"""Seeded inputs shared by make_golden.py (which ran the reference on them) and the tests (which replay them).
Everything comes from numpy's Philox bit generator, so the tensors are identical on every box."""
from __future__ import annotations

import os

import numpy as np
import torch

from oracle import showo_oracle as O

HERE = os.path.dirname(os.path.abspath(__file__))
TINY = dict(hidden=256, n_layers=2, n_heads=4, ffn=1024)


def rng(seed):
    return np.random.Generator(np.random.Philox(seed))


def load(name):
    return np.load(os.path.join(HERE, name))


def record_observed(name, key, value):
    """Adds `key: value` to the JSON file `name` in $SHOWO_OBSERVED_DIR (nothing is written when it is unset).  The variant
    tests run the parity tests in parallel processes that record into the same file, so each update holds an exclusive
    lock on it from the read to the end of the write."""
    import fcntl
    import json
    out = os.environ.get("SHOWO_OBSERVED_DIR")
    if not out:
        return
    os.makedirs(out, exist_ok=True)
    with open(os.path.join(out, name), "a+") as f:
        fcntl.flock(f, fcntl.LOCK_EX)
        f.seek(0)
        text = f.read()
        d = json.loads(text) if text else {}
        d[key] = value
        f.truncate(0)
        json.dump(d, f, indent=1)


def unpack_mask(z, key):
    shape = tuple(int(v) for v in z[key + "_shape"])
    n = int(np.prod(shape))
    return torch.from_numpy(np.unpackbits(z[key])[:n].reshape(shape).astype(bool))


def mask_rows(voc):
    """id rows covering: long / short / no left padding (t2i), and mmu rows whose eoi position differs from row 0."""
    cond, uncond = O.make_t2i_prompts(3, voc, seed=5, min_len=8, max_len=64)
    full = cond[:1].clone()
    r = rng(9)
    full[0, :129] = torch.from_numpy(r.integers(0, 50257, size=129).astype("int64"))     # no padding at all
    full[0, 0] = O.T2I
    t2i = torch.cat([cond, uncond[:1], full])
    codes = torch.from_numpy(r.integers(0, 8192, size=(2, 256)).astype("int64"))
    mmu = O.make_mmu_prompts(2, voc, codes, q_len=12, seed=3)
    return {"t2i": t2i, "mmu": mmu}


def sampler_cases():
    return [dict(step=0, T=18, w=5.0, B=2, N=256, seed=100), dict(step=7, T=18, w=5.0, B=2, N=256, seed=101),
            dict(step=17, T=18, w=0.0, B=2, N=256, seed=102), dict(step=3, T=8, w=2.0, B=1, N=1024, seed=103),
            dict(step=11, T=12, w=1.5, B=3, N=64, seed=104)]


def sampler_case(case, voc, C=8192):
    r = rng(case["seed"])
    B, N = case["B"], case["N"]
    cond = torch.from_numpy(r.standard_normal(size=(B, N, C), dtype=np.float32)) * 1.2
    unc = torch.from_numpy(r.standard_normal(size=(B, N, C), dtype=np.float32)) * 1.2
    w = case["w"]
    logits = (1 + w) * cond - w * unc if w > 0 else cond
    ids_minus = torch.full((B, N), voc.mask_token_id, dtype=torch.int64)
    known = torch.from_numpy(r.random(size=(B, N), dtype=np.float32) < (case["step"] / case["T"]))
    codes = torch.from_numpy(r.integers(0, C, size=(B, N)).astype("int64"))
    ids_minus = torch.where(known, codes, ids_minus)
    expo = torch.from_numpy(r.standard_exponential(size=(B * N, C), dtype=np.float32))
    unif = torch.from_numpy(r.random(size=(B, N), dtype=np.float32))
    temp_in = 1.0
    for s in range(case["step"]):
        temp_in = temp_in * (1.0 - (s + 1) / case["T"])
    return dict(B=B, N=N, cond=cond, unc=unc, logits=logits, ids_minus=ids_minus, expo=expo, unif=unif, temp_in=temp_in)


def tiny_t2i_inputs(voc):
    cond, uncond = O.make_t2i_prompts(2, voc, seed=11)
    r = rng(12)
    fill = torch.from_numpy(r.random(size=(2, 256), dtype=np.float32) < 0.4)
    codes = torch.from_numpy(r.integers(0, 8192, size=(2, 256)).astype("int64")) + voc.image_offset
    cond[:, 130:386] = torch.where(fill, codes, cond[:, 130:386])
    uncond[:, 129:] = cond[:, 129:]
    mask = O.create_attention_mask_predict_next(torch.cat([cond, uncond]))
    return cond, uncond, mask


def tiny_mmu_inputs(voc):
    r = rng(13)
    codes = torch.from_numpy(r.integers(0, 8192, size=(3, 256)).astype("int64"))
    return O.make_mmu_prompts(3, voc, codes, q_len=10, seed=14)


def full_row_inputs(voc):
    cond, _ = O.make_t2i_prompts(1, voc, seed=1234)
    r = rng(15)
    fill = torch.from_numpy(r.random(size=(1, 256), dtype=np.float32) < 0.5)
    codes = torch.from_numpy(r.integers(0, 8192, size=(1, 256)).astype("int64")) + voc.image_offset
    cond[:, 130:386] = torch.where(fill, codes, cond[:, 130:386])
    return cond, O.create_attention_mask_predict_next(cond)


def magvit_inputs():
    r = rng(16)
    codes = torch.from_numpy(r.integers(0, 8192, size=(1, 256)).astype("int64"))
    pixels = torch.from_numpy(r.random(size=(1, 3, 256, 256), dtype=np.float32)) * 2 - 1
    return codes, pixels


TRAIN_COEFF = (1.0, 0.1, 1.0)          # loss = c0 * loss_t2i + c1 * loss_lm + c2 * loss_mmu (train.py:603-606 shape)


def train_batch(voc):
    """A mixed training batch the way training/train.py assembles it (2 t2i + 1 lm + 2 mmu rows, L = 387):
    ids, additive mask [5,1,L,L], labels (-100 = ignored), and the three batch sizes.
    t2i rows: image codes with ~60 % of the positions replaced by the mask token, labels = the true image-token ids there
    (mask_or_random_replace_tokens semantics, training/utils.py:77-154); lm row: next-token labels over a full text row;
    mmu rows: [mmu, soi, 256 codes, eoi, bos, text]: labels only on the text part."""
    r = rng(21)
    L = 387
    cond, _ = O.make_t2i_prompts(2, voc, seed=22)
    codes = torch.from_numpy(r.integers(0, 8192, size=(2, 256)).astype("int64")) + voc.image_offset
    masked = torch.from_numpy(r.random(size=(2, 256), dtype=np.float32) < 0.6)
    t2i = cond.clone()
    t2i[:, 130:386] = torch.where(masked, torch.full_like(codes, voc.mask_token_id), codes)
    lab_t2i = torch.full((2, L), -100, dtype=torch.int64)
    lab_t2i[:, 130:386] = torch.where(masked, codes, torch.full_like(codes, -100))
    lm = torch.from_numpy(r.integers(0, 50257, size=(1, L)).astype("int64"))
    lm[0, 0] = O.BOS
    lm[0, -1] = O.EOS
    lab_lm = lm.clone()
    mcodes = torch.from_numpy(r.integers(0, 8192, size=(2, 256)).astype("int64"))
    mmu = O.make_mmu_prompts(2, voc, mcodes, q_len=L - 260, seed=23)
    assert mmu.shape[1] == L
    lab_mmu = mmu.clone()
    lab_mmu[:, :260] = -100
    ids = torch.cat([t2i, lm, mmu])
    labels = torch.cat([lab_t2i, lab_lm, lab_mmu])
    mask = torch.cat([O.create_attention_mask_predict_next(torch.cat([t2i, lm])), O.create_attention_mask_for_mmu(mmu)])
    return ids, mask, labels, (2, 1, 2)


TRAIN_GRAD_PROBES = ["showo.model.layers.0.self_attn.q_proj.weight", "showo.model.layers.0.self_attn.k_layernorm.weight",
                     "showo.model.layers.1.mlp.fc2.bias", "showo.model.layers.1.self_attn.dense.weight",
                     "showo.model.final_layernorm.weight", "showo.lm_head.bias"]


# ---------------------------------------------------------------- full-size cases (make_golden_full.py / test_gpu_full_size.py)
def full_cfg1_inputs(voc):
    """BASELINE configs[1]: 8 prompts (SURVEY 8d seed 1234), CFG pair rows, all 256 image positions masked."""
    cond, uncond = O.make_t2i_prompts(8, voc, seed=1234)
    mask = O.create_attention_mask_predict_next(torch.cat([cond, uncond]))
    return cond, uncond, mask


def full_cfg1_noise(step, B=8, N=256, C=8192):
    """The noise denoise step `step` consumes, in the reference's order ([B*N, C] exponentials, then [B, N] uniforms)."""
    r = rng(1000 + step)
    expo = torch.from_numpy(r.standard_exponential(size=(B * N, C), dtype=np.float32))
    unif = torch.from_numpy(r.random(size=(B, N), dtype=np.float32))
    return expo, unif


def full_cfg2_inputs(voc):
    """BASELINE configs[2]: 16 MMU rows [mmu, soi, 256 codes, eoi, bos, 16 question ids], L0 = 276."""
    r = rng(31)
    codes = torch.from_numpy(r.integers(0, 8192, size=(16, 256)).astype("int64"))
    return O.make_mmu_prompts(16, voc, codes, q_len=16, seed=32)


def full_cfg3_inputs(voc1024):
    """BASELINE configs[3] geometry: one CFG pair at N = 1024 (L = 1155), half of the image tokens already decided."""
    cond, uncond = O.make_t2i_prompts(1, voc1024, seed=77)
    r = rng(33)
    fill = torch.from_numpy(r.random(size=(1, 1024), dtype=np.float32) < 0.5)
    codes = torch.from_numpy(r.integers(0, 8192, size=(1, 1024)).astype("int64")) + voc1024.image_offset
    cond[:, 130:1154] = torch.where(fill, codes, cond[:, 130:1154])
    uncond[:, 129:] = cond[:, 129:]
    mask = O.create_attention_mask_predict_next(torch.cat([cond, uncond]))
    return cond, uncond, mask
