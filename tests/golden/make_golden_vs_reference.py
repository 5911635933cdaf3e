"""Golden vectors for tests/test_oracle_vs_reference.py and tests/test_reference_call_shapes.py, generated from the UNMODIFIED
reference checkout (located by ref_loader: SHOWO_REFERENCE) so that both tests run without it.

    SHOWO_REFERENCE=<reference checkout> python tests/golden/make_golden_vs_reference.py
        -> tests/golden/oracle_vs_reference.npz   the reference's outputs on the tests' seeded inputs (large tensors sampled)
        -> tests/golden/reference_calls.json      every call the reference's scripts make on the objects the drop-in replaces
"""
from __future__ import annotations

import ast
import json
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, HERE)
import fixtures as FX  # noqa: E402
import ref_loader as R  # noqa: E402
from oracle import magvit_oracle as MO  # noqa: E402
from oracle import showo_oracle as O  # noqa: E402

VOC = O.ShowoVocab()

# ---------------------------------------------------------------- inputs shared with tests/test_oracle_vs_reference.py
T2I_CASES = ((5.0, 4), (0.0, 3))                          # (guidance_scale, timesteps) of the t2i_generate replay
MMU_SAMPLED_CASES = ((None, 0.8), (5, 1.3), (1, 0.5))     # (top_k, temperature) of the sampled mmu decode
SCHEDULES = (("cosine", {}), ("linear", {}), ("pow2", {}), ("pow0.5", {}), ("pow3", {}), ("sigmoid", {}),
             ("sigmoid", dict(start=-2, end=4, tau=0.7)))
N_SAMPLE = 32768                                          # entries kept of the logits / decoded pixels


def sample_index(n: int, seed: int) -> np.ndarray:
    """fixed flat positions at which a large output is stored"""
    return FX.rng(seed).integers(0, n, size=N_SAMPLE)


def noise_probe() -> np.ndarray:
    """the first draws of the two torch CPU streams the sampled paths consume (t2i: Generator(11), mmu: global seed 17);
    where a host's streams differ from these the sampled comparisons cannot be replayed"""
    a = torch.empty(8).exponential_(1, generator=torch.Generator().manual_seed(11))
    torch.manual_seed(17)
    b = torch.empty(8).exponential_(1)
    return torch.cat([a, b]).numpy()


def mask_case_rows():
    cond, uncond = O.make_t2i_prompts(3, VOC, seed=5)
    codes = torch.from_numpy(FX.rng(41).integers(0, 8192, size=(2, 256)).astype("int64"))
    return torch.cat([cond, uncond]), O.make_mmu_prompts(2, VOC, codes, q_len=9)


def mmu_case_rows():
    codes = torch.randint(0, 8192, (1, 256), generator=torch.Generator().manual_seed(2))
    mm = O.make_mmu_prompts(1, VOC, codes, q_len=7)
    return mm, O.create_attention_mask_for_mmu(mm)


def magvit_case_inputs():
    x = torch.rand(1, 3, 256, 256, generator=torch.Generator().manual_seed(0)) * 2 - 1
    ids = torch.randint(0, 8192, (1, 256), generator=torch.Generator().manual_seed(1))
    return x, ids


def schedule_points():
    return [torch.tensor(float(i) / 18) for i in range(19)] + [torch.rand(7, generator=torch.Generator().manual_seed(1))]


def logits_summary(lg: torch.Tensor) -> dict:
    """full-coverage digest of [n, L, V] logits: per-position argmax and logsumexp (float64), plus a fixed sample"""
    flat = lg.reshape(-1)
    return {"argmax": lg.argmax(-1).numpy().astype(np.int32), "lse": torch.logsumexp(lg.double(), -1).numpy(),
            "sample": flat[torch.from_numpy(sample_index(flat.numel(), 42))].numpy()}


def pixels_summary(img: torch.Tensor) -> dict:
    """full-coverage digest of decoded pixels [1, 3, H, W]: per (channel, row) mean (float64), plus a fixed sample"""
    flat = img.reshape(-1)
    return {"row_mean": img.double().mean(-1).numpy(), "sample": flat[torch.from_numpy(sample_index(flat.numel(), 43))].numpy()}


def pack_mask(add: torch.Tensor, key: str, out: dict):
    """an additive mask is 0 where attention is allowed and one fill value elsewhere: stored as bits + that value"""
    neg = float(add.min())
    assert add.dtype == torch.float32 and bool(((add == 0) | (add == neg)).all())
    out[key] = np.packbits((add == 0).numpy())
    out[key + "_shape"] = np.array(add.shape)
    out[key + "_neg"] = np.array([neg], dtype=np.float32)


# ---------------------------------------------------------------- call shapes of the reference's scripts
CALL_SCRIPTS = ["inference_t2i.py", "inference_mmu.py", "training/train.py", "training/train_w_clip_vit.py"]
CALL_OBJECTS = ["model", "vq_model", "vision_tower"]
CALL_FUNCS = ["get_mask_chedule", "mask_or_random_replace_tokens"]


def script_calls(path):
    """[object or None, method, positional count, keyword names, line] of every call on CALL_OBJECTS / CALL_FUNCS"""
    tree = ast.parse(open(path).read())
    out = []
    for node in ast.walk(tree):
        if not isinstance(node, ast.Call):
            continue
        f = node.func
        kws = [k.arg for k in node.keywords if k.arg]
        if isinstance(f, ast.Attribute) and isinstance(f.value, ast.Name) and f.value.id in CALL_OBJECTS:
            out.append([f.value.id, f.attr, len(node.args), kws, node.lineno])
        elif isinstance(f, ast.Name) and f.id in CALL_OBJECTS:             # model(input_ids, ...)
            out.append([f.id, "forward", len(node.args), kws, node.lineno])
        elif isinstance(f, ast.Name) and f.id in CALL_FUNCS:
            out.append([None, f.id, len(node.args), kws, node.lineno])
    return out


def main():
    torch.set_num_threads(8)
    mods = R.load_modules()
    out = {"noise_probe": noise_probe()}

    # ------------------------------------------------------------ tiny Showo (2 layers, full vocabulary)
    dims = O.PhiDims(**FX.TINY)
    W = O.make_showo_weights(dims, seed=3)
    model, _ = R.build_showo(dims, W)
    sd = {k: v for k, v in model.state_dict().items() if "rotary_emb" not in k}
    out["state_names"] = np.array(sorted(sd))
    out["state_shapes"] = np.array(["x".join(str(s) for s in sd[k].shape) for k in sorted(sd)])

    ids, mm = mask_case_rows()
    pack_mask(mods.prompting.create_attention_mask_predict_next(ids, pad_id=O.PAD, soi_id=O.SOI, eoi_id=O.EOI, rm_pad_in_image=True),
              "mask_t2i", out)
    pack_mask(mods.prompting.create_attention_mask_predict_next(ids, pad_id=O.PAD, soi_id=O.SOI, eoi_id=O.EOI, rm_pad_in_image=False),
              "mask_t2i_keep_pad", out)
    pack_mask(mods.prompting.create_attention_mask_for_mmu(mm, eoi_id=O.EOI), "mask_mmu", out)

    cond, uncond = O.make_t2i_prompts(2, VOC, seed=5)
    mask = O.create_attention_mask_predict_next(torch.cat([cond, uncond]))
    with torch.no_grad():
        lg = model(torch.cat([cond, uncond]), attention_mask=mask)
    out.update({"logits_" + k: v for k, v in logits_summary(lg).items()})
    for i, (w, T) in enumerate(T2I_CASES):
        c1 = cond.clone()
        with torch.no_grad():
            r = model.t2i_generate(input_ids=c1, uncond_input_ids=uncond.clone(), attention_mask=mask if w > 0 else mask[:2],
                                   guidance_scale=w, timesteps=T, generator=torch.Generator().manual_seed(11), config=R.t2i_config(VOC))
        out[f"t2i_ids_{i}"], out[f"t2i_final_input_ids_{i}"] = r.numpy(), c1.numpy()

    mm1, mk1 = mmu_case_rows()
    with torch.no_grad():
        out["mmu_greedy"] = torch.stack(model.mmu_generate(mm1, attention_mask=mk1, max_new_tokens=5, top_k=1)).numpy()
    for i, (top_k, temp) in enumerate(MMU_SAMPLED_CASES):
        torch.manual_seed(17)
        with torch.no_grad():
            r = model.mmu_generate(mm1, attention_mask=mk1, max_new_tokens=4, temperature=temp, top_k=top_k)
        out[f"mmu_sampled_{i}"] = torch.stack(r).numpy()

    for i, (method, kw) in enumerate(SCHEDULES):
        f = mods.sampling.get_mask_chedule(method, **kw)
        vals = [f(t) for t in schedule_points()]
        assert all(v.dtype == torch.float32 for v in vals)
        out[f"schedule_{i}"] = torch.cat([v.reshape(-1) for v in vals]).numpy()
    del model

    # ------------------------------------------------------------ MAGVIT-v2
    Wm = MO.make_magvit_weights(1)
    vq, _ = R.build_magvit(Wm)
    out["magvit_state_names"] = np.array(sorted(k for k in vq.state_dict() if not k.startswith("quantize.")))
    x, codes = magvit_case_inputs()
    with torch.no_grad():
        out["magvit_codes"] = vq.get_code(x).numpy()
        out.update({"magvit_decode_" + k: v for k, v in pixels_summary(vq.decode_code(codes)).items()})
    np.savez_compressed(os.path.join(HERE, "oracle_vs_reference.npz"), **out)
    print("oracle_vs_reference.npz", os.path.getsize(os.path.join(HERE, "oracle_vs_reference.npz")), "bytes")

    # ------------------------------------------------------------ call shapes
    calls = {s: script_calls(os.path.join(R.REF, s)) for s in CALL_SCRIPTS if os.path.exists(os.path.join(R.REF, s))}
    with open(os.path.join(HERE, "reference_calls.json"), "w") as f:      # one call per line
        f.write('{"objects": %s,\n "functions": %s,\n "calls": {\n' % (json.dumps(CALL_OBJECTS), json.dumps(CALL_FUNCS)))
        f.write(",\n".join(f'  {json.dumps(s)}: [\n' + ",\n".join("   " + json.dumps(c) for c in cs) + "]" for s, cs in calls.items()))
        f.write("}}\n")
    print("reference_calls.json", {s: len(c) for s, c in calls.items()})


if __name__ == "__main__":
    main()
