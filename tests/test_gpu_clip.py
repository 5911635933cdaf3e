"""GPU parity tests of the CLIP ViT vision tower on the engine (clip_forward, csrc/clip.cu) through the drop-in class
show-o_b200/clip_tower.py, against oracle/clip_oracle.py (itself pinned to the live `transformers` model in
tests/test_oracle_golden.py) on seeded weights and pixels.

Tolerance: bf16 operands with fp32 accumulation and an fp32 residual stream against an fp32 reference; the features are the
penultimate block's residual stream (std about 1 with these weights).  Bounds are stated next to each assert, the observed errors are
recorded in $SHOWO_OBSERVED_DIR/parity_observed.json when that variable is set.
"""
import os

import numpy as np
import pytest
import torch

import fixtures as FX
import showo_b200
from oracle import clip_oracle as CO
from showo_b200 import CLIPVisionTower

pytestmark = pytest.mark.gpu


def _record(key, value):
    FX.record_observed("parity_observed.json", key, value)


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda", 0)


def _pixels(seed, B, S):
    r = np.random.Generator(np.random.Philox(seed))
    return torch.from_numpy(r.standard_normal(size=(B, 3, S, S), dtype=np.float32))       # image-processor output is ~N(0, 1) per channel


def _tower(d, dev, seed=2):
    W = CO.make_clip_weights(d, seed=seed)
    t = CLIPVisionTower(dict(image_size=d.image_size, patch_size=d.patch_size, hidden=d.hidden, n_layers=d.n_layers, n_heads=d.n_heads, ffn=d.ffn))
    t.load_weights(W, device=dev)
    return W, t


@pytest.mark.parametrize("geo", [dict(image_size=56, patch_size=14, hidden=256, n_layers=3, n_heads=4, ffn=512),        # 17 tokens: mma.sync attention only
                                 dict(image_size=224, patch_size=14, hidden=128, n_layers=2, n_heads=2, ffn=256)])      # 257 tokens: two tcgen05 tiles + 1 tail row
def test_clip_tower_small_geometries_against_the_oracle(dev, geo):
    d = CO.ClipDims(**geo)
    W, t = _tower(d, dev)
    x = _pixels(7, 3, d.image_size)
    with torch.no_grad():
        hs = CO.hidden_states(x, W, d)
    got = t(x.to(dev)).cpu()
    ref = hs[-2][:, 1:]
    err = (got - ref).abs()
    print(f"clip {geo['image_size']}px/{d.n_layers}L: max {err.max():.4f} mean {err.mean():.5f} (ref std {ref.std():.3f})")
    _record(f"clip_small_{geo['image_size']}", {"max_abs": float(err.max()), "mean_abs": float(err.mean()), "ref_std": float(ref.std())})
    assert got.shape == ref.shape and err.max().item() < 0.025 and err.mean().item() < 0.004      # observed 0.0106 / 0.0018
    # the other selections of clip_encoder.py:29-37 and every hidden_states index
    t.select_feature = "cls_patch"
    assert (t(x.to(dev)).cpu() - hs[-2]).abs().max().item() < 0.025
    t.select_feature = "patch"
    for sel in (0, 1, -1):
        t.select_layer = sel
        assert (t(x.to(dev)).cpu() - hs[sel][:, 1:]).abs().max().item() < 0.025, sel
    t.select_layer = -2
    # list input (clip_encoder.py:41-46), dtype of the input kept, batch independence bit for bit
    fl = t([x[0].to(dev), x[1].to(dev).half()])
    assert fl[0].shape == (1, d.n_tokens - 1, d.hidden) and fl[1].dtype == torch.float16
    assert torch.equal(fl[0][0].cpu(), got[0])
    assert t.kernel_launches() > 0
    t.select_feature = "pooled"
    with pytest.raises(ValueError):
        t(x.to(dev))


def test_clip_vit_l14_336_full_size_against_the_oracle(dev):
    """openai/clip-vit-large-patch14-336 geometry (24 layers, hidden 1024, 16 heads, MLP 4096, 577 tokens), seeded weights: the features
    the MMU path consumes ([B, 576, 1024], hidden_states[-2] without CLS) vs the fp32 oracle; then through Showo.mm_projector like
    inference_mmu.py:128-131 does."""
    d = CO.ClipDims()
    W, t = _tower(d, dev)
    x = _pixels(11, 2, 336)
    torch.set_num_threads(max(1, os.cpu_count() or 1))
    with torch.no_grad():
        ref = CO.tower_features(x, W, d)
    got = t(x.to(dev))
    assert got.shape == (2, 576, 1024) and torch.isfinite(got).all()
    err = (got.cpu() - ref).abs()
    rel = float((got.cpu() - ref).norm() / ref.norm())
    print(f"clip ViT-L/14-336: rel L2 {rel:.5f}, max {err.max():.4f}, mean {err.mean():.5f} (ref std {ref.std():.3f}, max {ref.abs().max():.2f}); "
          f"{t.kernel_launches()} launches")
    _record("clip_vit_l14_336", {"rel_l2": rel, "max_abs": float(err.max()), "mean_abs": float(err.mean()), "ref_std": float(ref.std()),
                                 "ref_max": float(ref.abs().max()), "launches": t.kernel_launches()})
    assert rel < 0.012 and err.max().item() < 0.16          # observed rel L2 0.0058, max 0.076 (ref std 2.7, max 13.1)
    # timing of one batch of 16 images (a config-3 MMU batch), device-side
    xb = _pixels(12, 16, 336).to(dev)
    t(xb)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(3):
        t(xb)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / 3
    flop = 16 * 23 * (577 * 2 * (4 * 1024 * 1024 + 2 * 1024 * 4096) + 4 * 577 * 577 * 1024) + 16 * 576 * 2 * 1024 * 588
    print(f"clip ViT-L/14-336, 16 images: {ms:.2f} ms = {16e3 / ms:.0f} images/s, {flop / ms / 1e9:.0f} TFLOP/s")
    _record("clip_vit_l14_336_speed", {"ms_per_16_images": ms, "tflops": flop / ms / 1e9})


def test_inference_mmu_w_clip_vit_call_shape_end_to_end(dev):
    """The w_clip_vit branch of inference_mmu.py:100-151 as the script writes it, every stage on the engine: `vision_tower(pixel_values[None])`
    (CLIP ViT, 336 x 336 -> [1, 576, 1024]) -> `model.mm_projector(...)` -> `model.showo.model.embed_tokens(input_ids_llava)` -> cat around the
    image embeddings -> `create_attention_mask_for_mmu_vit` (dense) -> `model.mmu_generate(input_embeddings=, attention_mask=, top_k=1, eot_token=)`
    -> `torch.stack(cont_toks_list).squeeze()[None]`.  A 1-layer backbone of the real width (the projector's output is 2048 wide) and a 3-layer
    ViT of the real width; the input embeddings and the first generated token against the oracles' fp32 flow."""
    from oracle import showo_oracle as O
    dims = O.PhiDims(hidden=2048, n_layers=1, n_heads=32, ffn=2048)
    W = O.make_showo_weights(dims, seed=8, w_clip_vit=True)
    m = showo_b200.Showo(True, dims.vocab_size, 50295, phi_dims=dict(hidden=2048, n_layers=1, n_heads=32, ffn=2048)).to(dev)
    m.load_state_dict(W, strict=True)
    m.eval()
    cd = CO.ClipDims(n_layers=3)
    CW, vision_tower = _tower(cd, dev)
    SYS = 28
    r = np.random.Generator(np.random.Philox(23))
    pixel_values = _pixels(21, 1, 336)[0]
    mmu, soi, eoi = 50301, 50296, 50297
    sys_ids = torch.from_numpy(r.integers(0, 50257, size=(1, SYS)).astype("int64"))
    q_ids = torch.from_numpy(r.integers(0, 50257, size=(1, 12)).astype("int64"))
    input_ids_llava = torch.cat([torch.full((1, 1), mmu), sys_ids, torch.full((1, 1), soi), torch.full((1, 1), eoi), q_ids], dim=1).long()
    with torch.no_grad():
        images_embeddings = vision_tower(pixel_values[None].to(dev))
        assert images_embeddings.shape == (1, 576, 1024)
        images_embeddings = m.mm_projector(images_embeddings)
        text_embeddings = m.showo.model.embed_tokens(input_ids_llava.to(dev))
        part1, part2 = text_embeddings[:, :2 + SYS, :], text_embeddings[:, 2 + SYS:, :]
        input_embeddings = torch.cat((part1, images_embeddings, part2), dim=1)
        L = input_embeddings.shape[1]
        attention_mask_llava = O.additive_from_allowed(O.mask_allowed_mmu_vit(1, L, system_prompt_len=SYS)).to(dev)      # create_attention_mask_for_mmu_vit
        cont_toks_list = m.mmu_generate(input_embeddings=input_embeddings, attention_mask=attention_mask_llava[0].unsqueeze(0),
                                        max_new_tokens=6, top_k=1, eot_token=50256)
    cont = torch.stack(cont_toks_list).squeeze()[None]
    assert 1 <= cont.numel() <= 6 and cont.dtype == torch.int64          # (a single token squeezes to [1], like in the reference)
    # ---- the oracles' flow in fp32
    with torch.no_grad():
        f_ref = CO.tower_features(pixel_values[None], CW, cd)
        h = torch.nn.functional.gelu(f_ref @ W["mm_projector.0.weight"].T + W["mm_projector.0.bias"])
        v_ref = h @ W["mm_projector.2.weight"].T + W["mm_projector.2.bias"]
        e_ref = W["showo.model.embed_tokens.weight"][input_ids_llava]
        emb_ref = torch.cat((e_ref[:, :2 + SYS], v_ref, e_ref[:, 2 + SYS:]), dim=1)
        lg = O.showo_logits(W, dims, input_embeddings=emb_ref, add_mask=attention_mask_llava.cpu())[:, -1]
    rel = float((input_embeddings.cpu() - emb_ref).norm() / emb_ref.norm())
    top2 = lg.topk(2)
    first = int(cont.reshape(-1)[0])
    print(f"inference_mmu w_clip_vit flow: input embeddings rel L2 {rel:.5f}; first token {first} (oracle {int(top2.indices[0, 0])}, margin {float(top2.values[0, 0] - top2.values[0, 1]):.4f})")
    _record("inference_mmu_w_clip_vit_flow", {"input_embeddings_rel_l2": rel, "first_token_equal": first == int(top2.indices[0, 0])})
    assert rel < 0.01
    if first != int(top2.indices[0, 0]):
        assert float(top2.values[0, 0] - top2.values[0, 1]) < 0.06 and first == int(top2.indices[0, 1])
