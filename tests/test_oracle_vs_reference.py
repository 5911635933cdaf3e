"""Pin of the oracle against the UNMODIFIED reference Python on the same seeded inputs: what the reference computed is stored in
tests/golden/oracle_vs_reference.npz (tests/golden/make_golden_vs_reference.py ran it), so the comparison needs no reference
checkout.  Large outputs are kept as a full-coverage digest (per-position argmax / logsumexp, per-row means) plus a fixed sample."""
import numpy as np
import pytest
import torch

import fixtures as FX
import make_golden_vs_reference as G
from oracle import magvit_oracle as MO
from oracle import showo_oracle as O

VOC = O.ShowoVocab()


@pytest.fixture(scope="module")
def z():
    return FX.load("oracle_vs_reference.npz")


@pytest.fixture(scope="module")
def tiny():
    dims = O.PhiDims(hidden=256, n_layers=2, n_heads=4, ffn=1024)
    return dims, O.make_showo_weights(dims, seed=3)


def _require_reference_noise(z):
    """the sampled paths replay torch's CPU noise streams: only comparable where they match the ones the reference drew"""
    if not np.array_equal(G.noise_probe(), z["noise_probe"]):
        pytest.skip("torch CPU exponential_ stream differs on this host; the sampled replay needs identical noise")


def _mask(z, key):
    allowed = FX.unpack_mask(z, key)
    return torch.zeros(allowed.shape).masked_fill_(~allowed, float(z[key + "_neg"][0]))


def test_state_dict_keys_match_reference(tiny, z):
    dims, W = tiny
    ref = {str(k): tuple(int(s) for s in str(v).split("x")) for k, v in zip(z["state_names"], z["state_shapes"])}
    assert set(ref) == set(W.keys())
    import showo_b200
    ours = showo_b200.Showo(False, dims.vocab_size, VOC.llm_vocab_size, phi_dims=dict(hidden=256, n_layers=2, n_heads=4, ffn=1024))
    assert set(ours.state_dict().keys()) == set(ref)
    for k, v in ours.state_dict().items():
        assert tuple(v.shape) == ref[k], k


def test_masks_equal_reference(z):
    ids, mm = G.mask_case_rows()
    assert torch.equal(_mask(z, "mask_t2i"), O.create_attention_mask_predict_next(ids))
    assert torch.equal(_mask(z, "mask_t2i_keep_pad"), O.create_attention_mask_predict_next(ids, rm_pad_in_image=False))
    assert torch.equal(_mask(z, "mask_mmu"), O.create_attention_mask_for_mmu(mm))


def test_logits_and_t2i_generate_equal_reference(tiny, z):
    dims, W = tiny
    cond, uncond = O.make_t2i_prompts(2, VOC, seed=5)
    mask = O.create_attention_mask_predict_next(torch.cat([cond, uncond]))
    with torch.no_grad():
        lo = O.showo_logits(W, dims, input_ids=torch.cat([cond, uncond]), add_mask=mask)
    got = G.logits_summary(lo)
    assert np.abs(got["sample"] - z["logits_sample"]).max() < 1e-5
    assert np.abs(got["lse"] - z["logits_lse"]).max() < 1e-5
    # the reference's argmax is (within the same bound) a maximum of ours: robust to exact ties
    at_ref = lo.gather(-1, torch.from_numpy(z["logits_argmax"]).long()[..., None])[..., 0]
    assert (lo.max(-1).values - at_ref).max().item() < 1e-5
    _require_reference_noise(z)
    for i, (w, T) in enumerate(G.T2I_CASES):
        c2 = cond.clone()
        with torch.no_grad():
            o = O.t2i_generate(W, dims, VOC, c2, uncond.clone(), mask if w > 0 else mask[:2], guidance_scale=w, timesteps=T,
                               generator=torch.Generator().manual_seed(11))
        assert np.array_equal(o.numpy(), z[f"t2i_ids_{i}"]) and np.array_equal(c2.numpy(), z[f"t2i_final_input_ids_{i}"])


def test_mmu_generate_equals_reference(tiny, z):
    dims, W = tiny
    mm, mk = G.mmu_case_rows()
    with torch.no_grad():
        o = O.mmu_generate(W, dims, mm, mk, max_new_tokens=5, top_k=1)
    assert np.array_equal(torch.stack(o).numpy(), z["mmu_greedy"])
    # sampled decode (modeling_showo.py:219-228): temperature, top-k filter, softmax, torch.multinomial(p, 1) -- whose
    # single-sample path is the exponential race the oracle (and the CUDA kernel) restate; both draw from the global RNG
    _require_reference_noise(z)
    for i, (top_k, temp) in enumerate(G.MMU_SAMPLED_CASES):
        torch.manual_seed(17)
        with torch.no_grad():
            o = O.mmu_generate(W, dims, mm, mk, max_new_tokens=4, temperature=temp, top_k=top_k)
        assert np.array_equal(torch.stack(o).numpy(), z[f"mmu_sampled_{i}"]), (top_k, temp)


def test_magvit_equals_reference(z):
    W = MO.make_magvit_weights(1)
    assert set(str(k) for k in z["magvit_state_names"]) == set(W.keys())
    x, ids = G.magvit_case_inputs()
    with torch.no_grad():
        assert np.array_equal(MO.get_code(x, W).numpy(), z["magvit_codes"])
        got = G.pixels_summary(MO.decode_code(ids, W))
    assert np.abs(got["sample"] - z["magvit_decode_sample"]).max() < 1e-5
    assert np.abs(got["row_mean"] - z["magvit_decode_row_mean"]).max() < 1e-5


def test_mask_schedules_equal_reference(z):
    """get_mask_chedule (sic) and every schedule it hands out, bit for bit on the fp32 grid the sampler evaluates them on
    (models/sampling.py:39-78)."""
    import showo_b200
    for i, (method, kw) in enumerate(G.SCHEDULES):
        ours = showo_b200.get_mask_chedule(method, **kw)
        vals = [ours(t) for t in G.schedule_points()]
        assert all(v.dtype == torch.float32 for v in vals), method
        assert np.array_equal(torch.cat([v.reshape(-1) for v in vals]).numpy(), z[f"schedule_{i}"]), (method, kw)
    with pytest.raises(ValueError):
        showo_b200.get_mask_chedule("nope")
