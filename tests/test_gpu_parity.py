"""GPU parity tests (run with -m gpu on the B200 box): every CUDA kernel and the assembled hot path against the CPU
oracle on seeded inputs and against the committed golden vectors, all calls going through the C ABI.

Tolerances (stated once): the engine computes in bf16 with fp32 accumulation, the reference in fp32.
  * integer / index outputs given identical fp32 logits + noise (sampler, LFQ bits above the sign margin): bit-exact
  * backbone logits: |d| <= 0.03 for the 2-layer test geometry, <= 0.08 for the full 24-layer model (logit std 0.91;
    SURVEY.md section 7 'hard parts' measured 0.045-0.054 for bf16 autocast on CPU)
  * token decisions made from engine logits may differ from the oracle only where the oracle's decision margin is
    below 2x the measured logit error (a flip needs two logits to cross)
"""
import ctypes as C
import math
import os

import numpy as np
import pytest
import torch

import fixtures as FX
import showo_b200
from oracle import magvit_oracle as MO
from oracle import showo_oracle as O
from showo_b200 import _lib, masks as M

pytestmark = pytest.mark.gpu
VOC = O.ShowoVocab()
TOL_TINY, TOL_FULL = 0.03, 0.08


def _record(key, value):
    FX.record_observed("parity_observed.json", key, value)


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda", 0)


@pytest.fixture(scope="module")
def lib():
    return _lib.require_gpu()


def S():
    return _lib.current_stream_ptr()


def cfg_ns(n_tok=256):
    from types import SimpleNamespace as NS
    return NS(model=NS(showo=NS(num_vq_tokens=n_tok, num_new_special_tokens=10, llm_vocab_size=50295)),
              dataset=NS(preprocessing=NS(max_seq_length=128)))


@pytest.fixture(scope="module")
def tiny(dev):
    dims = O.PhiDims(**FX.TINY)
    W = O.make_showo_weights(dims, seed=3)
    m = showo_b200.Showo(False, dims.vocab_size, VOC.llm_vocab_size, phi_dims=FX.TINY, materialize=False)
    m.load_weights(W, device=dev)
    return dims, W, m


# ------------------------------------------------------------------------------------------------ kernels
@pytest.mark.parametrize("Mm,N,K,bn", [(128, 256, 64, 256), (128, 64, 128, 64), (300, 520, 192, 128), (1, 64, 64, 64),
                                       (4128, 2048, 2048, 256), (1000, 2048, 10240, 256), (16, 58498, 256, 64),
                                       (257, 1000, 200, 0), (129, 8192, 2048, 128)])
def test_gemm_tcgen05_against_fp32(lib, dev, Mm, N, K, bn):
    g = torch.Generator(device=dev).manual_seed(Mm * 7 + N)
    A = (torch.randn(Mm, K, device=dev, generator=g) * 0.5).bfloat16()
    Bw = (torch.randn(N, K, device=dev, generator=g) * 0.05).bfloat16()
    bias = torch.randn(N + 1, device=dev, generator=g)[1:]          # deliberately NOT 16-byte aligned
    ref = A.float() @ Bw.float().t() + bias
    out = torch.full((Mm, N), float("nan"), device=dev)
    _lib.check(lib.showo_gemm_bf16(_lib.ptr(A), K, _lib.ptr(Bw), K, Mm, N, K, _lib.ptr(out), N, _lib.ptr(bias), None, 0, N, 2, bn, S()))
    assert (out - ref).abs().max().item() < 1e-3
    gf = (N // 2) // 32 * 32
    out16 = torch.zeros(Mm, N, device=dev, dtype=torch.bfloat16)
    _lib.check(lib.showo_gemm_bf16(_lib.ptr(A), K, _lib.ptr(Bw), K, Mm, N, K, _lib.ptr(out16), N, _lib.ptr(bias), None, 0, gf, 0, bn, S()))
    r16 = ref.clone()
    r16[:, gf:] = O.gelu_new(ref[:, gf:])
    assert ((out16.float() - r16).abs() <= r16.abs() * 2 ** -7 + 1e-2).all()
    res = torch.randn(Mm, N, device=dev, generator=g)
    outr = res.clone()
    _lib.check(lib.showo_gemm_bf16(_lib.ptr(A), K, _lib.ptr(Bw), K, Mm, N, K, _lib.ptr(outr), N, _lib.ptr(bias), _lib.ptr(outr), N, N, 1, bn, S()))
    assert (outr - (ref + res)).abs().max().item() < 1e-3


@pytest.mark.parametrize("Mf,Nf,K", [(2048, 10240, 9240), (640, 128, 100), (128, 384, 77), (58498, 256, 300), (14336, 2048, 1155)])
def test_gemm_token_major_operands_against_fp32(lib, dev, Mf, Nf, K):
    """weight-gradient form dW = dY^T X: both operands [tokens, features] as they lie (MN-major UMMA descriptors), ragged token counts,
    feature counts that leave tiles partly empty, row strides wider than the feature count."""
    g = torch.Generator(device=dev).manual_seed(Mf + Nf + K)
    lda, ldb = (Mf + 7) // 8 * 8 + 8, Nf + 16
    A = torch.zeros(K, lda, device=dev, dtype=torch.bfloat16)
    Bx = torch.zeros(K, ldb, device=dev, dtype=torch.bfloat16)
    A[:, :Mf] = (torch.randn(K, Mf, device=dev, generator=g) * 0.1).bfloat16()
    Bx[:, :Nf] = (torch.randn(K, Nf, device=dev, generator=g) * 0.5).bfloat16()
    A[:, Mf:] = 7.0                                   # the pad columns must not leak into the product
    Bx[:, Nf:] = 7.0
    ref = A[:, :Mf].float().t() @ Bx[:, :Nf].float()
    out = torch.full((Mf, Nf), float("nan"), device=dev)
    _lib.check(lib.showo_gemm_bf16(_lib.ptr(A), lda, _lib.ptr(Bx), ldb, Mf, Nf, K, _lib.ptr(out), Nf, None, None, 0, Nf, 3, 0, S()))
    assert not torch.isnan(out).any()
    assert (out - ref).abs().max().item() < 2e-3 * max(1.0, (K / 256) ** 0.5)
    out2 = torch.full((Mf, Nf), float("nan"), device=dev)
    _lib.check(lib.showo_gemm_bf16(_lib.ptr(A), lda, _lib.ptr(Bx), ldb, Mf, Nf, K, _lib.ptr(out2), Nf, None, None, 0, Nf, 3, 0, S()))
    assert torch.equal(out, out2)


@pytest.mark.parametrize("Mm,N,K", [(16, 2048, 10240), (16, 58498, 2048), (3, 1000, 256), (16, 14336, 2048), (1, 64, 64),
                                    (9, 2048, 2048)])
def test_skinny_weight_streaming_gemm(lib, dev, Mm, N, K):
    """decode path (M <= 16, block_n = 0): mma.sync weight streaming with deterministic split-K."""
    g = torch.Generator(device=dev).manual_seed(Mm + N)
    A = (torch.randn(Mm, K, device=dev, generator=g) * 0.5).bfloat16()
    Bw = (torch.randn(N, K, device=dev, generator=g) * 0.05).bfloat16()
    bias = torch.randn(N, device=dev, generator=g)
    ref = A.float() @ Bw.float().t() + bias
    outs = []
    for _ in range(2):
        out = torch.full((Mm, N), float("nan"), device=dev)
        _lib.check(lib.showo_gemm_bf16(_lib.ptr(A), K, _lib.ptr(Bw), K, Mm, N, K, _lib.ptr(out), N, _lib.ptr(bias), None, 0, N, 2, 0, S()))
        outs.append(out)
    assert (outs[0] - ref).abs().max().item() < 2e-3
    assert torch.equal(outs[0], outs[1])                      # split-K partials are summed in a fixed order
    gf = (N // 2) // 64 * 64
    out16 = torch.zeros(Mm, N, device=dev, dtype=torch.bfloat16)
    _lib.check(lib.showo_gemm_bf16(_lib.ptr(A), K, _lib.ptr(Bw), K, Mm, N, K, _lib.ptr(out16), N, _lib.ptr(bias), None, 0, gf, 0, 0, S()))
    r16 = ref.clone()
    r16[:, gf:] = O.gelu_new(ref[:, gf:])
    assert ((out16.float() - r16).abs() <= r16.abs() * 2 ** -7 + 1e-2).all()
    res = torch.randn(Mm, N, device=dev, generator=g)
    outr = res.clone()
    _lib.check(lib.showo_gemm_bf16(_lib.ptr(A), K, _lib.ptr(Bw), K, Mm, N, K, _lib.ptr(outr), N, _lib.ptr(bias), _lib.ptr(outr), N, N, 1, 0, S()))
    assert (outr - (ref + res)).abs().max().item() < 2e-3


def test_gemm_streamk_residual_epilogue_exact_and_deterministic(lib, dev):
    """the layer's second GEMM at full size (4128 x 2048 x 10240, x += A W^T + b: 136 pair tiles on 74 clusters -> stream-K with parked
    partial tiles): exact on small-integer operands whatever the split, identical from run to run, strided A like the engine's."""
    Mm, N, K, ld = 4128, 2048, 10240, 14336
    g = torch.Generator(device=dev).manual_seed(11)
    buf = torch.randint(-4, 5, (Mm, ld), device=dev, generator=g).to(torch.bfloat16)
    Bw = torch.randint(-2, 3, (N, K), device=dev, generator=g).to(torch.bfloat16)
    bias = torch.randint(-8, 9, (N,), device=dev, generator=g).float()
    res = torch.randint(-64, 65, (Mm, N), device=dev, generator=g).float()
    A = buf[:, ld - K:]
    ref = A.float() @ Bw.float().t() + bias + res
    outs = []
    for _ in range(3):
        x = res.clone()
        _lib.check(lib.showo_gemm_bf16(_lib.ptr(A), ld, _lib.ptr(Bw), K, Mm, N, K, _lib.ptr(x), N, _lib.ptr(bias), _lib.ptr(x), N, N, 1, 0, S()))
        outs.append(x)
    assert torch.equal(outs[0], ref)
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[1], outs[2])
    # random bf16 operands: fp32 accuracy with the partial sums added in a fixed order
    A2 = (torch.randn(Mm, K, device=dev, generator=g) * 0.5).bfloat16()
    B2 = (torch.randn(N, K, device=dev, generator=g) * 0.02).bfloat16()
    ref2 = A2.float() @ B2.float().t() + bias + res
    x1, x2 = res.clone(), res.clone()
    for x in (x1, x2):
        _lib.check(lib.showo_gemm_bf16(_lib.ptr(A2), K, _lib.ptr(B2), K, Mm, N, K, _lib.ptr(x), N, _lib.ptr(bias), _lib.ptr(x), N, N, 1, 0, S()))
    assert (x1 - ref2).abs().max().item() < 2e-3 and torch.equal(x1, x2)


def test_gemm_linearity_and_strided_operands(lib, dev):
    """size-independent properties at full size: C(A1 + A2) = C(A1) + C(A2) for exactly representable sums; A may be
    a strided column block of a wider buffer (the engine reads attn|act out of the k|v|q|act buffer)."""
    Mm, N, K, ld = 4128, 2048, 10240, 14336
    g = torch.Generator(device=dev).manual_seed(5)
    buf = torch.randint(-4, 5, (Mm, ld), device=dev, generator=g).to(torch.bfloat16)
    Bw = torch.randint(-2, 3, (N, K), device=dev, generator=g).to(torch.bfloat16)
    A = buf[:, ld - K:]
    out = torch.empty(Mm, N, device=dev)
    _lib.check(lib.showo_gemm_bf16(_lib.ptr(A), ld, _lib.ptr(Bw), K, Mm, N, K, _lib.ptr(out), N, None, None, 0, N, 2, 0, S()))
    ref = A.float() @ Bw.float().t()              # small integers: exact in fp32 whatever the summation order
    assert torch.equal(out, ref)


def test_layernorm(lib, dev):
    for D in (256, 2048):
        x = torch.randn(777, D, device=dev) * 2 + 0.3
        g, b = torch.randn(D, device=dev), torch.randn(D, device=dev)
        out = torch.zeros(777, D, device=dev, dtype=torch.bfloat16)
        _lib.check(lib.showo_layernorm_test(_lib.ptr(x), _lib.ptr(g), _lib.ptr(b), 1e-5, _lib.ptr(out), 777, D, S()))
        ref = torch.nn.functional.layer_norm(x, (D,), g, b, 1e-5)
        assert ((out.float() - ref).abs() <= ref.abs() * 2 ** -8 + 1e-3).all()


def _attn_ref(qkv, n_seq, rows, pos0, H, qg, qb, kg, kb, descs, dev, kprev=None, vprev=None):
    D = H * 64
    x = qkv.float().view(n_seq, rows, -1)
    k = x[..., :D].reshape(n_seq, rows, H, 64).transpose(1, 2)
    v = x[..., D:2 * D].reshape(n_seq, rows, H, 64).transpose(1, 2)
    q = x[..., 2 * D:3 * D].reshape(n_seq, rows, H, 64).transpose(1, 2)
    q = torch.nn.functional.layer_norm(q, (64,), qg, qb, 1e-5)
    k = torch.nn.functional.layer_norm(k, (64,), kg, kb, 1e-5)
    cos, sin = O.rotary_tables(O.PhiDims(), pos0 + rows)
    cos, sin = cos.to(dev)[pos0:], sin.to(dev)[pos0:]
    q = O.apply_partial_rotary(q, cos, sin, 32).bfloat16().float()
    k = O.apply_partial_rotary(k, cos, sin, 32).bfloat16().float()
    if kprev is not None:
        k, v = torch.cat([kprev, k], 2), torch.cat([vprev, v], 2)
    L = k.shape[2]
    s = (q @ k.transpose(-1, -2)) / 8.0
    for i, d in enumerate(descs):
        s[i, :, ~M.predicate(L, d, dev)[pos0:pos0 + rows]] = float("-inf")
    return (torch.softmax(s, -1) @ v).transpose(1, 2).reshape(n_seq, rows, D), k, v


@pytest.mark.parametrize("n_seq,rows,descs", [
    (2, 387, [(100, 129, 387, 0, 0), (0, 129, 387, 0, 0)]),          # t2i rows, with / without left padding
    (2, 200, [(0, 0, 0, 0, 0), (0, 0, 0, 3, 150)]),                  # pure causal (lm), mmu_vit-style window
    (1, 64, [(5, 0, 0, 0, 0)]), (1, 1, [(0, 0, 0, 0, 0)]),           # one full tile, a single row
    (3, 130, [(20, 60, 130, 0, 0), (0, 0, 0, 0, 77), (128, 0, 0, 0, 0)]),
    (1, 1155, [(60, 129, 1155, 0, 0)]),                              # 512x512 geometry
])
def test_omni_attention_prefill(lib, dev, n_seq, rows, descs):
    H = 4
    D, ld = H * 64, 3 * H * 64 + 128
    g = torch.Generator(device=dev).manual_seed(rows)
    Lmax = (rows + 63) // 64 * 64
    qkv = torch.randn(n_seq * rows, ld, device=dev, generator=g).bfloat16()
    qg, kg = 1 + 0.1 * torch.randn(64, device=dev, generator=g), 1 + 0.1 * torch.randn(64, device=dev, generator=g)
    qb, kb = 0.1 * torch.randn(64, device=dev, generator=g), 0.1 * torch.randn(64, device=dev, generator=g)
    ref, kk, vv = _attn_ref(qkv, n_seq, rows, 0, H, qg, qb, kg, kb, descs, dev)
    kc = torch.zeros(n_seq, H, Lmax, 64, device=dev, dtype=torch.bfloat16)
    vc = torch.zeros(n_seq, H, 64, Lmax, device=dev, dtype=torch.bfloat16)
    buf = qkv.clone()
    _lib.check(lib.showo_attention_test(_lib.ptr(buf), ld, n_seq, rows, 0, H, _lib.ptr(qg), _lib.ptr(qb), _lib.ptr(kg), _lib.ptr(kb),
                                        1e-5, 10000.0, 32, _lib.ptr(kc), _lib.ptr(vc), Lmax, rows, _lib.masks_array(descs), S()))
    got = buf.view(n_seq, rows, ld)[..., 2 * D:3 * D].float()
    assert (kc[:, :, :rows].float() - kk).abs().max().item() < 0.04          # 1 bf16 ulp of |k| < 8
    assert torch.equal(vc[:, :, :, :rows].float(), vv.transpose(-1, -2))
    for i, d in enumerate(descs):
        assert (got[i, d[0]:] - ref[i, d[0]:]).abs().max().item() < 0.02, (i, d)
    assert not torch.isnan(got).any()
    assert torch.equal(buf.view(n_seq, rows, ld)[..., 3 * D:], qkv.view(n_seq, rows, ld)[..., 3 * D:])   # act block untouched


def test_omni_attention_step_and_decode_against_cache(lib, dev):
    """denoise-step style (prefix K/V already cached, queries at pos0 = 129) and single-query decode."""
    H, n_seq, P, R = 4, 2, 129, 258
    D, ld, L, Lmax = H * 64, 3 * H * 64 + 128, P + R, 448
    descs = [(40, P, L, 0, 0), (126, P, L, 0, 0)]
    g = torch.Generator(device=dev).manual_seed(3)
    full = torch.randn(n_seq * L, ld, device=dev, generator=g).bfloat16()
    one, zero = torch.ones(64, device=dev), torch.zeros(64, device=dev)
    ref, _, _ = _attn_ref(full, n_seq, L, 0, H, one, zero, one, zero, descs, dev)
    kc = torch.zeros(n_seq, H, Lmax, 64, device=dev, dtype=torch.bfloat16)
    vc = torch.zeros(n_seq, H, 64, Lmax, device=dev, dtype=torch.bfloat16)
    f3 = full.view(n_seq, L, ld)
    pre, img = f3[:, :P].reshape(-1, ld).clone(), f3[:, P:].reshape(-1, ld).clone()
    args = (_lib.ptr(one), _lib.ptr(zero), _lib.ptr(one), _lib.ptr(zero), 1e-5, 10000.0, 32, _lib.ptr(kc), _lib.ptr(vc), Lmax)
    _lib.check(lib.showo_attention_test(_lib.ptr(pre), ld, n_seq, P, 0, H, *args, P, _lib.masks_array(descs), S()))
    _lib.check(lib.showo_attention_test(_lib.ptr(img), ld, n_seq, R, P, H, *args, L, _lib.masks_array(descs), S()))
    for i, d in enumerate(descs):
        assert (pre.view(n_seq, P, ld)[i, d[0]:, 2 * D:3 * D].float() - ref[i, d[0]:P]).abs().max().item() < 0.02
        assert (img.view(n_seq, R, ld)[i, :, 2 * D:3 * D].float() - ref[i, P:]).abs().max().item() < 0.02
    q1 = f3[:, L - 1:L].reshape(-1, ld).clone()
    _lib.check(lib.showo_attention_test(_lib.ptr(q1), ld, n_seq, 1, L - 1, H, *args, L, _lib.masks_array(descs), S()))
    assert (q1.view(n_seq, 1, ld)[:, 0, 2 * D:3 * D].float() - ref[:, L - 1]).abs().max().item() < 0.02


@pytest.mark.parametrize("NB,H,W,cin,cout,taps", [(2, 16, 16, 64, 512, 9), (1, 32, 32, 128, 128, 9), (2, 64, 64, 256, 128, 1),
                                                  (1, 16, 16, 512, 13, 9), (1, 256, 256, 128, 128, 9), (3, 24, 40, 64, 64, 9)])
def test_conv_implicit_gemm(lib, dev, NB, H, W, cin, cout, taps):
    k = 3 if taps == 9 else 1
    g = torch.Generator(device=dev).manual_seed(cin + cout)
    x = torch.randn(NB, H, W, cin, device=dev, generator=g).bfloat16()
    w = (torch.randn(cout, k, k, cin, device=dev, generator=g) / math.sqrt(cin * k * k)).bfloat16()
    b = torch.randn(cout, device=dev, generator=g)
    res = torch.randn(NB, H, W, cout, device=dev, generator=g).bfloat16()
    cout_pad = (cout + 63) // 64 * 64
    wp = torch.zeros(cout_pad, taps * cin, device=dev, dtype=torch.bfloat16)
    wp[:cout] = w.reshape(cout, taps * cin)
    out = torch.zeros(NB * H * W, cout, device=dev, dtype=torch.bfloat16)
    _lib.check(lib.showo_conv_test(_lib.ptr(x), _lib.ptr(wp), _lib.ptr(b), _lib.ptr(res), _lib.ptr(out), NB, H, W, cin, cout, taps, S()))
    ref = torch.nn.functional.conv2d(x.float().permute(0, 3, 1, 2), w.float().permute(0, 3, 1, 2), b, padding=k // 2)
    ref = ref + res.float().permute(0, 3, 1, 2)
    got = out.view(NB, H, W, cout).permute(0, 3, 1, 2).float()
    assert ((got - ref).abs() <= ref.abs() * 2 ** -7 + 1e-2).all()


# ------------------------------------------------------------------------------------------------ sampler
def _run_sampler(lib, dev, c, case, logits_cond, logits_unc, w):
    B, N = c["B"], c["N"]
    floors, temps = showo_b200.step_schedule(showo_b200.cosine_schedule, case["T"], N, 1.0)
    L = 129 + N + 2
    ids = torch.full((B, L), 7, dtype=torch.int64)
    ids[:, 130:130 + N] = torch.where(c["ids_minus"] == VOC.mask_token_id, c["ids_minus"], c["ids_minus"] + VOC.image_offset)
    ids_d, lc = ids.to(dev), logits_cond.contiguous().to(dev)
    lu = logits_unc.contiguous().to(dev) if logits_unc is not None else None
    ex, un = c["expo"].to(dev), c["unif"].to(dev)
    out = torch.zeros(B, N, dtype=torch.int64, device=dev)
    mk = torch.zeros(B, N, dtype=torch.uint8, device=dev)
    _lib.check(lib.showo_sampler_step(_lib.ptr(lc), _lib.ptr(lu), B, N, 8192, w, _lib.ptr(ids_d), L, 130, VOC.image_offset,
                                      VOC.mask_token_id, floors[case["step"]], temps[case["step"]], _lib.ptr(ex), _lib.ptr(un), 0,
                                      case["step"], _lib.ptr(out), _lib.ptr(mk), S()))
    torch.cuda.synchronize()
    return out.cpu(), mk.cpu().bool(), ids_d.cpu()


def test_sampler_bit_exact_against_golden_and_oracle(lib, dev):
    z = FX.load("sampler.npz")
    for ci, case in enumerate(FX.sampler_cases()):
        c = FX.sampler_case(case, VOC)
        w = case["w"]
        out, mk, ids = _run_sampler(lib, dev, c, case, c["cond"], c["unc"] if w > 0 else None, w)
        assert np.array_equal(out.numpy(), z[f"sampled_{ci}"]), ci                 # reference golden
        assert np.array_equal(mk.numpy(), z[f"masking_{ci}"]), ci
        samp, masking, _, _ = O.t2i_sample_step(c["logits"], c["ids_minus"], case["step"], case["T"], c["temp_in"],
                                                VOC.mask_token_id, c["N"], c["expo"], c["unif"])
        assert torch.equal(out, samp) and torch.equal(mk, masking)
        new_ids = torch.where(masking, VOC.mask_token_id, samp + VOC.image_offset)
        assert torch.equal(ids[:, 130:130 + c["N"]], new_ids) and (ids[:, :130] == 7).all() and (ids[:, 130 + c["N"]:] == 7).all()
        assert int(mk.sum(1).min()) == int(mk.sum(1).max()) or case["step"] > 0        # step 0: exactly mask_len masked


def test_sampler_philox_mode_properties(lib, dev):
    B, N = 4, 256
    g = torch.Generator(device=dev).manual_seed(0)
    logits = torch.randn(B, N, 8192, device=dev, generator=g)
    outs = []
    for seed in (1234, 1234, 99):
        ids = torch.full((B, 387), VOC.mask_token_id, dtype=torch.int64, device=dev)
        out = torch.zeros(B, N, dtype=torch.int64, device=dev)
        mk = torch.zeros(B, N, dtype=torch.uint8, device=dev)
        _lib.check(lib.showo_sampler_step(_lib.ptr(logits), None, B, N, 8192, 0.0, _lib.ptr(ids), 387, 130, VOC.image_offset,
                                          VOC.mask_token_id, 200, 0.9, None, None, seed, 0, _lib.ptr(out), _lib.ptr(mk), S()))
        assert int(out.min()) >= 0 and int(out.max()) < 8192 and mk.sum(1).tolist() == [200] * B
        assert (ids[:, 130:386] == VOC.mask_token_id).sum(1).tolist() == [200] * B
        outs.append(out.cpu())
    assert torch.equal(outs[0], outs[1]) and not torch.equal(outs[0], outs[2])
    # the draw follows the distribution: a strongly peaked row always returns its mode
    peaked = torch.zeros(1, 8, 8192, device=dev)
    peaked[0, torch.arange(8), torch.arange(8) * 1000] = 50.0
    ids = torch.full((1, 20), VOC.mask_token_id, dtype=torch.int64, device=dev)
    out = torch.zeros(1, 8, dtype=torch.int64, device=dev)
    _lib.check(lib.showo_sampler_step(_lib.ptr(peaked), None, 1, 8, 8192, 0.0, _lib.ptr(ids), 20, 5, VOC.image_offset,
                                      VOC.mask_token_id, 3, 0.5, None, None, 7, 0, _lib.ptr(out), None, S()))
    assert out.cpu()[0].tolist() == [i * 1000 for i in range(8)]


# ------------------------------------------------------------------------------------------------ backbone
def test_forward_tiny_against_oracle_and_golden(tiny, dev):
    dims, W, m = tiny
    z = FX.load("tiny_t2i.npz")
    cond, uncond, mask = FX.tiny_t2i_inputs(VOC)
    ids = torch.cat([cond, uncond])
    with torch.no_grad():
        ref = O.showo_logits(W, dims, input_ids=ids, add_mask=mask)
    got = m(ids.to(dev), attention_mask=mask.to(dev)).cpu()
    assert got.shape == ref.shape == (4, 387, 58498) and got.dtype == torch.float32
    descs = M.descriptors_from_dense(mask)
    for b in range(4):
        assert (got[b, descs[b][0]:] - ref[b, descs[b][0]:]).abs().max().item() < TOL_TINY
    sl = got[:, 130:386, VOC.image_offset:-1]
    assert np.abs(sl[:, ::16].numpy() - z["logits_slice"]).max() < TOL_TINY          # reference golden
    # decisions: argmax may differ only where the reference's top-2 margin is below 2x the measured error
    err = (sl - ref[:, 130:386, VOC.image_offset:-1]).abs().max().item()
    top2 = ref[:, 130:386, VOC.image_offset:-1].topk(2, -1).values
    flips = sl.argmax(-1) != torch.from_numpy(z["argmax"]).long()
    assert ((top2[..., 0] - top2[..., 1])[flips] <= 2 * err).all()


def test_prefix_reuse_equals_full_recompute(tiny, dev):
    dims, W, m = tiny
    cond, uncond, mask = FX.tiny_t2i_inputs(VOC)
    ids = torch.cat([cond, uncond]).to(dev)
    full = m(ids, attention_mask=mask.to(dev))[:, 130:386, VOC.image_offset:-1]
    step = m.t2i_step_logits(cond.to(dev), uncond.to(dev), mask.to(dev), guidance_scale=5.0, config=cfg_ns())
    one = m.t2i_step_logits(cond[:1].to(dev), None, mask[:1].to(dev), guidance_scale=0.0, config=cfg_ns())
    if os.environ.get("SHOWO_ATTN_TC") == "0":
        # mma.sync attention: every row is reduced in the same order whatever tile it lands in -> bitwise identical
        assert torch.equal(step, full)
        assert torch.equal(one[0], full[0])     # batch-size independence (B=1, no CFG branch)
    else:
        # tcgen05 attention (default): a row's 64-key blocks start at its tile's first visible key and the tile / tail split
        # depends on the row offset of the pass, so the two passes sum in different orders: equal to fp32-reordering accuracy
        d1, d2 = (step - full).abs().max().item(), (one[0] - full[0]).abs().max().item()
        print(f"prefix reuse vs full recompute: max|dlogit| {d1:.2e} (B=1: {d2:.2e})")
        _record("prefix_reuse_vs_full", {"max_abs_dlogit": d1, "max_abs_dlogit_b1": d2})
        assert d1 < 5e-3 and d2 < 5e-3


def test_forward_masks_lm_mmu_and_embeddings_input(tiny, dev):
    dims, W, m = tiny
    mm = FX.tiny_mmu_inputs(VOC)
    for mask in (O.create_attention_mask_for_mmu(mm), O.additive_from_allowed(torch.tril(torch.ones(3, mm.shape[1], mm.shape[1], dtype=torch.bool)))):
        with torch.no_grad():
            ref = O.showo_logits(W, dims, input_ids=mm, add_mask=mask)
        got = m(mm.to(dev), attention_mask=mask.to(dev)).cpu()
        assert (got - ref).abs().max().item() < TOL_TINY
    emb = W["showo.model.embed_tokens.weight"][mm]
    mask = O.additive_from_allowed(O.mask_allowed_mmu_vit(3, mm.shape[1], system_prompt_len=4, n_vis=100))
    with torch.no_grad():
        ref = O.showo_logits(W, dims, input_embeddings=emb, add_mask=mask)
    got = m(None, input_embeddings=emb.to(dev), attention_mask=mask.to(dev)).cpu()
    assert (got - ref).abs().max().item() < TOL_TINY


def test_mm_projector_on_engine(dev):
    """Showo.mm_projector (modeling_showo.py:49-54, inference_mmu.py:131) through the drop-in class: Linear(1024, 2048) -> exact GELU ->
    Linear(2048, 2048) on the engine vs torch fp32 on the same parameters; bf16 operands: |d| <= 1 % of the output scale."""
    torch.manual_seed(3)
    m = showo_b200.Showo(True, 58498, 50295, phi_dims=FX.TINY).to(dev)
    x = torch.randn(2, 576, 1024, device=dev)
    got = m.mm_projector(x)
    seq = torch.nn.Sequential(*list(m.mm_projector.children()))
    with torch.no_grad():
        ref = seq(x)
    assert got.shape == (2, 576, 2048) and got.dtype == torch.float32
    err, scale = (got - ref).abs().max().item(), ref.abs().max().item()
    print(f"mm_projector: max|d| {err:.4f} of scale {scale:.3f}")
    _record("mm_projector", {"max_abs": err, "ref_max": scale})
    assert err < 0.01 * scale
    # a tiny batch (M <= 16) takes the same tensor-core path, and a parameter update is picked up
    assert (m.mm_projector(x[:1, :3]) - ref[:1, :3]).abs().max().item() < 0.01 * scale
    with torch.no_grad():
        m.mm_projector[2].bias.add_(1.0)
    assert (m.mm_projector(x) - ref - 1.0).abs().max().item() < 0.01 * scale


def test_mmu_generate_from_input_embeddings(tiny, lib, dev):
    """the w_clip_vit branch of mmu_generate (modeling_showo.py:231-233, inference_mmu.py:100-151): the prompt arrives as embeddings
    under the mmu_vit window mask.  (a) embeddings produced by the engine's own embed_tokens give the SAME tokens as the ids branch,
    bit for bit; (b) the first generated token equals the oracle's argmax on the same embeddings unless the oracle's own top-2 margin
    is inside the logit tolerance; (c) the early stop at eot_token cuts the lengths."""
    dims, W, m = tiny
    mm = FX.tiny_mmu_inputs(VOC)
    B, L0 = mm.shape
    n_new = 6
    emb = torch.empty(B * L0, dims.hidden, device=dev)
    _lib.check(lib.showo_embed_tokens(m._engine, _lib.ptr(mm.to(dev).contiguous()), B * L0, _lib.ptr(emb), S()), "embed_tokens")
    emb = emb.view(B, L0, dims.hidden)
    descs = M.descriptors_mmu_vit(B, system_prompt_len=4, n_vis=100)
    t_ids, _ = m.mmu_generate_batched(mm.to(dev), attention_mask=descs, max_new_tokens=n_new, top_k=1)
    t_emb, l_emb = m.mmu_generate_batched(None, input_embeddings=emb, attention_mask=descs, max_new_tokens=n_new, top_k=1)
    assert torch.equal(t_ids, t_emb) and l_emb.tolist() == [n_new] * B
    mask = O.additive_from_allowed(O.mask_allowed_mmu_vit(B, L0, system_prompt_len=4, n_vis=100))
    with torch.no_grad():
        lg = O.showo_logits(W, dims, input_embeddings=emb.cpu(), add_mask=mask)[:, -1]
    top2 = lg.topk(2)
    for b in range(B):
        if int(t_emb[b, 0]) != int(top2.indices[b, 0]):
            assert float(top2.values[b, 0] - top2.values[b, 1]) < 2 * TOL_TINY and int(t_emb[b, 0]) == int(top2.indices[b, 1])
    # early stop: a token that row 0 produces at step 2 is declared eot -> lengths <= position of its first occurrence + 1, tokens unchanged
    eot = int(t_emb[0, 2])
    t2, l2 = m.mmu_generate_batched(None, input_embeddings=emb, attention_mask=descs, max_new_tokens=n_new, top_k=1, eot_token=eot)
    for b in range(B):
        hit = (t_emb[b] == eot).nonzero()
        want = int(hit[0]) + 1 if hit.numel() else n_new
        assert int(l2[b]) == want and torch.equal(t2[b, :want], t_emb[b, :want])


def test_t2i_generate_teacher_forced_parity(tiny, lib, dev):
    """Each denoise step is replayed from the ORACLE's input ids: logits within tolerance, the sampler on the oracle's
    logits is bit-exact, and on the engine's logits a token may differ only below the 2x-error decision margin."""
    dims, W, m = tiny
    B, T, w = 2, 5, 5.0
    cond, uncond = O.make_t2i_prompts(B, VOC, seed=11)
    mask = O.create_attention_mask_predict_next(torch.cat([cond, uncond]))
    trace = []
    with torch.no_grad():
        O.t2i_generate(W, dims, VOC, cond.clone(), uncond.clone(), mask, guidance_scale=w, timesteps=T,
                       generator=torch.Generator().manual_seed(21), trace=trace)
    floors, temps = showo_b200.step_schedule(showo_b200.cosine_schedule, T, 256, 1.0)
    md, ud = mask.to(dev), uncond.to(dev)
    for s, tr in enumerate(trace):
        ids_in = tr.input_ids_in.to(dev)
        sl = m.t2i_step_logits(ids_in, ud, md, guidance_scale=w, config=cfg_ns())
        lg = ((1 + w) * sl[:B] - w * sl[B:]).cpu()
        err = (lg - tr.logits).abs().max().item()
        assert err < (1 + 2 * w) * TOL_TINY, (s, err)
        ex, un = tr.expo.to(dev), tr.uniform.to(dev)
        for lc, lu, ww, exact in ((tr.logits.contiguous().to(dev), None, 0.0, True), (sl[:B].contiguous(), sl[B:].contiguous(), w, False)):
            ids_d = ids_in.clone()
            out = torch.zeros(B, 256, dtype=torch.int64, device=dev)
            mk = torch.zeros(B, 256, dtype=torch.uint8, device=dev)
            _lib.check(lib.showo_sampler_step(_lib.ptr(lc), _lib.ptr(lu), B, 256, 8192, ww, _lib.ptr(ids_d), 387, 130, VOC.image_offset,
                                              VOC.mask_token_id, floors[s], temps[s], _lib.ptr(ex), _lib.ptr(un), 0, s, _lib.ptr(out),
                                              _lib.ptr(mk), S()))
            if exact:
                assert torch.equal(out.cpu(), tr.sampled_ids) and torch.equal(mk.cpu().bool(), tr.masking), s
            else:
                race = (tr.logits.reshape(-1, 8192) - torch.log(tr.expo)).topk(2, -1).values
                margin = (race[:, 0] - race[:, 1]).view(B, 256)
                diff = out.cpu() != tr.sampled_ids
                assert (margin[diff] <= 2 * err).all(), (s, margin[diff], err)
                assert diff.float().mean().item() < 0.05


def test_t2i_generate_loop_equals_its_own_steps(tiny, lib, dev):
    """showo_t2i_generate == prefix + T x (step logits -> sampler) composed by hand with the same noise."""
    dims, W, m = tiny
    B, T, w = 2, 4, 3.0
    cond, uncond = O.make_t2i_prompts(B, VOC, seed=31)
    mask = O.create_attention_mask_predict_next(torch.cat([cond, uncond])).to(dev)
    ids_a = cond.clone().to(dev)
    out_a = m.t2i_generate(ids_a, uncond.to(dev), mask, guidance_scale=w, timesteps=T, generator=torch.Generator(device=dev).manual_seed(5),
                           config=cfg_ns())
    g = torch.Generator(device=dev).manual_seed(5)
    expo = torch.empty(T, B * 256, 8192, device=dev)
    unif = torch.empty(T, B, 256, device=dev)
    for s in range(T):
        expo[s].exponential_(1, generator=g)
        unif[s].uniform_(0, 1, generator=g)
    floors, temps = showo_b200.step_schedule(showo_b200.cosine_schedule, T, 256, 1.0)
    ids_b = cond.clone().to(dev)
    out_b = torch.zeros(B, 256, dtype=torch.int64, device=dev)
    for s in range(T):
        sl = m.t2i_step_logits(ids_b, uncond.to(dev), mask, guidance_scale=w, config=cfg_ns())
        lc, lu = sl[:B].contiguous(), sl[B:].contiguous()
        _lib.check(lib.showo_sampler_step(_lib.ptr(lc), _lib.ptr(lu), B, 256, 8192, w, _lib.ptr(ids_b), 387, 130, VOC.image_offset,
                                          VOC.mask_token_id, floors[s], temps[s], _lib.ptr(expo[s]), _lib.ptr(unif[s]), 0, s,
                                          _lib.ptr(out_b), None, S()))
    assert torch.equal(out_a, out_b) and torch.equal(ids_a, ids_b)
    # quirk kept from the reference: the last step still re-masks mask_len = max(1, .) = 1 token in input_ids, while the
    # returned sampled_ids are complete (modeling_showo.py:166-181)
    assert ((ids_a[:, 130:386] == VOC.mask_token_id).sum(1) <= 1).all()
    assert int(out_a.min()) >= 0 and int(out_a.max()) < 8192


def test_t2i_generate_variants(tiny, dev):
    dims, W, m = tiny
    cond, uncond = O.make_t2i_prompts(3, VOC, seed=41)
    mask = O.create_attention_mask_predict_next(torch.cat([cond, uncond])).to(dev)
    # no CFG (guidance 0): single branch, B descriptors
    out = m.t2i_generate(cond.clone().to(dev), None, mask[:3], guidance_scale=0, timesteps=3, config=cfg_ns())
    assert out.shape == (3, 256) and int(out.max()) < 8192
    # single step, philox noise, reproducible through torch's seed
    torch.manual_seed(7)
    a = m.t2i_generate(cond.clone().to(dev), uncond.to(dev), mask, guidance_scale=2.0, timesteps=1, config=cfg_ns())
    torch.manual_seed(7)
    b = m.t2i_generate(cond.clone().to(dev), uncond.to(dev), mask, guidance_scale=2.0, timesteps=1, config=cfg_ns())
    assert torch.equal(a, b)
    # inpainting-style: known tokens are kept (modeling_showo.py:153-154)
    c2 = cond.clone()
    known = torch.arange(256) % 3 == 0
    c2[:, 130:386][:, known] = torch.arange(int(known.sum())) + VOC.image_offset
    out = m.t2i_generate(c2.clone().to(dev), uncond.to(dev), mask, guidance_scale=2.0, timesteps=4, config=cfg_ns()).cpu()
    assert torch.equal(out[:, known], (torch.arange(int(known.sum())))[None].expand(3, -1))


def test_t2i_512_geometry_tiny_model(dev):
    """N = 1024 image tokens, L = 1155 (showo_demo_512x512.yaml geometry) on the 2-layer test model."""
    dims = O.PhiDims(**FX.TINY)
    W = O.make_showo_weights(dims, seed=3)
    m = showo_b200.Showo(False, dims.vocab_size, VOC.llm_vocab_size, phi_dims=FX.TINY, materialize=False, num_vq_tokens=1024)
    m.load_weights(W, device=dev)
    voc = O.ShowoVocab(num_vq_tokens=1024)
    cond, uncond = O.make_t2i_prompts(1, voc, seed=51)
    mask = O.create_attention_mask_predict_next(torch.cat([cond, uncond]))
    with torch.no_grad():
        ref = O.showo_logits(W, dims, input_ids=torch.cat([cond, uncond]), add_mask=mask)[:, 130:1154, voc.image_offset:-1]
    got = m.t2i_step_logits(cond.to(dev), uncond.to(dev), mask.to(dev), guidance_scale=5.0, config=cfg_ns(1024)).cpu()
    assert (got - ref).abs().max().item() < TOL_TINY
    out = m.t2i_generate(cond.to(dev), uncond.to(dev), mask.to(dev), guidance_scale=5.0, timesteps=2, config=cfg_ns(1024))
    assert out.shape == (1, 1024)


def test_mmu_generate_batched_equals_rowwise_reference(tiny, dev):
    """Row b of the batched KV-cached decode == the oracle's B=1 greedy decode of row b, up to the first step where the
    oracle's own top-2 margin is inside the logit tolerance (after which the sequences legitimately differ)."""
    dims, W, m = tiny
    z = FX.load("tiny_t2i.npz")
    mm = FX.tiny_mmu_inputs(VOC)
    n_new = 8
    toks, lens = m.mmu_generate_batched(mm.to(dev), attention_mask=O.create_attention_mask_for_mmu(mm).to(dev),
                                        max_new_tokens=n_new, top_k=1)
    toks = toks.cpu()
    assert lens.tolist() == [n_new] * 3
    agree_rows = 0
    for b in range(3):
        ref = torch.from_numpy(z["mmu_tokens"][b]).long()                 # reference golden, B=1 calls
        if torch.equal(toks[b], ref):
            agree_rows += 1
            continue
        t = int((toks[b] != ref).nonzero()[0])
        seq = torch.cat([mm[b:b + 1], ref[None, :t]], 1)
        mk = O.additive_from_allowed(M.predicate(seq.shape[1], (0, 0, 0, 0, 259))[None])
        with torch.no_grad():
            lg = O.showo_logits(W, dims, input_ids=seq, add_mask=mk)[0, -1]
        top2 = lg.topk(2).values
        assert float(top2[0] - top2[1]) < 2 * TOL_TINY, (b, t, float(top2[0] - top2[1]))
        assert int(toks[b, t]) in lg.topk(2).indices.tolist()
    assert agree_rows >= 2
    # eot handling + the reference-shaped list API (B = 1)
    eot = int(toks[1, 3])
    first = int((toks[1] == eot).nonzero()[0])
    lst = m.mmu_generate(mm[1:2].to(dev), attention_mask=O.create_attention_mask_for_mmu(mm[1:2]).to(dev), max_new_tokens=n_new,
                         top_k=1, eot_token=eot)
    assert len(lst) == first + 1 and int(lst[-1]) == eot and all(t.dim() == 0 and t.dtype == torch.int64 for t in lst)
    # sampled decode (top_k=None / k>1, modeling_showo.py:219-228), noise drawn by torch in the reference's order: every
    # drawn token must be what the oracle's draw gives on the engine's own teacher-forced logits with the same noise
    for top_k, temp in ((None, 0.8), (5, 1.3)):
        gen = torch.Generator(device=dev).manual_seed(11)
        toks_s, _ = m.mmu_generate_batched(mm.to(dev), attention_mask=O.create_attention_mask_for_mmu(mm).to(dev),
                                           max_new_tokens=4, temperature=temp, top_k=top_k, generator=gen)
        gen = torch.Generator(device=dev).manual_seed(11)
        V = dims.vocab_size
        expo = torch.empty(4, 3, V, device=dev)
        for t in range(4):
            expo[t].exponential_(1, generator=gen)
        ok = 0
        for t in range(4):
            seq = torch.cat([mm.to(dev), toks_s[:, :t]], 1)
            desc = [(0, 0, 0, 0, 259)] * 3
            lg = m(seq, attention_mask=desc)[:, -1] / temp                      # prefill-path logits (bf16-level noise)
            if top_k is not None:
                v, _ = torch.topk(lg, top_k)
                assert (lg.gather(1, toks_s[:, t:t + 1]) >= v[:, [-1]] - 2 * TOL_TINY / temp).all()
                lg = lg.masked_fill(lg < v[:, [-1]], -float("inf"))
            pick = O.categorical_from_exponential(torch.softmax(lg, -1), expo[t])
            ok += int((pick == toks_s[:, t]).sum())
        assert ok >= 10, ok                                                     # 12 draws; near-ties may flip a few
    # no generator: the library's own Philox stream, reproducible under torch.manual_seed
    torch.manual_seed(3)
    a1, _ = m.mmu_generate_batched(mm.to(dev), attention_mask=O.create_attention_mask_for_mmu(mm).to(dev), max_new_tokens=4, top_k=None)
    torch.manual_seed(3)
    a2, _ = m.mmu_generate_batched(mm.to(dev), attention_mask=O.create_attention_mask_for_mmu(mm).to(dev), max_new_tokens=4, top_k=None)
    assert torch.equal(a1, a2) and int(a1.min()) >= 0 and int(a1.max()) < dims.vocab_size


def test_cross_entropy_terms_against_torch(lib, dev):
    """showo_cross_entropy == F.cross_entropy(ignore_index=-100) on the reference's three slices (modeling_showo.py:81-100),
    including an empty slice (NaN) and a slice whose rows are all ignored."""
    import torch.nn.functional as F
    B, L, V, P = 4, 37, 58498, 9
    g = torch.Generator(device=dev).manual_seed(3)
    logits = torch.randn(B, L, V, device=dev, generator=g) * 2.0
    labels = torch.randint(0, V, (B, L), device=dev, generator=g)
    labels[torch.rand(B, L, device=dev, generator=g) < 0.3] = -100
    labels[3] = -100
    out = torch.zeros(2, device=dev)

    def ce(b0, nb, t0, nt, shift):
        _lib.check(lib.showo_cross_entropy(_lib.ptr(logits), _lib.ptr(labels), L, V, b0, nb, t0, nt, shift, -100, _lib.ptr(out), S()))
        return out.clone().cpu()

    got = ce(0, 2, P, L - P, 0)
    ref = F.cross_entropy(logits[:2, P:].reshape(-1, V), labels[:2, P:].reshape(-1), ignore_index=-100)
    assert abs(got[0].item() - ref.item()) < 2e-5 and int(got[1]) == int((labels[:2, P:] != -100).sum())
    got = ce(2, 1, 0, L - 1, 1)
    ref = F.cross_entropy(logits[2:3, :-1].reshape(-1, V), labels[2:3, 1:].reshape(-1), ignore_index=-100)
    assert abs(got[0].item() - ref.item()) < 2e-5
    assert torch.isnan(ce(2, 0, 0, L - 1, 1)[0])                      # empty slice: mean over nothing
    assert torch.isnan(ce(3, 1, 0, L - 1, 1)[0])                      # every row ignored: 0 / 0
    a, b2 = ce(0, B, 0, L - 1, 1), ce(0, B, 0, L - 1, 1)
    assert torch.equal(a, b2)                                         # fixed-order reduction


def test_forward_with_labels_losses_against_reference_golden(tiny, dev):
    """Showo.forward(labels=...) on the mixed t2i / lm / mmu training batch (modeling_showo.py:81-100): logits from the CUDA
    engine (three different mask kinds in one batch), the three cross-entropies against the reference's values."""
    dims, W, m = tiny
    z = FX.load("train_step.npz")
    ids, mask, labels, (bt, bl, bm) = FX.train_batch(VOC)
    logits, l1, l2, l3 = m(ids.to(dev), attention_mask=mask.to(dev), labels=labels.to(dev), batch_size_t2i=bt, batch_size_lm=bl,
                           batch_size_mmu=bm, max_seq_length=128)
    assert logits.shape == (5, 387, dims.vocab_size) and logits.dtype == torch.float32
    assert np.abs(logits[:, ::32, ::997].cpu().numpy() - z["logits_slice"]).max() < TOL_TINY
    got = np.array([l1.item(), l2.item(), l3.item()])
    assert np.abs(got - z["losses"]).max() < TOL_TINY, (got, z["losses"])


def test_decode_megakernel_equals_per_kernel_path(tiny, dev, monkeypatch):
    """The persistent decode kernel (SHOWO_DECODE_MEGA=1: all layers of a step in one launch, weights and KV chunks through
    one TMA ring, grid barriers between phases) produces the same tokens as the per-kernel decode path."""
    dims, W, m = tiny
    mm = FX.tiny_mmu_inputs(VOC)
    mk = O.create_attention_mask_for_mmu(mm).to(dev)
    monkeypatch.setenv("SHOWO_DECODE_MEGA", "0")
    ref, _ = m.mmu_generate_batched(mm.to(dev), attention_mask=mk, max_new_tokens=12, top_k=1)
    n0 = m.kernel_launches()
    monkeypatch.setenv("SHOWO_DECODE_MEGA", "1")
    got, _ = m.mmu_generate_batched(mm.to(dev), attention_mask=mk, max_new_tokens=12, top_k=1)
    assert m.kernel_launches() < n0                      # one launch per step instead of four per layer
    assert torch.equal(ref, got)


@pytest.mark.parametrize("V,top_k,temp", [(58498, 0, 1.0), (58498, 1, 0.7), (58498, 5, 0.7), (58498, 200, 1.5), (1000, 1000, 1.0),
                                          (1000, 4000, 2.0), (777, 13, 0.3)])
def test_mmu_next_token_draw_bit_exact(lib, dev, V, top_k, temp):
    """showo_mmu_sample == the reference's temperature / top-k / softmax / multinomial (modeling_showo.py:219-228) on
    the same logits and the same Exp(1) noise (torch.multinomial(p,1) == argmax(p/q)); ties in the k-th value are kept."""
    B = 16
    g = torch.Generator(device=dev).manual_seed(V + top_k)
    logits = torch.randn(B, V, device=dev, generator=g) * 3.0
    logits[:, 5] = logits[:, 9]                                # exact ties
    if 1 < top_k < V:
        kth = logits.topk(top_k).values[:, -1]
        logits[:, 17] = kth                                    # a duplicate of the k-th largest value stays in
    expo = torch.empty(B, V, device=dev).exponential_(1, generator=g)
    out = torch.full((B,), -1, dtype=torch.int64, device=dev)
    _lib.check(lib.showo_mmu_sample(_lib.ptr(logits), V, B, V, temp, top_k, _lib.ptr(expo), 0, 0, _lib.ptr(out), S()))
    lg = logits.cpu() / temp
    if top_k > 0:
        v, _ = torch.topk(lg, min(top_k, V))
        lg[lg < v[:, [-1]]] = -float("inf")
    ref = O.categorical_from_exponential(torch.softmax(lg, -1), expo.cpu())
    assert torch.equal(out.cpu(), ref)
    # Philox mode: in range, deterministic in (seed, step), different across steps
    o1, o2, o3 = (torch.empty(B, dtype=torch.int64, device=dev) for _ in range(3))
    _lib.check(lib.showo_mmu_sample(_lib.ptr(logits), V, B, V, temp, top_k, None, 77, 0, _lib.ptr(o1), S()))
    _lib.check(lib.showo_mmu_sample(_lib.ptr(logits), V, B, V, temp, top_k, None, 77, 0, _lib.ptr(o2), S()))
    _lib.check(lib.showo_mmu_sample(_lib.ptr(logits), V, B, V, temp, top_k, None, 77, 1, _lib.ptr(o3), S()))
    assert torch.equal(o1, o2) and int(o1.min()) >= 0 and int(o1.max()) < V
    if top_k != 1:
        assert not torch.equal(o1, o3)
    if 0 < top_k < V:
        kept = lg.gather(1, o1.cpu()[:, None])
        assert torch.isfinite(kept).all()


# ------------------------------------------------------------------------------------------------ MAGVIT-v2
@pytest.fixture(scope="module")
def vq(dev):
    v = showo_b200.MAGVITv2(materialize=False)
    v.load_weights(MO.make_magvit_weights(1), device=dev)
    return v


def test_magvit_decode_against_golden_and_oracle(vq, dev):
    z = FX.load("magvit.npz")
    codes_in, _ = FX.magvit_inputs()
    got = vq.decode_code(codes_in.to(dev)).cpu()
    ref = torch.from_numpy(z["decode"].astype(np.float32))
    d = (got - ref).abs()
    print(f"magvit decode: max {d.max():.4f} mean {d.mean():.5f} (ref std {ref.std():.3f})")
    _record("magvit_decode", {"max_abs": float(d.max()), "mean_abs": float(d.mean()), "ref_std": float(ref.std())})
    assert got.shape == (1, 3, 256, 256) and d.max().item() < 0.2 and d.mean().item() < 0.012
    u8 = vq.decode_code_uint8(codes_in.to(dev)).cpu()
    ref_u8 = torch.from_numpy((torch.clamp((ref + 1) / 2, 0, 1) * 255).permute(0, 2, 3, 1).numpy().astype("uint8"))
    d8 = (u8.int() - ref_u8.int()).abs()
    _record("magvit_decode_u8", {"max_levels": int(d8.max()), "mean_levels": float(d8.float().mean())})
    assert u8.shape == (1, 256, 256, 3) and d8.float().mean().item() < 1.5 and int(d8.max()) <= 24
    # uint8 path == clamp/scale of the fp32 path of the same engine
    own = (torch.clamp((got + 1) / 2, 0, 1) * 255).permute(0, 2, 3, 1).numpy().astype("uint8")
    assert np.array_equal(u8.numpy(), own)
    # batch independence + non-square grid (extrapolation mode, inference_t2i.py:276)
    g = torch.Generator().manual_seed(2)
    ids3 = torch.cat([codes_in, torch.randint(0, 8192, (2, 256), generator=g)])
    assert torch.equal(vq.decode_code(ids3.to(dev))[:1].cpu(), got)
    wide = torch.randint(0, 8192, (1, 16 * 32), generator=g)
    with torch.no_grad():
        refw = MO.decode_code(wide, MO.make_magvit_weights(1), shape=(16, 32))
    gotw = vq.decode_code(wide.to(dev), shape=(16, 32)).cpu()
    assert gotw.shape == (1, 3, 256, 512) and (gotw - refw).abs().mean().item() < 0.012


def test_magvit_get_code_against_golden(vq, dev):
    z = FX.load("magvit.npz")
    _, pixels = FX.magvit_inputs()
    codes = vq.get_code(pixels.to(dev)).cpu()
    assert codes.shape == (1, 256) and codes.dtype == torch.int64
    bits_ref = torch.from_numpy(z["z"] > 0).reshape(1, 13, -1)
    bits_got = ((codes[:, None, :] >> torch.arange(12, -1, -1)[None, :, None]) & 1).bool()
    mism = bits_ref != bits_got
    zabs = torch.from_numpy(np.abs(z["z"])).reshape(1, 13, -1)
    print(f"get_code: {int(mism.sum())}/{mism.numel()} sign bits differ, max|z| there {float(zabs[mism].max()) if mism.any() else 0:.4f}")
    codes_ref = torch.from_numpy(z["codes"].astype(np.int64)).reshape(1, -1)
    _record("magvit_get_code", {"sign_bits_differing": int(mism.sum()), "sign_bits": int(mism.numel()),
                                "max_abs_z_at_differing_bit": float(zabs[mism].max()) if mism.any() else 0.0,
                                "codes_differing": int((codes != codes_ref).sum()), "codes": int(codes.numel()),
                                "bits_with_abs_z_below_0p03": int((zabs < 0.03).sum())})
    # observed on B200 (profiles/r2_parity_observed.json): 19 of 3328 bits (0.57 %), largest |z| at a differing bit 0.0122 -- the
    # bounds are 2x that; 360 bits of the fixture have |z| < 0.03, so 'below the margin' does not mean 'free to differ'
    assert (zabs[mism] < 0.025).all() and mism.float().mean().item() < 0.012     # only bits whose pre-sign value is ~0
    # encode -> decode -> encode is stable for codes away from the sign boundary (round trip through the engine)
    rec = vq.decode_code(codes.to(dev))
    assert rec.shape == (1, 3, 256, 256) and torch.isfinite(rec).all()


# ------------------------------------------------------------------------------------------------ dense mask -> descriptors
def test_mask_descriptor_kernel_equals_host_derivation(dev):
    """showo_mask_descriptors (one kernel, derive + verify) == the torch derivation of masks.descriptors_from_dense on the CPU
    for every mask kind of the reference (t2i with long / short / no padding, lm, mmu, mmu_vit), additive fp32 and bool;
    a tensor that is not an omni mask is rejected."""
    rows = FX.mask_rows(VOC)
    dense = [O.create_attention_mask_predict_next(rows["t2i"]), O.create_attention_mask_for_mmu(rows["mmu"]),
             O.additive_from_allowed(O.mask_allowed_mmu_vit(2, 700, system_prompt_len=28))]
    for m in dense:
        want = M.descriptors_from_dense(m)                          # CPU tensors: torch path
        assert M.descriptors_from_dense(m.to(dev)) == want          # CUDA tensors: the kernel
        assert M.descriptors_from_dense((m == 0).to(dev)) == want   # bool masks
        assert M.descriptors_from_dense(m.to(dev).half()) == want   # other float dtypes are widened first
    bad = dense[0].clone()
    bad[1, 0, 300, 200] = bad[1, 0, 300, 200] - 1.0 if bad[1, 0, 300, 200] == 0 else 0.0
    with pytest.raises(NotImplementedError):
        M.descriptors_from_dense(bad.to(dev))
    # strided view of a larger batch (the shim slices [:n_seq])
    big = torch.cat([dense[0], dense[0]]).to(dev)
    assert M.descriptors_from_dense(big[:3]) == M.descriptors_from_dense(dense[0])[:3]


def test_magvit_fp32_verification_path(vq, dev):
    """The engine's fp32 verification path (SURVEY section 7; fp32 NCHW activations and weights, CUDA cores only) against the reference
    golden / the oracle at fp32 re-association level, and the FAST path against it: the bf16 fast path's LFQ sign flips sit only where
    the verification path's own pre-sign value is ~0, i.e. they are rounding, not defects."""
    g = FX.load("magvit.npz")
    codes_in, pixels = FX.magvit_inputs()
    # ---- decode
    with torch.no_grad():
        ref = MO.decode_code(codes_in, MO.make_magvit_weights(1))
    got32 = vq.decode_code_fp32(codes_in.to(dev)).cpu()
    d32 = (got32 - ref).abs()
    fast = vq.decode_code(codes_in.to(dev)).cpu()
    dfast = (fast - got32).abs()
    print(f"magvit decode, fp32 verification path vs oracle: max {d32.max():.2e} mean {d32.mean():.2e}; fast path vs verification path: "
          f"max {dfast.max():.4f} mean {dfast.mean():.5f}")
    _record("magvit_decode_fp32_path", {"max_abs_vs_oracle": float(d32.max()), "mean_abs_vs_oracle": float(d32.mean()),
                                        "fast_vs_fp32_max": float(dfast.max()), "fast_vs_fp32_mean": float(dfast.mean())})
    assert got32.shape == (1, 3, 256, 256) and d32.max().item() < 2e-4          # observed 2.9e-5
    assert (got32 - torch.from_numpy(g["decode"].astype(np.float32))).abs().max().item() < 2e-3        # the reference's own output (stored in half precision)
    assert dfast.max().item() < 0.2 and dfast.mean().item() < 0.012
    # non-square grid
    wide = torch.randint(0, 8192, (1, 8 * 24), generator=torch.Generator().manual_seed(3))
    with torch.no_grad():
        refw = MO.decode_code(wide, MO.make_magvit_weights(1), shape=(8, 24))
    assert (vq.decode_code_fp32(wide.to(dev), shape=(8, 24)).cpu() - refw).abs().max().item() < 5e-4
    # ---- get_code
    codes32, z32 = vq.get_code_fp32(pixels.to(dev), return_z=True)
    codes32, z32 = codes32.cpu(), z32.cpu()
    z_ref = torch.from_numpy(g["z"].astype(np.float32))
    codes_ref = torch.from_numpy(g["codes"].astype(np.int64)).reshape(1, -1)
    dz = (z32 - z_ref).abs()
    print(f"magvit get_code, fp32 verification path: max |dz| vs the reference {dz.max():.2e}; codes differing {(codes32 != codes_ref).sum().item()} of 256; "
          f"smallest |z| of the fixture {z_ref.abs().min():.2e}")
    assert dz.max().item() < 5e-5          # observed 5.7e-6
    bits_ref = z_ref.reshape(1, 13, -1) > 0
    bits32 = ((codes32[:, None, :] >> torch.arange(12, -1, -1)[None, :, None]) & 1).bool()
    assert ((bits32 != bits_ref) <= (z_ref.reshape(1, 13, -1).abs() < 2 * dz.max())).all()            # identical unless |z| is inside the fp32 noise
    codes_fast = vq.get_code(pixels.to(dev)).cpu()
    bits_fast = ((codes_fast[:, None, :] >> torch.arange(12, -1, -1)[None, :, None]) & 1).bool()
    flip = bits_fast != bits32
    zabs = z32.reshape(1, 13, -1).abs()
    print(f"fast path vs verification path: {int(flip.sum())} of {flip.numel()} sign bits differ, largest |z| (fp32 path) at a differing bit "
          f"{float(zabs[flip].max()) if flip.any() else 0:.4f}")
    _record("magvit_get_code_fp32_path", {"max_abs_dz_vs_reference": float(dz.max()), "codes_differing_vs_reference": int((codes32 != codes_ref).sum()),
                                          "fast_path_bits_differing": int(flip.sum()), "max_abs_z_at_fast_path_flip": float(zabs[flip].max()) if flip.any() else 0.0})
    assert (zabs[flip] < 0.025).all()


def test_backbone_fp32_verification_forward(lib, dev):
    """showo_forward_fp32 (SURVEY section 7's verification mode: fp32 activations + fp32 master weights on CUDA cores, the reference's
    six separate Linear layers per block) pins the engine to the oracle at fp32 re-association level on every mask kind -- and with
    logits that close the TOKEN DECISIONS are bit-identical: a whole t2i_generate run replayed step by step from the verification
    logits (the engine's sampler kernel, the oracle's noise) reproduces the oracle's ids exactly.  The fast bf16 path is then measured
    against it: this is the 'logit error' the tolerances of this file are multiples of."""
    dims = O.PhiDims(**FX.TINY)
    W = O.make_showo_weights(dims, seed=3)
    m = showo_b200.Showo(False, dims.vocab_size, VOC.llm_vocab_size, phi_dims=FX.TINY, materialize=False)
    m.enable_optimizer(device=dev)
    m.load_weights(W, device=dev)
    rows = FX.mask_rows(VOC)
    worst = {}
    for kind, ids, dense in (("t2i", rows["t2i"], O.create_attention_mask_predict_next(rows["t2i"])),
                             ("mmu", rows["mmu"], O.create_attention_mask_for_mmu(rows["mmu"]))):
        with torch.no_grad():
            ref = O.showo_logits(W, dims, input_ids=ids, add_mask=dense)
        descs = M.descriptors_from_dense(dense)
        got = m.forward_fp32(ids.to(dev), attention_mask=descs).cpu()
        fast = m(ids.to(dev), attention_mask=descs).cpu()
        nonpad = torch.stack([torch.arange(ids.shape[1]) >= d[0] for d in descs])          # pad rows are never read by anyone (SURVEY 8a-5)
        e32 = (got - ref).abs()[nonpad].max().item()
        ebf = (fast - got).abs()[nonpad].max().item()
        worst[kind] = (e32, ebf)
        print(f"{kind}: verification path vs oracle max |dlogit| {e32:.2e}; fast bf16 path vs verification path {ebf:.4f}")
        assert e32 < 5e-5 and ebf < TOL_TINY          # observed 2e-6 / 0.0094
        assert torch.equal(got[nonpad].argmax(-1), ref[nonpad].argmax(-1))
    _record("backbone_fp32_path", {k: {"fp32_vs_oracle": v[0], "bf16_vs_fp32": v[1]} for k, v in worst.items()})
    # ---- a whole generation, decisions bit-identical
    B, T, w = 2, 4, 3.0
    cond, uncond = O.make_t2i_prompts(B, VOC, seed=61)
    mask = O.create_attention_mask_predict_next(torch.cat([cond, uncond]))
    descs = M.descriptors_from_dense(mask)
    trace = []
    with torch.no_grad():
        ref_ids = O.t2i_generate(W, dims, VOC, cond.clone(), uncond.clone(), mask, guidance_scale=w, timesteps=T,
                                 generator=torch.Generator().manual_seed(33), trace=trace)
    floors, temps = showo_b200.step_schedule(showo_b200.cosine_schedule, T, 256, 1.0)
    unc_d = uncond.to(dev)
    out = torch.zeros(B, 256, dtype=torch.int64, device=dev)
    off = VOC.image_offset
    n_diff, on_trajectory = 0, True
    ids_run = cond.clone().to(dev)
    for s, tr in enumerate(trace):
        if not torch.equal(ids_run.cpu(), tr.input_ids_in):               # a decision inside the fp32 noise moved the run: continue teacher-forced
            on_trajectory = False
            ids_run = tr.input_ids_in.clone().to(dev)
        unc_step = torch.cat([unc_d[:, :129], ids_run[:, 129:]], dim=1)
        full = m.forward_fp32(torch.cat([ids_run, unc_step]), attention_mask=descs)
        lc = full[:B, 130:386, off:off + 8192].contiguous()
        lu = full[B:, 130:386, off:off + 8192].contiguous()
        err = (((1 + w) * lc - w * lu).cpu() - tr.logits).abs().max().item()
        assert err < 5e-5 * (1 + 2 * w), (s, err)
        ex, un = tr.expo.to(dev), tr.uniform.to(dev)
        mk = torch.zeros(B, 256, dtype=torch.uint8, device=dev)
        _lib.check(lib.showo_sampler_step(_lib.ptr(lc), _lib.ptr(lu), B, 256, 8192, w, _lib.ptr(ids_run), 387, 130, off, VOC.mask_token_id,
                                          floors[s], temps[s], _lib.ptr(ex), _lib.ptr(un), 0, s, _lib.ptr(out), _lib.ptr(mk), S()))
        diff = out.cpu() != tr.sampled_ids
        if diff.any():                                                    # only where the oracle's own race was inside the fp32 noise
            race = (tr.logits.reshape(-1, 8192) - torch.log(tr.expo)).topk(2, -1).values
            margin = (race[:, 0] - race[:, 1]).view(B, 256)
            assert (margin[diff] <= 4 * err).all(), (s, margin[diff], err)
        n_diff += int(diff.sum()) + int((mk.cpu().bool() != tr.masking).sum())
    _record("backbone_fp32_path_generation", {"decisions_differing": n_diff, "tokens_decided": B * 256 * T, "stayed_on_the_oracle_trajectory": on_trajectory,
                                              "last_step_max_abs_dlogit": err})
    assert n_diff <= 2
    if n_diff == 0:
        assert on_trajectory and torch.equal(out.cpu(), ref_ids)
    print(f"t2i_generate replayed from verification logits: {n_diff} of {B * 256 * T} decisions differ from the oracle over {T} steps "
          f"(on the oracle's trajectory throughout: {on_trajectory}; last step max |dlogit| {err:.2e})")


def test_philox_noise_is_keyed_by_the_global_row(tiny, dev):
    """SURVEY 8e: with the library's own noise (no generator) a row's image must not depend on how the batch is split over GPUs.  The Philox
    counters are keyed by (seed, GLOBAL row, token, step): four rows generated in one call == the same rows generated as two 'ranks' of two
    rows with their row offsets and the same seed, bit for bit; without the offset the second half differs (the noise really is per row)."""
    dims, W, m = tiny
    cond, uncond = O.make_t2i_prompts(4, VOC, seed=71)
    kw = dict(guidance_scale=2.0, timesteps=3, config=cfg_ns())

    def run(rows, offset):
        c, u = cond[rows].clone().to(dev), uncond[rows].to(dev)
        mask = O.create_attention_mask_predict_next(torch.cat([cond[rows], uncond[rows]])).to(dev)
        torch.manual_seed(123)                        # the kernel's seed is drawn from torch's global generator
        return m.t2i_generate(c, u, mask, rng_row_offset=offset, **kw).cpu()
    whole = run(slice(0, 4), 0)
    a, b = run(slice(0, 2), 0), run(slice(2, 4), 2)
    assert torch.equal(torch.cat([a, b]), whole)
    assert not torch.equal(run(slice(2, 4), 0), whole[2:])
    # sampled MMU decode: the same keying per sequence (recorded, not asserted: the decode GEMMs' bitwise batch invariance is not a stated contract)
    mm = FX.tiny_mmu_inputs(VOC)
    descs = M.descriptors_mmu(mm, O.EOI)

    def dec(lo, hi, offset):
        torch.manual_seed(77)
        t, _ = m.mmu_generate_batched(mm[lo:hi].to(dev), attention_mask=descs[lo:hi], max_new_tokens=4, temperature=1.0, top_k=None,
                                      rng_row_offset=offset)
        return t.cpu()
    whole_t, part_t = dec(0, 3, 0), dec(1, 3, 1)
    same = bool(torch.equal(part_t, whole_t[1:]))
    print(f"sampled MMU decode, rows 1..2 generated alone with row offset 1 == their rows of the 3-row call: {same}")
    _record("philox_global_row_keying", {"t2i_split_equals_whole": True, "mmu_sampled_split_equals_whole": same})
