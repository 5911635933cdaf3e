"""GPU parity tests of the training step (run with -m gpu): showo_train_forward / showo_backward / showo_read_grad and
the attention backward kernel, through the C ABI, against (a) the reference's own losses and gradients committed in
tests/golden/train_step.npz and (b) the oracle's forward differentiated by torch autograd (CPU, fp32) for every parameter.

Tolerances: the engine multiplies in bf16 with fp32 accumulation and keeps bf16 activations; gradients are compared as a
relative L2 error per tensor (||g - ref|| / ||ref||) and as a norm ratio against the reference's golden norms.  The bound
is stated next to each assert; the observed values are printed and recorded in
$SHOWO_OBSERVED_DIR/train_parity.json when that variable is set.
"""
import numpy as np
import pytest
import torch

import fixtures as FX
import showo_b200
from oracle import showo_oracle as O
from showo_b200 import _lib, masks as M

pytestmark = pytest.mark.gpu
VOC = O.ShowoVocab()
REL_L2_TOL = 0.06            # bf16 operands + bf16 activations, 2 layers + head; observed worst 0.030 (profiles/r2_train_parity_observed.json)
NORM_TOL = 0.01              # observed worst 0.0049


@pytest.fixture(scope="module")
def dev():
    return torch.device("cuda", 0)


@pytest.fixture(scope="module")
def lib():
    return _lib.require_gpu()


def S():
    return _lib.current_stream_ptr()


def _record(key, value):
    FX.record_observed("train_parity.json", key, value)


def _dense_allowed(desc, L):
    q = torch.arange(L)[:, None]
    k = torch.arange(L)[None, :]
    return O.omni_predicate(q, k, *desc)


@pytest.mark.parametrize("n_seq,L,H,descs", [
    (1, 64, 2, [(0, 0, 0, 0, 0)]),                                        # pure causal, one tile
    (2, 200, 2, [(17, 130, 200, 0, 0), (0, 0, 0, 0, 0)]),                 # t2i row with left pads + full span, and an lm row
    (2, 387, 4, [(60, 129, 387, 0, 0), (0, 0, 0, 0, 259)]),               # t2i + mmu window
    (1, 1155, 2, [(100, 129, 1155, 0, 0)]),                               # 512x512 geometry
])
def test_attention_backward_against_autograd(lib, dev, n_seq, L, H, descs):
    g = torch.Generator().manual_seed(L + H)
    D = H * 64
    q, k, v, d_o = (torch.randn(n_seq * L, D, generator=g).bfloat16() for _ in range(4))
    qf, kf, vf = (t.float().view(n_seq, L, H, 64).transpose(1, 2).clone().requires_grad_(True) for t in (q, k, v))
    allowed = torch.stack([_dense_allowed(d, L) for d in descs])[:, None]
    s = (qf @ kf.transpose(-1, -2)) / 8.0
    s = s.masked_fill(~allowed, float("-inf"))
    p = s.softmax(-1)
    o = p @ vf
    lse2 = torch.logsumexp(s, -1) / np.log(2.0)                                 # exp2 domain
    dof = d_o.float().view(n_seq, L, H, 64).transpose(1, 2)
    (o * dof).sum().backward()
    o_bf = o.detach().transpose(1, 2).reshape(n_seq * L, D).bfloat16()
    lse_d = lse2.detach().transpose(1, 2).reshape(n_seq * L, H).contiguous().float().to(dev)
    dq, dk, dv = (torch.full((n_seq * L, D), float("nan"), dtype=torch.bfloat16, device=dev) for _ in range(3))
    qd, kd, vd, od, dod = (t.contiguous().to(dev) for t in (q, k, v, o_bf, d_o))
    _lib.check(lib.showo_attention_bwd_test(_lib.ptr(qd), _lib.ptr(kd), _lib.ptr(vd), _lib.ptr(od), _lib.ptr(dod), _lib.ptr(lse_d),
                                            _lib.ptr(dq), _lib.ptr(dk), _lib.ptr(dv), n_seq, L, H, _lib.masks_array(descs), S()),
               "attention_bwd_test")
    torch.cuda.synchronize()
    errs = {}
    for name, got, ref in (("dq", dq, qf.grad), ("dk", dk, kf.grad), ("dv", dv, vf.grad)):
        r = ref.transpose(1, 2).reshape(n_seq * L, D)
        gt = got.float().cpu()
        assert torch.isfinite(gt).all(), name
        errs[name] = float((gt - r).norm() / r.norm())
    print(f"attention backward L={L}: rel L2 {errs}")
    _record(f"attention_bwd_L{L}", errs)
    assert max(errs.values()) < 0.006, errs          # bf16 P / dS operands, bf16 outputs; observed 0.0027


@pytest.fixture(scope="module")
def tiny_train(dev):
    dims = O.PhiDims(**FX.TINY)
    W = O.make_showo_weights(dims, seed=3)
    m = showo_b200.Showo(False, dims.vocab_size, VOC.llm_vocab_size, phi_dims=FX.TINY, materialize=False)
    m.load_weights(W, device=dev)
    return dims, W, m


def _oracle_grads(dims, W, ids, mask, labels, sizes, coeff, input_embeddings=None):
    Wg = {k: v.clone().requires_grad_(True) for k, v in W.items()}
    if input_embeddings is not None:
        input_embeddings = input_embeddings.clone().requires_grad_(True)
        logits = O.showo_logits(Wg, dims, input_embeddings=input_embeddings, add_mask=mask)
    else:
        logits = O.showo_logits(Wg, dims, input_ids=ids, add_mask=mask)
    l = O.showo_losses(logits, labels, *sizes, 128)
    (coeff[0] * l[0] + coeff[1] * l[1] + coeff[2] * l[2]).backward()
    return logits.detach(), [float(x) for x in l], {k: v.grad for k, v in Wg.items()}, (input_embeddings.grad if input_embeddings is not None else None)


def test_train_step_against_reference_golden_and_oracle_autograd(tiny_train, dev):
    """losses + gradient norms + gradient probes of the reference (train_step.npz), and every parameter's gradient against the
    oracle's forward differentiated by autograd."""
    dims, W, m = tiny_train
    z = FX.load("train_step.npz")
    ids, mask, labels, sizes = FX.train_batch(VOC)
    B, L = ids.shape
    descs = M.descriptors_from_dense(mask.to(dev))
    terms = m._loss_terms(B, L, *sizes, 128)
    logits, losses = m.train_forward(ids.to(dev), None, descs, labels.to(dev), terms)
    got_l = losses[:, 0].cpu().numpy()
    print("losses", got_l, "reference", z["losses"], "counts", losses[:, 1].cpu().numpy())
    assert np.allclose(got_l, z["losses"], rtol=2e-3)
    dl = np.abs(logits[:, ::32, ::997].cpu().numpy() - z["logits_slice"]).max()
    assert dl < 0.03, dl
    # training forward == inference forward of the same engine up to the bf16 rounding of the un-fused q/k/fc1 buffer
    inf = m(ids.to(dev), attention_mask=descs)
    assert (inf - logits).abs().max().item() < 0.03
    m.backward(FX.TRAIN_COEFF)
    names = [str(n) for n in z["grad_names"]]
    _, ref_l, ref_g, _ = _oracle_grads(dims, W, ids, mask, labels, sizes, FX.TRAIN_COEFF)
    table, worst = {}, 0.0
    for i, k in enumerate(names):
        g = m.read_grad(k, like=W[k]).cpu()
        assert torch.isfinite(g).all(), k
        ref = ref_g[k]
        rel = float((g - ref).norm() / (ref.norm() + 1e-30))
        ratio = float(g.double().norm() / z["grad_norms"][i])
        table[k] = (rel, ratio)
        worst = max(worst, rel)
    for k, (rel, ratio) in sorted(table.items(), key=lambda kv: -kv[1][0])[:12]:
        print(f"  {k:60s} rel L2 {rel:.4f}  norm ratio vs reference {ratio:.4f}")
    _record("tiny_train_step", {"loss_rel_err": float(np.abs(got_l / z["losses"] - 1).max()), "worst_rel_l2": worst,
                                "worst_norm_ratio_dev": float(max(abs(r - 1) for _, r in table.values()))})
    bad = {k: v for k, v in table.items() if v[0] > REL_L2_TOL or abs(v[1] - 1) > NORM_TOL}
    assert not bad, bad
    for k in FX.TRAIN_GRAD_PROBES:
        g = m.read_grad(k, like=W[k]).cpu()
        got = (g[:8, :8] if g.dim() == 2 else g[:64]).numpy()
        ref = z["grad:" + k]
        assert np.abs(got - ref).max() <= 0.08 * np.abs(ref).max() + 1e-9, (k, np.abs(got - ref).max(), np.abs(ref).max())
    # the backward is deterministic except for the embedding scatter-add (fp32 atomics)
    m.train_forward(ids.to(dev), None, descs, labels.to(dev), terms, want_logits=False)
    m.backward(FX.TRAIN_COEFF)
    k = "showo.model.layers.0.self_attn.q_proj.weight"
    a = m.read_grad(k, like=W[k])
    m.train_forward(ids.to(dev), None, descs, labels.to(dev), terms, want_logits=False)
    m.backward(FX.TRAIN_COEFF)
    assert torch.equal(a, m.read_grad(k, like=W[k]))


def test_train_step_embeddings_input_and_loss_term_quirks(tiny_train, dev):
    """input_embeddings path (train_w_clip_vit.py): gradient wrt the embeddings; batch_size_mmu = 0 makes the mmu term cover
    the whole batch (python's -0 slice) and an empty lm slice gives NaN -- both reproduced, and the NaN term does not
    poison the gradients of the other terms when its coefficient is 0."""
    dims, W, m = tiny_train
    ids, mask, labels, _ = FX.train_batch(VOC)
    ids, mask, labels = ids[:3], mask[:3], labels[:3]
    B, L = ids.shape
    emb = W["showo.model.embed_tokens.weight"][ids]
    sizes, coeff = (2, 0, 0), (1.0, 0.0, 0.5)
    descs = M.descriptors_from_dense(mask.to(dev))
    terms = m._loss_terms(B, L, *sizes, 128)
    _, losses = m.train_forward(None, emb.to(dev), descs, labels.to(dev), terms, want_logits=False)
    demb = m.backward(coeff, want_input_grad_like=emb.to(dev)).cpu()
    _, ref_l, ref_g, ref_demb = _oracle_grads(dims, W, ids, mask, labels, sizes, coeff, input_embeddings=emb)
    got = losses[:, 0].cpu().numpy()
    assert np.isnan(got[1]) and np.isnan(ref_l[1])
    assert np.allclose(got[[0, 2]], [ref_l[0], ref_l[2]], rtol=2e-3)
    rel = float((demb - ref_demb).norm() / ref_demb.norm())
    print("d input_embeddings rel L2", rel)
    assert torch.isfinite(demb).all() and rel < REL_L2_TOL
    k = "showo.lm_head.weight"
    g = m.read_grad(k, like=W[k]).cpu()
    assert float((g - ref_g[k]).norm() / ref_g[k].norm()) < REL_L2_TOL
    assert float(m.read_grad("showo.model.embed_tokens.weight", like=W["showo.model.embed_tokens.weight"]).abs().max()) == 0.0


def test_autograd_bridge_matches_engine_gradients(dev):
    """Showo.forward(labels=...) under autograd + loss.backward() (training/train.py:589-612): parameters of the torch module
    receive exactly what showo_read_grad returns, an optimizer step re-packs the engine weights, and the loss goes down."""
    dims = O.PhiDims(**FX.TINY)
    W = O.make_showo_weights(dims, seed=3)
    m = showo_b200.Showo(False, dims.vocab_size, VOC.llm_vocab_size, phi_dims=FX.TINY).to(dev)
    m.load_state_dict({k: v for k, v in W.items()}, strict=True)
    ids, mask, labels, sizes = FX.train_batch(VOC)
    kw = dict(attention_mask=mask.to(dev), labels=labels.to(dev), batch_size_t2i=sizes[0], batch_size_lm=sizes[1],
              batch_size_mmu=sizes[2], max_seq_length=128)
    opt = torch.optim.SGD(m.parameters(), lr=0.05)
    logits, l1, l2, l3 = m(ids.to(dev), **kw)
    assert not logits.requires_grad and l1.requires_grad
    loss0 = FX.TRAIN_COEFF[0] * l1 + FX.TRAIN_COEFF[1] * l2 + FX.TRAIN_COEFF[2] * l3
    loss0.backward()
    p = dict(m.named_parameters())
    for k in ("showo.model.layers.1.mlp.fc2.weight", "showo.model.layers.0.self_attn.k_layernorm.weight", "showo.lm_head.bias"):
        assert torch.equal(p[k].grad, m.read_grad(k, like=p[k])), k
    assert all(q.grad is not None and torch.isfinite(q.grad).all() for q in m.parameters())
    opt.step()
    with torch.no_grad():
        _, a1, a2, a3 = m(ids.to(dev), **kw)
    loss1 = FX.TRAIN_COEFF[0] * a1 + FX.TRAIN_COEFF[1] * a2 + FX.TRAIN_COEFF[2] * a3
    print("loss before / after one SGD step", float(loss0), float(loss1))
    assert float(loss1) < float(loss0)
    # writes through .data are invisible to autograd's version counter: refresh_engine() is the documented way to pick them up
    with torch.no_grad():
        before = m(ids.to(dev), attention_mask=mask.to(dev))
        p["showo.lm_head.bias"].data.add_(1.0)
        stale = m(ids.to(dev), attention_mask=mask.to(dev))
        m.refresh_engine()
        fresh = m(ids.to(dev), attention_mask=mask.to(dev))
    assert torch.equal(before, stale) and (fresh - before - 1.0).abs().max().item() < 1e-4


def test_engine_adamw_matches_torch_adamw(dev):
    """showo_adamw_step on the engine's fp32 masters == torch.optim.AdamW as training/train.py:211-236 builds it (weight decay on every
    parameter whose name has no "bias": the reference's other no_decay patterns match no Phi parameter), three steps, every parameter --
    fed with the engine's own gradients, so only the optimizer arithmetic and the parameter mapping (fused W1 / W2 blocks, the two
    biases that share a gradient) are compared."""
    dims = O.PhiDims(**FX.TINY)
    W = O.make_showo_weights(dims, seed=3)
    # non-trivial biases / LayerNorm parameters so that the decay split is visible
    g = torch.Generator().manual_seed(9)
    W = {k: (v + 0.05 * torch.randn(v.shape, generator=g) if (k.endswith("bias") or "layernorm" in k) else v) for k, v in W.items()}
    m = showo_b200.Showo(False, dims.vocab_size, VOC.llm_vocab_size, phi_dims=FX.TINY, materialize=False)
    m.enable_optimizer(device=dev)
    m.load_weights(W, device=dev)
    ref = {k: v.clone().to(dev).requires_grad_(True) for k, v in W.items()}
    no_decay = ["bias", "layer_norm.weight", "mlm_ln.weight", "embeddings.weight"]                  # train.py:211
    hp = dict(lr=1e-3, betas=(0.9, 0.999), eps=1e-8)
    opt = torch.optim.AdamW([{"params": [p for n, p in ref.items() if not any(nd in n for nd in no_decay)], "weight_decay": 0.01},
                             {"params": [p for n, p in ref.items() if any(nd in n for nd in no_decay)], "weight_decay": 0.0}], **hp)
    ids, mask, labels, sizes = FX.train_batch(VOC)
    B, L = ids.shape
    descs = M.descriptors_from_dense(mask.to(dev))
    terms = m._loss_terms(B, L, *sizes, 128)
    losses = []
    for step in range(3):
        _, ls = m.train_forward(ids.to(dev), None, descs, labels.to(dev), terms, want_logits=False)
        losses.append(float((ls[:, 0] * torch.tensor(FX.TRAIN_COEFF, device=dev)).sum()))
        m.backward(FX.TRAIN_COEFF)
        for k, p in ref.items():
            p.grad = m.read_grad(k, like=p)
        opt.step()
        m.adamw_step(weight_decay=0.01, **hp)
        worst = 0.0
        for k, p in ref.items():
            got = m.read_param(k, like=p)
            err = float((got - p.detach()).abs().max() / (p.detach().abs().max() + 1e-12))
            worst = max(worst, err)
            assert err < 2e-6, (step, k, err)
        print(f"adamw step {step}: loss {losses[-1]:.4f}, worst relative parameter difference vs torch {worst:.2e}")
    assert losses[2] < losses[0]                  # the engine trains on its own updated bf16 working copies
    # a decayed LayerNorm weight and an undecayed bias really moved differently from their gradients alone
    k_w, k_b = "showo.model.layers.0.input_layernorm.weight", "showo.model.layers.0.input_layernorm.bias"
    assert not torch.equal(m.read_param(k_w, like=ref[k_w]), W[k_w].to(dev)) and not torch.equal(m.read_param(k_b, like=ref[k_b]), W[k_b].to(dev))
    _record("adamw_vs_torch", {"worst_rel_param_diff": worst, "losses": losses})


def test_mm_projector_backward_against_torch_autograd(dev):
    """Showo.mm_projector under autograd (training/train_w_clip_vit.py:599-601 trains it through `input_embeddings`): the drop-in's
    call is differentiable, its backward is showo_mm_projector_backward (two weight-gradient GEMMs on token-major operands, one dgrad
    GEMM against the transposed 2.weight, exact-erf GELU derivative), and the four parameters receive gradients within bf16 tolerance of
    torch fp32 autograd on the same parameters.  Row count 117: not a multiple of the GEMMs' 128-wide token block.  Then the
    engine-side AdamW moves the four tensors exactly like torch.optim.AdamW (weights decayed, biases not)."""
    torch.manual_seed(5)
    m = showo_b200.Showo(True, 58498, 50295, phi_dims=FX.TINY).to(dev)
    with torch.no_grad():
        for p in m.mm_projector.parameters():
            if p.dim() == 1:
                p.add_(0.05 * torch.randn_like(p))
    x = torch.randn(3, 39, 1024, device=dev)
    gy = torch.randn(3, 39, 2048, device=dev) * 0.1
    out = m.mm_projector(x)
    assert out.requires_grad
    (out * gy).sum().backward()
    seq = torch.nn.Sequential(torch.nn.Linear(1024, 2048), torch.nn.GELU(), torch.nn.Linear(2048, 2048)).to(dev)
    seq.load_state_dict({k: v.detach().clone() for k, v in m.mm_projector.state_dict().items()})
    (seq(x) * gy).sum().backward()
    table = {}
    for (k, p), q in zip(m.mm_projector.named_parameters(), seq.parameters()):
        assert p.grad is not None and torch.isfinite(p.grad).all(), k
        table[k] = float((p.grad - q.grad).norm() / q.grad.norm())
        assert torch.equal(p.grad, m.read_grad("mm_projector." + k, like=p)), k
    print("mm_projector gradients, rel L2 vs torch fp32:", {k: round(v, 4) for k, v in table.items()})
    _record("mm_projector_backward", table)
    assert max(table.values()) < 0.02, table
    with torch.no_grad():                       # no autograd: the plain engine call, same values
        assert torch.equal(m.mm_projector(x), out.detach())
    with pytest.raises(_lib.ShowoError):
        m.mm_projector(x.clone().requires_grad_(True))      # the CLIP features are frozen in the reference: no gradient for them
    with pytest.raises(_lib.ShowoError):
        m.mm_projector_backward(gy[:2])                      # differentiates the LAST call: row count must match

    # ---- optimizer: engine AdamW on the projector vs torch.optim.AdamW fed with the engine's gradients
    m2 = showo_b200.Showo(True, 58498, 50295, phi_dims=FX.TINY).to(dev)
    m2.load_state_dict(m.state_dict())
    m2.enable_optimizer()
    ref = {k: p.detach().clone().requires_grad_(True) for k, p in m2.mm_projector.named_parameters()}
    hp = dict(lr=1e-3, betas=(0.9, 0.999), eps=1e-8)
    opt = torch.optim.AdamW([{"params": [p for n, p in ref.items() if "bias" not in n], "weight_decay": 0.01},
                             {"params": [p for n, p in ref.items() if "bias" in n], "weight_decay": 0.0}], **hp)
    dims = O.PhiDims(**FX.TINY)
    ids, mask, labels, sizes = FX.train_batch(VOC)
    descs = M.descriptors_from_dense(mask.to(dev))
    terms = m2._loss_terms(ids.shape[0], ids.shape[1], *sizes, 128)
    for step in range(2):
        m2.train_forward(ids.to(dev), None, descs, labels.to(dev), terms, want_logits=False)      # adamw_step wants backbone gradients too
        m2.backward(FX.TRAIN_COEFF)
        with torch.no_grad():
            m2.mm_projector(x)
        m2.mm_projector_backward(gy)
        for k, p in ref.items():
            p.grad = m2.read_grad("mm_projector." + k, like=p)
        opt.step()
        m2.adamw_step(weight_decay=0.01, **hp)
        for k, p in ref.items():
            got = m2.read_param("mm_projector." + k, like=p)
            err = float((got - p.detach()).abs().max() / (p.detach().abs().max() + 1e-12))
            assert err < 2e-6, (step, k, err)
    # the projector's bf16 working copy follows the masters: its output moved, and matches torch on the updated parameters
    seq.load_state_dict({k: p.detach() for k, p in ref.items()})
    with torch.no_grad():
        new = m2._project(x)
        want = seq(x)
    assert (new - want).abs().max().item() < 0.01 * want.abs().max().item() and not torch.equal(new, out.detach())
    # a step without a projector backward leaves the projector alone
    m2.train_forward(ids.to(dev), None, descs, labels.to(dev), terms, want_logits=False)
    m2.backward(FX.TRAIN_COEFF)
    before = m2.read_param("mm_projector.2.weight", like=ref["2.weight"])
    m2.adamw_step(weight_decay=0.01, **hp)
    assert torch.equal(before, m2.read_param("mm_projector.2.weight", like=ref["2.weight"]))


def test_train_step_mixed_ids_and_embeddings_input(tiny_train, dev):
    """showo_train_forward with BOTH ids and embeddings = the rows of train_w_clip_vit.py:532-537 without the torch-side embed / cat:
    positions with ids >= 0 come from the engine's table, positions with ids < 0 take the caller's vector (the mm_projector output).
    Losses, the embedding-table gradient (scatter-add over the ids >= 0 positions only) and the gradient handed back for the ids < 0
    positions against the oracle differentiated by autograd with the same mixed input."""
    dims, W, m = tiny_train
    ids, mask, labels, sizes = FX.train_batch(VOC)
    B, L = ids.shape
    g = torch.Generator().manual_seed(17)
    vis = torch.zeros(B, L, dtype=torch.bool)
    vis[-sizes[2]:, 3:60] = True                                   # a visual span inside the mmu rows
    given = torch.randn(B, L, dims.hidden, generator=g) * 0.02
    ids_mixed = torch.where(vis, torch.full_like(ids, -1), ids)
    labels = torch.where(vis, torch.full_like(labels, -100), labels)
    descs = M.descriptors_from_dense(mask.to(dev))
    terms = m._loss_terms(B, L, *sizes, 128)
    _, losses = m.train_forward(ids_mixed.to(dev), given.to(dev), descs, labels.to(dev), terms, want_logits=False)
    demb = m.backward(FX.TRAIN_COEFF, want_input_grad_like=given.to(dev)).cpu()
    # oracle: the same mixed embeddings built in torch, differentiated wrt the table and the given vectors
    Wg = {k: v.clone().requires_grad_(True) for k, v in W.items()}
    gv = given.clone().requires_grad_(True)
    emb = torch.where(vis[..., None], gv, Wg["showo.model.embed_tokens.weight"][ids])
    logits = O.showo_logits(Wg, dims, input_embeddings=emb, add_mask=mask)
    l = O.showo_losses(logits, labels, *sizes, 128)
    (FX.TRAIN_COEFF[0] * l[0] + FX.TRAIN_COEFF[1] * l[1] + FX.TRAIN_COEFF[2] * l[2]).backward()
    assert np.allclose(losses[:, 0].cpu().numpy(), [float(v) for v in l], rtol=2e-3)
    k = "showo.model.embed_tokens.weight"
    ge = m.read_grad(k, like=W[k]).cpu()
    rel_e = float((ge - Wg[k].grad).norm() / Wg[k].grad.norm())
    rel_v = float((demb[vis] - gv.grad[vis]).norm() / gv.grad[vis].norm())
    print(f"mixed input: embedding-table gradient rel L2 {rel_e:.4f}, visual-span gradient rel L2 {rel_v:.4f}")
    _record("mixed_input", {"embed_rel_l2": rel_e, "visual_rel_l2": rel_v})
    assert rel_e < REL_L2_TOL and rel_v < REL_L2_TOL
    k2 = "showo.model.layers.0.mlp.fc1.weight"
    assert float((m.read_grad(k2, like=W[k2]).cpu() - Wg[k2].grad).norm() / Wg[k2].grad.norm()) < REL_L2_TOL


def test_train_w_clip_vit_call_shape_end_to_end(dev):
    """The training step as training/train_w_clip_vit.py:532-537,599-612 writes it, on a 1-layer model of the real width (the projector's
    output is 2048 wide): `model.showo.model.embed_tokens(ids)` and `model.mm_projector(feats)` are called from outside, concatenated
    into `input_embeddings`, `model(...)` returns the losses under autograd and `loss.backward()` reaches the backbone (showo_backward),
    the projector (showo_mm_projector_backward, through the gradient of `input_embeddings`) and the embedding table (torch's own
    nn.Embedding backward, as in the reference).  Compared with the oracle's forward differentiated by autograd on the same weights."""
    dims = O.PhiDims(hidden=2048, n_layers=1, n_heads=32, ffn=2048)
    W = O.make_showo_weights(dims, seed=8, w_clip_vit=True)
    m = showo_b200.Showo(True, dims.vocab_size, VOC.llm_vocab_size, phi_dims=dict(hidden=2048, n_layers=1, n_heads=32, ffn=2048)).to(dev)
    m.load_state_dict(W, strict=True)
    B, sysl, n_vis, n_txt = 2, 4, 576, 40
    L = 1 + sysl + 1 + n_vis + 1 + n_txt
    r = FX.rng(31)
    ids = torch.from_numpy(r.integers(0, 50257, size=(B, L)).astype("int64"))
    feats = torch.from_numpy(r.standard_normal(size=(B, n_vis, 1024), dtype=np.float32))
    labels = torch.full((B, L), -100, dtype=torch.int64)
    labels[:, L - n_txt:] = ids[:, L - n_txt:]
    b0 = 1 + sysl + 1
    allowed = O.mask_allowed_mmu_vit(B, L, system_prompt_len=sysl, n_vis=n_vis)
    mask = O.additive_from_allowed(allowed)

    # ---- the drop-in, reference call shape
    ids_d, feats_d = ids.to(dev), feats.to(dev)
    emb_text = m.showo.model.embed_tokens(ids_d)
    vis = m.mm_projector(feats_d)
    input_embeddings = torch.cat([emb_text[:, :b0], vis, emb_text[:, b0 + n_vis:]], dim=1)
    logits, l_t2i, l_lm, l_mmu = m(None, input_embeddings=input_embeddings, attention_mask=mask.to(dev), labels=labels.to(dev),
                                   batch_size_t2i=0, batch_size_lm=0, batch_size_mmu=B, max_seq_length=128)
    l_mmu.backward()
    # ---- the oracle
    Wg = {k: v.clone().requires_grad_(True) for k, v in W.items()}
    e_ref = Wg["showo.model.embed_tokens.weight"][ids]
    h = torch.nn.functional.gelu(feats @ Wg["mm_projector.0.weight"].T + Wg["mm_projector.0.bias"])
    v_ref = h @ Wg["mm_projector.2.weight"].T + Wg["mm_projector.2.bias"]
    lg = O.showo_logits(Wg, dims, input_embeddings=torch.cat([e_ref[:, :b0], v_ref, e_ref[:, b0 + n_vis:]], dim=1), add_mask=mask)
    ref_l = O.showo_losses(lg, labels, 0, 0, B, 128)
    ref_l[2].backward()
    print("loss_mmu", float(l_mmu), "oracle", float(ref_l[2]))
    assert abs(float(l_mmu) / float(ref_l[2]) - 1) < 2e-3
    table = {}
    p = dict(m.named_parameters())
    for k in ("mm_projector.0.weight", "mm_projector.0.bias", "mm_projector.2.weight", "mm_projector.2.bias",
              "showo.model.embed_tokens.weight", "showo.model.layers.0.self_attn.q_proj.weight", "showo.model.layers.0.mlp.fc2.weight",
              "showo.lm_head.weight"):
        assert p[k].grad is not None and torch.isfinite(p[k].grad).all(), k
        table[k] = float((p[k].grad.cpu() - Wg[k].grad).norm() / Wg[k].grad.norm())
    print("train_w_clip_vit flow, rel L2 vs oracle autograd:", {k: round(v, 4) for k, v in table.items()})
    _record("train_w_clip_vit_flow", table)
    assert max(table.values()) < REL_L2_TOL, table
