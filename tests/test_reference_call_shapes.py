"""Static drop-in check: every call the reference's scripts make on the objects this repo replaces -- `model` (Showo), `vq_model`
(MAGVITv2), `get_mask_chedule`, `mask_or_random_replace_tokens`, `uni_prompting` for the t2i rows -- was parsed out of inference_t2i.py /
inference_mmu.py / training/train.py / training/train_w_clip_vit.py into tests/golden/reference_calls.json
(tests/golden/make_golden_vs_reference.py) and is bound here against the drop-in's signatures: the method has to exist and accept the
positional count and every keyword the script passes (or swallow it through **kwargs like the reference does).  Besides the GPU tests
that drive the same methods with the scripts' argument shapes, this is the strongest offline statement of "runs unchanged"."""
import inspect
import json
import os

import pytest
import torch

import fixtures as FX
import showo_b200
from showo_b200 import train_inputs

# instances, not classes: mm_projector only exists on a w_clip_vit model (like in the reference)
TARGETS = {"model": showo_b200.Showo(True, 58498, 50295, phi_dims=dict(hidden=128, n_layers=1, n_heads=2, ffn=256)),
           "vq_model": showo_b200.MAGVITv2(materialize=False),
           # the CLIP-ViT tower of inference_mmu.py:74,133 / train_w_clip_vit.py:216-218,531 (constructed from dims: no checkpoint offline)
           "vision_tower": showo_b200.CLIPVisionTower(dict(image_size=336, patch_size=14, hidden=1024, n_layers=24, n_heads=16, ffn=4096))}
FUNCS = {"get_mask_chedule": showo_b200.get_mask_chedule, "mask_or_random_replace_tokens": train_inputs.mask_or_random_replace_tokens}
# attribute chains the scripts read (not call) on the model objects
ATTRS = {"model": ["config", "showo", "mm_projector", "output_size"], "vq_model": [], "vision_tower": []}
# nn.Module / HF plumbing both sides inherit or that is exercised elsewhere: not part of the hot-path surface
SKIP_METHODS = {"to", "eval", "train", "requires_grad_", "parameters", "named_parameters", "state_dict", "load_state_dict", "from_pretrained",
                "module", "get", "resize_token_embeddings"}


def _reference_calls():
    with open(os.path.join(FX.HERE, "reference_calls.json")) as f:
        ref = json.load(f)
    assert ref["objects"] == list(TARGETS) and ref["functions"] == list(FUNCS)
    return ref["calls"]


def _accepts(fn, n_pos, kws, bound):
    sig = inspect.signature(fn)
    params = list(sig.parameters.values())
    if bound and params and params[0].name in ("self", "cls"):
        params = params[1:]
    has_var_kw = any(p.kind == p.VAR_KEYWORD for p in params)
    has_var_pos = any(p.kind == p.VAR_POSITIONAL for p in params)
    positional = [p for p in params if p.kind in (p.POSITIONAL_ONLY, p.POSITIONAL_OR_KEYWORD)]
    if n_pos > len(positional) and not has_var_pos:
        return f"takes {len(positional)} positional arguments, the script passes {n_pos}"
    names = {p.name for p in params if p.kind in (p.POSITIONAL_OR_KEYWORD, p.KEYWORD_ONLY)}
    missing = [k for k in kws if k not in names and not has_var_kw]
    return f"does not accept keyword(s) {missing}" if missing else None


@pytest.mark.parametrize("script", ["inference_t2i.py", "inference_mmu.py", "training/train.py", "training/train_w_clip_vit.py"])
def test_every_call_of_the_reference_scripts_binds_to_the_drop_in(script):
    calls = _reference_calls()[script]
    assert calls, f"no calls on {list(TARGETS)} found in {script}"
    problems, checked = [], 0
    for obj, meth, n_pos, kws, line in calls:
        if meth in SKIP_METHODS:
            continue
        if obj is None:
            why = _accepts(FUNCS[meth], n_pos, kws, bound=False)
        else:
            inst = TARGETS[obj]
            if not hasattr(inst, meth):
                problems.append(f"{script}:{line}: {obj}.{meth} does not exist on {type(inst).__name__}")
                continue
            fn = getattr(inst, meth)
            why = _accepts(fn.forward if isinstance(fn, torch.nn.Module) else fn, n_pos, kws, bound=False)
        checked += 1
        if why:
            problems.append(f"{script}:{line}: {obj or ''}.{meth}({n_pos} positional, {kws}) {why}")
    assert checked > 0 and not problems, "\n".join(problems)


def test_attributes_the_scripts_read_exist():
    m = TARGETS["model"]
    for a in ATTRS["model"]:
        assert hasattr(m, a), a
    assert hasattr(m.config, "mask_token_id") and m.config.mask_token_id == 58497          # inference_t2i.py:70
    assert callable(m.showo.model.embed_tokens)                                             # inference_mmu.py:136
    assert hasattr(train_inputs.UniversalPrompting, "t2i_prompt") and hasattr(train_inputs.UniversalPrompting, "__call__")
    assert hasattr(train_inputs.UniversalPrompting, "t2i_gen_prompt")                        # inference_t2i.py:115,118 ('t2i_gen')
    vt = TARGETS["vision_tower"]                                                             # models/clip_encoder.py:53-82
    for a in ("dummy_feature", "dtype", "device", "config", "hidden_size", "num_patches_per_side", "num_patches", "image_processor", "is_loaded"):
        assert hasattr(vt, a), a
    assert vt.num_patches == 576 and vt.hidden_size == 1024
