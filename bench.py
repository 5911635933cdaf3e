#!/usr/bin/env python
"""bench.py -- headline benchmark of the Show-o hot path on B200 (contract: see the task brief / DESIGN.md section 6).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
  torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...          (N > 1: one rank per GPU, NCCL)

A "step" = one batch of the configs[1] workload of BASELINE.json on every rank: showo_demo.yaml t2i 256x256,
18 denoise steps, CFG 5, batch 8 per GPU (weak scaling) -> t2i_generate + MAGVIT decode_code + uint8 conversion
(SURVEY.md section 8d, config 2), then (N > 1) an NCCL all-gather of the uint8 images.
Prints ONE JSON line on rank 0.

--dump-outputs DIR: after the timed steps, rank 0 saves what the last headline step returned to it as float32
DIR/codes.npy ([8, 256] image-token ids from t2i_generate) and DIR/images.npy ([8, 256, 256, 3] uint8 pixel values),
6.3 MB in all.  Weights, prompts and torch's RNG are seeded, so the same arguments give the same inputs on every run
and two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import sys
import threading
import time
from types import SimpleNamespace as NS

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "t2i_256x256_images_per_sec_18steps_cfg5"
UNIT = "images/s"
B_PER_GPU, N_TOK, T_STEPS, CFG_W, L_SEQ, P_TXT, CODEBOOK = 8, 256, 18, 5.0, 387, 129, 8192
D, NL, H, F, V = 2048, 24, 32, 8192, 58498
# algorithmic FLOPs (SURVEY.md section 8d): per-token 24-layer GEMM, attention per (q,k) pair, head per position
G_TOK = 2 * NL * (4 * D * D + 2 * D * F)
A_PAIR = 4 * D * NL
F_IMG = T_STEPS * 2 * ((N_TOK + 2) * (G_TOK + A_PAIR * L_SEQ) + N_TOK * 2 * D * CODEBOOK) + 2 * P_TXT * (G_TOK + A_PAIR * P_TXT / 2)
F_DEC = 300.9e9           # MAGVIT-v2 decode, per 256x256 image (SURVEY.md section 6, probed)


def t2i_config():
    return NS(model=NS(showo=NS(num_vq_tokens=N_TOK, num_new_special_tokens=10, llm_vocab_size=50295)),
              dataset=NS(preprocessing=NS(max_seq_length=P_TXT - 1)))


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(bf16_burst=d.get("bf16_tflops", 1590.0), bf16_sustained=d.get("bf16_tflops_sustained", 1400.0),
                    hbm=d.get("hbm_gbs", 6650.0), source="measured (MEASURED_PEAKS.json)")
    return dict(bf16_burst=1590.0, bf16_sustained=1400.0, hbm=6650.0, source="fallback (B200_PROFILING.md)")


def ncu_traffic():
    """dram bytes per launch of the dominant kernel from the committed ncu --set full captures (profiles/r2_traffic.json)."""
    try:
        t = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))["gemm_tcgen05_kernel"]
        return {k: {"dram_bytes": v["dram_bytes"], "algorithmic_bytes": v["algorithmic_bytes"]} for k, v in t.items()}
    except Exception:
        return None


class ClockSampler(threading.Thread):
    """nvidia-smi style clock / throttle-reason sampling during the timed region (pynvml)."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index, self.samples, self.reasons, self.stop_flag, self.max_mhz = index, [], set(), False, None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def run(self):
        if self.nv is None:
            return
        nv = self.nv
        names = {nv.nvmlClocksThrottleReasonHwSlowdown: "hw_slowdown",
                 nv.nvmlClocksThrottleReasonHwThermalSlowdown: "hw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwThermalSlowdown: "sw_thermal_slowdown",
                 nv.nvmlClocksThrottleReasonSwPowerCap: "sw_power_cap"}
        while not self.stop_flag:
            try:
                self.samples.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, n in names.items():
                    if r & bit:
                        self.reasons.add(n)
            except Exception:
                pass
            time.sleep(0.1)

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons),
                "samples": len(s)}


def synth_prompts(torch, batch, seed):
    """Synthetic t2i_gen rows (prompting_utils.py:92-123): left-padded [t2i][bos] text [eos] + [soi] 256 x mask [eoi]."""
    g = torch.Generator().manual_seed(seed)
    PAD, SOI, EOI, T2I, BOS = 50295, 50296, 50297, 50300, 50256
    cond = torch.full((batch, L_SEQ), PAD, dtype=torch.int64)
    unc = torch.full((batch, L_SEQ), PAD, dtype=torch.int64)
    descs_c, descs_u = [], []
    for b in range(batch):
        n = int(torch.randint(8, 65, (1,), generator=g))
        text = torch.randint(0, 50257, (n,), generator=g)
        row = torch.cat([torch.tensor([T2I, BOS]), text, torch.tensor([BOS])])
        cond[b, P_TXT - row.numel():P_TXT] = row
        unc[b, P_TXT - 3:P_TXT] = torch.tensor([T2I, BOS, BOS])
        for r in (cond, unc):
            r[b, P_TXT] = SOI
            r[b, P_TXT + 1:P_TXT + 1 + N_TOK] = V - 1
            r[b, P_TXT + 1 + N_TOK] = EOI
        descs_c.append((P_TXT - row.numel(), P_TXT, L_SEQ, 0, 0))
        descs_u.append((P_TXT - 3, P_TXT, L_SEQ, 0, 0))
    return cond, unc, descs_c + descs_u


def dense_mask_like_reference(torch, ids, pad_id=50295, soi_id=50296, eoi_id=50297):
    """What the reference's caller does before every t2i_generate (inference_t2i.py:300 -> create_attention_mask_predict_next,
    training/prompting_utils.py:466-511, rm_pad_in_image=True): dense additive fp32 [2B, 1, L, L] on the device."""
    n, L = ids.shape
    is_pad = ids == pad_id
    is_soi, is_eoi = ids == soi_id, ids == eoi_id
    in_img = (torch.cumsum(is_soi, 1) - torch.cumsum(is_eoi, 1)) > 0
    in_img = in_img | is_eoi
    causal = torch.tril(torch.ones(L, L, dtype=torch.bool, device=ids.device))
    allowed = causal[None] | in_img[:, :, None]
    allowed = allowed & ~(is_pad[:, None, :] & ~is_pad[:, :, None])
    add = torch.zeros(n, 1, L, L, dtype=torch.float32, device=ids.device)
    add.masked_fill_(~allowed[:, None], float(torch.iinfo(torch.int64).min))
    return add


def gpu_random_weights(torch, dev, seed=0):
    """Random-init Phi-1.5-sized state_dict generated on the device (N(0,0.02) matrices, zero biases, LN 1/0 --
    PhiPreTrainedModel._init_weights, phi.py:833-842).  Yields (name, tensor) one at a time to bound memory."""
    g = torch.Generator(device=dev).manual_seed(seed)

    def mat(o, i):
        return torch.randn(o, i, device=dev, generator=g) * 0.02
    yield "showo.model.embed_tokens.weight", mat(V, D)
    for l in range(NL):
        p = f"showo.model.layers.{l}."
        for n, (o, i) in {"self_attn.q_proj": (D, D), "self_attn.k_proj": (D, D), "self_attn.v_proj": (D, D),
                          "self_attn.dense": (D, D), "mlp.fc1": (F, D), "mlp.fc2": (D, F)}.items():
            yield p + n + ".weight", mat(o, i)
            yield p + n + ".bias", torch.zeros(o, device=dev)
        for n, c in {"input_layernorm": D, "self_attn.q_layernorm": 64, "self_attn.k_layernorm": 64}.items():
            yield p + n + ".weight", torch.ones(c, device=dev)
            yield p + n + ".bias", torch.zeros(c, device=dev)
    yield "showo.model.final_layernorm.weight", torch.ones(D, device=dev)
    yield "showo.model.final_layernorm.bias", torch.zeros(D, device=dev)
    yield "showo.lm_head.weight", mat(V, D)
    yield "showo.lm_head.bias", torch.zeros(V, device=dev)


def gpu_random_magvit_weights(torch, dev, seed=1):
    """Random-init MAGVIT-v2 state_dict (nn.Conv2d default: U(+-1/sqrt(fan_in)); GroupNorm 1/0) generated on the device."""
    from showo_b200.magvit_model import _param_shapes
    g = torch.Generator(device=dev).manual_seed(seed)
    W = {}
    shapes = _param_shapes()
    for name, shp in shapes.items():
        if len(shp) == 4:
            bound = 1.0 / math.sqrt(shp[1] * shp[2] * shp[3])
            W[name] = (torch.rand(shp, device=dev, generator=g) * 2 - 1) * bound
        elif ".norm" in name:
            W[name] = torch.ones(shp, device=dev) if name.endswith("weight") else torch.zeros(shp, device=dev)
        else:
            ws = shapes[name[:-5] + ".weight"]
            bound = 1.0 / math.sqrt(ws[1] * ws[2] * ws[3])
            W[name] = (torch.rand(shp, device=dev, generator=g) * 2 - 1) * bound
    return W


# ======================================================================================================= ours
def run_ours(args):
    import torch
    import torch.distributed as dist
    import showo_b200
    from showo_b200 import _lib

    from showo_b200 import parallel as P
    rank, local, world = P.env_world()
    assert world == args.gpus, f"--gpus {args.gpus} but WORLD_SIZE={world}: launch with torchrun for N > 1"
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    P.init("nccl", dev)
    lib = _lib.require_gpu()
    torch.manual_seed(0)          # t2i_generate draws its sampler seed from torch's RNG: identical runs for identical arguments

    model = showo_b200.Showo(False, V, 50295, materialize=False)
    model._make_engine(dev)
    for name, t in gpu_random_weights(torch, dev, seed=0):      # streamed one tensor at a time (no 5.8 GB fp32 copy)
        _lib.check(lib.showo_load_weight(model._engine, name.encode(), _lib.ptr(t), t.numel(), 1), f"load {name}")
    _lib.check(lib.showo_weights_complete(model._engine), "weights_complete")
    model._streamed = True
    vq = showo_b200.MAGVITv2(materialize=False)
    vq.load_weights(gpu_random_magvit_weights(torch, dev, seed=1), device=dev)

    cfg = t2i_config()
    cond_h, unc_h, descs = synth_prompts(torch, B_PER_GPU, seed=1234 + rank)
    cond_pin, unc_pin = cond_h.pin_memory(), unc_h.pin_memory()
    unc_d = unc_h.to(dev)
    imgs_pin = torch.empty(B_PER_GPU, 256, 256, 3, dtype=torch.uint8).pin_memory()
    gather_buf = torch.empty(world * B_PER_GPU, 256, 256, 3, dtype=torch.uint8, device=dev) if world > 1 else None
    ids_d = torch.empty_like(cond_h, device=dev)
    cond_d0 = cond_h.to(dev)

    phase_s = {"mask": 0.0, "generate_call": 0.0, "decode_call": 0.0, "tail_sync": 0.0}
    e2e_step_ms = []

    def one_step(e2e: bool):
        t0 = time.perf_counter()
        if e2e:
            ids_d.copy_(cond_pin, non_blocking=True)           # H2D of this step's prompts (pinned)
            unc_d.copy_(unc_pin, non_blocking=True)
            # the reference's call shape (inference_t2i.py:300,321): the caller builds the DENSE [2B,1,L,L] mask and hands it to
            # t2i_generate; the shim recovers + verifies the closed-form descriptors from it (showo_mask_descriptors, one
            # kernel + a 24 B/sequence read-back) -- all inside the timed region
            mask = dense_mask_like_reference(torch, torch.cat([ids_d, unc_d]))
        else:
            ids_d.copy_(cond_d0)                               # device-resident inputs
            mask = descs
        t1 = time.perf_counter()
        codes = model.t2i_generate(ids_d, unc_d, mask, guidance_scale=CFG_W, timesteps=T_STEPS, config=cfg)
        t2 = time.perf_counter()
        imgs = vq.decode_code_uint8(torch.clamp(codes, 0, CODEBOOK - 1))
        if world > 1:
            dist.all_gather_into_tensor(gather_buf, imgs)
        t3 = time.perf_counter()
        if e2e:
            imgs_pin.copy_(imgs, non_blocking=True)            # D2H of the step's result
            torch.cuda.current_stream().synchronize()
            t4 = time.perf_counter()                           # host-side split of the e2e step (reported under e2e.host_phases_ms)
            phase_s["mask"] += t1 - t0; phase_s["generate_call"] += t2 - t1; phase_s["decode_call"] += t3 - t2; phase_s["tail_sync"] += t4 - t3
            e2e_step_ms.append(round(1e3 * (t4 - t0), 1))
        return codes, imgs

    def timed(e2e: bool, steps: int):
        """device time of `steps` steps, and what the last one returned"""
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            last = one_step(e2e)
        e1.record()
        torch.cuda.synchronize()
        ms = P.max_over_ranks(e0.elapsed_time(e1), dev)       # the slowest rank's device time
        if world > 1:
            dist.barrier()
        return ms, last

    for _ in range(max(args.warmup, 3)):      # both call shapes warm up (first-use allocations, pinned-copy set-up, mempool creation)
        one_step(False)
        one_step(True)
    sampler = ClockSampler(local)
    sampler.start()
    ms_dev, (codes, imgs) = timed(False, args.steps)
    launches = model.kernel_launches() + vq.kernel_launches()
    for k in phase_s:
        phase_s[k] = 0.0
    ms_e2e, _ = timed(True, args.steps)
    host_phases = {k: round(1e3 * v / args.steps, 2) for k, v in phase_s.items()}
    sampler.stop_flag = True
    sampler.join(timeout=2)
    if args.dump_outputs and rank == 0:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, t in (("codes", codes), ("images", imgs)):
            np.save(os.path.join(args.dump_outputs, name + ".npy"), t.float().cpu().numpy())

    # ---- secondaries run on EVERY rank (weak scaling like the headline) and are aggregated below
    if os.environ.get("SHOWO_BENCH_HEADLINE_ONLY"):           # A/B runs while tuning: the headline line only
        if rank == 0:
            print(json.dumps({"metric": METRIC, "value": round(world * B_PER_GPU * args.steps / (ms_dev / 1e3), 3), "ms_per_step": round(ms_dev / args.steps, 3),
                              "e2e_ms_per_step": round(ms_e2e / args.steps, 3), "e2e_host_phases_ms": host_phases, "e2e_step_ms_all": e2e_step_ms, "clocks": sampler.summary(),
                              "env": {k: v for k, v in os.environ.items() if k.startswith("SHOWO_")}}), flush=True)
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return None
    mmu_local = mmu_decode_bench(torch, model, vq, dev, measured_peaks(), seed=5 + rank)
    mmu_agg = torch.tensor([mmu_local["ms_per_decode_step"], mmu_local["value"]], device=dev, dtype=torch.float64)

    def guarded(name, fn):
        """a secondary must never take the headline line down with it (same code on every rank: a failure is a failure everywhere)"""
        try:
            return fn()
        except Exception as e:          # noqa: BLE001
            import traceback
            traceback.print_exc()
            return {"metric": name, "error": f"{type(e).__name__}: {e}"[:400]}
    t512 = guarded("t2i_512x512", lambda: t2i512_bench(torch, dist, model, vq, dev, world, rank))
    train = None if os.environ.get("SHOWO_BENCH_SKIP_TRAIN") else guarded("train_step", lambda: train_step_bench(torch, dist, model, dev, world, rank))
    if world > 1:
        mx = mmu_agg.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(mmu_agg, op=dist.ReduceOp.SUM)
        mmu_local["ms_per_decode_step_max_over_ranks"] = round(float(mx[0]), 4)
        mmu_local["value_rank0"] = mmu_local["value"]
        # whole-job tokens/s: every rank decodes its own 16 sequences; time = the slowest rank's step
        mmu_local["value"] = round(world * 16 * 1000.0 / float(mx[0]), 1)
        mmu_local["n_gpus"] = world

    n_img = world * B_PER_GPU * args.steps
    value = n_img / (ms_dev / 1e3)
    e2e_value = n_img / (ms_e2e / 1e3)
    peaks = measured_peaks()

    out = None
    if rank == 0:
        # ---- dominant kernel (tcgen05 GEMM) timed alone with CUDA events on its launch stream: the three shapes of a step
        S = _lib.current_stream_ptr
        shapes = [("qkv_fc1", 16 * 258, 3 * D + F, D, 0, NL), ("dense_fc2", 16 * 258, D, D + F, 1, NL), ("head_img", 16 * 256, CODEBOOK, D, 2, 1)]
        tot_f = tot_ms = 0.0
        per_shape = {}
        for name, m_, n_, k_, epi, count in shapes:
            A = (torch.randn(m_, k_, device=dev) * 0.5).bfloat16()
            Bw = (torch.randn(n_, k_, device=dev) * 0.02).bfloat16()
            o = torch.empty(m_, n_, device=dev, dtype=torch.bfloat16 if epi == 0 else torch.float32)
            r = torch.zeros(m_, n_, device=dev) if epi == 1 else None
            for _ in range(3):
                lib.showo_gemm_bf16(_lib.ptr(A), k_, _lib.ptr(Bw), k_, m_, n_, k_, _lib.ptr(o), n_, None, _lib.ptr(r), n_, n_, epi, 0, S())
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(20):
                lib.showo_gemm_bf16(_lib.ptr(A), k_, _lib.ptr(Bw), k_, m_, n_, k_, _lib.ptr(o), n_, None, _lib.ptr(r), n_, n_, epi, 0, S())
            e1.record()
            torch.cuda.synchronize()
            ms = e0.elapsed_time(e1) / 20
            fl = 2.0 * m_ * n_ * k_
            per_shape[name] = {"ms": round(ms, 4), "tflops": round(fl / ms / 1e9, 1)}
            tot_f += fl * count
            tot_ms += ms * count
            del A, Bw, o, r
        kern_tflops = tot_f / tot_ms / 1e9
        # ---- second half of BASELINE.json's metric: MMU decode tokens/s (configs[2]: 256x256 image -> get_code ->
        #      [mmu][soi] 256 codes [eoi][bos] 16 question ids, greedy 100-token decode, batch 16, KV cache)
        mmu = mmu_local
        if world == 1 and not os.environ.get("SHOWO_BENCH_SKIP_CPU"):
            mmu["cpu_baseline"] = cpu_mmu_sample()
        # ---- CPU baseline: the oracle (port of the reference) on the host cores, bounded sample
        # (rank 0 at N = 1 only: at N > 1 the other ranks are waiting in the closing barrier)
        cpu = None if (world > 1 or os.environ.get("SHOWO_BENCH_SKIP_CPU")) else cpu_reference_sample(steps=1, warmup=1, quiet=True)
        clocks = sampler.summary()
        out = {
            "metric": METRIC, "value": round(value, 3), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": max(args.warmup, 3), "ms_per_step": round(ms_dev / args.steps, 3), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
            "config": {"workload": "showo_demo.yaml t2i 256x256, 18 denoise steps, CFG 5, batch 8 per GPU "
                                   "(t2i_generate + MAGVIT-v2 decode_code + uint8), random-init Phi-1.5 (1.45 B params)",
                       "global_batch": world * B_PER_GPU, "seq_len": L_SEQ, "timesteps": T_STEPS, "guidance": CFG_W,
                       "parallelism": f"dp{world}", "l2": "weights 2.9 GB bf16 streamed every step >> 126 MB L2 (no flush needed)"},
            "e2e": {"value": round(e2e_value, 3), "unit": UNIT, "h2d_bytes_per_step": int(2 * cond_h.numel() * 8),
                    "d2h_bytes_per_step": int(imgs_pin.numel()), "ms_per_step": round(ms_e2e / args.steps, 3), "host_phases_ms": host_phases},
            "gpu_launches": int(launches * args.steps),
            "clocks": clocks,
            "roofline": {"bound": "tensor", "achieved": round(kern_tflops, 1), "peak": peaks["bf16_burst"], "unit": "TFLOP/s",
                         "frac": round(kern_tflops / peaks["bf16_burst"], 4),
                         "job_frac": round((F_IMG + F_DEC) * value / world / 1e12 / peaks["bf16_sustained"], 4),
                         "traffic": ncu_traffic(),
                         "kernel": "gemm_tcgen05_kernel (FLOP-weighted over the 24x2 layer GEMMs + image-vocab head of one "
                                   "denoise step, each shape timed alone with CUDA events)", "peak_source": peaks["source"],
                         "per_shape": per_shape},
            "roofline_job": {"algorithmic_tflop_per_image": round((F_IMG + F_DEC) / 1e12, 3),
                             "achieved": round((F_IMG + F_DEC) * value / world / 1e12, 1), "peak": peaks["bf16_sustained"],
                             "unit": "TFLOP/s per GPU", "frac": round((F_IMG + F_DEC) * value / world / 1e12 / peaks["bf16_sustained"], 4)},
            "cpu_baseline": cpu,
            "secondary": mmu,
            "secondary_t2i512": t512,
            "secondary_train": train,
        }
        print(json.dumps(out), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return out


def t2i512_bench(torch, dist, model, vq, dev, world, rank, warm=1, steps=2):
    """BASELINE.json configs[3]: showo_demo_512x512.yaml t2i, N = 1024 image tokens (L = 1155), 18 steps, CFG 5, 8 images per GPU
    (batch 64 over 8 GPUs), decode_code -> uint8 [8,512,512,3], NCCL all-gather of the images for N > 1.  Device-resident ids."""
    N5, L5, B5 = 1024, P_TXT + 1 + 1024 + 1, B_PER_GPU
    g = torch.Generator().manual_seed(4321 + rank)
    PAD, SOI, EOI, T2I, BOS = 50295, 50296, 50297, 50300, 50256
    cond = torch.full((B5, L5), PAD, dtype=torch.int64)
    unc = torch.full((B5, L5), PAD, dtype=torch.int64)
    descs_c, descs_u = [], []
    for b in range(B5):
        n = int(torch.randint(8, 65, (1,), generator=g))
        row = torch.cat([torch.tensor([T2I, BOS]), torch.randint(0, 50257, (n,), generator=g), torch.tensor([BOS])])
        cond[b, P_TXT - row.numel():P_TXT] = row
        unc[b, P_TXT - 3:P_TXT] = torch.tensor([T2I, BOS, BOS])
        for r in (cond, unc):
            r[b, P_TXT] = SOI
            r[b, P_TXT + 1:P_TXT + 1 + N5] = V - 1
            r[b, P_TXT + 1 + N5] = EOI
        descs_c.append((P_TXT - row.numel(), P_TXT, L5, 0, 0))
        descs_u.append((P_TXT - 3, P_TXT, L5, 0, 0))
    descs = descs_c + descs_u
    cfg5 = NS(model=NS(showo=NS(num_vq_tokens=N5, num_new_special_tokens=10, llm_vocab_size=50295)),
              dataset=NS(preprocessing=NS(max_seq_length=P_TXT - 1)))
    cond_d0, unc_d = cond.to(dev), unc.to(dev)
    ids_d = torch.empty_like(cond_d0)
    gather = torch.empty(world * B5, 512, 512, 3, dtype=torch.uint8, device=dev) if world > 1 else None

    def step():
        ids_d.copy_(cond_d0)
        codes = model.t2i_generate(ids_d, unc_d, descs, guidance_scale=CFG_W, timesteps=T_STEPS, config=cfg5)
        imgs = vq.decode_code_uint8(torch.clamp(codes, 0, CODEBOOK - 1), shape=(32, 32))
        if world > 1:
            dist.all_gather_into_tensor(gather, imgs)
        return imgs
    for _ in range(warm):
        step()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        imgs = step()
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item())
    assert tuple(imgs.shape) == (B5, 512, 512, 3)
    f_img = T_STEPS * 2 * ((N5 + 2) * (G_TOK + A_PAIR * L5) + N5 * 2 * D * CODEBOOK) + 2 * P_TXT * (G_TOK + A_PAIR * P_TXT / 2) + 1205e9
    value = world * B5 * steps / (ms / 1e3)
    peaks = measured_peaks()
    return {"metric": "t2i_512x512_images_per_sec_18steps_cfg5", "value": round(value, 3), "unit": UNIT, "n_gpus": world,
            "ms_per_step": round(ms / steps, 2), "steps": steps, "warmup": warm,
            "config": {"workload": "showo_demo_512x512.yaml t2i 512x512 (N=1024, L=1155), 18 steps, CFG 5, 8 images per GPU, "
                                   "t2i_generate + decode_code + uint8 (+ all-gather)", "global_batch": world * B5, "seq_len": L5},
            "roofline": {"bound": "tensor", "achieved": round(f_img * value / world / 1e12, 1), "peak": peaks["bf16_sustained"],
                         "unit": "TFLOP/s per GPU", "frac": round(f_img * value / world / 1e12 / peaks["bf16_sustained"], 4),
                         "algorithmic_tflop_per_image": round(f_img / 1e12, 2), "kernel": "whole job (SURVEY 8d F_img at N=1024 + decode)"}}



class _BenchTokenizer:
    """id layout of the Show-o tokenizer (phi-1.5 vocabulary + [PAD] + the nine task / span tokens); tokenisation itself is host work
    outside the hot path, the bench feeds synthetic caption ids"""
    bos_token_id = eos_token_id = 50256
    pad_token_id = 50295
    _ids = {"[PAD]": 50295, "<|soi|>": 50296, "<|eoi|>": 50297, "<|sov|>": 50298, "<|eov|>": 50299, "<|t2i|>": 50300,
            "<|mmu|>": 50301, "<|t2v|>": 50302, "<|v2v|>": 50303, "<|lvg|>": 50304}

    def add_special_tokens(self, d):
        return 0

    def add_tokens(self, t):
        return 0

    def convert_tokens_to_ids(self, t):
        return [self._ids[x] for x in t] if isinstance(t, (list, tuple)) else self._ids[t]

    def __len__(self):
        return 50305


def train_step_bench(torch, dist, model, dev, world, rank, warm=1, steps=2):
    """BASELINE.json configs[4]: showo_demo_w_clip_vit_512x512.yaml mixed t2i + lm + mmu training step, forward / backward in bf16
    (fp32 master gradients), per-GPU micro-batch 8 rows of L = 1155 (3 t2i + 1 lm + 4 mmu-vit, SURVEY 8d config 5), data parallel:
    the t2i rows come from the device-side producer (showo_t2i_train_prep); the mmu rows are [mmu, 28 system ids, soi] || 576 visual
    positions || [eoi, 548 text ids] whose visual positions carry mm_projector(N(0,1) [4, 576, 1024]) (the CLIP tower is frozen and
    excluded, its features are synthetic) -- handed to the engine as the mixed ids / embeddings input; the backward returns the
    gradient of those positions and showo_mm_projector_backward turns it into the projector's gradients.  The fp32 gradients (5.8 GB +
    the projector's 25 MB) are all-reduced per layer on a side stream while the earlier layers' backward runs; the step ends with the
    engine's AdamW (showo_adamw_step: fp32 masters and moments, decay on non-bias parameters like training/train.py:211-236, projector
    included) which also rewrites the bf16 working weights."""
    from showo_b200 import train_inputs as TI
    L5, N5, B_T2I, B_LM, B_MMU = 1155, 1024, 3, 1, 4
    SYS, NVIS = 28, 576
    V0 = 1 + SYS + 1                                             # first visual position
    g = torch.Generator().manual_seed(777 + rank)
    up = TI.UniversalPrompting(_BenchTokenizer(), max_text_len=P_TXT - 1, ignore_id=-100, cond_dropout_prob=0.1)

    class _Cfg(dict):
        __getattr__ = dict.get
    cfg = _Cfg(training=_Cfg(min_masking_rate=0.0, noise_type="mask"))
    codes = (torch.randint(0, CODEBOOK, (B_T2I, N5), generator=g) + 50305).to(dev)
    texts = [torch.randint(0, 50256, (int(torch.randint(8, 65, (1,), generator=g)),), generator=g).tolist() for _ in range(B_T2I)]
    lm_ids = torch.randint(0, 50257, (B_LM, L5), generator=g).to(dev)
    mmu_ids = torch.randint(0, 50257, (B_MMU, L5), generator=g)
    mmu_lab = torch.full((B_MMU, L5), -100, dtype=torch.int64)
    mmu_lab[:, L5 - 548:] = mmu_ids[:, L5 - 548:]
    mmu_ids[:, V0:V0 + NVIS] = -1                                # visual positions: their vectors come from the projector
    mmu_ids, mmu_lab = mmu_ids.to(dev), mmu_lab.to(dev)
    feats = torch.randn(B_MMU, NVIS, 1024, generator=g).to(dev)  # synthetic CLIP-ViT features (SURVEY 8d config 5)
    B = B_T2I + B_LM + B_MMU
    emb_full = torch.zeros(B, L5, D, device=dev)                 # only the ids < 0 positions are read
    vis_rows = (slice(B_T2I + B_LM, B), slice(V0, V0 + NVIS))
    loss_w = torch.tensor([1.0, 0.1, 1.0], device=dev)          # training.t2i_coeff / lm_coeff / mmu_coeff of the yaml
    comm = torch.cuda.Stream(dev) if world > 1 else None
    # optimizer state in the engine (fp32 masters + Adam moments): enable, then hand the weights over again so that their fp32 values are kept
    from showo_b200 import _lib
    lib = _lib.require_gpu()
    model.enable_optimizer()
    gp = torch.Generator(device=dev).manual_seed(4)
    proj = {"mm_projector.0.weight": torch.randn(2048, 1024, device=dev, generator=gp) * 0.02, "mm_projector.0.bias": torch.zeros(2048, device=dev),
            "mm_projector.2.weight": torch.randn(2048, 2048, device=dev, generator=gp) * 0.02, "mm_projector.2.bias": torch.zeros(2048, device=dev)}
    for name, t in gpu_random_weights(torch, dev, seed=0):
        _lib.check(lib.showo_load_weight(model._engine, name.encode(), _lib.ptr(t), t.numel(), 1), f"load {name}")
    for name, t in proj.items():
        _lib.check(lib.showo_load_weight(model._engine, name.encode(), _lib.ptr(t), t.numel(), 1), f"load {name}")
    _lib.check(lib.showo_weights_complete(model._engine), "weights_complete")
    model._streamed = True

    def step():
        torch.manual_seed(1000 + rank)
        ids_t2i, lab_t2i, _, descs_t2i = up.t2i_train_rows(texts, codes, V - 1, cfg, showo_b200_cosine())
        ids = torch.cat([ids_t2i, lm_ids, mmu_ids])
        labels = torch.cat([lab_t2i, lm_ids, mmu_lab])
        descs = [tuple(r) for r in descs_t2i.tolist()] + [(0, 0, 0, 0, 0)] * B_LM + [(0, 0, 0, V0, V0 + NVIS)] * B_MMU
        terms = model._loss_terms(ids.shape[0], L5, B_T2I, B_LM, B_MMU, P_TXT - 1)
        emb_full[vis_rows] = model._project(feats)               # model.mm_projector(images_embeddings), train_w_clip_vit.py:599-601
        _, losses = model.train_forward(ids, emb_full, descs, labels, terms, want_logits=False)
        if world > 1:
            done = model.backward_overlapped(loss_w, comm_stream=comm, input_grad_like=emb_full, projector_rows=vis_rows)
            torch.cuda.current_stream().wait_event(done)
        else:
            demb = model.backward(loss_w, want_input_grad_like=emb_full)
            model.mm_projector_backward(demb[vis_rows])
        model.adamw_step(lr=1e-4, betas=(0.9, 0.999), eps=1e-8, weight_decay=0.01)      # optimizer.params of the yaml
        return losses
    for _ in range(warm):
        step()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        losses = step()
    e1.record()
    torch.cuda.synchronize()
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = float(ms.item()) / steps
    f_step = 3 * B * L5 * (G_TOK + A_PAIR * L5 + 2 * D * V)
    peaks = measured_peaks()
    return {"metric": "train_step_tokens_per_sec_mixed_t2i_lm_mmu_L1155_fwd_bwd_adamw", "value": round(world * B * L5 / ms * 1e3, 1), "unit": "tokens/s",
            "n_gpus": world, "ms_per_step": round(ms, 2), "steps": steps, "warmup": warm,
            "config": {"workload": "showo_demo_w_clip_vit_512x512.yaml geometry: forward + backward of 8 rows x L=1155 per GPU (3 t2i from the "
                                   "device-side producer + 1 lm + 4 mmu-vit whose 576 visual positions are mm_projector(synthetic CLIP "
                                   "features), projector forward + backward included), bf16 operands / fp32 gradients, per-layer gradient "
                                   "all-reduce (fp32, 5.8 GB) overlapped with backward for N > 1, then the engine-side AdamW step (fp32 "
                                   "masters + moments, backbone + projector)",
                       "global_batch": world * B, "seq_len": L5},
            "losses": [round(float(x), 4) for x in losses[:, 0].tolist()],
            "roofline": {"bound": "tensor", "achieved": round(f_step / ms / 1e9, 1), "peak": peaks["bf16_sustained"], "unit": "TFLOP/s per GPU",
                         "frac": round(f_step / ms / 1e9 / peaks["bf16_sustained"], 4), "algorithmic_tflop_per_step": round(f_step / 1e12, 2),
                         "kernel": "whole step (3 x forward FLOPs of the backbone, SURVEY 8d config 5; the projector's 0.09 TFLOP are not counted)"}}


def showo_b200_cosine():
    from showo_b200 import cosine_schedule
    return cosine_schedule

def cpu_mmu_sample(n_tokens=2):
    """The reference's MMU path on the host cores (modeling_showo.py:183-240: B = 1, NO KV cache, the whole sequence is
    re-run for every new token; 16 prompts are processed one after the other): bounded sample = `n_tokens` greedy tokens of ONE
    L0 = 276 row through the oracle port; tokens/s = 1 / (seconds per token), linear extrapolation to 16 x 100 tokens."""
    import torch
    from oracle import showo_oracle as O
    cores = host_cores()
    torch.set_num_threads(cores)
    dims = O.PhiDims()
    W = cpu_random_weights(torch, dims)
    voc = O.ShowoVocab()
    g = torch.Generator().manual_seed(5)
    codes = torch.randint(0, CODEBOOK, (1, N_TOK), generator=g)
    row = O.make_mmu_prompts(1, voc, codes, q_len=16, seed=6)
    mk = O.create_attention_mask_for_mmu(row)
    t0 = time.perf_counter()
    with torch.no_grad():
        O.mmu_generate(W, dims, row, mk, max_new_tokens=n_tokens, top_k=1)
    dt = (time.perf_counter() - t0) / n_tokens
    return {"value": round(1.0 / dt, 4), "unit": "tokens/s", "cores": cores, "kind": "port",
            "sample": f"{n_tokens} greedy tokens of 1 row (L0=276, full re-forward per token, fp32) = {dt:.2f} s per token; "
                      f"the reference decodes its 16 prompts sequentially, so tokens/s = 1 / t_token (extrapolated to 16 x 100 tokens)"}


def mmu_decode_bench(torch, model, vq, dev, peaks, B=16, q_len=16, n_new=100, seed=5):
    """MMU decode tokens/s on rank 0 (SURVEY.md section 8d config 3).  decode time = t(100 tokens) - t(1 token), i.e. 99
    KV-cached decode steps of 16 sequences; prefill and get_code are reported separately."""
    g = torch.Generator().manual_seed(seed)
    pixels = (torch.rand(B, 3, 256, 256, generator=g) * 2 - 1).to(dev)

    def ev():
        return torch.cuda.Event(enable_timing=True)
    vq.get_code(pixels)
    e0, e1 = ev(), ev()
    e0.record(); codes = vq.get_code(pixels); e1.record(); torch.cuda.synchronize()
    t_code = e0.elapsed_time(e1)
    MMU, SOI, EOI, BOS = 50301, 50296, 50297, 50256
    q = torch.randint(0, 50257, (B, q_len), generator=g).to(dev)
    ids = torch.cat([torch.full((B, 1), MMU, device=dev), torch.full((B, 1), SOI, device=dev), codes + 50305,
                     torch.full((B, 1), EOI, device=dev), torch.full((B, 1), BOS, device=dev), q], 1).contiguous()
    L0 = ids.shape[1]
    descs = [(0, 0, 0, 0, 259)] * B              # create_attention_mask_for_mmu: columns <= eoi (258) visible to all rows

    def run(n):
        e0, e1 = ev(), ev()
        e0.record()
        toks, _ = model.mmu_generate_batched(ids, attention_mask=descs, max_new_tokens=n, top_k=1)
        e1.record(); torch.cuda.synchronize()
        return e0.elapsed_time(e1), toks
    run(n_new)
    t1 = min(run(1)[0] for _ in range(3))
    tn = min(run(n_new)[0] for _ in range(3))
    steps = n_new - 1
    ms_step = (tn - t1) / steps
    tok_s = B * 1000.0 / ms_step
    w_bytes = (NL * (4 * D * D + 2 * D * F) + D * V) * 2.0                     # bf16 weights streamed per step
    kv_bytes = B * NL * 2 * D * 2.0 * (L0 + n_new / 2.0)                      # K and V^T rows read per step (mean length)
    gbs = (w_bytes + kv_bytes) / (ms_step * 1e-3) / 1e9
    return {"metric": "mmu_decode_tokens_per_sec_b16_greedy100", "value": round(tok_s, 1), "unit": "tokens/s",
            "ms_per_decode_step": round(ms_step, 4), "prefill_ms": round(t1, 3), "get_code_ms": round(t_code, 3),
            "config": {"workload": "showo_demo.yaml MMU, 256x256 input, L0=%d, greedy %d new tokens, batch %d, KV cache" % (L0, n_new, B)},
            "roofline": {"bound": "hbm", "achieved": round(gbs, 1), "peak": peaks["hbm"], "unit": "GB/s",
                         "frac": round(gbs / peaks["hbm"], 4), "traffic": None,
                         "bytes_per_step": int(w_bytes + kv_bytes), "kernel": "whole decode step (weights + KV streamed once)"}}


# ======================================================================================================= reference arm (CPU)
def host_cores():
    """threads the process can actually use: the affinity mask, capped by the container's CPU quota (cgroup v2 cpu.max) -- on the
    round-1 GPU box the mask showed 128 CPUs but the quota was 16 cores, and 128 threads ran 3x slower than 16."""
    try:
        cores = len(os.sched_getaffinity(0))
    except Exception:
        cores = os.cpu_count() or 1
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            cores = max(1, min(cores, int(math.ceil(int(quota) / int(period)))))
    except Exception:
        pass
    return cores


def cpu_random_weights(torch, dims, seed=0):
    """Random-init state_dict with the initialisation the tests use (N(0, 0.02) matrices, zero biases, LayerNorm 1 / 0)."""
    g = torch.Generator().manual_seed(seed)
    W = {}
    Dd, Ff, Vv = dims.hidden, dims.ffn, dims.vocab_size
    W["showo.model.embed_tokens.weight"] = torch.randn(Vv, Dd, generator=g) * 0.02
    for i in range(dims.n_layers):
        p = f"showo.model.layers.{i}."
        for n, (o, ii) in {"self_attn.q_proj": (Dd, Dd), "self_attn.k_proj": (Dd, Dd), "self_attn.v_proj": (Dd, Dd),
                           "self_attn.dense": (Dd, Dd), "mlp.fc1": (Ff, Dd), "mlp.fc2": (Dd, Ff)}.items():
            W[p + n + ".weight"] = torch.randn(o, ii, generator=g) * 0.02
            W[p + n + ".bias"] = torch.zeros(o)
        for n, c in {"input_layernorm": Dd, "self_attn.q_layernorm": 64, "self_attn.k_layernorm": 64}.items():
            W[p + n + ".weight"] = torch.ones(c)
            W[p + n + ".bias"] = torch.zeros(c)
    W["showo.model.final_layernorm.weight"] = torch.ones(Dd)
    W["showo.model.final_layernorm.bias"] = torch.zeros(Dd)
    W["showo.lm_head.weight"] = torch.randn(Vv, Dd, generator=g) * 0.02
    W["showo.lm_head.bias"] = torch.zeros(Vv)
    return W


def cpu_reference_sample(steps: int, warmup: int, quiet: bool = False, full: bool = False):
    """Times the oracle (CPU port of the reference's fp32 path; the Python reference itself cannot travel to the GPU box)
    on the host cores.  Bounded mode: one sample = ONE of the 18 denoise-step forwards of ONE image as the reference executes
    it (cond + uncond rows, L = 387, full 58498-way head), MAGVIT decode of one image timed once, images/s EXTRAPOLATED as
    1 / (18 * t_step + t_decode).  full=True: one COMPLETE image (t2i_generate: 18 forwards + sampler, then decode_code)."""
    import torch
    from oracle import magvit_oracle as MO
    from oracle import showo_oracle as O
    cores = host_cores()
    torch.set_num_threads(cores)
    dims = O.PhiDims()
    W = cpu_random_weights(torch, dims)
    voc = O.ShowoVocab()
    cond, unc = O.make_t2i_prompts(1, voc, seed=1234)
    ids = torch.cat([cond, unc])
    mask = O.create_attention_mask_predict_next(ids)
    g = torch.Generator().manual_seed(0)
    Wm = MO.make_magvit_weights(1)
    if full:
        with torch.no_grad():
            t0 = time.perf_counter()
            codes = O.t2i_generate(W, dims, voc, cond.clone(), unc.clone(), mask, guidance_scale=CFG_W, timesteps=T_STEPS, generator=g)
            t_gen = time.perf_counter() - t0
            t0 = time.perf_counter()
            MO.decode_code(torch.clamp(codes, 0, CODEBOOK - 1), Wm)
            t_dec = time.perf_counter() - t0
        return {"value": round(1.0 / (t_gen + t_dec), 6), "unit": UNIT, "cores": cores, "kind": "port",
                "sample": f"1 complete image: t2i_generate (18 denoise steps, CFG 5, fp32, sampler included) = {t_gen:.1f} s + "
                          f"decode_code = {t_dec:.2f} s; no extrapolation",
                "t_step_s": round(t_gen / T_STEPS, 3), "t_decode_s": round(t_dec, 3), "extrapolated": False}
    times = []
    with torch.no_grad():
        for it in range(warmup + steps):
            t0 = time.perf_counter()
            logits = O.showo_logits(W, dims, input_ids=ids, add_mask=mask)
            lg = (1 + CFG_W) * logits[:1] - CFG_W * logits[1:]
            _ = lg[:, -(N_TOK + 1):-1, voc.image_offset:-1].softmax(-1)
            dt = time.perf_counter() - t0
            if it >= warmup:
                times.append(dt)
        codes = torch.randint(0, CODEBOOK, (1, N_TOK), generator=g)
        t0 = time.perf_counter()
        MO.decode_code(codes, Wm)
        t_dec = time.perf_counter() - t0
    t_step = sum(times) / len(times)
    value = 1.0 / (T_STEPS * t_step + t_dec)
    return {"value": round(value, 6), "unit": UNIT, "cores": cores, "kind": "port",
            "sample": f"{len(times)} x (1 of 18 denoise-step forwards of 1 image: cond+uncond rows, L=387, fp32, full head) "
                      f"= {t_step:.2f} s each + 1 MAGVIT decode = {t_dec:.2f} s; images/s EXTRAPOLATED = 1/(18*t_step + t_decode)",
            "t_step_s": round(t_step, 3), "t_decode_s": round(t_dec, 3), "extrapolated": True}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # --steps >= 18: one COMPLETE 18-step image (about a minute on 16 cores); fewer: bounded sample, extrapolated
    full = args.steps >= T_STEPS
    cpu = cpu_reference_sample(steps=max(1, args.steps), warmup=min(args.warmup, 1), full=full)
    t_step = cpu["t_step_s"]
    how = ("one complete image (18 steps + sampler + decode)" if full
           else "bounded sample, EXTRAPOLATED: each step = 1 of 18 denoise-step forwards of 1 image")
    out = {"impl": "reference", "metric": METRIC, "value": cpu["value"], "unit": UNIT, "n_gpus": args.gpus,
           "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(1e3 * t_step, 1), "higher_is_better": True,
           "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
           "config": {"workload": "showo_demo.yaml t2i 256x256, 18 denoise steps, CFG 5 -- reference fp32 CPU path (oracle port), " + how,
                      "parallelism": "cpu"},
           "cpu_baseline": cpu,
           "e2e": {"value": cpu["value"], "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out), flush=True)


if __name__ == "__main__":
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--dump-outputs", metavar="DIR", help="save the last timed step's outputs as DIR/<name>.npy (float32)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and a.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    if a.impl == "reference":
        run_reference(a)
    else:
        run_ours(a)
