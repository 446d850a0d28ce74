#!/usr/bin/env python
"""bench.py -- images/sec of the VisualCloze denoising hot path on B200 (BASELINE.json metric).

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload B|A|Bp|D|E] [--dump-outputs DIR]

One "step" = one image of the workload: the flow-matching Euler loop over the FLUX-DiT (30 time points = 29 model
evaluations for the 384 grid 2x3 layout, SURVEY.md section 8) plus the VAE decode of the query row, on synthetic
inputs of the reference's shapes with random-init weights of the reference's geometry (no checkpoints offline).

  value   images/sec with the inputs already resident in HBM (device-timed, CUDA events, max over ranks)
  e2e     the same through the public API with HOST (pinned) buffers: H2D of the step's inputs and D2H of the
          result inside the timed region
  roofline / roofline_attention   achieved TFLOP/s of the GEMM / attention kernels (algorithmic FLOPs over the sum of
          their launch durations, CUDA events around every launch of one instrumented image) vs the measured peak
  cpu_baseline   the CPU oracle port (the reference's algorithm, un-merged LoRA, bf16 autocast semantics) timed on
          the host cores on a bounded sample (1 double + 1 single block at full width and full token count),
          extrapolated to images/sec -- a reported baseline, not the target.

`--dump-outputs DIR` writes what the last timed step returned -- the decoded query-row image tile, uint8 values, gathered over
the replicas -- to DIR/query_row_image.npy as float32.  Inputs and weights come from fixed seeds, so two builds run with the
same arguments can be compared output for output.

`--impl reference` times the reference arm: the UNMODIFIED reference modules of oracle/_ref (DoubleStreamBlock /
SingleStreamBlock of models/modules/layers.py with LoRA r=256, bf16 autocast, attention through SDPA because flash-attn is
CUDA-only) on the host cores -- `cpu_baseline.kind` "reference"; the restated oracle ("port") only if oracle/_ref is absent.

With N > 1 GPUs the default line is replica throughput (weak scaling, the contract's line); after it the same process group
runs the sequence-parallel single-image mode for a few images and reports it under `extra.sp` (strong scaling, one image over
the N GPUs), so the driver's scaling record also carries the NVLink path.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

import torch

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

BF16 = torch.bfloat16
WORKLOADS = {  # key: (grid_h, grid_w, res, num_steps, do_shift, strength, description)
    "A": (1, 1, 384, 4, True, None, "single 384x384 1x1 grid, 4 Euler time points (3 NFE)"),
    "B": (2, 3, 384, 30, True, None, "384 grid 2x3 in-context, 30 Euler time points (29 NFE), batch 1 per GPU"),
    "Bp": (3, 3, 384, 30, True, None, "384 grid 3x3 (2 demos + query), 30 time points (29 NFE)"),
    "C": (2, 3, 512, 30, True, None, "512 grid 2x3, 30 time points (29 NFE), batch 1 per GPU"),
    "D": (3, 4, 384, 30, True, None, "384 grid 3x4 multi-task layout, 30 time points (29 NFE)"),
    "E": (1, 1, 1024, 20, False, 0.4, "SDEdit upsampling 1024^2, 20 time points (19 NFE), strength 0.4"),
}


def peaks():
    p = os.path.join(REPO, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d["hbm_gbs"], tf_burst=d["bf16_tflops"], tf=d["bf16_tflops_sustained"], src="measured")
    return dict(hbm=6650.0, tf_burst=1590.0, tf=1400.0, src="fallback")


# ------------------------------------------------------------------------------------------------------
# synthetic inputs (SURVEY.md 8d): generated on CPU from a seeded generator, identical bits on every rank/run
# ------------------------------------------------------------------------------------------------------
def make_inputs(workload: str, seed: int):
    gh, gw, res, *_ = WORKLOADS[workload]
    g = torch.Generator().manual_seed(seed)
    h, w = res // 16, gw * res // 16
    ids = []
    for j in range(gh):
        t = torch.zeros(h, w, 3)
        t[..., 0] = j + 1
        t[..., 1] += torch.arange(h)[:, None]
        t[..., 2] += torch.arange(w)[None, :]
        ids.append(t.reshape(-1, 3))
    img_ids = torch.cat(ids)[None]
    Li, Lt = img_ids.shape[1], 512
    x = torch.randn(1, Li, 64, generator=g).to(BF16)                       # packed noise rows (visualcloze.py:394-403)
    fill_cond = torch.randn(1, Li, 64, generator=g).to(BF16)
    fill_mask = torch.zeros(1, gh, h, gw, res // 16, 256)
    fill_mask[:, -1, :, -1] = 1.0                                            # target = last cell of the query row
    cond = torch.cat((fill_cond, fill_mask.reshape(1, Li, 256).to(BF16)), dim=-1)
    kw = dict(txt=(0.1 * torch.randn(1, Lt, 4096, generator=g)).to(BF16), txt_ids=torch.zeros(1, Lt, 3),
              txt_mask=torch.ones(1, Lt, dtype=torch.int32), y=torch.randn(1, 768, generator=g).to(BF16),
              img_ids=img_ids, img_mask=torch.ones(1, Li, dtype=torch.int32), cond=cond,
              guidance=torch.full((1,), 30.0, dtype=BF16))
    return x, kw, Li, Lt


def flops_per_image(Li, Lt, nfe, H=3072, mlp=12288, heads=24, in_ch=384, out_ch=64, depth=19, depth_single=38):
    """Algorithmic FLOPs of the launched GEMMs / attention calls (merged LoRA), SURVEY.md 8d."""
    L = Li + Lt
    per_eval = 2 * Li * in_ch * H + depth * 24 * L * H * H + depth_single * 24 * L * H * H + 2 * Li * H * out_ch
    prep = 2 * Lt * 4096 * H + 2 * nfe * H * H * (depth * 12 + depth_single * 3 + 2) + 2 * nfe * (256 * H + H * H) \
        + 2 * (256 * H + H * H) + 2 * (768 * H + H * H)
    attn = (depth + depth_single) * 4 * L * L * H
    return nfe * per_eval + prep, nfe * attn


# ------------------------------------------------------------------------------------------------------
# clocks during the timed region
# ------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index: int):
        self.rows = []
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200",
                                          "-i", str(index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:  # noqa: BLE001
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        self.th.join(timeout=2)
        sm = sorted(float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit())
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(len(r) > 3 + i and r[3 + i].lower().startswith("active") for r in self.rows)]
        pw = [float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "power_w_max": max(pw) if pw else None, "samples": len(self.rows)}


# ------------------------------------------------------------------------------------------------------
# CPU port of the reference (oracle) on a bounded sample
# ------------------------------------------------------------------------------------------------------
def host_threads() -> int:
    """Threads this process may really use: the affinity mask, capped by the cgroup CPU quota (a container on a 128-thread
    host often owns far fewer; asking torch for all 128 then oversubscribes and slows the CPU arm several-fold)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()
        if quota != "max":
            n = max(1, min(n, math.ceil(int(quota) / int(period))))
    except (OSError, ValueError):
        pass
    return n


def cpu_reference_sample(workload: str, threads=None):
    """Times 1 DoubleStreamBlock + 1 SingleStreamBlock of the reference at full width on the workload's token count and
    extrapolates to one image (x 19 / x 38 blocks x NFE; embedders, final layer and the VAE decode -- together < 0.5 % of the
    image's FLOPs, SURVEY.md 8 -- are not in the sample).  Preferred: the UNMODIFIED reference modules from oracle/_ref under
    ``torch.autocast("cpu", bf16)`` (kind "reference"); fallback: the restated oracle (kind "port").

    ``threads`` = None tries host_threads() and its halves down to 1/8 (>= 4), each once after a warm-up pass, and reports the
    FASTEST -- the reference arm gets the thread count that suits it, not a blind os.cpu_count()."""
    import contextlib
    from oracle import flux_oracle as fo
    from oracle import ref_runner as rr
    gh, gw, res, num_steps, *_ = WORKLOADS[workload]
    cfg = fo.FluxConfig(depth=1, depth_single_blocks=1, lora_rank=256)
    H = cfg.hidden_size
    g = torch.Generator().manual_seed(0)
    shapes = fo.param_shapes(cfg)
    p = {}
    for k, shp in shapes.items():
        if k.startswith("double_blocks.") or k.startswith("single_blocks."):
            std = 0.02 if (k.endswith(".bias") or "lora_B" in k) else 1.0 / math.sqrt(shp[-1])
            p[k] = (torch.randn(shp, generator=g) * std).to(BF16) if not k.endswith(".scale") else torch.ones(shp, dtype=BF16)
    Li, Lt = gh * gw * (res // 16) ** 2, 512
    L = Li + Lt
    img = torch.randn(1, Li, H, generator=g).to(BF16)
    txt = torch.randn(1, Lt, H, generator=g).to(BF16)
    vec = torch.randn(1, H, generator=g).to(BF16)
    ids = torch.zeros(1, L, 3)
    ids[0, Lt:, 1] = torch.arange(Li) // 72
    ids[0, Lt:, 2] = torch.arange(Li) % 72
    mask = torch.ones(1, L, dtype=torch.int32)
    kind = "port"
    if rr.available():
        kind = "reference"
        rr.apply_cpu_patches()
        _, ref_layers, _, _ = rr._import()
        from models.modules.lora import replace_linear_with_lora
        dbl = ref_layers.DoubleStreamBlock(H, cfg.num_heads, mlp_ratio=cfg.mlp_ratio, qkv_bias=True)
        sgl = ref_layers.SingleStreamBlock(H, cfg.num_heads, mlp_ratio=cfg.mlp_ratio)
        for blk, pre in ((dbl, "double_blocks.0."), (sgl, "single_blocks.0.")):
            replace_linear_with_lora(blk, max_rank=256, scale=1.0)
            blk.load_state_dict({k[len(pre):]: v for k, v in p.items() if k.startswith(pre)}, strict=True)
            blk.to(BF16).eval().requires_grad_(False)
        pe = ref_layers.EmbedND(dim=128, theta=cfg.theta, axes_dim=list(cfg.axes_dim))(ids)
        ctx = torch.autocast("cpu", dtype=BF16)
    else:
        cos, sin = fo.rope_table(ids, cfg.axes_dim, cfg.theta)
        nm = fo.Numerics("cuda_bf16")
        ctx = contextlib.nullcontext()

    def one_pass():
        with torch.no_grad(), ctx:
            t0 = time.perf_counter()
            if kind == "reference":
                img2, txt2 = dbl(img=img, txt=txt, vec=vec, pe=pe, img_mask=mask[:, Lt:], txt_mask=mask[:, :Lt])
            else:
                img2, txt2 = fo.double_block(p, 0, cfg, img, txt, vec, cos, sin, mask, nm, 1.0)
            t1 = time.perf_counter()
            if kind == "reference":
                sgl(torch.cat((txt2, img2), 1), vec=vec, pe=pe, attn_mask=mask)
            else:
                fo.single_block(p, 0, cfg, torch.cat((txt2, img2), 1), vec, cos, sin, mask, nm, 1.0)
            t2 = time.perf_counter()
        return t1 - t0, t2 - t1

    nfe = num_steps - 1
    if threads is None:
        top = host_threads()
        cands = sorted({max(4, top >> s) if top >= 4 else top for s in range(4)}, reverse=True)
    else:
        cands = [int(threads)]
    tried, best = {}, None
    for n in cands:
        torch.set_num_threads(n)
        one_pass()                                   # warm-up at this thread count (thread pool, allocator, oneDNN primitives)
        td, ts = one_pass()
        sec = nfe * (19 * td + 38 * ts)
        tried[n] = round(sec, 1)
        if best is None or sec < best[0]:
            best = (sec, n, td, ts)
    sec, n, td, ts = best
    return 1.0 / sec, dict(double_block_s=td, single_block_s=ts, tokens=L, kind=kind, threads=n, host_threads=host_threads(),
                           tried_threads_sec_per_image=tried)


def cpu_sample_text(info: dict, nfe: int) -> str:
    what = ("UNMODIFIED reference modules from oracle/_ref, autocast cpu bf16, SDPA attention" if info["kind"] == "reference"
            else "restated oracle")
    return (f"1 DoubleStreamBlock + 1 SingleStreamBlock ({what}, un-merged LoRA r=256) at hidden 3072 on {info['tokens']} tokens: "
            f"{info['double_block_s']:.2f}s + {info['single_block_s']:.2f}s on {info['threads']} threads (fastest of the thread counts tried, "
            f"s/image: {info['tried_threads_sec_per_image']}; the process may use {info['host_threads']}), extrapolated x(19,38) blocks x {nfe} "
            "evaluations; embedders / final layer / VAE decode (< 0.5 % of the image's FLOPs) not in the sample; each timed once after a warm-up pass")


# ------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="B", choices=list(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's output to DIR/<name>.npy (float32)")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp8", "fp8_all"],
                    help="bf16 = the reference's numerics (the headline); fp8 = opt-in e4m3 projections for the LayerNorm-fed Linears "
                         "(a separate line with its own tolerance contract, never the headline)")
    ap.add_argument("--mode", default="replicas", choices=["replicas", "sp"],
                    help="N>1: 'replicas' = one image per GPU (throughput, weak scaling; the default and the contract's line); "
                         "'sp' = ONE image sharded by token rows over the N GPUs (latency, strong scaling; SURVEY.md 8f-2)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    gh, gw, res, num_steps, do_shift, strength, desc = WORKLOADS[args.workload]
    nfe = num_steps - 1
    config = {"workload": f"{args.workload}: {desc}", "grid": f"{gh}x{gw}", "resolution": res, "num_steps": num_steps,
              "nfe": nfe, "batch_per_gpu": 1, "parallelism": f"replicas x{world} (no per-step collective; all_gather of result tiles)",
              "lora": "merged r=256", "l2": "per-evaluation working set is 24 GB of weights >> 126 MB L2 (no flush needed)"}

    sp_mode = args.mode == "sp" and world > 1
    if sp_mode:
        config["parallelism"] = (f"sequence-parallel x{world}: one image, token rows sharded over the GPUs, attention all-to-alls fused "
                                 "into the QKV-GEMM / attention epilogues as NVLink peer stores (no NCCL on the per-step path)")
        config["batch_per_gpu"] = f"1/{world}"
    if args.impl == "reference":
        if rank != 0:
            return
        # one bounded sample per group (the result is an extrapolation of two block timings; repeating it --steps times would
        # only multiply the host time): per thread count one warm-up pass and ONE timed pass, the fastest count is reported
        v, info = cpu_reference_sample(args.workload)
        cores = info["threads"]
        sample = cpu_sample_text(info, nfe)
        print(json.dumps({"impl": "reference", "metric": "images/sec", "value": v, "unit": "images/s", "n_gpus": args.gpus,
                          "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1000.0 / v, "higher_is_better": True,
                          "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": config,
                          "sample_repeats": 1,
                          "cpu_baseline": {"value": v, "unit": "images/s", "cores": cores, "kind": info["kind"], "sample": sample},
                          "e2e": {"value": v, "unit": "images/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    # ---------------- our arm ----------------
    if not torch.cuda.is_available():
        raise SystemExit("bench.py --impl ours needs a B200: the hot path has no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        import datetime
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(minutes=5))   # a stuck rank ends the run, not the lease
    from visualcloze_b200 import _lib, model as M, transport as T
    lib = _lib.lib()
    with torch.device(dev):
        model = M.FluxLoraWrapper(lora_rank=256, params=M.flux_dev_fill_params())
    model.init_synthetic(0)
    if args.precision != "bf16":
        model.set_linear_precision(args.precision)
        config["precision"] = (("fp8: qkv / mlp.0 / linear1 (58 % of the GEMM FLOPs)" if args.precision == "fp8" else
                                "fp8_all: every Linear of the blocks (qkv, proj, mlp.0, mlp.2, linear1, linear2; inputs of the gated-residual ones "
                                "quantised row-wise by quantize_rows_e4m3_kernel, booked under other_ms)") +
                               " on e4m3 operands (tcgen05 kind::f8f6f4, per-row activation and per-channel weight scales); everything else bf16.  "
                               "NOT the reference's numerics: tests/test_fp8_gpu.py")
    model.engine()
    decoder = None
    try:
        from visualcloze_b200 import vae as V
        decoder = V.AutoEncoderDecoder(device=dev).init_synthetic(0)
    except ImportError:
        config["vae_decode"] = "NOT INCLUDED (kernel not built yet): value covers the denoise loop only"
    sampler = T.Sampler(T.create_transport("Linear", "velocity", do_shift=True))
    fn = sampler.sample_ode(sampling_method="euler", num_steps=num_steps, atol=1e-6, rtol=1e-3, reverse=False,
                            do_shift=do_shift, time_shifting_factor=1, strength=strength)
    if sp_mode:
        from visualcloze_b200.parallel import SequenceParallel
        model.enable_sequence_parallel(SequenceParallel(timeout_ms=20000))
    x_h, kw_h, Li, Lt = make_inputs(args.workload, 1234 + (0 if sp_mode else rank))
    pin = lambda t: t.pin_memory()
    x_h, kw_h = pin(x_h), {k: pin(v) for k, v in kw_h.items()}
    x_d, kw_d = x_h.to(dev), {k: v.to(dev) for k, v in kw_h.items()}
    row_tokens = Li // gh

    def finish(latent):
        """query row -> decoded image tile (uint8) -> gathered across replicas"""
        q = latent[:, Li - row_tokens:, :]
        if decoder is not None:
            tile = decoder.decode_packed(q, res // 16, gw * res // 16)
        else:
            tile = q
        if world > 1 and not sp_mode:     # sp: every rank holds the whole latent after the trajectory gather and decodes it
            out = torch.empty((world,) + tuple(tile.shape), dtype=tile.dtype, device=dev)
            dist.all_gather_into_tensor(out, tile.contiguous())
            return out
        return tile

    def step_resident():
        return finish(fn(x_d, model.forward, kw_d)[-1])

    def step_e2e():
        x = x_h.to(dev, non_blocking=True)
        kw = {k: v.to(dev, non_blocking=True) for k, v in kw_h.items()}
        return finish(fn(x, model.forward, kw)[-1]).cpu()

    last = [None]                     # what the most recent timed step returned

    def timed(step, k):
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            last[0] = step()
        e1.record()
        torch.cuda.synchronize()
        ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            dist.barrier()
        return float(ms)

    for _ in range(args.warmup):
        step_resident()
    clocks = ClockSampler(local) if rank == 0 else None
    lib.vcb_reset_launch_count()
    ms = timed(step_resident, args.steps)
    launches = lib.vcb_launch_count()
    clk = clocks.stop() if clocks else None
    if args.dump_outputs and rank == 0:
        import numpy as np
        os.makedirs(args.dump_outputs, exist_ok=True)
        np.save(os.path.join(args.dump_outputs, "query_row_image.npy"), last[0].float().cpu().numpy())
    step_e2e()
    ms_e2e = timed(step_e2e, args.steps)
    h2d = x_h.numel() * x_h.element_size() + sum(v.numel() * v.element_size() for v in kw_h.values())
    d2h_t = finish(fn(x_d, model.forward, kw_d)[-1])
    d2h = d2h_t.numel() * d2h_t.element_size()

    # one instrumented image: CUDA events around every launch, per kernel category and per launch
    eng = model.engine()

    def instrumented():
        lib.vcb_profile_begin()
        step_resident()
        return _lib.profile_end(max_records=20000)

    cat, recs = instrumented()
    variants = eng.softmax_variants()
    # the same image with every block on the exact online-max softmax (what a checkpoint whose QK-norm scales leave the safe
    # range runs; the synthetic scales 1 + 0.1 N(0,1) put every block on the fixed-reference variant)
    eng.use_score_bounds(False)
    step_resident()
    ms_exact = timed(step_resident, 2) / 2
    cat_x, _ = instrumented()
    eng.use_score_bounds(True)

    # ---- sequence-parallel single-image mode on the same process group (strong scaling; N > 1 only) ----
    sp_extra = None
    if world > 1 and not sp_mode and args.precision != "bf16":
        sp_extra = {"skipped": "the sequence-parallel mode runs the bf16 projections only (vcb_flux_sp_attach refuses an fp8 engine)"}
    elif world > 1 and not sp_mode:
        from visualcloze_b200.parallel import SequenceParallel
        try:
            x_s, kw_s, _, _ = make_inputs(args.workload, 1234)              # every rank: the SAME sample
            x_sd, kw_sd = x_s.to(dev), {k: v.to(dev) for k, v in kw_s.items()}
            model.enable_sequence_parallel(SequenceParallel(timeout_ms=20000))

            def step_sp():
                latent = fn(x_sd, model.forward, kw_sd)[-1]
                q = latent[:, Li - row_tokens:, :]
                return decoder.decode_packed(q, res // 16, gw * res // 16) if decoder is not None else q

            step_sp(); step_sp()
            n_sp = 3
            ms_sp = timed(step_sp, n_sp) / n_sp
            lib.vcb_profile_begin()
            step_sp()
            cat_s, _ = _lib.profile_end()
            Lq, Hh = Li + Lt, 3072
            sent = 57 * ((Lq // world) * 3 * Hh * 2 + Lq * (Hh // world) * 2) * (world - 1) / world
            sp_extra = {"ms_per_image": ms_sp, "images_per_s": 1000.0 / ms_sp, "timed_images": n_sp, "scaling": "strong",
                        "gemm_ms": cat_s["gemm"][0], "attention_ms": cat_s["attention"][0], "ln_modulate_ms": cat_s["ln_modulate"][0],
                        "barrier_and_other_ms": cat_s["other"][0], "vae_ms": cat_s["vae_conv3x3"][0] + cat_s["vae_elementwise"][0],
                        "nvlink_bytes_per_eval_per_rank": int(sent),
                        "note": "ONE image, token rows sharded over the GPUs; q/k/v and attention-output all-to-alls are TMA tile stores into "
                                "peer memory from the GEMM / attention epilogues; per-rank kernel times are rank 0's"}
            model.enable_sequence_parallel(None)
        except Exception as e:  # noqa: BLE001  (the replica line must survive a failure of the extra measurement)
            sp_extra = {"error": f"{type(e).__name__}: {e}"[:300]}
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    pk = peaks()
    gemm_fl, attn_fl = flops_per_image(Li, Lt, nfe)
    # AdaLN LayerNorm passes per evaluation: 2 per double block and 1 per single block over all L rows, 1 over the img rows
    ln_bytes = nfe * 4.0 * 3072 * ((2 * 19 + 38) * (Li + Lt) + Li)
    if sp_mode:                       # rank 0's kernels did 1/W of the image's GEMM rows and attention heads
        gemm_fl, attn_fl, ln_bytes = gemm_fl / world, attn_fl / world, ln_bytes / world
    traffic = {}
    import glob
    tps = sorted(glob.glob(os.path.join(REPO, "profiles", "r*_ncu_traffic.json")))   # committed ncu --set full captures, latest round
    if tps:
        traffic = json.load(open(tps[-1]))
        traffic["source"] = os.path.relpath(tps[-1], REPO)
    pms = [cat[k][0] for k in _lib.PROF_CATEGORIES]
    pl = [cat[k][1] for k in _lib.PROF_CATEGORIES]
    # the GEMM category also holds the VAE decoder's 1x1 convolutions / mid-attention GEMMs (M = pixels): split them off by shape
    EPI = {0: "bias", 1: "bias_gelu", 2: "gate_res", 3: "qkv_rmsnorm_rope", 4: "linear1_split", 5: "bias_f32"}
    shapes, conv_fl, conv_ms, vae_gemm_ms, vae_gemm_fl = {}, 0.0, 0.0, 0.0, 0.0
    for r in recs:
        i = list(r.info)
        if r.category == 0:
            fl = 2.0 * i[0] * i[1] * i[2]
            if (i[3] >> 24) & 1:                                             # launched from inside the VAE engine
                vae_gemm_ms += r.ms; vae_gemm_fl += fl
                continue
            key = (i[0], i[1], i[2], i[3] & 255, 32 * ((i[3] >> 8) & 255), (i[3] >> 16) & 255)
            e = shapes.setdefault(key, [0, 0.0, fl])
            e[0] += 1; e[1] += r.ms
        elif r.category == 4:
            conv_fl += 2.0 * i[0] * i[1] * i[2]; conv_ms += r.ms
    shape_rows = [{"M": k[0], "N": k[1], "K": k[2], "epilogue": EPI.get(k[3], str(k[3])), "block_n": k[4], "cta_group": k[5], "launches": v[0],
                   "avg_us": 1e3 * v[1] / v[0], "tflops": v[2] / (v[1] / v[0]) / 1e9, "frac_of_sustained_peak": v[2] / (v[1] / v[0]) / 1e9 / pk["tf"],
                   "share_of_gemm_time": v[1] / max(pms[0], 1e-9)}
                  for k, v in sorted(shapes.items(), key=lambda kv: -kv[1][1]) if v[1] > 0.002 * pms[0]]
    dit_gemm_ms = pms[0] - vae_gemm_ms
    jobs = 1 if sp_mode else world    # images per step over the whole job
    value = jobs * args.steps / (ms / 1000.0)
    attn_ms_x = cat_x["attention"][0]
    out = {
        "metric": "images/sec", "value": value, "unit": "images/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "strong" if sp_mode else "weak", "vs_baseline": None,
        "dtype": "bf16" if args.precision == "bf16" else "fp8(e4m3 projections)+bf16", "data": "synthetic", "config": config, "clocks": clk,
        "gpu_launches": int(launches),
        "e2e": {"value": jobs * args.steps / (ms_e2e / 1000.0), "unit": "images/s", "h2d_bytes_per_step": int(h2d),
                "d2h_bytes_per_step": int(d2h)},
        "roofline": {"kernel": "gemm_bf16_tcgen05_kernel (all fused-epilogue GEMMs of the FLUX-DiT for one image)", "bound": "tensor",
                     "achieved": gemm_fl / (dit_gemm_ms / 1000.0) / 1e12, "peak": pk["tf"], "unit": "TFLOP/s",
                     "frac": gemm_fl / (dit_gemm_ms / 1000.0) / 1e12 / pk["tf"],
                     "traffic": traffic.get("gemm", {}).get("avg_dram_bytes_per_launch"), "traffic_source": traffic.get("source"), "peak_source": pk["src"] + " sustained",
                     "launches": int(pl[0]), "avg_launch_ms": pms[0] / max(1, pl[0]), "flops_per_image": gemm_fl,
                     **({"peak_note": ("58 % of these FLOPs" if args.precision == "fp8" else "the blocks' FLOPs (all but img_in / final / modulation)") +
                                      " ran on e4m3 operands, whose dense peak is 2x the bf16 peak used as the denominator here"}
                        if args.precision != "bf16" else {})},
        "roofline_attention": {"kernel": "attn_fwd4_tcgen05_kernel (persistent schedule; fixed-reference softmax where the block's QK-norm bound applies)",
                               "bound": "tensor", "achieved": attn_fl / (pms[1] / 1000.0) / 1e12,
                               "peak": pk["tf"], "unit": "TFLOP/s", "frac": attn_fl / (pms[1] / 1000.0) / 1e12 / pk["tf"],
                               "launches": int(pl[1]), "avg_launch_ms": pms[1] / max(1, pl[1]), "softmax_variant_per_block": variants,
                               "traffic": traffic.get("attention", {}).get("avg_dram_bytes_per_launch")},
        "roofline_ln_modulate": {"kernel": "ln_modulate_stats_kernel (statistics from the producing GEMM's epilogue; ln_modulate2_kernel for the first LayerNorm of an evaluation)"
                                 if args.precision == "bf16" else "ln_modulate_fp8_kernel (e4m3 rows + per-row scales) + ln_modulate2_kernel", "bound": "hbm", "unit": "GB/s", "peak": pk["hbm"],
                                 "achieved": ln_bytes / (pms[2] / 1000.0) / 1e9, "frac": ln_bytes / (pms[2] / 1000.0) / 1e9 / pk["hbm"],
                                 "launches": int(pl[2]), "avg_launch_ms": pms[2] / max(1, pl[2]),
                                 "note": "algorithmic bytes = read + write of the normalised rows; CUDA events around a ~14 us kernel (ncu: 14.0 us, profiles/r02_summary.md) include ~4 us of launch latency"},
        "roofline_vae": {"kernel": "gemm_bf16_tcgen05_kernel<A_CONV3X3> (implicit-GEMM 3x3 convolutions of the decoder, query row)",
                         "bound": "tensor", "unit": "TFLOP/s", "peak": pk["tf"], "achieved": conv_fl / max(conv_ms, 1e-9) / 1e9,
                         "frac": conv_fl / max(conv_ms, 1e-9) / 1e9 / pk["tf"], "launches": int(pl[4]), "conv_ms": conv_ms,
                         "conv_flops": conv_fl, "other_gemm_ms": vae_gemm_ms, "other_gemm_flops": vae_gemm_fl,
                         "elementwise_ms": pms[5], "elementwise_launches": int(pl[5]),
                         "decode_ms_total": conv_ms + vae_gemm_ms + pms[5]},
        "kernel_time_share": {"gemm_ms": dit_gemm_ms, "attention_ms": pms[1], "ln_modulate_ms": pms[2], "other_ms": pms[3],
                              "vae_conv_ms": conv_ms, "vae_gemm_ms": vae_gemm_ms, "vae_elementwise_ms": pms[5]},
        "gemm_shapes": shape_rows,
        "extra": {"attention_exact_softmax": {"ms_per_step": ms_exact, "images_per_s": jobs * 1000.0 / ms_exact,
                                              "attention_tflops": attn_fl / (attn_ms_x / 1000.0) / 1e12,
                                              "attention_frac": attn_fl / (attn_ms_x / 1000.0) / 1e12 / pk["tf"],
                                              "note": "same image with every block on the exact online-max softmax (score bounds disabled)"}},
    }
    if sp_extra is not None:
        out["extra"]["sp"] = sp_extra
    if world == 1 and not args.no_cpu_baseline:
        v, info = cpu_reference_sample(args.workload)
        out["cpu_baseline"] = {"value": v, "unit": "images/s", "cores": info["threads"], "kind": info["kind"],
                               "sample": cpu_sample_text(info, nfe)}
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
