#!/usr/bin/env python
"""bench.py — denoise-step throughput of the StreamingSVD hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" = ONE pass of the hot path over one batch: StreamingWrapper.forward (ControlNet on 2x7 frames + VideoUNet
with 13 CAM mergers on 2x25 frames, 576x1024 -> latent 72x128, classifier-free-guidance batch 2) followed by the
denoiser scalings, guider combine and Euler update of the sampler (denoiser.py:33-39, guiders.py:78-86,
sampling.py:100-103; two fused elementwise kernels, streamingt2v_b200/sampler.py) — the work of one of
the 150 autoregressive denoise steps of a 200-frame request (SURVEY.md §3.2).  181.96 TFLOP algorithmic.
Weights are random-init of the shipped architecture (no checkpoints offline), inputs synthetic; bf16 compute.

Timed region (per rank): [invalidate conditioning cache] K x forward(+sampler math), bracketed by barrier +
torch.cuda.synchronize(), CUDA events on the launching stream, max over ranks.  The step-invariant conditioning
work (ControlNet conditioning embedding, cross-attention vectors) is executed once INSIDE the timed region, as it
is once per 30-step chunk in the real pipeline.
  value  : steps/s with inputs resident in HBM (whole job: N replicas x per-GPU rate; the path does not shard —
           "replicas only", DESIGN.md §multi-GPU).
  e2e    : same through the public module API (B200StreamingWrapper.forward) with x, t read from pinned HOST
           memory and the result copied back to the host EVERY step; conditioning uploaded from the host once
           inside the timed region (it is constant over a chunk).
  roofline / cpu_baseline: see DESIGN.md §measurement.
  gpu_reference : the reference's own computation as eager PyTorch on the SAME B200 — the oracle port (functional
           restatement of StreamingWrapper.forward, pinned against the unmodified reference) under fp16 autocast
           with cuDNN / cuBLAS / flash-SDPA, same inputs and weights, CUDA-event timed, own clocks record.  A
           reported baseline ("are we faster than torch + libraries on this box?"), never the product path.
  chunk  : one full StreamingSVD chunk = 30 sampler steps (B200EulerEDMSampler) + temporal VAE decode of the 25
           frames, reported as frames/s of new video (18 kept frames per chunk, streaming_svd.py:347).
Multi-GPU (--gpus N, torchrun): default `--mode latency` = classifier-free-guidance halves on rank pairs (one NCCL
all-gather of the network output per step inside each pair, N/2 independent pairs); `--mode throughput` = N replicas.
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

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

STEP_TFLOP = 181.96          # SURVEY.md §8(d): UNet + 13 CAM mergers + ControlNet, T=25, 72x128, CFG 2
FULL_FRAME_PIXELS = 2 * 25 * 72 * 128
METRIC = "denoise_steps_per_sec"
UNIT = "steps/s"


def _parallelism(args):
    if args.gpus == 1:
        return "single GPU"
    if args.mode == "latency":
        return f"cfg-parallel pairs: 2 ranks per step (guidance halves, NCCL all-gather) x {args.gpus // 2} pair(s)"
    return f"replicas x{args.gpus}"


def _workload(args):
    return dict(workload="StreamingSVD denoise step (ControlNet+VideoUNet+CAM), 25 frames, 576x1024 (latent 72x128), "
                         "CFG batch 2 — BASELINE configs[1]/[2] per-step unit",
                frames=25, latent=[72, 128], cfg_batch=2, cam=True, step_tflop=STEP_TFLOP,
                l2="inputs larger than L2 (activations ~19 GB/step >> 126 MB)", parallelism=_parallelism(args))


# ----------------------------------------------------------------------------------------------------------------
# clocks sampling (nvidia-smi) during the timed region
# ----------------------------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index=0):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], 0.0, set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx = max(mx, float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons),
                "samples": len(sm)}


def _usable_cores(cap=32):
    """Host threads the CPU arm may really use: scheduler affinity and cgroup CPU quota (os.cpu_count() reports the
    machine, not the container: 128 threads on a quota of a few cores made one sample forward take 140 s instead of
    ~10 s), capped at 32 -- the bounded sample's convolutions / matmuls do not scale past that."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except AttributeError:
        pass
    try:
        with open("/sys/fs/cgroup/cpu.max") as fh:
            quota, period = fh.read().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except (OSError, ValueError):
        pass
    return max(1, min(n, cap))


# ----------------------------------------------------------------------------------------------------------------
# CPU reference arm / cpu_baseline (oracle port, fp32, torch CPU kernels, all host threads)
# ----------------------------------------------------------------------------------------------------------------
def oracle_flops(cfg, T, h, w, B=2):
    """FLOPs (2 x MAC) of one oracle forward, counted by torch's flop counter on meta tensors (no compute; SDPA
    decomposes to bmm there, so attention is included).  Full step: 181.958 TFLOP, as SURVEY.md section 8(d)."""
    import torch
    from torch.utils.flop_counter import FlopCounterMode
    from oracle import streaming_svd_oracle as orc
    from streamingt2v_b200 import arch
    me = lambda shapes: {k: torch.empty(sh, device="meta") for k, sh in shapes.items()}  # noqa: E731
    n = B * T
    x, t = torch.empty(n, 4, h, w, device="meta"), torch.empty(n, device="meta")
    c = {"concat": torch.empty(n, 4, h, w, device="meta"), "crossattn": torch.empty(n, 1, cfg.context_dim, device="meta"),
         "vector": torch.empty(n, cfg.adm_in_channels, device="meta")}
    ctrl = torch.empty(1, cfg.num_frame_conditioning, 3, 8 * h, 8 * w, device="meta")
    with torch.no_grad(), FlopCounterMode(display=False) as fc:
        orc.streaming_wrapper_forward(me(arch.unet_param_shapes(cfg)), me(arch.controlnet_param_shapes(cfg)), cfg, x, t,
                                      c, batch_size=B, num_video_frames=T, ctrl_frames=ctrl)
    return float(fc.get_total_flops())


def _oracle_weights(cfg, device="cpu", seed=0):
    """Full-size random weights for the oracle arms (unit norm gains, zero biases, fan-in scaled matrices)."""
    import torch
    from streamingt2v_b200 import arch
    g = torch.Generator(device=device).manual_seed(seed)

    def rnd(shapes):
        sd = {}
        for k, sh in shapes.items():
            fan = 1
            for d in sh[1:]:
                fan *= d
            if k.endswith("weight") and len(sh) == 1:
                sd[k] = torch.ones(sh, device=device)
            elif len(sh) <= 1:
                sd[k] = torch.zeros(sh, device=device) if k.endswith("bias") else torch.full(sh, 0.5, device=device)
            else:
                sd[k] = torch.randn(sh, generator=g, device=device) * fan ** -0.5
        return sd

    return rnd(arch.unet_param_shapes(cfg)), rnd(arch.controlnet_param_shapes(cfg))


def cpu_reference_sample(runs=1, warmup=0, budget_s=200.0, big_sample_budget_s=150.0):
    """Time the oracle (CPU restatement of StreamingWrapper.forward, pinned against the reference) on a bounded
    sample of the SAME full-size network and scale to full-step units by the FLOP ratio of the two shapes (torch flop
    counter on meta tensors).  Sample = B=2, T=8 frames at the FULL 72x128 latent (BASELINE.md section 3) when a probe
    at 32x32 predicts that it fits the budget on this host, else the 32x32 probe itself."""
    import torch
    from oracle import streaming_svd_oracle as orc
    from streamingt2v_b200 import arch, synth
    cores = _usable_cores()
    torch.set_num_threads(cores)
    cfg = arch.UNetConfig()
    if os.environ.get("B200SVD_BENCH_CONTRACT_TEST"):
        # tests/test_bench_contract.py only: exercise the arm's plumbing on the reduced-width network in seconds; the
        # printed sample says so and such a line is never a measurement
        cfg = arch.TINY
        big_sample_budget_s = 0.0
    sd_u, sd_c = _oracle_weights(cfg)
    full_flops = oracle_flops(cfg, 25, 72, 128)

    def timed(T, h, w, n_runs, n_warm, budget):
        x, t, c, kw = synth.make_inputs(cfg, T=T, h=h, w=w, seed=1)
        times = []
        t_begin = time.time()
        for i in range(n_warm + n_runs):
            t0 = time.time()
            with torch.no_grad():
                orc.streaming_wrapper_forward(sd_u, sd_c, cfg, x, t, c, **kw)
            dt = time.time() - t0
            over = (time.time() - t_begin) > budget
            if i >= n_warm or over:
                times.append(dt)
            if over:
                break
        return sum(times) / len(times), len(times)

    T = 8
    probe_dt, probe_n = timed(T, 32, 32, 1, 0, budget_s)
    f_probe, f_big = oracle_flops(cfg, T, 32, 32), oracle_flops(cfg, T, 72, 128)
    predicted = probe_dt * f_big / f_probe
    if predicted <= big_sample_budget_s:
        h, w, f_s = 72, 128, f_big
        dt, n = timed(T, h, w, runs, 0, budget_s)      # the probe was the warm-up
    else:
        h, w, f_s = 32, 32, f_probe
        dt, n = (timed(T, h, w, runs, warmup, budget_s) if runs > 1 else (probe_dt, probe_n))
    ratio = full_flops / f_s
    return dict(value=1.0 / (dt * ratio), unit=UNIT, cores=cores, kind="port",
                sample=("[CONTRACT TEST, reduced-width network — not a measurement] " if cfg is arch.TINY else "") +
                       f"oracle port (fp32 torch-CPU, {cores} threads) of StreamingWrapper.forward, full-size weights, "
                       f"B=2 T={T} latent {h}x{w} ({f_s / 1e12:.2f} TFLOP): {dt:.2f}s/forward over {n} run(s) "
                       f"= {f_s / dt / 1e12:.2f} TFLOP/s; scaled x{ratio:.2f} by the FLOP ratio (torch flop counter on "
                       f"meta tensors) to the 25-frame 72x128 step ({full_flops / 1e12:.2f} TFLOP); 32x32 probe "
                       f"{probe_dt:.2f}s predicted {predicted:.0f}s for the 72x128 sample",
                sample_seconds=dt, sample_tflop=f_s / 1e12, cpu_tflops=f_s / dt / 1e12)


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    # each "step" of this arm is one bounded-sample forward (~90 s on 16 host threads): at most two of them, so that the
    # whole run ends within a few minutes whatever --steps says (the value is a rate, not a count)
    cb = cpu_reference_sample(runs=max(1, min(args.steps, 2)), warmup=0)
    v = cb["value"]
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": 1e3 / v, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": _workload(args), "cpu_baseline": cb,
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0}))


# ----------------------------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------------------------
def gpu_reference_leg(cfg, sd_pair, inputs, dev, ours_out, steps=4, warmup=2, index=0):
    """The reference computation as eager PyTorch on this GPU: the oracle port under fp16 autocast (the reference
    runs its UNet under fp16 autocast; xformers == flash SDPA), cuDNN / cuBLAS / flash-SDPA kernels, same weights and
    inputs as our arm.  Returns timing, its own clocks record, and the relative L2 distance between the two outputs
    (a full-size cross-check of the bf16 path against an independent fp16 implementation)."""
    import torch
    from oracle import streaming_svd_oracle as orc
    sd_u, sd_c = sd_pair
    x, t, c, ctrl, B, T = inputs
    kw = dict(batch_size=B, num_video_frames=T, ctrl_frames=ctrl)

    def fwd():
        with torch.no_grad(), torch.autocast("cuda", dtype=torch.float16):
            return orc.streaming_wrapper_forward(sd_u, sd_c, cfg, x, t, c, **kw)

    for _ in range(warmup):
        out = fwd()
    torch.cuda.synchronize()
    sampler = ClockSampler(index)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        out = fwd()
    e1.record()
    torch.cuda.synchronize()
    clocks = sampler.stop()
    ms = e0.elapsed_time(e1) / steps
    out = out.float()
    rel = ((ours_out.float() - out).norm() / out.norm()).item() if ours_out is not None else None
    return dict(kind="oracle port as eager PyTorch on the same GPU: fp16 autocast, cuDNN/cuBLAS/flash-SDPA "
                     "(StreamingWrapper.forward only, no sampler math)",
                ms_per_step=ms, value=1e3 / ms, unit=UNIT, steps=steps, warmup=warmup, clocks=clocks,
                effective_tflops=STEP_TFLOP / (ms * 1e-3), finite=bool(torch.isfinite(out).all()),
                ours_vs_gpu_reference_rel_l2=rel,
                peak_mem_gib=torch.cuda.max_memory_allocated() / 2 ** 30)


def run_ours(args):
    import torch
    import torch.distributed as dist
    from streamingt2v_b200 import arch, dist_utils, ops, synth
    from streamingt2v_b200.sampler import B200EulerEDMSampler
    from streamingt2v_b200.wrapper import B200StreamingWrapper

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (B200); there is no CPU path for the product arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    pair_mode = world > 1 and args.mode == "latency"
    if pair_mode and world % 2:
        raise SystemExit("--mode latency needs an even number of ranks (guidance halves on rank pairs)")
    pair_group = None
    if world > 1:
        # NCCL prints its version banner (and NCCL_DEBUG output) on stdout when the communicator is created: keep
        # stdout for the one JSON line
        sys.stdout.flush()
        saved_fd = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group("nccl", device_id=dev)
            dist.barrier()
            if pair_mode:
                for p0 in range(0, world, 2):           # every rank must take part in every new_group call
                    grp = dist.new_group([p0, p0 + 1])
                    if rank in (p0, p0 + 1):
                        pair_group = grp
                warm = torch.zeros(8, device=dev)
                dist.all_gather_into_tensor(torch.empty(16, device=dev), warm, group=pair_group)
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_fd, 1)
            os.close(saved_fd)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    cfg = arch.UNetConfig()
    T, h, w, B = 25, 72, 128, 2
    sd_u = arch.synth_state_dict_device(arch.unet_param_shapes(cfg), dev, 1)
    sd_c = arch.synth_state_dict_device(arch.controlnet_param_shapes(cfg), dev, 2)
    model = B200StreamingWrapper(cfg, sd_u, sd_c, dev)
    want_gpu_ref = world == 1 and not args.no_gpu_reference
    if not want_gpu_ref:
        del sd_u, sd_c
    torch.cuda.empty_cache()
    # in pair mode both ranks of a pair integrate the SAME video (same seed); different pairs, different videos
    vid = rank // 2 if pair_mode else rank
    half = rank % 2 if pair_mode else None           # 0: unconditional rows, 1: conditional rows (guiders.py:88-97)
    x, t, c, kw = synth.make_inputs(cfg, T=T, h=h, w=w, seed=1 + vid)
    Bm = 1 if pair_mode else B
    rows = slice(half * T, (half + 1) * T) if pair_mode else slice(None)
    # host (pinned) copies for the e2e leg, device copies for the resident leg
    host = dict(x=x.pin_memory(), t=t[rows].contiguous().pin_memory(), ctrl=kw["ctrl_frames"].pin_memory(),
                **{k: v[rows].contiguous().pin_memory() for k, v in c.items()})
    xd, td = x.to(dev), t[rows].to(dev)
    cd = {k: v[rows].to(dev) for k, v in c.items()}
    ctrl_d = kw["ctrl_frames"].to(dev)
    scale = torch.linspace(1.5, 3.0, T).to(dev)                          # LinearPredictionGuider (guiders.py:60-86)
    sigmas = torch.exp(torch.linspace(math.log(700.0), math.log(0.002), args.steps + args.warmup + 2)).tolist()
    net_full = torch.empty((2 * T, 4, h, w), dtype=torch.float32, device=dev) if pair_mode else None
    ag_events = []

    def step(cur, tin, cc, ctrl, i, time_ag=False):
        """one sampler step around the seam (EulerEDMSampler.sampler_step, gamma = 0): input scaling + batch doubling
        (kernel), denoiser forward (the hot path), output scaling + CFG combine + Euler update (kernel).
        cur: the latent state [T,4,h,w]; returns the next state.  Pair mode: this rank evaluates its guidance half
        (a batch-1 forward), the halves are exchanged with one all-gather inside the pair, and both ranks do the
        (identical) combine + Euler update."""
        sig, sig_next = sigmas[i], sigmas[i + 1]
        c_skip, c_out, c_in, c_noise = B200EulerEDMSampler.scalings(sig)  # denoiser_scaling.py:51-59
        tin.fill_(c_noise)
        xin2 = ops.sampler_prepare(cur, c_in)
        if pair_mode:
            xin2 = xin2[:T]                                    # both halves of the doubled input are identical
        net = model(xin2, tin, cc, batch_size=Bm, num_video_frames=T, image_only_indicator=None, ctrl_frames=ctrl,
                    num_conditional_frames=7)
        if pair_mode:
            if time_ag:
                a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                a0.record()
            dist.all_gather_into_tensor(net_full, net.contiguous(), group=pair_group)
            if time_ag:
                a1.record()
                ag_events.append((a0, a1))
            net = net_full
        return ops.sampler_step(net, cur, scale, num_frames=T, c_skip=c_skip, c_out=c_out, sigma=sig,
                                next_sigma=sig_next)            # denoiser.py:33-39, guiders.py:78-86, sampling.py:100-103

    # ---------------- resident leg ----------------
    cur = xd[T:2 * T].clone()
    for i in range(args.warmup):
        cur = step(cur, td, cd, ctrl_d, i)
    # clock settling: the B200 runs this workload at its power cap (sw_power_cap, ~1.5-1.7 of 1.965 GHz); for the first
    # seconds of sustained load the governor overshoots and then over-throttles, which made the first timed leg up to
    # 6 % slower than the second on the same box (profiles/r02_bench_7*.json).  Extra UNTIMED steps until the load has
    # lasted about `--settle` seconds; the timed region is still exactly K steps.
    settle_steps = int(round(args.settle * 5))     # a fixed count (~0.2 s per step): every rank runs the same collectives
    for _ in range(settle_steps):
        cur = step(cur, td, cd, ctrl_d, max(args.warmup - 1, 0))
    torch.cuda.synchronize()
    model.engine.reset_conditioning()  # the conditioning hoist is re-done inside the timed region (once per chunk)
    sampler = ClockSampler(local)
    barrier()
    if rank == 0:
        sampler.start()
    l0 = ops.launches()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(args.steps):
        cur = step(cur, td, cd, ctrl_d, args.warmup + i)
    e1.record()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    launches = ops.launches() - l0
    ms = e0.elapsed_time(e1)
    finite = bool(torch.isfinite(cur).all())
    # what the last timed step handed back: the sampler's next latent state
    outputs = {"latent": cur.float().cpu().numpy()} if args.dump_outputs else None

    # ---------------- e2e leg: host buffers, H2D + D2H every step ----------------
    out_host = torch.empty((T, 4, h, w), dtype=torch.float32).pin_memory()
    x_host = host["x"]
    barrier()
    model.engine.reset_conditioning()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    cc2 = {k: host[k].to(dev, non_blocking=True) for k in ("concat", "crossattn", "vector")}
    ctrl2 = host["ctrl"].to(dev, non_blocking=True)
    cond_bytes = sum(v.numel() * 4 for v in cc2.values()) + ctrl2.numel() * 4
    for i in range(args.steps):
        xin = x_host[T:2 * T].to(dev, non_blocking=True)
        tin = host["t"].to(dev, non_blocking=True)
        nxt = step(xin, tin, cc2, ctrl2, args.warmup + i)
        out_host.copy_(nxt, non_blocking=True)
    f1.record()
    barrier()
    ms_e2e = f0.elapsed_time(f1)
    h2d = x_host[T:2 * T].numel() * 4 + host["t"].numel() * 4 + cond_bytes / args.steps
    d2h = out_host.numel() * 4

    # ---------------- all-gather cost (pair mode): CUDA events around the collective, a few extra steps -----------
    ag_us = None
    if pair_mode:
        for i in range(3):
            cur = step(cur, td, cd, ctrl_d, i, time_ag=True)
        torch.cuda.synchronize()
        ag_us = sorted(a0.elapsed_time(a1) * 1e3 for a0, a1 in ag_events)[len(ag_events) // 2]

    # ---------------- max over ranks ----------------
    ms, ms_e2e = dist_utils.max_over_ranks([ms, ms_e2e], device=dev)

    # ---------------- secondary leg at N > 1: plain replicas (throughput mode) ----------------
    replicas = None
    if pair_mode and not args.no_replicas_leg:
        xr, tr, cr, kwr = synth.make_inputs(cfg, T=T, h=h, w=w, seed=101 + rank)
        xrd, trd = xr.to(dev), tr.to(dev)
        crd = {k: v.to(dev) for k, v in cr.items()}
        ctrlr = kwr["ctrl_frames"].to(dev)

        def rstep(cur_, i):
            sig, sig_next = sigmas[i], sigmas[i + 1]
            c_skip, c_out, c_in, c_noise = B200EulerEDMSampler.scalings(sig)
            trd.fill_(c_noise)
            net = model(ops.sampler_prepare(cur_, c_in), trd, crd, batch_size=B, num_video_frames=T,
                        image_only_indicator=None, ctrl_frames=ctrlr, num_conditional_frames=7)
            return ops.sampler_step(net, cur_, scale, num_frames=T, c_skip=c_skip, c_out=c_out, sigma=sig,
                                    next_sigma=sig_next)

        curr = xrd[T:].clone()
        for i in range(max(2, args.warmup)):
            curr = rstep(curr, i)
        barrier()
        r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        r0.record()
        for i in range(args.steps):
            curr = rstep(curr, args.warmup + i)
        r1.record()
        barrier()
        (ms_r,) = dist_utils.max_over_ranks([r0.elapsed_time(r1)], device=dev)
        replicas = {"value": dist_utils.aggregate_throughput(args.steps, world, ms_r), "unit": UNIT,
                    "ms_per_step": ms_r / args.steps, "parallelism": f"replicas x{world}"}

    # ---------------- per-family live profile (one extra step, outside the timed regions) ----------------
    roof = None
    fam = None
    # every rank takes the step (in pair mode it contains the pair's all-gather); rank 0 reports
    with ops.profile() as prof:
        step(cur, td, cd, ctrl_d, 1)
    if rank == 0:
        fam = {k: dict(launches=v["launches"], ms=round(v["ms"], 3), tflops=round(v["flops"] / 1e12, 3),
                       gbytes=round(v["bytes"] / 1e9, 3)) for k, v in prof.families.items()}
        if os.environ.get("B200SVD_BENCH_SHAPES"):
            with open(os.environ["B200SVD_BENCH_SHAPES"], "w") as fh:
                for famname in ("mtgemm", "flash_attn", "pixel_attn", "small_attn", "groupnorm", "layernorm"):
                    fh.write(f"== {famname}\n")
                    for d_, n_, ms_, tf_ in ops.summarize_records(prof.launch_records, famname, 60):
                        fh.write(f"{ms_:9.3f} ms n={n_:3d} avg={ms_ / n_:7.3f} {tf_:7.1f} TF/s  {d_}\n")
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("bf16_tflops_sustained", 1400.0))
        which = "measured (MEASURED_PEAKS.json bf16_tflops_sustained)" if peaks else "fallback 1.4 PFLOP/s sustained"
        g = prof.families["mtgemm"]
        ach = g["flops"] / (g["ms"] * 1e-3) / 1e12
        roof = {"kernel": "mtgemm_kernel (tcgen05 multi-tap GEMM: all Linear / Conv2d / Conv3d)", "bound": "tensor",
                "achieved": ach, "peak": peak, "unit": "TFLOP/s", "frac": ach / peak, "peak_source": which,
                "launches": g["launches"], "avg_launch_ms": g["ms"] / g["launches"],
                "share_of_step": g["ms"] / sum(v["ms"] for v in prof.families.values()),
                "traffic": None, "traffic_note": "see profiles/ for the ncu --set full capture of this kernel"}
        try:
            tpath = os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")
            if not os.path.exists(tpath):
                tpath = os.path.join(ROOT, "profiles", "r01_ncu_traffic.json")
            tr = json.load(open(tpath))["mtgemm_conv3x3_L0_320to320"]
            roof["traffic"] = tr["traffic_bytes"]
            roof["traffic_note"] = (f"ncu --set full, one launch of the dominant conv shape ({tr['launch']}): "
                                    f"{tr['traffic_bytes'] / 1e6:.0f} MB DRAM vs {tr['algorithmic_bytes'] / 1e6:.0f} MB "
                                    f"algorithmic; roofline.achieved aggregates all {g['launches']} launches of the step")
        except Exception:
            pass
        hbm_peak = float(peaks.get("hbm_gbs", 6500.0))
        for k, v in fam.items():
            if v["tflops"] > 0 and v["ms"] > 0:
                v["tflops_per_s"] = round(v["tflops"] / (v["ms"] * 1e-3), 1)
                v["frac_of_tensor_peak"] = round(v["tflops_per_s"] / peak, 3)
            elif v["gbytes"] > 0 and v["ms"] > 0:
                v["gb_per_s"] = round(v["gbytes"] / (v["ms"] * 1e-3), 1)
                v["frac_of_hbm_peak"] = round(v["gb_per_s"] / hbm_peak, 3)

    # ---------------- one whole chunk: 30 sampler steps + temporal VAE decode (rank 0, single GPU) ----------------
    chunk = first_chunk = None
    if rank == 0 and world == 1 and not args.no_chunk:
        try:
            chunk = chunk_leg(model, cfg, dev, c, kw, T, h, w)
            first_chunk = chunk_leg(model, cfg, dev, c, kw, T, h, w, first=True)
        except Exception as exc:
            chunk = chunk or {"error": repr(exc)}
            first_chunk = first_chunk or {"error": repr(exc)}

    # ---------------- the reference computation as eager PyTorch on this GPU (rank 0, single GPU) ----------------
    gpu_ref = None
    if want_gpu_ref and rank == 0:
        try:
            ours = model(xd, td, cd, batch_size=B, num_video_frames=T, image_only_indicator=None, ctrl_frames=ctrl_d,
                         num_conditional_frames=7).clone()
            gpu_ref = gpu_reference_leg(cfg, (sd_u, sd_c), (xd, td, cd, ctrl_d, B, T), dev, ours, index=local)
        except Exception as exc:
            gpu_ref = {"error": repr(exc)}
        del sd_u, sd_c
        torch.cuda.empty_cache()

    if rank == 0:
        jobs = world // 2 if pair_mode else world            # independent videos advancing one step per `ms`
        sps = dist_utils.aggregate_throughput(args.steps, jobs, ms)
        sps_e2e = dist_utils.aggregate_throughput(args.steps, jobs, ms_e2e)
        line = {
            "metric": METRIC, "value": sps, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None,
            "dtype": "bf16", "data": "synthetic (random-init weights of the shipped architecture, seeded inputs)",
            "config": _workload(args), "clocks": clocks,
            "e2e": {"value": sps_e2e, "unit": UNIT, "ms_per_step": ms_e2e / args.steps,
                    "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h)},
            "gpu_launches": launches, "cuda_graph": bool(model.engine.use_cuda_graph), "settle_steps": settle_steps,
            "roofline": roof, "kernel_families": fam,
            "effective_tflops_per_gpu": STEP_TFLOP / (ms / args.steps * 1e-3) / (2 if pair_mode else 1),
            "finite": finite,
        }
        if pair_mode:
            line["scaling_note"] = ("1 -> 2 GPUs splits ONE step (strong: the two guidance halves); beyond 2, more "
                                    "pairs advance more videos (weak).  value = pairs x steps / s; ms_per_step = latency "
                                    "of one step on a pair")
            line["collective"] = {"op": "ncclAllGather of the network output inside the pair", "bytes": T * 4 * h * w * 4,
                                  "median_us": ag_us}
            line["replicas"] = replicas
        if chunk is not None:
            line["chunk"] = chunk
            line["first_chunk"] = first_chunk
            if "ms_per_chunk" in chunk and first_chunk and "ms_per_chunk" in first_chunk:
                # 200 output frames = the first 25-frame chunk + 10 autoregressive chunks of 18 new frames (25 + 180 >= 200,
                # inference_i2v.py:35, streaming_svd.py:347); conditioner, enhance stage and VFI are not part of this number
                t200 = (first_chunk["ms_per_chunk"] + 10 * chunk["ms_per_chunk"]) * 1e-3
                line["streamingsvd_stage_200_frames"] = {
                    "seconds": t200, "frames_per_sec": 200.0 / t200,
                    "what": "StreamingSVD stage of a 200-frame request on ONE GPU: first chunk (configs[1]) + 10 autoregressive "
                            "chunks (configs[2]); sampler + VAE decode only — conditioner, I2VGen-XL enhance stage and EMA-VFI "
                            "(BASELINE configs[3], [4]) are not built and not included"}
        if gpu_ref is not None:
            line["gpu_reference"] = gpu_ref
            if "ms_per_step" in gpu_ref:
                line["speedup_vs_gpu_reference"] = gpu_ref["ms_per_step"] / (ms / args.steps)
        if not args.no_cpu_baseline and world == 1:
            try:
                line["cpu_baseline"] = cpu_reference_sample()
            except Exception as exc:  # the GPU number must not be lost to a host-side problem
                line["cpu_baseline"] = {"error": repr(exc)}
        if outputs is not None:
            import numpy as np
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, arr in outputs.items():
                np.save(os.path.join(args.dump_outputs, f"{name}.npy"), arr)
        print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def chunk_leg(model, cfg, dev, c, kw, T, h, w, first=False):
    """BASELINE configs[2], one autoregressive chunk: B200EulerEDMSampler (30 AlignYourSteps Euler steps, CFG 1.5->3)
    over the seam + decode_first_stage (temporal VAE decoder, groups of <= 8 frames) -> 25 frames at 576x1024, of
    which 18 are new video (the first 7 re-generate the conditioning frames, streaming_svd.py:347)."""
    import torch
    from streamingt2v_b200 import arch, ops
    from streamingt2v_b200.sampler import B200EulerEDMSampler
    from streamingt2v_b200.vae import B200VaeDecoder
    vcfg = arch.VaeConfig()
    dec = B200VaeDecoder(vcfg, arch.synth_state_dict_device(arch.vae_decoder_param_shapes(vcfg), dev, 3), dev)
    if first:
        # BASELINE configs[1]: the plain SVD chunk that opens a request (StableVideoDiffusionPipeline, streaming_svd.py:390):
        # 25 Euler steps on Karras sigmas, guidance 1.0 -> 3.0, no ControlNet / CAM (159.9 TFLOP per step)
        smp = B200EulerEDMSampler(num_steps=25, num_frames=T, min_scale=1.0, max_scale=3.0, schedule="karras")
    else:
        smp = B200EulerEDMSampler(num_steps=30, num_frames=T)
    n_steps = smp.num_steps
    cond = {k: v[T:].to(dev) for k, v in c.items()}
    uc = {"crossattn": torch.zeros_like(cond["crossattn"]), "concat": torch.zeros_like(cond["concat"]),
          "vector": cond["vector"].clone()}
    extra = dict(image_only_indicator=None, num_video_frames=T, batch_size=2, num_conditional_frames=7,
                 ctrl_frames=None if first else kw["ctrl_frames"].to(dev))
    noise = torch.randn((T, 4, h, w), generator=torch.Generator(device=dev).manual_seed(7), device=dev)

    def decode(z):
        outs = [dec.decode(z[i:i + 8] / 0.18215, timesteps=len(z[i:i + 8])) for i in range(0, T, 8)]
        return torch.cat(outs, 0).clamp_(-1.0, 1.0)

    decode(smp(model, noise, cond, uc, num_steps=2, **extra))           # warm-up: caches, graphs, attributes
    model.engine.reset_conditioning()
    torch.cuda.synchronize()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    sampler = ClockSampler(dev.index or 0)
    sampler.start()
    l0 = ops.launches()
    ev[0].record()
    z = smp(model, noise, cond, uc, **extra)
    ev[1].record()
    frames = decode(z)
    ev[2].record()
    torch.cuda.synchronize()
    clocks = sampler.stop()
    ms_s, ms_d = ev[0].elapsed_time(ev[1]), ev[1].elapsed_time(ev[2])
    kept = T if first else T - 7
    return dict(workload=("first chunk of a request: 25 Euler steps on Karras sigmas (CFG 2, plain SVD UNet, no ControlNet / "
                          "CAM) + temporal VAE decode of 25 frames at 576x1024 (BASELINE configs[1])") if first else
                         ("one StreamingSVD chunk: 30 Euler steps (CFG 2, ControlNet+CAM) + temporal VAE decode of 25 "
                          "frames at 576x1024 (BASELINE configs[2] per-chunk unit)"),
                ms_per_chunk=ms_s + ms_d, sampler_ms=ms_s, sampler_ms_per_step=ms_s / n_steps, vae_decode_ms=ms_d,
                vae_ms_per_frame=ms_d / T, frames_decoded=T, new_frames_per_chunk=kept,
                stage_frames_per_sec=kept / ((ms_s + ms_d) * 1e-3), gpu_launches=ops.launches() - l0,
                finite=bool(torch.isfinite(frames).all()), clocks=clocks,
                note="frames/s of the StreamingSVD stage only (200-frame request = 1 SVD chunk + 10 such chunks, then "
                     "enhance + VFI, which are later rows); conditioner excluded (injected)")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--settle", type=float, default=3.0, help="seconds of untimed load before the timed region")
    ap.add_argument("--no-gpu-reference", action="store_true")
    ap.add_argument("--no-chunk", action="store_true")
    ap.add_argument("--no-replicas-leg", action="store_true")
    ap.add_argument("--mode", default="latency", choices=["latency", "throughput"],
                    help="N>1 only: latency = guidance halves on rank pairs (default), throughput = N replicas")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed to DIR/<name>.npy (float32), for comparing builds")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.impl == "reference":
        run_reference(args)
        return
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.gpus > 1 and world == 1:
        # convenience: relaunch under torchrun on this node
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", os.environ.get("MASTER_PORT", "29511"),
               os.path.abspath(__file__), "--gpus", str(args.gpus), "--steps", str(args.steps), "--warmup",
               str(args.warmup), "--mode", args.mode] + (["--no-cpu-baseline"] if args.no_cpu_baseline else []) + \
              (["--dump-outputs", args.dump_outputs] if args.dump_outputs else [])
        raise SystemExit(subprocess.call(cmd))
    run_ours(args)


if __name__ == "__main__":
    main()
