#!/usr/bin/env python
"""bench.py -- the hot path of ssTEM-restoration on B200: sepconv 51-tap fwd+bwd Mpix/s
(and the flow warp in GB/s) against the kernel rooflines, with the CPU path timed beside it.

    python bench.py --gpus N --steps K --warmup W            # this repo's sm_100a path
    python bench.py --impl reference --gpus N --steps K ...  # the CPU baseline arm

One "step" (default workload `c3_train_step`) is the sepconv work of ONE SFF interpolation
training step (BASELINE.json configs[2]; sff_scripts_interp/model/model_interp.py:94 and its
backward): two `SeparableConvolution.apply` calls on `in[16,3,562,562]`, `v,h[16,51,512,512]`,
each followed by its backward for grad_vertical / grad_horizontal (the input does not require
grad, exactly as in the reference's training loop).  One pixel = one output location of one
section (all channels): 2 x 16 x 512 x 512 = 8 388 608 pixels per step per GPU.

Prints ONE JSON line (rank 0).  `value` = device-resident throughput (CUDA events, max over
ranks); `e2e` = the same step through the public operator with HOST (pinned) buffers, H2D of
input/taps/upstream-grad and D2H of output and both tap gradients inside the timed region.
"""
from __future__ import annotations

import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

K = 51
FLOP_FWD = lambda C: 2 * C * K * (K + 1)            # noqa: E731  SURVEY.md 8(d): 5304*C per pixel
FLOP_BWD_TAPS = lambda C: 2 * (C + 2) * K * K       # noqa: E731  26 010 at C = 3
BYTES_WARP = lambda C: 8 + 8 * C                    # noqa: E731  flow + image read + write per pixel

METRIC = "sepconv_51tap_fwd_bwd_mpix_per_s"
UNIT = "Mpix/s"


# --------------------------------------------------------------------------------------- helpers
def _dist_env():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""

    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0: float, t1: float):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.25)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        rows = [l for (t, l) in self.lines if t0 <= t <= t1 + 0.3] or [l for (_, l) in self.lines]
        for l in rows:
            f = [x.strip() for x in l.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None, "samples": len(sm), "reasons": sorted(reasons)}


def cpu_warp_sample():
    """cpu_baseline leg for the warps (SURVEY 8d): the numpy `image_warp` (simu_sff/image_warp.py, restated bit-equal in
    oracle/) on a uint8 256x256 section and a float 1024x1024x3 one, and the numpy restatement of
    SpatialTransformation.forward on [1,3,1024,1024]; one host core (numpy fancy indexing is single-threaded)."""
    import numpy as np
    import oracle
    from sstem_restoration_b200 import synth
    res = {"cores": 1}
    for name, n, c in (("image_warp_u8_256", 256, 0), ("image_warp_f32_1024x3", 1024, 3)):
        sec = synth.em_section(n, n, 3)
        im = sec if c == 0 else np.repeat(sec[..., None].astype(np.float32), c, axis=2)
        flow, _ = synth.random_fold_flow(n, n, 555)
        oracle.image_warp_restated(im, flow)
        t0 = time.perf_counter()
        reps = 5 if n == 256 else 2
        for _ in range(reps):
            oracle.image_warp_restated(im, flow)
        dt = (time.perf_counter() - t0) / reps
        res[name + "_mpix_per_s"] = round(n * n / dt / 1e6, 2)
    n = 1024
    moving = np.repeat((synth.em_section(n, n, 4).astype(np.float32) / 255.0)[None, None], 3, 1)
    flow, _ = synth.random_fold_flow(n, n, 555)
    oracle.warp_torch_restated(moving, flow[None])
    t0 = time.perf_counter()
    oracle.warp_torch_restated(moving, flow[None])
    dt = time.perf_counter() - t0
    res["spatial_transformation_1024x3_mpix_per_s"] = round(n * n / dt / 1e6, 2)
    res["spatial_transformation_1024x3_gb_per_s"] = round(32 * n * n / dt / 1e9, 3)
    return res


def cpu_simu_sff_sample(calls: int = 10):
    """cpu_baseline leg for BASELINE config 1: the reference's numpy SimuSFF (degradation + noise) restated in
    oracle/ (bit-equal to simu_sff/simuSFF.py:96-144), one host core, 256x256 sections.  -> seconds per call."""
    import random
    import oracle
    from sstem_restoration_b200 import synth
    img = synth.em_section(256, 256, 1)
    rng = random.Random(5)
    t0 = time.perf_counter()
    for _ in range(calls):
        d, _, _ = oracle.sff_degradation_restated(img, 256, rng)
        oracle.sff_noise_restated(d, 256, rng)
    return (time.perf_counter() - t0) / calls


def run_simu_sff(pkg, dev):
    """BASELINE config 1 on the GPU: sff_sim.simu_sff on a 256x256 section (host accept loop included), and the
    degrade kernel alone at the config-5 section size."""
    import random
    import torch
    from sstem_restoration_b200 import sff_sim, synth
    img = torch.from_numpy(synth.em_section(256, 256, 1)).to(dev)
    rng = random.Random(5)
    for _ in range(3):
        sff_sim.simu_sff(img, 256, rng=rng)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    n = 20
    for _ in range(n):
        sff_sim.simu_sff(img, 256, rng=rng)
    torch.cuda.synchronize()
    call_ms = (time.perf_counter() - t0) / n * 1e3
    big = torch.from_numpy(synth.em_section(512, 512, 2)).to(dev).repeat(8, 8)[None].contiguous()
    k, b = synth.gen_line([0, 1400], [4096, 2700])
    prm = [sff_sim.fold_line_params(k, b, 12, 60, 0.05)]
    for _ in range(3):
        sff_sim.gen_flow_warp(big, prm, want_flow=False, want_mask=False)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10):
        sff_sim.gen_flow_warp(big, prm, want_flow=False, want_mask=False)
    e1.record()
    torch.cuda.synchronize()
    kms = e0.elapsed_time(e1) / 10
    cpu_s = cpu_simu_sff_sample()
    return {"config": "c1: SimuSFF (degradation + noise) on a uint8 256x256 EM-like section; bit-equal to the reference's numpy run",
            "gpu_ms_per_call_256": round(call_ms, 4), "gpu_mpix_per_s_256": round(256 * 256 / call_ms / 1e3, 1),
            "cpu_numpy_ms_per_call_256": round(cpu_s * 1e3, 3), "cpu_mpix_per_s_256": round(256 * 256 / cpu_s / 1e6, 2), "cpu_cores": 1,
            "degrade_kernel_4096_ms": round(kms, 4), "degrade_kernel_4096_gpix_per_s": round(4096 * 4096 / kms / 1e6, 1),
            "note": "the 256x256 call is launch- and sync-bound (one 8-byte read per accept attempt); NOT the headline"}


def _cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.lower().startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def _traffic():
    """DRAM bytes per launch from the committed ncu captures (profiles/traffic_r2.json; round 1's as fall-back)."""
    path = os.path.join(ROOT, "profiles", "traffic_r2.json")
    if not os.path.exists(path):
        path = os.path.join(ROOT, "profiles", "traffic_r1.json")
    try:
        return json.load(open(path))
    except Exception:
        return {}


def _peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        try:
            return json.load(open(path)), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md: 6.65 TB/s)"


# --------------------------------------------------------------------------------------- CPU baseline
def cpu_sepconv_sample(steps: int, warmup: int, threads: int | None = None):
    """The CPU path BASELINE.json names for sepconv: unfold-based torch-CPU evaluation of
    kernel.cu:45-49, fwd + autograd bwd for grad_v / grad_h, all host threads; one step =
    in[1,3,306,306] (a 256x256 section).  Returns (Mpix/s, seconds per step, description)."""
    import numpy as np
    import torch
    import oracle
    from sstem_restoration_b200 import synth

    threads = threads or os.cpu_count() or 1
    torch.set_num_threads(threads)
    H = W = 256
    inp = torch.from_numpy(synth.section_to_input(synth.em_section(H, W, 0))[None])
    v = torch.from_numpy(synth.unit_taps(1, K, H, W, seed=1)).requires_grad_(True)
    h = torch.from_numpy(synth.unit_taps(1, K, H, W, seed=2)).requires_grad_(True)
    g = torch.from_numpy(np.random.default_rng(99).standard_normal((1, 3, H, W)).astype(np.float32))

    def step():
        v.grad = None
        h.grad = None
        out = oracle.sepconv_unfold_torch(inp, v, h)
        out.backward(g)
        return out

    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / max(steps, 1)
    return H * W / dt / 1e6, dt, f"unfold torch-CPU fwd+bwd(gv,gh) of in[1,3,306,306], v,h[1,51,256,256], {steps} steps"


def cpu_sepconv_fast_port_sample(steps: int = 3):
    """The strongest CPU implementation in the tree, reported BESIDE the baseline BASELINE.json prescribes (unfold-based
    torch): the factored fp32 C port with OpenMP over pixels (oracle/sepconv_oracle.c), same 256x256 workload.  -> Mpix/s."""
    import numpy as np
    import oracle
    from sstem_restoration_b200 import synth
    H = W = 256
    inp = synth.section_to_input(synth.em_section(H, W, 0))[None]
    v, h = synth.unit_taps(1, K, H, W, seed=1), synth.unit_taps(1, K, H, W, seed=2)
    g = np.random.default_rng(99).standard_normal((1, 3, H, W)).astype(np.float32)
    oracle.sepconv_fwd_bwd_fast(inp, v, h, g)
    t0 = time.perf_counter()
    for _ in range(steps):
        oracle.sepconv_fwd_bwd_fast(inp, v, h, g)
    return H * W / ((time.perf_counter() - t0) / steps) / 1e6


def run_reference_arm(args):
    rank, _, world = _dist_env()
    if rank != 0:
        return
    steps = max(1, min(args.steps, 20))
    warm = max(1, min(args.warmup, 3))
    cores = os.cpu_count() or 1
    val, dt, sample = cpu_sepconv_sample(steps, warm, cores)
    line = {
        "impl": "reference", "metric": METRIC, "value": round(val, 4), "unit": UNIT, "n_gpus": args.gpus, "steps": steps,
        "warmup": warm, "ms_per_step": round(dt * 1e3, 3), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "c3_train_step (bounded CPU sample: one 256x256 section per step; linear in pixels)",
                   "note": "the reference's sepconv is GPU-only (libs/sepconv/SeparableConvolution.py:47-48); per BASELINE.json "
                           "the CPU arm is an unfold-based torch-CPU evaluation of the same filter on all host cores"},
        "cpu_baseline": {"value": round(val, 4), "unit": UNIT, "cores": cores, "kind": "port", "sample": sample,
                         "cpu_model": _cpu_model(), "torch_threads": cores},
        "e2e": {"value": round(val, 4), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


# --------------------------------------------------------------------------------------- GPU arm
def run_gpu_arm(args):
    import numpy as np
    import torch
    import torch.distributed as dist
    import sstem_restoration_b200 as pkg
    from sstem_restoration_b200 import shard, synth

    rank, local_rank, world = _dist_env()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "").upper() in ("VERSION", ""):
            os.environ["NCCL_DEBUG"] = "WARN"            # keep stdout to the one JSON line
        dist.init_process_group("nccl", device_id=dev)
    sep = pkg.SeparableConvolution.apply
    # The headline runs the GENERAL 3-channel path (the roofline's flop count is the 3-channel one).  The package default
    # ("auto") would detect that the synthetic sections are gray x3 -- as every reference caller's are -- and compute one
    # plane; that path is measured separately below (extra.gray_x3_shortcut: asserted and auto-detected).
    pkg.set_gray_replicated("off")

    B, C, H, W = args.batch, 3, args.size, args.size
    calls = 2                                           # model_interp.py:94: two sepconv calls per step
    pix_per_step = calls * B * H * W

    # ---- synthetic EM-like inputs, resident in HBM before the timed region ------------------
    gen = torch.Generator(device=dev).manual_seed(4321 + rank)
    sets = []
    for k in range(calls):
        secs = np.stack([synth.section_to_input(synth.em_section(H, W, 100 * rank + 16 * k + b)) for b in range(B)])
        inp = torch.from_numpy(secs).to(dev)
        v = torch.softmax(torch.randn((B, K, H, W), device=dev, generator=gen), 1).requires_grad_(True)
        h = torch.softmax(torch.randn((B, K, H, W), device=dev, generator=gen), 1).requires_grad_(True)
        g = torch.randn((B, C, H, W), device=dev, generator=gen)
        sets.append((inp, v, h, g))
    ev = lambda: torch.cuda.Event(enable_timing=True)   # noqa: E731
    kern_events = []

    # The path's only exchange -- gathering the restored outputs -- runs on a side stream so that it
    # overlaps the next step's kernels (it is still inside the timed region: the region ends with a
    # wait on the side stream).  Two gather buffers alternate.
    comm_stream = torch.cuda.Stream(device=dev) if world > 1 else None
    comm_done = [None, None]
    step_no = [0]
    gatherer = None
    if world > 1 and not args.no_gather:
        gatherer = shard.SectionGatherer((C, H, W), torch.float32, calls * B, dev, dst=0, force_collective=args.nccl_gather)

    def step(record=False):
        outs = []
        for (inp, v, h, g) in sets:
            v.grad = None
            h.grad = None
            if record:
                e0, e1, e2 = ev(), ev(), ev()
                e0.record()
            out = sep(inp, v, h)
            if record:
                e1.record()
            out.backward(g)
            if record:
                e2.record()
                kern_events.append((e0, e1, e2))
            outs.append(out.detach())
        if world > 1 and not args.no_gather:
            local = torch.cat(outs, 0)
            ready = ev()
            ready.record()
            k = step_no[0] & 1
            with torch.cuda.stream(comm_stream):
                comm_stream.wait_event(ready)
                local.record_stream(comm_stream)
                gatherer.gather(local)                     # to rank 0, as DataParallel does (copy-engine peer writes)
                comm_done[k] = torch.cuda.Event()
                comm_done[k].record(comm_stream)
            step_no[0] += 1
        return outs

    def drain_comm():
        if comm_stream is not None:
            torch.cuda.current_stream(dev).wait_stream(comm_stream)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(max(args.warmup, 3)):
        step()
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    n0 = pkg.launch_count()
    t_start, t_stop = ev(), ev()
    barrier()
    w0 = time.time()
    t_start.record()
    for _ in range(args.steps):
        outs = step(record=True)
    drain_comm()
    t_stop.record()
    barrier()
    w1 = time.time()
    launches = pkg.launch_count() - n0
    ms_total = t_start.elapsed_time(t_stop)
    clocks = sampler.stop(w0, w1) if rank == 0 else None
    per_rank = None
    if world > 1:
        allt = [torch.zeros(1, device=dev, dtype=torch.float64) for _ in range(world)]
        dist.all_gather(allt, torch.tensor([ms_total / args.steps], device=dev, dtype=torch.float64))
        per_rank = [round(float(t.item()), 4) for t in allt]
    tmax = torch.tensor([ms_total], device=dev, dtype=torch.float64)
    lsum = torch.tensor([launches], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(lsum, op=dist.ReduceOp.SUM)
    ms_total = float(tmax.item())
    ms_step = ms_total / args.steps
    value = world * pix_per_step / (ms_step * 1e-3) / 1e6

    fwd_ms = statistics.mean(e0.elapsed_time(e1) for e0, e1, _ in kern_events)
    bwd_ms = statistics.mean(e1.elapsed_time(e2) for _, e1, e2 in kern_events)
    if args.dump_outputs and rank == 0:                 # before the legs below run more steps on the same tensors
        dump_outputs(args.dump_outputs, {f"call{k}_{name}": t for k, (out, (_, v, h, _)) in enumerate(zip(outs, sets))
                                         for name, t in (("output", out), ("grad_vertical", v.grad), ("grad_horizontal", h.grad))})

    # ---- the reference's actual inputs are gray sections replicated x3: opt-in shortcut, reported aside
    gray = None
    if all(bool(torch.equal(s_[0][:, 0], s_[0][:, 1])) and bool(torch.equal(s_[0][:, 0], s_[0][:, 2])) for s_ in sets):
        pkg.set_gray_replicated("assert")
        try:
            for _ in range(2):
                step()
            g0, g1 = ev(), ev()
            barrier()
            g0.record()
            for _ in range(args.steps):
                step()
            drain_comm()
            g1.record()
            barrier()
            gms = g0.elapsed_time(g1) / args.steps
            pkg.set_gray_replicated("detect")               # device-side plane comparison + two gated launches, no host sync
            for _ in range(2):
                step()
            barrier()
            g0.record()
            for _ in range(args.steps):
                step()
            drain_comm()
            g1.record()
            barrier()
            dms = g0.elapsed_time(g1) / args.steps
            gray = {"mpix_per_s": round(world * pix_per_step / (gms * 1e-3) / 1e6, 1), "ms_per_step": round(gms, 4),
                    "detected_on_device_mpix_per_s": round(world * pix_per_step / (dms * 1e-3) / 1e6, 1), "detected_on_device_ms_per_step": round(dms, 4),
                    "note": "same step with SSTEM_SEPCONV_GRAY_REPLICATED asserted (identical channel planes: one plane computed, "
                            "t = (sum_c g_c) * in_0); NOT the headline -- the headline runs the general 3-channel path"}
        finally:
            pkg.set_gray_replicated("off")

    # ---- e2e: same step through the public operator with HOST buffers -----------------------
    e2e = None
    if not args.no_e2e:
        e2e = run_e2e(args, pkg, dev, sets, calls, B, C, H, W, world, dist if world > 1 else None)

    # free the headline tensors before the other configurations (config 5 alone needs ~16 GB)
    del sets
    torch.cuda.empty_cache()
    peaks, peak_src = _peaks()
    hbm = float(peaks.get("hbm_gbs", 6650.0))
    fp32_peak, probe_mhz = pkg.fp32_peak_probe()

    # ---- config 5 (every rank takes part: strong scaling over the 98 targets) and its host-buffer form
    c5 = c5_host = c5_tiled = c5_prod = None
    if not args.no_stack:
        c5 = run_c5_stack(pkg, dev, rank, world, dist if world > 1 else None, args.sections, args.section_size)
        if e2e is not None:
            c5_host = run_c5_stack(pkg, dev, rank, world, dist if world > 1 else None, args.sections, args.section_size, to_host=True)
        c5_tiled = run_c5_stack(pkg, dev, rank, world, dist if world > 1 else None, args.sections, args.section_size, tiled_taps=True)
        c5_prod = run_c5_stack(pkg, dev, rank, world, dist if world > 1 else None, args.sections, args.section_size, producer=True)
        torch.cuda.empty_cache()

    # ---- warp (configs 4 / 5), the other BASELINE configurations, section-8f rows: rank 0, beside the headline
    warp = run_warp(args, pkg, dev) if not args.no_warp else None
    tail = run_tail(pkg, dev, B, H, W) if (not args.no_warp and rank == 0) else None
    simu = run_simu_sff(pkg, dev) if (not args.no_warp and rank == 0) else None
    configs = None
    if not args.no_warp and rank == 0:
        configs = {}
        configs.update(run_c2_c4_sepconv(pkg, dev, fp32_peak, hbm))
        configs.update(run_c4_warps(pkg, dev, hbm))
        configs["n2_tap_producer_2048"] = run_tap_producer(pkg, dev, peaks)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if configs is not None:
        configs["c1_simu_sff"] = simu
        configs["c3_train_step"] = "the headline (value / roofline / rooflines)"
        configs["c5_stack"] = c5
        if c5_host is not None:
            configs["c5_stack_host_out"] = c5_host
        if c5_tiled is not None:
            configs["c5_stack_tile_major_taps"] = c5_tiled
        if c5_prod is not None:
            configs["c5_stack_with_tap_producers"] = c5_prod
    if e2e is not None and c5_host is not None:
        e2e["e2e_u8"] = {"what": "config 5 through restore_stack with HOST buffers both ways: uint8 sections in pinned memory -> restored uint8 "
                                 "sections in pinned memory (1 byte per pixel up per section, 3 bytes per target down; every rank keeps its own targets)",
                         "mpix_per_s": c5_host["mpix_per_s"], "sections_per_s": c5_host["sections_per_s"], "seconds": c5_host["seconds"],
                         "h2d_bytes_rank0": c5_host["h2d_bytes_rank0"], "d2h_bytes_rank0": c5_host["d2h_bytes_rank0"]}

    px_call = B * H * W
    fwd_tflops = FLOP_FWD(C) * px_call / (fwd_ms * 1e-3) / 1e12
    bwd_tflops = FLOP_BWD_TAPS(C) * px_call / (bwd_ms * 1e-3) / 1e12
    rooflines = {
        "sepconv_fwd": {"bound": "fp32", "achieved": round(fwd_tflops, 3), "peak": round(fp32_peak, 2), "unit": "TFLOP/s",
                        "frac": round(fwd_tflops / fp32_peak, 4), "ms_per_launch": round(fwd_ms, 4),
                        "flop_per_pixel": FLOP_FWD(C), "traffic": None},
        "sepconv_bwd_taps": {"bound": "fp32", "achieved": round(bwd_tflops, 3), "peak": round(fp32_peak, 2), "unit": "TFLOP/s",
                             "frac": round(bwd_tflops / fp32_peak, 4), "ms_per_launch": round(bwd_ms, 4),
                             "flop_per_pixel": FLOP_BWD_TAPS(C), "traffic": None},
    }
    if warp:
        rooflines["warp"] = {"bound": "hbm", "achieved": round(warp["gbs"], 1), "peak": hbm, "unit": "GB/s",
                             "frac": round(warp["gbs"] / hbm, 4), "ms_per_launch": round(warp["ms"], 5),
                             "bytes_per_pixel": BYTES_WARP(3), "traffic": None, "peak_source": peak_src}
    traffic = _traffic()
    for name, r in rooflines.items():
        t = traffic.get(name)
        if t and (name == "warp" or (B * H * W == t.get("pixels_per_launch"))):
            r["traffic"] = t["dram_bytes_per_launch"]
            r["traffic_source"] = t["source"]
            r["algorithmic_bytes_per_launch"] = t["algorithmic_bytes_per_launch"]
    dominant = "sepconv_bwd_taps" if bwd_ms >= fwd_ms else "sepconv_fwd"
    roof = dict(rooflines[dominant])
    roof["kernel"] = dominant
    roof["peak_source"] = ("FFMA probe on this GPU in this run (sstem_fp32_peak_probe: best of 3 register-resident FMA loops; SM "
                           "clocks in `clocks`); nominal 148 SM x 128 lanes x 2 x 1.965 GHz = 74.4 TFLOP/s; MEASURED_PEAKS.json has "
                           "no fp32 row")

    cpu_val, cpu_dt, cpu_sample = cpu_sepconv_sample(steps=3, warmup=1)
    if warp:
        warp["cpu_baseline"] = cpu_warp_sample()
    line = {
        "metric": METRIC, "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": round(ms_step, 4), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": "c3_train_step", "calls_per_step": calls, "input": [B, C, H + 50, W + 50],
                   "taps": [B, K, H, W], "pixels_per_step_per_gpu": pix_per_step, "parallelism": f"dp{world} (batch shards, no data-path collective; outputs gathered to rank 0 on a side stream"
                                  + (f", {gatherer.mode}" + (f" [{gatherer.why}]" if gatherer.why else "") if gatherer is not None else "") + ")",
                   "l2": "working set 7 GB per step >> 126 MB L2 (no flush needed)"},
        "roofline": roof, "rooflines": rooflines,
        "cpu_baseline": {"value": round(cpu_val, 4), "unit": UNIT, "cores": os.cpu_count(), "kind": "port", "sample": cpu_sample,
                         "cpu_model": _cpu_model(), "torch_threads": os.cpu_count(),
                         "fast_c_port_openmp_mpix_per_s": round(cpu_sepconv_fast_port_sample(), 4),
                         "note": "`value` is the baseline BASELINE.json prescribes (unfold-based torch-CPU); the factored C / OpenMP port "
                                 "in oracle/ is the fastest CPU form in the tree and is reported beside it"},
        "e2e": e2e, "gpu_launches": int(lsum.item()), "clocks": clocks,
        "extra": {"fwd_mpix_per_s": round(px_call / (fwd_ms * 1e-3) / 1e6, 1), "bwd_taps_mpix_per_s": round(px_call / (bwd_ms * 1e-3) / 1e6, 1),
                  "configs": configs, "warp": warp, "gray_x3_shortcut": gray, "fused_interp_tail": tail, "simu_sff_c1": simu,
                  "ms_per_step_by_rank": per_rank},
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


DUMP_BYTES = 60 * 10 ** 6                           # --dump-outputs writes at most this many bytes of array data


def dump_outputs(dirname, arrays):
    """Writes each tensor of `arrays` as DIR/<name>.npy in float32.  When they do not fit in DUMP_BYTES together, each is
    written as a 1-D sample of its flattened elements instead: sorted flat indices drawn from a seed fixed by the tensor's
    position in `arrays`, so that two runs with the same arguments write the same elements."""
    import numpy as np
    import torch
    os.makedirs(dirname, exist_ok=True)
    sample = sum(t.numel() for t in arrays.values()) * 4 > DUMP_BYTES
    per = DUMP_BYTES // 4 // len(arrays)
    for i, (name, t) in enumerate(arrays.items()):
        t = t.detach()
        if sample and t.numel() > per:
            idx = np.unique(np.random.default_rng(i).integers(0, t.numel(), per))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(dirname, name + ".npy"), t.float().cpu().numpy())


def _bind_near_gpu(dev):
    """Best effort: run this rank (and first-touch its pinned buffers) on the CPUs local to its GPU."""
    try:
        import torch
        bus = torch.cuda.get_device_properties(dev).pci_bus_id
        dom = torch.cuda.get_device_properties(dev).pci_domain_id
        devid = torch.cuda.get_device_properties(dev).pci_device_id
        path = f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{devid:02x}.0/local_cpulist"
        cpus = set()
        for part in open(path).read().strip().split(","):
            lo, _, hi = part.partition("-")
            cpus.update(range(int(lo), int(hi or lo) + 1))
        if cpus:
            os.sched_setaffinity(0, cpus)
            return len(cpus)
    except Exception:
        pass
    return None


def run_e2e(args, pkg, dev, sets, calls, B, C, H, W, world, dist):
    """Host (pinned) buffers in, host buffers out: the step through the host-buffer entry point
    (sepconv_forward_backward_host: chunked H2D -> C-ABI kernels -> D2H on rotating streams)."""
    import torch
    # pinned buffers are first-touched by this thread: allocate them on the CPUs next to the GPU (a cross-socket
    # hop costs ~10 % of PCIe throughput), then give the process its full affinity back for the CPU baseline
    old_affinity = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else None
    numa_cpus = _bind_near_gpu(dev)
    host_in = [tuple(t.detach().cpu().pin_memory() for t in s) for s in sets]
    host_out = [(torch.empty((B, C, H, W)).pin_memory(), torch.empty((B, K, H, W)).pin_memory(), torch.empty((B, K, H, W)).pin_memory())
                for _ in sets]
    h2d = sum(t.numel() * 4 for s in host_in for t in s)
    d2h = sum(t.numel() * 4 for s in host_out for t in s)

    def step():
        for (hi, hv, hh, hg), ho in zip(host_in, host_out):
            pkg.sepconv_forward_backward_host(hi, hv, hh, hg, device=dev, out=ho, join=False)
        pkg.join_host_pipeline(dev)                      # results of the step are complete on the current stream

    steps = max(2, min(args.steps, 5))
    step()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    t0 = time.perf_counter()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    ms = max(e0.elapsed_time(e1), wall * 1e3)
    t = torch.tensor([ms], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t.item()) / steps
    # spot-check the host path against the device-resident path (same kernels, same inputs)
    ref = pkg.SeparableConvolution.apply(sets[0][0][:1], sets[0][1][:1].detach(), sets[0][2][:1].detach())
    same = bool(torch.equal(ref.cpu(), host_out[0][0][:1]))
    if old_affinity is not None:
        try:
            os.sched_setaffinity(0, old_affinity)
        except Exception:
            pass
    del host_in, host_out
    ceil_s = run_copy_ceiling(dev, h2d, d2h, world, dist)
    return {"value": round(world * calls * B * H * W / (ms * 1e-3) / 1e6, 2), "unit": UNIT, "ms_per_step": round(ms, 3),
            "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "steps": steps, "matches_device_path": same,
            "copy_ceiling": {"what": "the same H2D and D2H byte counts per step as raw pinned-memory copies on two streams, no kernels "
                                     "(max over ranks): the host link's own limit for this step",
                             "ms_per_step": round(ceil_s * 1e3, 3), "mpix_per_s": round(world * calls * B * H * W / ceil_s / 1e6, 2),
                             "gb_per_s_per_gpu_both_directions": round((h2d + d2h) / ceil_s / 1e9, 1),
                             "e2e_fraction_of_ceiling": round(ceil_s * 1e3 / ms, 3)},
            "note": "the e2e step ships 816 B/pixel of taps up and 816 B/pixel of tap gradients down -- traffic that does not exist in the "
                    "reference pipeline (taps are produced and consumed on the GPU); `e2e_u8` is the stack job with uint8 on the wire",
            "cpus_bound_near_gpu": numa_cpus,
            "api": "sepconv_forward_backward_host(pinned input, vertical, horizontal, grad_output) -> pinned output, grad_vertical, "
                   "grad_horizontal; two samples per chunk on 3 streams (H2D, C-ABI fwd+bwd kernels, D2H overlapped); the step's two calls are queued back to back and joined once"}


def _time_warp(pkg, dev, H, W, nsets, reps):
    import numpy as np
    import torch
    from sstem_restoration_b200 import synth
    st = pkg.SpatialTransformation(True)
    flow_np, _ = synth.random_fold_flow(H, W, 555)
    planar0 = torch.from_numpy(np.ascontiguousarray(flow_np.transpose(2, 0, 1))[None]).to(dev)
    sec = torch.from_numpy(synth.em_section(H, W, 50).astype(np.float32) / 255.0).to(dev)
    bufs = []
    for i in range(nsets):
        im = torch.roll(sec, shifts=17 * i, dims=1)[None, None].expand(1, 3, H, W).contiguous()   # gray x3, as the callers feed
        bufs.append((im, (planar0 + 0.01 * i).permute(0, 2, 3, 1)))
    for _ in range(10):                                 # warm-up: the preceding e2e leg is PCIe-bound and lets the clocks drop
        for im, fl in bufs:
            st(im, fl)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        for im, fl in bufs:
            st(im, fl)
    e1.record()
    torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / (reps * nsets)
    del bufs
    torch.cuda.empty_cache()
    return ms


def run_warp(args, pkg, dev):
    """Flow warp (SpatialTransformation) on the SFF fold flow, planar-strided flow view, rotating buffer sets > L2:
    the config-5 section size (4096^2, the roofline entry) and the config-4 size (2048^2, launch-latency share larger)."""
    ms5 = _time_warp(pkg, dev, 4096, 4096, nsets=3, reps=20)       # 3 x 537 MB
    ms4 = _time_warp(pkg, dev, 2048, 2048, nsets=6, reps=20)       # 6 x 134 MB
    g = lambda n, ms: BYTES_WARP(3) * n * n / (ms * 1e-3) / 1e9
    return {"metric": "warp_gb_per_s", "gbs": g(4096, ms5), "ms": ms5, "gpix_per_s": 4096 * 4096 / (ms5 * 1e-3) / 1e9,
            "config": "c5 section warp: im[1,3,4096,4096], flow planar [1,2,4096,4096] viewed as [1,4096,4096,2], SFF fold flow "
                      "(gen_flow, seed 555); 3 rotating buffer sets (1.6 GB > L2); through the SpatialTransformation module",
            "c4_2048": {"gbs": g(2048, ms4), "ms": ms4, "gpix_per_s": 2048 * 2048 / (ms4 * 1e-3) / 1e9,
                        "config": "c4 warp: im[1,3,2048,2048], same flow family; 6 rotating buffer sets (805 MB > L2)"}}



def _events_ms(fn, reps, warm=3):
    import torch
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / reps


def run_c2_c4_sepconv(pkg, dev, fp32_peak, hbm_gbs):
    """BASELINE configs 2 and 4 (sepconv part): forward of one 256x256 section (C = 1 literal, C = 3 as the reference
    calls it) and of one 2048x2048 section, unit-scale taps, rotating input sets larger than L2."""
    import torch
    sep = pkg.SeparableConvolution.apply
    gen = torch.Generator(device=dev).manual_seed(77)
    res = {}
    for name, C, n, nsets, reps in (("c2_fwd_c1", 1, 256, 6, 50), ("c2_fwd_c3", 3, 256, 6, 50), ("c4_sepconv_fwd_2048", 3, 2048, 2, 5)):
        sets = []
        for _ in range(nsets):
            inp = torch.rand((1, C, n + 50, n + 50), device=dev, generator=gen)
            v = torch.softmax(torch.randn((1, K, n, n), device=dev, generator=gen), 1)
            h = torch.softmax(torch.randn((1, K, n, n), device=dev, generator=gen), 1)
            sets.append((inp, v, h))

        def step():
            for inp, v, h in sets:
                sep(inp, v, h)
        ms = _events_ms(step, reps) / nsets
        tf = FLOP_FWD(C) * n * n / (ms * 1e-3) / 1e12
        tap_gbs = 408.0 * n * n / (ms * 1e-3) / 1e9
        res[name] = {"input": [1, C, n + 50, n + 50], "ms_per_call": round(ms, 5), "mpix_per_s": round(n * n / (ms * 1e-3) / 1e6, 1),
                     "tflops": round(tf, 3), "frac_fp32_probe": round(tf / fp32_peak, 4), "taps_gb_per_s": round(tap_gbs, 1),
                     "frac_hbm_taps": round(tap_gbs / hbm_gbs, 4), "l2": f"{nsets} rotating input sets ({nsets * 2 * K * n * n * 4 / 1e6:.0f} MB of taps)"}
        if n == 256:
            res[name]["note"] = "one 256x256 section is 512 CTA tiles on 148 SMs: launch / tail-latency bound, neither roofline applies"
        del sets
        torch.cuda.empty_cache()
    return res


def run_c4_warps(pkg, dev, hbm_gbs):
    """BASELINE config 4 (warp part): im[1,3,2048,2048], planar-strided flow view; SFF fold flow and the N(0, 5 px) flow."""
    import numpy as np
    import torch
    from sstem_restoration_b200 import synth
    st = pkg.SpatialTransformation(True)
    n, nsets, reps = 2048, 6, 20
    sec = torch.from_numpy(synth.em_section(n, n, 50).astype(np.float32) / 255.0).to(dev)
    res = {}
    for name, flow_np in (("c4_warp_fold", synth.random_fold_flow(n, n, 555)[0]), ("c4_warp_noise5px", synth.noise_flow(n, n, 5.0))):
        planar0 = torch.from_numpy(np.ascontiguousarray(flow_np.transpose(2, 0, 1))[None]).to(dev)
        bufs = []
        for i in range(nsets):
            im = torch.roll(sec, shifts=17 * i, dims=1)[None, None].expand(1, 3, n, n).contiguous()
            bufs.append((im, (planar0 + 0.01 * i).permute(0, 2, 3, 1)))

        def step():
            for im, fl in bufs:
                st(im, fl)
        ms = _events_ms(step, reps, warm=5) / nsets
        gbs = BYTES_WARP(3) * n * n / (ms * 1e-3) / 1e9
        res[name] = {"ms_per_call": round(ms, 5), "gb_per_s": round(gbs, 1), "frac_hbm": round(gbs / hbm_gbs, 4),
                     "gpix_per_s": round(n * n / (ms * 1e-3) / 1e9, 2), "l2": f"{nsets} rotating buffer sets ({nsets * 134} MB)"}
        del bufs
        torch.cuda.empty_cache()
    return res


def run_tap_producer(pkg, dev, peaks):
    """SURVEY 8f N2, producer side, at config 4's size: the last two layers of a tap branch (upsample x2 -> Conv2d(51,51,3);
    model_interp.py:18, 130-137) as the fused tcgen05 kernel writing tile-major taps, and the producer -> consumer chain
    (two tap tensors -> sepconv_forward_tiled) with no [B,51,H,W] tensor in between.  Roofline: tensor-bound work, measured
    against half the dense bf16 figure of MEASURED_PEAKS.json (TF32 runs at half the bf16 rate), burst value -- the
    kernel is timed alone.  The library chain it replaces (F.interpolate -> cuDNN TF32 conv -> layout conversion) is timed
    beside it by tools/bench_tapconv.py (profiles/tapconv_r2.md); bench.py runs none of torch's operators."""
    import torch
    n = 2048
    gen = torch.Generator(device=dev).manual_seed(99)
    nrot = 4                                                   # 4 x (53 MB in + 855 MB out) >> L2
    xs = [torch.relu(torch.randn((1, 51, n // 2, n // 2), device=dev, generator=gen)) for _ in range(nrot)]
    w = torch.randn((51, 51, 3, 3), device=dev, generator=gen) / 21.4
    bias = 0.1 * torch.randn(51, device=dev, generator=gen)
    packed = pkg.pack_tap_conv_weight(w)
    outs = [None, None]
    it = [0]

    def step():
        it[0] += 1
        outs[it[0] & 1] = pkg.tap_conv3x3(xs[it[0] % nrot], packed, bias, upsample=True, tiled=True)
    ms = _events_ms(step, 20, warm=5)
    flop = 2.0 * 51 * 51 * 9 * n * n
    tf32_peak = float(peaks.get("bf16_tflops", 2250.0)) / 2
    res = {"ms_per_tap_tensor": round(ms, 4), "tflops_useful": round(flop / ms / 1e9, 1), "flop_per_pixel": 2 * 51 * 51 * 9,
           "roofline": {"bound": "tensor", "achieved": round(flop / ms / 1e9, 1), "peak": round(tf32_peak, 1), "unit": "TFLOP/s",
                        "frac": round(flop / ms / 1e9 / tf32_peak, 4),
                        "peak_source": "MEASURED_PEAKS.json bf16_tflops (burst) / 2: TF32 is half the bf16 rate" if "bf16_tflops" in peaks else "nominal 1125 TFLOP/s TF32 dense",
                        "note": "useful flops only (51 of the 64 padded output channels, 51 of 56 padded input channels: the tensor core does 1.38x this)"},
           "hbm_gb_per_s": round((51 * (n // 2) ** 2 + 51 * n * n) * 4 / ms / 1e6, 1),
           "kernel": "tap_conv3x3_kernel<UPS, TILED>: tcgen05.mma kind::tf32 M128 N64 K8, accumulators in TMEM, upsample fused into the operand producer"}
    # producer -> consumer without NCHW taps: two branches feed one sepconv forward
    frame = torch.rand((1, 3, n + 50, n + 50), device=dev, generator=gen)

    def chain():
        v = pkg.tap_conv3x3(xs[0], packed, bias, upsample=True, tiled=True)
        h = pkg.tap_conv3x3(xs[1], packed, bias, upsample=True, tiled=True)
        return pkg.sepconv_forward_tiled(frame, v, h)
    cms = _events_ms(chain, 10, warm=3)
    res["chain_2_producers_1_sepconv_ms"] = round(cms, 4)
    res["chain_mpix_per_s"] = round(n * n / cms / 1e3, 1)
    # the interpolation tail on tile-major taps against the fused tail on [1,51,H,W] taps (gray x3 sections, as config 5 feeds)
    tiled = [pkg.tap_conv3x3(xs[i], packed, bias, upsample=True, tiled=True) for i in range(4)]
    i1, i2 = (torch.rand((1, 1, n, n), device=dev, generator=gen).expand(1, 3, n, n).contiguous() for _ in range(2))
    pkg.set_gray_replicated("assert")
    try:
        tms = _events_ms(lambda: pkg.interpolation_tail_tiled(i1, i2, *tiled), 10, warm=3)
        del frame
        nchw = [pkg.tap_conv3x3(xs[i], packed, bias, upsample=True, tiled=False) for i in range(4)]
        fms = _events_ms(lambda: pkg.interpolation_tail(i1, i2, *nchw), 10, warm=3)
    finally:
        pkg.set_gray_replicated("off")
    res["tail_tiled_taps_ms"] = round(tms, 4)
    res["tail_fused_nchw_taps_ms"] = round(fms, 4)
    res["tail_note"] = ("gray x3 sections: interpolation_tail_tiled = frame_mean_pad x2 + two one-plane persistent forwards on tile-major taps "
                        "(second accumulates); interpolation_tail = the fused generation-1 kernel on [1,51,H,W] taps")
    del tiled, nchw
    del xs, outs
    torch.cuda.empty_cache()
    return res


def run_c5_stack(pkg, dev, rank, world, dist, sections=100, size=4096, to_host=False, tiled_taps=False, producer=False):
    """BASELINE config 5: a synthetic 100-section 4096x4096 stack, 98 targets (k-1, k+1) -> k
    (sff_scripts_interp/inference.py:69-70) through restore_stack: uint8 sections uploaded from pinned host memory
    inside the timed region, fused interpolation tail + flow warp + stitch per target, targets sharded contiguously
    over the ranks (STRONG scaling: the job is fixed), restored uint8 sections gathered to rank 0.  Taps / flow are
    synthetic and reused for every target (the KPN and the flow net are out of scope; their values do not affect speed)."""
    import numpy as np
    import torch
    from sstem_restoration_b200 import shard, synth
    H = W = size
    gen = torch.Generator(device=dev).manual_seed(4321 + rank)
    taps = [torch.softmax(torch.randn((1, K, H, W), device=dev, generator=gen), 1) for _ in range(4)]
    if tiled_taps:                                            # the layout the tap producer writes (DESIGN 4.10 / 4.11): restore_stack then
        taps = [pkg.taps_to_tiled(t) for t in taps]          # takes the tile-major tail
    taps_fn = lambda k, x: taps
    if producer:
        # the four tap branches' last two layers run per target: half-resolution activations (synthetic, fixed) -> tile-major taps
        del taps
        acts = [torch.relu(torch.randn((1, K, H // 2, W // 2), device=dev, generator=gen)) for _ in range(4)]
        prods = [pkg.ModuleTapProducer(tiled=True).to(dev) for _ in range(4)]
        taps = None
        taps_fn = lambda k, x: [m(a) for m, a in zip(prods, acts)]
    flow_np, _ = synth.random_fold_flow(H, W, 555)
    flow = torch.from_numpy(np.ascontiguousarray(flow_np.transpose(2, 0, 1))[None]).to(dev).permute(0, 2, 3, 1)
    tile = synth.em_section(min(H, 1024), min(W, 1024), 0)
    base = torch.from_numpy(np.tile(tile, (H // tile.shape[0], W // tile.shape[1])))
    targets = shard.stack_targets(sections)
    lo, hi = shard.shard_range(len(targets), rank, world)
    stack = torch.empty((sections, H, W), dtype=torch.uint8).pin_memory()
    for k in range(max(lo, 0), min(hi + 2, sections)):       # only the sections this rank touches are materialised
        stack[k] = torch.roll(base, shifts=7 * k, dims=1)
    pkg.set_gray_replicated("assert")                         # sections are gray x3 by construction (inference.py:71-74)
    try:
        kw = dict(rank=rank, world_size=world, dst=0, device=dev, to_host=to_host)
        if to_host:                                            # pinned result buffers exist before the timed region, like the stack
            kw["host_out"] = {n: torch.empty((hi - lo, H, W), dtype=torch.uint8).pin_memory() for n in ("interp", "warped", "stitch")}
        warm = torch.empty((4, H, W), dtype=torch.uint8).pin_memory()
        warm[:] = stack[lo:lo + 4] if hi - lo >= 2 else 0
        pkg.restore_stack(warm, taps_fn, lambda k, xk, interp: flow, rank=0, world_size=1, device=dev)   # warm-up
        # allocator warm-up: blocks of the sizes the timed call will ask for (its three [targets,H,W] outputs, the gathered copies
        # on rank 0) are obtained from the driver now and handed to torch's cache -- the timed region measures the job, not
        # cudaMalloc of gigabytes (which moved config 5 between 84 and 149 sections/s, profiles/c5_order_r2.md)
        pre = [torch.empty((hi - lo, H, W), dtype=torch.uint8, device=dev) for _ in range(3)]
        if world > 1 and not to_host:
            m = shard.max_units_per_rank(len(targets), world)
            if hi - lo < m:                                    # a rank with fewer targets pads its shard for the gather
                pre.append(torch.empty((m, H, W), dtype=torch.uint8, device=dev))
            if rank == 0:                                      # receive buffers [world * m, H, W] and, if ragged, the trimmed copies
                pre += [torch.empty((world * m, H, W), dtype=torch.uint8, device=dev) for _ in range(3)]
                if world * m != len(targets):
                    pre += [torch.empty((len(targets), H, W), dtype=torch.uint8, device=dev) for _ in range(3)]
        del pre
        if world > 1:
            shard.gather_sections(torch.zeros((1, 8, 8), dtype=torch.uint8, device=dev), world, dst=0)             # communicator
        # (no nvidia-smi sampler here: its start-up attaches to the driver and stalls the ~1000 launches / copies of this job --
        #  measured 107 instead of 148 sections/s with it; the headline region above is the one that is sampled)
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        t0 = time.perf_counter()
        e0.record()
        out = pkg.restore_stack(stack, taps_fn, lambda k, xk, interp: flow, **kw)
        e1.record()
        torch.cuda.synchronize()
        wall_ms = (time.perf_counter() - t0) * 1e3
    finally:
        pkg.set_gray_replicated("off")
    ms = torch.tensor([max(e0.elapsed_time(e1), wall_ms if to_host else 0.0)], device=dev, dtype=torch.float64)
    per_rank_ms = [round(float(ms.item()), 2)]
    if dist is not None:
        allms = [torch.zeros_like(ms) for _ in range(world)]
        dist.all_gather(allms, ms)
        per_rank_ms = [round(float(t.item()), 2) for t in allms]
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    sec = float(ms.item()) * 1e-3
    per_rank_max = -(-len(targets) // world)
    st = out["stats"]
    res = {"workload": f"{sections} sections {H}x{W}, {len(targets)} targets", "n_gpus": world, "scaling": "strong",
           "seconds": round(sec, 4), "sections_per_s": round(len(targets) / sec, 2), "mpix_per_s": round(len(targets) * H * W / sec / 1e6, 1),
           "per_rank_ms": per_rank_ms,
           "targets_on_busiest_rank": per_rank_max, "ideal_speedup_at_this_n": round(len(targets) / per_rank_max, 3),
           "ms_per_target_on_busiest_rank": round(sec * 1e3 / per_rank_max, 3),
           "h2d_bytes_rank0": st["h2d_bytes"], "d2h_bytes_rank0": st["d2h_bytes"], "kernel_launches_rank0": st["kernel_launches"],
           "outputs": ("interp, warped, stitch: uint8, each rank downloads its own targets into pinned host memory (one async copy per target, no collective)"
                       if to_host else "interp, warped, stitch: uint8 [98,H,W] each, gathered to rank 0 (device memory)"),
           "taps": ("produced per target by 4 x ModuleTapProducer (upsample x2 + conv 3x3, tcgen05 TF32) from half-resolution activations, tile-major"
                    if producer else "tile-major [1,H/8,W/8,51,8,8] (interpolation_tail_tiled)" if tiled_taps else "[1,51,H,W] (fused interpolation_tail)"),
           "api": "sstem_restoration_b200.restore_stack(stack_u8_pinned, taps_fn, flow_fn, rank, world_size, dst=0)"}
    del taps, taps_fn, flow, stack, out
    # (no empty_cache() here: handing the blocks back makes the NEXT config-5 run cudaMalloc gigabytes inside its timed region --
    #  measured 84 - 161 instead of 148 / 176 sections/s, profiles/c5_order_r2.md; main() frees once after the last variant)
    return res


def run_copy_ceiling(dev, h2d_bytes, d2h_bytes, world, dist, chunks=8, steps=3):
    """What the host link alone allows for the e2e step: the same byte counts, pinned buffers, H2D and D2H running
    concurrently on two streams, no kernels.  -> seconds per step (max over ranks)."""
    import torch
    n_up, n_dn = h2d_bytes // chunks, d2h_bytes // chunks
    hu, hd = torch.empty(n_up, dtype=torch.uint8).pin_memory(), torch.empty(n_dn, dtype=torch.uint8).pin_memory()
    du, dd = torch.empty(n_up, dtype=torch.uint8, device=dev), torch.empty(n_dn, dtype=torch.uint8, device=dev)
    s_up, s_dn = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)

    def step():
        for _ in range(chunks):
            with torch.cuda.stream(s_up):
                du.copy_(hu, non_blocking=True)
            with torch.cuda.stream(s_dn):
                hd.copy_(dd, non_blocking=True)
        s_up.synchronize()
        s_dn.synchronize()
    step()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    t = torch.tensor([dt], device=dev, dtype=torch.float64)
    if dist is not None:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def run_tail(pkg, dev, B, H, W, reps=5):
    """Fused interpolation tail (SURVEY 8f N1) against the unfused expression it replaces, gray x3 frames."""
    import torch
    gen = torch.Generator(device=dev).manual_seed(11)
    f = [torch.rand((B, 1, H, W), device=dev, generator=gen).expand(B, 3, H, W).contiguous() for _ in range(2)]
    taps = [torch.softmax(torch.randn((B, K, H, W), device=dev, generator=gen), 1) for _ in range(4)]
    pad = torch.nn.ReplicationPad2d(K // 2)

    def unfused():
        y = pkg.SeparableConvolution.apply(pad(f[1]), taps[2], taps[3]) + pkg.SeparableConvolution.apply(pad(f[0]), taps[0], taps[1])
        return torch.mean(y, dim=1, keepdim=True)

    def timed(fn):
        for _ in range(2):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    res = {"shape": [B, 3, H, W], "ms_unfused_expression": round(timed(unfused), 4)}
    for mode in ("off", "assert"):
        pkg.set_gray_replicated(mode)
        try:
            ms = timed(lambda: pkg.interpolation_tail(f[0], f[1], *taps))
        finally:
            pkg.set_gray_replicated("off")
        res["ms_fused_gray_" + mode] = round(ms, 4)
        res["mpix_per_s_gray_" + mode] = round(B * H * W / (ms * 1e-3) / 1e6, 1)
    res["note"] = ("interpolation_tail = 2x ReplicationPad2d + 2x sepconv + add + channel mean in one launch "
                   "(model_interp.py:90-97); 816 B of taps per output pixel; NOT the headline")
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=30)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--batch", type=int, default=16)
    ap.add_argument("--size", type=int, default=512)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-warp", action="store_true")
    ap.add_argument("--no-gather", action="store_true", help="diagnostic: skip the output gather at N > 1")
    ap.add_argument("--nccl-gather", action="store_true", help="diagnostic: gather with the NCCL collective instead of copy-engine peer writes")
    ap.add_argument("--no-stack", action="store_true", help="skip BASELINE config 5 (the 100-section stack job)")
    ap.add_argument("--sections", type=int, default=100)
    ap.add_argument("--section-size", type=int, default=4096)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the last step's outputs and tap gradients as DIR/<name>.npy (float32; "
                         "a fixed seeded sample of each when they exceed 60 MB together)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        run_reference_arm(args)
    else:
        run_gpu_arm(args)


if __name__ == "__main__":
    main()
