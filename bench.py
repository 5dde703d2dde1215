#!/usr/bin/env python
"""bench.py — ARTDECO hot-path benchmark (driver contract: one JSON line on stdout from rank 0).

metric   rasterizer fwd+bwd Gpix/s @ 1M splats, 1080p (BASELINE.json `metric`; workload = SURVEY.md §8d
         `raster_scene(1_000_000)`, cameras v = 0..7, dense N(0,1) upstream gradients).
step     ONE OPTIMISER STEP of BASELINE config 4: forward + backward of an 8-VIEW BATCH against the same 1M Gaussians,
         gradients summed over the 8 views.  Per view: project+SH -> tile-bucketed intersection -> blend fwd -> blend bwd;
         then one multi-view projection/SH backward.  value = 8 * 1920*1080 pixels / step time.
N > 1    STRONG scaling of that step: the 8 views are split over the ranks (rank g renders views {v : v mod N = g}), every
         rank holds a replica of the scene, and the per-Gaussian gradients are exchanged once per step
         (parallel.MultiViewExchange: all-gather of the 12 B/view colour gradients + all-reduce of the 11 geometry floats,
         overlapped with the backward kernels) so that every rank ends with the sum over all 8 views.
value    whole-job Gpix/s with inputs resident in HBM, the local compute replayed as one CUDA graph, timed with CUDA events,
         max over ranks.
e2e      same metric through the public operator surface (artdeco_b200.rasterization(C views) + L1 + fused_ssim + autograd):
         per step the cameras and the ground-truth images of the local views come from PINNED HOST memory (H2D inside the
         timed region, prefetched on a copy stream) and the loss is read back (D2H).  Gaussian parameters are optimiser state
         and stay resident, as in the reference (h3dgsv3.py keeps them on device_mapper).
--impl reference   the reference's CPU implementation of the path on the host cores: gsplat has no CPU path and is not
         installable offline, so this arm times the CPU oracle port (oracle/raster_oracle.c, OpenMP, all host threads;
         `cpu_baseline.kind` = "port"), one view of the same batch per step, plus the PyTorch-CPU MASt3R restatement.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
_T0 = time.time()


def log(msg):
    """Progress to stderr (stdout carries exactly one JSON line)."""
    print(f"[bench +{time.time() - _T0:6.1f}s] {msg}", file=sys.stderr, flush=True)


import numpy as np  # noqa: E402
import torch  # noqa: E402

N_GAUSS = 1_000_000
N_VIEWS = 8
W, H = 1920, 1080
KEYS = ("means", "quats", "scales", "opacities", "sh")
METRIC = "rasterizer fwd+bwd Gpix/s @1M splats 1080p"
WORKLOAD = ("raster_scene(1M) 1080p, one optimiser step = fwd+bwd of the 8-view batch (views 0..7, BASELINE config 4), "
            "dense N(0,1) upstream grads, gradients summed over the views")
MAST3R_FLOP_PER_PAIR = 2.806e12   # SURVEY.md §8a (torch FlopCounterMode on the reference module, 512x512)


def _peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            return json.load(f), True
    return {"hbm_gbs": 6650.0, "bf16_tflops_sustained": 1400.0, "sm_max_mhz": 1965.0}, False


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index: int):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--id={index}", f"--query-gpu={q}", "--format=csv,noheader,nounits",
                                       "-lms", "100"], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.p = None

    def stop(self):
        if self.p is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.p.kill()
        self.f.flush()
        self.f.seek(0)
        rows = [r.strip().split(", ") for r in self.f.read().strip().splitlines() if r.strip()]
        os.unlink(self.f.name)
        sm, smax, reasons = [], None, set()
        for r in rows:
            if len(r) < 7:
                continue
            try:
                sm.append(float(r[0]))
                smax = float(r[1])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                if v.strip().lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": smax, "reasons": sorted(reasons),
                "samples": len(sm)}


def host_threads() -> int:
    """Usable host cores for the CPU legs: min(affinity mask, cgroup CPU quota, physical cores).  Oversubscribing (e.g. one
    thread per logical CPU of a box the container may only use a quarter of) makes OpenMP spin-wait and costs 5-15x."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    try:
        import psutil
        phys = psutil.cpu_count(logical=False)
        if phys:
            n = min(n, phys)
    except Exception:  # noqa: BLE001
        pass
    try:
        with open("/sys/fs/cgroup/cpu.max") as f:
            quota, period = f.read().split()[:2]
        if quota != "max":
            n = min(n, max(1, int(int(quota) / int(period))))
    except Exception:  # noqa: BLE001
        pass
    return max(1, n)


def cpu_thread_setup():
    """Leaves the default thread counts alone unless the launcher restricted them (torchrun exports OMP_NUM_THREADS=1)."""
    want = host_threads()
    if torch.get_num_threads() < max(2, want // 2):
        torch.set_num_threads(want)
    return want


def cpu_oracle_leg(steps: int, warmup: int, n: int, views):
    """Times the CPU oracle's fwd+bwd (one view per step, cycling through `views`) on the host cores.
    Returns (Gpix/s, seconds/step, n_isect of the last view, threads)."""
    import oracle
    from artdeco_b200 import synthetic
    want = cpu_thread_setup()
    threads = oracle.num_threads()
    if threads < max(2, want // 2):
        threads = oracle.set_num_threads(want)
    sc = synthetic.raster_scene(n, seed=0)
    args = [sc[k].numpy() for k in KEYS]
    ts = []
    n_isect = 0
    for i in range(warmup + steps):
        view = float(views[i % len(views)])
        V, K = synthetic.camera(W, H, view=view)
        vc, va = synthetic.upstream_grads(W, H, seed=1 + int(view))
        vcn, van = vc[0].numpy(), va[0, ..., 0].numpy()
        t0 = time.perf_counter()
        f = oracle.rasterize_fwd(*args, V.numpy(), K.numpy(), W, H)
        oracle.rasterize_bwd(*args, V.numpy(), f, vcn, van)
        dt = time.perf_counter() - t0
        n_isect = len(f["keys"])
        if i >= warmup:
            ts.append(dt)
    sec = float(np.mean(ts))
    return W * H / sec / 1e9, sec, n_isect, threads


def cpu_mast3r_leg(passes: int = 3):
    """PyTorch-CPU restatement of the reference model (oracle/mast3r_torch.py), 1 warm-up + `passes` timed 512x512 pairs,
    median (BASELINE.md plan), all host threads."""
    from artdeco_b200.mast3r import FULL_CFG
    from artdeco_b200.mast3r.shapes import random_state_dict
    from oracle import mast3r_torch as mt
    cpu_thread_setup()
    sd_cpu = random_state_dict(FULL_CFG, "cpu", seed=0)
    g = torch.Generator().manual_seed(100)
    i1 = torch.rand(1, 3, 512, 512, generator=g) * 2 - 1
    i2 = torch.rand(1, 3, 512, 512, generator=g) * 2 - 1
    ts = []
    with torch.inference_mode():
        for i in range(1 + passes):
            t0 = time.perf_counter()
            mt.forward_pair(sd_cpu, FULL_CFG, i1, i2)
            if i:
                ts.append(time.perf_counter() - t0)
    sec = float(np.median(ts))
    return {"value": 1.0 / sec, "unit": "pairs/s", "cores": torch.get_num_threads(), "kind": "port",
            "sample": f"1 warm-up + {passes} timed 512x512 pairs through oracle/mast3r_torch.py (PyTorch CPU fp32, all host "
                      "threads), median", "seconds_per_pair": sec, "seconds_all": ts}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    steps, warm = max(1, args.steps), max(1, args.warmup)
    gpix, sec, n_isect, threads = cpu_oracle_leg(steps, warm, N_GAUSS, list(range(N_VIEWS)))
    line = {
        "impl": "reference", "metric": METRIC, "value": gpix, "unit": "Gpix/s", "n_gpus": args.gpus, "steps": steps,
        "warmup": warm, "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
        "dtype": "f32", "data": "synthetic",
        "config": {"workload": WORKLOAD, "n_gaussians": N_GAUSS, "width": W, "height": H, "n_views": N_VIEWS,
                   "n_isect_last_view": n_isect, "sh_degree": 3, "eps2d": 0.01,
                   "note": "gsplat (the live reference renderer) is an un-vendored pip dependency with no CPU path; this arm "
                           "times the CPU oracle port with all host threads; each step is a bounded sample of the 8-view "
                           "batch: ONE view's fwd+bwd (views cycle 0..7), same Gpix/s unit"},
        "cpu_baseline": {"value": gpix, "unit": "Gpix/s", "cores": threads, "kind": "port",
                         "sample": f"{steps} single-view fwd+bwd passes (views cycling 0..7) of the 1M/1080p workload"},
        "e2e": {"value": gpix, "unit": "Gpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    if not args.no_mast3r:
        log("reference arm: PyTorch-CPU MASt3R (1 + 3 pairs)")
        m = cpu_mast3r_leg(3)
        line["mast3r"] = {"impl": "reference", "metric": "MASt3R pairs/s @512^2", "value": m["value"], "unit": "pairs/s",
                          "ms_per_step": m["seconds_per_pair"] * 1e3, "cpu_baseline": m,
                          "e2e": {"value": m["value"], "unit": "pairs/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


class Watchdog:
    """Fires ``on_fire`` from a timer thread unless cancelled first.  A device-side hang cannot be recovered in-process
    (synchronize never returns), so the callback is expected to print what has already been measured and ``os._exit``."""

    def __init__(self, seconds: float, on_fire):
        import threading
        self._t = threading.Timer(seconds, on_fire)
        self._t.daemon = True

    def start(self):
        self._t.start()
        return self

    def cancel(self):
        self._t.cancel()


def timed(fn, steps, warmup, dev, world):
    """W warm-up calls, then K calls between CUDA events, barrier + synchronize on both sides, max over ranks."""
    import torch.distributed as dist
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(steps):
        fn()
    b.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    ms = torch.tensor([a.elapsed_time(b)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    return float(ms) / steps


DUMP_GAUSSIANS = 65536      # gradient rows sampled per parameter (59 floats each: 15.5 MB)
DUMP_PIXELS = 262144        # pixels sampled over the local views (colour+depth and alpha: 5.2 MB)


def dump_outputs(out_dir, engine):
    """Writes what ``engine.step()`` computed in its last call as float32 ``<name>.npy``: the gradients it returns, summed
    over the views (v_means, v_quats, v_scales, v_opac, v_sh), for a fixed seeded sample of the Gaussians, and the local
    views' render (colors [.., 4] = RGB + depth, alphas) for a fixed seeded sample of their pixels.  The samples depend only
    on the sizes, so two builds of the project can be compared array for array."""
    os.makedirs(out_dir, exist_ok=True)
    g = torch.Generator().manual_seed(0)
    rows = torch.randperm(engine.N, generator=g)[:DUMP_GAUSSIANS].sort().values.to(engine.dev)
    for name in ("v_means", "v_quats", "v_scales", "v_opac", "v_sh"):
        np.save(os.path.join(out_dir, f"{name}.npy"), engine.grads[name][rows].float().cpu().numpy())
    cols, alps = engine.render
    pix = torch.randperm(len(cols) * H * W, generator=g)[:DUMP_PIXELS].sort().values.to(engine.dev)
    np.save(os.path.join(out_dir, "colors.npy"), torch.stack(cols).reshape(-1, 4)[pix].cpu().numpy())
    np.save(os.path.join(out_dir, "alphas.npy"), torch.stack(alps).reshape(-1)[pix].cpu().numpy())


def event_ms(fn, reps, warmup=3):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(reps):
        fn()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / reps


def bench_mast3r(dev, world, rank, steps, warmup, want_baselines):
    """MASt3R pair inference (2x _encode_image + _decoder + 2x _downstream_head) at 512x512, B pairs per GPU per step;
    pairs are split across GPUs with no collective (SURVEY.md §8e)."""
    from artdeco_b200 import _lib
    from artdeco_b200.mast3r import BENCH_PAIRS_PER_GPU, FULL_CFG, AsymmetricMASt3R, GraphedForwardPair, forward_pair
    from artdeco_b200.mast3r.shapes import random_state_dict
    B = int(os.environ.get("ADB_MAST3R_B", str(BENCH_PAIRS_PER_GPU)))
    sd = random_state_dict(FULL_CFG, dev, seed=0)
    model = AsymmetricMASt3R(precision="bf16x3", **FULL_CFG).load_state_dict(sd).to(dev)
    g = torch.Generator().manual_seed(100 + rank)
    h1 = (torch.rand(B, 3, 512, 512, generator=g) * 2 - 1).pin_memory()
    h2 = (torch.rand(B, 3, 512, 512, generator=g) * 2 - 1).pin_memory()
    d1, d2 = h1.to(dev), h2.to(dev)
    out_host = [torch.empty(B, 512, 512, 4).pin_memory() for _ in range(2)]

    graphed = GraphedForwardPair(model, B, 512, 512)     # one CUDA graph replay per step (two streams)

    def step():
        graphed(d1, d2)

    def e2e_step():
        r1, r2 = graphed(h1, h2)                          # H2D copies of both image batches from pinned host memory
        for o, r in zip(out_host, (r1, r2)):
            o[..., :3].copy_(r["pts3d"], non_blocking=True)
            o[..., 3].copy_(r["conf"], non_blocking=True)

    log("mast3r model resident; timing")
    k = max(3, min(steps, 10))
    ms = timed(step, k, max(3, warmup), dev, world)
    ms_e2e = timed(e2e_step, k, 3, dev, world)
    # B = 1: the Frontend's per-frame latency (VSLAM/CameraTracker.py:59-61 runs one pair per tracked frame)
    graphed1 = GraphedForwardPair(model, 1, 512, 512)
    ms_b1 = timed(lambda: graphed1(d1[:1], d2[:1]), k, 3, dev, world)
    del graphed1
    # live duration of the tensor-core kernels over one step (eager, single stream: event times are not inflated by overlap)
    for name in ("adb_gemm_bf16", "adb_gemm_bf16_rope", "adb_conv3x3_bf16", "adb_attention_bf16", "adb_layernorm", "adb_split_bf16",
                 "adb_rope_heads", "adb_softmax_rows", "adb_im2col_patch16", "adb_upsample2x_nhwc", "adb_head_postprocess"):
        _lib.LAUNCHES.setdefault(name, 1)
    _lib.TIMER = _lib.StageTimer()
    model.concurrent = False
    forward_pair(model, d1, d2)
    torch.cuda.synchronize()
    model.concurrent = True
    tot = _lib.TIMER.totals_ms()
    launches = _lib.TIMER.launches
    _lib.TIMER = None
    gemm_ms = sum(tot.get(n, (0.0, 0))[0] for n in ("adb_gemm_bf16", "adb_gemm_bf16_rope", "adb_conv3x3_bf16", "adb_attention_bf16"))
    pairs_s = world * B / (ms * 1e-3)
    peaks, measured = _peaks()
    peak_tf = float(peaks.get("bf16_tflops_sustained", 1400.0))
    peak_src = "measured (MEASURED_PEAKS.json bf16_tflops_sustained)" if measured else "fallback (B200_PROFILING.md ~1.4 PFLOP/s sustained)"
    algo_tf = MAST3R_FLOP_PER_PAIR * B / (gemm_ms * 1e-3) / 1e12          # over the GEMM kernels' own time
    traffic = None
    prof = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(prof):
        try:
            with open(prof) as f:
                traffic = json.load(f).get("gemm_tc_kernel")
        except Exception:  # noqa: BLE001
            pass
    res = {
        "metric": "MASt3R pairs/s @512^2", "value": pairs_s, "unit": "pairs/s", "ms_per_step": ms, "pairs_per_gpu_per_step": B,
        "b1_latency_ms": ms_b1, "b1_pairs_per_s": world / (ms_b1 * 1e-3),
        "precision": "bf16x3 (3 tcgen05 MMAs per product: fp32-class accuracy, 1e-4 pointmap tolerance)",
        "e2e": {"value": world * B / (ms_e2e * 1e-3), "unit": "pairs/s", "ms_per_step": ms_e2e,
                "h2d_bytes_per_step": 2 * h1.numel() * 4, "d2h_bytes_per_step": 2 * out_host[0].numel() * 4,
                "what": "two image batches from pinned host memory -> forward_pair -> pts3d+conf of both views copied back"},
        "gpu_launches": launches,
        "roofline": {"bound": "tensor", "kernel": "gemm_tc_kernel + attn_fused_kernel (tcgen05 GEMM / implicit-GEMM conv / fused attention)",
                     "achieved": algo_tf, "peak": peak_tf, "unit": "TFLOP/s", "frac": algo_tf / peak_tf,
                     "tensor_work_achieved": 3 * algo_tf, "tensor_work_frac": 3 * algo_tf / peak_tf,
                     "peak_source": peak_src, "traffic": traffic, "kernel_ms_per_step": gemm_ms,
                     "note": "achieved = 2.806 TFLOP/pair algorithmic FLOPs / live GEMM-kernel time; bf16x3 issues 3x that "
                             "many tensor FLOPs (tensor_work_*), which is what the pipe actually sustains",
                     "whole_step": {"achieved": MAST3R_FLOP_PER_PAIR * B / (ms * 1e-3) / 1e12,
                                    "frac": MAST3R_FLOP_PER_PAIR * B / (ms * 1e-3) / 1e12 / peak_tf},
                     "stage_ms": {k2.replace("adb_", ""): v[0] for k2, v in tot.items()}},
    }
    if want_baselines and rank == 0:
        # the reference's own GPU mode on this box: torch eager fp32 with TF32 matmuls (croco.py:13 sets allow_tf32), same batch
        log("mast3r: reference GPU mode (torch eager fp32+TF32 restatement) on the same B200")
        try:
            from oracle import mast3r_torch as mt
            prev = torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32
            torch.backends.cuda.matmul.allow_tf32 = torch.backends.cudnn.allow_tf32 = True
            with torch.inference_mode():
                ms_ref = event_ms(lambda: mt.forward_pair(sd, FULL_CFG, d1, d2), 3, 2)
                ms_ref1 = event_ms(lambda: mt.forward_pair(sd, FULL_CFG, d1[:1], d2[:1]), 3, 2)
            torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.allow_tf32 = prev
            res["gpu_reference"] = {"what": "oracle/mast3r_torch.forward_pair (the reference model restated op for op) in torch "
                                            "eager fp32+TF32 on the same GPU — the reference's own GPU mode (croco.py:13)",
                                    "batch": B, "ms_per_step": ms_ref, "pairs_per_s": B / (ms_ref * 1e-3), "b1_latency_ms": ms_ref1,
                                    "speedup_batched": ms_ref / ms, "speedup_b1": ms_ref1 / ms_b1}
        except Exception as e:  # noqa: BLE001
            res["gpu_reference"] = {"error": repr(e)[:200]}
    del graphed, model, sd
    torch.cuda.empty_cache()
    if want_baselines and rank == 0:
        log("mast3r GPU legs done; timing the CPU restatement (PyTorch fp32, 1 + 3 pairs)")
        res["cpu_baseline"] = cpu_mast3r_leg(3)
    return res


def bench_ops(dev):
    """Roofline fractions of the other operators on the path (SURVEY.md §8d algorithmic bytes), each timed alone with CUDA
    events, next to the reference's own CUDA build (oracle/_ref) where one exists on this box."""
    from artdeco_b200 import synthetic
    from artdeco_b200.adam import adamUpdate
    from artdeco_b200.cull import lod_select
    from artdeco_b200.knn import distCUDA2
    from artdeco_b200.ssim import fused_ssim
    peaks, _ = _peaks()
    hbm = float(peaks["hbm_gbs"])
    out = {}
    try:
        a, b = synthetic.ssim_pair(1, 3, H, W, seed=0)
        a, b = a.to(dev).requires_grad_(True), b.to(dev)

        def ssim_step():
            a.grad = None
            fused_ssim(a, b).backward()
        ms = event_ms(ssim_step, 20)
        by = 52 * 3 * W * H
        out["fused_ssim_fwd_bwd_1x3x1080p"] = {"ms": ms, "algorithmic_bytes": by, "GBps": by / ms / 1e6, "frac_hbm": by / ms / 1e6 / hbm}
        try:
            from oracle import build_ref
            rb = build_ref.load("fused_ssim_ref")
            C1, C2 = 0.01 ** 2, 0.03 ** 2
            up = torch.full_like(b, 1.0 / b.numel())

            def ref_step():
                m, d1, d2, d3 = rb.fusedssim(C1, C2, a.detach(), b, True)
                m.mean()
                rb.fusedssim_backward(C1, C2, a.detach(), b, up, d1, d2, d3)
            ms_r = event_ms(ref_step, 20)
            out["fused_ssim_fwd_bwd_1x3x1080p"].update(reference_build_ms=ms_r, speedup_vs_reference_build=ms_r / ms)
        except Exception as e:  # noqa: BLE001
            out["fused_ssim_fwd_bwd_1x3x1080p"]["reference_build"] = f"unavailable: {repr(e)[:120]}"
        sc = synthetic.raster_scene(N_GAUSS, seed=0)
        pts = sc["means"].to(dev)
        ms = event_ms(lambda: distCUDA2(pts), 10)
        by = N_GAUSS * (12 + 16 + 12 + 4)
        out["distCUDA2_1M"] = {"ms": ms, "algorithmic_bytes": by, "GBps": by / ms / 1e6, "frac_hbm": by / ms / 1e6 / hbm}
        try:
            from oracle import build_ref
            rk = build_ref.load("simple_knn_ref")
            ms_r = event_ms(lambda: rk.distCUDA2(pts), 3, 1)
            out["distCUDA2_1M"].update(reference_build_ms=ms_r, speedup_vs_reference_build=ms_r / ms)
        except Exception as e:  # noqa: BLE001
            out["distCUDA2_1M"]["reference_build"] = f"unavailable: {repr(e)[:120]}"
        M = 59
        prm, grd = torch.randn(N_GAUSS, M, device=dev), torch.randn(N_GAUSS, M, device=dev)
        m1, m2 = torch.zeros_like(prm), torch.zeros_like(prm)
        vis = torch.ones(N_GAUSS, dtype=torch.bool, device=dev)
        lr = torch.tensor(1e-3, device=dev)
        ms = event_ms(lambda: adamUpdate(prm, grd, m1, m2, vis, lr, 0.5, 0.99, 1e-15, N_GAUSS, M), 20)
        by = N_GAUSS * M * 28
        out["adamUpdate_1Mx59"] = {"ms": ms, "algorithmic_bytes": by, "GBps": by / ms / 1e6, "frac_hbm": by / ms / 1e6 / hbm}
        dmax = sc["d_max"].to(dev)
        cam = torch.zeros(3, device=dev)
        ms = event_ms(lambda: lod_select(pts, dmax, cam), 20)
        by = N_GAUSS * 16
        out["lod_select_1M"] = {"ms": ms, "algorithmic_bytes": by, "GBps": by / ms / 1e6, "frac_hbm": by / ms / 1e6 / hbm}
        # global Gauss-Newton on a loop-closure-sized graph: 32 key frames, 128 two-way edges, 512x384 pointmaps, 5 iterations
        from artdeco_b200 import gn
        g = torch.Generator().manual_seed(0)
        Kp, n, E = 32, 512 * 384, 128
        T = torch.zeros(Kp, 8)
        T[:, 6] = 1.0
        T[:, 7] = 1.0
        T[:, :3] = torch.randn(Kp, 3, generator=g) * 0.1
        Xg = (torch.randn(Kp, n, 3, generator=g) + torch.tensor([0.0, 0.0, 4.0])).to(dev)
        Cg, Qg = (torch.rand(Kp, n, 1, generator=g) + 1).to(dev), (torch.rand(E, n, 1, generator=g) + 1).to(dev)
        ei = torch.randint(0, Kp, (E,), generator=g)
        ej = (ei + 1 + torch.randint(0, Kp - 1, (E,), generator=g)) % Kp
        idxg = torch.randint(0, n, (E, n), generator=g).to(dev)
        vmg = (torch.rand(E, n, 1, generator=g) > 0.3).to(dev)
        Td = T.to(dev)

        def gn_step():
            gn.gauss_newton_rays(Td.clone(), Xg, Cg, ei.to(dev), ej.to(dev), idxg, vmg, Qg, 0.003, 10.0, 0.0, 1.5, 5, 0.0)
        ms = event_ms(gn_step, 5, 2)
        by = 5 * E * n * (12 + 12 + 4 + 4 + 8 + 1 + 4)
        out["gauss_newton_rays_32kf_128edges_5it"] = {"ms": ms, "ms_per_iteration": ms / 5, "algorithmic_bytes": by,
                                                       "GBps": by / ms / 1e6, "frac_hbm": by / ms / 1e6 / hbm,
                                                       "note": "whole solve on the device (normal equations + dense double "
                                                               "Cholesky of 217 unknowns + retraction), no host sync; the "
                                                               "reference copies the blocks to the host and factorises with "
                                                               "Eigen every iteration (its extension needs Eigen: not buildable here)"}
    except Exception as e:  # noqa: BLE001
        out["error"] = repr(e)[:300]
    torch.cuda.empty_cache()
    return out


def bench_config5(dev, world, rank):
    """BASELINE config 5 (SURVEY.md §8d/§8e): raster_scene(10M) with the LoD d_max cull INSIDE the timed call, 4k evaluation
    render (forward only, as the reference's evaluation renders are), one view per GPU (replicas by view, no collective)."""
    import torch.distributed as dist
    from artdeco_b200 import synthetic
    from artdeco_b200.scene import render_lod
    N5, W5, H5 = 10_000_000, 3840, 2160
    sc = synthetic.raster_scene(N5, seed=0)
    V, K = synthetic.camera(W5, H5, view=float(rank % 8))
    kw = dict(xyz=sc["means"].to(dev), opacity=sc["opacities"][:, None].to(dev), f_dc=sc["sh"][:, :1].contiguous().to(dev),
              f_rest=sc["sh"][:, 1:].contiguous().to(dev), scaling=sc["scales"].to(dev), rotation=sc["quats"].to(dev),
              d_max=sc["d_max"].to(dev), tanfovx=W5 / (2 * float(K[0, 0])), tanfovy=H5 / (2 * float(K[1, 1])), sh_degree=3,
              eps2d=0.01)
    del sc
    Vd = V.to(dev)
    info = {}

    def step():
        with torch.no_grad():
            pkg = render_lod(W5, H5, Vd, **kw)
        info.update(n_selected=pkg["n_selected"], n_isect=pkg["n_isect"])
    ms = timed(step, 5, 3, dev, world)
    res = {"workload": "raster_scene(10M) + d_max ~ U(4,40), LoD cull inside the call, 3840x2160 forward render, one view per GPU",
           "ms_per_render": ms, "value": world * W5 * H5 / (ms * 1e-3) / 1e9, "unit": "Gpix/s (forward only)",
           "n_gaussians": N5, "n_selected": info["n_selected"], "n_isect": info["n_isect"],
           "host_syncs_per_render": 2, "note": "public path: lod_select count + intersection count are read back (as gsplat does)"}
    del kw
    torch.cuda.empty_cache()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-mast3r", action="store_true")
    ap.add_argument("--no-extra", action="store_true", help="skip the config-3 stream and config-5 legs")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (rank 0, sampled)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    import torch.distributed as dist
    from artdeco_b200 import _lib, synthetic
    from artdeco_b200 import raster as R
    from artdeco_b200.multiview import MultiViewStep
    from artdeco_b200.parallel import views_for_rank
    from artdeco_b200.ssim import fused_ssim

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device; there is no CPU fallback (use --impl reference for the CPU oracle)")
    if N_VIEWS % world:
        raise SystemExit(f"--gpus must divide the {N_VIEWS}-view batch")
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=dev)

    views = views_for_rank(N_VIEWS, world, rank)
    Cl = len(views)
    sc = synthetic.raster_scene(N_GAUSS, seed=0)
    t = {k: sc[k].to(dev) for k in KEYS}
    cams = [synthetic.camera(W, H, view=float(v)) for v in views]
    Vs = torch.stack([c[0] for c in cams]).to(dev)
    Ks = torch.stack([c[1] for c in cams]).to(dev)
    engine = MultiViewStep(t, Vs, Ks, W, H, world=world)
    for j, v in enumerate(views):
        vc, va = synthetic.upstream_grads(W, H, seed=1 + v)
        engine.v_colors[j].copy_(vc[0])
        engine.v_alphas[j].copy_(va[0, ..., 0])
    n_isect_local = engine.calibrate()
    log(f"raster scene resident; local views {views}, n_isect {n_isect_local}; timing device-resident steps")
    sampler = ClockSampler(local_rank) if rank == 0 else None
    ms_step = timed(engine.step, args.steps, args.warmup, dev, world)
    n_isect_local = engine.check_overflow()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, engine)     # before the stage-timing steps below overwrite the buffers

    # per-stage live timing + launch count over K more steps, eager (CUDA events on the launching stream)
    engine.use_graph = False
    ov, engine.overlap_views = engine.overlap_views, False     # one stream: per-kernel event times are not inflated by overlap
    _lib.TIMER = _lib.StageTimer()
    k_stage = max(2, min(args.steps, 5))
    for _ in range(k_stage):
        engine.step()
    torch.cuda.synchronize()
    tot = _lib.TIMER.totals_ms()
    launches = _lib.TIMER.launches // k_stage * args.steps     # launches inside the timed region (graph replays the same nodes)
    _lib.TIMER = None
    engine.use_graph = True
    engine.overlap_views = ov
    # per LAUNCH; the *_hits entry points are the same blend kernels sharing their culling decisions (one byte per intersection)
    short = lambda k: k.replace("adb_raster_", "").replace("_hits", "")  # noqa: E731
    stage_ms = {short(k): v[0] / v[1] for k, v in tot.items()}
    stage_calls = {short(k): v[1] // k_stage for k, v in tot.items()}

    # the exchange alone (world > 1): time and achieved bus bandwidth of the two collectives on the real buffers
    collective = None
    if world > 1:
        ex = engine.exchange
        g_loc = engine.grads["g_rgb"]

        def comm_only():
            ex.start_gather(g_loc, engine.P)
            ex.start_reduce()
            ex.wait_gather()
            ex.wait_reduce()
        ms_comm = timed(comm_only, 10, 3, dev, world)
        moved = (world - 1) / world * (N_VIEWS * N_GAUSS * 12) + 2 * (world - 1) / world * N_GAUSS * 44
        peer = type(ex).__name__ == "PeerExchange"
        if peer:
            ex.check()
        collective = {"ms": ms_comm, "impl": ("own kernels over NVLink peer memory (csrc/peer_exchange.cu): masked colour rows stored into "
                                             "every rank's table; reduce-scatter by push + owner sum + broadcast; release/acquire "
                                             "step counters") if peer else "NCCL all_gather_into_tensor + all_reduce",
                      "bytes_all_gather_total": N_VIEWS * N_GAUSS * 12, "bytes_all_reduce_payload": N_GAUSS * 44,
                      "bus_GBps": moved / ms_comm / 1e6,
                      "dense_all_reduce_payload_replaced": N_GAUSS * 59 * 4,
                      "what": "gather of g_rgb [views,N,3] + sum of [N,11] over ranks issued together, timed alone; inside "
                              "the step both overlap the backward kernels"}
    n_isect_all = n_isect_local
    if world > 1:
        gathered = [None] * world
        dist.all_gather_object(gathered, list(zip(views, n_isect_local)))
        n_isect_all = [n for _, n in sorted(sum(gathered, []))]

    log(f"raster value leg done: {ms_step:.3f} ms/step ({Cl} local views)")
    # ---- e2e through the public operator surface, host buffers for the per-step inputs ----
    gt_host = torch.rand(Cl, H, W, 3, generator=torch.Generator().manual_seed(2 + rank)).pin_memory()
    V_host, K_host = Vs.cpu().pin_memory(), Ks.cpu().pin_memory()
    params = {k: t[k].clone().requires_grad_(True) for k in KEYS}
    loss_host = torch.empty((), dtype=torch.float32).pin_memory()
    h2d = gt_host.numel() * 4 + Cl * (16 + 9) * 4
    d2h = 8
    copy_stream = torch.cuda.Stream(device=dev)
    gt_buf = [torch.empty(Cl, H, W, 3, device=dev) for _ in range(2)]
    copied = [torch.cuda.Event() for _ in range(2)]
    used = [torch.cuda.Event() for _ in range(2)]
    state = {"i": 0}

    def prefetch(slot):
        copy_stream.wait_event(used[slot])           # the step that last read this buffer has finished with it
        with torch.cuda.stream(copy_stream):
            gt_buf[slot].copy_(gt_host, non_blocking=True)
            copied[slot].record(copy_stream)

    for slot in range(2):
        used[slot].record()
    prefetch(0)
    exchange = engine.exchange
    caps = list(engine.capacity)
    flag_host = torch.zeros(1, dtype=torch.int32).pin_memory()

    def e2e_step():
        i = state["i"]
        state["i"] = i + 1
        prefetch((i + 1) % 2)                        # next step's images, overlapped with this step's kernels
        torch.cuda.current_stream().wait_event(copied[i % 2])
        gt = gt_buf[i % 2]
        Ve = V_host.to(dev, non_blocking=True).requires_grad_(True)
        Ke = K_host.to(dev, non_blocking=True)
        for p in params.values():
            p.grad = None
        colors, alphas, meta = R.rasterization(params["means"], params["quats"], params["scales"], params["opacities"],
                                               params["sh"], Ve, Ke, W, H, render_mode="RGB+D", sh_degree=3, eps2d=0.01,
                                               grad_exchange=exchange, isect_capacity=caps)
        img = colors[..., :3]
        l1 = (img - gt).abs().mean()
        ssim = fused_ssim(img.permute(0, 3, 1, 2), gt.permute(0, 3, 1, 2))
        loss = 0.8 * l1 + 0.2 * (1.0 - ssim) + 0.01 * colors[..., 3].mean() + 0.01 * alphas.mean()
        loss.backward()
        used[i % 2].record()
        loss_host.copy_(loss.detach(), non_blocking=True)
        flag_host.copy_(meta["isect_overflow"], non_blocking=True)      # read back with the loss: no extra sync

    e2e_steps = max(3, min(args.steps, 10))
    ms_e2e = timed(e2e_step, e2e_steps, 3, dev, world)
    if int(flag_host):
        raise SystemExit("e2e leg: intersection capacity exceeded")
    log(f"raster e2e leg done: {ms_e2e:.3f} ms/step")

    P = W * H
    gpix = N_VIEWS * P / (ms_step * 1e-3) / 1e9
    gpix_e2e = N_VIEWS * P / (ms_e2e * 1e-3) / 1e9
    peaks, measured = _peaks()
    peak = float(peaks["hbm_gbs"])
    peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)" if measured else "fallback (B200_PROFILING.md 6.65 TB/s)"
    I_mean = float(np.mean(n_isect_all))
    I_loc = float(np.mean(n_isect_local))
    # algorithmic bytes (SURVEY.md §8d): per view 568N + 112I + 68P; dominant kernel = blend_bwd: 44I + 44P per launch
    step_bytes = N_VIEWS * (568 * N_GAUSS + 68 * P) + 112 * float(np.sum(n_isect_all))
    per_launch_bytes = {"project_fwd": 284 * N_GAUSS, "project_fwd_counts": 284 * N_GAUSS, "tile_count_scan": 16 * N_GAUSS, "tile_scatter_sort": 16 * N_GAUSS + 28 * I_loc,
                        "blend_fwd": 44 * I_loc + 24 * P, "blend_bwd": 44 * I_loc + 44 * P,
                        "project_bwd_multi": N_GAUSS * (40 + 44 + Cl * 104), "sh_bwd_multi": N_GAUSS * (204 + 204 + N_VIEWS * 12),
                        "sh_dir_bwd_multi": N_GAUSS * (204 + 24 + Cl * 48), "sh_expand_multi": N_GAUSS * (12 + 192 + N_VIEWS * 12)}
    dom = max((k for k in stage_ms if k in per_launch_bytes), key=lambda k: stage_ms[k] * stage_calls.get(k, 1))
    dom_gbs = per_launch_bytes[dom] / (stage_ms[dom] * 1e-3) / 1e9
    # secondary bound (SURVEY.md §7.4/§8d): FP32 issue.  No-cull model: 256 pixel-threads x I splats x (25 FLOP + 1 MUFU)
    # forward, 2.5x that backward, at 4 warp-instructions per clock per SM; the kernels beat it because warp-level culling
    # never evaluates most (pixel, splat) pairs.
    sm_mhz = float(peaks.get("sm_max_mhz", 1965.0))
    issue_rate = 148 * 4 * sm_mhz * 1e6                       # warp-instructions / s
    fwd_issue_ms = 8 * I_loc * 26 / issue_rate * 1e3
    issue = {"model": "256 px x I x (25 FLOP + 1 MUFU) / 32 lanes at 148 SM x 4 issue/clk (no culling)", "sm_mhz": sm_mhz,
             "blend_fwd_bound_ms": fwd_issue_ms, "blend_bwd_bound_ms": 2.5 * fwd_issue_ms,
             "blend_fwd_measured_ms": stage_ms.get("blend_fwd"), "blend_bwd_measured_ms": stage_ms.get("blend_bwd")}
    roofline = {"bound": "hbm", "kernel": dom, "achieved": dom_gbs, "peak": peak, "unit": "GB/s",
                "frac": dom_gbs / peak, "traffic": None, "peak_source": peak_src,
                "algorithmic_bytes_per_launch": per_launch_bytes[dom], "launch_ms": stage_ms[dom],
                "launches_per_step": stage_calls.get(dom),
                "step": {"algorithmic_bytes": step_bytes, "achieved": step_bytes / world / (ms_step * 1e-3) / 1e9,
                         "frac": step_bytes / world / (ms_step * 1e-3) / 1e9 / peak,
                         "note": "per GPU: the batch's algorithmic bytes / ranks / step time"},
                "fp32_issue_bound": issue,
                "stage_ms_per_launch": stage_ms, "stage_launches_per_step": stage_calls}
    prof = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(prof):
        try:
            with open(prof) as f:
                roofline["traffic"] = json.load(f).get(dom)
        except Exception:  # noqa: BLE001
            pass

    # free the rasterizer's working set before the other legs
    del params, t, engine, exchange, gt_buf
    torch.cuda.empty_cache()
    ops = bench_ops(dev) if (world == 1 and not args.no_cpu_baseline) else None
    config5 = config3 = None
    if not args.no_extra:
        try:
            log("config 5: 10M Gaussians, LoD cull, 4k render")
            config5 = bench_config5(dev, world, rank)
        except Exception as e:  # noqa: BLE001
            config5 = {"error": repr(e)[:300]}
            torch.cuda.empty_cache()
        if world == 1 and not args.no_mast3r:
            try:
                log("config 3: synthetic stream (Frontend + mapper sharing the GPU)")
                from artdeco_b200 import stream
                config3 = stream.run(dev, frames=30, keyframe_every=5, grow=40000, mapper_iters=2)
            except Exception as e:  # noqa: BLE001
                config3 = {"error": repr(e)[:300]}
            torch.cuda.empty_cache()

    def make_line(mast3r, clocks):
        return {
            "metric": METRIC, "value": gpix, "unit": "Gpix/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32",
            "data": "synthetic",
            "config": {"workload": WORKLOAD, "n_gaussians": N_GAUSS, "width": W, "height": H, "n_views": N_VIEWS,
                       "views_per_gpu": Cl, "n_isect_per_view": n_isect_all, "n_isect_mean": I_mean, "sh_degree": 3, "eps2d": 0.01,
                       "l2": "working set per step (params 236 MB + per-view records/keys/accumulators ~150 MB x views + grads "
                             "236 MB) exceeds the 126 MB L2; no explicit flush",
                       "parallelism": f"view-parallel dp{world}: 8-view batch split over ranks, one gradient exchange per step"
                                      + (" (all-gather 12 B/view colour grads + all-reduce [N,11], overlapped)" if world > 1 else ""),
                       "graph": "local compute of the value leg replayed as one CUDA graph (no host sync inside the step)"},
            "clocks": clocks,
            "e2e": {"value": gpix_e2e, "unit": "Gpix/s", "ms_per_step": ms_e2e, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h,
                    "what": "rasterization(C local views, isect_capacity=...: no host sync)+L1+fused_ssim loss+backward via autograd (+ gradient exchange); per step: "
                            "the local views' gt images (prefetched on a copy stream, double-buffered) + cameras from pinned host "
                            "memory, loss + overflow flag read back"},
            "gpu_launches": launches,
            "roofline": roofline,
            "collective": collective,
            "ops": ops,
            "config5_lod_4k": config5,
            "config3_stream": config3,
            "mast3r": mast3r,
        }

    def emit(mast3r, clocks, cpu):
        line = make_line(mast3r, clocks)
        if cpu:
            line["cpu_baseline"] = cpu
        print(json.dumps(line), flush=True)

    # The headline (rasterizer) numbers exist at this point.  If the second leg wedges the device, report them anyway.
    limit = float(os.environ.get("ADB_BENCH_MAST3R_TIMEOUT", "480"))

    def on_hang():
        if rank == 0:
            log(f"MASt3R leg exceeded {limit:.0f} s: reporting the rasterizer line without it")
            try:
                clocks = sampler.stop() if sampler else None
            except Exception:  # noqa: BLE001
                clocks = None
            emit({"metric": "MASt3R pairs/s @512^2", "error": f"leg exceeded {limit:.0f} s (device hang?)"}, clocks, None)
        os._exit(0)

    mast3r = None
    if not args.no_mast3r:
        wd = Watchdog(limit, on_hang).start()
        mast3r = bench_mast3r(dev, world, rank, args.steps, args.warmup,
                              want_baselines=(world == 1 and not args.no_cpu_baseline))
        wd.cancel()
    clocks = sampler.stop() if sampler else None   # sampled across every timed GPU leg (raster, e2e, MASt3R)
    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return
    if mast3r:
        log(f"mast3r leg done: {mast3r['ms_per_step']:.2f} ms/step")
    cpu = None
    if world == 1 and not args.no_cpu_baseline:
        g, sec, _, threads = cpu_oracle_leg(4, 1, N_GAUSS, [0, 3, 5, 7])
        cpu = {"value": g, "unit": "Gpix/s", "cores": threads, "kind": "port",
               "sample": "4 single-view fwd+bwd passes (views 0,3,5,7 of the batch) of the same 1M/1080p workload through "
                         "oracle/raster_oracle.c (OpenMP)", "seconds_per_view": sec}
    emit(mast3r, clocks, cpu)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
