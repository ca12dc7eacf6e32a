#!/usr/bin/env python
"""Benchmark of the GS/GD hologram path (BASELINE.json metric: iterations/s at 1024^2, holograms/s, % of HBM roofline).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--only headline,gs_1024,...]

ONE JSON line on stdout.  Its top level is the headline workload -- BASELINE.json configs[1]: gradient descent, 100
iterations, 1024x1024, followed by the wavefront-mask add + 8-bit quantisation; a *step* is one batch of 32 such
holograms per GPU, inputs resident in HBM, `value` = iterations/s summed over the ranks (weak scaling: every rank runs
its own batch, the path has no collective).  `verified` says whether plane 0 of the timed batch reproduced the
reference's error curve and 8-bit frame (tests/golden/gd_noise_1024x1024_curves.npz, made by the unmodified reference).

`e2e` is the same work through the reference-facing API with HOST buffers (algorithms.gradient_descent(target, args) ->
numpy, then display_holograms.hologram_to_grey), host<->device copies inside the timed region, summed over the ranks.

The line stays under 4 KB (tools that collect a run's output may keep only its tail): it ends with `summary`, one flat
object with the main figure of every further workload.  The full record -- the same keys with every sub-record, the
kernels' rooflines and notes -- is written to stderr as one JSON line.  Its `configs` holds one sub-record per further
workload of BASELINE.json, each timed like the headline (device events, warm-up, max over ranks):
    gs_1024   Gerchberg-Saxton, batch 32 x 1024^2 x 100 iterations (the metric names GS and GD)
    fp64      GD and GS at 1024^2 in the fp64 parity mode
    config1   ONE 512x512 GS hologram, 20 iterations: device latency and through gerchberg_saxton(target, args)
    config3   optical-trap movie, 1024 frames 768x1024 x GS 50 iterations through sequence_holograms: host frames in, host
              results out (uint8 SLM frames and float64 holograms); under --gpus N the frames are sharded over the ranks
              and gathered on rank 0 inside the timed region (strong scaling)
    config4   compare_error_evolution_algorithms shape: 256 targets x 2048^2, GD then GS, 50 iterations, all 512 curves
              (targets sharded over the ranks)
    config5   one 16384^2 GS hologram, 20 iterations, slab-decomposed over the ranks (1 GPU: the same code, world = 1);
              config5_gd: the same plane through gradient descent
    size_4096 GD and GS at 4096^2 (the upper end of the north star's range)

`--impl reference` times the CPU implementation (the oracle's numpy restatement of the reference, scipy.fft with all
host threads) on a bounded sample of the headline workload.

`--dump-outputs DIR` writes what the headline's last timed step computed on rank 0, so that two builds can be compared
output for output (the inputs are seeded: the same arguments give the same inputs):
    hologram.npy  float64 [batch, n]      the holograms at n pixels per plane (n <= 65536, the same pixels for every
                                          plane, drawn without replacement by np.random.default_rng(0), in ascending order)
    frames.npy    float32 [batch, n]      the 8-bit SLM frames (mask add + quantisation) at the same pixels
    errors.npy    float64 [batch, loops]  every plane's error curve
"""
from __future__ import annotations

import argparse
import contextlib
import io
import json
import os
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

ALL_SECTIONS = ["headline", "gs_1024", "fp64", "config1", "config3", "config4", "config5", "size_4096", "e2e", "cpu"]


def parse():
    p = argparse.ArgumentParser()
    p.add_argument("--gpus", type=int, default=1)
    p.add_argument("--steps", type=int, default=10)
    p.add_argument("--warmup", type=int, default=3)
    p.add_argument("--impl", default="b200", choices=["b200", "reference"])
    p.add_argument("--alg", default="gd", choices=["gd", "gs"])
    p.add_argument("--precision", default="fp32", choices=["fp32", "fp64"])
    p.add_argument("--size", type=int, default=1024)
    p.add_argument("--height", type=int, default=0, help="plane height (default: --size)")
    p.add_argument("--batch", type=int, default=32)
    p.add_argument("--loops", type=int, default=100)
    p.add_argument("--e2e-steps", type=int, default=5)
    p.add_argument("--cpu-loops", type=int, default=40, help="iterations of the CPU baseline sample")
    p.add_argument("--only", default="", help="comma-separated sections (default: all): " + ",".join(ALL_SECTIONS))
    p.add_argument("--movie-frames", type=int, default=1024)
    p.add_argument("--movie-batch", type=int, default=0, help="frames per device batch of config3 (0: the driver's own choice)")
    p.add_argument("--config4-targets", type=int, default=256)
    p.add_argument("--slab-size", type=int, default=16384)
    p.add_argument("--workload", default="batch", choices=["batch", "slab"],
                   help="slab: only config5 as the line's own workload (one --size^2 plane row-split over the ranks)")
    p.add_argument("--dump-outputs", metavar="DIR", default="",
                   help="write the headline's outputs of its last timed step to DIR/<name>.npy (see the module docstring)")
    a = p.parse_args()
    if a.steps < 1:
        p.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl != "b200" or a.workload != "batch"):
        p.error("--dump-outputs writes the headline's outputs: it needs --impl b200 --workload batch")
    return a


def env_rank():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))


def workload_name(a, shape):
    alg = "gradient_descent" if a.alg == "gd" else "gerchberg_saxton"
    return (f"{alg} {shape[0]}x{shape[1]} uint8 noise targets, {a.loops} iterations, batch {a.batch}/GPU, "
            f"+ wavefront-mask add + 8-bit quantise (BASELINE.json configs[1])")


# ---- byte models ------------------------------------------------------------------------------------------------------
def survey_bytes_per_px(alg, precision):
    """SURVEY.md 8(d): four passes per iteration -- GS (8c+4), GD (9c+4) bytes per pixel."""
    c = 8 if precision == "fp32" else 16
    return (8 * c + 4) if alg == "gs" else (9 * c + 4)


def design_bytes_per_px(alg, precision, gd_passes=1):
    """What this design must move (DESIGN.md 4): the two transforms that meet at a pointwise step share one pass --
    GS (4c+4); GD (6c+4) with one Fourier-plane pass per iteration, (8c+4) in the two-pass form."""
    c = 8 if precision == "fp32" else 16
    return (4 * c + 4) if alg == "gs" else ((6 * c + 4) if gd_passes == 1 else (8 * c + 4))


def kernel_bytes_per_px(kind, alg, precision):
    """Algorithmic bytes per pixel of ONE launch of a pass kernel (every plane the pass must read or write once, the
    8-bit target accounted at 4 B/px as in SURVEY 8d)."""
    c = 8 if precision == "fp32" else 16
    if kind == "col_pass":
        return 2 * c + 4                         # read X, write Y, read target
    if kind == "row_pass":
        return 2 * c if alg == "gs" else 4 * c   # GS: read Y, write X; GD: + read x, write x
    if kind == "col_stats":
        return 2 * c                             # the max pass of the two-pass GD form keeps the transform: read X, write X
    raise KeyError(kind)


def measured_traffic(key):
    """DRAM bytes (read + write) per launch from the committed ncu capture (profiles/traffic.json), or None."""
    path = os.path.join(ROOT, "profiles", "traffic.json")
    if not os.path.exists(path):
        return None
    return json.load(open(path)).get(key)


def measured_peak():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        return float(json.load(open(path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """SM clock / throttle-reason samples DURING the timed region, taken with NVML from a background
    thread (an `nvidia-smi -lms` child process perturbed the timed region on this pool: bimodal step times)."""
    THROTTLE = {"hw_slowdown": 0x8, "sw_thermal_slowdown": 0x20, "hw_thermal_slowdown": 0x40, "sw_power_cap": 0x4}

    def __init__(self, index, period_s=None):
        period_s = float(os.environ.get("SLM_BENCH_SAMPLER_PERIOD", "0.05")) if period_s is None else period_s
        self.index, self.period, self.samples, self._stop, self.thread, self.err = index, period_s, [], False, None, None

    def start(self):
        import threading
        try:
            import pynvml
            pynvml.nvmlInit()
            visible = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(visible.split(",")[self.index]) if visible and visible.split(",")[self.index].isdigit() else self.index
            self.nv, self.h = pynvml, pynvml.nvmlDeviceGetHandleByIndex(phys)
        except Exception as exc:
            self.err = f"nvml unavailable: {exc}"
            return

        def loop():
            nv, h = self.nv, self.h
            while not self._stop:
                try:
                    t_s = time.time()
                    row = (t_s, nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM),
                           nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM),
                           nv.nvmlDeviceGetCurrentClocksEventReasons(h), nv.nvmlDeviceGetPowerUsage(h) / 1000.0)
                    self.samples.append(row + (time.time() - t_s,))
                except Exception as exc:
                    self.err = str(exc)
                    return
                time.sleep(self.period)
        self.thread = threading.Thread(target=loop, daemon=True)
        self.thread.start()

    def stop(self, t_begin=None, t_end=None):
        self._stop = True
        if self.thread:
            self.thread.join(timeout=2)
        rows = [r for r in self.samples if t_begin is None or t_begin - 0.05 <= r[0] <= t_end + 0.05] or self.samples[-1:]
        if not rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [self.err or "no samples"]}
        reasons = sorted(k for k, bit in self.THROTTLE.items() if any(r[3] & bit for r in rows))
        return {"sm_mhz": float(np.median([r[1] for r in rows])), "sm_max_mhz": float(max(r[2] for r in rows)),
                "reasons": reasons, "samples": len(rows), "power_w_max": max(r[4] for r in rows), "source": "nvml",
                "sample_ms_max": round(1e3 * max(r[5] for r in rows), 2)}


# ---- CPU arm ------------------------------------------------------------------------------------------------------------
def cpu_port_iterations_per_s(alg, shape, loops, workers):
    """Time the oracle's restatement of the reference loop on the host."""
    import scipy.fft
    from oracle import numpy_port as P
    from spatial_light_modulator_module_b200 import synthetic
    t = synthetic.noise_target(shape, seed=0)
    with scipy.fft.set_workers(workers), np.errstate(all="ignore"):
        t0 = time.perf_counter()
        if alg == "gd":
            P.gd_run(t, loops)
        else:
            P.gs_run(t, loops)
        dt = time.perf_counter() - t0
    return loops / dt, dt


def run_reference(a):
    rank, _, world = env_rank()
    if rank != 0:
        return
    shape = (a.height or a.size, a.size)
    cores = os.cpu_count() or 1
    sample_loops = max(2, min(a.loops, 10))
    times = []
    for i in range(a.warmup + a.steps):
        _, dt = cpu_port_iterations_per_s(a.alg, shape, sample_loops, cores)
        if i >= a.warmup:
            times.append(dt)
    total = sum(times)
    value = sample_loops * a.steps / total
    sample = (f"each step = 1 hologram x {sample_loops} iterations of the numpy restatement (oracle/numpy_port.py) "
              f"incl. setup, scipy.fft workers={cores}")
    emit(({
        "impl": "reference", "metric": "GS/GD iterations/sec at 1024^2", "value": value, "unit": "iterations/s",
        "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup, "ms_per_step": 1e3 * total / a.steps,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
        "config": {"workload": workload_name(a, shape)},
        "cpu_baseline": {"value": value, "unit": "iterations/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "iterations/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ---- device arm -----------------------------------------------------------------------------------------------------------
class Harness:
    """Timing rules of the contract: warm-up, barrier + synchronize on both sides, CUDA events, max over ranks."""

    def __init__(self, torch, dist, world, dev):
        self.torch, self.dist, self.world, self.dev = torch, dist, world, dev

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, value):
        if self.world == 1:
            return float(value)
        t = self.torch.tensor([value], device=self.dev, dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, value):
        if self.world == 1:
            return float(value)
        t = self.torch.tensor([value], device=self.dev, dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return float(t.item())

    def all_ok(self, flag):
        if self.world == 1:
            return bool(flag)
        t = self.torch.tensor([1.0 if flag else 0.0], device=self.dev, dtype=self.torch.float64)
        self.dist.all_reduce(t, op=self.dist.ReduceOp.MIN)
        return bool(t.item() > 0.5)

    def time_steps(self, step, warmup, steps):
        """-> (total ms of `steps` steps as the max over ranks, per-step ms of this rank, result of the last step)"""
        torch = self.torch
        out = None
        for _ in range(warmup):
            out = step()
        self.barrier()
        e0 = torch.cuda.Event(enable_timing=True)
        marks = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
        self.barrier()
        e0.record()
        for i in range(steps):
            out = step()
            marks[i].record()
        self.barrier()
        ms = e0.elapsed_time(marks[-1])
        step_ms = [round(([e0] + marks)[i].elapsed_time(marks[i]), 3) for i in range(steps)]
        return self.max_over_ranks(ms), step_ms, out

    def wall_steps(self, step, warmup, steps):
        """Host-clock timing for end-to-end calls (host buffers in and out): seconds per step, max over ranks."""
        out = None
        for _ in range(warmup):
            out = step()                 # (kept alive like a timed step's result: see time_steps)
        self.barrier()
        t0 = time.perf_counter()
        for _ in range(steps):
            out = step()
        self.torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / steps
        self.barrier()
        return self.max_over_ranks(dt), out


def roofline_record(name, alg, precision, npx_total, avg_ms, kind, share, peak, peak_src, traffic_key=None):
    """traffic_key: "<kind>|<alg>|<precision>|<H>x<W>|batch<B>" in profiles/traffic.json (ncu --set full, per launch)"""
    bts = kernel_bytes_per_px(kind, alg, precision) * npx_total
    ach = bts / (avg_ms * 1e-3) / 1e9
    return {"bound": "hbm", "kernel": name, "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak,
            "traffic": measured_traffic(traffic_key) if traffic_key else None, "peak_source": peak_src,
            "alg_bytes_per_launch": bts, "avg_launch_ms": avg_ms, "share_of_step": share}


def iteration_rooflines(alg, precision, npx, per_iter_s, peak, gd_passes=1):
    sv, ds = survey_bytes_per_px(alg, precision) * npx, design_bytes_per_px(alg, precision, gd_passes) * npx
    return {"survey_model": {"bytes_per_iteration": sv, "achieved_gbs": sv / per_iter_s / 1e9, "frac": sv / per_iter_s / 1e9 / peak,
                             "note": "SURVEY 8(d): (8c+4) GS / (9c+4) GD B/px -- four unfused passes; a fused design moves fewer bytes, so "
                                     "this fraction can exceed what the memory system really delivers"},
            "design_model": {"bytes_per_iteration": ds, "achieved_gbs": ds / per_iter_s / 1e9, "frac": ds / per_iter_s / 1e9 / peak,
                             "note": "bytes this design must move: (4c+4) GS, (6c+4) GD B/px (one Fourier-plane pass per iteration)"},
            "peak": peak, "unit": "GB/s"}


def kernel_names(alg, gd_form):
    col = {"gs": "col_warp_kernel<GS> (Fourier-plane pass)",
           "gd": {"pipe": "col_warp_kernel<GD_PIPE> (Fourier-plane pass, one per iteration)",
                  "fused": "col_warp_kernel<GD_FUSED> (Fourier-plane pass, one per iteration)",
                  "two_pass": "col_warp_kernel<GD_POST> (gradient pass)"}[gd_form]}[alg]
    return {"col_pass": col, "row_pass": f"row_pass_kernel<{'GS' if alg == 'gs' else 'GD'}> (SLM-plane pass)",
            "col_stats": "col_warp_kernel<STATS_KEEP> (max pass, keeps the transform)"}


def profile_kernels(eng, step, steps, alg, precision, npx_total, peak, peak_src, gd_form="pipe", names=None, traffic_prefix=None):
    """Instrumented re-run of the same steps: per-kernel CUDA-event times from the engine (slm_ctx_profile)."""
    eng.profile(True)
    eng.profile_read()
    for _ in range(steps):
        step()
    prof = eng.profile_read()
    eng.profile(False)
    names = names or kernel_names(alg, gd_form)
    kernels = {}
    tsum = sum(v[0] for v in prof.values()) or 1.0
    for kind in ("col_pass", "row_pass", "col_stats"):
        tot, cnt = prof[kind]
        if cnt:
            rec = roofline_record(names[kind], alg, precision, npx_total, tot / cnt, kind, tot / tsum, peak, peak_src,
                                  f"{kind}|{traffic_prefix}" if traffic_prefix else None)
            rec["launches"] = cnt
            kernels[kind] = rec
    dom = max(kernels, key=lambda k: kernels[k]["share_of_step"])
    return kernels, dict(kernels[dom])


def batched_loop_record(h, a, alg, precision, shape, batch, loops, steps, warmup, peak, peak_src, verify=None, extra_step=None):
    """One sub-record: `batch` holograms of `shape`, `loops` iterations each, device resident; optionally the mask add +
    quantise behind it (extra_step).  Returns (record, engine state for follow-ups)."""
    import torch
    from spatial_light_modulator_module_b200 import host_logic as hl, synthetic
    from spatial_light_modulator_module_b200.engine import Engine
    rank = env_rank()[0]
    npx = shape[0] * shape[1]
    eng = Engine(shape, precision, batch)
    tg = [synthetic.noise_target(shape, seed=(0 if (i == 0 and verify) else 1000 * rank + i + 1)) for i in range(batch)]
    targets = torch.from_numpy(np.stack(tg)).to(h.dev)
    norms = targets.reshape(batch, -1).amax(dim=1).double().cpu().numpy()
    during, _ = hl.learning_rate_schedule(0.005, 0, loops)
    x0 = x = None
    if alg == "gd":
        rng = np.random.default_rng(rank)
        x0 = torch.from_numpy(np.exp(2j * np.pi * rng.random((batch,) + shape)).astype(eng.complex_dtype)).to(h.dev)
        if verify:                                  # plane 0: the reference's own start, random.seed(42) (algorithms.py:117-121)
            u = eng.python_random_uniform(42, shape)
            x0[0].copy_(eng.random_phasor_guess(u, 1.0)[0])
        x = torch.empty_like(x0)
    state = {}

    def step():
        if alg == "gd":
            x.copy_(x0)
            res, _ = eng.gd(targets, x, during, loops, want_expected=False, norms=norms)
        else:
            res = eng.gs(targets, loops, want_expected=False, norms=norms)
        state["res"] = res
        return extra_step(eng, res) if extra_step else res.hologram

    n0 = eng.launch_count()
    ms, step_ms, out = h.time_steps(step, max(warmup, 3), steps)
    timed_res = state["res"]                         # the profiled re-run below replaces state["res"]
    launches = (eng.launch_count() - n0) * steps // (max(warmup, 3) + steps)
    iters = batch * loops * steps * h.world
    per_iter_s = ms * 1e-3 / (batch * loops * steps)
    sms = torch.cuda.get_device_properties(h.dev).multi_processor_count
    form = os.environ.get("SLM_GD_FORM") or ("two_pass" if os.environ.get("SLM_NO_FUSED_GD") else ("pipe" if batch * (shape[1] // 8) > 4 * sms else "fused"))
    if precision == "fp64" or shape[0] not in (768, 1024):
        form = "two_pass"                            # the one-pass forms exist in the warp-per-column kernel (fp32, 768/1024 rows)
    rec = {"workload": f"{'gradient_descent' if alg == 'gd' else 'gerchberg_saxton'} {shape[0]}x{shape[1]}, batch {batch}/GPU, {loops} iterations, "
                       f"{precision}, device resident", "value": iters / (ms * 1e-3), "unit": "iterations/s",
           "holograms_per_s": batch * steps * h.world / (ms * 1e-3), "ms_per_step": ms / steps, "steps": steps, "step_ms": step_ms,
           "gpu_launches": int(launches), "iteration_roofline": iteration_rooflines(alg, precision, npx, per_iter_s, peak, 1 if form != "two_pass" else 2)}
    if alg == "gd":
        rec["gd_form"] = form
    if rank == 0:
        names = kernel_names(alg, form)
        if precision == "fp64" or shape[0] not in (768, 1024):
            names = {k: v.replace("col_warp_kernel", "col_group_kernel" if shape[0] < 4096 else "col_pass_kernel / col_plain_kernel") for k, v in names.items()}
        kernels, roof = profile_kernels(eng, step, min(steps, 3), alg, precision, npx * batch, peak, peak_src, form, names,
                                        f"{alg}|{precision}|{shape[0]}x{shape[1]}|batch{batch}")
        rec["kernels"], rec["roofline"] = kernels, roof
        if alg == "gd" and form == "pipe" and roof:
            roof["note"] = ("one launch does what round 1's two did (max pass: read + write the transform, 16 B/px; gradient pass: 20 B/px -- "
                            "0.104 + 0.164 = 0.268 ms): it moves 20 B/px in 0.24 ms and is bound by the planes' barriers and the SM "
                            "(issue slots 32 % busy), not by DRAM; the whole iteration's fractions are in iteration_roofline")
    state.update(eng=eng, targets=targets, norms=norms, during=during, x0=x0, x=x, res=timed_res, out=out, step=step)
    return rec, state


def verify_headline(state, shape, loops, precision):
    """Plane 0 of the timed batch against the reference's own run (fixture made by the unmodified reference): error
    curve within the north star's fp32 tolerance 1e-3 (fp64: 1e-9), 8-bit frame within +-1 LSB on <= 2e-3 of the pixels."""
    path = os.path.join(ROOT, "tests", "golden", f"gd_noise_{shape[0]}x{shape[1]}_curves.npz")
    if not os.path.exists(path) or loops != 100:
        return None, {"skipped": "no reference fixture for this configuration"}
    g = np.load(path)
    res, eng = state["res"], state["eng"]
    e = res.errors[0]
    ok_len = len(e) == len(g["errors"])
    curve = float(np.max(np.abs(e - g["errors"]) / g["errors"])) if ok_len else float("inf")
    frame = eng.to_host(state["out"][0:1])[0][::4, ::4].astype(np.int32)
    d = (frame - g["q3_sub"].astype(np.int32)) % 256
    d = np.minimum(d, 256 - d)
    frac = float(np.mean(d != 0))
    tol = 1e-3 if precision == "fp32" else 1e-9
    ok = bool(ok_len and curve < tol and d.max() <= 1 and frac <= 2e-3)
    return ok, {"error_curve_max_rel": curve, "curve_tolerance": tol, "frame_max_lsb": int(d.max()), "frame_fraction_differing": frac, "frame_fraction_allowed": 2e-3,
                "fixture": "tests/golden/gd_noise_1024x1024_curves.npz (unmodified reference, algorithms.py:60-112 + move_traps.py:135-140)"}


def dump_outputs(out_dir, state):
    """--dump-outputs: the headline's last timed step (module docstring), at most 64 MB in all."""
    import torch
    res, frames = state["res"], state["out"]
    batch = frames.shape[0]
    npx = frames[0].numel()
    n = min(npx, 1 << 16, (48 << 20) // (12 * batch))            # 8 B (hologram) + 4 B (frame) per sampled pixel
    idx = torch.from_numpy(np.sort(np.random.default_rng(0).choice(npx, size=n, replace=False))).to(frames.device)
    arrays = {"hologram": res.hologram.reshape(batch, -1).index_select(1, idx).cpu().numpy(),
              "frames": frames.reshape(batch, -1).index_select(1, idx).float().cpu().numpy(),
              "errors": np.stack(res.errors).astype(np.float64)}
    os.makedirs(out_dir, exist_ok=True)
    for name, arr in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), arr)


def run_b200(a):
    import torch
    import torch.distributed as dist

    rank, local_rank, world = env_rank()
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    from spatial_light_modulator_module_b200 import _ffi, algorithms, display_holograms, synthetic
    from spatial_light_modulator_module_b200.engine import Engine

    dev = torch.device("cuda", local_rank)
    h = Harness(torch, dist, world, dev)
    only = [s for s in a.only.split(",") if s] or ALL_SECTIONS
    shape = (a.height or a.size, a.size)
    npx = shape[0] * shape[1]
    peak, peak_src = measured_peak()
    mask_dev = torch.from_numpy(synthetic.random_mask(shape, seed=1)).to(dev)
    quant = lambda eng, res: eng.quantize(res.hologram, mask_dev, 256, _ffi.QUANT_FLOOR)      # noqa: E731

    # ---- headline: configs[1] ---------------------------------------------------------------------------------------
    sampler = ClockSampler(local_rank)
    if rank == 0 and not os.environ.get("SLM_BENCH_NO_SAMPLER"):
        sampler.start()
    wall0 = time.time()
    head, st = batched_loop_record(h, a, a.alg, a.precision, shape, a.batch, a.loops, a.steps, a.warmup, peak, peak_src,
                                   verify=(a.alg == "gd"), extra_step=quant)
    wall1 = time.time()
    clocks = sampler.stop(wall0, wall1) if rank == 0 else None
    verified, verification = (None, {"skipped": "GS free-running is chaotic on dense targets (DESIGN.md 2); see tests"})
    if a.alg == "gd":
        verified, verification = verify_headline(st, shape, a.loops, a.precision)
    if verified is not None:
        verified = h.all_ok(verified)
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, st)
    csz = 8 if a.precision == "fp32" else 16
    line = {
        "metric": "GS/GD iterations/sec at 1024^2", "value": head["value"], "unit": "iterations/s", "n_gpus": world,
        "steps": a.steps, "warmup": max(a.warmup, 3), "ms_per_step": head["ms_per_step"], "step_ms": head["step_ms"],
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32" if a.precision == "fp32" else "f64",
        "data": "synthetic",
        "config": {"workload": workload_name(a, shape), "algorithm": a.alg, "shape": list(shape), "batch_per_gpu": a.batch,
                   "iterations": a.loops, "precision_mode": f"{a.precision} (north star: fp32 mode with 1e-3 tolerances, fp64 parity mode with 1e-9; "
                                                            "the reference computes in complex128 -- see configs.fp64)",
                   "l2": f"inputs larger than L2: {3 * a.batch * npx * csz / 2**20:.0f} MiB of field planes per GPU",
                   "seeds": "targets default_rng(1000*rank+i+1) (plane 0: seed 0 = the reference fixture), mask default_rng(1)",
                   "gd_form": head.get("gd_form")},
        "holograms_per_s": head["holograms_per_s"], "gpu_launches": head["gpu_launches"], "clocks": clocks,
        "verified": verified, "verification": verification,
        "roofline": head.get("roofline"), "iteration_roofline": head["iteration_roofline"], "kernels": head.get("kernels"),
        "targets": {"north_star": ">= 70 % of 8 TB/s on SURVEY 8(d) bytes", "gd_iterations_per_s": 0.7 * 8e12 / (survey_bytes_per_px("gd", "fp32") * npx),
                    "gs_iterations_per_s": 0.7 * 8e12 / (survey_bytes_per_px("gs", "fp32") * npx)},
    }
    configs = {}

    # ---- latency of ONE hologram (batch 1), device resident ---------------------------------------------------------
    if "headline" in only:
        eng1 = Engine(shape, a.precision, 1)
        t1, x01 = st["targets"][:1].contiguous(), (st["x0"][:1].contiguous() if st["x0"] is not None else None)
        x1 = torch.empty_like(x01) if x01 is not None else None

        def step1():
            if a.alg == "gd":
                x1.copy_(x01)
                r, _ = eng1.gd(t1, x1, st["during"], a.loops, want_expected=False, norms=st["norms"][:1])
            else:
                r = eng1.gs(t1, a.loops, want_expected=False, norms=st["norms"][:1])
            return eng1.quantize(r.hologram, mask_dev, 256, _ffi.QUANT_FLOOR)
        ms1, _, _ = h.time_steps(step1, 3, a.steps)
        lat = ms1 / a.steps
        line["single_hologram"] = {"ms_per_hologram": lat, "iterations_per_s": a.loops / (lat * 1e-3),
                                   "note": "batch 1 (the unit the reference API hands over): the working set fits in L2, launch/latency bound"}
        eng1.close()
    st["eng"].close()
    del st

    if "gs_1024" in only:
        rec, s2 = batched_loop_record(h, a, "gs", "fp32", (1024, 1024), a.batch, a.loops, max(3, a.steps // 2), 3, peak, peak_src, extra_step=quant)
        s2["eng"].close()
        configs["gs_1024"] = rec
    if "fp64" in only:
        m64 = torch.from_numpy(synthetic.random_mask((1024, 1024), seed=1)).to(dev)
        q64 = lambda eng, res: eng.quantize(res.hologram, m64, 256, _ffi.QUANT_FLOOR)      # noqa: E731
        sub = {}
        for alg in ("gd", "gs"):
            rec, s2 = batched_loop_record(h, a, alg, "fp64", (1024, 1024), 16, a.loops, 3, 3, peak, peak_src, verify=(alg == "gd"), extra_step=q64)
            if alg == "gd":
                ok, info = verify_headline(s2, (1024, 1024), a.loops, "fp64")
                rec["verified"], rec["verification"] = (h.all_ok(ok) if ok is not None else None), info
            s2["eng"].close()
            sub[alg] = rec
        configs["fp64"] = sub
    if "size_4096" in only:
        sub = {}
        for alg in ("gd", "gs"):
            rec, s2 = batched_loop_record(h, a, alg, "fp32", (4096, 4096), 2, 20, 3, 3, peak, peak_src)
            s2["eng"].close()
            sub[alg] = rec
        configs["size_4096"] = sub
    if "config1" in only:
        configs["config1"] = run_config1(h, a, local_rank)
    if "config3" in only:
        configs["config3"] = run_config3(h, a)
    if "config4" in only:
        configs["config4"] = run_config4(h, a, local_rank, peak)
    if "config5" in only:
        configs["config5"] = run_config5(h, a.slab_size, 20, "fp32", 2, 1, peak)
        configs["config5_gd"] = run_config5(h, a.slab_size, 20, "fp32", 2, 1, peak, alg="gd")

    # ---- end to end through the drop-in API with host buffers, every rank at once -------------------------------------
    if "e2e" in only:
        ns = argparse.Namespace(incomming_intensity="uniform", tolerance=0, max_loops=a.loops, gif=False, print_info=False,
                                plot_error=False, initial_guess="random", random_seed=42, white_attention=1,
                                learning_rate=0.005, unsettle=0, precision=a.precision, device=local_rank)
        host_targets = [synthetic.noise_target(shape, seed=77 + i + 100 * rank) for i in range(a.e2e_steps + 1)]
        host_mask = synthetic.random_mask(shape, seed=1)
        fn = algorithms.gradient_descent if a.alg == "gd" else algorithms.gerchberg_saxton
        it = {"i": 0}

        def e2e_once():
            t = host_targets[it["i"] % len(host_targets)]
            it["i"] += 1
            with contextlib.redirect_stdout(io.StringIO()):
                holo, exp, errs = fn(t, ns)
            ns.learning_rate = 0.005
            return display_holograms.hologram_to_grey(holo, host_mask, 256)
        e2e_s, _ = h.wall_steps(e2e_once, 2, a.e2e_steps)     # (2 warm-ups: the engine page-locks a host array it is handed twice -- the mask)
        h2d = npx * 1 + npx * 8 + npx * 8                    # target; hologram + mask for the quantiser (the GD initial guess is drawn on the device)
        d2h = npx * 8 * 2 + a.loops * 8 + npx                # hologram, expected, error curve, grey frame
        line["e2e"] = {"value": world * a.loops / e2e_s, "unit": "iterations/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                       "ms_per_hologram": 1e3 * e2e_s, "holograms_per_s": world / e2e_s, "ranks": world,
                       "api": f"algorithms.{fn.__name__}(target_uint8, args) -> numpy; display_holograms.hologram_to_grey(h, mask, 256); "
                              "one hologram at a time per rank, all ranks at once, value = sum over ranks",
                       "note": "random.seed(42) initial guess: the MT19937 stream is a pure function of (seed, size) and is memoised on the device "
                               "(the reference's CLI always seeds 42, generate_hologram.py:370); SLM_NO_GUESS_MEMO=1 disables the memo"}

    # ---- CPU baseline (oracle port, single core as the reference runs it), at every N on rank 0 ---------------------------
    cpu = None
    if "cpu" in only and rank == 0:
        v, dt = cpu_port_iterations_per_s(a.alg, shape, min(a.cpu_loops, a.loops), 1)
        cores = os.cpu_count() or 1
        v_all, dt_all = cpu_port_iterations_per_s(a.alg, shape, min(a.cpu_loops, a.loops), cores)
        cpu = {"value": v, "unit": "iterations/s", "cores": 1, "kind": "port",
               "sample": f"1 hologram x {min(a.cpu_loops, a.loops)} iterations of oracle/numpy_port.py ({dt:.1f} s), "
                         f"scipy.fft workers=1 as in the reference; host has {cores} cores",
               "all_cores": {"value": v_all, "cores": cores, "sample": f"the same with scipy.fft workers={cores} ({dt_all:.1f} s); numpy's "
                                                                       "elementwise work stays on one core"}}
    line["cpu_baseline"] = cpu
    line["configs"] = configs
    if rank == 0:
        sys.stderr.write(json.dumps(line) + "\n")
        sys.stderr.flush()
        emit(result_line(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_config1(h, a, local_rank):
    """BASELINE configs[0]: ONE 512x512 GS hologram, 20 iterations (the reference's own CPU-runnable case)."""
    import torch
    from spatial_light_modulator_module_b200 import algorithms, synthetic
    from spatial_light_modulator_module_b200.engine import Engine
    shape, loops = (512, 512), 20
    eng = Engine(shape, "fp32", 1)
    t = synthetic.noise_target(shape, seed=0)
    td = torch.from_numpy(t[None]).to(h.dev)
    norms = np.array([float(t.max())])
    ms, _, _ = h.time_steps(lambda: eng.gs(td, loops, want_expected=True, norms=norms).hologram, 5, 20)
    ns = argparse.Namespace(incomming_intensity="uniform", tolerance=0, max_loops=loops, gif=False, print_info=False,
                            plot_error=False, precision="fp32", device=local_rank)

    def once():
        with contextlib.redirect_stdout(io.StringIO()):
            return algorithms.gerchberg_saxton(t, ns)
    s, out = h.wall_steps(once, 3, 20)
    eng.close()
    return {"workload": "gerchberg_saxton(target 512x512 uint8 noise, max_loops=20): one hologram (BASELINE.json configs[0])",
            "device_ms_per_hologram": ms / 20, "device_iterations_per_s": loops / (ms / 20 * 1e-3),
            "e2e_ms_per_hologram": 1e3 * s, "e2e_iterations_per_s": loops / s, "e2e_holograms_per_s": 1 / s,
            "final_error": float(out[2][-1]), "h2d_bytes": 512 * 512, "d2h_bytes": 2 * 512 * 512 * 8 + loops * 8,
            "note": "latency bound: 2 MB of field, 41 launches; the device figure includes setup (ifft2 of the amplitude), the final "
                    "hologram and the expected outcome"}


def run_config3(h, a):
    """BASELINE configs[2]: optical-trap movie, GS 50 iterations per frame, frames sharded over the ranks, results gathered
    on rank 0 -- through generate_hologram_sequence.sequence_holograms with host frames in and host results out."""
    from spatial_light_modulator_module_b200 import generate_hologram_sequence as ghs, synthetic
    frames_n, loops, shape = a.movie_frames, 50, (768, 1024)
    frames = synthetic.movie_frames(frames_n)
    mask = synthetic.random_mask(shape, seed=1)
    dots = synthetic.movie_frame_dots(frames_n)
    rec = {"workload": f"{frames_n} trap frames {shape[0]}x{shape[1]} (two circulating dots, generate_traps_image_sequence.py:48-58), GS {loops} "
                       f"iterations each, sharded over {h.world} GPU(s), gathered on rank 0 (BASELINE.json configs[2])", "frames": frames_n}
    variants = {
        "uint8_frames": dict(output="uint8", mask=mask, ct2pi=256),
        "float64_holograms": dict(output="float64"),
        "uint8_frames_device_rasterised": dict(output="uint8", mask=mask, ct2pi=256, trap_dots=(dots, frames_n, shape)),
    }
    for name, kw in variants.items():
        src = None if "trap_dots" in kw else frames

        def once():
            return ghs.sequence_holograms(src, loops, precision="fp32", batch=a.movie_batch or None, gather=True, **kw)
        s, out = h.wall_steps(once, 2, 2)          # (two warm-ups: the result of call k is alive while call k+1 allocates its own)
        per_frame = shape[0] * shape[1] * (1 if kw["output"] == "uint8" else 8)
        rec[name] = {"holograms_per_s": frames_n / s, "iterations_per_s": frames_n * loops / s, "seconds": s,
                     "h2d_bytes": 0 if src is None else int(frames.nbytes), "d2h_bytes": frames_n * per_frame,
                     "gathered_bytes": 0 if h.world == 1 else frames_n * per_frame * (h.world - 1) // h.world,
                     "final_error_frame0": float(out[2][0][-1]) if env_rank()[0] == 0 else None}
    # the loop of the same workload alone, device resident, with its kernels' rooflines
    peak, peak_src = measured_peak()
    dev_rec, st = batched_loop_record(h, a, "gs", "fp32", shape, 32, loops, 3, 3, peak, peak_src)
    st["eng"].close()
    dev_rec["workload"] = f"gerchberg_saxton {shape[0]}x{shape[1]} (the SLM shape), batch 32/GPU, {loops} iterations, fp32, device resident (noise targets)"
    rec["device_resident_loop"] = dev_rec
    rec["note"] = ("timed region: host uint8 frames -> device, 50 iterations per frame, mask add + quantisation (uint8 variants) and the gather: "
                   "rank 0's result arrays lie in host memory shared by the ranks of the node, every rank reads its own frames back into them "
                   "over its own PCIe link (shared_host.py; SLM_GATHER=device: device-to-device gather on rank 0 over NCCL, then ONE link); "
                   "uint8 SLM frames are what display_holograms.py:253-266 consumes, float64 holograms what the reference saves (6 MiB per frame)")
    return rec


def run_config4(h, a, local_rank, peak):
    """BASELINE configs[3]: compare_error_evolution_algorithms over many large targets: GD then GS, all curves."""
    from spatial_light_modulator_module_b200 import compare_error_evolution_algorithms as cmp, host_logic as hl, synthetic
    rank, world = env_rank()[0], h.world
    n_total, shape, loops = a.config4_targets, (2048, 2048), 50
    lo, hi = hl.shard_range(n_total, rank, world)
    kinds = []
    for i in range(lo, hi):                                # the mix of SURVEY 8(d): noise, shapes, sparse traps
        if i % 3 == 0:
            kinds.append(synthetic.noise_target(shape, seed=i))
        elif i % 3 == 1:
            kinds.append(np.roll(synthetic.shapes_target(shape), 7 * i, axis=1))
        else:
            kinds.append(synthetic.traps_target(shape, [((37 * i) % shape[0], (91 * i) % shape[1]), ((211 * i) % shape[0], (503 * i) % shape[1])]))
    targets = np.stack(kinds)
    ns = argparse.Namespace(max_loops=loops, learning_rate=0.005, white_attention=1, unsettle=0, initial_guess="random", random_seed=42,
                            precision="fp32", device=local_rank)
    cmp.fill_unnecessary_args(ns)

    def once():
        return cmp.error_evolution_curves(targets, ns, batch=32)
    s, (gd, gs) = h.wall_steps(once, 1, 1)
    npx = shape[0] * shape[1]
    it = 2 * n_total * loops
    bytes_it = (survey_bytes_per_px("gd", "fp32") + survey_bytes_per_px("gs", "fp32")) / 2 * npx
    return {"workload": f"compare_error_evolution_algorithms.error_evolution_curves: {n_total} targets x 2048x2048 (noise / shapes / traps), GD then "
                        f"GS, {loops} iterations each, host uint8 targets in, {2 * n_total} error curves out, targets sharded over {world} GPU(s) "
                        "(BASELINE.json configs[3])",
            "seconds": s, "holograms_per_s": 2 * n_total / s, "iterations_per_s": it / s, "curves": 2 * n_total,
            "h2d_bytes": int(n_total * npx), "d2h_bytes": int(2 * n_total * loops * 8),
            "iteration_roofline_survey_bytes": {"achieved_gbs_per_gpu": bytes_it * it / s / 1e9 / world, "frac": bytes_it * it / s / 1e9 / world / peak,
                                                "note": "whole call incl. the host->device copy of the targets and the drawing of the random guess"},
            "gd_final_error_mean": float(np.mean([c[-1] for c in gd])), "gs_final_error_mean": float(np.mean([c[-1] for c in gs])),
            "gd_curve0_decreasing": bool(gd[0][-1] < gd[0][0]) if len(gd) else None}


def run_config5(h, n, loops, precision, steps, warmup, peak, alg="gs"):
    """BASELINE configs[4]: one n x n GS hologram, slab-decomposed over the ranks (strong scaling); ``alg="gd"``: the
    same plane through gradient descent (algorithms.py:60-112), whose Fourier plane is passed twice per iteration."""
    import torch
    from spatial_light_modulator_module_b200 import host_logic as hl
    from spatial_light_modulator_module_b200.slab import SlabEngine
    rank, world = env_rank()[0], h.world
    rows = n // world
    eng = SlabEngine(n, world, rank, precision)
    slab = eng._mem_upload((np.random.default_rng(100 + rank).random((rows, n)) * 255).astype(np.uint8))   # resident in HBM
    state = {}
    if alg == "gd":
        u = eng._mem_upload(np.random.default_rng(200 + rank).random((rows, n)))
        x0 = eng._mem_empty((rows, n), eng.complex_dtype)
        eng._check(eng._lib.slm_random_phasor(eng._ctx, eng._mem_ptr(u), eng._mem_ptr(x0), rows * n, 1.0))
        del u
        run = lambda k: eng.gd(slab, x0, hl.learning_rate_schedule(0.005, 0, k)[0], k, want_expected=False, on_device=True)
    else:
        run = lambda k: eng.gs(slab, k, want_expected=False, on_device=True)

    def step():
        state["out"] = run(loops)
        return state["out"][0]
    # Warm-up: twice at least, results kept alive like a timed step's -- a step allocates its result before the previous
    # one is released, so the allocator needs TWO result blocks, and a fresh 1 GB cudaMalloc with peer mappings in place
    # costs ~100 ms (seen as a first timed step of 188 instead of 90 ms on 2 GPUs).
    for _ in range(max(warmup, 2)):
        state["out"] = run(2)
    n0 = eng.launch_count()
    ms, step_ms, _ = h.time_steps(step, 0, steps)
    launches = eng.launch_count() - n0
    errs = state["out"][2]
    it_bytes = survey_bytes_per_px(alg, precision) * n * n          # SURVEY 8(d)'s four-pass model (the exchanges are not in it)
    per_it = ms * 1e-3 / (steps * loops)
    eng_info = argparse.Namespace(enqueue_s=getattr(eng, "enqueue_s", 0.0))
    eng.close()
    del slab
    torch.cuda.empty_cache()
    what = ("gerchberg_saxton", "2 all-to-alls + 1 all-reduce", "BASELINE.json configs[4]") if alg == "gs" else \
        ("gradient_descent", "2 all-to-alls + 2 all-reduces", "the plane of configs[4] through the other algorithm")
    return {"workload": f"{what[0]}, one {n}x{n} uint8 noise target, {loops} iterations incl. setup and the final hologram, rows split over "
                        f"{world} GPU(s), {what[1]} per iteration ({what[2]})",
            "value": 1.0 / per_it, "unit": "iterations/s", "scaling": "strong", "ms_per_hologram": ms / steps, "step_ms": step_ms,
            "gpu_launches": int(launches), "final_error": float(errs[-1]), "iterations": len(errs),
            "host_enqueue_ms": round(1e3 * getattr(eng_info, "enqueue_s", 0.0), 3),
            "iteration_roofline": {"survey_bytes_per_iteration": it_bytes, "achieved_gbs_per_gpu": it_bytes / per_it / 1e9 / world,
                                   "frac": it_bytes / per_it / 1e9 / world / peak, "peak": peak, "unit": "GB/s per GPU"}}


def run_slab(a):
    """`--workload slab`: config 5 alone, as the line's own workload."""
    import torch
    import torch.distributed as dist
    rank, local_rank, world = env_rank()
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    h = Harness(torch, dist, world, torch.device("cuda", local_rank))
    peak, _ = measured_peak()
    sampler = ClockSampler(local_rank)
    if rank == 0 and not os.environ.get("SLM_BENCH_NO_SAMPLER"):
        sampler.start()
    wall0 = time.time()
    rec = run_config5(h, a.size, a.loops, a.precision, a.steps, max(a.warmup, 1), peak)
    clocks = sampler.stop(wall0, time.time()) if rank == 0 else None
    if rank == 0:
        emit({"metric": f"GS iterations/sec on one {a.size}^2 plane (slab-decomposed)", "value": rec["value"], "unit": "iterations/s",
              "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 1), "ms_per_step": rec["ms_per_hologram"], "higher_is_better": True,
              "scaling": "strong", "vs_baseline": None, "dtype": "f32" if a.precision == "fp32" else "f64", "data": "synthetic",
              "config": {"workload": rec["workload"]}, "gpu_launches": rec["gpu_launches"], "final_error": rec["final_error"], "clocks": clocks,
              "iteration_roofline": rec["iteration_roofline"]})
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# (summary key, path into the full record): the main figure of every further workload, in the order the run makes them
SUMMARY = [
    ("iteration_frac", ("iteration_roofline", "survey_model", "frac")),
    ("single_ms", ("single_hologram", "ms_per_hologram")),
    ("gs_1024_its", ("configs", "gs_1024", "value")),
    ("fp64_gd_its", ("configs", "fp64", "gd", "value")),
    ("fp64_gd_verified", ("configs", "fp64", "gd", "verified")),
    ("fp64_gs_its", ("configs", "fp64", "gs", "value")),
    ("s4096_gd_its", ("configs", "size_4096", "gd", "value")),
    ("s4096_gs_its", ("configs", "size_4096", "gs", "value")),
    ("c1_dev_ms", ("configs", "config1", "device_ms_per_hologram")),
    ("c1_e2e_ms", ("configs", "config1", "e2e_ms_per_hologram")),
    ("c3_u8_hps", ("configs", "config3", "uint8_frames", "holograms_per_s")),
    ("c3_f64_hps", ("configs", "config3", "float64_holograms", "holograms_per_s")),
    ("c3_u8_raster_hps", ("configs", "config3", "uint8_frames_device_rasterised", "holograms_per_s")),
    ("c4_hps", ("configs", "config4", "holograms_per_s")),
    ("c5_gs_its", ("configs", "config5", "value")),
    ("c5_gd_its", ("configs", "config5_gd", "value")),
]


def result_line(full: dict) -> dict:
    """The stdout line of the batch workload (module docstring): the headline's own keys without the prose, then
    `summary`."""
    line = {k: full[k] for k in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                                 "scaling", "vs_baseline", "dtype", "data", "holograms_per_s", "gpu_launches", "clocks",
                                 "verified")}
    line["config"] = {k: full["config"][k] for k in ("workload", "algorithm", "shape", "batch_per_gpu", "iterations", "gd_form")}
    line["verification"] = {k: v for k, v in full["verification"].items() if k != "fixture"}
    if full.get("roofline"):
        line["roofline"] = {k: v for k, v in full["roofline"].items() if k != "note"}
    if full.get("cpu_baseline"):
        line["cpu_baseline"] = {k: full["cpu_baseline"][k] for k in ("value", "unit", "cores", "kind")}
    if full.get("e2e"):
        line["e2e"] = {k: full["e2e"][k] for k in ("value", "unit", "h2d_bytes_per_step", "d2h_bytes_per_step", "ms_per_hologram")}
    summary = {}
    for key, path in SUMMARY:
        v = full
        for p in path:
            v = v.get(p) if isinstance(v, dict) else None
        if v is not None:
            summary[key] = v
    line["summary"] = summary
    return line


def emit(line: dict) -> None:
    """The ONE JSON line of this run, on the process's real stdout."""
    os.write(_REAL_STDOUT, (json.dumps(line) + "\n").encode())


_REAL_STDOUT = 1

if __name__ == "__main__":
    sys.dont_write_bytecode = True      # a run leaves nothing in the source tree (which may be read-only)
    args = parse()
    # watchdog: a run that takes absurdly long (default 20 min; SLM_BENCH_WATCHDOG=seconds) dumps every thread's stack
    # to stderr and exits instead of hanging its launcher
    import faulthandler
    faulthandler.dump_traceback_later(float(os.environ.get("SLM_BENCH_WATCHDOG", "1200")), exit=True)
    # libraries (NCCL's version banner, ...) write to file descriptor 1: keep it for the JSON line alone
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    elif args.workload == "slab":
        run_slab(args)
    else:
        run_b200(args)
