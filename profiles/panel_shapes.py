"""GS and GD iterations/s at the 1920x1152 / 1280x1024 panel shapes and 1920^2, beside in-process controls at 2048^2 and
4096^2 that run the same column kernels; fp32, and fp64 at 1152x1920 and 1024x1280 beside an fp64 2048^2 control.
Device resident, 100 iterations per hologram; every figure is the median
of REPEATS timed runs (torch.cuda.synchronize around each, after WARMUP untimed runs).  Also one 100-iteration GD
hologram at 1152x1920 through the drop-in algorithms.gradient_descent(target, args), and the fraction of the HBM peak the
SURVEY 8(d) byte model of bench.py implies.  Prints one JSON line.

    python profiles/panel_shapes.py
"""
import argparse
import contextlib
import io
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from spatial_light_modulator_module_b200 import algorithms, host_logic as hl, synthetic  # noqa: E402
from spatial_light_modulator_module_b200.engine import Engine  # noqa: E402

LOOPS, WARMUP, REPEATS = 100, 2, 5
HBM_GBS = 8000.0                       # B200 HBM3e nominal
CASES = [((1152, 1920), 8, "fp32"), ((1024, 1280), 8, "fp32"), ((1920, 1920), 8, "fp32"), ((2048, 2048), 8, "fp32"),
         ((4096, 4096), 2, "fp32"), ((1152, 1920), 8, "fp64"), ((1024, 1280), 8, "fp64"), ((2048, 2048), 8, "fp64")]


def survey_bytes_per_px(alg, precision):
    """SURVEY.md 8(d), as bench.py: four passes per iteration -- GS (8c+4), GD (9c+4) bytes per pixel."""
    c = 8 if precision == "fp32" else 16
    return (8 * c + 4) if alg == "gs" else (9 * c + 4)


def timed(fn):
    for _ in range(WARMUP):
        fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(REPEATS):
        t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize()
        out.append(time.perf_counter() - t0)
    return statistics.median(out), out


def rates(shape, batch, precision, dev):
    eng = Engine(shape, precision, batch)
    t = torch.from_numpy(np.stack([synthetic.noise_target(shape, seed=i + 1) for i in range(batch)])).to(dev)
    norms = t.reshape(batch, -1).amax(dim=1).double().cpu().numpy()
    x0 = torch.from_numpy(np.exp(2j * np.pi * np.random.default_rng(0).random((batch,) + shape)).astype(eng.complex_dtype)).to(dev)
    x = torch.empty_like(x0)
    during, _ = hl.learning_rate_schedule(0.005, 0, LOOPS)

    def gd():
        x.copy_(x0)
        eng.gd(t, x, during, LOOPS, want_expected=False, norms=norms)

    def gs():
        eng.gs(t, LOOPS, want_expected=False, norms=norms)

    npx = shape[0] * shape[1]
    rec = {"shape": list(shape), "batch": batch, "precision": precision, "mpx": npx / 1e6}
    for name, fn in (("gd", gd), ("gs", gs)):
        med, all_s = timed(fn)
        its = batch * LOOPS / med
        rec[name + "_it_s"] = round(its, 1)
        rec[name + "_px_it_s"] = its * npx                     # per-pixel rate: comparable across shapes
        rec[name + "_runs_ms"] = [round(1e3 * s, 3) for s in all_s]
        rec[name + "_survey_frac"] = round(survey_bytes_per_px(name, precision) * npx * its / 1e9 / HBM_GBS, 4)
    eng.close()
    return rec


def card():
    props = torch.cuda.get_device_properties(0)
    info = {"name": props.name}
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        info["nvidia_smi"] = q
    except Exception as e:                                    # noqa: BLE001 -- reported, not fatal
        info["nvidia_smi"] = f"unavailable: {e}"
    return info


def dropin_gd():
    shape = (1152, 1920)
    tgt = synthetic.noise_target(shape, seed=3)
    args = argparse.Namespace(incomming_intensity="uniform", tolerance=0, max_loops=LOOPS, gif=False, gif_skip=1,
                              gif_type="i", print_info=False, plot_error=False, initial_guess="random", random_seed=42,
                              white_attention=1, learning_rate=0.005, unsettle=0, correspond_to2pi=256, precision="fp32")
    with contextlib.redirect_stdout(io.StringIO()):
        algorithms.gradient_descent(tgt, args)                 # first call: context, graph capture
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        algorithms.gradient_descent(tgt, args)
        torch.cuda.synchronize()
    return {"shape": list(shape), "iterations": LOOPS, "ms": round(1e3 * (time.perf_counter() - t0), 2)}


def main():
    dev = torch.device("cuda", 0)
    out = {"card": card(), "loops": LOOPS, "repeats": REPEATS, "hbm_gbs_model": HBM_GBS, "cases": []}
    for shape, batch, precision in CASES:
        out["cases"].append(rates(shape, batch, precision, dev))
    ctl = next(c for c in out["cases"] if c["shape"] == [4096, 4096])
    for c in out["cases"]:
        if c["precision"] != "fp32":
            continue
        for k in ("gd", "gs"):
            c[k + "_per_px_vs_4096"] = round(c[k + "_px_it_s"] / ctl[k + "_px_it_s"], 3)
    out["dropin_gd_1152x1920"] = dropin_gd()
    print(json.dumps(out))


if __name__ == "__main__":
    main()
