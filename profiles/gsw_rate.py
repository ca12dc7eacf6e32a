"""GS and weighted GS (GSW) iterations/s and column-pass time per iteration: fp32 at 32 x 1024^2, 32 x 768x1024 and
8 x 1152x1920, fp64 at 16 x 1024^2.  Device-resident uint8 noise targets, 100 iterations per run, no expected outcome;
GSW starts every run from weights of 1 (copied in before the run, inside the timed window: one plane-stack copy).  Rates
are the median of REPEATS timed runs (torch.cuda.synchronize around each, after WARMUP untimed runs).  The column-pass
time comes from a separate profiled run (CUDA events around every launch, Engine.profile): its total over the run's
column passes / iterations.  Prints one JSON line, with the card's name, power limit and clock.

    python profiles/gsw_rate.py
"""
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
from spatial_light_modulator_module_b200 import synthetic  # noqa: E402
from spatial_light_modulator_module_b200.engine import Engine  # noqa: E402

LOOPS, WARMUP, REPEATS = 100, 2, 5
CASES = [((1024, 1024), 32, "fp32"), ((768, 1024), 32, "fp32"), ((1152, 1920), 8, "fp32"), ((1024, 1024), 16, "fp64")]


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


def col_pass_ms(eng, fn):
    """column-pass milliseconds per iteration of one profiled run (the GS / GSW Fourier-plane pass only; the max
    pre-pass of iteration 0 is a launch kind of its own)"""
    eng.profile(True)
    eng.profile_read()
    fn()
    prof = eng.profile_read()
    eng.profile(False)
    ms, n = prof["col_pass"]
    return round(ms / max(n, 1), 4), n


def rates(shape, batch, precision, dev):
    eng = Engine(shape, precision, batch)
    t = torch.from_numpy(np.stack([synthetic.noise_target(shape, seed=i + 1) for i in range(batch)])).to(dev)
    norms = t.reshape(batch, -1).amax(dim=1).double().cpu().numpy()
    ones = torch.ones((batch,) + shape, dtype=torch.float32 if precision == "fp32" else torch.float64, device=dev)
    w = torch.empty_like(ones)

    def gs():
        eng.gs(t, LOOPS, want_expected=False, norms=norms)

    def gsw():
        w.copy_(ones)
        eng.gsw(t, LOOPS, weights=w, want_expected=False, norms=norms)

    rec = {"shape": list(shape), "batch": batch, "precision": precision}
    for name, fn in (("gs", gs), ("gsw", gsw)):
        med, all_s = timed(fn)
        rec[name + "_it_s"] = round(batch * LOOPS / med, 1)
        rec[name + "_runs_ms"] = [round(1e3 * s, 3) for s in all_s]
        rec[name + "_col_pass_ms"], rec[name + "_col_passes"] = col_pass_ms(eng, fn)
    rec["gsw_vs_gs"] = round(rec["gsw_it_s"] / rec["gs_it_s"], 3)
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


def main():
    dev = torch.device("cuda", 0)
    out = {"card": card(), "loops": LOOPS, "repeats": REPEATS, "cases": [rates(s, b, p, dev) for s, b, p in CASES]}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
