"""Multi-plane GS and GD against GS and GD at a fixed number of planes in flight (32): plane-iterations/s of GS (GD)
on 32 planes and of multi-plane GS (GD) with K = 1, 2, 4 planes per hologram and 32 / K holograms, at 768x1024 and
1024^2 in fp32 and 1024^2 in fp64.  Device-resident uint8 noise targets, 100 iterations per run, no expected outcome;
defocus alpha = 0, +1e-3, -1e-3, +5e-4 for planes 0..3 (K = 1 is alpha = 0: the lens products are skipped, the
kernel's own overhead is left).  GD runs from a random phasor per hologram at the reference's learning rate, in the
Fourier-plane form the engine picks for 32 planes.  Rates are the median of REPEATS timed runs (torch.cuda.synchronize
around each, after WARMUP untimed runs).  From a separate profiled run (CUDA events around every launch,
Engine.profile): the SLM-plane (row) pass time per launch and per plane -- row_pass_kernel and row_multiplane_kernel --
and the plain column pass per plane (0 where the column groups run it).  Prints one JSON line, with the card's name,
power limit and clock.

    python profiles/multiplane_rate.py [gs] [gd]      (default: both)
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

LOOPS, WARMUP, REPEATS, PLANES = 100, 2, 5, 32
CASES = [((768, 1024), "fp32"), ((1024, 1024), "fp32"), ((1024, 1024), "fp64")]
ALPHAS = [0.0, 1e-3, -1e-3, 5e-4]


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


def pass_ms(eng, fn):
    """(row pass ms per launch, launches, column pass ms per launch) of one profiled run"""
    eng.profile(True)
    eng.profile_read()
    fn()
    prof = eng.profile_read()
    eng.profile(False)
    (rms, rn), (cms, cn) = prof["row_pass"], prof["col_pass"]
    return rms / max(rn, 1), rn, cms / max(cn, 1)


def rates(shape, precision, dev, alg):
    eng = Engine(shape, precision, PLANES)
    t = torch.from_numpy(np.stack([synthetic.noise_target(shape, seed=i + 1) for i in range(PLANES)])).to(dev)
    norms = t.reshape(PLANES, -1).amax(dim=1).double().cpu().numpy()
    lr = np.full(LOOPS, 0.005)

    def x0(n):
        return eng.random_phasor_guess(np.random.default_rng(n).random((n,) + shape))
    if alg == "gs":
        runs = [("gs", lambda: eng.gs(t, LOOPS, want_expected=False, norms=norms))]
    else:
        x = x0(PLANES)
        runs = [("gd", lambda: eng.gd(t, x, lr, LOOPS, want_expected=False, norms=norms))]
    for k in (1, 2, 4):
        g = PLANES // k
        tk = t.reshape(g, k, *shape)
        if alg == "gs":
            runs.append((f"mp{k}", lambda tk=tk, k=k: eng.gs_multiplane(tk, ALPHAS[:k], LOOPS, want_expected=False, norms=norms)))
        else:
            runs.append((f"mp{k}", lambda tk=tk, k=k, x=x0(g): eng.gd_multiplane(tk, ALPHAS[:k], x, lr, LOOPS,
                                                                                 want_expected=False, norms=norms)))
    rec = {"algorithm": alg, "shape": list(shape), "precision": precision, "planes": PLANES}
    for name, fn in runs:
        med, all_s = timed(fn)
        row_ms, row_n, col_ms = pass_ms(eng, fn)
        rec[name] = {"plane_it_s": round(PLANES * LOOPS / med, 1), "runs_ms": [round(1e3 * s, 3) for s in all_s],
                     "row_ms_per_launch": round(row_ms, 4), "row_launches": row_n,
                     "row_ms_per_plane": round(row_ms / PLANES, 5), "col_ms_per_plane": round(col_ms / PLANES, 5)}
    for k in (1, 2, 4):
        rec[f"mp{k}_vs_{alg}"] = round(rec[f"mp{k}"]["plane_it_s"] / rec[alg]["plane_it_s"], 3)
        rec[f"mp{k}_row_vs_{alg}_row"] = round(rec[f"mp{k}"]["row_ms_per_plane"] / rec[alg]["row_ms_per_plane"], 3)
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
    algs = sys.argv[1:] or ["gs", "gd"]
    out = {"card": card(), "loops": LOOPS, "repeats": REPEATS,
           "cases": [rates(s, p, dev, a) for a in algs for s, p in CASES]}
    print(json.dumps(out))


if __name__ == "__main__":
    main()
