"""Multi-plane GD checks shared by the CPU suite (host emulation of the kernel sources) and the GPU suite (the real
library on a B200).  Each check takes ``make_engine(shape, precision, max_batch)`` and compares
``Engine.gd_multiplane`` with the oracle (oracle/multiplane_gd.py), with ``Engine.gd``, or with itself.

Tolerances are GD's (tests/parity_checks.py TOL): fp64 error curve rel 1e-9, phase 1e-8 rad, intensity 1e-10 of the
plane's max; fp32 1e-4, 1e-3 rad and 1e-4.  The phase is weighted by |x| / max |x|, as multi-plane GS weights it by
|A|: where x is small its phase carries no light.
"""
from __future__ import annotations

import numpy as np
import pytest

from oracle import multiplane as MP
from oracle import multiplane_gd as MPGD
from oracle import numpy_port as P
from spatial_light_modulator_module_b200 import host_logic as hl
from tests import multiplane_checks as mc
from tests import parity_checks as pc


def x0_for(shape, seed=42):
    return hl.host_initial_guess("random", shape, seed)


def weighted_phase(holo, x):
    """Largest |x|-weighted distance [rad] between ``holo`` and angle(x)."""
    return float((pc.circ(holo, np.angle(x)) * np.abs(x) / np.abs(x).max()).max())


def check_oracle_k1_is_gd_run(shape=(128, 128), loops=8):
    """The oracle with one plane at alpha = 0 is numpy_port.gd_run bit for bit: hologram, output, error curve and final
    learning rate, with the unsettle rule doubling the rate during the run."""
    for kind in ("noise", "shapes"):
        t = pc.targets(shape)[kind]
        x0 = x0_for(shape)
        h1, o1, e1, lr1 = P.gd_run(t, loops, x0=x0, unsettle=3, learning_rate=0.01)
        h2, o2, e2, lr2 = MPGD.mpgd_run([t], [0.0], x0, loops, unsettle=3, learning_rate=0.01)
        np.testing.assert_array_equal(h1, h2)
        np.testing.assert_array_equal(o1, o2[0])
        assert e1 == e2[0] and lr1 == lr2 == 0.16                     # doubled at iterations 2, 4, 6 and 8


def check_k1_is_gd(make_engine, shape, precision, loops=5):
    """planes = 1, alpha = 0: hologram, expected outcome, error curve and final x are Engine.gd's bits, for 8-bit and
    real targets, with uniform and non-uniform illumination, under whatever GD form the environment selects."""
    eng = make_engine(shape, precision, 1)
    kinds = pc.targets(shape)
    inc = np.sqrt(1.0 + 0.5 * np.cos(np.arange(shape[1]) / 7.0)[None, :] * np.ones((shape[0], 1)))
    during, _ = hl.learning_rate_schedule(0.005, 1, loops)
    for t in (kinds["noise"], kinds["shapes"], kinds["noise"].astype(np.float32)):
        for illum in (None, inc):
            x0 = x0_for(shape)
            r_gd, x_gd = eng.gd(t, x0, during, loops, inc_amp=illum)
            r_mp, x_mp = eng.gd_multiplane(t[None], [0.0], x0, during, loops, inc_amp=illum)
            np.testing.assert_array_equal(r_mp.errors[0][0], r_gd.errors[0])
            np.testing.assert_array_equal(eng.to_host(r_mp.hologram), eng.to_host(r_gd.hologram))
            np.testing.assert_array_equal(eng.to_host(r_mp.expected)[:, 0], eng.to_host(r_gd.expected))
            np.testing.assert_array_equal(eng.to_host(x_mp), eng.to_host(x_gd))
    eng.close()


def free_running_deviation(make_engine, shape, precision, k, loops=10):
    """``loops`` iterations in one run from the oracle's x0: (largest relative error-curve deviation, |x|-weighted
    hologram phase deviation [rad], largest intensity deviation relative to each plane's max) from the oracle's run."""
    ts, al = mc.plane_targets(shape, k), mc.alphas(shape, k)
    x0 = x0_for(shape)
    during, _ = hl.learning_rate_schedule(0.005, 0, loops)
    eng = make_engine(shape, precision, k)
    res, _ = eng.gd_multiplane(ts, al, x0, during, loops)
    st = MPGD.mpgd_setup(list(ts), al, x0, max_loops=loops)
    _, outs, errs, _ = MPGD.mpgd_loop(st)
    curve = max(np.max(np.abs(np.asarray(res.errors[0][j]) - errs[j]) / np.abs(errs[j])) for j in range(k))
    phase = weighted_phase(eng.to_host(res.hologram)[0], st.x)
    exp = eng.to_host(res.expected)[0]
    inten = max(np.abs(exp[j] - outs[j]).max() / outs[j].max() for j in range(k))
    eng.close()
    return float(curve), phase, float(inten)


def check_free_running(make_engine, shape, precision, k, loops=10):
    tol = pc.TOL[precision]
    curve, phase, inten = free_running_deviation(make_engine, shape, precision, k, loops)
    assert curve < tol["gd_curve"] and phase < tol["gd_phase"] and inten < tol["gd_inten"], (curve, phase, inten)


def check_batch_equals_single_runs(make_engine, shape, precision, k=2, loops=5):
    """Three holograms of ``k`` planes, each from its own x0, in one call give the bits of three one-hologram calls."""
    groups = [mc.plane_targets(shape, k, offset=o) for o in (0, 1, 2)]
    x0s = np.stack([x0_for(shape, 42 + g) for g in range(3)])
    al = mc.alphas(shape, k)
    during, _ = hl.learning_rate_schedule(0.005, 0, loops)
    eng = make_engine(shape, precision, 3 * k)
    res, x = eng.gd_multiplane(np.stack(groups), al, x0s.copy(), during, loops)
    holo, exp, xb = eng.to_host(res.hologram), eng.to_host(res.expected), eng.to_host(x)
    assert holo.shape == (3,) + tuple(shape) and exp.shape == (3, k) + tuple(shape)
    for g, ts in enumerate(groups):
        r, x1 = eng.gd_multiplane(ts, al, x0s[g], during, loops)
        np.testing.assert_array_equal(holo[g], eng.to_host(r.hologram)[0])
        np.testing.assert_array_equal(exp[g], eng.to_host(r.expected)[0])
        np.testing.assert_array_equal(xb[g], eng.to_host(x1)[0])
        for j in range(k):
            np.testing.assert_array_equal(res.errors[g][j], r.errors[0][j])
    eng.close()


def check_tolerance(make_engine, shape, precision, loops=10):
    """Two holograms of two planes, one tolerance: each hologram stops where the oracle stops (all its curves that
    long), the two stop at different iterations, a plane below the tolerance early keeps iterating until its
    hologram stops, and the final holograms match the oracle's -- which they would not if the update of the last
    iteration were skipped or applied twice (checked against the oracle's x one update either side)."""
    tol_k = pc.TOL[precision]
    al = mc.alphas(shape, 2)
    groups = [mc.plane_targets(shape, 2, offset=1), mc.plane_targets(shape, 2, offset=0)]
    x0s = np.stack([x0_for(shape, 42 + g) for g in range(2)])
    curves = []
    for g, ts in enumerate(groups):
        st = MPGD.mpgd_setup(list(ts), al, x0s[g], max_loops=loops)
        MPGD.mpgd_loop(st)
        curves.append(st.errors)
    worst = sorted(set(np.concatenate([np.max(np.array(c), axis=0) for c in curves])))
    tol = None
    for lo, hi in zip(worst[:-1], worst[1:]):
        cand = float(np.sqrt(lo * hi))
        stops = [mc._stop(c, cand, loops) for c in curves]
        if hi / lo > 1.01 and stops[0] != stops[1] and max(stops) < loops - 1:
            tol = cand
            break
    assert tol is not None
    stops = [mc._stop(c, tol, loops) for c in curves]
    during, _ = hl.learning_rate_schedule(0.005, 0, loops)
    eng = make_engine(shape, precision, 4)
    res, _ = eng.gd_multiplane(np.stack(groups), al, x0s.copy(), during, loops, tol)
    holo = eng.to_host(res.hologram)
    early = False
    for g, ts in enumerate(groups):
        assert res.iterations[g] == stops[g]
        for j in range(2):
            dev = np.asarray(res.errors[g][j])
            assert len(dev) == stops[g]
            ref = np.asarray(curves[g][j][:stops[g]])
            assert np.all(np.abs(dev - ref) <= 10 * tol_k["gd_curve"] * np.abs(ref))
            early = early or bool(np.any(~(ref[:-1] > tol)))
        # the oracle's x after stops - 1, stops and stops + 1 updates
        st = MPGD.mpgd_setup(list(ts), al, x0s[g], max_loops=loops)
        xs = [None] * 3
        for i in range(stops[g] + 1):
            if i >= stops[g] - 1:
                xs[i - stops[g] + 1] = st.x.copy()
            MPGD.mpgd_step(st)
        xs[2] = st.x.copy()
        d = [weighted_phase(holo[g], x) for x in xs]
        assert d[1] < tol_k["gd_phase"], d
        assert d[0] > 10 * tol_k["gd_phase"] and d[2] > 10 * tol_k["gd_phase"], d
    assert early
    eng.close()


def check_fourier_guess(make_engine, shape, precision, k):
    """The multi-plane "fourier" guess against the oracle, at GS's setup tolerances (tests/multiplane_checks.py's
    amplitude-weighted phase of A): |x| = inc, and the phase weighted by |A|.  8-bit targets take the complex64
    setup, so they are held to the fp32 gate in both precisions."""
    ts, al = mc.plane_targets(shape, k), mc.alphas(shape, k)
    eng = make_engine(shape, precision, k)
    inc = np.sqrt(1.0 + 0.5 * np.cos(np.arange(shape[0]) / 5.0)[:, None] * np.ones((1, shape[1])))
    for targets, c64 in ((ts, True), (ts.astype(np.float64), precision == "fp32")):
        for illum in (None, inc):
            x = eng.to_host(eng.multiplane_fourier_guess(targets, al, illum))
            assert x.shape == (1,) + tuple(shape)
            ref = MPGD.fourier_guess(list(targets), al, "uniform" if illum is None else illum ** 2)
            A = MP.mp_setup(list(targets), al).A
            amp = np.abs(A) / np.abs(A).max()
            gate = pc.TOL["fp32" if c64 else precision]["wphase"]
            assert (pc.circ(np.angle(x[0]), np.angle(ref)) * amp).max() < gate
            assert np.abs(np.abs(x[0]) - np.abs(ref)).max() < pc.TOL[precision]["fft"] * np.abs(ref).max()
    eng.close()
    # two one-plane holograms in one call: each its own guess, bit for bit
    pair = mc.plane_targets(shape, 2)
    eng = make_engine(shape, precision, 2)
    both = eng.to_host(eng.multiplane_fourier_guess(pair[:, None], al[:1]))
    for g in range(2):
        np.testing.assert_array_equal(both[g], eng.to_host(eng.multiplane_fourier_guess(pair[g:g + 1], al[:1]))[0])
    eng.close()


def check_argument_errors(make_engine, shape, precision):
    ts = mc.plane_targets(shape, 2)
    eng = make_engine(shape, precision, 4)
    n = max(shape)
    x0 = x0_for(shape)
    lr = np.full(2, 0.005)
    with pytest.raises(ValueError, match="plane 1 aliases"):
        eng.gd_multiplane(ts, [0.0, 1.01 * np.pi / n], x0, lr, 2)
    with pytest.raises(ValueError, match="defocus coefficients"):
        eng.gd_multiplane(ts, [0.0], x0, lr, 2)
    with pytest.raises(ValueError, match="max_batch"):
        eng.gd_multiplane(np.stack([ts, ts, ts]), [0.0, 0.001], np.stack([x0] * 3), lr, 2)
    with pytest.raises(ValueError, match="multi-plane GD takes 1 to 8"):
        eng.gd_multiplane(np.zeros((9,) + tuple(shape), np.uint8), np.zeros(9), x0, lr, 2)
    with pytest.raises(ValueError, match="x0"):
        eng.gd_multiplane(ts, [0.0, 0.001], np.stack([x0, x0]), lr, 2)
    with pytest.raises(ValueError, match="x0"):
        eng.gd_multiplane(ts, [0.0, 0.001], x0[:, : shape[1] // 2], lr, 2)
    with pytest.raises(ValueError, match="lr_schedule"):
        eng.gd_multiplane(ts, [0.0, 0.001], x0, np.full(3, 0.005), 2)
    with pytest.raises(ValueError, match="not finite"):
        eng.gd_multiplane(ts, [0.0, float("nan")], x0, lr, 2)
    with pytest.raises(UnboundLocalError, match="output"):
        eng.gd_multiplane(ts, [0.0, 0.001], x0, np.zeros(0), 0)
    with pytest.raises(ValueError, match="aliases"):
        eng.multiplane_fourier_guess(ts, [0.0, 1.01 * np.pi / n])
    # the C ABI refuses by itself, naming the argument
    t8 = eng._mem_upload(np.concatenate([ts, ts]))
    holo = eng._mem_empty((4,) + tuple(shape), np.float64)
    x = eng._mem_upload(np.stack([x0, x0]).astype(eng.complex_dtype))
    xg = eng._mem_empty((2,) + tuple(shape), eng.complex_dtype)
    norms = np.full(4, 255.0)
    mask_lut = hl.gd_mask_lut(1)

    def call(holograms, planes, alphas):
        d = None if alphas is None else eng._dp(np.ascontiguousarray(alphas, dtype=np.float64))
        rc = eng._lib.slm_gd_multiplane_run(eng._ctx, holograms, planes, eng._mem_ptr(t8), None, None, eng._dp(mask_lut),
                                            eng._dp(norms), d, None, eng._mem_ptr(x), eng._dp(lr), 2, 0.0,
                                            eng._mem_ptr(holo), None)
        return rc, eng._lib.slm_last_error()

    def guess(holograms, planes, alphas):
        d = None if alphas is None else eng._dp(np.ascontiguousarray(alphas, dtype=np.float64))
        rc = eng._lib.slm_multiplane_fourier_guess(eng._ctx, holograms, planes, eng._mem_ptr(t8), None,
                                                   eng._dp(eng._amp_lut), d, None, 1, eng._mem_ptr(xg))
        return rc, eng._lib.slm_last_error()
    for fn, who in ((call, b"slm_gd_multiplane_run"), (guess, b"slm_multiplane_fourier_guess")):
        for planes in (0, 9):
            rc, msg = fn(1, planes, np.zeros(9))
            assert rc == -1 and b"planes" in msg and who in msg
        rc, msg = fn(3, 2, np.zeros(2))
        assert rc == -1 and b"holograms * planes" in msg
        rc, msg = fn(1, 2, None)
        assert rc == -1 and b"defocus" in msg
        rc, msg = fn(1, 2, [0.0, float("inf")])
        assert rc == -1 and b"defocus[1]" in msg
        assert fn(2, 2, [0.0, 0.001])[0] == 0
    assert eng._lib.slm_version() == 104
    eng.close()


# ---- traps in three planes (tests/test_gpu_multiplane_gd.py) ------------------------------------------------------
TRAP_SHAPE, TRAP_ALPHAS, TRAP_LOOPS, TRAP_LR = (768, 1024), [0.0, 2e-3, -2e-3], 50, 0.005


def trap_evenness(expected, trap_sets):
    """Per plane: the spread of its traps' intensities, std / mean."""
    return [float(np.std(e[s]) / np.mean(e[s])) for e, s in zip(expected, trap_sets)]


def oracle_trap_scores():
    """The oracle on the CPU: 3 planes of 12 traps (multiplane_checks.trap_planes) at TRAP_SHAPE and TRAP_ALPHAS,
    TRAP_LOOPS iterations at the reference's learning rate from the multi-plane "fourier" guess -> (share, ratio) per
    plane (multiplane_checks.intensity_scores); and plain GD on the Fourier-plane target from its own "fourier" guess,
    each lens applied to its hologram afterwards -> (share, ratio)."""
    from scipy.fft import fft2
    planes, sets = mc.trap_planes(TRAP_SHAPE)
    x0 = MPGD.fourier_guess(list(planes), TRAP_ALPHAS)
    _, outs, _, _ = MPGD.mpgd_run(list(planes), TRAP_ALPHAS, x0, TRAP_LOOPS, learning_rate=TRAP_LR)
    h, _, _, _ = P.gd_run(planes[0], TRAP_LOOPS, initial_guess_kind="fourier", learning_rate=TRAP_LR)
    inten = [np.abs(fft2(np.exp(1j * h) * MP.lens_field(TRAP_SHAPE, a))) ** 2 for a in TRAP_ALPHAS]
    return mc.intensity_scores(outs, sets), mc.intensity_scores(inten, sets)
