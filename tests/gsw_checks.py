"""Weighted GS checks shared by the CPU suite (host emulation of the kernel sources) and the GPU suite (the real
library on a B200).  Each check takes ``make_engine(shape, precision, max_batch)`` and compares ``Engine.gsw`` with the
oracle (oracle/gsw.py), with ``Engine.gs``, or with itself.

Tolerances are GS's (tests/parity_checks.py): fp64 error rel 1e-12, amplitude-weighted phase 1e-10 rad; fp32 1e-5 and
1e-4 rad.  Weights are held to the phase's bound, weighted by |C| / max |C| the same way: where |C| is small, so is the
accuracy of |C|^2 and of the weight made from it.
"""
from __future__ import annotations

import numpy as np
import pytest

from oracle import gsw as G
from oracle import numpy_port as P
from tests import parity_checks as pc


def target(shape, kind, dtype=np.uint8):
    t = pc.targets(shape)[kind]
    return t if dtype == np.uint8 else t.astype(dtype)


def trap_array(shape, n=200, seed=1):
    """``n`` single-pixel traps at seeded random places, clear of the edges by an eighth of the side (at most 64)."""
    rng = np.random.default_rng(seed)
    t = np.zeros(shape, np.uint8)
    my, mx = min(64, shape[0] // 8), min(64, shape[1] // 8)
    t[rng.integers(my, shape[0] - my, n), rng.integers(mx, shape[1] - mx, n)] = 255
    return t


def intensity_cv(expected, t):
    """coefficient of variation of I / T over the signal set"""
    v = expected[t > 0] / t[t > 0].astype(np.float64)
    return float(v.std() / v.mean())


def check_teacher_forced(make_engine, shape, precision, kind="noise", dtype=np.uint8, steps=(0, 1, 4)):
    """The oracle's state entering iteration k (B_k, w_{k-1}) -> ONE engine iteration from it -> error, expected
    outcome, angle of the next field and the weights w_k against the oracle's iteration from the same state."""
    tol = pc.TOL[precision]
    t = target(shape, kind, dtype)
    eng = make_engine(shape, precision, 1)
    st = G.gsw_setup(t)
    for k in range(max(steps) + 1):
        B, w0 = st.B.copy(), st.w.copy()
        G.gsw_step(st)
        if k not in steps:
            continue
        fresh = G.gsw_start(t, B, w0)
        C, exp_ref, err_ref = G.gsw_step(fresh)
        res, w = eng.gsw(t, 1, phasor0=B, weights=w0)
        assert len(res.errors[0]) == 1
        assert abs(res.errors[0][0] - err_ref) <= tol["err"] * abs(err_ref) + 1e-300
        exp = eng.to_host(res.expected)[0]
        assert np.abs(exp - exp_ref).max() <= tol["inten"] * exp_ref.max()
        holo = eng.to_host(res.hologram)[0]
        amp = np.abs(fresh.A) / np.abs(fresh.A).max()
        assert (pc.circ(holo, np.angle(fresh.A)) * amp).max() < tol["wphase"]
        cw = np.abs(C) / np.abs(C).max()
        assert (np.abs(eng.to_host(w)[0] - fresh.w) / fresh.w * cw).max() < tol["wphase"]
    eng.close()


def check_free_running(make_engine, shape, loops=3):
    """fp64, three iterations in one run from the oracle's B_0: inside a run sigma_k = S_T / P_{k-1} lags P by one
    iteration.  On a trap array the weights stay far from the clamp, so sigma scales them uniformly: the lag shows in
    the weights (taking sigma from the pass's own P moves them by 1.5e-5 at 2048^2, 3e-3 at 128^2, amplitude-weighted)
    and nowhere else, and the run stays as close to the oracle as one teacher-forced iteration.  (On the noise target,
    where many weights sit at the clamp, rounding differences grow about 1000-fold per iteration, more at larger
    planes, so a free run there cannot be held to a fixed bound.)"""
    t = trap_array(shape)
    eng = make_engine(shape, "fp64", 1)
    st = G.gsw_setup(t)
    res, w = eng.gsw(t, loops, phasor0=st.B.copy())
    for _ in range(loops):
        C, _, _ = G.gsw_step(st)
    assert np.max(np.abs(res.errors[0] - st.errors) / np.array(st.errors)) < 1e-10
    amp = np.abs(st.A) / np.abs(st.A).max()
    assert (pc.circ(eng.to_host(res.hologram)[0], np.angle(st.A)) * amp).max() < 1e-10
    cw = np.abs(C) / np.abs(C).max()
    assert (np.abs(eng.to_host(w)[0] - st.w) / st.w * cw).max() < 1e-10
    eng.close()


def check_weight_limit_one_is_gs(make_engine, shape, precision, loops=6):
    """c = 1: the weights stay exactly 1.0 and hologram, expected outcome and error curve are GS's bits (one-plane
    context, where GS runs on the one-CTA-per-tile column kernel too), from the device setup and from a given field."""
    for t in (target(shape, "noise"), target(shape, "shapes"), target(shape, "noise", np.float32)):
        eng = make_engine(shape, precision, 1)
        for phasor in (None, P.gs_first_phasor(P.gs_setup(t))):
            r_gs = eng.gs(t, loops, phasor0=phasor)
            r_w, w = eng.gsw(t, loops, phasor0=phasor, weight_limit=1.0)
            np.testing.assert_array_equal(r_w.errors[0], r_gs.errors[0])
            np.testing.assert_array_equal(eng.to_host(r_w.hologram), eng.to_host(r_gs.hologram))
            np.testing.assert_array_equal(eng.to_host(r_w.expected), eng.to_host(r_gs.expected))
            assert np.all(eng.to_host(w) == 1.0)
        eng.close()


def check_batch_equals_single_runs(make_engine, shape, precision, loops=5):
    """Four different targets in one batch give the bits of four one-plane runs in the same context."""
    ts = [target(shape, "noise"), target(shape, "shapes"), target(shape, "traps"),
          trap_array(shape, n=20, seed=3) if min(shape) > 128 else target(shape, "noise")[::-1].copy()]
    eng = make_engine(shape, precision, 4)
    res, w = eng.gsw(np.stack(ts), loops)
    holo, exp, wts = eng.to_host(res.hologram), eng.to_host(res.expected), eng.to_host(w)
    for i, t in enumerate(ts):
        r, wi = eng.gsw(t, loops)
        np.testing.assert_array_equal(res.errors[i], r.errors[0])
        np.testing.assert_array_equal(holo[i], eng.to_host(r.hologram)[0])
        np.testing.assert_array_equal(exp[i], eng.to_host(r.expected)[0])
        np.testing.assert_array_equal(wts[i], eng.to_host(wi)[0])
    eng.close()


def check_tolerance_stops_planes(make_engine, shape, precision, loops=10):
    """Loop condition per plane: the planes of one batch stop independently, each equal to its one-plane run, and a
    plane that stopped early equals (weights included) a run of exactly that many iterations."""
    order = ["noise", "shapes", "traps"]
    tt = {k: target(shape, k) for k in order}
    eng = make_engine(shape, precision, 3)
    singles = {}
    for k in order:
        r, w = eng.gsw(tt[k], loops)
        singles[k] = (r.errors[0], eng.to_host(r.hologram)[0], eng.to_host(w)[0])
    e_sh = singles["shapes"][0]
    tol = float(np.sort(e_sh)[len(e_sh) // 2])
    res, w = eng.gsw(np.stack([tt[k] for k in order]), loops, tol)
    holo, wts = eng.to_host(res.hologram), eng.to_host(w)
    stops = []
    for i, k in enumerate(order):
        ref = singles[k][0]
        stop = int(np.argmax(~(ref > tol))) + 1 if np.any(~(ref > tol)) else loops
        stops.append(stop)
        assert len(res.errors[i]) == stop == res.iterations[i]
        np.testing.assert_array_equal(res.errors[i], ref[:stop])
        r2, w2 = eng.gsw(tt[k], stop)
        np.testing.assert_array_equal(holo[i], eng.to_host(r2.hologram)[0])
        np.testing.assert_array_equal(wts[i], eng.to_host(w2)[0])
    assert min(stops) < loops
    eng.close()


def check_weight_bounds(make_engine, shape, precision, loops=8):
    """Weights stay finite and within [1/c, c] (c = 3 and 10), and keep their initial values off the signal set."""
    rdt = np.float32 if precision == "fp32" else np.float64
    eng = make_engine(shape, precision, 2)
    t = np.stack([target(shape, "noise"), target(shape, "traps")])
    t[0, :5] = 0                                          # some dark pixels in the dense target too
    w0 = np.ones(t.shape)
    w0[t == 0] = 7.5                                      # off the signal set: must come back unchanged
    for c in (3.0, 10.0):
        _, w = eng.gsw(t, loops, weight_limit=c, weights=w0)
        wd = eng.to_host(w)
        on = t > 0
        assert np.all(np.isfinite(wd))
        assert wd[on].min() >= rdt(1 / c) and wd[on].max() <= rdt(c)
        assert np.all(wd[~on] == 7.5)
        assert wd[on].min() < 1 < wd[on].max()          # the weights did move
    eng.close()


def check_argument_errors(make_engine, shape, precision):
    t = target(shape, "noise")
    eng = make_engine(shape, precision, 2)
    for c in (0.5, 0.0, -1.0, float("nan")):
        with pytest.raises(ValueError):
            eng.gsw(t, 3, weight_limit=c)
    with pytest.raises(ValueError):
        eng.gsw(t, 3, weights=np.ones((2,) + shape))                 # batch of 1, weights for 2
    with pytest.raises(ValueError):
        eng.gsw(t, 3, weights=np.ones((shape[0], shape[1] // 2)))
    wrong = np.float64 if precision == "fp32" else np.float32
    with pytest.raises(TypeError):
        eng.gsw(t, 3, weights=eng._mem_upload(np.ones((1,) + shape, wrong)))
    with pytest.raises(UnboundLocalError):
        eng.gsw(t, 0)
    # the C ABI refuses a weight limit below 1 (and NaN) by itself
    w = eng._mem_upload(np.ones((1,) + shape, eng.real_dtype))
    holo = eng._mem_empty((1,) + shape, np.float64)
    norms, sums = np.array([float(t.max())]), np.array([float(t.sum())])
    for c in (0.999, float("nan")):
        rc = eng._lib.slm_gsw_run(eng._ctx, 1, eng._mem_ptr(eng._mem_upload(t[None])), None, None, eng._dp(eng._amp_lut),
                                  eng._dp(norms), None, None, 1, 2, 0.0, eng._mem_ptr(holo), None, eng._dp(sums),
                                  eng._mem_ptr(w), c)
        assert rc == -1 and b"weight_limit" in eng._lib.slm_last_error()
    assert eng._lib.slm_version() == 104
    eng.close()


def check_sequence_driver(make_engine, shape, precision, n_frames=6, batch=4, loops=3):
    """A weighted movie in batches with a ragged tail: every frame equals its one-plane GSW run bit for bit (weights
    start at 1 for every frame)."""
    from spatial_light_modulator_module_b200 import generate_hologram_sequence as ghs
    frames = np.stack([trap_array(shape, n=30, seed=s) for s in range(n_frames)])
    holos, exps, errors, _ = ghs.sequence_holograms(frames, loops, precision=precision, batch=batch, want_expected=True,
                                                    engine_factory=make_engine, weighted=True, weight_limit=5.0)
    eng = make_engine(shape, precision, 1)
    for i in range(n_frames):
        r, _ = eng.gsw(frames[i], loops, weight_limit=5.0)
        np.testing.assert_array_equal(holos[i], eng.to_host(r.hologram)[0])
        np.testing.assert_array_equal(exps[i], eng.to_host(r.expected)[0])
        np.testing.assert_array_equal(errors[i], r.errors[0])
    eng.close()
