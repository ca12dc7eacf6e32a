"""Multi-plane GS checks shared by the CPU suite (host emulation of the kernel sources) and the GPU suite (the real
library on a B200).  Each check takes ``make_engine(shape, precision, max_batch)`` and compares
``Engine.gs_multiplane`` with the oracle (oracle/multiplane.py), with ``Engine.gs``, or with itself.

Tolerances are GS's (tests/parity_checks.py): fp64 error rel 1e-12, intensity 1e-12 of the plane's max, amplitude-
weighted phase 1e-10 rad; fp32 1e-5, 1e-5 and 1e-4 rad.
"""
from __future__ import annotations

import numpy as np
import pytest

from oracle import multiplane as MP
from oracle import numpy_port as P
from tests import parity_checks as pc

KINDS = ("noise", "shapes", "traps")
# defocus coefficients per plane count [rad / pixel^2] for planes of up to 256 points a side (|alpha| <= 0.012 keeps
# the phase step at the edge, |alpha| max(H, W), below pi); larger planes take them scaled by 256 / max(H, W)
ALPHAS = {1: [0.009], 2: [0.0, -0.012], 3: [0.0, 0.012, -0.007], 4: [0.0, 0.01, -0.008, 0.005]}


def alphas(shape, k):
    s = min(1.0, 256 / max(shape))
    return [a * s for a in ALPHAS[k]]


def trap_array(shape, n, seed):
    """``n`` single-pixel traps at seeded distinct places, clear of the edges by an eighth of the side (at most 64)."""
    rng = np.random.default_rng(seed)
    my, mx = min(64, shape[0] // 8), min(64, shape[1] // 8)
    cells = rng.choice((shape[0] - 2 * my) * (shape[1] - 2 * mx), n, replace=False)
    t = np.zeros(shape, np.uint8)
    t[my + cells // (shape[1] - 2 * mx), mx + cells % (shape[1] - 2 * mx)] = 255
    return t


def plane_targets(shape, k, offset=0):
    """``k`` different target planes: the synthetic kinds, then trap arrays."""
    kinds = pc.targets(shape)
    out = []
    for i in range(offset, offset + k):
        out.append(kinds[KINDS[i]] if i < len(KINDS) else trap_array(shape, 20, seed=i))
    return np.stack(out)


def check_k1_is_gs(make_engine, shape, precision, max_batch=1, loops=6):
    """planes = 1, alpha = 0: hologram, expected outcome and error curve are Engine.gs's bits, from the device setup
    (8-bit and real targets) and from a given first phasor, on the same engine."""
    eng = make_engine(shape, precision, max_batch)
    kinds = pc.targets(shape)
    for t in (kinds["noise"], kinds["shapes"], kinds["noise"].astype(np.float32)):
        for phasor in (None, P.gs_first_phasor(P.gs_setup(t))):
            r_gs = eng.gs(t, loops, phasor0=phasor)
            r_mp = eng.gs_multiplane(t[None], [0.0], loops, phasor0=phasor)
            np.testing.assert_array_equal(r_mp.errors[0][0], r_gs.errors[0])
            np.testing.assert_array_equal(eng.to_host(r_mp.hologram), eng.to_host(r_gs.hologram))
            np.testing.assert_array_equal(eng.to_host(r_mp.expected)[:, 0], eng.to_host(r_gs.expected))
    eng.close()


def check_teacher_forced(make_engine, shape, precision, k, steps=(0, 1, 2)):
    """The oracle's B entering iteration i -> ONE engine iteration from it -> every plane's error and expected outcome,
    and the hologram (amplitude-weighted phase of A), against the oracle's iteration from the same B."""
    tol = pc.TOL[precision]
    ts, al = plane_targets(shape, k), alphas(shape, k)
    eng = make_engine(shape, precision, k)
    st = MP.mp_setup(list(ts), al)
    for i in range(max(steps) + 1):
        B = MP.mp_first_phasor(st)
        if i in steps:
            fresh = MP.mp_start(list(ts), al, B)
            _, exps, errs = MP.mp_step(fresh)
            res = eng.gs_multiplane(ts, al, 1, phasor0=B)
            assert res.expected.shape == (1, k) + tuple(shape)
            for j in range(k):
                assert len(res.errors[0][j]) == 1
                assert abs(res.errors[0][j][0] - errs[j]) <= tol["err"] * abs(errs[j]), (j, res.errors[0][j][0], errs[j])
            exp = eng.to_host(res.expected)[0]
            for j in range(k):
                assert np.abs(exp[j] - exps[j]).max() <= tol["inten"] * exps[j].max()
            amp = np.abs(fresh.A) / np.abs(fresh.A).max()
            assert (pc.circ(eng.to_host(res.hologram)[0], np.angle(fresh.A)) * amp).max() < tol["wphase"]
        MP.mp_step(st)
    eng.close()


def free_running_deviation(make_engine, shape, k, loops=10):
    """fp64, ``loops`` iterations in one run from the oracle's first phasor: (largest relative error-curve deviation,
    amplitude-weighted hologram phase deviation [rad]) from the oracle's run."""
    ts, al = plane_targets(shape, k), alphas(shape, k)
    eng = make_engine(shape, "fp64", k)
    st = MP.mp_setup(list(ts), al)
    res = eng.gs_multiplane(ts, al, loops, phasor0=MP.mp_first_phasor(st))
    MP.mp_loop(st, loops)
    curve = max(np.max(np.abs(np.asarray(res.errors[0][j]) - st.errors[j]) / np.abs(st.errors[j])) for j in range(k))
    amp = np.abs(st.A) / np.abs(st.A).max()
    phase = (pc.circ(eng.to_host(res.hologram)[0], np.angle(st.A)) * amp).max()
    eng.close()
    return float(curve), float(phase)


def check_batch_equals_single_runs(make_engine, shape, precision, k=2, loops=5):
    """Three holograms of ``k`` planes (noise, shapes, traps and trap arrays, mixed differently in each) in one call
    give the bits of three one-hologram calls on the same context."""
    groups = [plane_targets(shape, k, offset=o) for o in (0, 1, 2)]
    al = alphas(shape, k)
    eng = make_engine(shape, precision, 3 * k)
    res = eng.gs_multiplane(np.stack(groups), al, loops)
    holo, exp = eng.to_host(res.hologram), eng.to_host(res.expected)
    assert holo.shape == (3,) + tuple(shape) and exp.shape == (3, k) + tuple(shape)
    for g, ts in enumerate(groups):
        r = eng.gs_multiplane(ts, al, loops)
        np.testing.assert_array_equal(holo[g], eng.to_host(r.hologram)[0])
        np.testing.assert_array_equal(exp[g], eng.to_host(r.expected)[0])
        for j in range(k):
            np.testing.assert_array_equal(res.errors[g][j], r.errors[0][j])
    eng.close()


def _stop(curves, tol, loops):
    """The oracle's loop condition over the planes: iterations run until every plane's error is <= tol."""
    worst = np.max(np.array(curves), axis=0)
    below = np.nonzero(~(worst > tol))[0]
    return int(below[0]) + 1 if below.size else loops


def check_tolerance(make_engine, shape, precision, loops=10):
    """Two holograms of two planes, one tolerance: each hologram's curves all have the oracle's length, the two stop
    at different iterations, and a plane below the tolerance early keeps iterating (its curve follows the oracle's)
    until the other plane of its hologram gets there too.  Both runs start from the oracle's first phasor."""
    tol_k = pc.TOL[precision]
    al = alphas(shape, 2)
    groups = [plane_targets(shape, 2, offset=1), plane_targets(shape, 2, offset=0)]
    states = [MP.mp_setup(list(ts), al) for ts in groups]
    phasors = np.stack([MP.mp_first_phasor(s) for s in states])
    curves = []
    for s in states:
        MP.mp_loop(s, loops)
        curves.append(s.errors)
    # a tolerance halfway (geometrically) between two neighbouring values of the holograms' worst-plane curves, so
    # that rounding cannot move a stop, with the holograms stopping at different iterations before max_loops
    worst = sorted(set(np.concatenate([np.max(np.array(c), axis=0) for c in curves])))
    tol = None
    for lo, hi in zip(worst[:-1], worst[1:]):
        cand = float(np.sqrt(lo * hi))
        stops = [_stop(c, cand, loops) for c in curves]
        if hi / lo > 1.01 and stops[0] != stops[1] and max(stops) < loops:
            tol = cand
            break
    assert tol is not None
    stops = [_stop(c, tol, loops) for c in curves]
    eng = make_engine(shape, precision, 4)
    res = eng.gs_multiplane(np.stack(groups), al, loops, tol, phasor0=phasors)
    early = False
    for g in range(2):
        assert res.iterations[g] == stops[g]
        for j in range(2):
            dev = np.asarray(res.errors[g][j])
            assert len(dev) == stops[g]
            ref = np.asarray(curves[g][j][:stops[g]])
            assert np.all(np.abs(dev - ref) <= 10 * tol_k["err"] * np.abs(ref))
            early = early or bool(np.any(~(ref[:-1] > tol)))
    assert early                                           # some plane was below the tolerance before its hologram stopped
    eng.close()


def intensity_scores(expected, trap_sets):
    """Per plane k: the share of its intensity on its own traps, and the mean intensity on its traps over the mean on
    the other planes' trap positions."""
    share, ratio = [], []
    for k, e in enumerate(expected):
        own = e[trap_sets[k]]
        other = np.concatenate([e[trap_sets[m]] for m in range(len(trap_sets)) if m != k])
        share.append(float(own.sum() / e.sum()))
        ratio.append(float(own.mean() / other.mean()))
    return share, ratio


def trap_planes(shape, k=3, n=12, seed=7):
    """``k`` target planes of ``n`` single-pixel traps each, all k*n positions distinct."""
    t = trap_array(shape, k * n, seed)
    ys, xs = np.nonzero(t)
    order = np.random.default_rng(seed).permutation(len(ys))
    planes = np.zeros((k,) + tuple(shape), np.uint8)
    sets = []
    for i in range(k):
        sel = order[i * n:(i + 1) * n]
        planes[i, ys[sel], xs[sel]] = 255
        sets.append(planes[i] > 0)
    return planes, sets


def check_argument_errors(make_engine, shape, precision):
    ts = plane_targets(shape, 2)
    eng = make_engine(shape, precision, 4)
    n = max(shape)
    with pytest.raises(ValueError, match="plane 1 aliases"):
        eng.gs_multiplane(ts, [0.0, 1.01 * np.pi / n], 2)
    with pytest.raises(ValueError, match="focal length"):
        eng.gs_multiplane(ts, [-1.01 * np.pi / n, 0.0], 2)
    with pytest.raises(ValueError, match="defocus coefficients"):
        eng.gs_multiplane(ts, [0.0], 2)
    with pytest.raises(ValueError, match="max_batch"):
        eng.gs_multiplane(np.stack([ts, ts, ts]), [0.0, 0.001], 2)
    with pytest.raises(ValueError, match="phasor0"):
        eng.gs_multiplane(ts, [0.0, 0.001], 2, phasor0=np.ones((2,) + tuple(shape), np.complex128))
    with pytest.raises(ValueError, match="phasor0"):
        eng.gs_multiplane(ts, [0.0, 0.001], 2, phasor0=np.ones((shape[0], shape[1] // 2), np.complex128))
    with pytest.raises(ValueError, match="not finite"):
        eng.gs_multiplane(ts, [0.0, float("nan")], 2)
    with pytest.raises(UnboundLocalError):
        eng.gs_multiplane(ts, [0.0, 0.001], 0)
    # the C ABI refuses by itself, naming the argument
    t8 = eng._mem_upload(np.concatenate([ts, ts]))
    holo = eng._mem_empty((4,) + tuple(shape), np.float64)
    norms = np.full(4, 255.0)

    def call(holograms, planes, alphas):
        d = None if alphas is None else eng._dp(np.ascontiguousarray(alphas, dtype=np.float64))
        rc = eng._lib.slm_gs_multiplane_run(eng._ctx, holograms, planes, eng._mem_ptr(t8), None, None,
                                            eng._dp(eng._amp_lut), eng._dp(norms), d, None, None, 1, 2, 0.0,
                                            eng._mem_ptr(holo), None)
        return rc, eng._lib.slm_last_error()
    for planes in (0, 9):
        rc, msg = call(1, planes, np.zeros(9))
        assert rc == -1 and b"planes" in msg
    rc, msg = call(3, 2, np.zeros(2))
    assert rc == -1 and b"holograms * planes" in msg
    rc, msg = call(1, 2, None)
    assert rc == -1 and b"defocus" in msg
    rc, msg = call(1, 2, [0.0, float("inf")])
    assert rc == -1 and b"defocus[1]" in msg
    assert call(2, 2, [0.0, 0.001])[0] == 0
    assert eng._lib.slm_version() == 104
    eng.close()
