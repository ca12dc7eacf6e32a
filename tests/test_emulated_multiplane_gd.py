"""Multi-plane GD (Engine.gd_multiplane, row_multiplane_kernel<ALG_MPGD>) on the CPU through the host emulation of the
kernel sources (tests/emu): against the oracle (oracle/multiplane_gd.py), against GD with one plane at alpha = 0, and
against itself across batches and tolerance stops.  tests/test_gpu_multiplane_gd.py repeats the checks on the B200."""
import argparse
import contextlib
import io

import numpy as np
import pytest

from spatial_light_modulator_module_b200 import algorithms, constants, host_logic as hl
from tests import multiplane_checks as mc
from tests import multiplane_gd_checks as gc
from tests.emu.emu_engine import EmuEngine


def make_engine(shape, precision, max_batch):
    return EmuEngine(shape, precision, max_batch)


SHAPES = [(128, 128), (192, 256)]
PRECISIONS = ["fp32", "fp64"]


def test_oracle_one_plane_is_gd():
    gc.check_oracle_k1_is_gd_run()


# The emulated grid has 3 CTAs, so GD picks the fused form at 128^2; each form is forced in turn, and SLM_NO_GROUPS=1
# takes the one-CTA-per-tile column kernels.
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("form", ["two_pass", "fused", "pipe", "no_groups"])
def test_one_plane_is_gd(monkeypatch, form, precision):
    if form == "no_groups":
        monkeypatch.setenv("SLM_NO_GROUPS", "1")
    else:
        monkeypatch.setenv("SLM_GD_FORM", form)
    gc.check_k1_is_gd(make_engine, (128, 128), precision)


# fp32 columns of 768 and 1024 points run on the warp-per-column kernel (col_warp.cuh), in its fused and pipelined
# one-pass GD forms
@pytest.mark.parametrize("form", ["fused", "pipe"])
@pytest.mark.parametrize("rows", [768, 1024])
def test_one_plane_is_gd_warp_column_kernel(monkeypatch, rows, form):
    monkeypatch.setenv("SLM_GD_FORM", form)
    gc.check_k1_is_gd(make_engine, (rows, 64), "fp32", loops=3)


@pytest.mark.parametrize("form", ["fused", "pipe"])
@pytest.mark.parametrize("rows", [768, 1024])
def test_warp_column_kernel_free_running(monkeypatch, rows, form):
    monkeypatch.setenv("SLM_GD_FORM", form)
    gc.check_free_running(make_engine, (rows, 64), "fp32", 2, loops=4)


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("k", [1, 2, 3])
@pytest.mark.parametrize("shape", SHAPES)
def test_free_running(shape, k, precision):
    gc.check_free_running(make_engine, shape, precision, k)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_batch_equals_single_runs(precision):
    gc.check_batch_equals_single_runs(make_engine, (128, 128), precision)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_tolerance(precision):
    gc.check_tolerance(make_engine, (128, 128), precision)


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("k", [1, 3])
def test_fourier_guess(k, precision):
    gc.check_fourier_guess(make_engine, (128, 128), precision, k)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_argument_errors(precision):
    gc.check_argument_errors(make_engine, (128, 128), precision)


def ns(**kw):
    base = dict(incomming_intensity="uniform", tolerance=0, max_loops=6, gif=False, print_info=False, plot_error=False,
                initial_guess="random", random_seed=42, learning_rate=0.005, unsettle=2, white_attention=1)
    base.update(kw)
    return argparse.Namespace(**base)


@pytest.fixture
def emu_engines(monkeypatch):
    """algorithms.get_engine -> cached EmuEngines, one per (shape, precision)"""
    cache = {}

    def get_engine(shape, precision="fp32", max_batch=1, device=None):
        key = (tuple(int(s) for s in shape), precision)
        if key not in cache or cache[key].max_batch < max_batch:
            cache[key] = EmuEngine(key[0], precision, max_batch)
        return cache[key]
    monkeypatch.setattr(algorithms, "get_engine", get_engine)
    return cache


@pytest.mark.parametrize("guess", ["random", "old", "ones"])
@pytest.mark.parametrize("precision", PRECISIONS)
def test_drop_in_one_plane_is_gradient_descent(emu_engines, precision, guess):
    t = mc.plane_targets((128, 128), 1)[0]
    a1, a2 = ns(precision=precision, initial_guess=guess), ns(precision=precision, initial_guess=guess)
    with contextlib.redirect_stdout(io.StringIO()):
        h1, e1, r1 = algorithms.gradient_descent(t, a1)
        h2, e2, r2 = algorithms.multiplane_gradient_descent([t], [None], a2)
    np.testing.assert_array_equal(h1, h2)
    np.testing.assert_array_equal(e1, e2[0])
    assert r1 == r2[0] and all(isinstance(e, np.float64) for e in r2[0])
    assert a1.learning_rate == a2.learning_rate == 0.04                    # unsettle = 2: doubled at iterations 2, 4 and 6


def test_drop_in(emu_engines):
    ts = mc.plane_targets((128, 128), 3)
    fl = [None, 40.0, -60.0]
    args = ns(precision="fp64", print_info=True, initial_guess="fourier")
    with contextlib.redirect_stdout(io.StringIO()) as out:
        holo, exp, errs = algorithms.multiplane_gradient_descent(list(ts), fl, args)
    assert "loop 6/6" in out.getvalue() and "plane 2" in out.getvalue()
    assert args.learning_rate == 0.04
    eng = emu_engines[((128, 128), "fp64")]
    alphas = [hl.defocus_coefficient(f, constants.px_distance, constants.wavelength) for f in fl]
    x0 = eng.multiplane_fourier_guess(ts, alphas)
    during, _ = hl.learning_rate_schedule(0.005, 2, 6)
    res, _ = eng.gd_multiplane(ts, alphas, x0, during, 6)
    np.testing.assert_array_equal(holo, eng.to_host(res.hologram)[0])
    np.testing.assert_array_equal(exp, eng.to_host(res.expected)[0])
    assert holo.shape == (128, 128) and exp.shape == (3, 128, 128)
    assert [len(e) for e in errs] == [6, 6, 6]
    np.testing.assert_array_equal(np.array(errs), np.array(res.errors[0]))


def test_drop_in_refusals(emu_engines):
    ts = list(mc.plane_targets((128, 128), 2))
    with pytest.raises(ValueError, match="GIF"):
        algorithms.multiplane_gradient_descent(ts, [None, 50.0], ns(gif=True))
    with pytest.raises(ValueError, match="focal lengths"):
        algorithms.multiplane_gradient_descent(ts, [None], ns())
    with pytest.raises(ValueError, match="all zero"):
        algorithms.multiplane_gradient_descent([ts[0], np.zeros_like(ts[0])], [None, 50.0], ns())
    with pytest.raises(UnboundLocalError, match="output"):
        with contextlib.redirect_stdout(io.StringIO()):
            algorithms.multiplane_gradient_descent(ts, [None, 50.0], ns(max_loops=0))
    with pytest.raises(ValueError, match="aliases"):
        algorithms.multiplane_gradient_descent(ts, [None, 0.1], ns())
    assert "multiplane_gradient_descent" in algorithms.__all__
