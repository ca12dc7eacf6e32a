"""Multi-plane GS (Engine.gs_multiplane, row_multiplane_kernel) on the CPU through the host emulation of the kernel
sources (tests/emu): against the oracle (oracle/multiplane.py), against GS with one plane at alpha = 0, and against
itself across batches and tolerance stops.  tests/test_gpu_multiplane.py repeats the checks on the B200."""
import argparse
import contextlib
import io

import numpy as np
import pytest

from oracle import multiplane as MP
from oracle import numpy_port as P
from spatial_light_modulator_module_b200 import algorithms, constants, host_logic as hl
from tests import multiplane_checks as mc
from tests import parity_checks as pc
from tests.emu.emu_engine import EmuEngine


def make_engine(shape, precision, max_batch):
    return EmuEngine(shape, precision, max_batch)


SHAPES = [(128, 128), (192, 256)]
PRECISIONS = ["fp32", "fp64"]


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("groups", ["plain", "pipeline"])
def test_one_plane_is_gs(monkeypatch, groups, precision):
    # the emulated grid has 3 CTAs: GS takes the column pipeline unless the column groups are off
    monkeypatch.setenv("SLM_NO_GROUPS" if groups == "plain" else "SLM_GS_GROUPS", "1")
    mc.check_k1_is_gs(make_engine, (128, 128), precision)


def test_oracle_one_plane_is_gs():
    for kind in ("noise", "shapes"):
        t = pc.targets((128, 128))[kind]
        h1, e1, r1 = P.gs_run(t, 6)
        h2, e2, r2 = MP.mp_run([t], [0.0], 6)
        np.testing.assert_array_equal(h1, h2)
        np.testing.assert_array_equal(e1, e2[0])
        assert r1 == r2[0]


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("k", [1, 2, 3])
@pytest.mark.parametrize("shape", SHAPES)
def test_teacher_forced(shape, k, precision):
    mc.check_teacher_forced(make_engine, shape, precision, k)


@pytest.mark.parametrize("k", [2, 3])
@pytest.mark.parametrize("shape", SHAPES)
def test_free_running_fp64(shape, k):
    """Ten iterations in one run track the oracle's run.  Measured on this emulator: error curves within 1.2e-14
    (128^2) and 8.8e-14 (192x256) relative, hologram within 8.2e-14 and 6.3e-13 rad (amplitude-weighted); the gates
    leave a factor of ten or more.  (One plane with a lens does not track: the lens cancels between the two passes,
    so the run is plain GS, whose rounding differences grow -- 0.4 of the error at 192x256 after ten iterations.)"""
    curve, phase = mc.free_running_deviation(make_engine, shape, k)
    assert curve < 1e-12 and phase < 1e-11, (curve, phase)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_batch_equals_single_runs(precision):
    mc.check_batch_equals_single_runs(make_engine, (128, 128), precision)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_tolerance(precision):
    mc.check_tolerance(make_engine, (128, 128), precision)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_argument_errors(precision):
    mc.check_argument_errors(make_engine, (128, 128), precision)


def test_defocus_coefficient_and_aliasing_limit():
    px, lam = constants.px_distance, constants.wavelength
    assert hl.defocus_coefficient(None, px, lam) == 0.0 and hl.defocus_coefficient(float("inf"), px, lam) == 0.0
    assert MP.defocus_coefficient(2.0) == hl.defocus_coefficient(2.0, px, lam) == -np.pi * px ** 2 / (lam * 2.0)
    # the shortest focal lengths the refusal allows with the project's constants: 2.49 m at 768x1024, 4.68 m at 1152x1920
    for shape, f_min in (((768, 1024), 2.49), ((1152, 1920), 4.68)):
        hl.check_defocus([hl.defocus_coefficient(f_min * 1.01, px, lam)], shape, px, lam)
        hl.check_defocus([hl.defocus_coefficient(-f_min * 1.01, px, lam)], shape, px, lam)
        with pytest.raises(ValueError, match=f"{f_min:.3g} m"):
            hl.check_defocus([0.0, hl.defocus_coefficient(f_min * 0.99, px, lam)], shape, px, lam)


def test_paraxial_lens_matches_reference_lens():
    """alpha rho^2 is the reference's lens phase k (1 - sqrt(1 + r^2 / f^2)) up to its next term, k r^4 / (8 f^3):
    0.027 rad at the corners of a 768x1024 plane at the shortest focal length allowed there."""
    px, lam, f = constants.px_distance, constants.wavelength, 2.5
    i = np.arange(768)[:, None] - 384.0
    j = np.arange(1024)[None, :] - 512.0
    r2 = (i * i + j * j) * px ** 2
    exact = 2 * np.pi * f / lam * (1 - np.sqrt(1 + r2 / f ** 2))
    paraxial = hl.defocus_coefficient(f, px, lam) * (i * i + j * j)
    quartic = 2 * np.pi * f / lam * r2 ** 2 / (8 * f ** 4)
    assert np.abs(exact - paraxial).max() < 0.03
    assert np.abs(exact - paraxial - quartic).max() < 1e-4


def ns(**kw):
    base = dict(incomming_intensity="uniform", tolerance=0, max_loops=5, gif=False, print_info=False, plot_error=False)
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


def test_drop_in(emu_engines):
    ts = mc.plane_targets((128, 128), 3)
    fl = [None, 40.0, -60.0]
    with contextlib.redirect_stdout(io.StringIO()) as out:
        holo, exp, errs = algorithms.multiplane_gerchberg_saxton(list(ts), fl, ns(precision="fp64", print_info=True))
    assert "loop 5/5" in out.getvalue() and "plane 2" in out.getvalue()
    eng = emu_engines[((128, 128), "fp64")]
    res = eng.gs_multiplane(ts, [hl.defocus_coefficient(f, constants.px_distance, constants.wavelength) for f in fl], 5)
    np.testing.assert_array_equal(holo, eng.to_host(res.hologram)[0])
    np.testing.assert_array_equal(exp, eng.to_host(res.expected)[0])
    assert holo.shape == (128, 128) and exp.shape == (3, 128, 128)
    assert [len(e) for e in errs] == [5, 5, 5] and all(isinstance(e, np.float64) for e in errs[0])
    np.testing.assert_array_equal(np.array(errs), np.array(res.errors[0]))


def test_drop_in_refusals(emu_engines):
    ts = list(mc.plane_targets((128, 128), 2))
    with pytest.raises(ValueError, match="GIF"):
        algorithms.multiplane_gerchberg_saxton(ts, [None, 50.0], ns(gif=True))
    with pytest.raises(ValueError, match="focal lengths"):
        algorithms.multiplane_gerchberg_saxton(ts, [None], ns())
    with pytest.raises(ValueError, match="all zero"):
        algorithms.multiplane_gerchberg_saxton([ts[0], np.zeros_like(ts[0])], [None, 50.0], ns())
    with pytest.raises(UnboundLocalError):
        with contextlib.redirect_stdout(io.StringIO()):
            algorithms.multiplane_gerchberg_saxton(ts, [None, 50.0], ns(max_loops=0))
    with pytest.raises(ValueError, match="aliases"):
        algorithms.multiplane_gerchberg_saxton(ts, [None, 0.1], ns())
