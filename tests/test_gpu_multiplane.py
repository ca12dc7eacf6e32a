"""Multi-plane GS on the B200 at SLM and panel sizes: the checks of tests/test_emulated_multiplane.py
(tests/multiplane_checks.py) at 768x1024, 1024^2 and 1152x1920 with 2 and 4 planes, plus the property multi-plane GS
exists for -- traps in several focal planes from one hologram -- and the drop-in function end to end."""
import argparse
import contextlib
import io

import numpy as np
import pytest

from tests import multiplane_checks as mc

pytestmark = pytest.mark.gpu

SHAPES = [(768, 1024), (1024, 1024), (1152, 1920)]
PRECISIONS = ["fp32", "fp64"]


def make_engine(shape, precision, max_batch):
    from spatial_light_modulator_module_b200.engine import Engine
    return Engine(shape, precision, max_batch)


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("groups", ["plain", "pipeline"])
def test_one_plane_is_gs(monkeypatch, groups, precision):
    # SLM_NO_GROUPS=1: the one-CTA-per-tile column kernel; SLM_GS_GROUPS=1: the column pipeline
    monkeypatch.setenv("SLM_NO_GROUPS" if groups == "plain" else "SLM_GS_GROUPS", "1")
    mc.check_k1_is_gs(make_engine, (768, 1024), precision)


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("k", [2, 4])
@pytest.mark.parametrize("shape", SHAPES)
def test_teacher_forced(shape, k, precision):
    mc.check_teacher_forced(make_engine, shape, precision, k)


@pytest.mark.parametrize("k", [2, 4])
@pytest.mark.parametrize("shape", SHAPES)
def test_free_running_fp64(shape, k):
    """Ten iterations in one run track the oracle's run (GS's fp64 gates; the emulator measures 1e-13 at 192x256)."""
    curve, phase = mc.free_running_deviation(make_engine, shape, k)
    assert curve < 1e-10 and phase < 1e-10, (curve, phase)


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("shape", SHAPES)
def test_batch_equals_single_runs(shape, precision):
    mc.check_batch_equals_single_runs(make_engine, shape, precision)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_tolerance(precision):
    mc.check_tolerance(make_engine, (768, 1024), precision)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_argument_errors(precision):
    mc.check_argument_errors(make_engine, (768, 1024), precision)


# The oracle (oracle/multiplane.py) on the CPU, 3 planes of 12 single-pixel traps each at 768x1024 (trap_planes()),
# alpha = 0, +2e-3, -2e-3, 30 iterations: per plane, the share of its intensity on its own traps, and the mean on its
# traps over the mean on the other planes' traps.
ORACLE_SHARE = [0.26292559927944564, 0.26362841253320823, 0.26315087372753065]
ORACLE_RATIO = [14113.660724249341, 17848.693021664705, 25209.116411441606]
# Plain GS on the Fourier-plane target alone, 30 iterations, each lens applied to its hologram afterwards: the
# defocused planes get 1.7e-5 of their intensity on their traps, and no more there than on the other planes' traps.
GS_SHARE = [0.7936248021200267, 1.6815267060042555e-05, 1.641270720887861e-05]
GS_RATIO = [471241.0198515872, 1.035595865385792, 0.9984269004384992]


@pytest.mark.parametrize("precision", PRECISIONS)
def test_traps_in_three_planes(precision):
    shape = (768, 1024)
    planes, sets = mc.trap_planes(shape)
    al = [0.0, 2e-3, -2e-3]
    eng = make_engine(shape, precision, 3)
    res = eng.gs_multiplane(planes, al, 30)
    share, ratio = mc.intensity_scores(list(eng.to_host(res.expected)[0]), sets)
    np.testing.assert_allclose(share, ORACLE_SHARE, rtol=0.1)
    np.testing.assert_allclose(ratio, ORACLE_RATIO, rtol=0.1)
    # plain GS for the Fourier-plane traps, the lenses added afterwards, on the device
    from oracle import multiplane as MP
    r = eng.gs(planes[0], 30)
    h = eng.to_host(r.hologram)[0]
    fields = np.stack([np.exp(1j * h) * MP.lens_field(shape, a) for a in al])
    inten = np.abs(eng.to_host(eng.fft2(fields.astype(eng.complex_dtype)))) ** 2
    gs_share, gs_ratio = mc.intensity_scores(list(inten), sets)
    np.testing.assert_allclose(gs_share[1:], GS_SHARE[1:], rtol=0.5)
    for k in (1, 2):
        assert gs_share[k] < 1e-3 * share[k] and gs_ratio[k] < 10 and ratio[k] > 1e3
    eng.close()


def test_drop_in_end_to_end():
    from spatial_light_modulator_module_b200 import algorithms, constants, host_logic as hl
    from spatial_light_modulator_module_b200.display_holograms import hologram_to_grey
    shape = (768, 1024)
    planes, sets = mc.trap_planes(shape)
    f_min = constants.px_distance ** 2 * max(shape) / constants.wavelength          # 2.49 m
    fl = [None, 2 * f_min, -2 * f_min]
    args = argparse.Namespace(max_loops=20, tolerance=0, incomming_intensity="uniform", print_info=False,
                              plot_error=False, gif=False, precision="fp32")
    with contextlib.redirect_stdout(io.StringIO()):
        holo, exp, errs = algorithms.multiplane_gerchberg_saxton(list(planes), fl, args)
    assert holo.shape == shape and holo.dtype == np.float64 and exp.shape == (3,) + shape
    assert [len(e) for e in errs] == [20, 20, 20] and np.all(np.isfinite(errs))
    share, _ = mc.intensity_scores(list(exp), sets)
    assert min(share) > 0.2
    grey = hologram_to_grey(holo)
    assert grey.shape == shape and grey.dtype == np.uint8 and len(np.unique(grey)) > 200
    alphas = [hl.defocus_coefficient(f, constants.px_distance, constants.wavelength) for f in fl]
    eng = algorithms.get_engine(shape, "fp32", 3)
    r = eng.gs_multiplane(planes, alphas, 20)
    np.testing.assert_array_equal(holo, eng.to_host(r.hologram)[0])
