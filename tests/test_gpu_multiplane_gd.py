"""Multi-plane GD on the B200 at SLM and panel sizes: the checks of tests/test_emulated_multiplane_gd.py
(tests/multiplane_gd_checks.py) at 768x1024, 1024^2 and 1152x1920 with 2 and 4 planes, one plane against GD under each
Fourier-plane form, the property multi-plane GD exists for -- traps in several focal planes from one hologram -- and
the drop-in function end to end."""
import argparse
import contextlib
import io

import numpy as np
import pytest

from tests import multiplane_checks as mc
from tests import multiplane_gd_checks as gc

pytestmark = pytest.mark.gpu

SHAPES = [(768, 1024), (1024, 1024), (1152, 1920)]
PRECISIONS = ["fp32", "fp64"]


def make_engine(shape, precision, max_batch):
    from spatial_light_modulator_module_b200.engine import Engine
    return Engine(shape, precision, max_batch)


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("form", ["two_pass", "fused", "pipe", "no_groups"])
def test_one_plane_is_gd(monkeypatch, form, precision):
    if form == "no_groups":
        monkeypatch.setenv("SLM_NO_GROUPS", "1")
    else:
        monkeypatch.setenv("SLM_GD_FORM", form)
    gc.check_k1_is_gd(make_engine, (768, 1024), precision)


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("k", [2, 4])
@pytest.mark.parametrize("shape", SHAPES)
def test_free_running(shape, k, precision):
    gc.check_free_running(make_engine, shape, precision, k)


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("shape", SHAPES)
def test_batch_equals_single_runs(shape, precision):
    gc.check_batch_equals_single_runs(make_engine, shape, precision)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_tolerance(precision):
    gc.check_tolerance(make_engine, (768, 1024), precision)


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("k", [2, 4])
def test_fourier_guess(k, precision):
    gc.check_fourier_guess(make_engine, (768, 1024), precision, k)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_argument_errors(precision):
    gc.check_argument_errors(make_engine, (768, 1024), precision)


# The oracle on the CPU (oracle/multiplane_gd.py), 3 planes of 12 single-pixel traps each at 768x1024, alpha = 0,
# +2e-3, -2e-3, 50 iterations at learning rate 0.005 from the multi-plane "fourier" guess: per plane, the share of its
# intensity on its own traps and the mean on its traps over the mean on the other planes' traps; then plain GD on the
# Fourier-plane target from its own "fourier" guess, each lens applied to its hologram afterwards.  Produced by
#     python -c "from tests import multiplane_gd_checks as g; print(g.oracle_trap_scores())"
ORACLE_SHARE = [0.26182046185506697, 0.26333524835956634, 0.2634759686030083]
ORACLE_RATIO = [13783.775848915771, 17499.760142494026, 25723.164066823054]
GD_SHARE = [0.7934125619222016, 1.6946397965073276e-05, 1.637473728225413e-05]
GD_RATIO = [504287.58652623586, 1.0574315723354402, 1.003856546553973]


@pytest.mark.parametrize("precision", PRECISIONS)
def test_traps_in_three_planes(precision):
    shape, al = gc.TRAP_SHAPE, gc.TRAP_ALPHAS
    planes, sets = mc.trap_planes(shape)
    eng = make_engine(shape, precision, 3)
    x0 = eng.multiplane_fourier_guess(planes, al)
    res, _ = eng.gd_multiplane(planes, al, x0, np.full(gc.TRAP_LOOPS, gc.TRAP_LR), gc.TRAP_LOOPS)
    exp = list(eng.to_host(res.expected)[0])
    share, ratio = mc.intensity_scores(exp, sets)
    np.testing.assert_allclose(share, ORACLE_SHARE, rtol=0.1)
    np.testing.assert_allclose(ratio, ORACLE_RATIO, rtol=0.1)
    # plain GD for the Fourier-plane traps, the lenses added afterwards, on the device
    from oracle import multiplane as MP
    r, _ = eng.gd(planes[0], eng.fourier_guess(planes[0]), np.full(gc.TRAP_LOOPS, gc.TRAP_LR), gc.TRAP_LOOPS)
    h = eng.to_host(r.hologram)[0]
    fields = np.stack([np.exp(1j * h) * MP.lens_field(shape, a) for a in al])
    inten = np.abs(eng.to_host(eng.fft2(fields.astype(eng.complex_dtype)))) ** 2
    gd_share, gd_ratio = mc.intensity_scores(list(inten), sets)
    np.testing.assert_allclose(gd_share[1:], GD_SHARE[1:], rtol=0.5)
    for k in (1, 2):
        assert gd_share[k] < 1e-3 * share[k] and gd_ratio[k] < 10 and ratio[k] > 1e3
    # reported, not gated: how even the trap intensities are (std / mean per plane) against multi-plane GS's
    gs = eng.gs_multiplane(planes, al, gc.TRAP_LOOPS)
    print(f"\ntrap evenness {precision}: multi-plane GD {gc.trap_evenness(exp, sets)}, "
          f"multi-plane GS {gc.trap_evenness(list(eng.to_host(gs.expected)[0]), sets)}")
    eng.close()


def test_drop_in_end_to_end():
    from spatial_light_modulator_module_b200 import algorithms, constants, host_logic as hl
    from spatial_light_modulator_module_b200.display_holograms import hologram_to_grey
    shape = gc.TRAP_SHAPE
    planes, sets = mc.trap_planes(shape)
    f_min = constants.px_distance ** 2 * max(shape) / constants.wavelength          # 2.49 m
    fl = [None, 2 * f_min, -2 * f_min]
    args = argparse.Namespace(max_loops=20, tolerance=0, incomming_intensity="uniform", print_info=False,
                              plot_error=False, gif=False, precision="fp32", initial_guess="fourier", random_seed=42,
                              learning_rate=0.005, unsettle=1, white_attention=1)
    with contextlib.redirect_stdout(io.StringIO()):
        holo, exp, errs = algorithms.multiplane_gradient_descent(list(planes), fl, args)
    assert holo.shape == shape and holo.dtype == np.float64 and exp.shape == (3,) + shape
    assert [len(e) for e in errs] == [20, 20, 20] and np.all(np.isfinite(errs))
    assert args.learning_rate == 0.02
    share, _ = mc.intensity_scores(list(exp), sets)
    assert min(share) > 0.2
    grey = hologram_to_grey(holo)
    assert grey.shape == shape and grey.dtype == np.uint8 and len(np.unique(grey)) > 200
    alphas = [hl.defocus_coefficient(f, constants.px_distance, constants.wavelength) for f in fl]
    eng = algorithms.get_engine(shape, "fp32", 3)
    during, _ = hl.learning_rate_schedule(0.005, 1, 20)
    r, _ = eng.gd_multiplane(planes, alphas, eng.multiplane_fourier_guess(planes, alphas), during, 20)
    np.testing.assert_array_equal(holo, eng.to_host(r.hologram)[0])
