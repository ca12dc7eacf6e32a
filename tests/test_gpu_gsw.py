"""Weighted GS on the B200 at SLM and panel sizes: the checks of tests/test_emulated_gsw.py (tests/gsw_checks.py) at
768x1024, 1024^2, 1152x1920 and 2048^2, plus the property GSW exists for -- even trap intensities -- the drop-in function
and the command line end to end, and a weighted movie with a ragged last batch."""
import argparse
import contextlib
import io
import os

import numpy as np
import pytest

from oracle import gsw as G
from oracle import numpy_port as P
from tests import gsw_checks as gc
from tests import parity_checks as pc

pytestmark = pytest.mark.gpu

SHAPES = [(768, 1024), (1024, 1024), (1152, 1920), (2048, 2048)]
PRECISIONS = ["fp32", "fp64"]


def make_engine(shape, precision, max_batch):
    from spatial_light_modulator_module_b200.engine import Engine
    return Engine(shape, precision, max_batch)


def quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("kind,dtype", [("noise", np.uint8), ("noise", np.float32)])
@pytest.mark.parametrize("shape", SHAPES)
def test_teacher_forced(shape, kind, dtype, precision):
    gc.check_teacher_forced(make_engine, shape, precision, kind, dtype)


@pytest.mark.parametrize("shape", SHAPES)
def test_free_running_fp64(shape):
    gc.check_free_running(make_engine, shape)


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("shape", SHAPES)
def test_weight_limit_one_is_gs(monkeypatch, shape, precision):
    # GS of a one-plane context takes the column pipeline where a plane has more tiles than the device has SMs (2048^2)
    monkeypatch.setenv("SLM_NO_GROUPS", "1")
    gc.check_weight_limit_one_is_gs(make_engine, shape, precision)


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("shape", SHAPES)
def test_batch_equals_single_runs(shape, precision):
    gc.check_batch_equals_single_runs(make_engine, shape, precision)


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("shape", SHAPES)
def test_planes_stop_independently(shape, precision):
    gc.check_tolerance_stops_planes(make_engine, shape, precision)


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("shape", SHAPES)
def test_weight_bounds(shape, precision):
    gc.check_weight_bounds(make_engine, shape, precision)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_argument_errors(precision):
    gc.check_argument_errors(make_engine, (768, 1024), precision)


def test_trap_array_intensities_768x1024():
    """200 single-pixel traps, 50 iterations from the device's own setup: GSW's coefficient of variation of I/T over
    the traps is below 1e-3 and GS's above 1e-2 -- first on the oracle, then on the device in both precisions."""
    shape = (768, 1024)
    t = gc.trap_array(shape)
    _, e_gs, _ = P.gs_run(t, 50)
    _, e_w, _, _ = G.gsw_run(t, 50)
    assert gc.intensity_cv(e_gs, t) > 1e-2 and gc.intensity_cv(e_w, t) < 1e-3
    for precision in PRECISIONS:
        eng = make_engine(shape, precision, 1)
        cv_gs = gc.intensity_cv(eng.to_host(eng.gs(t, 50).expected)[0], t)
        res, _ = eng.gsw(t, 50)
        cv_w = gc.intensity_cv(eng.to_host(res.expected)[0], t)
        print(f"\ntrap CV of I/T after 50 iterations, {precision}: GS {cv_gs:.3g}, GSW {cv_w:.3g}")
        assert cv_gs > 1e-2 and cv_w < 1e-3
        eng.close()


def ns(**kw):
    base = dict(incomming_intensity="uniform", tolerance=0, max_loops=10, gif=False, gif_skip=1, gif_type="i",
                print_info=False, plot_error=False, initial_guess="random", random_seed=42, white_attention=1,
                learning_rate=0.005, unsettle=0, correspond_to2pi=256)
    base.update(kw)
    return argparse.Namespace(**base)


def test_dropin_weighted_gs_768x1024():
    """algorithms.weighted_gerchberg_saxton on a trap array.  From the device's own setup a trap target's field is
    noise-seeded at its nodes (tests/parity_checks.check_gs_device_setup), so the run is held to the oracle's first
    error within 1e-2 and to what GSW must reach: even traps, a falling error, the expected outcome's max at the
    target's.  The result is the engine's own run bit for bit."""
    from spatial_light_modulator_module_b200 import algorithms, engine as E
    shape = (768, 1024)
    t = gc.trap_array(shape)
    holo, exp, errs = quiet(algorithms.weighted_gerchberg_saxton, t, ns(max_loops=30, precision="fp64", weight_limit=10.0))
    _, _, ref_errs, _ = G.gsw_run(t, 1)
    assert len(errs) == 30 and holo.shape == shape and np.all(np.abs(holo) <= np.pi + 1e-12)
    assert abs(errs[0] - ref_errs[0]) <= 1e-2 * ref_errs[0]
    assert abs(exp.max() - 255.0) < 1e-9 * 255
    assert gc.intensity_cv(exp, t) < 1e-3 and errs[-1] < errs[0]
    eng = E.get_engine(shape, "fp64")                    # the drop-in's own engine
    res, _ = eng.gsw(t, 30)
    np.testing.assert_array_equal(holo, eng.to_host(res.hologram)[0])


def test_generate_hologram_cli_weighted(tmp_path, monkeypatch):
    """generate_hologram's command line with -alg weighted_gerchberg_saxton writes the hologram of the drop-in call."""
    from PIL import Image as im
    from spatial_light_modulator_module_b200 import algorithms, generate_hologram as gh
    monkeypatch.chdir(tmp_path)
    os.makedirs("images")
    t = gc.trap_array((768, 1024), n=40, seed=7)
    im.fromarray(t).save("images/traps.png")
    quiet(gh.cli, ["traps.png", "-alg", "weighted_gerchberg_saxton", "--weight_limit", "5", "-l", "12",
                   "--precision", "fp64", "-dest_dir", "out"])
    files = os.listdir("out")
    assert len(files) == 1 and "_weighted_gerchberg_saxton" in files[0]
    saved = np.load(os.path.join("out", files[0]))
    a = gh.build_parser().parse_args(["traps.png", "--precision", "fp64", "-l", "12", "--weight_limit", "5"])
    a.random_seed, a.print_info, a.correspond_to2pi = 42, False, 256
    holo, _, _ = quiet(algorithms.weighted_gerchberg_saxton, gh.prepare_target("traps.png", a), a)
    np.testing.assert_array_equal(saved, holo)


def test_sequence_driver_weighted_ragged_batch():
    gc.check_sequence_driver(make_engine, (768, 1024), "fp64", n_frames=6, batch=4)


def test_sequence_driver_weighted_uint8_frames():
    """The weighted movie's 8-bit frames (output="uint8", floor rule of move_traps.py:135-140) are the frames of the
    float64 holograms of the same run."""
    from spatial_light_modulator_module_b200 import generate_hologram_sequence as ghs
    shape = (768, 1024)
    frames = np.stack([gc.trap_array(shape, n=30, seed=s) for s in range(5)])
    mask = np.random.default_rng(1).uniform(0, 2 * np.pi, size=shape)
    holos, _, _, _ = ghs.sequence_holograms(frames, 8, precision="fp32", batch=2, engine_factory=make_engine, weighted=True)
    q, _, _, _ = ghs.sequence_holograms(frames, 8, precision="fp32", batch=2, engine_factory=make_engine, weighted=True,
                                        output="uint8", mask=mask, ct2pi=256)
    np.testing.assert_array_equal(q, P.quantize_q3(holos, mask, 256))
