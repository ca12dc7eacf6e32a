"""Weighted GS (Engine.gsw, col_pass_tile<ALG_GSW>, col_gsw_stats_kernel) on the CPU through the host emulation of
the kernel sources (tests/emu): against the oracle (oracle/gsw.py), against GS with weight_limit = 1, and against
itself across batches and tolerance stops.  tests/test_gpu_gsw.py repeats the checks on the B200."""
import argparse

import numpy as np
import pytest

from oracle import gsw as G
from tests import gsw_checks as gc
from tests.emu.emu_engine import EmuEngine


def make_engine(shape, precision, max_batch):
    return EmuEngine(shape, precision, max_batch)


SHAPES = [(128, 128), (192, 256)]
PRECISIONS = ["fp32", "fp64"]


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("kind,dtype", [("noise", np.uint8), ("traps", np.uint8), ("noise", np.float32)])
@pytest.mark.parametrize("shape", SHAPES)
def test_teacher_forced(shape, kind, dtype, precision):
    gc.check_teacher_forced(make_engine, shape, precision, kind, dtype)


@pytest.mark.parametrize("shape", SHAPES)
def test_free_running_fp64(shape):
    gc.check_free_running(make_engine, shape)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_weight_limit_one_is_gs(monkeypatch, precision):
    monkeypatch.setenv("SLM_NO_GROUPS", "1")             # the emulated grid has 3 CTAs: GS would take the column pipeline
    gc.check_weight_limit_one_is_gs(make_engine, (128, 128), precision)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_batch_equals_single_runs(precision):
    gc.check_batch_equals_single_runs(make_engine, (128, 128), precision)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_planes_stop_independently(precision):
    gc.check_tolerance_stops_planes(make_engine, (128, 128), precision)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_weight_bounds(precision):
    gc.check_weight_bounds(make_engine, (128, 128), precision)


@pytest.mark.parametrize("precision", PRECISIONS)
def test_argument_errors(precision):
    gc.check_argument_errors(make_engine, (128, 128), precision)


def test_sequence_driver_weighted():
    gc.check_sequence_driver(make_engine, (128, 128), "fp64", n_frames=3, batch=2)


def test_oracle_trap_gates_small():
    """The oracle itself at 256^2 (the issue's evidence): GSW evens out the traps that GS leaves uneven."""
    from oracle import numpy_port as P
    shape = (256, 256)
    rng = np.random.default_rng(0)
    t = np.zeros(shape, np.uint8)
    t[rng.integers(20, 236, 25), rng.integers(20, 236, 25)] = 255
    _, e_gs, _ = P.gs_run(t, 50)
    _, e_w, errs, w = G.gsw_run(t, 50)
    assert gc.intensity_cv(e_gs, t) > 1e-2 and gc.intensity_cv(e_w, t) < 1e-10
    assert errs[-1] < 0.1 * errs[0]


def test_weighted_gs_refuses_gif_snapshots():
    from spatial_light_modulator_module_b200 import algorithms
    a = argparse.Namespace(gif=True, max_loops=3, tolerance=0, incomming_intensity="uniform")
    with pytest.raises(ValueError, match="GIF"):
        algorithms.weighted_gerchberg_saxton(np.zeros((64, 64), np.uint8), a)


def test_command_lines_route_weighted_gs():
    from spatial_light_modulator_module_b200 import algorithms, generate_hologram as gh, generate_hologram_sequence as ghs
    a = gh.build_parser().parse_args(["t.png", "-alg", "weighted_gerchberg_saxton", "--weight_limit", "4"])
    assert gh.ALGORITHMS[a.algorithm] is algorithms.weighted_gerchberg_saxton and a.weight_limit == 4.0
    assert gh.ALGORITHMS[gh.build_parser().parse_args(["t.png", "-alg", "gradient_descent"]).algorithm] is algorithms.gradient_descent
    assert gh.build_parser().parse_args(["t.png"]).weight_limit == 10.0
    s = ghs.build_parser().parse_args(["d", "-ct2pi", "256", "--weighted", "--weight_limit", "3"])
    assert s.weighted and s.weight_limit == 3.0
    assert not ghs.build_parser().parse_args(["d", "-ct2pi", "256"]).weighted
