"""The drop-in functions of algorithms.py (gerchberg_saxton, weighted_gerchberg_saxton, gradient_descent) on the CPU:
``algorithms.get_engine`` hands out engines over the host emulation of the kernel sources (tests/emu), so the whole
call runs -- argument checks, GIF chunks, progress text -- as it does on the B200 (tests/test_gpu_parity.py)."""
import argparse
import contextlib
import io
import random

import numpy as np
import pytest

from spatial_light_modulator_module_b200 import algorithms, synthetic
from tests import parity_checks as pc
from tests.emu.emu_engine import EmuEngine


def ns(**kw):
    base = dict(incomming_intensity="uniform", tolerance=0, max_loops=10, gif=False, gif_skip=1, gif_type="i",
                print_info=False, plot_error=False, initial_guess="random", random_seed=42, white_attention=1,
                learning_rate=0.005, unsettle=0, correspond_to2pi=256)
    base.update(kw)
    return argparse.Namespace(**base)


def quiet(fn, *a, **k):
    with contextlib.redirect_stdout(io.StringIO()):
        return fn(*a, **k)


@pytest.fixture
def emu_engines(monkeypatch):
    """algorithms.get_engine -> cached EmuEngines, one per (shape, precision), grown like the package's cache."""
    cache = {}

    def get_engine(shape, precision="fp32", max_batch=1, device=None):
        key = (tuple(int(s) for s in shape), precision)
        if key not in cache or cache[key].max_batch < max_batch:
            cache[key] = EmuEngine(key[0], precision, max_batch)
        return cache[key]
    monkeypatch.setattr(algorithms, "get_engine", get_engine)
    yield cache
    for eng in cache.values():
        eng.close()


@pytest.mark.parametrize("precision", ["fp32", "fp64"])
def test_gif_snapshots(emu_engines, tmp_path, precision):
    pc.check_gif_snapshots(None, precision, tmp_path,
                           lambda t, a: quiet(algorithms.gerchberg_saxton, t, a),
                           lambda t, a: quiet(algorithms.gradient_descent, t, a), ns)


def test_gif_gs_launches(emu_engines, tmp_path):
    """A GS run with GIF snapshots makes the launches of its chunks, and one phasor launch after every chunk that does
    not end the run -- the last chunk of a run that reaches max_loops included."""
    from spatial_light_modulator_module_b200 import host_logic as hl
    t = synthetic.shapes_target((128, 128))
    a = ns(max_loops=7, gif=True, gif_skip=3, gif_source_dir=str(tmp_path), precision="fp64")
    quiet(algorithms.gerchberg_saxton, t, a)
    eng = emu_engines[((128, 128), "fp64")]
    n0 = eng.launch_count()
    quiet(algorithms.gerchberg_saxton, t, a)
    gif = eng.launch_count() - n0
    n0, phasor = eng.launch_count(), None
    for n in hl.snapshot_chunks(7, 3):
        phasor = eng.phase_phasor(eng.gs(t, n, phasor0=phasor).hologram)
    assert gif == eng.launch_count() - n0


@pytest.mark.parametrize("precision", ["fp32", "fp64"])
def test_weighted_drop_in_is_engine_gsw(emu_engines, precision):
    t = synthetic.traps_target((128, 128))
    holo, exp, errs = quiet(algorithms.weighted_gerchberg_saxton, t, ns(max_loops=6, weight_limit=3.0, precision=precision))
    eng = EmuEngine((128, 128), precision, 1)
    res, _w = eng.gsw(t, 6, 0.0, weight_limit=3.0)
    np.testing.assert_array_equal(holo, eng.to_host(res.hologram)[0])
    np.testing.assert_array_equal(exp, eng.to_host(res.expected)[0])
    np.testing.assert_array_equal(errs, res.errors[0])
    assert all(type(e) is np.float64 for e in errs)
    eng.close()


def test_zero_loops(emu_engines, capsys):
    t = synthetic.traps_target((64, 64))
    for fn in (algorithms.gerchberg_saxton, algorithms.weighted_gerchberg_saxton):
        with pytest.raises(UnboundLocalError, match="expected_outcome"):
            fn(t, ns(max_loops=0, print_info=True))
        assert capsys.readouterr().out == "\n"
    # gradient descent draws its initial guess first: the module-level generator is left where the reference's
    # per-pixel loop leaves it, and "computing hologram" is printed, before the loop count is refused
    random.seed(0)
    with pytest.raises(UnboundLocalError, match="output"):
        algorithms.gradient_descent(t, ns(max_loops=0, print_info=True))
    after = random.random()
    assert capsys.readouterr().out == "computing hologram\n\n"
    random.seed(42)
    for _ in range(t.size):
        random.random()
    assert after == random.random()


def test_print_info(emu_engines, capsys):
    t = synthetic.traps_target((64, 64))
    for fn, head in ((algorithms.gerchberg_saxton, ""), (algorithms.weighted_gerchberg_saxton, ""),
                     (algorithms.gradient_descent, "computing hologram\n")):
        _, _, errs = fn(t, ns(max_loops=4, print_info=True))
        assert capsys.readouterr().out == f"{head}\rloop 4/4\n\nerror: {errs[-1]}\nnumber of loops: 4\n"
        fn(t, ns(max_loops=3))
        assert capsys.readouterr().out == "\rloop 3/3\n"
