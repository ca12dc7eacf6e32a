"""Slab-decomposed transform of one large plane (BASELINE config 5) on CPU: the row-slab kernels run in
the host emulation, the all-to-all transposes and the 4-scalar all-reduce over gloo with 2 ranks."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

from tests.conftest import free_port
import torch.multiprocessing as mp
from scipy.fft import fft, ifft

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _slab_factory(n, world, rank, precision, *a):
    from tests.emu.emu_engine import EmuSlabEngine
    return EmuSlabEngine(n, world, rank, precision)


@pytest.mark.parametrize("n,precision", [(8192, "fp32"), (16384, "fp32"), (8192, "fp64"), (1024, "fp32")])
def test_long_line_transforms(n, precision):
    """Lines of 8192 / 16384 points (32 points per thread, fft_tile.cuh) against scipy, both directions,
    plain and exchange-layout addressing."""
    from tests.emu.emu_engine import EmuSlabEngine
    rows = 32
    eng = EmuSlabEngine(n, n // rows, 0, precision)
    rng = np.random.default_rng(2)
    x = (rng.standard_normal((rows, n)) + 1j * rng.standard_normal((rows, n))).astype(eng.complex_dtype)
    tol = 3e-6 if precision == "fp32" else 5e-14
    xd, out = eng._mem_upload(x), eng._mem_empty((rows, n), eng.complex_dtype)
    for inverse in (False, True):
        eng._rows_fft(xd, out, inverse)
        ref = (ifft(x.astype(np.complex128), axis=1) * n) if inverse else fft(x.astype(np.complex128), axis=1)
        assert np.abs(eng.to_host(out) - ref).max() / np.abs(ref).max() < tol
    # exchange layout in and out: block q holds [rows][rows] = elements q*rows .. of every line
    xb = np.ascontiguousarray(x.reshape(rows, n // rows, rows).transpose(1, 0, 2))
    ob = eng._mem_empty(xb.shape, eng.complex_dtype)
    eng._rows_fft(eng._mem_upload(xb), ob, False, block_in=rows, block_out=rows)
    got = eng.to_host(ob).transpose(1, 0, 2).reshape(rows, n)
    ref = fft(x.astype(np.complex128), axis=1)
    assert np.abs(got - ref).max() / np.abs(ref).max() < tol
    eng.close()


def test_transpose_blocks_roundtrip():
    from tests.emu.emu_engine import EmuSlabEngine
    n, world = 256, 4
    eng = EmuSlabEngine(n, world, 0, "fp32")
    h = n // world
    for dtype, eb in ((np.complex64, 8), (np.uint8, 1), (np.complex128, 16)):
        a = (np.arange(h * n) % 251).reshape(h, n).astype(dtype)
        send, back = eng._mem_empty((world, h, h), dtype), eng._mem_empty((h, n), dtype)
        eng._transpose(eng._mem_upload(a), send, eb, False)
        s = eng.to_host(send)
        for q in range(world):
            np.testing.assert_array_equal(s[q], a[:, q * h:(q + 1) * h].T)
        eng._transpose(send, back, eb, True)
        np.testing.assert_array_equal(eng.to_host(back), a)
    eng.close()


@pytest.mark.parametrize("precision", ["fp32", "fp64"])
def test_slab_gs_single_rank_equals_plane_engine(precision):
    """world = 1: the slab path is the same arithmetic as the ordinary engine, bit for bit."""
    from spatial_light_modulator_module_b200 import synthetic
    from tests.emu.emu_engine import EmuEngine, EmuSlabEngine
    n = 256
    t = synthetic.shapes_target((n, n))
    ref = EmuEngine((n, n), precision, 1)
    r = ref.gs(t, 4)
    eng = EmuSlabEngine(n, 1, 0, precision)
    h, e, errs = eng.gs(t, 4)
    np.testing.assert_array_equal(h, ref.to_host(r.hologram)[0])
    np.testing.assert_array_equal(e, ref.to_host(r.expected)[0])
    assert np.max(np.abs(np.array(errs) - r.errors[0]) / r.errors[0]) < 1e-12
    # a tolerance between two errors of the curve ends the loop where the ordinary engine ends it (algorithms.py:29)
    stop_at = float(0.5 * (errs[0] + errs[1]))
    r2 = ref.gs(t, 4, tolerance=stop_at)
    h2, _, errs2 = eng.gs(t, 4, tolerance=stop_at)
    assert len(errs2) == len(r2.errors[0]) == 2
    assert np.max(np.abs(np.array(errs2) - r2.errors[0]) / r2.errors[0]) < 1e-12
    np.testing.assert_array_equal(h2, ref.to_host(r2.hologram)[0])
    eng.close(); ref.close()


@pytest.mark.parametrize("precision", ["fp32", "fp64"])
def test_slab_gs_exact_zero_error(precision):
    """One bright pixel at the origin is a fixed point of GS: the first error is exactly 0, so the default tolerance 0
    ends the loop there.  The slab path, which runs every iteration and cuts the curve, gives the ordinary engine's
    hologram, expected outcome and curve."""
    from tests.emu.emu_engine import EmuEngine, EmuSlabEngine
    n = 256
    t = np.zeros((n, n), np.uint8)
    t[0, 0] = 255
    ref = EmuEngine((n, n), precision, 1)
    r = ref.gs(t, 2)
    eng = EmuSlabEngine(n, 1, 0, precision)
    h, e, errs = eng.gs(t, 2)
    assert errs == [0.0] and list(r.errors[0]) == [0.0]
    np.testing.assert_array_equal(h, ref.to_host(r.hologram)[0])
    np.testing.assert_array_equal(e, ref.to_host(r.expected)[0])
    eng.close(); ref.close()


def _worker(rank, world, port, n, loops, out_dir):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    from spatial_light_modulator_module_b200 import slab, synthetic
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    try:
        t = synthetic.noise_target((n, n), seed=6)
        h, e, errs = slab.gerchberg_saxton_slab(t, loops, precision="fp32", engine_factory=_slab_factory)
        np.savez(os.path.join(out_dir, f"r{rank}.npz"), h=h, e=e, errs=np.array(errs))
    finally:
        dist.destroy_process_group()


def test_two_rank_slab_gs_matches_single_rank(tmp_path):
    from spatial_light_modulator_module_b200 import synthetic
    from tests.emu.emu_engine import EmuSlabEngine
    n, loops = 256, 4
    mp.spawn(_worker, args=(2, free_port(), n, loops, str(tmp_path)), nprocs=2, join=True)
    t = synthetic.noise_target((n, n), seed=6)
    eng = EmuSlabEngine(n, 1, 0, "fp32")
    h, e, errs = eng.gs(t, loops)
    r0, r1 = np.load(tmp_path / "r0.npz"), np.load(tmp_path / "r1.npz")
    np.testing.assert_array_equal(np.concatenate([r0["h"], r1["h"]]), h)      # fields are bit-identical
    np.testing.assert_allclose(np.concatenate([r0["e"], r1["e"]]), e, rtol=1e-12)
    np.testing.assert_array_equal(r0["errs"], r1["errs"])                     # every rank closes the loop identically
    assert np.max(np.abs(r0["errs"] - np.array(errs)) / np.array(errs)) < 1e-12
    eng.close()


# ---- gradient descent on the distributed plane -------------------------------------------------------------------
@pytest.mark.parametrize("precision", ["fp32", "fp64"])
def test_slab_gd_single_rank_equals_plane_engine_and_oracle(precision):
    """world = 1: GD on the slab path (two Fourier-plane passes per iteration, loop state on the device) against the
    ordinary engine -- the same arithmetic per element, the error sums in another order -- and against the oracle."""
    from oracle import numpy_port as P
    from spatial_light_modulator_module_b200 import host_logic as hl, synthetic
    from tests.emu.emu_engine import EmuEngine, EmuSlabEngine
    n, loops = 256, 5
    t = synthetic.noise_target((n, n), seed=8)
    x0 = hl.host_initial_guess("random", (n, n), 42)
    during, _ = hl.learning_rate_schedule(0.01, 1, loops)             # (with one doubling of the learning rate on the way)
    ref = EmuEngine((n, n), precision, 1)
    r, _ = ref.gd(t, x0.copy(), during, loops)
    eng = EmuSlabEngine(n, 1, 0, precision)
    h, e, errs = eng.gd(t, x0, during, loops)
    np.testing.assert_array_equal(h, ref.to_host(r.hologram)[0])
    np.testing.assert_allclose(e, ref.to_host(r.expected)[0], rtol=1e-12)
    assert np.max(np.abs(np.array(errs) - r.errors[0]) / r.errors[0]) < (1e-6 if precision == "fp32" else 1e-12)
    ref_h, ref_e, ref_errs, _ = P.gd_run(t, loops, learning_rate=0.01, unsettle=1)
    tol = 1e-9 if precision == "fp64" else 1e-4
    assert np.max(np.abs(np.array(errs) - np.array(ref_errs)) / np.array(ref_errs)) < tol
    # a tolerance ends the loop where the reference does (algorithms.py:83)
    stop_at = float(0.5 * (errs[1] + errs[2]))
    h2, _, errs2 = eng.gd(t, x0, during, loops, tolerance=stop_at)
    assert len(errs2) == 3 and errs2 == errs[:3]
    r2, _ = ref.gd(t, x0.copy(), during[:3], 3)
    np.testing.assert_array_equal(h2, ref.to_host(r2.hologram)[0])
    # device-resident target and guess (what bench.py hands over): the same result, the guess left as it was
    xd = eng._mem_upload(x0.astype(eng.complex_dtype))
    h3, _, errs3 = eng.gd(eng._mem_upload(t), xd, during, loops, want_expected=False)
    np.testing.assert_array_equal(h3, h)
    assert errs3 == errs
    np.testing.assert_array_equal(eng.to_host(xd), x0.astype(eng.complex_dtype))
    eng.close(); ref.close()


def test_slab_gs_after_gd_on_the_same_engine():
    """A GD run that ends on its tolerance leaves the context's loop-ended flags set; the next GS run on the same engine
    starts from a reset context and gives the bits of a fresh engine."""
    from spatial_light_modulator_module_b200 import host_logic as hl, synthetic
    from tests.emu.emu_engine import EmuSlabEngine
    n, loops = 256, 4
    t = synthetic.shapes_target((n, n))
    fresh = EmuSlabEngine(n, 1, 0, "fp32")
    h, e, errs = fresh.gs(t, loops)
    fresh.close()
    eng = EmuSlabEngine(n, 1, 0, "fp32")
    during, _ = hl.learning_rate_schedule(0.005, 0, loops)
    _, _, gd_errs = eng.gd(t, hl.host_initial_guess("random", (n, n), 42), during, loops, tolerance=1e9)
    assert len(gd_errs) == 1                                           # (stopped on the tolerance)
    h2, e2, errs2 = eng.gs(t, loops)
    np.testing.assert_array_equal(h2, h)
    np.testing.assert_array_equal(e2, e)
    assert errs2 == errs
    eng.close()


def _gd_worker(rank, world, port, n, loops, out_dir):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    from spatial_light_modulator_module_b200 import host_logic as hl, synthetic
    dist.init_process_group("gloo", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world)
    try:
        t = synthetic.shapes_target((n, n))
        x0 = hl.host_initial_guess("random", (n, n), 7)
        during, _ = hl.learning_rate_schedule(0.005, 0, loops)
        lo, hi = rank * (n // world), (rank + 1) * (n // world)
        eng = _slab_factory(n, world, rank, "fp64")
        h, e, errs = eng.gd(t[lo:hi], x0[lo:hi], during, loops, white_attention=2.5)
        np.savez(os.path.join(out_dir, f"gd{rank}.npz"), h=h, e=e, errs=np.array(errs))
        eng.close()
    finally:
        dist.destroy_process_group()


def test_two_rank_slab_gd_matches_single_rank(tmp_path):
    from spatial_light_modulator_module_b200 import host_logic as hl, synthetic
    from tests.emu.emu_engine import EmuSlabEngine
    n, loops = 256, 4
    mp.spawn(_gd_worker, args=(2, free_port(), n, loops, str(tmp_path)), nprocs=2, join=True)
    t = synthetic.shapes_target((n, n))
    x0 = hl.host_initial_guess("random", (n, n), 7)
    during, _ = hl.learning_rate_schedule(0.005, 0, loops)
    eng = EmuSlabEngine(n, 1, 0, "fp64")
    h, e, errs = eng.gd(t, x0, during, loops, white_attention=2.5)
    r0, r1 = np.load(tmp_path / "gd0.npz"), np.load(tmp_path / "gd1.npz")
    np.testing.assert_array_equal(np.concatenate([r0["h"], r1["h"]]), h)
    np.testing.assert_allclose(np.concatenate([r0["e"], r1["e"]]), e, rtol=1e-12)
    np.testing.assert_array_equal(r0["errs"], r1["errs"])
    assert np.max(np.abs(r0["errs"] - np.array(errs)) / np.array(errs)) < 1e-12
    eng.close()


def test_gradient_descent_slab_entry_point():
    """The reference-style entry (learning rate, unsettle, initial guess by name) against the oracle's GD."""
    from oracle import numpy_port as P
    from spatial_light_modulator_module_b200 import slab, synthetic
    n, loops = 256, 6
    t = synthetic.noise_target((n, n), seed=3)
    h, e, errs, lr_after = slab.gradient_descent_slab(t, loops, learning_rate=0.01, unsettle=2, precision="fp64",
                                                      engine_factory=_slab_factory)
    ref_h, ref_e, ref_errs, ref_lr = P.gd_run(t, loops, learning_rate=0.01, unsettle=2)
    assert np.max(np.abs(np.array(errs) - np.array(ref_errs)) / np.array(ref_errs)) < 1e-9
    assert lr_after == ref_lr
    d = np.abs(np.angle(np.exp(1j * (h - ref_h))))
    assert d.max() < 1e-6
    np.testing.assert_allclose(e, ref_e, rtol=1e-7, atol=1e-9)
    with pytest.raises(ValueError):
        slab.gradient_descent_slab(t, loops, initial_guess="fourier", engine_factory=_slab_factory)


@pytest.mark.parametrize("dtype", [np.complex64, np.complex128, np.uint8])
def test_peer_store_kernel_is_the_all_to_all(dtype):
    """slm_transpose_blocks_peer with every "peer" a buffer of this process: the stores of all ranks together are the
    all-to-all of the transposed blocks, on the way out and on the way back."""
    from tests.emu.emu_engine import EmuSlabEngine
    n, world = 256, 4
    h = n // world
    rng = np.random.default_rng(4)
    eb = np.dtype(dtype).itemsize
    if dtype == np.uint8:
        slabs = [rng.integers(0, 256, (h, n)).astype(np.uint8) for _ in range(world)]
    else:
        slabs = [(rng.standard_normal((h, n)) + 1j * rng.standard_normal((h, n))).astype(dtype) for _ in range(world)]
    engs = [EmuSlabEngine(n, world, r, "fp32") for r in range(world)]
    recv = [engs[r]._mem_upload(np.zeros((world, h, h), dtype)) for r in range(world)]
    table = (C.c_void_p * world)(*[b.ctypes.data for b in recv])
    for r, eng in enumerate(engs):
        src = eng._mem_upload(slabs[r])
        eng._check(eng._lib.slm_transpose_blocks_peer(eng._ctx, eng._mem_ptr(src), table, world, r, h, n, eb, 0))
    for q in range(world):
        for p in range(world):                                    # rank q's block p = rank p's columns q*h.., transposed
            np.testing.assert_array_equal(np.asarray(recv[q])[p], slabs[p][:, q * h:(q + 1) * h].T)
    # way back: lines into the peers' row slabs
    back = [engs[r]._mem_upload(np.zeros((h, n), dtype)) for r in range(world)]
    table = (C.c_void_p * world)(*[b.ctypes.data for b in back])
    lines = [np.ascontiguousarray(np.stack([slabs[p][:, q * h:(q + 1) * h].T for p in range(world)])) for q in range(world)]
    for q, eng in enumerate(engs):
        src = eng._mem_upload(lines[q])
        eng._check(eng._lib.slm_transpose_blocks_peer(eng._ctx, eng._mem_ptr(src), table, world, q, h, n, eb, 1))
    for p in range(world):
        got = np.asarray(back[p])
        for q in range(world):
            np.testing.assert_array_equal(got[:, q * h:(q + 1) * h], slabs[p][:, q * h:(q + 1) * h])
    for eng in engs:
        eng.close()


def test_slab_gs_with_illumination_plane():
    """A non-uniform illumination amplitude (algorithms.py:14-19,30) on the slab path: the ordinary engine's bits."""
    from spatial_light_modulator_module_b200 import synthetic
    from tests.emu.emu_engine import EmuEngine, EmuSlabEngine
    n = 256
    t = synthetic.shapes_target((n, n))
    yy, xx = np.mgrid[0:n, 0:n]
    inc = np.exp(-((yy - n / 2) ** 2 + (xx - n / 2) ** 2) / (2 * (n / 3) ** 2))
    ref = EmuEngine((n, n), "fp64", 1)
    r = ref.gs(t, 4, inc_amp=inc)
    eng = EmuSlabEngine(n, 1, 0, "fp64")
    h, e, errs = eng.gs(t, 4, inc_amp_slab=inc)
    np.testing.assert_array_equal(h, ref.to_host(r.hologram)[0])
    np.testing.assert_array_equal(e, ref.to_host(r.expected)[0])
    assert np.max(np.abs(np.array(errs) - r.errors[0]) / r.errors[0]) < 1e-12
    h0, _, errs0 = eng.gs(t, 4)
    assert not np.array_equal(h0, h)                                   # (the plane does change the result)
    eng.close(); ref.close()
