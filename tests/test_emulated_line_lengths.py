"""CPU checks of the 1152-, 1280- and 1920-point line transforms through the host emulation of the kernel sources
(tests/emu): 1280 = 16*5*16 (radix-5 middle stage), 1152 = 8*(2*3*3)*8 and 1920 = 8*(2*3*5)*8 (composite middles).
Each length runs as the rows and as the columns of a plane whose other side is 64, in both precisions.

The columns of these lengths run on the one-CTA-per-tile kernels (col_pass_kernel / col_plain_kernel) in both
precisions: the column-group kernel is built only for plans with a single own-code middle stage."""
import ctypes
import re

import numpy as np
import pytest

from tests import parity_checks as pc
from tests.emu.emu_engine import EmuEngine, emu_library

NEW_LENGTHS = [1152, 1280, 1920]
SHAPES = [s for L in NEW_LENGTHS for s in ((L, 64), (64, L))]
PRECISIONS = ["fp32", "fp64"]


def make_engine(shape, precision, max_batch):
    return EmuEngine(shape, precision, max_batch)


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("shape", SHAPES)
def test_fft2_matches_scipy(shape, precision):
    pc.check_fft2(make_engine, shape, precision)


@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("kind", ["noise", "shapes"])
@pytest.mark.parametrize("shape", SHAPES)
def test_gs_teacher_forced(shape, kind, precision):
    pc.check_gs_teacher_forced(make_engine, shape, precision, kind, steps=(0, 2))


@pytest.mark.parametrize("batch", [1, 2])
@pytest.mark.parametrize("precision", PRECISIONS)
@pytest.mark.parametrize("shape", SHAPES)
def test_gd_vs_oracle(shape, precision, batch):
    pc.check_gd_vs_oracle(make_engine, shape, precision, "noise", loops=3, batch=batch)


# one shape per new length and precision class as columns, and the new length as rows
@pytest.mark.parametrize("shape,precision", [((1152, 64), "fp32"), ((1280, 64), "fp32"), ((1920, 64), "fp64"),
                                             ((64, 1920), "fp32")])
def test_gs_tolerance_and_batch(shape, precision):
    pc.check_gs_tolerance_and_batch(make_engine, precision, shape=shape)


@pytest.mark.parametrize("shape,precision", [((1152, 64), "fp32"), ((1280, 64), "fp32"), ((1920, 64), "fp64"),
                                             ((64, 1920), "fp32")])
def test_gd_tolerance_and_batch(shape, precision):
    pc.check_gd_tolerance_and_batch(make_engine, precision, shape=shape, loops=6)


def test_supported_lengths_and_shape_error():
    lib = emu_library()
    buf = (ctypes.c_int * 64)()
    n = lib.slm_supported_lengths(buf, 64)
    lengths = list(buf[:n])
    assert set(NEW_LENGTHS) <= set(lengths)
    assert 1080 not in lengths
    with pytest.raises(ValueError) as ei:
        make_engine((1080, 1920), "fp32", 1)
    msg = str(ei.value)
    assert "1080x1920" in msg
    listed = re.search(r"\(([^()]*)\)\s*$", msg)
    assert listed, msg
    both, _, rows_only = listed.group(1).partition("; row length only: ")
    assert {int(x) for x in both.split(", ")} == {64, 128, 192, 256, 512, 768, 1024, 1152, 1280, 1920, 2048, 4096}
    assert {int(x) for x in rows_only.split(", ")} == {8192, 16384}
    assert set(lengths) == {64, 128, 192, 256, 512, 768, 1024, 1152, 1280, 1920, 2048, 4096, 8192, 16384}


@pytest.mark.parametrize("n", [1152, 1280, 1920])
def test_slab_path_rejects_lines_that_are_not_whole_warps(n):
    """The slab Fourier-plane kernel reduces a line's partial sums per warp; 144, 80 and 240 threads per line are
    neither within one warp nor whole warps, so the row-slab context refuses these lengths."""
    from tests.emu.emu_engine import EmuSlabEngine
    with pytest.raises(ValueError, match="slab path"):
        EmuSlabEngine(n, 1, 0, "fp32")


def test_new_lengths_in_a_full_panel_shape_context():
    """A 1152x1920 context is accepted and its transform round-trips (one plane, fp32)."""
    eng = make_engine((1152, 1920), "fp32", 1)
    rng = np.random.default_rng(1)
    x = (rng.standard_normal((1, 1152, 1920)) + 1j * rng.standard_normal((1, 1152, 1920))).astype(np.complex64)
    y = eng.to_host(eng.fft2(eng.fft2(x, False), True))
    assert np.abs(y - x).max() < 1e-5 * np.abs(x).max()
    eng.close()


def test_new_lengths_use_the_one_cta_per_tile_column_kernel():
    """The radix-5 and composite middle stages stay out of the column-group kernel (it spilled under its register cap):
    a context of each new column length runs its column passes without that kernel, and the 1024-point context still
    uses it."""
    class LineTable(ctypes.Structure):
        _fields_ = [("L", ctypes.c_int), ("prec", ctypes.c_int), ("rows_per_cta", ctypes.c_int), ("row_threads", ctypes.c_int),
                    ("row_smem", ctypes.c_size_t), ("cols_per_cta", ctypes.c_int), ("col_threads", ctypes.c_int),
                    ("col_smem", ctypes.c_size_t)] + [(f"fn{i}", ctypes.c_void_p) for i in range(5)] + \
                   [("group_ok", ctypes.c_int), ("group_row_bytes", ctypes.c_int), ("group_fused", ctypes.c_int)]
    lib = emu_library()

    def table(L, p):
        name = f"line_table_{L}_{p}"
        return LineTable.in_dll(lib, f"_ZN3slm{len(name)}{name}E")
    for L in NEW_LENGTHS:
        for p in (0, 1):
            t = table(L, p)
            assert t.L == L and t.prec == p and t.group_ok == 0 and t.group_fused == 0
            assert t.col_threads % 32 == 0 and t.col_threads == t.cols_per_cta * (L // (16 if L == 1280 else 8))
    assert table(1024, 0).group_ok == 1 and table(1024, 1).group_ok == 1
