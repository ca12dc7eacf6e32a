"""CPU checks of the CUDA kernel SOURCES through their host emulation (tests/emu): the same
.cu/.cuh files the product compiles with nvcc are compiled with g++ -DSLM_EMULATE and driven
through the C ABI by the package's Engine class, then compared with the oracle and the golden
fixtures.  This proves the kernels' logic (indexing, butterflies, fused pointwise steps,
reductions, loop control) without a GPU; the `-m gpu` suite repeats the same checks on the B200.
"""
import pytest

from tests import parity_checks as pc
from tests.emu.emu_engine import EmuEngine


def make_engine(shape, precision, max_batch):
    return EmuEngine(shape, precision, max_batch)


@pytest.mark.parametrize("precision", ["fp32", "fp64"])
@pytest.mark.parametrize("shape", [(64, 64), (128, 192), (192, 256), (256, 512), (64, 768), (768, 64), (1024, 64),
                                   (64, 2048), (64, 4096), (4096, 64)])
def test_fft2_matches_scipy(shape, precision):
    pc.check_fft2(make_engine, shape, precision)


@pytest.mark.parametrize("precision", ["fp32", "fp64"])
@pytest.mark.parametrize("kind", ["noise", "shapes"])
@pytest.mark.parametrize("shape", [(128, 128), (192, 256)])
def test_gs_teacher_forced(shape, kind, precision):
    pc.check_gs_teacher_forced(make_engine, shape, precision, kind)


@pytest.mark.parametrize("precision", ["fp32", "fp64"])
@pytest.mark.parametrize("kind", ["noise", "shapes", "traps"])
def test_gs_device_setup(kind, precision):
    pc.check_gs_device_setup(make_engine, (128, 128), precision, kind)


# fp32 columns of 1024 and 768 points run on the warp-per-column kernel (col_warp.cuh): every mode of it, several
# tiles per CTA (the emulated grid has 3 CTAs), both compute groups, a batch, the stop markers
@pytest.mark.parametrize("rows", [1024, 768])
@pytest.mark.parametrize("kind", ["noise", "shapes"])
def test_warp_column_kernel_gs(kind, rows):
    pc.check_gs_teacher_forced(make_engine, (rows, 64), "fp32", kind, steps=(0, 2))


@pytest.mark.parametrize("rows", [1024, 768])
def test_warp_column_kernel_gs_device_setup(rows):
    pc.check_gs_device_setup(make_engine, (rows, 64), "fp32", "noise", loops=3)


@pytest.mark.parametrize("rows,batch", [(1024, 1), (1024, 2), (768, 2)])
def test_warp_column_kernel_gd(rows, batch):
    pc.check_gd_vs_oracle(make_engine, (rows, 64), "fp32", "noise", loops=3, batch=batch)


@pytest.mark.parametrize("rows,batch", [(1024, 2), (768, 3), (1024, 5)])
def test_warp_column_kernel_gd_pipelined_one_pass_form(monkeypatch, rows, batch):
    """CGM_GD_PIPE: the CTA's two compute groups split each tile (forward transform + plane max | gradient step +
    inverse transform); tiles wait for the other tiles of their plane held by the other CTAs of a cooperative grid
    (the emulation co-schedules its 3 CTAs).  Against the oracle, and bit-identical to the two-pass form."""
    import numpy as np
    from spatial_light_modulator_module_b200 import host_logic as hl, synthetic
    monkeypatch.setenv("SLM_GD_FORM", "pipe")
    pc.check_gd_vs_oracle(make_engine, (rows, 64), "fp32", "noise", loops=3, batch=batch)
    shape, loops = (rows, 64), 4
    t = np.stack([synthetic.noise_target(shape, seed=i) for i in range(batch)])
    x0 = np.stack([hl.host_initial_guess("random", shape, 42 + i) for i in range(batch)])
    during, _ = hl.learning_rate_schedule(0.005, 0, loops)
    out = {}
    for form in ("pipe", "two_pass"):
        monkeypatch.setenv("SLM_GD_FORM", form)
        eng = make_engine(shape, "fp32", batch)
        n0 = eng.launch_count()
        r, _ = eng.gd(t, x0.copy(), during, loops)
        out[form] = (np.array(r.errors), eng.to_host(r.hologram), eng.to_host(r.expected), eng.launch_count() - n0)
        eng.close()
    assert out["pipe"][3] < out["two_pass"][3]                    # one Fourier-plane pass per iteration instead of two
    for i in range(3):
        np.testing.assert_array_equal(out["pipe"][i], out["two_pass"][i])


@pytest.mark.parametrize("shape,precision,gd_form", [((1024, 64), "fp32", "two_pass"), ((1024, 64), "fp32", "pipe"),
                                                     ((128, 128), "fp64", None)])
def test_deferred_and_in_kernel_closing_agree(monkeypatch, shape, precision, gd_form):
    """When a batch has more tiles than 4 per CTA, the planes are closed by a kernel behind the column pass;
    SLM_NO_DEFER_CLOSE=1 has the publisher warp of the pass close them.  Same bits for GS and GD from both persistent
    column kernels: the warp-per-column kernel (fp32 1024 rows; GD in two passes or pipelined) and the column-group
    kernel (fp64 128 rows)."""
    import numpy as np
    from spatial_light_modulator_module_b200 import host_logic as hl, synthetic
    if gd_form:
        monkeypatch.setenv("SLM_GD_FORM", gd_form)
    batch, loops = 2, 3
    t = np.stack([synthetic.noise_target(shape, seed=i) for i in range(batch)])
    x0 = np.stack([hl.host_initial_guess("random", shape, 42 + i) for i in range(batch)])
    during, _ = hl.learning_rate_schedule(0.005, 0, loops)
    out = {}
    for name in ("deferred", "in_kernel"):
        if name == "in_kernel":
            monkeypatch.setenv("SLM_NO_DEFER_CLOSE", "1")
        eng = make_engine(shape, precision, batch)
        n0 = eng.launch_count()
        g = eng.gs(t, loops)
        r, _ = eng.gd(t, x0.copy(), during, loops)
        out[name] = ([np.array(g.errors), eng.to_host(g.hologram), eng.to_host(g.expected),
                      np.array(r.errors), eng.to_host(r.hologram), eng.to_host(r.expected)], eng.launch_count() - n0)
        eng.close()
    assert out["deferred"][1] > out["in_kernel"][1]                # the closing kernels ran
    for a, b in zip(out["deferred"][0], out["in_kernel"][0]):
        np.testing.assert_array_equal(a, b)


def test_warp_column_kernel_gd_pipelined_tolerance(monkeypatch):
    monkeypatch.setenv("SLM_GD_FORM", "pipe")
    pc.check_gd_tolerance_and_batch(make_engine, "fp32", shape=(768, 64), loops=6)


def test_warp_column_kernel_tolerance_and_batch():
    pc.check_gs_tolerance_and_batch(make_engine, "fp32", shape=(1024, 64))
    pc.check_gd_tolerance_and_batch(make_engine, "fp32", shape=(768, 64), loops=6)


@pytest.mark.parametrize("precision", ["fp32", "fp64"])
def test_gd_tolerance_and_batch(precision):
    pc.check_gd_tolerance_and_batch(make_engine, precision)


GD_CASES = ["gd_noise_random_128x128", "gd_shapes_fourier_192x256", "gd_traps_unsettle_128x128",
            "gd_noise_wa2int_128x128", "gd_noise_wa05_128x128", "gd_shapes_old_128x128",
            "gd_shapes_unnormed_128x128", "gd_shapes_zeros_128x128", "gd_shapes_ones_128x128",
            "gd_traps_tol_128x128"]


@pytest.mark.parametrize("precision", ["fp32", "fp64"])
@pytest.mark.parametrize("name", GD_CASES)
def test_gd_matches_reference_golden(golden, name, precision):
    pc.check_gd_golden(make_engine, golden, name, precision)


@pytest.mark.parametrize("precision", ["fp32", "fp64"])
def test_gs_tolerance_and_batch(precision):
    pc.check_gs_tolerance_and_batch(make_engine, precision)


@pytest.mark.parametrize("precision", ["fp32", "fp64"])
def test_gs_real_valued_targets(golden, precision):
    pc.check_gs_real_targets(make_engine, golden, precision)


@pytest.mark.parametrize("precision", ["fp32", "fp64"])
def test_illumination(precision):
    pc.check_illumination(make_engine, precision)


def test_analytic_and_quantisers_bit_exact(golden):
    pc.check_analytic_and_quantisers(make_engine, golden)


@pytest.mark.parametrize("precision", ["fp32", "fp64"])
def test_expected_outcome(golden, precision):
    pc.check_expected_outcome(make_engine, golden, precision)


@pytest.mark.parametrize("precision", ["fp32", "fp64"])
def test_random_phasor_guess(golden, precision):
    pc.check_random_phasor_guess(make_engine, golden, precision)


def test_single_trap_and_device_frames(golden):
    pc.check_single_trap_and_frames(make_engine, golden)


def test_device_mt19937_stream():
    pc.check_device_mt19937(make_engine)


def test_sequence_driver_with_illumination_plane():
    """The movie driver hands a non-uniform illumination amplitude (algorithms.py:14-19) to every frame."""
    import numpy as np
    from spatial_light_modulator_module_b200 import generate_hologram_sequence as ghs, synthetic
    shape = (128, 128)
    frames = np.stack([synthetic.noise_target(shape, seed=s) for s in range(3)])
    yy, xx = np.mgrid[0:shape[0], 0:shape[1]]
    inc = np.sqrt(np.exp(-((yy - 64.0) ** 2 + (xx - 64.0) ** 2) / 3000.0) * 255).astype(np.float16).astype(np.float64)
    holos, exps, errors, _ = ghs.sequence_holograms(frames, 4, precision="fp64", batch=2, want_expected=True,
                                                    engine_factory=make_engine, inc_amp=inc)
    eng = make_engine(shape, "fp64", 1)
    for i in range(3):
        r = eng.gs(frames[i], 4, inc_amp=inc)
        np.testing.assert_array_equal(holos[i], eng.to_host(r.hologram)[0])
        np.testing.assert_array_equal(exps[i], eng.to_host(r.expected)[0])
        np.testing.assert_array_equal(errors[i], r.errors[0])
    eng.close()


def test_sequence_driver_warm_start():
    """Opt-in warm start: frame n starts from frame n-1's hologram; equals the hand-made chain, and on a slowly
    moving trap pattern the warm-started frames begin from a far smaller error than cold ones."""
    import numpy as np
    from spatial_light_modulator_module_b200 import generate_hologram_sequence as ghs, synthetic
    frames = synthetic.movie_frames(3, rescale_parameter=0.2)[:, :128, :128].copy()
    frames[:, 40, 50] = 255
    holos, _, errors, _ = ghs.sequence_holograms(frames, 5, precision="fp64", engine_factory=make_engine, warm_start=True)
    eng = make_engine(frames.shape[1:], "fp64", 1)
    phasor = None
    for i in range(3):
        r = eng.gs(frames[i], 5, phasor0=phasor)
        np.testing.assert_array_equal(holos[i], eng.to_host(r.hologram)[0])
        np.testing.assert_array_equal(errors[i], r.errors[0])
        phasor = eng.phase_phasor(r.hologram)
    cold, _, cold_errors, _ = ghs.sequence_holograms(frames, 5, precision="fp64", engine_factory=make_engine)
    assert errors[2][0] < cold_errors[2][0]
    eng.close()


def test_batched_algorithm_comparison_matches_single_runs():
    """compare_error_evolution_algorithms.error_evolution_curves (BASELINE config 4) at reduced size: chunks of two
    targets, a ragged last chunk -- the curves of the one-target-at-a-time runs."""
    import argparse
    import numpy as np
    from spatial_light_modulator_module_b200 import compare_error_evolution_algorithms as cmp, host_logic as hl, synthetic
    shape = (128, 128)
    targets = np.stack([synthetic.noise_target(shape, seed=1), synthetic.shapes_target(shape), synthetic.traps_target(shape)])
    a = argparse.Namespace(max_loops=5, precision="fp64", tolerance=0, learning_rate=0.005, unsettle=0, initial_guess="random",
                           random_seed=42, white_attention=1)
    cmp.fill_unnecessary_args(a)
    gd, gs = cmp.error_evolution_curves(targets, a, batch=2, engine_factory=make_engine)
    assert len(gd) == len(gs) == 3
    eng = make_engine(shape, "fp64", 1)
    during, _ = hl.learning_rate_schedule(0.005, 0, 5)
    for i, t in enumerate(targets):
        r, _ = eng.gd(t, hl.host_initial_guess("random", shape, 42), during, 5)
        np.testing.assert_allclose(gd[i], r.errors[0], rtol=1e-12)
        np.testing.assert_allclose(gs[i], eng.gs(t, 5).errors[0], rtol=1e-12)
    eng.close()
