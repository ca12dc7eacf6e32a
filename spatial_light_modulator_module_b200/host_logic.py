"""Host-side logic of the drop-in shims: everything the reference decides with Python / numpy
*scalars and dtypes* before or after the heavy array work (which runs on the device).

Nothing here touches a device, so it is covered by the CPU test-suite.
"""
from __future__ import annotations

import random as _pyrandom
from typing import List, Tuple

import numpy as np

TWO_PI = 2 * np.pi


# --------------------------------------------------------------------------------------------
# targets
# --------------------------------------------------------------------------------------------
def amplitude_lut() -> np.ndarray:
    """|sqrt(T)| for every 8-bit grey level, evaluated by numpy itself so the float16 rounding of
    ``np.sqrt(uint8)`` (algorithms.py:21, SURVEY A.1) is reproduced exactly."""
    return np.abs(np.sqrt(np.arange(256, dtype=np.uint8))).astype(np.float64)


def gd_mask_lut(white_attention) -> np.ndarray:
    """``1 + white_attention * T / 255`` (algorithms.py:80) per grey level.  Computed with the
    caller's own ``white_attention`` object so numpy's promotion applies (a Python int keeps the
    product in uint8 and wraps, SURVEY A.2)."""
    grey = np.arange(256, dtype=np.uint8)
    return np.asarray(1 + white_attention * grey / 255, dtype=np.float64)


def classify_target(target: np.ndarray):
    """How a target plane is handed to the engine.

    Returns ``("u8", None, None, setup_c64)`` for uint8 targets (amplitude / mask come from
    256-entry tables) or ``("real", T_float64, amp_float64, setup_c64)`` otherwise, where ``amp``
    is ``np.abs(np.sqrt(target))`` in the dtype numpy picks and ``setup_c64`` says whether scipy's
    first ``ifft2`` of that amplitude runs in complex64 (float16/float32 data) or complex128.
    """
    target = np.asarray(target)
    if target.dtype == np.uint8:
        return "u8", None, None, True
    amp = np.sqrt(target)
    setup_c64 = amp.dtype in (np.dtype(np.float16), np.dtype(np.float32))
    return "real", target.astype(np.float64), np.abs(amp).astype(np.float64), setup_c64


def plane_norms(targets: np.ndarray) -> np.ndarray:
    """np.amax(demanded_output) per plane (algorithms.py:23,74) as float64."""
    t = np.asarray(targets)
    return t.reshape(t.shape[0], -1).max(axis=1).astype(np.float64)


# --------------------------------------------------------------------------------------------
# gradient descent bookkeeping
# --------------------------------------------------------------------------------------------
def learning_rate_schedule(learning_rate, unsettle, max_loops) -> Tuple[np.ndarray, List[float]]:
    """Learning rate in force during iteration k, and ``args.learning_rate`` as it stands after k
    completed iterations (index k), following algorithms.py:102-104 literally (Python's banker's
    ``round``; ZeroDivisionError when the period rounds to 0)."""
    lr = learning_rate
    during = np.empty(max_loops, dtype=np.float64)
    after = [lr]
    for i in range(1, max_loops + 1):
        during[i - 1] = lr
        if unsettle and i % int(round(max_loops / (unsettle + 1))) == 0:
            lr *= 2
        after.append(lr)
    return during, after


def snapshot_chunks(max_loops: int, gif_skip: int) -> List[int]:
    """Iteration counts of consecutive runs that end exactly at the iterations i with i % gif_skip == 0
    (where algorithms.py:40,94 dump a GIF frame), plus the remainder."""
    if gif_skip < 1:
        raise ZeroDivisionError("integer modulo by zero")          # i % 0 in the reference
    ends = [i for i in range(max_loops) if i % gif_skip == 0]       # snapshot after iteration i (0-based)
    chunks, done = [], 0
    for e in ends:
        chunks.append(e + 1 - done)
        done = e + 1
    if done < max_loops:
        chunks.append(max_loops - done)
    return chunks


def python_random_stream(seed, count: int) -> np.ndarray:
    """``count`` successive ``random.random()`` values after ``random.seed(seed)``.

    CPython's MT19937 state is transplanted into numpy's RandomState, which draws the same
    53-bit doubles in bulk (SURVEY A.4).  The module-level ``random`` state is left exactly where
    the reference's per-pixel loop would leave it (algorithms.py:117-150)."""
    _pyrandom.seed(seed)
    state = _pyrandom.getstate()
    rs = np.random.RandomState()
    rs.set_state(("MT19937", np.array(state[1][:-1], dtype=np.uint32), state[1][-1]))
    out = rs.random_sample(count)
    key, pos = rs.get_state()[1:3]
    _pyrandom.setstate((state[0], tuple(int(k) for k in key) + (int(pos),), state[2]))
    return out


def uniform_stream_guess(kind: str, shape, seed):
    """For the families that are exp(1j*2*pi*u)[/100] ("random", "zeros"): the uniform plane u and
    the divisor, so the exponential can be evaluated on the device.  None for other kinds."""
    h, w = shape
    if kind == "random":
        return python_random_stream(seed, h * w).reshape(h, w), 1.0
    if kind == "zeros":
        return python_random_stream(seed, h * w).reshape(h, w), 100.0
    return None


def host_initial_guess(kind: str, shape, seed):
    """The random families of make_initial_guess (algorithms.py:115-153) as complex128 planes.
    Returns None for "fourier" (computed on the device) and raises ValueError for unknown kinds."""
    h, w = shape
    if kind == "random":
        u = python_random_stream(seed, h * w).reshape(h, w)
        return np.exp(1j * 2 * np.pi * u)
    if kind == "old":
        u = python_random_stream(seed, 2 * h * w).reshape(h, w, 2)
        return np.sqrt(u[..., 0]) + 1j * np.sqrt(u[..., 1])
    if kind == "unnormed":
        u = python_random_stream(seed, 2 * h * w).reshape(h, w, 2)
        return ((u[..., 0] + 1j * u[..., 1]) - 0.5) * 2
    if kind == "zeros":
        u = python_random_stream(seed, h * w).reshape(h, w)
        return np.exp(1j * 2 * np.pi * u) / 100
    if kind == "ones":
        _pyrandom.seed(seed)
        return np.ones(shape) + 1j * np.zeros(shape)
    if kind == "fourier":
        _pyrandom.seed(seed)
        return None
    _pyrandom.seed(seed)
    raise ValueError("unknown type of initial guess")


# --------------------------------------------------------------------------------------------
# analytic hologram scalars (evaluated exactly as the reference's Python expressions)
# --------------------------------------------------------------------------------------------
def deflect_scalars(angle, px_distance, wavelength, unit_angle):
    """wavefront_correction.py:440-447: (const, sin(y*u), sin(x*u))."""
    x_angle, y_angle = angle
    const = 2 * np.pi * px_distance / wavelength
    return float(const), float(np.sin(y_angle * unit_angle)), float(np.sin(x_angle * unit_angle))


def lens_scalars(focal_length, wavelength):
    """generate_hologram.py:196-201: (2*pi*f/lambda, f**2)."""
    return float(2 * np.pi * focal_length / wavelength), float(focal_length ** 2)


def defocus_coefficient(focal_length, px_distance, wavelength) -> float:
    """Multi-plane GS: alpha = -pi px^2 / (lambda f) [rad / pixel^2], the paraxial form of the reference's ``lens(f)``
    (generate_hologram.py:189-203, phase k (1 - sqrt(1 + r^2/f^2)) ~ -pi r^2 / (lambda f)): the target plane that
    ``add_lens(hologram, f)`` brings into focus.  f = None or infinite: 0, the Fourier plane."""
    if focal_length is None or np.isinf(focal_length):
        return 0.0
    return float(-np.pi * px_distance ** 2 / (wavelength * focal_length))


def check_defocus(alphas, shape, px_distance, wavelength) -> None:
    """Multi-plane GS: refuse a defocus that aliases.  The phase alpha rho^2 steps by |alpha| max(H, W) per pixel at the
    plane's edge; above pi the sampled lens is a different lens.  The message names the plane and the shortest focal
    length allowed at ``px_distance`` and ``wavelength``."""
    n = max(shape)
    for k, a in enumerate(alphas):
        if not np.isfinite(a):
            raise ValueError(f"defocus of plane {k} is not finite: {a!r}")
        if abs(a) * n > np.pi:
            f_min = px_distance ** 2 * n / wavelength
            raise ValueError(f"the defocus of plane {k} aliases: its phase steps by |alpha| * max(H, W) = {abs(a) * n:.4g} rad "
                             f"per pixel at the edge of a {shape[0]}x{shape[1]} plane (at most pi); the shortest focal length "
                             f"allowed is |f| >= {f_min:.3g} m (pixel pitch {px_distance:g} m, wavelength {wavelength:g} m)")


# --------------------------------------------------------------------------------------------
# frame sharding (generate_hologram_sequence over ranks)
# --------------------------------------------------------------------------------------------
def shard_range(n_items: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous block [lo, hi) of ``n_items`` owned by ``rank`` (sizes differ by at most one)."""
    base, rem = divmod(n_items, world)
    lo = rank * base + min(rank, rem)
    return lo, lo + base + (1 if rank < rem else 0)
