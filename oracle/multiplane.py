"""Multi-plane Gerchberg-Saxton as this project defines it: the checker of ``Engine.gs_multiplane`` /
``slm_gs_multiplane_run``.

TEST INFRASTRUCTURE ONLY -- never imported by the shipped package.

The reference has no multi-plane GS; this module is the definition (after Haist et al., Opt. Commun. 140, 299 (1997),
and Whyte & Courtial, New J. Phys. 7, 117 (2005)).  K target planes T_k share one hologram.  Plane k lies where a lens
of phase alpha_k * rho^2 brings the Fourier plane, with rho^2 = (i - H/2)^2 + (j - W/2)^2 in pixels^2 (the centre of
the reference's ``lens``) and L_k = exp(1j * alpha_k * rho^2):

    setup      A_k = ifft2(amp_k) as GS computes it (numpy_port.gs_setup: complex64 for 8-bit targets)
               A   = sum_k A_k conj(L_k)
    iteration  B   = inc * exp(1j*angle(A))
               per plane: C_k = fft2(B L_k),  D_k = |amp_k| exp(1j*angle(C_k)),
                          expected_k = |C_k|^2 norm_k / max |C_k|^2,  err_k = error_f(expected_k, T_k, HW)
               A   = sum_k ifft2(D_k) conj(L_k)
    hologram   angle(A) after the last iteration; the loop runs while ANY plane's error > tolerance

Sums start from their first term, and a plane with alpha_k = 0 is not multiplied by L_k, so K = 1 with alpha = 0 is
numpy_port's GS operation for operation.  Like numpy_port's GS it is a setup / step state machine: a state made by
:func:`mp_start` from a given B is the state the engine starts a one-iteration run from.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import List, Optional

import numpy as np
from scipy.fft import fft2, ifft2

from . import numpy_port as P


def defocus_coefficient(focal_length, px_distance=P.PX_DISTANCE, wavelength=P.WAVELENGTH):
    """alpha = -pi px^2 / (lambda f) [rad / pixel^2]: the paraxial form of the reference's ``lens(f)``, whose phase
    k (1 - sqrt(1 + r^2/f^2)) is -pi r^2 / (lambda f) to first order.  f = None or inf: 0 (the Fourier plane)."""
    if focal_length is None or np.isinf(focal_length):
        return 0.0
    return float(-np.pi * px_distance ** 2 / (wavelength * focal_length))


def lens_field(shape, alpha):
    """L = exp(1j * alpha * rho^2) over a plane of ``shape``."""
    h, w = shape
    i = np.arange(h, dtype=np.float64)[:, None] - h / 2
    j = np.arange(w, dtype=np.float64)[None, :] - w / 2
    return np.exp(1j * (alpha * (i * i + j * j)))


@dataclass
class MPState:
    planes: List[P.GSState]       # per plane: GS's target, amplitude, norm, space norm; .A is unused
    alphas: List[float]
    lenses: List[Optional[np.ndarray]]   # L_k, None where alpha_k == 0
    inc_amp: np.ndarray
    B: Optional[np.ndarray] = None       # SLM-plane field of the next iteration (set by a start from B)
    A: Optional[np.ndarray] = None       # field summed over the planes
    expected: Optional[List[np.ndarray]] = None
    errors: List[List[float]] = field(default_factory=list)


def _sum(terms):
    total = None
    for t in terms:
        total = t if total is None else total + t
    return total


def _state(targets, alphas, incomming_intensity) -> MPState:
    targets = [np.asarray(t) for t in targets]
    if len(targets) != len(alphas):
        raise ValueError("one defocus coefficient per target plane")
    planes = [P.gs_setup(t, incomming_intensity) for t in targets]
    lenses = [None if a == 0 else lens_field(targets[0].shape, a) for a in alphas]
    return MPState(planes, [float(a) for a in alphas], lenses, planes[0].inc_amp, errors=[[] for _ in targets])


def mp_setup(targets, alphas, incomming_intensity="uniform") -> MPState:
    """A = sum_k A_k conj(L_k) from GS's setup of every plane."""
    st = _state(targets, alphas, incomming_intensity)
    st.A = _sum(p.A if L is None else p.A * np.conj(L) for p, L in zip(st.planes, st.lenses))
    return st


def mp_first_phasor(st: MPState) -> np.ndarray:
    """B of iteration 0 (carries the complex64 quirk when the sum is one unmultiplied 8-bit plane, as GS's does)."""
    return st.inc_amp * P.unit_phasor(st.A)


def mp_start(targets, alphas, B, incomming_intensity="uniform") -> MPState:
    """State entering an iteration from SLM-plane field ``B``."""
    st = _state(targets, alphas, incomming_intensity)
    st.B = np.asarray(B)
    return st


def mp_step(st: MPState):
    """One iteration.  Returns (C_k list, expected_k list, error_k list) and advances A (and B)."""
    B = st.inc_amp * P.unit_phasor(st.A) if st.B is None else st.B
    st.B = None
    Cs, exps, errs, terms = [], [], [], []
    for k, (p, L) in enumerate(zip(st.planes, st.lenses)):
        C = fft2(B if L is None else B * L)
        D = np.abs(p.target_amp) * P.unit_phasor(C)
        a = ifft2(D)
        terms.append(a if L is None else a * np.conj(L))
        expected = np.abs(C) ** 2
        expected *= p.norm / expected.max()
        err = P.mean_square_error(expected, p.target, p.space_norm)
        st.errors[k].append(err)
        Cs.append(C), exps.append(expected), errs.append(err)
    st.A = _sum(terms)
    st.expected = exps
    return Cs, exps, errs


def mp_loop(st: MPState, max_loops, tolerance=0):
    """The GS loop condition over all planes: run while any plane's error > tolerance (NaN: not above)."""
    errs = [tolerance + 1]
    i = 0
    while any(e > tolerance for e in errs) and i < max_loops:
        _, _, errs = mp_step(st)
        i += 1
    if st.expected is None:
        raise UnboundLocalError("expected_outcome")
    return np.angle(st.A), st.expected, st.errors


def mp_run(targets, alphas, max_loops, tolerance=0, incomming_intensity="uniform"):
    """Returns (hologram, [expected_k], [errors_k])."""
    return mp_loop(mp_setup(targets, alphas, incomming_intensity), max_loops, tolerance)
