"""Weighted Gerchberg-Saxton (GSW) as this project defines it: the checker of ``Engine.gsw`` / ``slm_gsw_run``.

TEST INFRASTRUCTURE ONLY -- never imported by the shipped package.

The reference has no GSW; this module is the definition (after Di Leonardo, Ianni & Ruocco, Opt. Express 15, 1913
(2007)).  It is GS as ``numpy_port`` restates it, with per-pixel weights w on the target amplitude.  Per plane:

    T      the target as GS reads it (grey levels or the real plane); amp = |sqrt(T)| as GS uses it
    Omega  {T > 0}, the signal set;  S_T = sum(T);  c = weight_limit >= 1
    iteration k:  C_k = fft2(B_k),  I_k = |C_k|^2,  P_k = sum over Omega of I_k
                  sigma_k = S_T / P_{k-1}  (sigma_0 = S_T / P_0: the first iteration of a run uses its own P)
                  w_k = clip(w_{k-1} * amp / sqrt(sigma_k * I_k), 1/c, c) on Omega where I_k > 0, else w_{k-1}
                  D_k = (amp * w_k) * exp(1j*angle(C_k)),   A = ifft2(D_k),   B_{k+1} = inc * exp(1j*angle(A))
    scale, expected outcome and error: GS's (numpy_port.gs_step).

Like numpy_port's GS it is a setup / step state machine, so tests can teacher-force single iterations: a state made
by :func:`gsw_start` from (B_k, w_{k-1}) is the state the engine starts a one-iteration run from.
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import List, Optional

import numpy as np
from scipy.fft import fft2, ifft2

from . import numpy_port as P


@dataclass
class GSWState:
    target: np.ndarray            # demanded_output as given
    inc_amp: np.ndarray           # incomming_amplitude
    amp: np.ndarray               # float64 |sqrt(T)| as GS uses it (float16-rounded for uint8 targets)
    signal: np.ndarray            # Omega = T > 0
    target_sum: float             # S_T
    space_norm: int
    norm: object                  # np.amax(target)
    weight_limit: float
    B: np.ndarray                 # SLM-plane field of the next iteration
    w: np.ndarray                 # weights w_{k-1}
    P_prev: Optional[float]       # P_{k-1}; None: the next iteration is the first of a run
    A: Optional[np.ndarray] = None
    expected: Optional[np.ndarray] = None
    errors: List[float] = field(default_factory=list)


def gsw_start(target, B, weights=None, weight_limit=10.0, incomming_intensity="uniform") -> GSWState:
    """State entering the first iteration of a run from SLM-plane field ``B`` and initial ``weights`` (None: ones)."""
    gs = P.gs_setup(target, incomming_intensity)
    t64 = np.asarray(target).astype(np.float64)
    w = np.ones(t64.shape) if weights is None else np.array(weights, dtype=np.float64)
    return GSWState(gs.target, gs.inc_amp, np.abs(gs.target_amp).astype(np.float64), t64 > 0, float(t64.sum()),
                    gs.space_norm, gs.norm, float(weight_limit), np.asarray(B), w, None)


def gsw_setup(target, weight_limit=10.0, incomming_intensity="uniform", weights=None) -> GSWState:
    """GS's setup (algorithms.py:14-30, including the complex64 first phasor) with weights w_{-1} (ones by default)."""
    gs = P.gs_setup(target, incomming_intensity)
    return gsw_start(target, P.gs_first_phasor(gs), weights, weight_limit, incomming_intensity)


def gsw_step(st: GSWState):
    """One iteration.  Returns (C, expected, error) and advances B, w and P_prev."""
    C = fft2(st.B)
    I = np.abs(C) ** 2
    p = float(I[st.signal].sum())
    sigma = st.target_sum / (p if st.P_prev is None else st.P_prev)
    m = st.signal & (I > 0)
    w = st.w.copy()
    c = st.weight_limit
    w[m] = np.clip(st.w[m] * st.amp[m] / np.sqrt(sigma * I[m]), 1 / c, c)
    D = (st.amp * w) * P.unit_phasor(C)
    st.A = ifft2(D)
    st.B = st.inc_amp * P.unit_phasor(st.A)
    expected = I * (st.norm / I.max())
    err = P.mean_square_error(expected, st.target, st.space_norm)
    st.w, st.P_prev, st.expected = w, p, expected
    st.errors.append(err)
    return C, expected, err


def gsw_run(target, max_loops, tolerance=0, weight_limit=10.0, incomming_intensity="uniform", weights=None):
    """The GS loop (algorithms.py:24-49) with GSW's iteration.  Returns (hologram, expected, errors, weights)."""
    st = gsw_setup(target, weight_limit, incomming_intensity, weights)
    error = tolerance + 1
    i = 0
    while error > tolerance and i < max_loops:
        _, _, error = gsw_step(st)
        i += 1
    if st.expected is None:
        raise UnboundLocalError("expected_outcome")
    return np.angle(st.A), st.expected, st.errors, st.w
