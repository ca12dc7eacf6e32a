"""Multi-plane gradient descent as this project defines it: the checker of ``Engine.gd_multiplane`` /
``slm_gd_multiplane_run``.

TEST INFRASTRUCTURE ONLY -- never imported by the shipped package.

The reference's GD (numpy_port.gd_step) for K target planes T_k that share one hologram, plane k where a lens of
phase alpha_k * rho^2 brings the Fourier plane (L_k = exp(1j * alpha_k * rho^2), oracle/multiplane.py).  The cost is
the MEAN of the planes' errors, so the learning rate keeps its one-plane meaning.  Per hologram: one variable x
(GD's ``input``), one illumination, one learning-rate schedule; per plane: T_k, norm_k = amax(T_k) and mask_k =
1 + white_attention T_k / 255 with numpy's dtype rules (numpy_port.gd_setup).  Each iteration:

    B     = x / |x| * inc
    per plane:  F_k   = fft2(B L_k)                        (B itself where alpha_k = 0)
                out_k = |F_k|^2 norm_k / amax(|F_k|^2)
                G_k   = ifft2(mask_k F_k (out_k - T_k))
                err_k = error_f(out_k, T_k, HW)
    dEdF  = (sum_k G_k conj(L_k)) inc / K                  (the sum starts from its first term; no product at alpha = 0)
    x    -= lr_i dEdX_complex(dEdF, x)

The loop runs while ANY plane's error is above the tolerance and i < max_loops, so a hologram's K curves have one
length; the learning rate follows numpy_port's unsettle rule.  K = 1 with alpha = 0 is numpy_port.gd_step operation
for operation (the / 1 is exact).
"""
from __future__ import annotations

from dataclasses import dataclass, field
from typing import List, Optional

import numpy as np
from scipy.fft import fft2, ifft2

from . import multiplane as MP
from . import numpy_port as P


@dataclass
class MPGDState:
    planes: List[P.GDState]              # per plane: GD's target, norm, mask, space norm; .x is unused
    lenses: List[Optional[np.ndarray]]   # L_k, None where alpha_k == 0
    inc_amp: np.ndarray
    x: np.ndarray
    learning_rate: float
    unsettle: int
    max_loops: int
    i: int = 0
    outputs: Optional[List[np.ndarray]] = None
    errors: List[List[float]] = field(default_factory=list)


def mpgd_setup(targets, alphas, x0, *, white_attention=1, learning_rate=0.005, unsettle=0, max_loops=100,
               incomming_intensity="uniform") -> MPGDState:
    """State before iteration 0 from the initial guess ``x0`` (one plane)."""
    targets = [np.asarray(t) for t in targets]
    if len(targets) != len(alphas):
        raise ValueError("one defocus coefficient per target plane")
    planes = [P.gd_setup(t, white_attention=white_attention, incomming_intensity=incomming_intensity,
                         max_loops=max_loops, x0=x0) for t in targets]
    lenses = [None if a == 0 else MP.lens_field(targets[0].shape, a) for a in alphas]
    return MPGDState(planes, lenses, planes[0].inc_amp, np.array(x0, dtype=complex), learning_rate, unsettle,
                     max_loops, errors=[[] for _ in targets])


def fourier_guess(targets, alphas, incomming_intensity="uniform"):
    """The "fourier" initial guess: inc exp(i angle(sum_k ifft2(sqrt(T_k)) conj(L_k))), multi-plane GS's setup sum
    (one plane at alpha = 0: numpy_port.initial_guess("fourier"))."""
    return MP.mp_first_phasor(MP.mp_setup(targets, alphas, incomming_intensity))


def mpgd_step(st: MPGDState):
    """One iteration.  Returns (outputs, errors) of the planes; updates st.x, st.learning_rate, st.i."""
    B = st.x / abs(st.x) * st.inc_amp
    outs, errs, terms = [], [], []
    for k, (p, L) in enumerate(zip(st.planes, st.lenses)):
        F = fft2(B if L is None else B * L)
        output_unnormed = abs(F) ** 2
        output = output_unnormed * p.norm / np.amax(output_unnormed)
        G = ifft2(p.mask * F * (output - p.target))
        terms.append(G if L is None else G * np.conj(L))
        err = P.mean_square_error(output, p.target, p.space_norm)
        st.errors[k].append(err)
        outs.append(output), errs.append(err)
    dEdF = MP._sum(terms) * st.inc_amp / len(terms)
    st.x = st.x - st.learning_rate * P.tangent_gradient_rows(dEdF, st.x)
    st.outputs = outs
    st.i += 1
    if st.unsettle and st.i % int(round(st.max_loops / (st.unsettle + 1))) == 0:
        st.learning_rate *= 2
    return outs, errs


def mpgd_loop(st: MPGDState, tolerance=0):
    """GD's loop condition over all planes: run while any plane's error > tolerance (NaN: not above)."""
    errs = [tolerance + 1]
    while any(e > tolerance for e in errs) and st.i < st.max_loops:
        _, errs = mpgd_step(st)
    if st.outputs is None:
        raise UnboundLocalError("output")
    return np.angle(st.x), st.outputs, st.errors, st.learning_rate


def mpgd_run(targets, alphas, x0, max_loops, tolerance=0, **kw):
    """Returns (hologram, [output_k], [errors_k], final learning rate)."""
    return mpgd_loop(mpgd_setup(targets, alphas, x0, max_loops=max_loops, **kw), tolerance)
