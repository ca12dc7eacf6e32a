"""Drop-in replacements for the reference's ``src/algorithms.py`` (same names, same
``(numpy array, argparse.Namespace) -> (hologram, expected_outcome, error_evolution)`` contract),
running on the B200 engine.

Optional attributes on ``args`` (absent => default) select engine behaviour without changing the
reference's signature:
    ``precision``  "fp32" (default; env SLM_PRECISION overrides the default) or "fp64"
    ``device``     CUDA device index (default: current device)

Differences a caller can observe are limited to: the ``\\rloop i/N`` progress text is printed once
at the end instead of after every iteration (the loop runs on the device without host round
trips), and floating-point results agree with numpy within the tolerances in DESIGN.md rather
than bit for bit.  With ``args.gif`` the loop is run in chunks that end at the iterations the
reference snapshots (``i % gif_skip == 0``, algorithms.py:40-41,94-101) and the same PNG frames
are written.
"""
from __future__ import annotations

import os

import numpy as np

from . import constants, host_logic as hl
from .engine import Engine, get_engine

__all__ = ["gerchberg_saxton", "weighted_gerchberg_saxton", "multiplane_gerchberg_saxton", "gradient_descent",
           "multiplane_gradient_descent", "make_initial_guess", "error_f", "printout", "complex_to_real_phase", "dEdX_complex",
           "add_gif_image"]


def _precision(args) -> str:
    return getattr(args, "precision", None) or os.environ.get("SLM_PRECISION", "fp32")


def _engine(shape, args, batch=1) -> Engine:
    return get_engine(shape, _precision(args), batch, getattr(args, "device", None))


def _illumination(args, shape):
    """algorithms.py:14-19 / :65-70 -> sqrt(illumination) plane or None for 'uniform'."""
    if args.incomming_intensity == "uniform":
        return None
    import PIL.Image as im
    plane = np.array(im.open(args.incomming_intensity))
    amp = np.sqrt(plane)                       # float16 for an 8-bit image, like the reference
    if amp.shape != tuple(shape):
        raise ValueError(f"operands could not be broadcast together with shapes {amp.shape} {tuple(shape)}")
    return amp.astype(np.float64)


def _progress(i, max_loops):
    print(f"\rloop {i}/{max_loops}", end="")
    print()


def _report(args, hologram, expected, errors):
    """The drop-ins' epilogue: progress line, then the reference's printout with ``args.print_info``."""
    _progress(len(errors), args.max_loops)
    if args.print_info:
        print()
        printout(errors[-1], len(errors), errors, args.plot_error)
    return hologram, expected, errors


def _to_host(eng, res):
    """One plane's LoopResult -> (hologram, expected, errors) on the host."""
    hologram, expected = (a[0] for a in eng.to_host_many([res.hologram, res.expected]))
    return hologram, expected, [np.float64(e) for e in res.errors[0]]


def _gs_family(demanded_output, args, run):
    """gerchberg_saxton and weighted_gerchberg_saxton: ``run(eng, target, max_loops, inc, phasor0)`` -> LoopResult."""
    target = np.asarray(demanded_output)
    inc = _illumination(args, target.shape)
    if args.max_loops < 1 or not (args.tolerance + 1 > args.tolerance):
        # the reference's loop body never runs and `expected_outcome` is unbound at :49
        print()
        raise UnboundLocalError("cannot access local variable 'expected_outcome' where it is not associated with a value")
    eng = _engine(target.shape, args)
    if not getattr(args, "gif", False):
        return _report(args, *_to_host(eng, run(eng, target, int(args.max_loops), inc, None)))
    phasor = None

    def restart(res):
        # the next chunk starts from B = inc*exp(1j*angle(A)) (algorithms.py:30), which is what the next iteration of
        # an uninterrupted run computes
        nonlocal phasor
        phasor = eng.phase_phasor(res.hologram, inc)
    return _report(args, *_with_snapshots(eng, args, lambda n, done: run(eng, target, n, inc, phasor), restart))


def gerchberg_saxton(demanded_output, args):
    """classical Gerchberg-Saxton algorithm for generating phase holograms in far field regime
    (reference: algorithms.py:10-49)."""
    return _gs_family(demanded_output, args, lambda eng, target, n, inc, phasor0:
                      eng.gs(target, n, float(args.tolerance), inc_amp=inc, phasor0=phasor0))


def weighted_gerchberg_saxton(demanded_output, args):
    """Weighted Gerchberg-Saxton (Di Leonardo, Ianni & Ruocco, Opt. Express 15, 1913 (2007)): GS whose target
    amplitude carries per-pixel weights, fed back each iteration so that the reconstructed intensity follows the
    target's levels -- plain GS leaves trap arrays with a spread of intensities.  The contract of
    :func:`gerchberg_saxton` (error curve and expected outcome are computed the same way, so the curves compare
    directly), plus the optional ``args.weight_limit`` (default 10): the weights stay within [1/limit, limit].
    ``args.gif`` snapshots are not offered (ValueError)."""
    if getattr(args, "gif", False):
        raise ValueError("weighted_gerchberg_saxton does not offer GIF snapshots (args.gif)")
    return _gs_family(demanded_output, args, lambda eng, target, n, inc, phasor0:
                      eng.gsw(target, n, float(args.tolerance), inc_amp=inc, phasor0=phasor0,
                              weight_limit=float(getattr(args, "weight_limit", 10.0)))[0])


def multiplane_gerchberg_saxton(demanded_outputs, focal_lengths, args):
    """Multi-plane Gerchberg-Saxton (Haist et al., Opt. Commun. 140, 299 (1997)): one phase hologram for several target
    images, image k in focus where ``add_lens(hologram, focal_lengths[k])`` would bring the Fourier plane (None or inf:
    the Fourier plane itself) -- traps in 3-D.  ``demanded_outputs``: K images of one shape (a list or a [K,H,W]
    array), K <= 8.  Returns ``(hologram, expected[K,H,W], [errors_k])``: each plane's expected outcome and error curve
    as :func:`gerchberg_saxton` computes them, every curve of the same length (the loop runs while any plane's error is
    above ``args.tolerance``).  Lenses use the paraxial phase -pi r^2 / (lambda f) at the pixel pitch and wavelength of
    ``constants``; a focal length short enough to alias at the plane's edge is refused (ValueError), as are
    ``args.gif``, an all-zero target image and a count of focal lengths other than K."""
    targets, focal_lengths = _multiplane_targets("multiplane_gerchberg_saxton", demanded_outputs, focal_lengths, args)
    inc = _illumination(args, targets.shape[1:])
    if args.max_loops < 1 or not (args.tolerance + 1 > args.tolerance):
        print()
        raise UnboundLocalError("cannot access local variable 'expected_outcome' where it is not associated with a value")
    alphas = _alphas(focal_lengths)
    eng = _engine(targets.shape[1:], args, batch=len(targets))
    res = eng.gs_multiplane(targets, alphas, int(args.max_loops), float(args.tolerance), inc_amp=inc)
    return _multiplane_report(args, eng, res)


def _multiplane_targets(name, demanded_outputs, focal_lengths, args):
    """The multi-plane drop-ins' refusals (``name`` in the messages) -> (targets as one [K,H,W] array, focal lengths
    as a list)."""
    if getattr(args, "gif", False):
        raise ValueError(f"{name} does not offer GIF snapshots (args.gif)")
    targets = np.stack([np.asarray(t) for t in demanded_outputs])
    focal_lengths = list(focal_lengths)
    if len(focal_lengths) != len(targets):
        raise ValueError(f"{len(targets)} target images need {len(targets)} focal lengths, not {len(focal_lengths)}")
    for k, t in enumerate(targets):
        if not np.any(t):
            raise ValueError(f"target image {k} is all zero: it has no intensity to place")
    return targets, focal_lengths


def _alphas(focal_lengths):
    return [hl.defocus_coefficient(f, constants.px_distance, constants.wavelength) for f in focal_lengths]


def _multiplane_report(args, eng, res):
    """The multi-plane drop-ins' epilogue: (hologram, expected[K,H,W], [errors_k]) on the host, progress line, and
    the reference's printout per plane with ``args.print_info``."""
    hologram, expected = (a[0] for a in eng.to_host_many([res.hologram, res.expected]))
    errors = [[np.float64(e) for e in curve] for curve in res.errors[0]]
    _progress(len(errors[0]), args.max_loops)
    if args.print_info:
        for k, curve in enumerate(errors):
            print(f"\nplane {k}")
            printout(curve[-1], len(curve), curve, args.plot_error)
    return hologram, expected, errors


def gradient_descent(demanded_output, args):
    """phase holograms by gradient descent on a complex field (reference: algorithms.py:60-112).
    ``args.learning_rate`` is updated by the ``unsettle`` rule exactly as the reference does."""
    target = np.asarray(demanded_output)
    inc = _illumination(args, target.shape)
    eng = _engine(target.shape, args)
    inc_amp = np.float64(1.0) if inc is None else inc        # (uniform illumination: make_initial_guess takes a scalar too)
    x = make_initial_guess(args.initial_guess, inc_amp, target, args.random_seed, _engine_hint=eng, _device=True)
    if args.print_info:
        print("computing hologram")
    if args.max_loops < 1 or not (args.tolerance + 1 > args.tolerance):
        print()
        raise UnboundLocalError("cannot access local variable 'output' where it is not associated with a value")
    during, after = hl.learning_rate_schedule(args.learning_rate, args.unsettle, int(args.max_loops))

    def chunk(n, done):
        nonlocal x
        res, x = eng.gd(target, x, during[done:done + n], n, float(args.tolerance),
                        white_attention=args.white_attention, inc_amp=inc)
        return res
    if getattr(args, "gif", False):
        hologram, expected, errors = _with_snapshots(eng, args, chunk)
    else:
        hologram, expected, errors = _to_host(eng, chunk(int(args.max_loops), 0))
    args.learning_rate = after[len(errors)]
    return _report(args, hologram, expected, errors)


def multiplane_gradient_descent(demanded_outputs, focal_lengths, args):
    """Multi-plane gradient descent: one phase hologram for several target images, image k in focus where
    ``add_lens(hologram, focal_lengths[k])`` would bring the Fourier plane (None or inf: the Fourier plane itself) --
    :func:`gradient_descent` for traps in 3-D.  It descends on the mean of the planes' errors, so
    ``args.learning_rate`` means what it means for one plane.  Arguments as :func:`gradient_descent`
    (``initial_guess``, ``random_seed``, ``learning_rate``, ``unsettle``, ``white_attention``,
    ``incomming_intensity``; one initial guess for the hologram, "fourier" being taken from the sum of the planes'
    setup fields as multi-plane GS takes it), targets and focal lengths as :func:`multiplane_gerchberg_saxton`, with its
    refusals.  Returns ``(hologram, expected[K,H,W], [errors_k])``, every curve of the same length (the loop runs while
    any plane's error is above ``args.tolerance``); ``args.learning_rate`` is updated as :func:`gradient_descent`
    updates it.  One plane with focal length None gives :func:`gradient_descent`'s results bit for bit, except from
    the "fourier" guess, whose phase is taken through the multi-plane setup sum."""
    targets, focal_lengths = _multiplane_targets("multiplane_gradient_descent", demanded_outputs, focal_lengths, args)
    alphas = _alphas(focal_lengths)
    inc = _illumination(args, targets.shape[1:])
    eng = _engine(targets.shape[1:], args, batch=len(targets))
    if args.initial_guess == "fourier":
        hl.host_initial_guess("fourier", targets.shape[1:], args.random_seed)     # seeds `random` as make_initial_guess does
        x = eng.multiplane_fourier_guess(targets, alphas, inc)
    else:
        inc_amp = np.float64(1.0) if inc is None else inc
        x = make_initial_guess(args.initial_guess, inc_amp, targets[0], args.random_seed, _engine_hint=eng, _device=True)
    if args.print_info:
        print("computing hologram")
    if args.max_loops < 1 or not (args.tolerance + 1 > args.tolerance):
        print()
        raise UnboundLocalError("cannot access local variable 'output' where it is not associated with a value")
    during, after = hl.learning_rate_schedule(args.learning_rate, args.unsettle, int(args.max_loops))
    res, _ = eng.gd_multiplane(targets, alphas, x, during, int(args.max_loops), float(args.tolerance),
                               white_attention=args.white_attention, inc_amp=inc)
    out = _multiplane_report(args, eng, res)
    args.learning_rate = after[len(out[2][0])]
    return out


def make_initial_guess(initial_guess_type, incomming_amplitude, demanded_output, seed, _engine_hint=None, _device=False):
    """reference: algorithms.py:115-158.  The random families are drawn on the host from the same
    MT19937 stream as the reference's per-pixel ``random.random()`` calls; "fourier" runs on the
    device."""
    target = np.asarray(demanded_output)
    if _device and initial_guess_type in ("random", "zeros"):
        # called from gradient_descent: the MT19937 stream and exp(2*pi*i*u) are both produced on the device
        u = _engine_hint.python_random_uniform(seed, target.shape)
        return _engine_hint.random_phasor_guess(u, 100.0 if initial_guess_type == "zeros" else 1.0)
    guess = hl.host_initial_guess(initial_guess_type, target.shape, seed)
    if guess is not None:
        return guess
    eng = _engine_hint or get_engine(target.shape, os.environ.get("SLM_PRECISION", "fp32"))
    inc = np.asarray(incomming_amplitude, dtype=np.float64)
    uniform = inc.shape == () or bool(np.all(inc == 1))
    x = eng.fourier_guess(target, None if uniform else np.broadcast_to(inc, target.shape))
    if _device:
        return x
    return eng.to_host(x)[0].astype(np.complex128)


def error_f(actual, correct, norm):
    """reference: algorithms.py:161-162 (host arrays; the loops compute this on the device)."""
    return np.sum((actual - correct) ** 2) / norm


def printout(error, loop_num, error_evol, plot_error):
    """reference: algorithms.py:165-172."""
    print(f"error: {error}")
    print(f"number of loops: {loop_num}")
    if plot_error:
        import matplotlib.pyplot as plt
        plt.plot(error_evol)
        plt.xlabel("loop number")
        plt.ylabel("error")
        plt.show()


def complex_to_real_phase(complex_phase, correspond_to2pi=256):
    """reference: algorithms.py:175-176."""
    return (np.angle(complex_phase) + np.pi) / (2 * np.pi) * correspond_to2pi


def dEdX_complex(dEdF, x):
    """reference: algorithms.py:179-185 (host helper; the GD loop fuses this into the SLM-plane pass)."""
    rE, iE = dEdF.real, dEdF.imag
    rx, ix = x.real, x.imag
    ax = abs(x)
    re_res = rE * (1 / ax - rx**2 / ax**3) + iE * (-(rx * ix) / ax**3)
    im_res = rE * (-(rx * ix) / ax**3) + iE * (1 / ax - ix**2 / ax**3)
    return re_res + 1j * im_res


def add_gif_image(args, expected_outcome, A, i):
    """reference: algorithms.py:52-57 (host-side PNG dump of one frame)."""
    import PIL.Image as im
    if args.gif_type == "h":
        img = im.fromarray((np.angle(A) + np.pi) * args.correspond_to2pi / (2 * np.pi))
    if args.gif_type == "i":
        img = im.fromarray(expected_outcome)
    img.convert("L").save(f"{args.gif_source_dir}/{i // args.gif_skip}.png")


def _save_snapshot(args, expected, hologram, i):
    """One GIF source frame exactly as the reference writes it (algorithms.py:52-57 / :94-101)."""
    import PIL.Image as im
    if args.gif_type == "h":
        img = im.fromarray((hologram + np.pi) * args.correspond_to2pi / (2 * np.pi))
    if args.gif_type == "i":
        img = im.fromarray(expected)
    img.convert("L").save(f"{args.gif_source_dir}/{i // args.gif_skip}.png")


def _with_snapshots(eng, args, chunk, restart=None):
    """The loop in chunks that end at the iterations the reference snapshots; ``chunk(n, done)`` runs the next ``n``
    iterations after ``done`` and returns their LoopResult; ``restart(result)`` follows every chunk that does not end
    the run."""
    errors, done, hologram, expected = [], 0, None, None
    for n in hl.snapshot_chunks(int(args.max_loops), int(args.gif_skip)):
        res = chunk(n, done)
        errors += [np.float64(e) for e in res.errors[0]]
        hologram, expected = eng.to_host(res.hologram)[0], eng.to_host(res.expected)[0]
        last = done + len(res.errors[0]) - 1
        if last % args.gif_skip == 0:
            _save_snapshot(args, expected, hologram, last)
        done += n
        # the loop condition (algorithms.py:29,83) holds across chunk borders: a chunk's last error ends the run too
        if len(res.errors[0]) < n or not (errors[-1] > float(args.tolerance)):
            break
        if restart:
            restart(res)
    return hologram, expected, errors
