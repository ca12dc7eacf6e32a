"""Python face of libslmholo: one :class:`Engine` per (plane shape, precision, device).

PyTorch is used only as the device-memory container (allocation, pinned staging, streams); every
computation is a kernel of ``lib/libslmholo.so`` reached through the C ABI of
``include/slm_holo.h``.  There is no CPU path: constructing an Engine without a CUDA device or
without the built library raises.
"""
from __future__ import annotations

import ctypes as C
from collections import namedtuple
from dataclasses import dataclass
from typing import List, Optional

import numpy as np

from . import _ffi, host_logic as hl

_NP_REAL = {"fp32": np.float32, "fp64": np.float64}
_NP_CPLX = {"fp32": np.complex64, "fp64": np.complex128}
_PREC = {"fp32": _ffi.PREC_F32, "fp64": _ffi.PREC_F64}


@dataclass
class LoopResult:
    """Per-plane results of a GS / GD run (device buffers unless converted)."""
    hologram: object                 # [B,H,W] float64: angle(A) / angle(x)
    expected: Optional[object]       # [B,H,W] float64 or None
    errors: List[np.ndarray]         # error_evolution per plane (length = iterations executed)
    iterations: np.ndarray           # int [B]


class Engine:
    """Device context for planes of one shape.

    ``gs`` / ``gd`` take a batch of targets (numpy or device tensors) and leave the results on the
    device; :meth:`to_host` brings them back.  Subclasses may override the ``_mem_*`` hooks and
    ``_load_library`` (the CPU test-suite drives the host emulation of the kernel sources that
    way); the package itself only ever uses this class.
    """

    def __init__(self, shape, precision: str = "fp32", max_batch: int = 1, device=None, stream=None):
        if precision not in _PREC:
            raise ValueError(f"precision must be 'fp32' or 'fp64', not {precision!r}")
        self.shape = (int(shape[0]), int(shape[1]))
        self.precision = precision
        self.max_batch = int(max_batch)
        self.real_dtype = _NP_REAL[precision]
        self.complex_dtype = _NP_CPLX[precision]
        self._lib = self._load_library()
        self._device_index = self._mem_init(device)
        self._stream_handle = self._mem_stream(stream)
        ctx = C.c_void_p()
        rc = self._lib.slm_ctx_create(C.byref(ctx), self._device_index, self.shape[0], self.shape[1],
                                      self.max_batch, _PREC[precision], self._stream_handle)
        if rc == _ffi_shape_error():
            raise ValueError(self._lib.slm_last_error().decode())
        _ffi.check(self._lib, rc)
        self._ctx = ctx
        self._amp_lut = hl.amplitude_lut()

    # ---- memory hooks (torch CUDA tensors) ------------------------------------------------------
    def _load_library(self):
        return _ffi.load()

    def _mem_init(self, device) -> int:
        import torch
        if not torch.cuda.is_available():
            raise _ffi.EngineError("no CUDA device: this engine has no CPU fallback")
        self._torch = torch
        self._dev = torch.device("cuda", torch.cuda.current_device() if device is None else
                                 (device if isinstance(device, int) else torch.device(device).index or 0))
        return self._dev.index

    def _mem_stream(self, stream):
        torch = self._torch
        self._stream = stream if stream is not None else torch.cuda.current_stream(self._dev)
        return C.c_void_p(self._stream.cuda_stream)

    def _mem_empty(self, shape, dtype):
        torch = self._torch
        tdt = {np.dtype(np.float32): torch.float32, np.dtype(np.float64): torch.float64,
               np.dtype(np.complex64): torch.complex64, np.dtype(np.complex128): torch.complex128,
               np.dtype(np.uint8): torch.uint8, np.dtype(np.int32): torch.int32}[np.dtype(dtype)]
        with torch.cuda.stream(self._stream):
            return torch.empty(tuple(shape), dtype=tdt, device=self._dev)

    def _mem_upload(self, array: np.ndarray):
        """Host array -> device tensor.  Large arrays travel on a copy stream of their own and the engine's stream waits
        for them by an event, so an upload neither waits for kernels already queued nor holds them up (the movie driver
        sends batch k+1 while batch k iterates)."""
        torch = self._torch
        array = np.ascontiguousarray(array)
        host = torch.from_numpy(array)
        nbytes = host.numel() * host.element_size()
        if not ((1 << 20) <= nbytes <= (1 << 30)):
            with torch.cuda.stream(self._stream):
                return host.to(self._dev, non_blocking=False)
        if getattr(self, "_upload_stream", None) is None:
            self._upload_stream = torch.cuda.Stream(self._dev)
        side = self._upload_stream
        with torch.cuda.stream(side):
            locked = _dma_ready(torch, host, array)
            if locked:
                # page-locked already (a result of to_host(), or a caller's array seen before, e.g. the one
                # wavefront-correction mask every frame is added to): DMA straight from it, no staging copy
                src = host
            else:
                src = torch.empty(host.shape, dtype=host.dtype, pin_memory=True)      # staging (pooled by torch, reused once its copy is done)
                src.copy_(host)
            dev = src.to(self._dev, non_blocking=True)
            done = torch.cuda.Event()
            done.record(side)
        self._stream.wait_event(done)
        dev.record_stream(self._stream)
        if locked:
            done.synchronize()            # the caller may change its array as soon as we return: wait for THIS copy (not for the kernels)
        return dev

    def upload(self, array):
        """Start sending a host array to the device (see :meth:`_mem_upload`); the result can be handed to gs / gd."""
        return self._mem_upload(np.asarray(array))

    def _mem_plane_max(self, dev) -> np.ndarray:
        """max over each plane of a uint8 device stack [B,H,W] -> float64 [B] on the host."""
        return np.ascontiguousarray(dev.reshape(dev.shape[0], -1).amax(dim=1).double().cpu().numpy(), dtype=np.float64)

    def _mem_plane_sum(self, dev) -> np.ndarray:
        """sum over each plane of a uint8 device stack [B,H,W] -> float64 [B] on the host (exact: integer sums)."""
        return np.ascontiguousarray(dev.reshape(dev.shape[0], -1).sum(dim=1, dtype=self._torch.float64).cpu().numpy(),
                                    dtype=np.float64)

    def _mem_contiguous(self, dev):
        return dev.contiguous()

    def _mem_fill(self, buf, value) -> None:
        """set every element of a device buffer, in order on the engine's stream"""
        with self._torch.cuda.stream(self._stream):
            buf.fill_(value)

    def _mem_repeat(self, plane, n: int):
        """[1,H,W] device plane -> [n,H,W] copies (every target of a batch starts from the same guess)"""
        return plane.expand(n, -1, -1).contiguous()

    def _mem_is_device(self, obj) -> bool:
        return hasattr(obj, "data_ptr")

    def _mem_ptr(self, buf) -> C.c_void_p:
        return C.c_void_p(buf.data_ptr()) if buf is not None else C.c_void_p(0)

    def _mem_download(self, buf) -> np.ndarray:
        torch = self._torch
        nbytes = buf.numel() * buf.element_size()
        if nbytes < (1 << 20) or nbytes > (1 << 30):       # tiny: not worth a pinned allocation; huge: pinning costs more than it saves
            self._stream.synchronize()
            return buf.cpu().numpy()
        with torch.cuda.stream(self._stream):
            host = torch.empty(buf.shape, dtype=buf.dtype, pin_memory=True)
            host.copy_(buf, non_blocking=True)
        self._stream.synchronize()
        return host.numpy()

    def _mem_download_many(self, bufs):
        """Several device buffers -> host arrays with one synchronisation."""
        torch = self._torch
        small = [b for b in bufs if not ((1 << 20) <= b.numel() * b.element_size() <= (1 << 30))]
        if small:
            return [self._mem_download(b) for b in bufs]
        with torch.cuda.stream(self._stream):
            hosts = [torch.empty(b.shape, dtype=b.dtype, pin_memory=True) for b in bufs]
            for h, b in zip(hosts, bufs):
                h.copy_(b, non_blocking=True)
        self._stream.synchronize()
        return [h.numpy() for h in hosts]

    def _mem_np_dtype(self, buf):
        return np.dtype(str(buf.dtype).replace("torch.", ""))

    # ---- helpers ----------------------------------------------------------------------------------
    def _check(self, rc):
        _ffi.check(self._lib, rc)

    def _as_device(self, obj, dtype, what):
        """numpy -> device (with dtype conversion on the host); device tensors must already match."""
        if obj is None:
            return None
        if self._mem_is_device(obj):
            if self._mem_np_dtype(obj) != np.dtype(dtype):
                raise TypeError(f"{what}: device tensor must have dtype {np.dtype(dtype)}")
            return obj
        return self._mem_upload(np.asarray(obj).astype(dtype, copy=False))

    def _targets(self, targets, norms=None):
        """-> (batch, u8_dev, real_dev, aux_source, norms, setup_c64)."""
        if self._mem_is_device(targets):
            if self._mem_np_dtype(targets) != np.uint8:
                raise TypeError("device-resident targets must be uint8")
            t = targets if len(targets.shape) == 3 else targets[None]
            self._shape_check(tuple(t.shape[1:]))
            if norms is None:
                norms = self._mem_plane_max(t)
            norms = np.ascontiguousarray(norms, dtype=np.float64)
            return t.shape[0], self._mem_contiguous(t), None, None, norms, True
        t = np.asarray(targets)
        if t.ndim == 2:
            t = t[None]
        self._shape_check(t.shape[1:])
        kind, treal, amp, c64 = hl.classify_target(t)
        if kind == "u8":
            dev = self._mem_upload(t)
            # np.amax(demanded_output) (algorithms.py:23): a large stack of frames is reduced where it now lies (a
            # host pass over 25 MB per movie batch costs as much as a sixth of the batch's iterations)
            norms = self._mem_plane_max(dev) if t.nbytes >= (4 << 20) else hl.plane_norms(t)
            return t.shape[0], dev, None, None, norms, True
        norms = hl.plane_norms(t)
        return t.shape[0], None, self._mem_upload(treal.astype(self.real_dtype)), amp, norms, c64

    def _shape_check(self, shape):
        if tuple(shape) != self.shape:
            raise ValueError(f"plane shape {tuple(shape)} does not match the engine's {self.shape}")

    def _collect(self, batch, max_loops, hologram, expected) -> LoopResult:
        err = np.empty((batch, max_loops), dtype=np.float64)
        iters = np.empty(batch, dtype=np.int32)
        self._check(self._lib.slm_read_curves(self._ctx, batch, max_loops,
                                              err.ctypes.data_as(C.POINTER(C.c_double)),
                                              iters.ctypes.data_as(C.POINTER(C.c_int))))
        return LoopResult(hologram, expected, [err[b, :iters[b]].copy() for b in range(batch)], iters)

    @staticmethod
    def _dp(a: np.ndarray):
        return a.ctypes.data_as(C.POINTER(C.c_double))

    # ---- transforms ---------------------------------------------------------------------------------
    def fft2(self, x, inverse: bool = False):
        """scipy.fft.fft2 / ifft2 over the last two axes of a [B,H,W] (or [H,W]) complex array."""
        xd = self._as_device(x, self.complex_dtype, "fft2 input")
        batch = 1 if len(xd.shape) == 2 else xd.shape[0]
        self._shape_check(tuple(xd.shape[-2:]))
        out = self._mem_empty(xd.shape, self.complex_dtype)
        self._check(self._lib.slm_fft2(self._ctx, batch, self._mem_ptr(xd), self._mem_ptr(out), int(inverse)))
        return out

    # ---- Gerchberg-Saxton (algorithms.py:10-49) -------------------------------------------------------
    # what _begin hands a run: the targets (fields of _targets), the illumination and the result buffers
    _Begun = namedtuple("_Begun", "batch t8 treal amp norms c64 inc hologram expected")

    def _begin(self, targets, max_loops, unbound, inc_amp, norms, want_expected):
        """What gs, gsw and gd do first.  ``unbound``: the reference's variable that a run without iterations
        leaves unbound."""
        if max_loops < 1:
            raise UnboundLocalError(f"cannot access local variable '{unbound}' where it is not associated with a value")
        batch, t8, treal, amp, norms, c64 = self._targets(targets, norms)
        inc_dev = self._as_device(inc_amp, self.real_dtype, "inc_amp")
        holo = self._mem_empty((batch,) + self.shape, np.float64)
        exp = self._mem_empty((batch,) + self.shape, np.float64) if want_expected else None
        return self._Begun(batch, t8, treal, amp, norms, c64, inc_dev, holo, exp)

    def _gs_run(self, entry, b, phasor0, max_loops, tolerance, *gsw_args) -> LoopResult:
        """slm_gs_run, or slm_gsw_run with its three further arguments ``gsw_args``, after :meth:`_begin` (``b``)."""
        amp_dev = self._mem_upload(b.amp.astype(self.real_dtype)) if b.amp is not None else None
        ph_dev = self._as_device(phasor0, self.complex_dtype, "phasor0")
        self._check(entry(
            self._ctx, b.batch, self._mem_ptr(b.t8), self._mem_ptr(b.treal), self._mem_ptr(amp_dev),
            self._dp(self._amp_lut), self._dp(b.norms), self._mem_ptr(b.inc), self._mem_ptr(ph_dev), int(b.c64),
            int(max_loops), float(tolerance), self._mem_ptr(b.hologram), self._mem_ptr(b.expected), *gsw_args))
        return self._collect(b.batch, max_loops, b.hologram, b.expected)

    def gs(self, targets, max_loops: int, tolerance: float = 0.0, inc_amp=None, phasor0=None,
           want_expected: bool = True, norms=None) -> LoopResult:
        begun = self._begin(targets, max_loops, "expected_outcome", inc_amp, norms, want_expected)
        return self._gs_run(self._lib.slm_gs_run, begun, phasor0, max_loops, tolerance)

    def gsw(self, targets, max_loops: int, tolerance: float = 0.0, inc_amp=None, phasor0=None, weight_limit: float = 10.0,
            weights=None, want_expected: bool = True, norms=None):
        """Weighted GS (include/slm_holo.h slm_gsw_run): GS whose target amplitude carries per-pixel weights, which
        even out the intensities of trap arrays.  ``weights``: initial weights [B,H,W] (host or device; a device tensor
        of the engine's real dtype is updated in place), None = ones.  ``weight_limit`` >= 1 bounds them to
        [1/weight_limit, weight_limit]; 1 gives GS's results bit for bit.  Scale, error curve, tolerance stop and
        expected outcome are GS's.  Returns (LoopResult, weights_device)."""
        if max_loops >= 1 and not float(weight_limit) >= 1.0:        # (max_loops < 1 raises first, in _begin)
            raise ValueError(f"weight_limit must be >= 1, not {weight_limit!r}")
        b = self._begin(targets, max_loops, "expected_outcome", inc_amp, norms, want_expected)
        if b.t8 is not None and self._mem_is_device(targets):
            sums = self._mem_plane_sum(b.t8)
        else:
            sums = np.asarray(targets).reshape(b.batch, -1).sum(axis=1, dtype=np.float64)    # S_T, like the norms
        sums = np.ascontiguousarray(sums, dtype=np.float64)
        shape = (b.batch,) + self.shape
        if weights is None:
            w = self._mem_empty(shape, self.real_dtype)
            self._mem_fill(w, 1.0)
        else:
            w = self._as_device(weights, self.real_dtype, "weights")
            if tuple(w.shape) == self.shape and b.batch == 1:
                w = w[None]
            if tuple(w.shape) != shape:
                raise ValueError(f"weights must have shape {shape}, not {tuple(w.shape)}")
        res = self._gs_run(self._lib.slm_gsw_run, b, phasor0, max_loops, tolerance,
                           self._dp(sums), self._mem_ptr(w), float(weight_limit))
        return res, w

    # ---- gradient descent (algorithms.py:60-112) --------------------------------------------------------
    def gd(self, targets, x0, lr_schedule, max_loops: int, tolerance: float = 0.0, white_attention=1,
           inc_amp=None, want_expected: bool = True, norms=None):
        """``x0``: complex initial guess [B,H,W] (host or device; a device tensor is updated in place).
        Returns (LoopResult, x_device)."""
        b = self._begin(targets, max_loops, "output", inc_amp, norms, want_expected)
        if b.t8 is not None:
            mask_lut, mask_dev = hl.gd_mask_lut(white_attention), None
        else:
            mask_lut = np.zeros(256)
            mask_dev = self._mem_upload(np.asarray(1 + white_attention * np.asarray(targets).reshape((b.batch,) + self.shape) / 255,
                                                   dtype=self.real_dtype))
        x = self._as_device(x0, self.complex_dtype, "x0")
        if len(x.shape) == 2:
            x = x[None]
        lr = np.ascontiguousarray(lr_schedule, dtype=np.float64)
        if lr.shape != (max_loops,):
            raise ValueError("lr_schedule must have max_loops entries")
        self._check(self._lib.slm_gd_run(
            self._ctx, b.batch, self._mem_ptr(b.t8), self._mem_ptr(b.treal), self._mem_ptr(mask_dev), self._dp(mask_lut),
            self._dp(b.norms), self._mem_ptr(b.inc), self._mem_ptr(x), self._dp(lr), int(max_loops), float(tolerance),
            self._mem_ptr(b.hologram), self._mem_ptr(b.expected)))
        return self._collect(b.batch, max_loops, b.hologram, b.expected), x

    def random_phasor_guess(self, u, divide_by=1.0):
        """exp(1j*2*pi*u)/divide_by on the device from a host-drawn uniform stream ``u`` [B,H,W] or [H,W]
        (make_initial_guess "random" / "zeros", algorithms.py:118-124,145-151)."""
        ud = self._as_device(u, np.float64, "u")
        if len(ud.shape) == 2:
            ud = ud[None]
        self._shape_check(tuple(ud.shape[1:]))
        x = self._mem_empty(ud.shape, self.complex_dtype)
        self._check(self._lib.slm_random_phasor(self._ctx, self._mem_ptr(ud), self._mem_ptr(x), _numel(ud), float(divide_by)))
        return x

    def python_random_uniform(self, seed, shape):
        """``prod(shape)`` successive ``random.random()`` draws after ``random.seed(seed)`` as a device
        float64 array (MT19937 continued on the device from CPython's own state); the module-level
        generator is left where the reference's per-pixel loop leaves it (algorithms.py:117-150).

        The stream is a pure function of (seed, count) -- and the reference's CLI always seeds with 42
        (generate_hologram.py:370) -- so the last few streams are kept on the device, keyed by the seeded
        generator state itself; set ``SLM_NO_GUESS_MEMO=1`` to regenerate on every call."""
        import os
        import random
        random.seed(seed)
        version, words, gauss = random.getstate()
        pos = int(words[624])
        n = int(np.prod(shape))
        if pos & 1:                                    # not reachable right after seed(); keep the host path for it
            return self._mem_upload(hl.python_random_stream(seed, n).reshape(shape))
        memo = None if os.environ.get("SLM_NO_GUESS_MEMO") else self.__dict__.setdefault("_stream_memo", {})
        key = (hash(words), n)
        if memo is not None and key in memo:
            u, final_words = memo[key]
            random.setstate((version, final_words, gauss))
            return u.reshape(tuple(shape))
        state = np.array(words[:624], dtype=np.uint32)
        u = self._mem_empty(tuple(shape), np.float64)
        out = np.empty(625, dtype=np.uint32)
        self._check(self._lib.slm_mt19937_uniform(self._ctx, state.ctypes.data_as(C.c_void_p), pos, self._mem_ptr(u), n,
                                                  out.ctypes.data_as(C.c_void_p)))
        final_words = tuple(int(w) for w in out[:624]) + (int(out[624]),)
        random.setstate((version, final_words, gauss))
        if memo is not None:
            while len(memo) >= 4:
                memo.pop(next(iter(memo)))
            memo[key] = (u, final_words)
        return u

    def phase_phasor(self, phase, inc_amp=None):
        """inc * exp(1j*phase) as complex<R> on the device (continue a GS run from a hologram)."""
        pd = self._as_device(phase, np.float64, "phase")
        if len(pd.shape) == 2:
            pd = pd[None]
        self._shape_check(tuple(pd.shape[1:]))
        inc_dev = self._as_device(inc_amp, self.real_dtype, "inc_amp")
        x = self._mem_empty(pd.shape, self.complex_dtype)
        self._check(self._lib.slm_phase_phasor(self._ctx, self._mem_ptr(pd), self._mem_ptr(inc_dev), self._mem_ptr(x),
                                               _numel(pd), self.shape[0] * self.shape[1]))
        return x

    def single_trap_phase(self, row, col, shape=None):
        """np.angle(ifft2(one-hot at (row, col))) in closed form (move_traps.py:64-68)."""
        h, w = shape or self.shape
        out = self._mem_empty((h, w), np.float64)
        self._check(self._lib.slm_single_trap_phase(self._ctx, h, w, int(row), int(col), self._mem_ptr(out)))
        return out

    def trap_frames(self, dots, n_frames, shape=None):
        """uint8 [n_frames,H,W] stack on the device with the pixels ``dots`` = int array [n,3] of
        (frame, y, x) set to 255 (traps_images.py:10-16,87-91 without the PNG round trip)."""
        h, w = shape or self.shape
        dots = np.ascontiguousarray(dots, dtype=np.int32).reshape(-1, 3)
        if dots.size and (dots.min() < 0 or dots[:, 0].max() >= n_frames or dots[:, 1].max() >= h or dots[:, 2].max() >= w):
            raise IndexError("trap position outside the frame")       # numpy raises IndexError at traps_images.py:89
        frames = self._mem_empty((n_frames, h, w), np.uint8)
        ddev = self._mem_upload(dots) if dots.size else None
        self._check(self._lib.slm_trap_frames(self._ctx, self._mem_ptr(frames), int(n_frames), h, w, self._mem_ptr(ddev), len(dots)))
        return frames

    def fourier_guess(self, targets, inc_amp=None):
        """make_initial_guess("fourier") (algorithms.py:154-157) on the device -> complex [B,H,W]."""
        batch, t8, _treal, amp, _norms, c64 = self._targets(targets)
        amp_dev = self._mem_upload(amp.astype(self.real_dtype)) if amp is not None else None
        inc_dev = self._as_device(inc_amp, self.real_dtype, "inc_amp")
        x = self._mem_empty((batch,) + self.shape, self.complex_dtype)
        self._check(self._lib.slm_fourier_guess(self._ctx, batch, self._mem_ptr(t8), self._mem_ptr(amp_dev),
                                                self._dp(self._amp_lut), self._mem_ptr(inc_dev), int(c64), self._mem_ptr(x)))
        return x

    # ---- preview, analytic holograms, quantisers -----------------------------------------------------------
    def expected_outcome(self, hologram, norm=255):
        """generate_hologram.py:24-29: |fft2(exp(1j*h))|^2 / max * norm."""
        h = self._as_device(hologram, np.float64, "hologram")
        hb = h if len(h.shape) == 3 else h[None]
        self._shape_check(tuple(hb.shape[1:]))
        norms = np.broadcast_to(np.asarray(norm, dtype=np.float64), (hb.shape[0],)).copy()
        out = self._mem_empty(hb.shape, np.float64)
        self._check(self._lib.slm_expected_outcome(self._ctx, hb.shape[0], self._mem_ptr(hb), self._dp(norms), self._mem_ptr(out)))
        return out if len(h.shape) == 3 else out[0]

    def deflect_phase(self, angle, px_distance, wavelength, unit_angle, shape=None):
        h, w = shape or self.shape
        const, sy, sx = hl.deflect_scalars(angle, px_distance, wavelength, unit_angle)
        out = self._mem_empty((h, w), np.float64)
        self._check(self._lib.slm_deflect_phase(self._ctx, h, w, const, sy, sx, self._mem_ptr(out)))
        return out

    def lens_phase(self, focal_length, px_distance, wavelength, shape=None, uint8_quirk=True):
        h, w = shape or self.shape
        k, f2 = hl.lens_scalars(focal_length, wavelength)
        out = self._mem_empty((h, w), np.float64)
        self._check(self._lib.slm_lens_phase(self._ctx, h, w, float(px_distance), k, f2, int(uint8_quirk), self._mem_ptr(out)))
        return out

    def add_mod2pi(self, a, b):
        """(a + b) % 2pi with ``b`` one plane broadcast over the batch of ``a``."""
        ad = self._as_device(a, np.float64, "a")
        bd = self._as_device(b, np.float64, "b")
        n, plane = _numel(ad), _numel(bd)
        if n % plane:
            raise ValueError("operands could not be broadcast together")
        out = self._mem_empty(ad.shape, np.float64)
        self._check(self._lib.slm_add_mod2pi(self._ctx, self._mem_ptr(ad), self._mem_ptr(bd), self._mem_ptr(out), n, plane))
        return out

    def quantize(self, phase, mask=None, ct2pi=256, mode=_ffi.QUANT_FLOOR):
        pd = self._as_device(phase, np.float64, "phase")
        md = self._as_device(mask, np.float64, "mask")
        n = _numel(pd)
        plane = _numel(md) if md is not None else n
        if n % plane:
            raise ValueError("operands could not be broadcast together")
        out = self._mem_empty(pd.shape, np.uint8)
        self._check(self._lib.slm_quantize(self._ctx, self._mem_ptr(pd), self._mem_ptr(md), float(ct2pi), int(mode),
                                           self._mem_ptr(out), n, plane))
        return out

    def quantize_grey(self, grey, mask, ct2pi):
        gd_ = self._as_device(grey, np.uint8, "grey")
        md = self._as_device(mask, np.float64, "mask")
        n, plane = _numel(gd_), _numel(md)
        out = self._mem_empty(gd_.shape, np.uint8)
        self._check(self._lib.slm_quantize_grey(self._ctx, self._mem_ptr(gd_), self._mem_ptr(md), float(ct2pi),
                                                self._mem_ptr(out), n, plane))
        return out

    # ---- misc ---------------------------------------------------------------------------------------------
    def to_host(self, buf) -> Optional[np.ndarray]:
        return None if buf is None else self._mem_download(buf)

    def to_host_many(self, bufs):
        return self._mem_download_many(list(bufs))

    def to_host_into(self, buf, out: np.ndarray, after=None):
        """Start copying a device buffer into the host array ``out`` (same shape and dtype) while the engine's
        stream goes on with other work; returns a handle whose ``join()`` waits for the copy.  ``after``: a
        torch.distributed work handle that must complete first (the collective that fills ``buf``)."""
        return self._mem_download_into(buf, out, after)

    def gather_to_root(self, buf, padded_shape, dtype, dist, dst: int = 0):
        """Device-to-device gather of one equally shaped block per rank onto rank ``dst`` (NCCL over NVLink), ordered
        behind the engine's stream and not waited for: returns ``.blocks`` (one device buffer per rank on ``dst``,
        else None) and ``.work`` (pass it to :meth:`to_host_into`).  ``buf`` may be None or shorter than
        ``padded_shape`` along the first axis (ragged last batch): the tail is padding nobody reads."""
        return self._mem_gather_to_root(buf, tuple(padded_shape), dtype, dist, dst)

    def _mem_gather_to_root(self, buf, padded_shape, dtype, dist, dst):
        torch = self._torch
        with torch.cuda.stream(self._stream):          # the collective is ordered behind the kernels of this stream
            if buf is None or tuple(buf.shape) != padded_shape:
                pad = self._mem_empty(padded_shape, dtype)
                if buf is not None:
                    pad[:buf.shape[0]].copy_(buf)
                buf = pad
            blocks = [torch.empty_like(buf) for _ in range(dist.get_world_size())] if dist.get_rank() == dst else None
            work = dist.gather(buf, blocks, dst=dst, async_op=True)
        return _Gathered(blocks, work, buf)

    def _mem_download_into(self, buf, out, after=None):
        import threading
        torch = self._torch
        if not out.flags.c_contiguous or out.dtype != self._mem_np_dtype(buf) or tuple(out.shape) != tuple(buf.shape):
            raise ValueError("to_host_into: destination must be a C-contiguous array of the buffer's shape and dtype")
        if getattr(self, "_copy_stream", None) is None:
            self._copy_stream = torch.cuda.Stream(self._dev)
        side = self._copy_stream
        ready = torch.cuda.Event()
        ready.record(self._stream)                       # everything that produced `buf`
        buf.record_stream(side)

        dst = torch.from_numpy(out)
        if dst.is_pinned():                              # page-locked destination (host_empty): a plain asynchronous DMA
            with torch.cuda.stream(side):
                if after is not None:
                    after.wait()                         # the copy stream (not the engine's) waits for the collective
                side.wait_event(ready)
                dst.copy_(buf, non_blocking=True)
                done = torch.cuda.Event()
                done.record(side)

            class Copy:
                def join(self_inner):
                    done.synchronize()
            return Copy()

        def work():
            with torch.cuda.device(self._dev), torch.cuda.stream(side):
                if after is not None:
                    after.wait()
                side.wait_event(ready)
                dst.copy_(buf)                           # device -> host array directly (the driver stages pageable memory)
                side.synchronize()
        th = threading.Thread(target=work, daemon=True)
        th.start()
        return th

    def host_empty(self, shape, dtype) -> np.ndarray:
        """Host array for results that are read back with :meth:`to_host_into`: page-locked (from PyTorch's caching
        host allocator, so repeated calls neither pin nor page-fault again) up to ``SLM_PINNED_RESULT_BYTES``
        (default 8 GiB: a 1024-frame movie of float64 holograms at the SLM shape is 6 GiB), ordinary memory beyond."""
        return self._mem_host_empty(shape, dtype)

    def _mem_host_empty(self, shape, dtype):
        import os
        torch = self._torch
        nbytes = int(np.prod(shape)) * np.dtype(dtype).itemsize
        if nbytes == 0 or nbytes > int(os.environ.get("SLM_PINNED_RESULT_BYTES", 8 << 30)):
            return np.empty(shape, dtype=dtype)
        tdt = {np.dtype(np.float64): torch.float64, np.dtype(np.float32): torch.float32, np.dtype(np.uint8): torch.uint8}[np.dtype(dtype)]
        return torch.empty(tuple(shape), dtype=tdt, pin_memory=True).numpy()

    KINDS = ("row_pass", "col_pass", "col_stats", "row_plain", "col_plain", "elementwise")

    def profile(self, enable: bool) -> None:
        """Bracket every kernel launch with CUDA events on the engine's stream (bench roofline)."""
        self._check(self._lib.slm_ctx_profile(self._ctx, int(enable)))

    def profile_read(self):
        """{kind: (total ms, launches)} since the last read; synchronises the stream."""
        ms = (C.c_double * 6)()
        cnt = (C.c_longlong * 6)()
        self._check(self._lib.slm_ctx_profile_read(self._ctx, ms, cnt))
        return {k: (ms[i], cnt[i]) for i, k in enumerate(self.KINDS)}

    def launch_count(self) -> int:
        return int(self._lib.slm_ctx_launch_count(self._ctx))

    def workspace_bytes(self) -> int:
        return int(self._lib.slm_ctx_workspace_bytes(self._ctx))

    def close(self):
        if getattr(self, "_ctx", None):
            self._lib.slm_ctx_destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass


class _Gathered:
    """Result of Engine.gather_to_root: keeps the source block alive until the collective has run."""

    def __init__(self, blocks, work, source):
        self.blocks, self.work, self.source = blocks, work, source


# Host arrays a caller passes again and again (same memory) are page-locked in place on their second use, so later
# uploads skip the staging copy.  The registration ends when the array that owns the memory is collected.
_SEEN_ONCE = {}
_LOCKED = {}
_LOCK_BUDGET = 1 << 30
_LOCK_MIN = 4 << 20           # cudaHostRegister costs ~2 ms whatever the size: not worth it for small arrays


def _dma_ready(torch, host, array: np.ndarray) -> bool:
    """May `array` be copied to the device asynchronously, straight from where it lies?  Yes for PyTorch's own pinned
    memory (results of to_host) and for ranges lying COMPLETELY inside memory this module has page-locked; an array
    that only begins in a locked range (``is_pinned`` looks at the first byte alone) must take the staged copy."""
    lo, hi = array.ctypes.data, array.ctypes.data + array.nbytes
    for (p, n) in _LOCKED:
        if p <= lo < p + n or p < hi <= p + n:
            return lo >= p and hi <= p + n
    if host.is_pinned():
        return True
    return array.nbytes >= _LOCK_MIN and _page_lock_if_reused(torch, array)


def _page_lock_if_reused(torch, array: np.ndarray) -> bool:
    import weakref
    owner = array
    while isinstance(getattr(owner, "base", None), np.ndarray):
        owner = owner.base
    if not isinstance(owner, np.ndarray) or owner.base is not None or not owner.flags.owndata:
        return False                                    # memory owned by something we cannot watch
    key = (array.ctypes.data, array.nbytes)
    if key in _LOCKED:
        return True
    if _SEEN_ONCE.pop(key, None) != id(owner):
        if len(_SEEN_ONCE) > 64:
            _SEEN_ONCE.clear()
        _SEEN_ONCE[key] = id(owner)
        return False
    if sum(n for _, n in _LOCKED) + array.nbytes > _LOCK_BUDGET:
        return False
    lib = _ffi.load()
    if lib.slm_host_register(C.c_void_p(array.ctypes.data), array.nbytes) != 0:
        return False
    _LOCKED[key] = True

    def release(k=key, ptr=array.ctypes.data):
        if _LOCKED.pop(k, None):
            try:
                lib.slm_host_unregister(C.c_void_p(ptr))
            except Exception:
                pass
    weakref.finalize(owner, release)
    return True


def _numel(buf) -> int:
    n = 1
    for s in buf.shape:
        n *= int(s)
    return n


def _ffi_shape_error() -> int:
    return -2


_ENGINES = {}


def get_engine(shape, precision="fp32", max_batch=1, device=None) -> Engine:
    """Cached engine for (shape, precision, device) able to hold at least ``max_batch`` planes."""
    import torch
    dev = torch.cuda.current_device() if device is None else device
    key = (tuple(int(s) for s in shape), precision, str(dev))
    eng = _ENGINES.get(key)
    if eng is None or eng.max_batch < max_batch:
        if eng is not None:
            eng.close()
        eng = Engine(shape, precision, max_batch, device)
        _ENGINES[key] = eng
    return eng


def supported_lengths() -> List[int]:
    lib = _ffi.load()
    buf = (C.c_int * 64)()
    n = lib.slm_supported_lengths(buf, 64)
    return [buf[i] for i in range(min(n, 64))]
