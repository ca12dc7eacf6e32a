"""Gerchberg-Saxton on ONE very large square plane split by rows over the ranks of a process group
(BASELINE config 5: a 16384^2 grid on 2/4/8 GPUs): slab-decomposed 2-D transforms with all-to-all
transposes.

Rank p owns rows [p*h, (p+1)*h) of the N x N field, h = N / world.  One GS iteration
(reference: algorithms.py:30-38) is

    row pass      finish ifft2 along the rows, B = exp(1j*angle(A)), start fft2 along the rows   (local)
    exchange      pack blocks -> all-to-all -> every rank holds h whole COLUMNS as contiguous lines
    Fourier pass  finish fft2 along those lines, amplitude replacement + error sums, start ifft2   (local)
    all-reduce    max |C|^2 and the three error sums (4 doubles)
    exchange      all-to-all back -> unpack into the row slab

i.e. two all-to-alls and one tiny all-gather per iteration; the target is exchanged once.  All array work is done by
kernels of libslmholo (``slm_rows_*``, ``slm_transpose_blocks*``).  The loop state (the context's scale, max, iteration
count and loop-ended flag, and the run's error curve) lives on the device: with ``tolerance <= 0`` -- every caller of the
reference -- no iteration waits for the host.

Two ways of moving the blocks:

* **peer memory** (GPUs, world > 1, ``torch.distributed._symmetric_memory`` available): the row slabs and receive
  buffers of all ranks are allocated symmetrically and mapped into every process; the transposing pack kernel stores
  each block straight into its destination rank's buffer (``slm_transpose_blocks_peer``), so the transposition IS the
  all-to-all -- the blocks cross NVLink while they are being transposed, nothing is staged -- and the ranks meet at a
  device-side barrier.  The four reduction numbers travel the same way.  No NCCL call inside the loop.
* **collectives** (fallback, and the CPU test-suite on gloo): pack -> ``all_to_all_single`` -> line pass -> ``all_gather``
  of four doubles -> ``all_to_all_single`` -> unpack, all ordered on the engine's stream.
"""
from __future__ import annotations

import ctypes as C
import time
from types import SimpleNamespace

import numpy as np

from . import _ffi, host_logic as hl
from .engine import Engine, _PREC, _NP_REAL, _NP_CPLX


class SlabEngine(Engine):
    """Row-slab context: ``rows`` = N / world lines of N points on this rank's device."""

    def __init__(self, n: int, world: int, rank: int, precision: str = "fp32", device=None, stream=None, group=None, peer=None):
        if n % world:
            raise ValueError("the grid size must be divisible by the number of ranks")
        self.n, self.world, self.rank, self.rows = int(n), int(world), int(rank), int(n) // int(world)
        self.precision = precision
        self.shape = (self.rows, self.n)
        self.max_batch = 1
        self.real_dtype, self.complex_dtype = _NP_REAL[precision], _NP_CPLX[precision]
        self.group = group
        self._lib = self._load_library()
        self._device_index = self._mem_init(device)
        self._stream_handle = self._mem_stream(stream)
        ctx = C.c_void_p()
        rc = self._lib.slm_rows_create(C.byref(ctx), self._device_index, self.rows, self.n, _PREC[precision], self._stream_handle)
        if rc == -2:
            raise ValueError(self._lib.slm_last_error().decode())
        _ffi.check(self._lib, rc)
        self._ctx = ctx
        self._amp_lut = hl.amplitude_lut()
        self._peer = None                     # symmetric allocation shared with the other ranks (peer-memory exchange)
        self.peer_status = "single rank" if self.world == 1 else "collectives"
        if self.world > 1 and peer is not False and self.world <= 16:
            self._peer_setup(required=bool(peer))

    # ---- peer memory (GPUs only; the CPU test-suite overrides this with a no-op) -----------------------------------
    def _peer_setup(self, required: bool):
        """One symmetric allocation per rank holding its two row slabs, its receive buffer and the gathered reduction
        numbers; every rank learns the others' base pointers (torch's symmetric memory does the mapping)."""
        try:
            torch = self._torch
            import torch.distributed as dist
            import torch.distributed._symmetric_memory as symm
            cs = np.dtype(self.complex_dtype).itemsize
            plane = self.rows * self.n * cs
            align = lambda v: (v + 1023) // 1024 * 1024       # noqa: E731
            offs, total = {}, 0
            for name, size in (("X", plane), ("Y", plane), ("Rv", plane), ("Tx", self.rows * self.n),
                               ("gathered", 2 * self.world * 32)):
                offs[name] = total
                total += align(size)
            with torch.cuda.stream(self._stream):
                buf = symm.empty((total,), dtype=torch.uint8, device=self._dev)
                group = self.group if self.group is not None else dist.group.WORLD
                hdl = symm.rendezvous(buf, group)
            ptrs = [int(p) for p in hdl.buffer_ptrs]
            if len(ptrs) != self.world:
                raise RuntimeError("symmetric memory handle does not cover the group")
            self._peer = {"buf": buf, "hdl": hdl, "ptrs": ptrs, "offs": offs}
            self.peer_status = "peer memory (torch symmetric memory over NVLink; transposing stores)"
        except Exception as exc:                  # no symmetric memory on this system: keep the collectives
            self._peer = None
            self.peer_status = f"collectives (peer memory unavailable: {type(exc).__name__}: {exc})"
            if required:
                raise

    def _peer_view(self, name, shape, dtype):
        torch = self._torch
        tdt = {np.dtype(np.complex64): torch.complex64, np.dtype(np.complex128): torch.complex128, np.dtype(np.uint8): torch.uint8,
               np.dtype(np.float64): torch.float64}[np.dtype(dtype)]
        n = int(np.prod(shape)) * np.dtype(dtype).itemsize
        off = self._peer["offs"][name]
        return self._peer["buf"][off:off + n].view(tdt).view(tuple(shape))

    def _peer_array(self, name, extra=0):
        """(void*)[world]: where `name` (+ `extra` bytes) lies in every rank's symmetric allocation"""
        off = self._peer["offs"][name] + extra
        return (C.c_void_p * self.world)(*[p + off for p in self._peer["ptrs"]])

    def _peer_barrier(self):
        with self._torch.cuda.stream(self._stream):
            self._peer["hdl"].barrier(channel=0)

    # ---- hooks the test-suite overrides together with the _mem_* ones ------------------------------------
    def _as_torch(self, buf):
        """torch view of a device buffer, as real numbers (NCCL has no complex types)."""
        torch = self._torch
        return torch.view_as_real(buf) if buf.is_complex() else buf

    def _dist(self):
        import torch.distributed as dist
        return dist

    # ---- collectives ---------------------------------------------------------------------------------------
    def _on_stream(self):
        """Collectives are ordered against torch's CURRENT stream: make that the engine's."""
        import contextlib
        torch = getattr(self, "_torch", None)
        return torch.cuda.stream(self._stream) if torch is not None and getattr(self, "_stream", None) is not None else contextlib.nullcontext()

    def _all_to_all(self, send, recv):
        if self.world == 1:
            self._copy(send, recv)
            return
        dist = self._dist()
        with self._on_stream():
            dist.all_to_all_single(self._as_torch(recv), self._as_torch(send), group=self.group)

    def _all_gather4(self, mine, gathered):
        """every rank's four reduction numbers (device double[4]) -> gathered [world][4] on every rank, rank order"""
        if self.world == 1:
            self._copy(mine, gathered[0])
            return
        dist = self._dist()
        with self._on_stream():
            dist.all_gather(list(self._as_torch(gathered).unbind(0)), self._as_torch(mine), group=self.group)

    def _all_reduce(self, values: np.ndarray, op: str) -> np.ndarray:
        if self.world == 1:
            return values
        import torch
        dist = self._dist()
        t = torch.from_numpy(np.ascontiguousarray(values, dtype=np.float64))
        if dist.get_backend(self.group) == "nccl":
            t = t.to(self._dev)
        with self._on_stream():
            dist.all_reduce(t, op=dist.ReduceOp.MAX if op == "max" else dist.ReduceOp.SUM, group=self.group)
        return t.cpu().numpy()

    def _sync(self):
        self._stream.synchronize()

    def _copy(self, src, dst):
        dst.copy_(src)

    # ---- kernels ----------------------------------------------------------------------------------------------
    def _transpose(self, src, dst, elem_bytes: int, from_exchange: bool):
        self._check(self._lib.slm_transpose_blocks(self._ctx, self._mem_ptr(src), self._mem_ptr(dst), self.rows, self.n,
                                                   elem_bytes, int(from_exchange)))

    def _exchange(self, slab, send, recv, elem_bytes, peer_name=None):
        """row slab -> exchange layout of the columns this rank owns (in ``recv``; ``peer_name``: recv is that symmetric
        buffer on every rank, so the blocks are stored straight into their destinations)."""
        if self.world == 1:
            self._transpose(slab, recv, elem_bytes, False)
            return
        if self._peer is not None and peer_name is not None:
            self._check(self._lib.slm_transpose_blocks_peer(self._ctx, self._mem_ptr(slab), self._peer_array(peer_name), self.world,
                                                            self.rank, self.rows, self.n, elem_bytes, 0))
            self._peer_barrier()                 # every block of `recv` has landed (and every rank is done with `slab`)
            return
        self._transpose(slab, send, elem_bytes, False)
        self._all_to_all(send, recv)

    def _exchange_back(self, lines, recv, slab, elem_bytes, peer_name=None):
        """exchange layout (after a pass over the owned columns) -> row slab (``peer_name``: the symmetric slab)."""
        if self.world == 1:
            self._transpose(lines, slab, elem_bytes, True)
            return
        if self._peer is not None and peer_name is not None:
            self._check(self._lib.slm_transpose_blocks_peer(self._ctx, self._mem_ptr(lines), self._peer_array(peer_name), self.world,
                                                            self.rank, self.rows, self.n, elem_bytes, 1))
            self._peer_barrier()
            return
        self._all_to_all(lines, recv)
        self._transpose(recv, slab, elem_bytes, True)

    def _rows_fft(self, src, dst, inverse, block_in=0, block_out=0, u8=None):
        lut = self._dp(self._amp_lut) if u8 is not None else None
        self._check(self._lib.slm_rows_fft(self._ctx, self._mem_ptr(src), self._mem_ptr(u8), lut, self._mem_ptr(dst),
                                           int(inverse), int(block_in), int(block_out)))

    # ---- what a GS and a GD run share ---------------------------------------------------------------------------------
    def _begin(self, target_slab, max_loops: int, want_expected: bool) -> SimpleNamespace:
        """Check this rank's uint8 target rows (host array or device buffer), take the plane's max over the ranks, exchange
        the target once into the column layout, allocate the run's buffers and reset the context's loop state."""
        if self._mem_is_device(target_slab):
            T = target_slab
            if tuple(T.shape) != self.shape or self._mem_np_dtype(T) != np.uint8:
                raise ValueError(f"target slab must be uint8 {self.shape}")
            local_max = float(self.to_host(T.max() if hasattr(T, "is_cuda") else np.asarray(T).max()))
        else:
            t = np.ascontiguousarray(target_slab)
            if t.dtype != np.uint8 or t.shape != self.shape:
                raise ValueError(f"target slab must be uint8 {self.shape}")
            T, local_max = self._mem_upload(t), float(t.max())
        norm = float(self._all_reduce(np.array([local_max]), "max")[0])
        peer = self._peer is not None
        blocks = (self.world, self.rows, self.rows)

        def buf(name, shape, dtype):                                      # the peers store into the symmetric ones
            return self._peer_view(name, shape, dtype) if peer else self._mem_empty(shape, dtype)

        r = SimpleNamespace(T=T, blocks=blocks, norm=norm, hw=float(self.n) * float(self.n), Tx=buf("Tx", blocks, np.uint8))
        self._exchange(T, None if peer else self._mem_empty(blocks, np.uint8), r.Tx, 1, "Tx")      # target columns, once
        r.X, r.Y = buf("X", self.shape, self.complex_dtype), buf("Y", self.shape, self.complex_dtype)   # row slabs
        r.S = self._mem_empty(blocks, self.complex_dtype)                 # exchange layout: lines (and the send side of the collectives)
        r.Rv = buf("Rv", blocks, self.complex_dtype)                      # receive side
        r.partial = self._mem_empty((self.rows, 4), np.float64)
        # the error curve and the ranks' sums (the rest of the loop state is the context's)
        r.curve = self._mem_empty((max_loops,), np.float64)
        r.mine = self._mem_empty((4,), np.float64)
        # (two slots used in turn: a rank may run one closing step ahead of a peer that is still reading the previous one)
        r.gathered = buf("gathered", (2, self.world, 4), np.float64)
        r.inten = self._mem_empty(blocks, np.float64) if want_expected else None
        self._slot = 0
        self._check(self._lib.slm_rows_reset(self._ctx))                 # (a finished run's flags would stop the row passes)
        return r

    def _close(self, r, kind: int, tolerance: float):
        """this rank's sums -> every rank -> the closing ``kind`` (``_ffi.CLOSE_*``) of slm_rows_close in the context's
        loop state (all on the device)"""
        peer = self._peer is not None
        slot, self._slot = self._slot, self._slot ^ 1
        self._check(self._lib.slm_rows_reduce(self._ctx, self._mem_ptr(r.partial), self.rows, self._mem_ptr(r.mine),
                                              self._peer_array("gathered", slot * self.world * 32) if peer else None,
                                              self.world if peer else 0, self.rank))
        if peer:
            self._peer_barrier()
        else:
            self._all_gather4(r.mine, r.gathered[slot])
        self._check(self._lib.slm_rows_close(self._ctx, self._mem_ptr(r.gathered[slot]), self.world, r.norm, r.hw, kind,
                                             float(tolerance), self._mem_ptr(r.curve)))

    def _state(self):
        """(scale, max, loop ended) of the context's loop state, read back"""
        scale, imax, done = C.c_double(), C.c_double(), C.c_int()
        self._check(self._lib.slm_rows_state(self._ctx, C.byref(scale), C.byref(imax), None, C.byref(done)))
        return scale.value, imax.value, done.value != 0

    def _curve(self, r, done_iters: int, tolerance: float):
        """the error curve, read back and cut where the reference stops (tolerance <= 0: the loop ran on)"""
        errors = [np.float64(e) for e in self.to_host(r.curve)[:done_iters]]
        for i, e in enumerate(errors):
            if not (e > tolerance):
                return errors[:i + 1]
        return errors

    def _expected(self, r, on_device: bool, scale: float, divisor: float = None):
        """the intensity the run kept, back in rows, times ``scale`` and then over ``divisor`` (GD: times norm, over the max,
        rounded as algorithms.py:86 rounds it); None if the run kept none"""
        if r.inten is None:
            return None
        exp_slab = self._mem_empty(self.shape, np.float64)
        if self.world == 1:
            self._transpose(r.inten, exp_slab, 8, True)
        else:
            recv_i = self._mem_empty(r.blocks, np.float64)
            self._all_to_all(r.inten, recv_i)
            self._transpose(recv_i, exp_slab, 8, True)
        if not on_device:
            exp_slab = self.to_host(exp_slab) * scale
            return exp_slab if divisor is None else exp_slab / divisor
        exp_slab *= scale
        if divisor is not None:
            exp_slab /= divisor
        return exp_slab

    # ---- Gerchberg-Saxton on the distributed plane --------------------------------------------------------------
    def gs(self, target_slab, max_loops: int, tolerance: float = 0.0, want_expected: bool = True, on_device: bool = False,
           inc_amp_slab=None):
        """``target_slab``: this rank's uint8 rows [rows, N] of the target (host array or device buffer).
        ``inc_amp_slab``: this rank's rows of the illumination amplitude (algorithms.py:14-19,30; None: uniform).
        Returns ``(hologram_slab float64 [rows, N], expected_slab or None, error_evolution list)``; the error
        curve is identical on every rank.  ``on_device`` leaves hologram / expected in device memory."""
        if max_loops < 1:
            raise UnboundLocalError("cannot access local variable 'expected_outcome' where it is not associated with a value")
        inc = self._as_device(inc_amp_slab, self.real_dtype, "inc_amp_slab")
        if inc is not None and tuple(inc.shape) != self.shape:
            raise ValueError(f"inc_amp_slab must have shape {self.shape}")
        r = self._begin(target_slab, max_loops, want_expected)
        cs = np.dtype(self.complex_dtype).itemsize
        # A = ifft2(sqrt(T))  (algorithms.py:27), unnormalised: only its phase is used.  For 8-bit targets the
        # reference computes it (and the first phasor) in complex64, so an fp64 plane borrows an fp32 engine.
        if self.precision == "fp32":
            self._setup_field(r.T, r.X, r.S, r.Rv, "Rv", "X")
            A0, field_kind = r.X, 1
        else:
            helper = type(self)(self.n, self.world, self.rank, "fp32", self._device_index, None, self.group, peer=False)
            A0 = helper._mem_empty(self.shape, np.complex64)
            helper._setup_field(r.T, A0, helper._mem_empty(r.blocks, np.complex64), helper._mem_empty(r.blocks, np.complex64))
            helper._sync()
            helper.close()
            field_kind = 2
        check_every = tolerance > 0                                           # the host must see every error to stop the loop
        src, field, done_iters = A0, field_kind, 0
        t_loop = time.perf_counter()
        for k in range(max_loops):
            cur = r.X if src is r.Y else r.Y                                  # receives the row-transformed B
            self._check(self._lib.slm_rows_gs_row_pass(self._ctx, self._mem_ptr(src), self._mem_ptr(cur), self._mem_ptr(inc), int(field), 0, None))
            self._exchange(cur, r.S, r.Rv, cs, "Rv")
            if k == 0:                                                        # exact scale of iteration 0: max pre-pass
                self._fourier(r, _ffi.RF_GS, r.Rv, self._amp_lut)
                self._close(r, _ffi.CLOSE_MAX, tolerance)
            last = k == max_loops - 1
            self._fourier(r, _ffi.RF_GS, r.Rv, self._amp_lut, r.inten if (last or check_every or k == 0) else None)
            self._close(r, _ffi.CLOSE_GS, tolerance)
            self._exchange_back(r.S, r.Rv, cur, cs, "X" if cur is r.X else "Y")   # D with the columns inverse-transformed
            src, field, done_iters = cur, 0, k + 1
            if check_every or (k == 0 and not r.norm > 0):                    # (an all-zero target ends the loop at once: 0/0, algorithms.py:29,37)
                if self._state()[2]:
                    break
        self.enqueue_s = time.perf_counter() - t_loop                        # host time to issue the loop (measurements: is the host the bound?)
        errors = self._curve(r, done_iters, tolerance)
        holo = self._mem_empty(self.shape, np.float64)
        self._check(self._lib.slm_rows_gs_row_pass(self._ctx, self._mem_ptr(src), None, None, 0, 1, self._mem_ptr(holo)))
        expected = self._expected(r, on_device, self._state()[0])            # expected_outcome *= norm / max, :37
        return (holo if on_device else self.to_host(holo)), expected, errors

    # ---- gradient descent on the distributed plane (algorithms.py:60-112) ------------------------------------------------
    def gd(self, target_slab, x0_slab, lr_schedule, max_loops: int, tolerance: float = 0.0, white_attention=1,
           want_expected: bool = True, on_device: bool = False):
        """``target_slab``: this rank's uint8 rows [rows, N] (host array or device buffer); ``x0_slab``: this rank's rows of the complex initial guess
        (host array; make_initial_guess draws the plane row-major, so rank p's rows are a contiguous part of the stream).
        Returns ``(hologram_slab, expected_slab or None, error_evolution)`` like :meth:`gs`.  Same exchange as GS (stores into
        peer memory or collectives), two Fourier-plane passes per iteration: the plane's max is needed before the gradient
        (algorithms.py:86), and here it lives on several devices."""
        if max_loops < 1:
            raise UnboundLocalError("cannot access local variable 'output' where it is not associated with a value")
        x_on_device = self._mem_is_device(x0_slab)
        x0 = x0_slab if x_on_device else np.asarray(x0_slab)
        if tuple(x0.shape) != self.shape or (x_on_device and not str(x0.dtype).endswith(np.dtype(self.complex_dtype).name)):
            raise ValueError(f"x0 slab must have shape {self.shape} (a device buffer: in the engine's complex type)")
        lr = np.ascontiguousarray(lr_schedule, dtype=np.float64)
        if lr.shape != (max_loops,):
            raise ValueError("lr_schedule must have max_loops entries")
        r = self._begin(target_slab, max_loops, want_expected)
        cs = np.dtype(self.complex_dtype).itemsize
        if x_on_device:                                                   # (the row pass updates x in place: work on a copy)
            x = self._mem_empty(self.shape, self.complex_dtype)
            self._copy(x0, x)
        else:
            x = self._mem_upload(x0.astype(self.complex_dtype))
        lr_dev = self._mem_upload(lr)
        mask_lut = hl.gd_mask_lut(white_attention)
        check_every = tolerance > 0
        done_iters = 0
        for k in range(max_loops):
            # SLM-plane pass: the update of the previous iteration (none yet at k = 0), x/|x|, rows of fft2
            self._check(self._lib.slm_rows_gd_row_pass(self._ctx, self._mem_ptr(r.Y), self._mem_ptr(x), self._mem_ptr(r.X), self._mem_ptr(lr_dev),
                                                       int(k == 0), 0, None))
            self._exchange(r.X, r.S, r.Rv, cs, "Rv")
            # the plane's max (the transform is kept in S), then the gradient step on it
            self._fourier(r, _ffi.RF_GD_MAX, r.Rv)
            self._close(r, _ffi.CLOSE_MAX, tolerance)
            last = k == max_loops - 1
            self._fourier(r, _ffi.RF_GD_POST, r.S, mask_lut, r.inten if (last or check_every or k == 0) else None)
            self._close(r, _ffi.CLOSE_GD, tolerance)
            self._exchange_back(r.S, r.Rv, r.Y, cs, "Y")
            done_iters = k + 1
            if check_every or (k == 0 and not r.norm > 0):
                if self._state()[2]:
                    break
        errors = self._curve(r, done_iters, tolerance)
        holo = self._mem_empty(self.shape, np.float64)
        self._check(self._lib.slm_rows_gd_row_pass(self._ctx, self._mem_ptr(r.Y), self._mem_ptr(x), None, self._mem_ptr(lr_dev), 0, 1,
                                                   self._mem_ptr(holo)))
        expected = self._expected(r, on_device, r.norm, self._state()[1])  # output_unnormed * norm / amax, algorithms.py:86
        return (holo if on_device else self.to_host(holo)), expected, errors

    def _setup_field(self, T, X, S, Rv, peer_recv=None, peer_slab=None):
        """A = ifft2(amplitude) of the distributed target into the row slab X (this engine's precision)."""
        h, cs = self.rows, np.dtype(self.complex_dtype).itemsize
        self._rows_fft(None, X, True, u8=T)
        self._exchange(X, S, Rv, cs, peer_recv)
        self._rows_fft(Rv, S, True, block_in=h, block_out=h)
        self._exchange_back(S, Rv, X, cs, peer_slab)

    def _fourier(self, r, mode, src, lut=None, inten=None):
        """Fourier-plane pass ``mode`` (``_ffi.RF_*``) over the received lines ``src`` into r.S (``lut``: the target's
        table by grey level, GS amplitude or GD mask)"""
        self._check(self._lib.slm_rows_fourier_pass(self._ctx, mode, self._mem_ptr(src), self._mem_ptr(r.S), self.rows,
                                                    self._mem_ptr(r.Tx), None if lut is None else self._dp(lut), r.norm,
                                                    self._mem_ptr(r.partial), self._mem_ptr(inten)))

    def close(self):
        self._peer = None                     # (releases this rank's symmetric allocation)
        super().close()


def _world_rank():
    """(world size, rank) of the default process group; (1, 0) without one."""
    try:
        import torch.distributed as dist
        return (dist.get_world_size(), dist.get_rank()) if dist.is_available() and dist.is_initialized() else (1, 0)
    except Exception:
        return 1, 0


def gerchberg_saxton_slab(target, max_loops: int, tolerance: float = 0.0, precision: str = "fp32", want_expected: bool = True,
                          engine_factory=None):
    """GS hologram of one large square uint8 ``target`` (every rank passes the same array, or only its
    own rows via ``target[lo:hi]`` semantics handled here) on all ranks of the default process group.
    Returns this rank's row slab of (hologram, expected) and the error curve."""
    world, rank = _world_rank()
    target = np.asarray(target)
    n = target.shape[1]
    lo, hi = rank * (n // world), (rank + 1) * (n // world)
    slab = target[lo:hi] if target.shape[0] == n else target
    eng = (engine_factory or SlabEngine)(n, world, rank, precision)
    try:
        return eng.gs(slab, max_loops, tolerance, want_expected)
    finally:
        eng.close()


def gradient_descent_slab(target, max_loops: int, learning_rate: float = 0.005, unsettle: int = 0, tolerance: float = 0.0,
                          white_attention=1, initial_guess: str = "random", random_seed: int = 42, precision: str = "fp32",
                          want_expected: bool = True, engine_factory=None):
    """GD hologram (algorithms.py:60-112) of one large square uint8 ``target`` on all ranks of the default process group;
    the arguments are the reference's ``args`` fields of the same names.  ``initial_guess``: the random families of make_initial_guess
    (algorithms.py:115-153; the MT19937 stream is drawn row-major for the whole plane, every rank keeps its own rows) --
    "fourier" is not offered here.  Returns this rank's row slab of (hologram, expected), the error curve and the learning rate the
    reference would leave in ``args.learning_rate``."""
    world, rank = _world_rank()
    target = np.asarray(target)
    n = target.shape[1]
    lo, hi = rank * (n // world), (rank + 1) * (n // world)
    if target.shape[0] != n:
        raise ValueError("gradient_descent_slab takes the whole plane (the initial guess is drawn for all of it)")
    if initial_guess == "fourier":
        raise ValueError('initial_guess "fourier" is not available on the slab path')
    during, after = hl.learning_rate_schedule(learning_rate, unsettle, int(max_loops))
    eng = (engine_factory or SlabEngine)(n, world, rank, precision)
    try:
        if initial_guess in ("random", "zeros"):
            # the MT19937 stream continued on the device (Engine.python_random_uniform); every rank draws the whole plane's
            # stream -- the last rank needs all of it anyway, and Python's generator is then left where the reference's
            # per-pixel loop leaves it (algorithms.py:117-124) on every rank -- and keeps its own rows
            u = eng.python_random_uniform(random_seed, (n, n))
            x0 = eng._mem_empty(eng.shape, eng.complex_dtype)
            eng._check(eng._lib.slm_random_phasor(eng._ctx, eng._mem_ptr(u[lo:hi]), eng._mem_ptr(x0), (hi - lo) * n,
                                                  100.0 if initial_guess == "zeros" else 1.0))
            del u
        else:
            x0 = hl.host_initial_guess(initial_guess, (n, n), random_seed)[lo:hi]
        h, e, errs = eng.gd(target[lo:hi], x0, during, int(max_loops), float(tolerance), white_attention, want_expected)
        return h, e, errs, after[len(errs)]
    finally:
        eng.close()
