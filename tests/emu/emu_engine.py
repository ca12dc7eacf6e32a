"""TEST INFRASTRUCTURE ONLY: drive the host emulation of the kernel sources (libslmholo_emu.so)
through the package's own Engine class, with numpy arrays standing in for device buffers.

Used by the CPU test-suite to check the kernels' logic against the oracle without a GPU.  The
package never imports this module and never loads the emulation library.
"""
from __future__ import annotations

import ctypes as C

import numpy as np

from spatial_light_modulator_module_b200 import _ffi
from spatial_light_modulator_module_b200.engine import Engine

from . import build_emu

_LIB = None


def emu_library():
    global _LIB
    if _LIB is None:
        _LIB = _ffi.declare(C.CDLL(build_emu.build()))
    return _LIB


class HostBuf(np.ndarray):
    """numpy array with the two tensor methods Engine uses on device buffers."""

    def data_ptr(self):
        return self.ctypes.data

    def dim(self):
        return self.ndim


class EmuEngine(Engine):
    def _load_library(self):
        return emu_library()

    def _mem_init(self, device):
        return 0

    def _mem_stream(self, stream):
        return C.c_void_p(0)

    def _mem_empty(self, shape, dtype):
        return np.full(tuple(shape), 0xFF, dtype=np.uint8).repeat(np.dtype(dtype).itemsize).view(dtype).reshape(shape).view(HostBuf) \
            if False else np.empty(tuple(shape), dtype=dtype).view(HostBuf)

    def _mem_upload(self, array):
        return np.array(array, copy=True, order="C").view(HostBuf)

    def _mem_is_device(self, obj):
        return isinstance(obj, HostBuf)

    def _mem_download(self, buf):
        return np.asarray(buf).copy()

    def _mem_plane_max(self, dev):
        a = np.asarray(dev)
        return a.reshape(a.shape[0], -1).max(axis=1).astype(np.float64)

    def _mem_plane_sum(self, dev):
        a = np.asarray(dev)
        return a.reshape(a.shape[0], -1).sum(axis=1, dtype=np.float64)

    def _mem_fill(self, buf, value):
        np.asarray(buf).fill(value)

    def _mem_contiguous(self, dev):
        return np.ascontiguousarray(dev).view(HostBuf)

    def _mem_repeat(self, plane, n):
        return np.repeat(np.asarray(plane), n, axis=0).view(HostBuf)

    def _mem_host_empty(self, shape, dtype):
        return np.empty(shape, dtype=dtype)

    def _mem_gather_to_root(self, buf, padded_shape, dtype, dist, dst):
        import torch
        from spatial_light_modulator_module_b200.engine import _Gathered
        pad = np.zeros(padded_shape, dtype=dtype)
        if buf is not None:
            pad[:buf.shape[0]] = np.asarray(buf)
        mine = torch.from_numpy(pad)
        bufs = [torch.empty_like(mine) for _ in range(dist.get_world_size())] if dist.get_rank() == dst else None
        work = dist.gather(mine, bufs, dst=dst, async_op=True)
        blocks = [b.numpy().view(HostBuf) for b in bufs] if bufs is not None else None
        return _Gathered(blocks, work, mine)

    def _mem_download_into(self, buf, out, after=None):
        if after is not None:
            after.wait()
        np.copyto(out, np.asarray(buf))

        class Done:
            def join(self):
                pass
        return Done()

    def _mem_download_many(self, bufs):
        return [self._mem_download(b) for b in bufs]

    def _mem_np_dtype(self, buf):
        return buf.dtype


from spatial_light_modulator_module_b200.slab import SlabEngine  # noqa: E402


class EmuSlabEngine(EmuEngine, SlabEngine):
    """Row-slab engine over the host emulation; torch CPU tensors (gloo) view the numpy buffers."""

    def _as_torch(self, buf):
        import torch
        t = torch.from_numpy(np.asarray(buf))
        return torch.view_as_real(t) if t.is_complex() else t

    def _sync(self):
        pass

    def _copy(self, src, dst):
        np.copyto(np.asarray(dst), np.asarray(src))
