"""Optical-trap movies: a sequence of target frames -> a sequence of GS holograms
(reference: ``generate_hologram_sequence.py:10-32``).

Frames are independent (the reference's loop carries no state from frame to frame), so they are
processed in device batches and, under ``torch.distributed``, split into contiguous blocks over
the ranks (one process per GPU) with no collective on the data path; only the finished holograms
are gathered.
"""
from __future__ import annotations

import os
from typing import Callable, List, Optional

import numpy as np

from . import host_logic as hl


def _dist():
    try:
        import torch.distributed as dist
        if dist.is_available() and dist.is_initialized():
            return dist
    except Exception:
        pass
    return None


def sequence_holograms(frames, max_loops: int, tolerance: float = 0.0, precision: str = "fp32",
                       batch: Optional[int] = None, want_expected: bool = False, engine_factory: Optional[Callable] = None,
                       gather: bool = True, inc_amp=None, warm_start: bool = False, output: str = "float64",
                       mask=None, ct2pi=256, trap_dots=None, on_batch: Optional[Callable] = None,
                       weighted: bool = False, weight_limit: float = 10.0):
    """GS holograms of ``frames`` (uint8 [F,H,W], a host array or a device tensor); ``inc_amp``: illumination amplitude
    plane [H,W] shared by all frames (algorithms.py:14-19), None = uniform.

    ``weighted``: weighted GS (Engine.gsw, weights bounded by ``weight_limit``) instead of GS, for trap intensities
    that follow the frames' grey levels.  Every frame's weights start at 1 (``warm_start`` carries only the phase).

    ``output``: "float64" -- the holograms as the reference saves them (generate_hologram_sequence.py:26, 8 bytes per
    pixel); "uint8" -- the frames the SLM is shown: wavefront-correction ``mask`` added (None: no mask) and quantised
    with ``ct2pi`` grey levels per 2 pi by the floor rule of move_traps.py:135-140 / display_holograms.py:253-266
    (1 byte per pixel: an eighth of the read-back and of the gather).

    ``trap_dots`` = (dots int[n,3] of (frame, y, x), number_of_frames, (H, W)) instead of ``frames``: the trap targets
    are rasterised on the device (traps_images.py:10-16,87-91) -- no frame stack crosses the host at all.

    ``warm_start`` (an extension, off by default because it changes the results): every frame of a rank's block
    starts from the previous frame's hologram (``B = inc * exp(1j * hologram)``) instead of the reference's
    ``ifft2(sqrt(target))`` setup, which lets a slowly moving trap pattern converge in a few iterations; the frames
    are then processed one after the other.

    ``on_batch(lo, hi, holograms, expected)`` is called from a writer thread as soon as global frames [lo, hi) lie in
    host memory (this rank's own frames; with a gather, rank 0 receives every rank's), while later batches iterate.

    Under an initialised process group every rank passes the SAME ``frames`` and computes only its contiguous block.
    With ``gather`` the full movie is returned on rank 0 (other ranks return their own block's error curves and empty
    arrays).  ``gather=True`` picks the way: all ranks on ONE node (and no ``on_batch``) -- rank 0's result arrays lie
    in shared host memory which every rank maps, page-locks and reads its own frames back into, each over its own
    PCIe link (``shared_host.py``; "host"); otherwise, or as ``gather="device"``, the finished frames travel device to
    device to rank 0 (``torch.distributed.gather`` per batch: NCCL over NVLink on GPUs), which alone reads them back.
    Either way batch k is read back while batch k+1 iterates.
    Returns ``(holograms [n,H,W] float64 | uint8, expected or None, errors list, (lo, hi))``.
    """
    if output not in ("float64", "uint8"):
        raise ValueError("output must be 'float64' or 'uint8'")
    dist = _dist()
    rank, world = (dist.get_rank(), dist.get_world_size()) if dist else (0, 1)
    if trap_dots is not None:
        dots, n_frames, shape = trap_dots
        dots = np.asarray(dots, dtype=np.int64).reshape(-1, 3)
        shape = tuple(int(v) for v in shape)
        frames = None
    else:
        if not hasattr(frames, "data_ptr"):
            frames = np.asarray(frames)
        if len(frames.shape) != 3:
            raise ValueError("frames must be [F,H,W]")
        n_frames, shape = int(frames.shape[0]), tuple(int(v) for v in frames.shape[1:])
    lo, hi = hl.shard_range(n_frames, rank, world)
    n_local = hi - lo
    blocks = [hl.shard_range(n_frames, r, world) for r in range(world)]
    n_max = max(h - l for l, h in blocks)
    if batch is None:
        # 64 frames per launch sequence are 5 % faster than 32, but a rank wants at least four batches so that the gather
        # and the read-back of one batch hide behind the iterations of the next
        batch = min(64, max(16, n_max // 4))
    batch = max(1, min(int(batch), max(n_max, 1)))
    if engine_factory is None:
        from .engine import get_engine
        eng = get_engine(shape, precision, batch)
    else:
        eng = engine_factory(shape, precision, batch)
    out_dtype = np.float64 if output == "float64" else np.uint8
    if gather not in (True, False, "host", "device"):
        raise ValueError("gather must be True, False, 'host' or 'device'")
    collect = bool(dist and world > 1 and gather)
    root = rank == 0
    shared = None                                         # the result arrays in host memory shared by the ranks of one node
    if collect and warm_start:
        raise ValueError("warm_start chains the frames of a block: gather=False only")
    if collect and gather != "device" and on_batch is None and n_frames > 0:
        from . import shared_host
        want = os.environ.get("SLM_GATHER", "host" if gather == "host" or shared_host.same_node(dist) else "device")
        if want == "host":
            specs = [((n_frames,) + shape, out_dtype)] + ([((n_frames,) + shape, np.float64)] if want_expected else [])
            shared = shared_host.shared_results(dist, specs, (lo, hi))
    n_host = n_frames if (collect and root) else (0 if collect else n_local)
    base = 0 if collect else lo                           # global index of holos[0]
    if shared is not None:
        holos, exps = shared[0], (shared[1] if want_expected else None)
    else:
        holos = eng.host_empty((n_host,) + shape, out_dtype)
        exps = eng.host_empty((n_host,) + shape, np.float64) if want_expected else None
    errors: List[np.ndarray] = []
    writer = _Writer(on_batch)

    def run(targets, phasor0=None):
        if weighted:
            return eng.gsw(targets, max_loops, tolerance, inc_amp=inc_amp, phasor0=phasor0, weight_limit=weight_limit,
                           want_expected=want_expected)[0]
        return eng.gs(targets, max_loops, tolerance, inc_amp=inc_amp, phasor0=phasor0, want_expected=want_expected)

    def finish(res):
        """device results of one batch in the requested output format"""
        if output == "float64":
            return res.hologram
        from . import _ffi
        return eng.quantize(res.hologram, mask, ct2pi, _ffi.QUANT_FLOOR)

    def targets_of(s, e):
        """this rank's frames [s, e) on the device (host frames: the copy is started here and not waited for)"""
        if e <= s:
            return None
        if frames is not None:
            block = frames[lo + s:lo + e]
            return block if hasattr(block, "data_ptr") else eng.upload(block)
        sel = dots[(dots[:, 0] >= lo + s) & (dots[:, 0] < lo + e)].copy()
        sel[:, 0] -= lo + s
        return eng.trap_frames(sel, e - s, shape)

    if warm_start:
        if collect:
            raise ValueError("warm_start chains the frames of a block: gather=False only")
        phasor = None
        for s in range(n_local):
            res = run(targets_of(s, s + 1), phasor0=phasor)
            holos[s] = eng.to_host(finish(res))[0]
            if want_expected:
                exps[s] = eng.to_host(res.expected)[0]
            errors.extend(res.errors)
            phasor = eng.phase_phasor(res.hologram, inc_amp)
            writer.put([], lo + s, lo + s + 1, holos[s:s + 1], exps[s:s + 1] if want_expected else None)
        n_local = n_max = 0                              # nothing left for the batched loop below
    # the read-back (and the gather) of one batch runs beside the iterations of the next one
    pending: list = []
    ahead = targets_of(0, min(batch, n_local))
    for s in range(0, n_max, batch):
        e = min(s + batch, n_local)
        res, cur = None, ahead
        ahead = targets_of(s + batch, min(s + 2 * batch, n_local))        # the next batch's frames travel beside this batch's iterations
        if e > s:
            res = run(cur)
            errors.extend(res.errors)
        for jobs, a, b in pending:
            writer.put(jobs, a, b, holos[a - base:b - base], exps[a - base:b - base] if want_expected else None)
        pending = []
        if not collect or shared is not None:
            off = lo if shared is not None else 0         # (shared arrays hold the whole movie: this rank fills its own rows)
            if e > s:
                jobs = [eng.to_host_into(finish(res), holos[off + s:off + e])]
                if want_expected:
                    jobs.append(eng.to_host_into(res.expected, exps[off + s:off + e]))
                pending.append((jobs, lo + s, lo + e))
            continue
        # gather this batch of every rank on rank 0's device; rank 0 reads the blocks back
        parts = [(finish(res) if res is not None else None, holos)]
        if want_expected:
            parts.append((res.expected if res is not None else None, exps))
        by_block = {}
        for dev_buf, host in parts:
            got = eng.gather_to_root(dev_buf, (batch,) + shape, host.dtype, dist)
            if not root:
                continue
            for r, (rl, rh) in enumerate(blocks):
                a, b = rl + s, min(rl + s + batch, rh)
                if b > a:
                    by_block.setdefault((a, b), []).append(eng.to_host_into(got.blocks[r][:b - a], host[a:b], after=got.work))
        pending = [(jobs, a, b) for (a, b), jobs in by_block.items()]
    for jobs, a, b in pending:
        writer.put(jobs, a, b, holos[a - base:b - base], exps[a - base:b - base] if want_expected else None)
    writer.close()                                        # (every copy of this rank has landed)
    if collect:
        errors = _gather_curves(dist, n_frames, errors, max_loops)      # also the point where rank 0 knows the others are done
        if root:
            lo, hi = 0, n_frames
        elif shared is not None:                          # like the device gather: only rank 0 holds the movie
            holos = np.empty((0,) + shape, out_dtype)
            exps = np.empty((0,) + shape, np.float64) if want_expected else None
    return holos, exps, errors, (lo, hi)


class _Writer:
    """Hands finished batches to ``on_batch`` from one background thread, in order, after their copies have landed
    (file output of batch k overlaps the iterations of batch k+1).  Without a callback it only joins the copies."""

    def __init__(self, on_batch):
        import queue
        import threading
        self.on_batch, self.error = on_batch, None
        self.q = queue.Queue() if on_batch else None
        self.thread = None
        if on_batch:
            self.thread = threading.Thread(target=self._run, daemon=True)
            self.thread.start()

    def put(self, jobs, lo, hi, holos, exps):
        if self.q is None:
            for j in jobs:
                j.join()
            return
        self.q.put((jobs, lo, hi, holos, exps))

    def _run(self):
        while True:
            item = self.q.get()
            if item is None:
                return
            jobs, lo, hi, holos, exps = item
            try:
                for j in jobs:
                    j.join()
                if self.error is None:
                    self.on_batch(lo, hi, holos, exps)
            except Exception as exc:                  # surfaced by close()
                self.error = exc

    def close(self):
        if self.q is not None:
            self.q.put(None)
            self.thread.join()
        if self.error is not None:
            raise self.error


def _gather_curves(dist, n_total, errors, max_loops):
    """The error curves of every rank's block on rank 0 (a few doubles per frame; the other ranks keep their own)."""
    import torch
    rank, world = dist.get_rank(), dist.get_world_size()
    dev = torch.device("cuda", torch.cuda.current_device()) if dist.get_backend() == "nccl" else torch.device("cpu")
    counts = [hl.shard_range(n_total, r, world) for r in range(world)]
    cap = max(h - l for l, h in counts)
    curves = np.full((cap, max_loops + 1), np.nan)
    for i, e in enumerate(errors):
        curves[i, 0] = len(e)
        curves[i, 1:1 + len(e)] = e
    mine = torch.from_numpy(curves).to(dev)
    bufs = [torch.empty_like(mine) for _ in range(world)] if rank == 0 else None
    dist.gather(mine, bufs, dst=0)
    if rank != 0:
        return errors
    rows = np.concatenate([bufs[r][:h - l].cpu().numpy() for r, (l, h) in enumerate(counts)], axis=0)
    return [row[1:1 + int(row[0])].copy() for row in rows]


def generate_hologram_sequence(args):
    """Drop-in for the reference driver (generate_hologram_sequence.py:10-32): reads
    ``images/moving_traps/<source_dir>/<i>.png``, writes ``<i>.npy`` holograms (and preview PNGs) -- from a writer
    thread, batch by batch, while the following batches iterate on the device.  Optional ``args.batch`` /
    ``args.precision`` tune the engine.  Under an initialised process group every rank computes and writes its own
    block of frames (no gather: the files are the result)."""
    from PIL import Image as im
    dest_dir_holograms = f"holograms/{args.source_dir}_{args.version}_holograms"
    dest_dir_preview = f"images/moving_traps/{args.source_dir}_{args.version}_preview"
    for dest_dir in [dest_dir_holograms, dest_dir_preview]:
        if not os.path.exists(dest_dir):
            os.makedirs(dest_dir, exist_ok=True)
    source_dir_path = f"images/moving_traps/{args.source_dir}"
    files = os.listdir(source_dir_path)
    frames = np.stack([np.array(im.open(f"{source_dir_path}/{i}.png")) for i in range(len(files))])
    if frames.dtype != np.uint8 or frames.ndim != 3:
        raise ValueError("trap frames must be single-channel 8-bit images")
    inc = None
    if getattr(args, "incomming_intensity", "uniform") != "uniform":
        from .algorithms import _illumination
        inc = _illumination(args, frames.shape[1:])
    from .display_holograms import preview_to_grey

    def write(lo, hi, holos, exps):
        for k in range(hi - lo):
            i = lo + k
            print(f"\rcreating {i}. hologram ", end="")
            np.save(f"{dest_dir_holograms}/{i}.npy", holos[k])
            if args.preview:
                im.fromarray(preview_to_grey(exps[k])).save(f"{dest_dir_preview}/{i}.png")

    _, _, errors, _ = sequence_holograms(
        frames, int(args.max_loops), float(args.tolerance), getattr(args, "precision", None) or
        os.environ.get("SLM_PRECISION", "fp32"), getattr(args, "batch", None), bool(args.preview), gather=False,
        inc_amp=inc, on_batch=write, weighted=bool(getattr(args, "weighted", False)),
        weight_limit=float(getattr(args, "weight_limit", 10.0)))
    plot_error_evolution([list(e) for e in errors])
    return errors


def plot_error_evolution(err_evl_list):
    """reference: generate_hologram_sequence.py:35-40 (skipped silently when matplotlib is absent)."""
    try:
        import matplotlib.pyplot as plt
    except Exception:
        return
    for i, err_evl in enumerate(err_evl_list):
        plt.plot(err_evl, label=i)
    plt.legend()
    plt.show()


def build_parser():
    """The reference's command line (generate_hologram_sequence.py:43-103): same arguments and defaults;
    ``--batch`` and ``--precision`` are additions."""
    import argparse
    p = argparse.ArgumentParser(formatter_class=argparse.ArgumentDefaultsHelpFormatter,
                                description="Holograms of a sequence of trap images (images/moving_traps/<source_dir>/<i>.png) "
                                            "-> holograms/<source_dir>_<version>_holograms/<i>.npy, computed in batches on a B200.")
    p.add_argument("source_dir", type=str, help="directory with the trap images, inside images/moving_traps")
    p.add_argument("-v", "--version", type=str, help="tag appended to the output directory names")
    p.add_argument("-ii", "--incomming_intensity", metavar="PATH", type=str, default="uniform", help="illumination image path, or 'uniform'")
    p.add_argument("-ct2pi", "--correspond_to2pi", metavar="INT", required=True, type=int, help="grey level that corresponds to a 2 pi phase shift")
    p.add_argument("-tol", "--tolerance", metavar="FLOAT", default=0, type=float, help="stop when the error falls to this value")
    p.add_argument("-loops", "--max_loops", metavar="INT", default=5, type=int, help="upper bound on the number of iterations")
    p.add_argument("-p", "--preview", action="store_true", help="also write the expected images of the holograms")
    p.add_argument("--batch", type=int, default=None, help="frames per device batch (default: chosen from the number of frames)")
    p.add_argument("--precision", default=None, choices=["fp32", "fp64"], help="engine arithmetic (default fp32)")
    p.add_argument("--weighted", action="store_true", help="weighted Gerchberg-Saxton: even trap intensities")
    p.add_argument("--weight_limit", default=10.0, type=float, metavar="FLOAT",
                   help="weighted GS: the weights stay within [1/limit, limit] (>= 1)")
    return p


def cli(argv=None):
    args = build_parser().parse_args(argv)
    args.gif = False                       # generate_hologram_sequence.py:105-107
    args.plot_error = False
    args.print_info = False
    generate_hologram_sequence(args)


if __name__ == "__main__":
    cli()
