"""torchrun --nproc-per-node N profiles/prof_slab.py [n]: per-phase device times of one slab GS iteration."""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch, torch.distributed as dist
rank, local, world = int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
torch.cuda.set_device(local)
if world > 1:
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
from spatial_light_modulator_module_b200.slab import SlabEngine
n = int(sys.argv[1]) if len(sys.argv) > 1 else 16384
for mode in ("peer", "coll"):
    eng = SlabEngine(n, world, rank, "fp32", peer=None if mode == "peer" else False)
    rows = n // world
    slab = eng._mem_upload((np.random.default_rng(100 + rank).random((rows, n)) * 255).astype(np.uint8))
    eng.gs(slab, 2, want_expected=False, on_device=True)
    torch.cuda.synchronize()
    if world > 1: dist.barrier()
    t0 = time.perf_counter()
    eng.gs(slab, 10, want_expected=False, on_device=True)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    eng.profile(True); eng.profile_read()
    eng.gs(slab, 10, want_expected=False, on_device=True)
    prof = eng.profile_read(); eng.profile(False)
    if rank == 0:
        print(f"[{mode}] {eng.peer_status}: 10 iterations + setup in {dt*1e3:.1f} ms")
        for k, (ms, cnt) in prof.items():
            if cnt: print(f"    {k:12s} {cnt:4d} launches  {ms:8.2f} ms total  {ms/cnt:7.3f} ms each")
    # the exchange alone
    peer = eng._peer is not None
    cs = 8
    X = eng._peer_view("X", eng.shape, np.complex64) if peer else eng._mem_empty(eng.shape, np.complex64)
    S = eng._mem_empty((world, rows, rows), np.complex64)
    Rv = eng._peer_view("Rv", (world, rows, rows), np.complex64) if peer else eng._mem_empty((world, rows, rows), np.complex64)
    for _ in range(2): eng._exchange(X, S, Rv, cs, "Rv")
    torch.cuda.synchronize()
    if world > 1: dist.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(10): eng._exchange(X, S, Rv, cs, "Rv")
    e1.record(); torch.cuda.synchronize()
    if rank == 0: print(f"    exchange (pack + all-to-all / peer stores + barrier): {e0.elapsed_time(e1)/10:.3f} ms each, {rows*n*cs*(world-1)/world/1e6:.0f} MB sent per rank")
    e0.record()
    for _ in range(10): eng._exchange_back(S, Rv, X, cs, "X")
    e1.record(); torch.cuda.synchronize()
    if rank == 0: print(f"    exchange back: {e0.elapsed_time(e1)/10:.3f} ms each")
    if peer:
        e0.record()
        for _ in range(20): eng._peer_barrier()
        e1.record(); torch.cuda.synchronize()
        if rank == 0: print(f"    device barrier: {e0.elapsed_time(e1)/20*1e3:.1f} us each")
    eng.close()
    del slab, X, S, Rv
    torch.cuda.empty_cache()
if world > 1:
    dist.barrier(); dist.destroy_process_group()
