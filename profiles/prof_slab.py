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
for mode in ("copy", "store", "peer1", "coll"):
    for k in ("SLM_SLAB_NO_PEER", "SLM_SLAB_PARTS", "SLM_SLAB_EXCHANGE"):
        os.environ.pop(k, None)
    os.environ.update({"copy": {"SLM_SLAB_PARTS": "4"}, "store": {"SLM_SLAB_PARTS": "4", "SLM_SLAB_EXCHANGE": "store"}, "peer1": {}, "coll": {"SLM_SLAB_NO_PEER": "1"}}[mode])
    eng = SlabEngine(n, world, rank, "fp32")
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
    if peer and getattr(eng, "_how", "") == "copy":
        B = eng._peer["comm_stream"]
        part = rows // eng._parts
        for rows_part, name in ((True, "copy engines, way out (strided runs)"), (False, "copy engines, way back (contiguous)")):
            torch.cuda.synchronize(); dist.barrier()
            e0.record(B)
            for _ in range(5):
                for j in range(eng._parts):
                    eng._copy_blocks(S, "Rv" if rows_part else "Rb", j * part, part, cs, rows_part)
            e1.record(B); torch.cuda.synchronize()
            if rank == 0: print(f"    {name}: {e0.elapsed_time(e1)/5:.3f} ms per exchange ({rows*n*cs*(world-1)/world/1e6/(e0.elapsed_time(e1)/5)*1e-3*1e3:.0f} GB/s to the peers)")
        # the passes alone (engine stream), then passes + copies together
        Tx = eng._peer_view("Tx", (world, rows, rows), np.uint8)
        state = eng._mem_upload(np.array([1.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0])); partial = eng._mem_empty((rows, 4), np.float64)
        Y = eng._peer_view("Y", eng.shape, np.complex64)
        torch.cuda.synchronize(); dist.barrier()
        e0.record()
        for _ in range(5):
            for j in range(eng._parts):
                eng._check(eng._lib.slm_rows_gs_row_pass_part(eng._ctx, eng._mem_ptr(X), eng._mem_ptr(Y), 0, j * part, part))
            for j in range(eng._parts):
                eng._fourier(Rv, S, Tx, state, partial, None, j * part, part)
        e1.record(); torch.cuda.synchronize()
        if rank == 0: print(f"    the two passes alone: {e0.elapsed_time(e1)/5:.3f} ms per iteration")
        torch.cuda.synchronize(); dist.barrier()
        e0.record()
        for _ in range(5):
            for j in range(eng._parts):
                eng._check(eng._lib.slm_rows_gs_row_pass_part(eng._ctx, eng._mem_ptr(X), eng._mem_ptr(Y), 0, j * part, part))
                eng._copy_blocks(S, "Rv", j * part, part, cs, True)
            for j in range(eng._parts):
                eng._fourier(Rv, S, Tx, state, partial, None, j * part, part)
                eng._copy_blocks(S, "Rb", j * part, part, cs, False)
        e1.record(); eng._after(eng._stream, B); e1.record(); torch.cuda.synchronize()
        if rank == 0: print(f"    passes + unordered copies on the second stream: {e0.elapsed_time(e1)/5:.3f} ms per iteration")
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
