"""torchrun --nproc-per-node N profiles/prof_slab_gd.py [n]: per-kernel device times of slab GD iterations."""
import os, sys, time
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch, torch.distributed as dist
rank, local, world = int(os.environ.get("RANK", 0)), int(os.environ.get("LOCAL_RANK", 0)), int(os.environ.get("WORLD_SIZE", 1))
torch.cuda.set_device(local)
if world > 1:
    dist.init_process_group("nccl", device_id=torch.device("cuda", local))
from spatial_light_modulator_module_b200 import host_logic as hl
from spatial_light_modulator_module_b200.slab import SlabEngine
n = int(sys.argv[1]) if len(sys.argv) > 1 else 16384
for mode in ("peer", "coll"):
    eng = SlabEngine(n, world, rank, "fp32", peer=None if mode == "peer" else False)
    rows = n // world
    slab = eng._mem_upload((np.random.default_rng(100 + rank).random((rows, n)) * 255).astype(np.uint8))
    u = eng._mem_upload(np.random.default_rng(200 + rank).random((rows, n)))
    x0 = eng._mem_empty((rows, n), eng.complex_dtype)
    eng._check(eng._lib.slm_random_phasor(eng._ctx, eng._mem_ptr(u), eng._mem_ptr(x0), rows * n, 1.0))
    del u
    run = lambda k: eng.gd(slab, x0, hl.learning_rate_schedule(0.005, 0, k)[0], k, want_expected=False, on_device=True)
    run(2)
    torch.cuda.synchronize()
    for loops in (2, 12, 20, 20):
        if world > 1: dist.barrier()
        t0 = time.perf_counter()
        run(loops)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if rank == 0: print(f"[{mode}] {eng.peer_status}: {loops} iterations + setup in {dt*1e3:.1f} ms")
    eng.profile(True); eng.profile_read()
    run(10)
    prof = eng.profile_read(); eng.profile(False)
    if rank == 0:
        for k, (ms, cnt) in prof.items():
            if cnt: print(f"    {k:12s} {cnt:4d} launches  {ms:8.2f} ms total  {ms/cnt:7.3f} ms each")
    eng.close()
    del slab, x0
    torch.cuda.empty_cache()
if world > 1:
    dist.barrier(); dist.destroy_process_group()
