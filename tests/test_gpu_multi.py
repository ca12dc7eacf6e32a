"""Frame-sharded movie on 2 GPUs (NCCL): every rank computes its contiguous block of frames on its
own device, rank 0 gathers; the result equals the single-GPU run frame for frame.  Skipped on a
single-GPU box (the CPU suite covers the same code path over gloo)."""
import os
import sys

import numpy as np
import pytest

from tests.conftest import free_port

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _worker(rank, world, port, n_frames, out_dir):
    sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist
    from spatial_light_modulator_module_b200 import generate_hologram_sequence as ghs, synthetic
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world,
                            device_id=torch.device("cuda", rank))
    try:
        frames = synthetic.movie_frames(n_frames, rescale_parameter=5.0)
        holos, exps, errors, (lo, hi) = ghs.sequence_holograms(frames, 6, precision="fp32", batch=3, want_expected=True)
        if rank == 0:
            np.savez(os.path.join(out_dir, "rank0.npz"), holos=holos, exps=exps, lo=lo, hi=hi,
                     errors=np.array([np.asarray(e) for e in errors]))
    finally:
        dist.destroy_process_group()


def test_two_gpu_movie_matches_single_gpu(tmp_path):
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    from spatial_light_modulator_module_b200 import generate_hologram_sequence as ghs, synthetic
    n = 7
    mp.spawn(_worker, args=(2, free_port(), n, str(tmp_path)), nprocs=2, join=True)
    ref_h, ref_e, ref_err, _ = ghs.sequence_holograms(synthetic.movie_frames(n, rescale_parameter=5.0), 6, precision="fp32",
                                                      batch=4, want_expected=True)
    r0 = np.load(tmp_path / "rank0.npz")
    assert (int(r0["lo"]), int(r0["hi"])) == (0, n)
    np.testing.assert_array_equal(r0["holos"], ref_h)
    np.testing.assert_array_equal(r0["exps"], ref_e)
    np.testing.assert_array_equal(r0["errors"], np.array(ref_err))


def _slab_worker(rank, world, port, n, loops, out_dir):
    sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist
    from spatial_light_modulator_module_b200 import slab, synthetic
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world,
                            device_id=torch.device("cuda", rank))
    try:
        t = synthetic.noise_target((n, n), seed=6)
        for tag, peer in (("peer", None), ("coll", False)):
            eng = slab.SlabEngine(n, world, rank, "fp32", peer=peer)
            h, e, errs = eng.gs(t[rank * (n // world):(rank + 1) * (n // world)], loops)
            np.savez(os.path.join(out_dir, f"slab_{tag}{rank}.npz"), h=h, e=e, errs=np.array(errs), status=np.array(eng.peer_status))
            eng.close()
    finally:
        dist.destroy_process_group()


def test_two_gpu_slab_gs_matches_single_gpu(tmp_path):
    """One 2048^2 plane over 2 GPUs: row slabs, NCCL all-to-all transposes, 4-scalar all-reduce."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    from spatial_light_modulator_module_b200 import synthetic
    from spatial_light_modulator_module_b200.slab import SlabEngine
    n, loops = 2048, 5
    mp.spawn(_slab_worker, args=(2, free_port(), n, loops, str(tmp_path)), nprocs=2, join=True)
    eng = SlabEngine(n, 1, 0, "fp32")
    h, e, errs = eng.gs(synthetic.noise_target((n, n), seed=6), loops)
    statuses = {}
    # transposing stores into the peer's memory / NCCL all-to-all: the same bits
    for tag in ("peer", "coll"):
        r0, r1 = np.load(tmp_path / f"slab_{tag}0.npz"), np.load(tmp_path / f"slab_{tag}1.npz")
        statuses[tag] = str(r0["status"])
        np.testing.assert_array_equal(np.concatenate([r0["h"], r1["h"]]), h)
        np.testing.assert_allclose(np.concatenate([r0["e"], r1["e"]]), e, rtol=1e-12)
        np.testing.assert_array_equal(r0["errs"], r1["errs"])
        assert np.max(np.abs(r0["errs"] - np.array(errs)) / np.array(errs)) < 1e-12
    print("slab exchange:", statuses)
    assert statuses["coll"].startswith("collectives")
    eng.close()


def _slab_gd_worker(rank, world, port, n, loops, out_dir):
    sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist
    from spatial_light_modulator_module_b200 import host_logic as hl, slab, synthetic
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world,
                            device_id=torch.device("cuda", rank))
    try:
        t = synthetic.noise_target((n, n), seed=6)
        x0 = hl.host_initial_guess("random", (n, n), 11)
        during, _ = hl.learning_rate_schedule(0.005, 1, loops)
        lo, hi = rank * (n // world), (rank + 1) * (n // world)
        for tag, peer in (("peer", None), ("coll", False)):
            eng = slab.SlabEngine(n, world, rank, "fp32", peer=peer)
            h, e, errs = eng.gd(t[lo:hi], x0[lo:hi], during, loops, white_attention=2.0)
            np.savez(os.path.join(out_dir, f"slabgd_{tag}{rank}.npz"), h=h, e=e, errs=np.array(errs))
            eng.close()
    finally:
        dist.destroy_process_group()


def test_two_gpu_slab_gd_matches_single_gpu(tmp_path):
    """GD on one 2048^2 plane over 2 GPUs (peer-memory exchange and collectives) against one GPU: the same bits."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    from spatial_light_modulator_module_b200 import host_logic as hl, synthetic
    from spatial_light_modulator_module_b200.slab import SlabEngine
    n, loops = 2048, 5
    mp.spawn(_slab_gd_worker, args=(2, free_port(), n, loops, str(tmp_path)), nprocs=2, join=True)
    eng = SlabEngine(n, 1, 0, "fp32")
    during, _ = hl.learning_rate_schedule(0.005, 1, loops)
    h, e, errs = eng.gd(synthetic.noise_target((n, n), seed=6), hl.host_initial_guess("random", (n, n), 11), during, loops,
                        white_attention=2.0)
    for tag in ("peer", "coll"):
        r0, r1 = np.load(tmp_path / f"slabgd_{tag}0.npz"), np.load(tmp_path / f"slabgd_{tag}1.npz")
        np.testing.assert_array_equal(np.concatenate([r0["h"], r1["h"]]), h)
        np.testing.assert_allclose(np.concatenate([r0["e"], r1["e"]]), e, rtol=1e-12)
        np.testing.assert_array_equal(r0["errs"], r1["errs"])
        assert np.max(np.abs(r0["errs"] - np.array(errs)) / np.array(errs)) < 1e-12
    eng.close()


def _frames_worker(rank, world, port, n_frames, out_dir):
    sys.path.insert(0, ROOT)
    import torch
    import torch.distributed as dist
    from spatial_light_modulator_module_b200 import generate_hologram_sequence as ghs, synthetic
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", init_method=f"tcp://127.0.0.1:{port}", rank=rank, world_size=world,
                            device_id=torch.device("cuda", rank))
    try:
        mask = synthetic.random_mask((768, 1024), seed=2)
        dots = synthetic.movie_frame_dots(n_frames, rescale_parameter=5.0)
        for how in ("device", "host"):                 # NCCL gather onto rank 0's device / host memory shared by the ranks
            frames, _, errors, (lo, hi) = ghs.sequence_holograms(None, 6, precision="fp32", batch=3, output="uint8", mask=mask, ct2pi=256,
                                                                 trap_dots=(dots, n_frames, (768, 1024)), gather=how)
            if rank == 0:
                import torch as _t
                np.savez(os.path.join(out_dir, f"frames0_{how}.npz"), frames=frames, lo=lo, hi=hi,
                         pinned=_t.from_numpy(frames[:1]).is_pinned())           # (rank 0 page-locks the rows it fills itself)
    finally:
        dist.destroy_process_group()


def test_two_gpu_uint8_frames_gathered(tmp_path):
    """Config 3's output format: device-rasterised trap targets, GS, mask add + quantisation, the 8-bit frames gathered
    on rank 0 both ways (NCCL onto its device; read back by every rank into shared host memory) -- equal to quantising
    the single-GPU float64 holograms."""
    import torch
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    import torch.multiprocessing as mp
    from spatial_light_modulator_module_b200 import display_holograms as dh, generate_hologram_sequence as ghs, synthetic
    n = 7
    mp.spawn(_frames_worker, args=(2, free_port(), n, str(tmp_path)), nprocs=2, join=True)
    ref_h, _, _, _ = ghs.sequence_holograms(synthetic.movie_frames(n, rescale_parameter=5.0), 6, precision="fp32", batch=4)
    mask = synthetic.random_mask((768, 1024), seed=2)
    for how in ("device", "host"):
        r0 = np.load(tmp_path / f"frames0_{how}.npz")
        assert (int(r0["lo"]), int(r0["hi"])) == (0, n) and r0["frames"].dtype == np.uint8
        assert bool(r0["pinned"])                                     # page-locked either way (shared memory: registered in place)
        for i in range(n):
            np.testing.assert_array_equal(r0["frames"][i], dh.hologram_to_grey(ref_h[i], mask, 256))
