"""GPU, NCCL: slab mode when only rank 0 holds the window (a real encoder's lookahead lives in one process).
sharding.SlabWindow.replicate_frames stages rank 0's frames on its GPU, broadcasts them and every rank ingests them
from device memory (tf_gpu_cache_frame_device).  Every rank's slots must equal a host upload of the same pixels, and
the slab-filtered, gathered frame and FRAME_DIFF must equal what one GPU computes alone.  Two GPUs for the real
thing (skipped with fewer); the one-rank group runs the same code on one GPU."""
import os
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
pytestmark = pytest.mark.gpu

# W, H, bit depth, frames, rank 0's frames as CUDA tensors (else host arrays)
CASES = {"cif8_n5_host": (352, 288, 8, 5, False), "1080p10_n5_tensors": (1920, 1080, 10, 5, True)}


def _worker(rank, world, port, case, q):
    sys.path.insert(0, HERE)
    sys.path.insert(0, os.path.dirname(HERE))
    import importlib
    import torch.distributed as dist
    import conftest
    import _clips
    import _params
    pkg = conftest.load_package()
    sh = importlib.import_module("aom_av1_psy_b200.sharding")
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    W, H, bd, N, as_tensors = CASES[case]
    p = _params.tf_params(W, H, N, bit_depth=bd, allow_hp=1)
    ctx = pkg.TemporalFilterGpu(device=rank, max_cached_frames=24)
    mb_rows = (H + 31) // 32
    sw = sh.SlabWindow(mb_rows, world, rank)
    ok = True
    for rep in range(2):  # two windows: the staging tensors are reused
        frames = _clips.moving_texture(W, H, N, bd, seed=300 + rep)  # only rank 0 hands them over
        if rank == 0 and as_tensors:
            own = [tuple(torch.from_numpy(a.view(np.int16) if bd > 8 else a).cuda() for a in f) for f in frames]
        else:
            own = frames
        ids = [100 * (rep + 1) + i for i in range(N)]
        got_ids = sw.replicate_frames(ctx, dist, torch, own if rank == 0 else None, ids if rank == 0 else None)
        ok = ok and got_ids == ids
        # every rank's slots equal a host upload of the same pixels (regenerated here only to check)
        host_ids = [5000 + i for i in range(N)]
        for hid, fid, (y, u, v) in zip(host_ids, ids, frames):
            b = pkg.Yv12Buffer(W, H, 1, 1, bd > 8, p["border"], frame_id=hid).set_planes(y, u, v, extend=False)
            ctx.cache_frame(b)
            db = ctx.device_border()
            for pl in range(3):
                k = 1 if pl else 0
                bx, by = (db >> 1, db >> 1) if k else (db, db)
                aw, ah = b.aligned[k]
                regions = []
                for i in (hid, fid):
                    dst = np.zeros((ah + 2 * by, aw + 2 * bx), b.dtype)
                    ctx._check(ctx.lib.tf_gpu_debug_read_plane(ctx.h, i, pl, dst.ctypes.data, dst.shape[1], -bx, -by,
                                                               dst.shape[1], dst.shape[0]))
                    regions.append(dst)
                ok = ok and bool((regions[0] == regions[1]).all())
        # slab-filtered, gathered frame == the frame one GPU computes from the host uploads
        _, diff = ctx.filter_resident(sw.params(p), ids)
        g, dsum = sw.gather(sw.device_slabs(ctx, torch, f"cuda:{rank}"),
                            torch.from_numpy(diff.copy()).to(f"cuda:{rank}"), dist, torch)
        torch.cuda.synchronize()
        if rank == 0:
            pitches = [ctx.output_device_plane(pl)[1] for pl in range(3)]
            planes = [t.cpu().numpy() for t in sw.assemble(g, pitches, torch.cat)]
            _, full_diff = ctx.filter_resident(dict(p, out_row_begin=0, out_row_end=0), host_ids)
            out = pkg.Yv12Buffer(W, H, 1, 1, bd > 8, p["border"])
            ctx.download_output(out)
            ok = ok and bool((dsum.cpu().numpy() == full_diff).all())
            for pl in range(3):
                want = out.full_blocks(pl)
                got = planes[pl][:, :want.shape[1] * want.itemsize].copy().view(want.dtype)
                ok = ok and got.shape == want.shape and bool((got == want).all())
        for i in host_ids + ids:
            ctx.evict_frame(i)
        dist.barrier()
    if rank == 0:
        q.put(ok)
    ctx.close()
    dist.destroy_process_group()


def _run(world, case, port):
    import torch.multiprocessing as mp
    mpc = mp.get_context("spawn")
    q = mpc.Queue()
    procs = [mpc.Process(target=_worker, args=(r, world, port, case, q)) for r in range(world)]
    for pr in procs:
        pr.start()
    for pr in procs:
        pr.join(timeout=600)
        assert pr.exitcode == 0
    assert q.get(timeout=10) is True


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two GPUs")
@pytest.mark.parametrize("case", sorted(CASES))
def test_replicated_slab_window_equals_one_gpu(case):
    _run(2, case, 29800 + (os.getpid() % 1000))


@pytest.mark.parametrize("case", sorted(CASES))
def test_replicate_frames_one_rank(case):
    _run(1, case, 28800 + (os.getpid() % 1000))
