"""CPU, world_size 2, gloo: SlabWindow.replicate_frames -- only the owner rank holds the window's frames (host arrays
of several shapes and dtypes, one monochrome frame, one plane a strided view); after the call every rank has handed
the owner's pixels, shapes, dtypes and frame ids, in order, to its context's cache_frame_tensor.  A stand-in context
records what it receives.  Run twice on one SlabWindow: the second window reuses the staging tensors."""
import os
import sys

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

HERE = os.path.dirname(os.path.abspath(__file__))


class _RecordingCtx:
    def __init__(self):
        self.calls = []

    def cache_frame_tensor(self, frame_id, y, u=None, v=None):
        self.calls.append((frame_id, [t.clone() for t in (y, u, v) if t is not None]))


def _window(seed):
    rng = np.random.default_rng(seed)
    wide = rng.integers(0, 1024, size=(36, 80)).astype(np.uint16)
    return [
        (rng.integers(0, 256, size=(24, 40)).astype(np.uint8), rng.integers(0, 256, size=(12, 20)).astype(np.uint8),
         rng.integers(0, 256, size=(12, 20)).astype(np.uint8)),
        (wide[:, 3:53], rng.integers(0, 1024, size=(18, 25)).astype(np.uint16),
         rng.integers(0, 1024, size=(18, 25)).astype(np.uint16)),
        (rng.integers(0, 4096, size=(17, 9)).astype(np.uint16), None, None),
    ]


def _worker(rank, world, port, q):
    sys.path.insert(0, HERE)
    sys.path.insert(0, os.path.dirname(HERE))
    import conftest
    conftest.load_package()
    import importlib
    sh = importlib.import_module("aom_av1_psy_b200.sharding")
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    sw = sh.SlabWindow(4, world, rank)
    ok = True
    for seed, ids in ((5, [11, 12, 13]), (6, [21, 22, 23])):
        want = _window(seed)
        ctx = _RecordingCtx()
        got_ids = sw.replicate_frames(ctx, dist, torch, want if rank == 0 else None, ids if rank == 0 else None)
        ok = ok and got_ids == ids and [c[0] for c in ctx.calls] == ids
        for (fid, planes), w in zip(ctx.calls, want):
            w = [a for a in w if a is not None]
            ok = ok and len(planes) == len(w)
            for t, a in zip(planes, w):
                ok = ok and t.device.type == "cpu" and tuple(t.shape) == a.shape
                ok = ok and t.dtype == (torch.uint8 if a.dtype == np.uint8 else torch.int16)
                ok = ok and bool((t.numpy().astype(a.dtype) == a).all())
    oks = [None] * world
    dist.all_gather_object(oks, ok)
    if rank == 0:
        q.put(oks)
    dist.destroy_process_group()


def test_replicate_frames_two_ranks_gloo():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 31500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    for p in procs:
        p.join(timeout=180)
        assert p.exitcode == 0
    assert q.get(timeout=10) == [True, True]
