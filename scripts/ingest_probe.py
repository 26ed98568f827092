"""Frame ingest from device memory vs host upload.

One GPU (default), at 4K 10-bit and 1080p 8-bit 4:2:0:
  * per-frame device ingest (tf_gpu_cache_frame_device: one ingest_plane_kernel per plane), CUDA events on the
    producer's stream around many calls;
  * per-frame host upload (tf_gpu_cache_frame: H2D copy + border kernel, a synchronous call) from pinned and from
    pageable memory, host clock;
  * the ingest's achieved bytes/s (crop area read + defined slot region written) against the 7.7 TB/s HBM3e
    figure of the B200 data sheet.
Sources and slots rotate over enough distinct frames that the traffic of one round exceeds twice the 126 MB L2.

--gpus N (under torchrun, one process per GPU): time until every rank holds a 15-frame 4K 10-bit window, per-rank
host uploads (pinned) vs owner upload + NCCL broadcast + device ingest (sharding.SlabWindow.replicate_frames).

Writes one JSON document (--out) with the card name and power limit beside the numbers.
    python scripts/ingest_probe.py --out probe.json
    torchrun --nproc-per-node 2 scripts/ingest_probe.py --gpus 2 --out probe_2gpu.json
"""
import argparse
import importlib
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests"))
sys.path.insert(0, ROOT)
HBM_TBPS = 7.7  # B200 data sheet, one GPU
L2_BYTES = 126e6


def _card():
    name = torch.cuda.get_device_name()
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                             str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001 -- recorded, not fatal
        pl = f"unknown ({e})"
    return {"name": name, "power_limit": pl}


def _frames(W, H, bd, k, seed):
    rng = np.random.default_rng(seed)
    dt = np.uint16 if bd > 8 else np.uint8
    cw, ch = (W + 1) >> 1, (H + 1) >> 1
    return [tuple(rng.integers(0, 1 << bd, size=s).astype(dt) for s in ((H, W), (ch, cw), (ch, cw))) for _ in range(k)]


def _bytes(W, H, bd, border):
    """(crop area read, defined slot region written) in bytes for a 4:2:0 frame; device border `border` luma."""
    es = 2 if bd > 8 else 1
    aw, ah = -(-W // 8) * 8, -(-H // 8) * 8
    read = (W * H + 2 * ((W + 1) >> 1) * ((H + 1) >> 1)) * es
    write = ((aw + 2 * border) * (ah + 2 * border) + 2 * ((aw >> 1) + border) * ((ah >> 1) + border)) * es
    return read, write


def single_gpu(pkg, W, H, bd, reps):
    border = pkg.load_library().tf_gpu_device_border()
    rd, wr = _bytes(W, H, bd, border)
    k = max(8, int(2 * L2_BYTES / (rd + wr)) + 1)
    ctx = pkg.TemporalFilterGpu(device=torch.cuda.current_device(), max_cached_frames=max(k, 24))
    frames = _frames(W, H, bd, k, seed=bd)
    tens = [[torch.from_numpy(a.view(np.int16) if bd > 8 else a).cuda() for a in f] for f in frames]
    ids = [1 + i for i in range(k)]
    for i, t in zip(ids, tens):  # warm-up: slots allocated, modules loaded
        ctx.cache_frame_tensor(i, *t)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    per, host = [], []
    for _ in range(reps):
        for i in ids:
            ctx.evict_frame(i)
        # the stream is held behind a sleep until all k calls are enqueued, so the events time the GPU work
        # (launches + cross-stream event waits + kernels), not the rate at which the host issues the calls
        torch.cuda._sleep(50_000_000)
        e0.record()
        t0 = time.perf_counter()
        for i, t in zip(ids, tens):
            ctx.cache_frame_tensor(i, *t)
        host.append((time.perf_counter() - t0) * 1e3 / k)
        e1.record()
        torch.cuda.synchronize()
        assert ctx.last_stats()[0] == 3
        per.append(e0.elapsed_time(e1) / k)
    ingest_ms = statistics.median(per)
    assert max(host) * k < 20, "host enqueue outran the sleep: the event time would include host time"

    def host_upload(pinned):
        bufs = []
        for i, (y, u, v) in enumerate(frames):
            b = pkg.Yv12Buffer(W, H, 1, 1, bd > 8, 160, frame_id=1000 + i).set_planes(y, u, v, extend=False)
            if pinned:
                for a in b.alloc:
                    ctx.host_register(a)
            bufs.append(b)
        for b in bufs:
            ctx.cache_frame(b)
        out = []
        for _ in range(reps):
            for b in bufs:
                ctx.evict_frame(b.frame_id)
            t0 = time.perf_counter()
            for b in bufs:
                ctx.cache_frame(b)
            out.append((time.perf_counter() - t0) * 1e3 / k)
        for b in bufs:
            ctx.evict_frame(b.frame_id)
            if pinned:
                for a in b.alloc:
                    ctx.host_unregister(a)
        return statistics.median(out)

    for i in ids:
        ctx.evict_frame(i)
    up_pinned = host_upload(True)
    up_pageable = host_upload(False)
    ctx.close()
    floor_ms = (rd + wr) / (HBM_TBPS * 1e12) * 1e3
    return {
        "frame": f"{W}x{H} {bd}-bit 4:2:0", "distinct_frames_per_round": k, "rounds": reps,
        "bytes_read": rd, "bytes_written": wr,
        "device_ingest_ms_per_frame": round(ingest_ms, 4),
        "host_call_ms_per_frame": round(statistics.median(host), 4),
        "host_upload_pinned_ms_per_frame": round(up_pinned, 4),
        "host_upload_pageable_ms_per_frame": round(up_pageable, 4),
        "ingest_GBps": round((rd + wr) / ingest_ms / 1e6, 1),
        "hbm_floor_ms": round(floor_ms, 4),
        "ingest_share_of_hbm_floor": round(floor_ms / ingest_ms, 3),
        "upload_pinned_over_ingest": round(up_pinned / ingest_ms, 1),
    }


def multi_gpu(pkg, sh, reps):
    import torch.distributed as dist
    rank, world = dist.get_rank(), dist.get_world_size()
    W, H, bd, N = 3840, 2160, 10, 15
    frames = _frames(W, H, bd, N, seed=7)  # every rank has them for the per-rank upload arm only
    ctx = pkg.TemporalFilterGpu(device=torch.cuda.current_device(), max_cached_frames=2 * N + 2)
    bufs = []
    for i, (y, u, v) in enumerate(frames):
        b = pkg.Yv12Buffer(W, H, 1, 1, True, 160, frame_id=1 + i).set_planes(y, u, v, extend=False)
        for a in b.alloc:
            ctx.host_register(a)
        bufs.append(b)
    sw = sh.SlabWindow((H + 31) // 32, world, rank)
    ids = [100 + i for i in range(N)]

    def timed(fn):
        out = []
        for r in range(reps + 1):
            dist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            fn()
            torch.cuda.synchronize()
            dist.barrier()
            if r:  # first round: warm-up
                out.append((time.perf_counter() - t0) * 1e3)
            for b in bufs:
                ctx.evict_frame(b.frame_id)
            for i in ids:
                ctx.evict_frame(i)
        return statistics.median(out)

    def per_rank_uploads():
        for b in bufs:
            ctx.cache_frame(b)

    def replicate():
        sw.replicate_frames(ctx, dist, torch, frames if rank == 0 else None, ids if rank == 0 else None)

    res = {"window": f"{N} x {W}x{H} {bd}-bit 4:2:0", "gpus": world, "rounds": reps,
           "per_rank_host_uploads_pinned_ms": round(timed(per_rank_uploads), 3),
           "owner_upload_broadcast_ingest_ms": round(timed(replicate), 3)}
    for b in bufs:
        for a in b.alloc:
            ctx.host_unregister(a)
    ctx.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default="ingest_probe.json")
    a = ap.parse_args()
    import conftest
    pkg = conftest.load_package()
    res = {"card": None}
    if a.gpus > 1:
        import torch.distributed as dist
        rank = int(os.environ["RANK"])
        torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
        dist.init_process_group("nccl", device_id=torch.device("cuda", torch.cuda.current_device()))
        sh = importlib.import_module("aom_av1_psy_b200.sharding")
        res["multi_gpu"] = multi_gpu(pkg, sh, a.reps)
        res["card"] = _card()
        dist.destroy_process_group()
        if rank:
            return
    else:
        res["card"] = _card()
        res["single_gpu"] = [single_gpu(pkg, 3840, 2160, 10, a.reps), single_gpu(pkg, 1920, 1080, 8, a.reps)]
    res["note"] = ("device ingest: CUDA events on the producer's stream, enqueued behind a sleep (GPU time of the "
                   "k calls of a round / k); host_call: host time of one cache_frame_tensor call (validation + "
                   "enqueue); host upload: host clock around the synchronous tf_gpu_cache_frame; HBM floor from the "
                   "7.7 TB/s data-sheet figure")
    txt = json.dumps(res, indent=1)
    print(txt)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        f.write(txt + "\n")


if __name__ == "__main__":
    main()
