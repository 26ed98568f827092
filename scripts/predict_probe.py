"""Throughput of tf_gpu_predict_device (TemporalFilterGpu.predict_tensors) on the B200.

Workloads: 4K 10-bit 4:2:0 and 1080p 8-bit 4:2:0, every 16x16 block of a source frame against 14 references (4K:
453,600 items).  The MVs come from a device motion search of those blocks (motion_search_tensors, zero starts); an
all-zero-MV control runs the copy path.  For each: the kernel time from CUDA events on the torch stream after
warm-up (median and spread over the repetitions), the bytes written (samples and status) and a lower bound on the
bytes read (the items, plus one read of each reference's crop area, every block of which is predicted), as GB/s
against the 7.7 TB/s data-sheet HBM3e figure; and the wall time of the search -> predict chain (host clock around
both calls and a synchronise).  The card's name and power limit are read in the same run.

    python scripts/predict_probe.py --out profiles/predict_probe_r07.json [--reps 20]
"""
import argparse
import ctypes as C
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
import _clips  # noqa: E402
import _params  # noqa: E402
import conftest  # noqa: E402

PEAK_BYTES_PER_S = 7.7e12
NUM_REFS = 14


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                       text=True).stdout.strip().splitlines()
    name, limit = [s.strip() for s in q[0].split(",")]
    return {"name": name, "power_limit": limit}


def time_ms(fn, reps, warmup=3):
    for _ in range(warmup):
        fn()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        ts.append(a.elapsed_time(b))
    return {"median_ms": statistics.median(ts), "min_ms": min(ts), "max_ms": max(ts), "reps": reps}


def workload(pkg, ctx, name, W, H, bd, reps):
    p = _params.tf_params(W, H, 1 + NUM_REFS, bit_depth=bd)
    frames = _clips.moving_texture(W, H, 1 + NUM_REFS, bd, motion=(1, 2))
    ids = []
    for i, planes in enumerate(frames):
        b = pkg.Yv12Buffer(W, H, 1, 1, p["use_hbd"], p["border"], frame_id=5_000_000 + 100 * bd + i)
        ctx.cache_frame(b.set_planes(*planes))
        ids.append(b.frame_id)
    del frames
    ah = -(-H // 8) * 8
    blocks = np.array([(x, y) for y in range(0, ah, 16) for x in range(0, W, 16)], np.int64)
    items = np.zeros((len(blocks) * NUM_REFS, 5), np.int64)
    items[:, 0:2] = np.tile(blocks, (NUM_REFS, 1))
    items[:, 4] = np.repeat(np.arange(NUM_REFS), len(blocks))
    d_items = torch.from_numpy(items).cuda()
    n = len(items)
    res = ctx.motion_search_tensors(p, ids[0], ids[1:], 16, d_items)
    mv_items = d_items.clone()
    mv_items[:, 2:4] = res[:, 3:5]
    torch.cuda.synchronize()
    es = 2 if p["use_hbd"] else 1
    num_pels = 256 + 2 * 64
    crop = W * H + 2 * ((W + 1) // 2) * ((H + 1) // 2)
    written = n * (num_pels * es + 4)
    read_lb = n * 16 + NUM_REFS * crop * es
    out = {"workload": name, "width": W, "height": H, "bit_depth": bd, "items": n, "refs": NUM_REFS,
           "bytes_written": written, "bytes_read_lower_bound": read_lb}
    frac = (res[:, 3:5] & 7 != 0).any(dim=1).float().mean().item()
    cp = pkg.make_params(p)
    ref_ids = (C.c_uint64 * NUM_REFS)(*ids[1:])
    pred = torch.empty(n * num_pels, dtype=torch.int16 if es == 2 else torch.uint8, device="cuda")
    status = torch.empty(n, dtype=torch.int32, device="cuda")
    for label, its in (("search_mvs", mv_items), ("zero_mv_copy", d_items)):
        packed = pkg.pack_motion_items(its)

        def call():  # the library call alone: items packed and outputs allocated beforehand
            rc = ctx.lib.tf_gpu_predict_device(ctx.h, C.byref(cp), ref_ids, NUM_REFS, 16, packed.data_ptr(), n,
                                               pred.data_ptr(), status.data_ptr(),
                                               torch.cuda.current_stream().cuda_stream)
            assert rc == 0, rc
        t = time_ms(call, reps)
        gbs = (written + read_lb) / (t["median_ms"] * 1e-3) / 1e9
        out[label] = dict(t, gb_per_s=gbs, share_of_7_7_tb_s=gbs * 1e9 / PEAK_BYTES_PER_S)
    out["search_mvs"]["items_with_subpel_mv"] = frac
    # wall time of the chain: search then predict at its MVs, one synchronise at the end
    walls = []
    for _ in range(5):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        r = ctx.motion_search_tensors(p, ids[0], ids[1:], 16, d_items)
        it2 = d_items.clone()
        it2[:, 2:4] = r[:, 3:5]
        ctx.predict_tensors(p, ids[1:], 16, it2)
        torch.cuda.synchronize()
        walls.append((time.perf_counter() - t0) * 1e3)
    out["chain_wall_ms"] = {"median_ms": statistics.median(walls), "min_ms": min(walls), "max_ms": max(walls)}
    for i in ids:
        ctx.evict_frame(i)
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True)
    ap.add_argument("--reps", type=int, default=20)
    args = ap.parse_args()
    pkg = conftest.load_package()
    ctx = pkg.TemporalFilterGpu(device=0, max_cached_frames=1 + NUM_REFS)
    rec = {"card": card(), "peak_bytes_per_s": PEAK_BYTES_PER_S, "workloads": [
        workload(pkg, ctx, "4k10", 3840, 2160, 10, args.reps),
        workload(pkg, ctx, "1080p8", 1920, 1080, 8, args.reps)]}
    rec["card_after"] = card()
    ctx.close()
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(rec, f, indent=1)
    print(json.dumps(rec, indent=1))


if __name__ == "__main__":
    main()
