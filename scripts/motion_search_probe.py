"""Throughput of tf_gpu_motion_search_batch (the per-block motion search over cached frames, several references in one
launch).

For each workload (a source frame and seven references, resident) and each block size, every block of the frame is
searched from a zero start against the first R references (R = 1, 2, 4, 7: n = blocks x R items in one call), with
the speed-4 settings (PRUNED_MORE sub-pel, LVL_2 mesh pruning) and the speed-2 settings (SUBPEL_TREE, mesh not
pruned).  Each configuration is warmed, then called `--reps` times; per call the probe records the search kernel's
device time (CUDA events around the launch, tf_gpu_last_stats) and the call's wall time (host clock; the call ends in
a stream synchronise, and includes the item / result copies).  items/s are reported from both.  The results of every
repetition are hashed: one hash per configuration shows they are identical.  For scale, the 16x16 search kernel of the
temporal filter (tf_gpu_last_kernel_times()[1]) on a 2-frame window of the same frames runs one 16x16 search per
16x16 block of the frame, the same count as the R = 1, 16x16 configuration; but it starts each search from the
full-pel rounding of its 32x32 block's MV, so the same items are also timed started that way ("tf_starts": the
starts come from a 32x32 call of the same settings).  The card's name and power limit are read in the same run.
    python scripts/motion_search_probe.py --out profiles/motion_search_probe_r03.json
"""
import argparse
import hashlib
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

import _clips  # noqa: E402
import _params  # noqa: E402

WORKLOADS = [  # name, width, height, bit depth
    ("1080p8", 1920, 1080, 8),
    ("1080p10", 1920, 1080, 10),
    ("4k10", 3840, 2160, 10),
]
REFS = (1, 2, 4, 7)
SPEEDS = (4, 2)


def _card():
    name = torch.cuda.get_device_name()
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                             str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001 -- recorded, not fatal
        pl = f"unknown ({e})"
    return {"name": name, "power_limit": pl}


def _rawpel(v):  # GET_MV_RAWPEL (mv.h:28): the full-pel start tf_motion_search() gives a 16x16 search
    return (v + 3 + (v >= 0)) >> 3


def _stats(v):
    return {"median": statistics.median(v), "min": min(v), "max": max(v), "all": v}


def probe_workload(pkg, wl, warmup, reps):
    name, W, H, bd = wl
    clip = _clips.moving_texture(W, H, 8, bd)
    ids = [700 + i for i in range(8)]  # source = frame 3 (ids[0]), references the other seven
    order = [3, 2, 4, 1, 5, 0, 6, 7]
    ctx = pkg.TemporalFilterGpu(device=0)
    p0 = _params.tf_params(W, H, 2, bit_depth=bd)
    for i, f in zip(ids, order):
        ctx.cache_frame(pkg.Yv12Buffer(W, H, 1, 1, bd > 8, p0["border"], frame_id=i).set_planes(*clip[f], extend=False))
    aw, ah = -(-W // 8) * 8, -(-H // 8) * 8
    out = []
    for speed in SPEEDS:
        p = _params.tf_params(W, H, 2, bit_depth=bd, speed=speed)
        # scale: the temporal filter's 16x16 search kernel on the 2-frame window (source, first reference)
        s16 = []
        for k in range(warmup + reps):
            ctx.filter_resident(dict(p, filter_frame_idx=0), [ids[0], ids[1]])
            if k >= warmup:
                s16.append(ctx.last_kernel_times()[1])
        for bsize in (16, 32):
            blocks = [(x, y) for y in range(0, ah, bsize) for x in range(0, aw, bsize)]
            for R in REFS:
                items = np.array([(x, y, 0, 0, r) for r in range(R) for x, y in blocks], np.int64)
                kern, wall, hashes = [], [], set()
                for k in range(warmup + reps):
                    torch.cuda.synchronize()
                    t0 = time.perf_counter()
                    res = ctx.motion_search_batch(p, ids[0], ids[1:1 + R], bsize, items)
                    t1 = time.perf_counter()
                    if k >= warmup:
                        kern.append(ctx.last_stats()[1])
                        wall.append((t1 - t0) * 1e3)
                        hashes.add(hashlib.sha256(res.tobytes()).hexdigest()[:16])
                n = len(items)
                r = {"workload": name, "speed": speed, "block": bsize, "refs": R, "items": n,
                     "kernel_ms": _stats(kern), "wall_ms": _stats(wall),
                     "items_per_s_kernel": n / (statistics.median(kern) * 1e-3),
                     "items_per_s_wall": n / (statistics.median(wall) * 1e-3),
                     "result_hashes": sorted(hashes), "identical_across_reps": len(hashes) == 1}
                if bsize == 16 and R == 1:
                    r["tf_search16_ms"] = _stats(s16)
                    r["tf_search16_searches"] = ((H + 31) // 32) * ((W + 31) // 32) * 4
                    r["kernel_over_tf_search16"] = statistics.median(kern) / statistics.median(s16)
                    b32 = {(x, y): i for i, (x, y) in enumerate((x, y) for y in range(0, ah, 32) for x in range(0, aw, 32))}
                    r32 = ctx.motion_search_batch(p, ids[0], ids[1:2], 32, [(x, y, 0, 0, 0) for x, y in b32])
                    tf_items = items.copy()
                    for k, (x, y) in enumerate(blocks):
                        m = r32[b32[(x // 32 * 32, y // 32 * 32)]]
                        tf_items[k, 2:4] = [_rawpel(int(m[3])), _rawpel(int(m[4]))]
                    tk = []
                    for k in range(warmup + reps):
                        ctx.motion_search_batch(p, ids[0], ids[1:2], bsize, tf_items)
                        if k >= warmup:
                            tk.append(ctx.last_stats()[1])
                    r["tf_starts_kernel_ms"] = _stats(tk)
                    r["tf_starts_kernel_over_tf_search16"] = statistics.median(tk) / statistics.median(s16)
                out.append(r)
                print(json.dumps({k: v for k, v in r.items() if k not in ("kernel_ms", "wall_ms")}), flush=True)
    ctx.close()
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="motion_search_probe.json")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--workloads", default=",".join(w[0] for w in WORKLOADS))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("motion_search_probe needs a CUDA device")
    import importlib.util
    spec = importlib.util.spec_from_file_location("aom_av1_psy_b200", os.path.join(ROOT, "aom-av1-psy_b200", "__init__.py"),
                                                  submodule_search_locations=[os.path.join(ROOT, "aom-av1-psy_b200")])
    pkg = importlib.util.module_from_spec(spec)
    sys.modules["aom_av1_psy_b200"] = pkg
    spec.loader.exec_module(pkg)
    doc = {"card": _card(), "method": __doc__.strip(), "results": []}
    for wl in WORKLOADS:
        if wl[0] in args.workloads.split(","):
            doc["results"] += probe_workload(pkg, wl, args.warmup, args.reps)
    doc["card_after"] = _card()
    with open(args.out, "w") as f:
        json.dump(doc, f, indent=1)


if __name__ == "__main__":
    main()
