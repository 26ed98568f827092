"""Host cost of the motion search with device-memory items and results (tf_gpu_motion_search_device, through
TemporalFilterGpu.motion_search_tensors) against the synchronous tf_gpu_motion_search_batch.

For each workload (a source frame and four references, resident; speed-4 settings) the probe measures, after
`--warmup` untimed calls, `--reps` times:
  - host time per call for every 16x16 block of the frame against each of the four references (n = 4 x blocks): the
    synchronous call (items from a host array, results back in a host array; the call ends in a stream synchronise)
    against the device call (items already a CUDA tensor; packing, the call and unpacking are enqueued and the host
    returns without waiting), each started from an idle GPU;
  - wall time of the two-stage chain of tests/test_gpu_motion_search_device.py: a 32x32 search of every block against
    the four references, the GET_MV_RAWPEL full-pel starts of its 16x16 blocks, then the 16x16 search -- driven
    from the host (numpy between two synchronous calls) against on the device (torch ops between two device calls on
    one stream); both end in a synchronise, and both results are compared.
The card's name and power limit are read in the same run.
    python scripts/motion_search_device_probe.py --out profiles/motion_search_device_probe_r04.json
"""
import argparse
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
    ("4k10", 3840, 2160, 10),
    ("1080p8", 1920, 1080, 8),
]
REFS = 4
SPEED = 4
OFFS = [(0, 0), (16, 0), (0, 16), (16, 16)]  # the 16x16 blocks of a 32x32 block


def _card():
    name = torch.cuda.get_device_name()
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                             str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001 -- recorded, not fatal
        pl = f"unknown ({e})"
    return {"name": name, "power_limit": pl}


def _stats(v):
    return {"median": statistics.median(v), "min": min(v), "max": max(v), "all": v}


def _rawpel(v):  # GET_MV_RAWPEL (mv.h:28)
    return (v + 3 + (v >= 0)) >> 3


def _timed(fn, warmup, reps):
    out, last = [], None
    for k in range(warmup + reps):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        last = fn()
        t1 = time.perf_counter()
        if k >= warmup:
            out.append((t1 - t0) * 1e3)
    torch.cuda.synchronize()
    return out, last


def probe_workload(pkg, wl, warmup, reps):
    name, W, H, bd = wl
    clip = _clips.moving_texture(W, H, 1 + REFS, bd)
    ids = [800 + i for i in range(1 + REFS)]
    ctx = pkg.TemporalFilterGpu(device=0)
    p = _params.tf_params(W, H, 2, bit_depth=bd, speed=SPEED)
    for i, f in zip(ids, clip):
        ctx.cache_frame(pkg.Yv12Buffer(W, H, 1, 1, bd > 8, p["border"], frame_id=i).set_planes(*f, extend=False))
    src, refs = ids[0], ids[1:]
    aw, ah = -(-W // 8) * 8, -(-H // 8) * 8
    res = {"workload": name, "width": W, "height": H, "bit_depth": bd, "speed": SPEED, "refs": REFS}

    i16 = np.array([(x, y, 0, 0, r) for r in range(REFS) for y in range(0, ah, 16) for x in range(0, aw, 16)], np.int64)
    d16 = torch.from_numpy(i16).cuda()
    sync_ms, want = _timed(lambda: ctx.motion_search_batch(p, src, refs, 16, i16), warmup, reps)
    dev_ms, got = _timed(lambda: ctx.motion_search_tensors(p, src, refs, 16, d16), warmup, reps)
    res["search16"] = {"items": len(i16), "sync_call_host_ms": _stats(sync_ms), "device_call_host_ms": _stats(dev_ms),
                       "equal": bool((got.cpu().numpy() == want).all())}

    i32 = np.array([(x, y, 0, 0, r) for r in range(REFS) for y in range(0, ah, 32) for x in range(0, aw, 32)], np.int64)
    # the 16x16 blocks of each 32x32 block that lie in the frame (at 4K the last 32x32 row has only its top two):
    # positions and parent blocks are known before the 32x32 search, only the starts come from it
    subs = [(k, x + dx, y + dy, r) for k, (x, y, _, _, r) in enumerate(i32.tolist()) for dx, dy in OFFS
            if y + dy < ah and x + dx < aw]
    parent = np.array([s[0] for s in subs], np.int64)
    sub_pos = np.array([s[1:] for s in subs], np.int64)  # x, y, ref
    d32_items = torch.from_numpy(i32).cuda()
    d_parent, d_pos = torch.from_numpy(parent).cuda(), torch.from_numpy(sub_pos).cuda()

    def host_chain():
        r32 = ctx.motion_search_batch(p, src, refs, 32, i32)
        st = _rawpel(r32[parent, 3:5])
        sub = np.stack([sub_pos[:, 0], sub_pos[:, 1], st[:, 0], st[:, 1], sub_pos[:, 2]], axis=1)
        return r32, ctx.motion_search_batch(p, src, refs, 16, sub)

    def device_chain():
        r32 = ctx.motion_search_tensors(p, src, refs, 32, d32_items)
        mv = r32[d_parent, 3:5]
        st = torch.bitwise_right_shift(mv + 3 + (mv >= 0).to(torch.int64), 3)
        sub = torch.stack([d_pos[:, 0], d_pos[:, 1], st[:, 0], st[:, 1], d_pos[:, 2]], dim=1)
        r16 = ctx.motion_search_tensors(p, src, refs, 16, sub)
        torch.cuda.synchronize()
        return r32, r16

    host_ms, (h32, h16) = _timed(host_chain, warmup, reps)
    chain_ms, (g32, g16) = _timed(device_chain, warmup, reps)
    res["chain"] = {"items32": len(i32), "items16": len(subs), "host_driven_wall_ms": _stats(host_ms),
                    "device_wall_ms": _stats(chain_ms),
                    "equal": bool((g32.cpu().numpy() == h32).all() and (g16.cpu().numpy() == h16).all())}
    ctx.close()
    print(json.dumps({k: v for k, v in res.items()}, default=str)[:2000], flush=True)
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="motion_search_device_probe.json")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--reps", type=int, default=15)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("motion_search_device_probe needs a CUDA device")
    import importlib.util
    spec = importlib.util.spec_from_file_location("aom_av1_psy_b200", os.path.join(ROOT, "aom-av1-psy_b200", "__init__.py"),
                                                  submodule_search_locations=[os.path.join(ROOT, "aom-av1-psy_b200")])
    pkg = importlib.util.module_from_spec(spec)
    sys.modules["aom_av1_psy_b200"] = pkg
    spec.loader.exec_module(pkg)
    doc = {"card": _card(), "method": __doc__.strip(), "results": []}
    for wl in WORKLOADS:
        doc["results"].append(probe_workload(pkg, wl, args.warmup, args.reps))
    doc["card_after"] = _card()
    with open(args.out, "w") as f:
        json.dump(doc, f, indent=1)


if __name__ == "__main__":
    main()
