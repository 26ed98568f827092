"""Batched windows (tf_gpu_filter_batch_async) against the other ways of running K windows on one GPU.

For each workload and K, K windows slide over one clip (window k = frames k .. k + N - 1, filtering its centre
frame) and are timed three ways:
  * batch:     one context, the K windows as one filter_batch call, calls back to back;
  * contexts:  K contexts in flight, each holding its own copy of its window's frames, driven as bench.py drives
               its windows (a context gets its next window as soon as its previous one is harvested);
  * serial:    one context, filter_resident for one window after another.
Each mode runs `--warmup` rounds first (every shape warmed), then `--reps` timed repetitions of `rounds` rounds (one
round = the K windows once); the host clock spans the repetition and ends in a device synchronise.  The outputs and
FRAME_DIFF of every window must be identical in all three modes.  Writes one JSON document (--out) with the card's
name and power limit, read in the same run, beside the numbers.
    python scripts/batch_probe.py --out profiles/batch_probe_r03.json
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

# name, width, height, bit depth, frames per window, windows per timed repetition (sizes the work to ~0.3-1 s)
WORKLOADS = [
    ("4k10_n15", 3840, 2160, 10, 15, 48),
    ("1080p10_n11", 1920, 1080, 10, 11, 128),
    ("1080p8_n7", 1920, 1080, 8, 7, 192),
    ("360p8_n7", 640, 360, 8, 7, 512),
]
KS = (2, 4, 8, 16)


def _card():
    name = torch.cuda.get_device_name()
    try:
        pl = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                             str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout.strip()
    except Exception as e:  # noqa: BLE001 -- recorded, not fatal
        pl = f"unknown ({e})"
    return {"name": name, "power_limit": pl}


def _cache(pkg, ctx, p, frames, ids):
    for i, planes in zip(ids, frames):
        b = pkg.Yv12Buffer(p["width"], p["height"], 1, 1, p["use_hbd"], p["border"], frame_id=i)
        b.set_planes(*planes, extend=False)
        ctx.cache_frame(b)


def _download(pkg, ctx, p, window=None):
    o = pkg.Yv12Buffer(p["width"], p["height"], 1, 1, p["use_hbd"], p["border"])
    if window is None:
        ctx.download_output(o)
    else:
        ctx.download_batch_output(window, o)
    return [o.full_blocks(pl).copy() for pl in range(3)]


def _time(fn, rounds, warmup, reps):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    out = []
    for _ in range(reps):
        t0 = time.perf_counter()
        for _ in range(rounds):
            fn()
        torch.cuda.synchronize()
        out.append((time.perf_counter() - t0) * 1e3 / rounds)
    return out


def probe(pkg, wl, K, warmup, reps, clip):
    name, W, H, bd, N, per_rep = wl
    p = _params.tf_params(W, H, N, bit_depth=bd)
    ids = [1 + i for i in range(N + K - 1)]
    wins = [ids[k:k + N] for k in range(K)]
    ps = [p] * K
    rounds = max(2, per_rep // K)

    batch = pkg.TemporalFilterGpu(device=0, max_cached_frames=max(24, N + K - 1))
    _cache(pkg, batch, p, clip[:N + K - 1], ids)
    ctxs = []
    for k in range(K):
        c = pkg.TemporalFilterGpu(device=0)
        _cache(pkg, c, p, clip[k:k + N], wins[k])
        ctxs.append(c)

    def run_batch():
        batch.filter_batch(ps, wins)

    pending = [False] * K

    def run_contexts():
        for k, c in enumerate(ctxs):
            if pending[k]:
                c.filter_resident_result()
            c.filter_resident_async(p, wins[k])
            pending[k] = True

    def drain():
        for k, c in enumerate(ctxs):
            if pending[k]:
                c.filter_resident_result()
                pending[k] = False

    def run_serial():
        for k in range(K):
            batch.filter_resident(p, wins[k])

    res = {"workload": name, "K": K, "rounds_per_rep": rounds}
    res["batch_ms"] = _time(run_batch, rounds, warmup, reps)
    res["contexts_ms"] = []
    for _ in range(reps):  # the pipeline is drained at the end of every repetition, inside its clock
        t = _time(run_contexts, rounds, 0 if res["contexts_ms"] else warmup, 1)
        t0 = time.perf_counter()
        drain()
        torch.cuda.synchronize()
        res["contexts_ms"].append(t[0] + (time.perf_counter() - t0) * 1e3 / rounds)
    res["serial_ms"] = _time(run_serial, rounds, warmup, reps)
    for m in ("batch", "contexts", "serial"):
        v = res[m + "_ms"]
        res[m] = {"median_ms_per_round": statistics.median(v), "min": min(v), "max": max(v),
                  "frames_per_s": K / (statistics.median(v) * 1e-3)}

    # identical outputs in all three modes
    _, bdiff = batch.filter_batch(ps, wins)
    b_out = [_download(pkg, batch, p, k) for k in range(K)]
    same = True
    for k in range(K):
        _, d = ctxs[k].filter_resident(p, wins[k])
        c_out = _download(pkg, ctxs[k], p)
        _, d2 = batch.filter_resident(p, wins[k])
        s_out = _download(pkg, batch, p)
        same &= bool((d == bdiff[k]).all() and (d2 == bdiff[k]).all())
        same &= all((a == b).all() and (a == c).all() for a, b, c in zip(b_out[k], c_out, s_out))
    res["outputs_identical"] = same
    for c in ctxs:
        c.close()
    batch.close()
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default="batch_probe.json")
    ap.add_argument("--warmup", type=int, default=2)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--workloads", default=",".join(w[0] for w in WORKLOADS))
    ap.add_argument("--ks", default=",".join(map(str, KS)))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("batch_probe needs a CUDA device")
    import importlib.util
    spec = importlib.util.spec_from_file_location("aom_av1_psy_b200", os.path.join(ROOT, "aom-av1-psy_b200", "__init__.py"),
                                                  submodule_search_locations=[os.path.join(ROOT, "aom-av1-psy_b200")])
    pkg = importlib.util.module_from_spec(spec)
    sys.modules["aom_av1_psy_b200"] = pkg
    spec.loader.exec_module(pkg)
    doc = {"card": _card(), "method": __doc__.strip().splitlines()[0], "results": []}
    ks = [int(k) for k in args.ks.split(",")]
    for wl in WORKLOADS:
        if wl[0] not in args.workloads.split(","):
            continue
        _, W, H, bd, N, _ = wl
        clip = _clips.moving_texture(W, H, N + max(ks) - 1, bd)
        for K in ks:
            try:
                r = probe(pkg, wl, K, args.warmup, args.reps, clip)
            except pkg.TfGpuError as e:  # e.g. memory: recorded as not measured
                r = {"workload": wl[0], "K": K, "not_measured": str(e)}
            doc["results"].append(r)
            print(json.dumps(r), flush=True)
    doc["card_after"] = _card()
    with open(args.out, "w") as f:
        json.dump(doc, f, indent=1)


if __name__ == "__main__":
    main()
