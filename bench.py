#!/usr/bin/env python3
"""bench.py -- ARF-filtered frames/s of the B200 temporal filter (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload 4k10_n15|1080p10_n11|1080p8_n7]
                    [--mode windows|slab] [--impl tfgpu|reference] [--dump-outputs DIR]

A step = one pass of the hot path over one ARF window = one filtered output frame
per GPU (mode windows, weak scaling: independent windows per GPU, no collective) or
one window sharded by 32-px block rows over all GPUs and gathered with NCCL (mode
slab, strong scaling).  Prints ONE JSON line (rank 0).

 value     frames/s with the windows resident in HBM (device-event time of K steps on the
           library's own streams, max over ranks).  A step filters `windows_in_flight_per_gpu`
           independent windows per GPU concurrently (one tf_gpu context each; SURVEY 8e config 5:
           batches of independent ARF windows): 2 at 4K, 4 at 1080p, 1 in slab mode
 e2e       the same through tf_gpu_filter() with HOST (pinned) buffers: H2D of all window
           frames + D2H of the filtered frame inside the timed region, every step
 roofline  HBM view of the block kernel (algorithmic bytes = (N+1) planes per launch) plus
           the INT view the survey says binds (SURVEY 8d): T_int from measured pipe rates
 cpu_baseline  the reference's C temporal filter (oracle/_ref, else the oracle port) on a
           bounded row sample of the same window, 1 core

--impl reference times the reference's own CPU implementation on all host cores (row
sharding across processes, the reference's own MT axis: av1/encoder/ethread.c:2062-2189).

--dump-outputs DIR writes, after the timed steps, what every context's last timed step returned:
DIR/ctx<c>_{y,u,v}.npy (the filtered planes, whole 32x32 blocks, float32) and DIR/ctx<c>_frame_diff.npy
(FRAME_DIFF sum and sse, float64); with several ranks the names start with rank<r>_.  In slab mode on several
GPUs rank 0 writes the frame the gather assembled and the all-reduced FRAME_DIFF: DIR/frame_{y,u,v,diff}.npy
(--impl tfgpu only: the reference arm times block-row samples and returns no frame).  The inputs are seeded,
so two builds run with the same arguments can be compared file for file.  Above 64 MB in all, each plane is
cut to the same fixed sample of its samples in every run (see write_outputs).
"""
import argparse
import importlib.util
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(ROOT, "tests"))

WORKLOADS = {
    # name: (width, height, bit_depth, num_frames, filter_strength)   SURVEY 8d configs
    "4k10_n15": (3840, 2160, 10, 15, 5),
    "1080p10_n11": (1920, 1080, 10, 11, 5),
    "1080p8_n7": (1920, 1080, 8, 7, 4),
    "cif8_n7": (352, 288, 8, 7, 5),
}
# Window parameters as aomenc itself passes them (profiles/aomenc_e2e_r02.json: TF_SEAM_WINDOW lines of the
# CONFIG_TF_GPU build on the same synthetic clips, --end-usage=q --cq-level=32): q_factor of the ARF window,
# allow_high_precision_mv = 1; the noise levels are estimated from the frame to filter in every run.
Q_FACTOR = 43
ALLOW_HP = 1
SPEED_CLASS = "good cpu-used=4 (PRUNED_MORE, prune mesh lvl2, skip-row SAD >= 720p)"


def workload_config(wl):
    """The `config` object of the JSON line: names the workload only, identical in the tfgpu and reference arms."""
    width, height, bd, n, strength = WORKLOADS[wl]
    return {"workload": wl, "width": width, "height": height, "bit_depth": bd, "chroma": "4:2:0", "num_frames": n,
            "filter_strength": strength, "q_factor": Q_FACTOR, "allow_hp": ALLOW_HP, "speed_class": SPEED_CLASS,
            "clip": "synthetic moving texture (tests/_clips.py), seeded",
            "l2": f"inputs larger than L2: one window = {plane_bytes(width, height, bd) * n / 1e6:.0f} MB, "
                  "several windows cycled"}


def load_package():
    name = "aom_av1_psy_b200"
    if name in sys.modules:
        return sys.modules[name]
    path = os.path.join(ROOT, "aom-av1-psy_b200", "__init__.py")
    spec = importlib.util.spec_from_file_location(name, path, submodule_search_locations=[os.path.dirname(path)])
    mod = importlib.util.module_from_spec(spec)
    sys.modules[name] = mod
    spec.loader.exec_module(mod)
    return mod


def make_window(width, height, bd, n, seed):
    import _clips
    return _clips.moving_texture(width, height, n, bd, seed=seed)


def plane_bytes(width, height, bd):
    es = 2 if bd > 8 else 1
    return (width * height + 2 * ((width + 1) // 2) * ((height + 1) // 2)) * es


DUMP_LIMIT_BYTES = 64_000_000
SMALL = 4096  # arrays of at most this many elements are always written whole


def write_outputs(path, arrays, limit=DUMP_LIMIT_BYTES):
    """Writes {name: integer array} as path/<name>.npy: 8- and 16-bit samples in float32, wider integers
    (FRAME_DIFF) in float64, both exact.  When that would exceed `limit` bytes in all, every larger array
    is cut to the same share of its elements, flattened: sorted flat indices drawn by
    numpy.random.default_rng(0), so every run with the same arguments keeps the same positions."""
    out = {}
    for name, a in arrays.items():
        a = np.asarray(a)
        out[name] = a.astype(np.float32 if a.dtype.itemsize <= 2 else np.float64)
    small = sum(a.nbytes for a in out.values() if a.size <= SMALL)
    big = sum(a.nbytes for a in out.values() if a.size > SMALL)
    if small + big > limit:
        share = (limit - small - 256 * len(out)) / big  # 256: room for each .npy header
        for name, a in out.items():
            if a.size > SMALL:
                idx = np.sort(np.random.default_rng(0).choice(a.size, int(a.size * share), replace=False))
                out[name] = a.ravel()[idx]
    os.makedirs(path, exist_ok=True)
    for name, a in out.items():
        np.save(os.path.join(path, name + ".npy"), a)


# ---------------------------------------------------------------------------------------
# INT roofline (SURVEY 8d): scalar-equivalent pixel operations per (block, reference frame)
# ---------------------------------------------------------------------------------------
def window_params(wl):
    import _params
    width, height, bd, n, strength = WORKLOADS[wl]
    return _params.tf_params(width, height, n, bit_depth=bd, q_factor=Q_FACTOR, filter_strength=strength,
                             allow_hp=ALLOW_HP)


def int_work_per_block_ref(allow_hp):
    sad = 141 * (512 + 4 * 128)              # 1x32x32 + 4x16x16 searches, 141 sites each, skip-row SAD
    var = 2 * 2048                           # full-pel variance re-scores
    evals = 5 * (3 if allow_hp else 2) + 1   # sub-pel candidates (PRUNED_MORE, iters 1)
    subpel = evals * 2048 * 6
    pred = 4 * (27 * 16 + 16 * 16) * 12 + 8 * (19 * 8 + 8 * 8) * 12
    weights = 1536 * 29
    return dict(sad=sad, var=var, subpel=subpel, pred=pred, weights=weights)


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region: NVML from a thread (sub-millisecond
    queries, so even short regions get samples), nvidia-smi -lms as the fallback."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.thread = None
        self.stop_flag = False
        self.sm, self.reasons, self.mx = [], set(), None

    def _nvml_loop(self, nv, h):
        bits = [("hw_slowdown", nv.nvmlClocksThrottleReasonHwSlowdown),
                ("hw_thermal_slowdown", nv.nvmlClocksThrottleReasonHwThermalSlowdown),
                ("sw_thermal_slowdown", nv.nvmlClocksThrottleReasonSwThermalSlowdown),
                ("sw_power_cap", nv.nvmlClocksThrottleReasonSwPowerCap)]
        while not self.stop_flag:
            try:
                self.sm.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                r = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                for nm, bit in bits:
                    if r & bit:
                        self.reasons.add(nm)
            except Exception:
                pass
            time.sleep(0.01)

    def start(self):
        try:
            import threading
            import pynvml as nv
            nv.nvmlInit()
            # NVML indexes physical devices: honour CUDA_VISIBLE_DEVICES when it is a plain index list
            vis = os.environ.get("CUDA_VISIBLE_DEVICES", "")
            idx = self.index
            if vis and all(x.strip().isdigit() for x in vis.split(",")):
                idx = int(vis.split(",")[self.index])
            h = nv.nvmlDeviceGetHandleByIndex(idx)
            self.mx = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            self.thread = threading.Thread(target=self._nvml_loop, args=(nv, h), daemon=True)
            self.thread.start()
            return
        except Exception:
            self.thread = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                 "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if self.thread is not None:
            self.stop_flag = True
            self.thread.join(timeout=2)
            return {"sm_mhz": float(np.median(self.sm)) if self.sm else None, "sm_max_mhz": self.mx,
                    "samples": len(self.sm), "reasons": sorted(self.reasons), "source": "nvml"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons), "source": "nvidia-smi"}


# ---------------------------------------------------------------------------------------
# CPU arm
# ---------------------------------------------------------------------------------------
SIMD_NOTE = ("avx2: SAD/variance/sub-pel variance/12-tap convolve/apply_temporal_filter bound to the reference's "
             "AVX2 intrinsics (oracle/_ref/libtf_ref_avx2.so; aom_sad16x16 single-ref stays C, its only SIMD is asm)")


def cpu_filter_class(simd="auto"):
    """(factory, kind, simd) -- the compiled reference when it travelled with the repo, else the
    oracle port.  simd: "auto" picks the AVX2-bound flavour when the host has AVX2."""
    import functools
    import _ref
    if _ref.available():
        if simd in ("auto", "avx2") and _ref.avx2_available():
            return functools.partial(_ref.RefFilter, avx2=True), "reference", "avx2"
        return _ref.RefFilter, "reference", "none (generic C)"
    import _oracle
    return _oracle.OracleFilter, "port", "none (scalar C port)"


def _time_rows(cls, p, frames, rows):
    f = cls(p, frames)
    t = time.perf_counter()
    f.run(record=False, rows=rows)
    dt = time.perf_counter() - t
    f.close()
    return dt


def cpu_baseline(p, frames, rows, mb_rows, simd="auto"):
    """1-core bounded sample: block rows `rows` of the window.  The headline value is the fastest
    faithful reference build available (AVX2-bound when the host has it); the generic-C figure of
    the same sample is reported beside it."""
    cls, kind, used = cpu_filter_class(simd)
    dt = _time_rows(cls, p, frames, rows)
    frac = (rows[1] - rows[0]) / mb_rows
    out = {"value": frac / dt, "unit": "frames/s", "cores": 1, "kind": kind, "simd": used,
           "sample": f"block rows [{rows[0]},{rows[1]}) of {mb_rows} of one window ({dt:.2f} s)"}
    if used == "avx2":
        out["simd_note"] = SIMD_NOTE
        cls_c, _, _ = cpu_filter_class("c")
        dt_c = _time_rows(cls_c, p, frames, rows)
        out["generic_c"] = {"value": frac / dt_c, "unit": "frames/s", "cores": 1, "sample_s": round(dt_c, 2)}
    return out


def _ref_worker(conn, filt):
    while True:
        msg = conn.recv()
        if msg is None:
            break
        t = time.perf_counter()
        if msg[1] > msg[0]:
            filt.run(record=False, rows=msg)
        conn.send(time.perf_counter() - t)


def run_reference_arm(args, wl):
    """The reference's CPU temporal filter on all host cores; rank 0 only."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import multiprocessing as mp
    import _params
    width, height, bd, n, strength = WORKLOADS[wl]
    frames = make_window(width, height, bd, n, seed=77 if bd > 8 else 1234)
    p = window_params(wl)
    cls, kind, simd = cpu_filter_class(args.ref_simd)
    filt = cls(p, frames)
    p["noise_levels"] = tuple(filt.estimate_noise())
    filt.close()
    filt = cls(p, frames)
    mb_rows = (height + 31) // 32
    ncores = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    # calibrate on one middle row, then size a step to about 3 s of wall time
    mid = mb_rows // 2
    t = time.perf_counter()
    filt.run(record=False, rows=(mid, mid + 1))
    t_row = time.perf_counter() - t
    rows_per_step = int(min(mb_rows, max(ncores, 3.0 * ncores / max(t_row, 1e-6))))
    nw = min(ncores, rows_per_step)
    ctx = mp.get_context("fork")
    workers = []
    for _ in range(nw):
        a, b = ctx.Pipe()
        pr = ctx.Process(target=_ref_worker, args=(b, filt), daemon=True)
        pr.start()
        workers.append((pr, a))
    r0 = max(0, (mb_rows - rows_per_step) // 2)
    bounds = [r0 + (rows_per_step * i) // nw for i in range(nw + 1)]

    def step():
        t0 = time.perf_counter()
        for i, (_, c) in enumerate(workers):
            c.send((bounds[i], bounds[i + 1]))
        for _, c in workers:
            c.recv()
        return time.perf_counter() - t0

    for _ in range(args.warmup):
        step()
    times = [step() for _ in range(args.steps)]
    for pr, c in workers:
        c.send(None)
    for pr, _ in workers:
        pr.join(timeout=5)
    total = sum(times)
    frac = rows_per_step / mb_rows
    value = frac * args.steps / total
    sample = f"block rows [{r0},{r0 + rows_per_step}) of {mb_rows} per step, sharded over {nw} processes"
    line = {
        "impl": "reference", "metric": "arf_filtered_frames_per_sec", "value": value, "unit": "frames/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * total / args.steps / frac,
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u16" if bd > 8 else "u8", "data": "synthetic",
        "config": workload_config(wl),
        "measurement": {"note": "ms_per_step is per whole frame (sample time / sampled fraction)"},
        "cpu_baseline": {"value": value, "unit": "frames/s", "cores": nw, "kind": kind, "simd": simd,
                         "sample": sample},
        "e2e": {"value": value, "unit": "frames/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


# ---------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------
_REAL_STDOUT = None


def _claim_stdout():
    """stdout carries exactly one JSON line: everything else any library prints there (NCCL's version
    banner, for one) is sent to stderr by pointing fd 1 at fd 2 for the duration of the run."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        sys.stdout.flush()
        os.write(_REAL_STDOUT, data)


def main():
    _claim_stdout()
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--workload", default="4k10_n15", choices=sorted(WORKLOADS))
    ap.add_argument("--mode", default="windows", choices=["windows", "slab"])
    ap.add_argument("--impl", default="tfgpu", choices=["tfgpu", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--ref-simd", default="auto", choices=["auto", "avx2", "c"],
                    help="CPU reference flavour: auto = AVX2-bound build when the host has AVX2, c = generic C")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--concurrent", type=int, default=0,
                    help="independent windows in flight per GPU (contexts); 0 = auto: 3 for 4K, 4 below")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned as DIR/*.npy (--impl tfgpu; "
                         "the reference arm times block-row samples in worker processes and returns no frame)")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "tfgpu":
        ap.error("--dump-outputs needs --impl tfgpu: the reference arm times block-row samples and returns no frame")
    args.warmup = max(args.warmup, 3) if args.impl == "tfgpu" else args.warmup
    wl = args.workload
    if args.impl == "reference":
        run_reference_arm(args, wl)
        return

    import torch
    import torch.distributed as dist
    import _params

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; the temporal filter has no CPU fallback")
    torch.cuda.set_device(local)
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    pkg = load_package()
    import importlib
    sharding = importlib.import_module("aom_av1_psy_b200.sharding")
    width, height, bd, n, strength = WORKLOADS[wl]
    slab_req = args.mode == "slab" and world > 1
    conc = args.concurrent if args.concurrent > 0 else (1 if slab_req else (3 if width >= 3000 else 4))
    ctxs = [pkg.TemporalFilterGpu(device=local, max_cached_frames=40) for _ in range(conc)]
    ctx = ctxs[0]

    use_hbd = bd > 8
    mb_rows, mb_cols = (height + 31) // 32, (width + 31) // 32
    p = window_params(wl)

    # windows resident on this GPU: enough distinct data to exceed L2 (126 MB) several times
    win_bytes = plane_bytes(width, height, bd) * n
    nwin = max(2, int(np.ceil(400e6 / win_bytes)))
    nwin = min(nwin, 40 // n) if 40 // n >= 1 else 1
    slab = args.mode == "slab" and world > 1
    if conc > 1:
        nwin = max(2, int(np.ceil(nwin / conc)))
    all_windows = []  # [context][window] -> (frames, bufs)
    for ci in range(conc):
        windows = []
        for w in range(nwin):
            seed = (77 if bd > 8 else 1234) + (0 if slab else 1000 * rank) + 100 * ci + w
            frames = make_window(width, height, bd, n, seed)
            bufs = []
            for i, (y, u, v) in enumerate(frames):
                b = pkg.Yv12Buffer(width, height, 1, 1, use_hbd, p["border"], frame_id=1 + w * 100 + i)
                b.set_planes(y, u, v, extend=False)
                for a in b.alloc:
                    ctxs[ci].host_register(a)
                bufs.append(b)
            windows.append((frames, bufs))
        all_windows.append(windows)
    windows = all_windows[0]
    out = pkg.Yv12Buffer(width, height, 1, 1, use_hbd, p["border"])
    for a in out.alloc:
        ctx.host_register(a)

    # noise levels of the frame to filter (tf_setup_filtering_buffer, temporal_filter.c:1023-1027)
    fi = p["filter_frame_idx"]
    p["noise_levels"] = tuple(ctx.estimate_noise_from_single_plane(windows[0][1][fi], pl, bd) for pl in range(3))
    for ci in range(conc):
        for _, bufs in all_windows[ci]:
            for b in bufs:
                ctxs[ci].cache_frame(b)

    if slab:
        p["out_row_begin"], p["out_row_end"] = sharding.slab_rows(mb_rows, world, rank)

    def barrier():
        for c in ctxs:
            c.synchronize()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()

    slab_win = sharding.SlabWindow(mb_rows, world, rank) if slab else None
    last_gather = [None, None]  # slab mode: rank 0's gathered slabs and the all-reduced FRAME_DIFF of the last step

    def slab_gather(diff):
        """NCCL gather of the disjoint output row slabs to rank 0 and a 16-byte all-reduce of
        FRAME_DIFF (SURVEY 8e; integer sums, so order independent like ethread.c:2161-2173)."""
        d = torch.from_numpy(diff.copy()).to(f"cuda:{local}")
        last_gather[:] = slab_win.gather(slab_win.device_slabs(ctx, torch, f"cuda:{local}"), d, dist, torch)
        torch.cuda.current_stream().synchronize()

    ids = [[b.frame_id for b in bufs] for _, bufs in windows]
    launches = 0
    ktimes = [0.0, 0.0, 0.0]

    pending = [False] * conc
    call_ms = [0.0] * conc
    last_diff = [None] * conc

    def harvest(ci):
        nonlocal launches
        m, diff = ctxs[ci].filter_resident_result()
        pending[ci] = False
        last_diff[ci] = diff
        call_ms[ci] += m
        launches += ctxs[ci].last_stats()[0]
        if ci == 0:
            for i, t in enumerate(ctxs[ci].last_kernel_times()):
                ktimes[i] += t
        if slab:
            slab_gather(diff)

    def run_steps(nsteps):
        """One step = one window per context.  The contexts run as a staggered pipeline: a context
        gets its next window as soon as its previous one is harvested, so the GPU never drains
        between steps; everything still in flight is harvested before returning."""
        for k in range(nsteps):
            for ci, c in enumerate(ctxs):
                if pending[ci]:
                    harvest(ci)
                c.filter_resident_async(p, ids[k % nwin])
                pending[ci] = True
        for ci in range(conc):
            if pending[ci]:
                harvest(ci)

    run_steps(args.warmup)
    sampler = ClockSampler(local)
    barrier()
    sampler.start()
    launches = 0
    ktimes = [0.0, 0.0, 0.0]
    call_ms = [0.0] * conc
    for c in ctxs:
        c.event_record(0)
    t0 = time.perf_counter()
    run_steps(args.steps)
    kernel_ms = max(call_ms)
    for c in ctxs:
        c.event_record(1)
    dev_ms = max(c.event_elapsed_ms(0, 1) for c in ctxs)
    barrier()
    wall_ms = (time.perf_counter() - t0) * 1e3
    clocks = sampler.stop()
    step_ms = max(dev_ms, wall_ms if slab else dev_ms)  # slab mode includes the NCCL gather (other stream)
    tmax = torch.tensor([step_ms, kernel_ms], device=f"cuda:{local}", dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    tot_ms, kern_ms_max = tmax.tolist()
    frames_done = args.steps * (1 if slab else world * conc)
    value = frames_done / (tot_ms * 1e-3)

    # ---- the timed configuration is verified: the frame every context produced last, with all contexts in
    # flight, must equal the same window filtered synchronously on an otherwise idle device --------------
    import hashlib
    vout = pkg.Yv12Buffer(width, height, 1, 1, use_hbd, p["border"])

    if args.dump_outputs and slab:
        if rank == 0:  # the frame the gather assembled, as measure_slab() reads it back
            pitches = [ctx.output_device_plane(pl)[1] for pl in range(3)]
            planes = slab_win.assemble(last_gather[0], pitches, torch.cat)
            dumped = {}
            for pl, plane in enumerate("yuv"):
                want = vout.full_blocks(pl)
                rows = planes[pl].cpu().numpy()[:, :want.shape[1] * want.itemsize]
                dumped[f"frame_{plane}"] = np.ascontiguousarray(rows).view(want.dtype)
            dumped["frame_diff"] = last_gather[1].cpu().numpy()
            write_outputs(args.dump_outputs, dumped)
    elif args.dump_outputs:
        dumped = {}
        prefix = f"rank{rank}_" if world > 1 else ""
        for ci, c in enumerate(ctxs):
            c.download_output(vout)
            for pl, plane in enumerate("yuv"):
                dumped[f"{prefix}ctx{ci}_{plane}"] = vout.full_blocks(pl).copy()
            dumped[f"{prefix}ctx{ci}_frame_diff"] = last_diff[ci]
        write_outputs(args.dump_outputs, dumped, DUMP_LIMIT_BYTES // world)  # every rank writes its share

    def out_hash(c):
        c.download_output(vout)
        h = hashlib.sha256()
        for pl in range(3):
            h.update(np.ascontiguousarray(vout.full_blocks(pl)).tobytes())
        return h.hexdigest()

    verified = None
    if not slab:
        last_w = (args.steps - 1) % nwin
        timed_hashes = [out_hash(c) for c in ctxs]
        sync_hashes = []
        for c in ctxs:
            c.filter_resident(p, ids[last_w])
            sync_hashes.append(out_hash(c))
        vt = torch.tensor([1.0 if timed_hashes == sync_hashes else 0.0], device=f"cuda:{local}", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(vt, op=dist.ReduceOp.MIN)
        verified = bool(vt.item() == 1.0)

    # ---- 4K on several GPUs: the slab-parallel partitioning of ONE window (BASELINE.json config 4), measured
    # in the same run as the window-parallel line and reported in its "slab" object ---------------------
    def measure_slab(nsteps):
        dev = f"cuda:{local}"
        sw = sharding.SlabWindow(mb_rows, world, rank)
        frames = make_window(width, height, bd, n, 77 if bd > 8 else 1234)  # the same pixels on every rank
        sids, sbufs = [], []
        for i, (y, u, v) in enumerate(frames):
            b = pkg.Yv12Buffer(width, height, 1, 1, use_hbd, p["border"], frame_id=9000 + i)
            ctx.cache_frame(b.set_planes(y, u, v, extend=False))
            sids.append(b.frame_id)
            sbufs.append(b)
        # the slab window's own noise levels (p carries those of this rank's first window, which differ per rank)
        sp = dict(p, noise_levels=tuple(ctx.estimate_noise_from_single_plane(sbufs[fi], pl, bd) for pl in range(3)))
        pf = dict(sp, out_row_begin=0, out_row_end=0)
        # one whole window on one GPU, nothing else in flight: the latency strong scaling is measured against
        for _ in range(3):
            ctx.filter_resident(pf, sids)
        barrier()
        ctx.event_record(2)
        for _ in range(nsteps):
            ctx.filter_resident(pf, sids)
        ctx.event_record(3)
        t_one = ctx.event_elapsed_ms(2, 3) / nsteps
        full_diff = ctx.filter_resident(pf, sids)[1]
        ctx.download_output(vout)
        full_planes = [vout.full_blocks(pl).copy() for pl in range(3)]
        ps = sw.params(sp)
        gather_ms = [0.0]
        chain_ms = [0.0]
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        last = {}

        def step():
            ctx.filter_resident_async(ps, sids)
            _, diff = ctx.filter_resident_result()
            chain_ms[0] += ctx.last_kernel_times()[0]
            d = torch.from_numpy(diff.copy()).to(dev)
            ev[0].record()
            g, dsum = sw.gather(sw.device_slabs(ctx, torch, dev), d, dist, torch)
            ev[1].record()
            torch.cuda.current_stream().synchronize()
            gather_ms[0] += ev[0].elapsed_time(ev[1])
            last["g"], last["d"] = g, dsum

        for _ in range(3):
            step()
        smp = ClockSampler(local)
        barrier()
        smp.start()
        gather_ms[0] = chain_ms[0] = 0.0
        t0 = time.perf_counter()
        for _ in range(nsteps):
            step()
        barrier()
        wall = (time.perf_counter() - t0) * 1e3 / nsteps
        clk = smp.stop()
        t = torch.tensor([wall, t_one, gather_ms[0] / nsteps, chain_ms[0] / nsteps], device=dev, dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        wall, t_one_max, g_ms, c_ms = t.tolist()
        ok = None
        if rank == 0:  # the gathered frame against this GPU's own full-frame result
            pitches = [ctx.output_device_plane(pl)[1] for pl in range(3)]
            planes = sw.assemble(last["g"], pitches, torch.cat)
            ok = bool((last["d"].cpu().numpy() == full_diff).all())
            detail = {"frame_diff_equal": ok, "mismatching_samples": []}
            for pl in range(3):
                want = full_planes[pl]
                got = np.ascontiguousarray(planes[pl].cpu().numpy()[:, :want.shape[1] * want.itemsize]).view(want.dtype)
                bad = int((got != want).sum()) if got.shape == want.shape else -1
                detail["mismatching_samples"].append(bad)
                ok = ok and bad == 0
        # ---- the same slabs without a gather: every rank stores its rows into rank 0's planes over NVLink ----
        peer = None
        try:
            perr = None
            try:
                sw.connect_peer_output(ctx, dist)
            except Exception as e:
                perr = e
            pflag = torch.tensor([0.0 if perr is None else 1.0], device=dev, dtype=torch.float64)
            dist.all_reduce(pflag, op=dist.ReduceOp.MAX)  # every rank takes the same branch
            if pflag.item() > 0:
                sw.disconnect_peer_output(ctx)
                raise RuntimeError(f"peer mapping failed on some rank ({perr!r})")
            if rank == 0:
                for t in sw.device_planes(ctx, torch, dev):
                    t.zero_()  # what is compared below can only have come from the timed steps
                torch.cuda.synchronize()
            plast = {}

            def pstep():
                ctx.filter_resident_async(ps, sids)
                _, diff = ctx.filter_resident_result()
                plast["d"] = sw.finish_peer(torch.from_numpy(diff.copy()).to(dev), dist)
                torch.cuda.current_stream().synchronize()

            for _ in range(3):
                pstep()
            barrier()
            t0 = time.perf_counter()
            for _ in range(nsteps):
                pstep()
            barrier()
            pwall = (time.perf_counter() - t0) * 1e3 / nsteps
            tp = torch.tensor([pwall], device=dev, dtype=torch.float64)
            dist.all_reduce(tp, op=dist.ReduceOp.MAX)
            pwall = tp.item()
            pok = None
            if rank == 0:
                ctx.download_output(vout)
                pok = bool((plast["d"].cpu().numpy() == full_diff).all())
                for pl in range(3):
                    pok = pok and bool((vout.full_blocks(pl) == full_planes[pl]).all())
            barrier()
            sw.disconnect_peer_output(ctx)
            peer = {"mode": "no gather: every rank stores its block rows into rank 0's output planes over NVLink "
                            "(CUDA IPC peer mapping, tf_gpu_output_ipc_export/import) + 16-byte all-reduce of FRAME_DIFF",
                    "ms_per_frame": pwall, "frames_per_sec": 1e3 / pwall, "speedup": t_one_max / pwall,
                    "efficiency": t_one_max / pwall / world, "verified": pok}
        except Exception as e:  # no peer access between the GPUs of this box: the NCCL figures above stand
            peer = {"unavailable": repr(e)[:200]}
        return {"mode": "block-row slabs of one window per GPU + NCCL gather to rank 0 (SlabWindow)",
                "peer_store": peer,
                "ms_per_frame": wall, "frames_per_sec": 1e3 / wall, "single_gpu_ms_per_frame": t_one_max,
                "speedup": t_one_max / wall, "efficiency": t_one_max / wall / world,
                "gather_ms": g_ms, "search32_chain_ms": c_ms, "steps": nsteps, "clocks": clk, "verified": ok,
                "verify_detail": detail if rank == 0 else None,
                "limiter": "the ref_mv chain: one tf_search32 launch per reference frame whose per-block latency "
                           "does not shrink with the number of block rows"}

    # executed work of one window (untimed, instrumented): SURVEY 8d "executed op count"
    ctx.collect_counters(1)
    ctx.filter_resident(p, ids[0])
    executed = ctx.read_counters()
    ctx.collect_counters(0)

    # ---- e2e: host buffers through tf_gpu_filter, copies inside the timed region --------
    e2e = None
    if not args.no_e2e and not slab:
        DEPTH = 2  # windows submitted per context before the oldest is waited for
        outs = []
        for ci in range(conc):
            row = []
            for d in range(DEPTH):
                if ci == 0 and d == 0:
                    row.append(out)
                    continue
                o = pkg.Yv12Buffer(width, height, 1, 1, use_hbd, p["border"])
                for a in o.alloc:
                    ctxs[ci].host_register(a)
                row.append(o)
            outs.append(row)
        for ci in range(conc):
            for _, bufs in all_windows[ci]:
                for b in bufs:
                    b.frame_id = 0  # never cached: every step uploads the whole window

        def e2e_steps(nsteps):
            """The public submit / wait calls with host buffers in and out, as an encoder would drive
            them: every context keeps DEPTH windows submitted (the uploads of the next window overlap
            the kernels of the current one) and the contexts are staggered; all tickets are waited
            for before returning."""
            queues = [[] for _ in range(conc)]
            for k in range(nsteps):
                for ci in range(conc):
                    if len(queues[ci]) == DEPTH:
                        ctxs[ci].wait(queues[ci].pop(0)[0])
                    queues[ci].append(ctxs[ci].submit(p, all_windows[ci][k % nwin][1], outs[ci][k % DEPTH]))
            for ci in range(conc):
                for t in queues[ci]:
                    ctxs[ci].wait(t[0])

        e2e_steps(2)
        barrier()
        t0 = time.perf_counter()
        e2e_steps(args.steps)
        barrier()
        e_ms = (time.perf_counter() - t0) * 1e3
        te = torch.tensor([e_ms], device=f"cuda:{local}", dtype=torch.float64)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        es = 2 if use_hbd else 1
        d2h = sum(out.full_blocks(pl).size for pl in range(3)) * es
        e2e = {"value": args.steps * world * conc / (te.item() * 1e-3), "unit": "frames/s",
               "h2d_bytes_per_step": plane_bytes(width, height, bd) * n * conc, "d2h_bytes_per_step": int(d2h) * conc}

    slab_section = None
    if world > 1 and not slab and width >= 3000:
        slab_section = measure_slab(args.steps)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    # ---- roofline ---------------------------------------------------------------------
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        hbm_peak, peak_src = json.load(open(peaks_path))["hbm_gbs"], "measured (MEASURED_PEAKS.json)"
    else:
        hbm_peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    rows_frac = ((p["out_row_end"] - p["out_row_begin"]) / mb_rows) if slab else 1.0
    es = 2 if use_hbd else 1
    kern_s = kern_ms_max * 1e-3 / args.steps
    # The search runs as one tf_search32 launch per reference frame on the library stream (the ref_mv
    # chain) with the tf_search16 launch of the same frame overlapped on a second stream; the events
    # on the library stream therefore give: [0] the chain of (N-1) search32 launches (with the 16x16
    # work running underneath), [1] the wait for the last search16 launch, [2] the filter kernel.
    nref = n - 1
    kt = [t / args.steps for t in ktimes]  # ms per step
    luma = width * height * es
    per_launch_ms = {"tf_search32_kernel": kt[0] / max(nref, 1), "tf_filter_kernel": kt[2]}
    # algorithmic bytes per launch: every input read once + every output written once
    alg_bytes = {"tf_search32_kernel": 2 * luma * rows_frac,  # frame to filter + one reference, luma
                 "tf_filter_kernel": (n + 1) * plane_bytes(width, height, bd) * rows_frac}
    shares = {"tf_search32_kernel": kt[0], "tf_filter_kernel": kt[2]}
    dom_name = max(shares, key=shares.get)
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic_r02.json")
    if not os.path.exists(tpath):
        tpath = os.path.join(ROOT, "profiles", "traffic_r01.json")
    if os.path.exists(tpath):
        traffic = json.load(open(tpath)).get(wl, {}).get(dom_name)
    achieved = alg_bytes[dom_name] / (per_launch_ms[dom_name] * 1e-3) / 1e9
    rates = {k: ctx.microbench(i) for i, k in enumerate(["iadd", "imad", "vabsdiff4", "vimnmx_u16x2", "idp4a", "dfma"])}
    W = int_work_per_block_ref(p["allow_hp"])
    # px per lane-instruction: 8-bit SAD = 4 px per VABSDIFF4.ACC; high bitdepth = 2 px per (max, min, sub-add)
    r_sad = rates["vabsdiff4"] * 4 if bd == 8 else rates["vimnmx_u16x2"] * 2 / 3
    t_int_block = (W["sad"] / r_sad + (W["var"] + W["subpel"] + W["pred"]) / rates["imad"] + W["weights"] / rates["iadd"]) / 1e9
    t_int = t_int_block * mb_rows * mb_cols * (n - 1) * rows_frac
    step_alg = (n + 1) * plane_bytes(width, height, bd) * rows_frac * conc
    nbr = mb_rows * mb_cols * (n - 1) * rows_frac
    w_exec = {"sad": executed[0] / nbr, "subpel": executed[1] * 6 / nbr, "var": executed[2] * 2 / nbr,
              "pred": W["pred"], "weights": W["weights"]}
    t_exec = nbr * (w_exec["sad"] / r_sad + (w_exec["var"] + w_exec["subpel"] + w_exec["pred"]) / rates["imad"]
                    + w_exec["weights"] / rates["iadd"]) / 1e9
    exec_info = {"work_per_block_ref": w_exec, "t_int_ms": t_exec * conc * 1e3, "frac": t_exec * conc / kern_s}
    # px-ops of the whole step / time: the binding (integer) roofline at top level, the HBM view nested
    w_step = sum(W.values()) * mb_rows * mb_cols * (n - 1) * rows_frac * conc
    roofline = {
        "bound": "int", "achieved": w_step / kern_s / 1e9, "peak": w_step / (t_int * conc) / 1e9, "unit": "Gpixel-op/s",
        "frac": t_int * conc / kern_s, "traffic": traffic,
        "note": "binding roofline per SURVEY 8d: T_int = sum_class W_class / R_class over pipe rates measured in this run "
                "(tf_gpu_microbench), whole step (all windows in flight); frac = T_int / T_step.  W = static-content floor "
                "per (block, reference frame); `executed` = instrumented counts of this clip",
        "kernel": dom_name, "kernel_ms": per_launch_ms[dom_name],
        "launches_per_step": {"tf_search32_kernel": nref, "tf_search16_kernel": nref, "tf_filter_kernel": 1},
        "phases_ms": {"search32_chain_with_search16_overlapped": kt[0], "search16_tail": kt[1], "filter": kt[2]},
        "work_per_block_ref": W, "rates_giga_lane_ops_per_s": rates, "t_int_ms": t_int * conc * 1e3,
        "executed": exec_info,
        "hbm": {"achieved": achieved, "peak": hbm_peak, "unit": "GB/s", "frac": achieved / hbm_peak,
                "peak_source": peak_src, "kernel": dom_name, "algorithmic_bytes_per_launch": alg_bytes[dom_name],
                "traffic_bytes_per_launch": traffic,
                "step": {"algorithmic_bytes": step_alg, "kernels_ms_sum": kern_s * 1e3,
                         "achieved_gbs": step_alg / kern_s / 1e9, "frac": step_alg / kern_s / 1e9 / hbm_peak}},
    }

    line = {
        "metric": "arf_filtered_frames_per_sec", "value": value, "unit": "frames/s", "n_gpus": world,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": tot_ms / args.steps, "higher_is_better": True,
        "scaling": "strong" if slab else "weak", "vs_baseline": None, "dtype": "u16" if use_hbd else "u8",
        "data": "synthetic",
        "config": workload_config(wl),
        "measurement": {"mode": "slab rows + NCCL gather" if slab else "independent windows per GPU",
                        "windows_in_flight_per_gpu": conc,
                        "resident_windows_cycled": f"{nwin} per context x {win_bytes / 1e6:.0f} MB",
                        "timing": "CUDA events on the library stream around K steps, max over ranks"},
        "verified": verified,
        "clocks": clocks, "gpu_launches": launches, "roofline": roofline,
    }
    if slab_section:
        line["slab"] = slab_section
    if e2e:
        line["e2e"] = e2e
    if not args.no_cpu_baseline and world == 1:
        mid = mb_rows // 2
        nrows = mb_rows  # one whole window: ~6 s (AVX2) + ~18 s (generic C) of one core at 4K 10-bit
        rows = (max(0, mid - nrows // 2), min(mb_rows, mid - nrows // 2 + nrows))
        pc = dict(p)
        pc["out_row_begin"] = pc["out_row_end"] = 0
        line["cpu_baseline"] = cpu_baseline(pc, windows[0][0], rows, mb_rows, args.ref_simd)
    emit(line)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
