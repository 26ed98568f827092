"""Latency of one block-row slab of one 4K 10-bit window on one GPU (what a rank of the slab mode computes),
for 1/1, 1/2, 1/4, 1/8 of the rows, for the library in TF_GPU_LIB (or the in-tree build)."""
import os, sys, time
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import bench
wl = "4k10_n15"
width, height, bd, n, strength = bench.WORKLOADS[wl]
pkg = bench.load_package()
ctx = pkg.TemporalFilterGpu(device=0, max_cached_frames=40)
p = bench.window_params(wl)
frames = bench.make_window(width, height, bd, n, 77)
bufs = []
for i, (y, u, v) in enumerate(frames):
    b = pkg.Yv12Buffer(width, height, 1, 1, True, p["border"], frame_id=1 + i).set_planes(y, u, v, extend=False)
    ctx.cache_frame(b); bufs.append(b)
fi = p["filter_frame_idx"]
p["noise_levels"] = tuple(ctx.estimate_noise_from_single_plane(bufs[fi], pl, bd) for pl in range(3))
ids = [b.frame_id for b in bufs]
mb_rows = (height + 31) // 32
out = {}
for parts in (1, 2, 4, 8):
    rows = (mb_rows + parts - 1) // parts
    pp = dict(p, out_row_begin=0 if parts == 1 else mb_rows // 2 - rows // 2, out_row_end=0 if parts == 1 else mb_rows // 2 - rows // 2 + rows)
    for _ in range(3): ctx.filter_resident(pp, ids)
    ctx.event_record(2)
    K = 10
    for _ in range(K): ctx.filter_resident(pp, ids)
    ctx.event_record(3)
    out[parts] = round(ctx.event_elapsed_ms(2, 3) / K, 3)
print(os.environ.get("TF_GPU_LIB", "cur"), out, {k: round(out[1] / v / k, 3) for k, v in out.items()})
