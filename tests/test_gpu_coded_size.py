"""GPU: coded sizes, mi grids and borders that differ from the frames' own (superres, spatial resize), through every
entry point that reads them, against the oracle (test_oracle_coded_size.py shows that each case reaches its regime).

The bar is test_gpu_fuzz.py's: MVs, MSEs, predictors, accum and count bit-exact, output within 1 LSB, FRAME_DIFF
equal.  At 4K and 1080p the oracle runs on sampled block rows (as in test_gpu_fullsize.py); case a's rows all hold
32x32 blocks whose column limits are inverted."""
import numpy as np
import pytest

import _coded
import _gpu
import _oracle
import _oracle_motion

pytestmark = pytest.mark.gpu

N = _coded.N
MAX_ORACLE_ITEMS = 20000  # per block size: every position of the grids here (4K coded at 1920x2160: 16200)


def _bufs(pkg, p, frames, id_base=0):
    return [pkg.Yv12Buffer(p["width"], p["height"], p["ss_x"], p["ss_y"], p["use_hbd"], p["border"], p["monochrome"],
                           frame_id=(id_base + i) if id_base else 0).set_planes(*f) for i, f in enumerate(frames)]


def _planes(out):
    return [out.full_blocks(pl).astype(np.uint16).copy() for pl in range(out.num_planes)]


def _check_rows(g, p, frames, rows, slab_diff):
    """The whole-frame dump g against the oracle on block rows `rows` (None: all of them)."""
    o = _oracle.OracleFilter(p, frames)
    mb_cols = o.mb_cols
    fi = p["filter_frame_idx"]
    sel = [f for f in range(N) if f != fi]
    for rr in rows or [(0, o.mb_rows)]:
        r = o.run(rows=rr)
        b0, b1 = rr[0] * mb_cols, rr[1] * mb_cols
        for k in ("mvs", "mses", "pred"):
            assert (g[k][b0:b1][:, sel] == r[k][b0:b1][:, sel]).all(), (k, rr)
        for k in ("accum", "count"):
            assert (g[k][b0:b1] == r[k][b0:b1]).all(), (k, rr)
        for pl, (a, b) in enumerate(zip(g["out"], r["out"])):
            bh = 32 >> (p["ss_y"] if pl else 0)
            d = np.abs(a[rr[0] * bh:rr[1] * bh].astype(np.int32) - b[rr[0] * bh:rr[1] * bh].astype(np.int32))
            assert d.max() <= 1, (pl, rr)
        want = r["diff"] if rows else g["diff"]
        assert (slab_diff(rr) == r["diff"]).all() and (want == r["diff"]).all(), rr
    o.close()


def _filter_case(pkg, tfgpu, p, frames, rows, id_base):
    """tf_gpu_filter_dump on the whole frame against the oracle (rows), then filter_resident on row slabs
    reassembled into the whole-frame output with FRAME_DIFF adding up."""
    g = _gpu.run_gpu(pkg, tfgpu, p, frames)
    bufs = _bufs(pkg, p, frames, id_base)
    for b in bufs:
        tfgpu.cache_frame(b)
    ids = [b.frame_id for b in bufs]
    try:
        def slab_diff(rr):
            return tfgpu.filter_resident(dict(p, out_row_begin=rr[0], out_row_end=rr[1]), ids)[1]
        _check_rows(g, p, frames, rows, slab_diff)
        mb_rows = (p["height"] + 31) // 32
        cuts = sorted({0, mb_rows // 3, 2 * mb_rows // 3 + 1, mb_rows})
        out = pkg.Yv12Buffer(p["width"], p["height"], p["ss_x"], p["ss_y"], p["use_hbd"], p["border"])
        diff = np.zeros(2, np.int64)
        for b, e in zip(cuts[:-1], cuts[1:]):
            diff += tfgpu.filter_resident(dict(p, out_row_begin=b, out_row_end=e), ids)[1]
            tfgpu.download_output(out, b, e)
        assert (diff == g["diff"]).all()
        assert all((a == b).all() for a, b in zip(_planes(out), g["out"]))
    finally:
        for i in ids:
            tfgpu.evict_frame(i)
    return g


@pytest.mark.parametrize("case", _coded.CASES, ids=[c[0] for c in _coded.CASES])
def test_filter_equals_oracle(pkg, tfgpu, case):
    p, frames = _coded.case_params(case), _coded.case_frames(case)
    _filter_case(pkg, tfgpu, p, frames, case[10], 7100000 + 100 * _coded.CASES.index(case))


@pytest.mark.parametrize("border", _coded.BORDERS)
@pytest.mark.parametrize("size", _coded.BORDER_SIZES, ids=[f"{s[0]}x{s[1]}" for s in _coded.BORDER_SIZES])
def test_border_filter_equals_oracle(pkg, tfgpu, size, border):
    W, H, rows = size
    p = _coded.border_params(W, H, border, N)
    frames = _coded.frames("large_motion", W, H, N, 8)
    _filter_case(pkg, tfgpu, p, frames, rows, 7200000 + 10 * border + (W > 640))


def test_zero_coded_size_equals_explicit_crop_size(pkg, tfgpu):
    case = _coded.CASES[3]
    p, frames = _coded.case_params(case), _coded.case_frames(case)
    base = dict(p, cm_width=0, cm_height=0)
    del base["mi_rows"], base["mi_cols"]
    a = _gpu.run_gpu(pkg, tfgpu, base, frames)
    b = _gpu.run_gpu(pkg, tfgpu, dict(base, cm_width=p["width"], cm_height=p["height"],
                                      mi_rows=_coded.align8(p["height"]) // 4, mi_cols=_coded.align8(p["width"]) // 4),
                     frames)
    for k in ("mvs", "mses", "pred", "accum", "count", "diff"):
        assert (a[k] == b[k]).all(), k
    assert all((x == y).all() for x, y in zip(a["out"], b["out"]))
    c = _gpu.run_gpu(pkg, tfgpu, p, frames)  # the coded size of the case changes the result
    assert not (c["mvs"] == a["mvs"]).all()


def test_batch_windows_with_different_coded_sizes(pkg, tfgpu):
    """One batch over one set of 1280x720 frames whose windows differ in coded size, grid and border: each window
    equals its single-window call."""
    W, H = 1280, 720
    frames = _coded.frames("large_motion", W, H, N, 10, seed=5)
    base = _coded.border_params(W, H, 160, N, bd=10, speed=3)
    windows = [
        _coded.coded_params(W, H, 640, 360, N, border=160, bit_depth=10, speed=3),
        _coded.coded_params(W, H, 960, 540, N, border=288, bit_depth=10, speed=3),
        dict(base, border=40),
        dict(base, border=47, cm_width=1280, cm_height=479, mi_rows=120, mi_cols=320),
        base,
    ]
    bufs = _bufs(pkg, base, frames, 7300000)
    for b in bufs:
        tfgpu.cache_frame(b)
    ids = [b.frame_id for b in bufs]
    try:
        _, diffs = tfgpu.filter_batch(windows, [ids] * len(windows))
        got = []
        for w in range(len(windows)):
            out = pkg.Yv12Buffer(W, H, 1, 1, True, 160)
            tfgpu.download_batch_output(w, out)
            got.append(_planes(out))
        for w, wp in enumerate(windows):
            _, d = tfgpu.filter_resident(wp, ids)
            out = pkg.Yv12Buffer(W, H, 1, 1, True, 160)
            tfgpu.download_output(out)
            assert (d == diffs[w]).all(), w
            assert all((a == b).all() for a, b in zip(_planes(out), got[w])), w
        # the two coded sizes change the result against the crop size's
        assert (diffs[0] != diffs[4]).any() and (diffs[1] != diffs[4]).any()
    finally:
        for i in ids:
            tfgpu.evict_frame(i)


def _grid_items(rng, p, bsize, cap=MAX_ORACLE_ITEMS):
    """Every bsize position (16 px in x, bsize in y) of the coded grid, from zero or random starts, ref drawn."""
    gw, gh = p["mi_cols"] * 4, p["mi_rows"] * 4
    xs, ys = list(range(0, gw, 16)), list(range(0, gh, bsize))
    items = [(x, y, 0 if k % 2 else int(rng.integers(-60, 61)), 0 if k % 2 else int(rng.integers(-60, 61)),
              int(rng.integers(0, N - 1))) for k, (y, x) in enumerate((y, x) for y in ys for x in xs)]
    if len(items) > cap:
        edge = [i for i, it in enumerate(items) if it[0] == xs[-1] or it[1] == ys[-1]]
        keep = sorted(set(rng.choice(len(items), cap, replace=False).tolist()) | set(edge))
        items = [items[i] for i in keep]
    return np.array(items, np.int64)


MOTION_CASES = list(_coded.CASES) + [
    ("g_360_b40", (640, 360), (640, 360), 40, 8, 0, 2, 1, 0, "large_motion", None, ()),
    ("g_360_b48", (640, 360), (640, 360), 48, 8, 0, 4, 0, 0, "large_motion", None, ()),
]


@pytest.mark.parametrize("bsize", [16, 32])
@pytest.mark.parametrize("case", MOTION_CASES, ids=[c[0] for c in MOTION_CASES])
def test_searches_equal_oracle(pkg, tfgpu, case, bsize):
    """motion_search_batch and motion_search_tensors against tfo_motion_search on all six fields, and
    fullpel_search_batch against tfo_full_pixel_search (200 of the items), on every position of the coded grid.
    Items past the coded grid but inside the frame fail the synchronous call and come back rejected from the device
    call."""
    import torch
    p, frames = _coded.case_params(case), _coded.case_frames(case)
    rng = np.random.default_rng(_coded.CASES.index(case) * 10 + bsize if case in _coded.CASES else bsize)
    items = _grid_items(rng, p, bsize)
    bufs = _bufs(pkg, p, frames, 7400000 + 100 * MOTION_CASES.index(case) + bsize)
    for b in bufs:
        tfgpu.cache_frame(b)
    ids = [b.frame_id for b in bufs]
    src, refs = ids[0], ids[1:]
    try:
        got = tfgpu.motion_search_batch(p, src, refs, bsize, items)
        dev = tfgpu.motion_search_tensors(p, src, refs, bsize, torch.from_numpy(items).cuda())
        assert (dev.cpu().numpy() == got).all()
        o = _oracle_motion.MotionOracle(p, frames)
        _oracle_motion.reset_stats()
        bad = []
        for it, g in zip(items.tolist(), got.tolist()):
            want = o.motion_search(0, 1 + it[4], bsize, *it[:4])
            if tuple(g) != want:
                bad.append((it, tuple(g), want))
        st = _oracle_motion.get_stats()
        o.close()
        assert not bad, (len(bad), len(items), bad[:5])
        if case[2] != case[1]:
            assert st["start_clamped"] > 0, st  # starts outside the shrunk limits
        if bsize == 32 and case[3] is not None and case[3] < 48:
            assert st["lim_border_bound"] > 0, st
        # the full-pel search alone, on host frames
        of = _oracle.OracleFilter(dict(p, num_frames=N, filter_frame_idx=0), frames)
        sub = rng.choice(len(items), min(len(items), 200), replace=False)
        for r in range(N - 1):
            sel = sub[items[sub, 4] == r]
            fp = tfgpu.fullpel_search_batch(p, bufs[0], bufs[1 + r], bsize, items[sel, :4].tolist())
            want = np.array([of.full_pixel_search(0, 1 + r, bsize, *it[:4]) for it in items[sel].tolist()],
                            np.int64).reshape(len(sel), 3)
            assert (fp == want).all(), r
            assert (fp == got[sel, :3]).all(), r
        of.close()
        # past the coded grid, inside the frame
        gw, gh = p["mi_cols"] * 4, p["mi_rows"] * 4
        outside = [(x, y, 0, 0, 0) for x, y in ((gw + 16 - gw % 16 if gw % 16 else gw, 0), (0, gh))
                   if x + 1 <= _coded.align8(p["width"]) and y + 1 <= _coded.align8(p["height"])]
        for it in outside:
            with pytest.raises(pkg.TfGpuError) as e:
                tfgpu.motion_search_batch(p, src, refs, bsize, [it])
            assert e.value.code == -1
            r = tfgpu.motion_search_tensors(p, src, refs, bsize, torch.tensor([list(items[0]), it]).cuda()).cpu()
            assert int(r[1, 2]) == pkg.TF_GPU_MOTION_REJECTED and int(r[1, 5]) == 2 ** 32 - 1
            assert (r[0].numpy() == got[0]).all()
        assert outside or case[2] == case[1]
    finally:
        for i in ids:
            tfgpu.evict_frame(i)


def test_grid_past_the_frame_is_rejected(pkg, tfgpu):
    """A grid larger than the frames' aligned size (by one mi unit, or far enough to overflow mi * 4) is rejected
    by every entry point with nothing enqueued, and the context then filters as a fresh one does."""
    case = _coded.CASES[5]
    p, frames = _coded.case_params(case), _coded.case_frames(case)
    aw, ah = _coded.align8(p["width"]), _coded.align8(p["height"])
    bufs = _bufs(pkg, p, frames, 7500000)
    for b in bufs:
        tfgpu.cache_frame(b)
    ids = [b.frame_id for b in bufs]
    bad = [dict(p, mi_rows=ah // 4 + 1), dict(p, mi_cols=aw // 4 + 1), dict(p, mi_cols=1 << 30),
           dict(p, mi_rows=(1 << 30) + 1), dict(p, mi_rows=(1 << 31) - 1)]
    try:
        for q in bad:
            calls = [lambda: _gpu.run_gpu(pkg, tfgpu, q, frames),
                     lambda: tfgpu.filter_resident(q, ids),
                     lambda: tfgpu.filter_batch([p, q], [ids, ids]),
                     lambda: tfgpu.fullpel_search_batch(q, bufs[0], bufs[1], 16, [(0, 0, 0, 0)]),
                     lambda: tfgpu.motion_search_batch(q, ids[0], ids[1:], 32, [(0, 0, 0, 0, 0)])]
            for k, call in enumerate(calls):
                with pytest.raises(pkg.TfGpuError) as e:
                    call()
                assert e.value.code == -1, (q["mi_rows"], q["mi_cols"], k)
    finally:
        for i in ids:
            tfgpu.evict_frame(i)
    a = _gpu.run_gpu(pkg, tfgpu, p, frames)
    fresh = pkg.TemporalFilterGpu()
    try:
        b = _gpu.run_gpu(pkg, fresh, p, frames)
    finally:
        fresh.close()
    for k in ("mvs", "mses", "pred", "accum", "count", "diff"):
        assert (a[k] == b[k]).all(), k
    assert all((x == y).all() for x, y in zip(a["out"], b["out"]))
