"""GPU: several windows over one frame cache in one call (tf_gpu_filter_batch_async, TemporalFilterGpu.filter_batch*).
Every window of a batch must equal the same window filtered alone (filter_resident) in the same context, bit for
bit on every output plane (full blocks) and on FRAME_DIFF; sampled block rows at 1080p and 4K equal the oracle.
Also: windows that differ in every per-window parameter, a sliding window over a clip, separate outputs, launch
counts, determinism, rejections and the tensor API."""
import ctypes as C

import numpy as np
import pytest
import torch

import _clips
import _oracle
import _params

pytestmark = pytest.mark.gpu


def _cache(pkg, ctx, p, frames, base_id):
    """Upload the frames under ids base_id, base_id + 1, ...; returns the ids."""
    ids = []
    for i, planes in enumerate(frames):
        b = pkg.Yv12Buffer(p["width"], p["height"], p["ss_x"], p["ss_y"], p["use_hbd"], p["border"], p["monochrome"],
                           frame_id=base_id + i)
        b.set_planes(*planes, extend=False)
        ctx.cache_frame(b)
        ids.append(base_id + i)
    return ids


def _out_buf(pkg, p):
    return pkg.Yv12Buffer(p["width"], p["height"], p["ss_x"], p["ss_y"], p["use_hbd"], p["border"], p["monochrome"])


def _planes(b):
    return [b.full_blocks(pl).copy() for pl in range(b.num_planes)]


def _single(pkg, ctx, p, ids):
    _, diff = ctx.filter_resident(p, ids)
    o = _out_buf(pkg, p)
    ctx.download_output(o)
    return _planes(o), diff


def _batch(pkg, ctx, ps, idss):
    _, diffs = ctx.filter_batch(ps, idss)
    outs = []
    for w, p in enumerate(ps):
        o = _out_buf(pkg, p)
        ctx.download_batch_output(w, o)
        outs.append(_planes(o))
    return outs, diffs


def _assert_equal(got, want, what):
    (gp, gd), (wp, wd) = got, want
    assert (np.asarray(gd) == np.asarray(wd)).all(), (what, gd, wd)
    assert len(gp) == len(wp)
    for pl, (a, b) in enumerate(zip(gp, wp)):
        assert (a == b).all(), (what, pl, int((a != b).sum()))


def _windows(p, ids):
    """Windows over one 7-frame clip that differ in every per-window parameter: the whole clip around its centre,
    a 5-frame window filtering its first frame, a 4-frame window filtering its last, and a single frame."""
    return [
        (dict(p), ids),
        (dict(p, num_frames=5, filter_frame_idx=0, filter_strength=3, q_factor=60, noise_levels=(4.5, 0.5, 2.0)),
         ids[1:6]),
        (dict(p, num_frames=4, filter_frame_idx=3, filter_strength=6, q_factor=140, compute_frame_diff=0), ids[3:7]),
        (dict(p, num_frames=1, filter_frame_idx=0, noise_levels=(1.0, 1.0, 1.0)), ids[2:3]),
    ]


# (W, H, bit depth, ss_x, ss_y, monochrome, parameter overrides)
CASES = {
    "8bit_420": (352, 288, 8, 1, 1, 0, {}),
    "10bit_420": (352, 288, 10, 1, 1, 0, {}),
    "12bit_444": (200, 136, 12, 0, 0, 0, {}),
    "8bit_422": (352, 288, 8, 1, 0, 0, {}),
    "10bit_422": (200, 136, 10, 1, 0, 0, {}),
    "mono_8": (200, 136, 8, 1, 1, 1, {}),
    "odd_353x289_8": (353, 289, 8, 1, 1, 0, {}),
    "odd_353x289_10": (353, 289, 10, 1, 1, 0, {}),
    "force_integer_mv": (352, 288, 8, 1, 1, 0, {"force_integer_mv": 1}),
    "subpel_tree_speed0": (352, 288, 10, 1, 1, 0, {"speed": 0}),
    "subpel_pruned_speed3": (352, 288, 8, 1, 1, 0, {"speed": 3}),
    "mesh_speed2_allow_hp": (352, 288, 8, 1, 1, 0, {"speed": 2, "allow_hp": 1}),
    "skip_sad": (352, 288, 10, 1, 1, 0, {"use_downsampled_sad": 1}),
}


@pytest.mark.parametrize("case", sorted(CASES))
def test_batch_windows_equal_single_window_calls(pkg, tfgpu, case):
    W, H, bd, sx, sy, mono, over = CASES[case]
    frames = _clips.moving_texture(W, H, 7, bd, ss_x=sx, ss_y=sy, monochrome=bool(mono))
    p = _params.tf_params(W, H, 7, bit_depth=bd, ss_x=sx, ss_y=sy, monochrome=mono, **over)
    ids = _cache(pkg, tfgpu, p, frames, 930001)
    try:
        wins = _windows(p, ids)
        outs, diffs = _batch(pkg, tfgpu, [w[0] for w in wins], [w[1] for w in wins])
        for k, (wp, wids) in enumerate(wins):
            _assert_equal((outs[k], diffs[k]), _single(pkg, tfgpu, wp, wids), (case, k))
        assert (diffs[2] == 0).all()  # compute_frame_diff off
    finally:
        for i in ids:
            tfgpu.evict_frame(i)


@pytest.mark.parametrize("n", [1, 2, 16])
def test_batch_sizes(pkg, tfgpu, n):
    W, H, bd = 352, 288, 8
    frames = _clips.moving_texture(W, H, 9, bd, seed=11)
    p = _params.tf_params(W, H, 5, bit_depth=bd)
    ids = _cache(pkg, tfgpu, p, frames, 931001)
    try:
        wins = []
        for k in range(n):  # 5-frame windows sliding over the 9 frames, the filtered frame moving through them
            s = k % 5
            wins.append((dict(p, filter_frame_idx=k % 5, filter_strength=3 + k % 4), ids[s:s + 5]))
        outs, diffs = _batch(pkg, tfgpu, [w[0] for w in wins], [w[1] for w in wins])
        assert tfgpu.last_stats()[0] == 3
        for k, (wp, wids) in enumerate(wins):
            _assert_equal((outs[k], diffs[k]), _single(pkg, tfgpu, wp, wids), (n, k))
    finally:
        for i in ids:
            tfgpu.evict_frame(i)


ORACLE_CASES = [("1080p10_n11", 1920, 1080, 10, 11, 77), ("4k10_n15", 3840, 2160, 10, 15, 77)]


@pytest.mark.parametrize("wl", ORACLE_CASES, ids=[w[0] for w in ORACLE_CASES])
def test_full_size_batch_rows_against_oracle(pkg, wl):
    _, W, H, bd, N, seed = wl
    ctx = pkg.TemporalFilterGpu(device=0)
    try:
        frames = _clips.moving_texture(W, H, N + 2, bd, seed=seed)
        p = _params.tf_params(W, H, N, bit_depth=bd)
        ids = _cache(pkg, ctx, p, frames, 932001)
        wins = [(p, ids[:N], frames[:N]),
                (dict(p, filter_strength=4, q_factor=50, noise_levels=(3.0, 1.5, 1.5)), ids[2:], frames[2:])]
        outs, diffs = _batch(pkg, ctx, [w[0] for w in wins], [w[1] for w in wins])
        mb_rows = (H + 31) // 32
        for k, (wp, _, wf) in enumerate(wins):
            o = _oracle.OracleFilter(wp, wf)
            for r in ((0, mb_rows // 2) if k == 0 else (mb_rows // 3, mb_rows - 1)):
                ref = o.run(record=False, rows=(r, r + 1))
                for pl in range(3):
                    bh = 32 >> (1 if pl else 0)
                    want = ref["out"][pl][r * bh:(r + 1) * bh]
                    have = outs[k][pl][r * bh:(r + 1) * bh].astype(np.uint16)
                    assert (want == have).all(), (k, pl, r, int((want != have).sum()))
            o.close()
            _assert_equal((outs[k], diffs[k]), _single(pkg, ctx, wp, wins[k][1]), k)
    finally:
        ctx.close()


def _cuda(a):
    return None if a is None else torch.from_numpy(a.view(np.int16) if a.dtype == np.uint16 else a).cuda()


def test_sliding_window_over_a_clip(pkg):
    """12 frames, half uploaded from host memory and half ingested from CUDA tensors; a 5-frame window centred on
    every frame (clamped at the ends), all 12 in two batches.  The batches read the cached frames only: no frame is
    uploaded twice or evicted."""
    W, H, bd, T, N = 352, 288, 10, 12, 5
    ctx = pkg.TemporalFilterGpu(device=0, max_cached_frames=24)
    try:
        frames = _clips.moving_texture(W, H, T, bd, seed=21)
        p = _params.tf_params(W, H, N, bit_depth=bd)
        ids = [933001 + i for i in range(T)]
        bufs = {}
        for i, planes in enumerate(frames):
            if i % 2 == 0:
                b = pkg.Yv12Buffer(W, H, 1, 1, True, p["border"], frame_id=ids[i])
                b.set_planes(*planes, extend=False)
                ctx.cache_frame(b)
            else:
                ctx.cache_frame_tensor(ids[i], *[_cuda(a) for a in planes])
            bufs[ids[i]] = planes
        wins = []
        for c in range(T):
            s = min(max(c - N // 2, 0), T - N)
            wins.append((dict(p, filter_frame_idx=c - s), ids[s:s + N]))
        results = []
        for half in (wins[:6], wins[6:]):
            outs, diffs = _batch(pkg, ctx, [w[0] for w in half], [w[1] for w in half])
            assert ctx.last_stats()[0] == 3  # the three kernels, no upload
            results += list(zip(outs, diffs))
        for k, (wp, wids) in enumerate(wins):
            _assert_equal(results[k], _single(pkg, ctx, wp, wids), k)
        for i in ids:  # every frame still resident, once, with its own pixels
            got = ctx.debug_read_plane(pkg.Yv12Buffer(W, H, 1, 1, True, frame_id=i), 0, 0, 0, W, H)
            assert (got == bufs[i][0]).all(), i
    finally:
        ctx.close()


def test_batch_and_single_window_outputs_are_separate(pkg, tfgpu):
    W, H, bd = 352, 288, 8
    frames = _clips.moving_texture(W, H, 7, bd, seed=31)
    p = _params.tf_params(W, H, 7, bit_depth=bd)
    ids = _cache(pkg, tfgpu, p, frames, 934001)
    try:
        wins = _windows(p, ids)
        ps, idss = [w[0] for w in wins[1:3]], [w[1] for w in wins[1:3]]
        # single window, then a batch, then the single window's output
        _, sdiff = tfgpu.filter_resident(p, ids)
        want_single = _single(pkg, tfgpu, p, ids)
        tfgpu.filter_resident(p, ids)
        tfgpu.filter_batch(ps, idss)
        o = _out_buf(pkg, p)
        tfgpu.download_output(o)
        _assert_equal((_planes(o), sdiff), want_single, "single after batch")
        # a batch, then a single window, then the batch's outputs
        want_batch = _batch(pkg, tfgpu, ps, idss)
        tfgpu.filter_batch(ps, idss)
        tfgpu.filter_resident(wins[3][0], wins[3][1])
        for w in range(2):
            o = _out_buf(pkg, ps[w])
            tfgpu.download_batch_output(w, o)
            _assert_equal((_planes(o), want_batch[1][w]), (want_batch[0][w], want_batch[1][w]), ("batch after single", w))
    finally:
        for i in ids:
            tfgpu.evict_frame(i)


def test_launch_counts_and_determinism(pkg, tfgpu):
    W, H, bd = 352, 288, 8
    frames = _clips.moving_texture(W, H, 7, bd, seed=41)
    p = _params.tf_params(W, H, 7, bit_depth=bd)
    ids = _cache(pkg, tfgpu, p, frames, 935001)
    try:
        wins = _windows(p, ids)
        ps, idss = [w[0] for w in wins], [w[1] for w in wins]
        a = _batch(pkg, tfgpu, ps, idss)
        assert tfgpu.last_stats()[0] == 3
        b = _batch(pkg, tfgpu, ps, idss)
        for w in range(len(ps)):
            _assert_equal((a[0][w], a[1][w]), (b[0][w], b[1][w]), ("determinism", w))
        # no 16x16 task in any window: the 16x16 launch is skipped
        ints = [dict(q, force_integer_mv=1) for q in ps]
        _batch(pkg, tfgpu, ints, idss)
        assert tfgpu.last_stats()[0] == 2
        _batch(pkg, tfgpu, [ints[0], ps[3]], [idss[0], idss[3]])
        assert tfgpu.last_stats()[0] == 2
        # no reference frame in any window: only the filter kernel
        singles = [dict(p, num_frames=1, filter_frame_idx=0) for _ in range(3)]
        outs, _ = _batch(pkg, tfgpu, singles, [[i] for i in ids[:3]])
        assert tfgpu.last_stats()[0] == 1
        for w in range(3):  # a window of one frame returns the frame
            fr = frames[w]
            for pl in range(3):
                assert (outs[w][pl][:fr[pl].shape[0], :fr[pl].shape[1]] == fr[pl]).all(), (w, pl)
    finally:
        for i in ids:
            tfgpu.evict_frame(i)


def _raw_batch(ctx, params_list, ids_list, n=None):
    """tf_gpu_filter_batch_async without the Python checks: (return code, error message)."""
    params_t = ctx.lib.tf_gpu_filter_batch_async.argtypes[2]._type_
    cps = (params_t * max(len(params_list), 1))(*params_list)
    arrs = [(C.c_uint64 * max(len(x), 1))(*x) for x in ids_list]
    ptrs = (C.POINTER(C.c_uint64) * max(len(arrs), 1))(*[C.cast(a, C.POINTER(C.c_uint64)) for a in arrs])
    rc = ctx.lib.tf_gpu_filter_batch_async(ctx.h, len(params_list) if n is None else n, cps, ptrs)
    return rc, (ctx.lib.tf_gpu_last_error(ctx.h) or b"").decode()


def test_rejections_leave_the_context_usable(pkg):
    W, H, bd = 352, 288, 8
    ctx = pkg.TemporalFilterGpu(device=0, max_cached_frames=24)
    try:
        frames = _clips.moving_texture(W, H, 7, bd, seed=51)
        p = _params.tf_params(W, H, 7, bit_depth=bd)
        ids = _cache(pkg, ctx, p, frames, 936001)
        other = _params.tf_params(200, 136, 1, bit_depth=bd)
        oid = _cache(pkg, ctx, other, _clips.moving_texture(200, 136, 1, bd), 936101)[0]
        ps, idss = [p, dict(p, num_frames=3, filter_frame_idx=1)], [ids, ids[2:5]]
        want = _batch(pkg, ctx, ps, idss)
        cp = pkg.make_params(p)
        lib, h = ctx.lib, ctx.h

        def err():
            return (lib.tf_gpu_last_error(h) or b"").decode()

        def check(rc, msg):
            assert rc == -1, (rc, msg)
            assert msg in err(), (msg, err())

        check(_raw_batch(ctx, [cp], [ids], n=0)[0], "batch of 0 windows out of [1,16]")
        check(_raw_batch(ctx, [cp] * 17, [ids] * 17)[0], "batch of 17 windows out of [1,16]")
        arr = (C.c_uint64 * 7)(*ids)
        ptrs = (C.POINTER(C.c_uint64) * 1)(C.cast(arr, C.POINTER(C.c_uint64)))
        check(lib.tf_gpu_filter_batch_async(h, 1, None, ptrs), "params / frame_ids is NULL")
        check(lib.tf_gpu_filter_batch_async(h, 1, (pkg.Params * 1)(cp), None), "params / frame_ids is NULL")
        check(lib.tf_gpu_filter_batch_async(h, 1, (pkg.Params * 1)(cp), (C.POINTER(C.c_uint64) * 1)()),
              "frame_ids[0] is NULL")
        check(_raw_batch(ctx, [cp, cp], [ids, ids[:6] + [999999]])[0], "window 1: frame id 999999 is not resident")
        check(_raw_batch(ctx, [cp, pkg.make_params(dict(p, num_frames=1, filter_frame_idx=0))], [ids, [oid]])[0],
              "window 1: the frames of a batch must share one geometry")
        many = [pkg.make_params(_params.tf_params(W, H, 15, bit_depth=bd))] * 2
        check(_raw_batch(ctx, many, [list(range(1, 16)), list(range(101, 116))])[0],
              "the batch reads 30 distinct frames, the frame cache holds 24")
        check(_raw_batch(ctx, [pkg.make_params(dict(p, out_row_begin=0, out_row_end=3))], [ids])[0],
              "window 0: a batch filters whole frames")
        check(_raw_batch(ctx, [cp, pkg.make_params(dict(p, extend_output_borders=1))], [ids, ids])[0],
              "window 1: a batch does not extend output borders")
        check(_raw_batch(ctx, [pkg.make_params(dict(p, filter_frame_idx=7))], [ids])[0], "filter_frame_idx out of range")
        ctx.collect_counters(True)
        check(_raw_batch(ctx, [cp], [ids])[0], "work counters are not collected for batches")
        ctx.collect_counters(False)
        check(lib.tf_gpu_download_batch_output(h, 2, C.byref(_out_buf(pkg, p).c_frame())),
              "window 2 is not in the last batch (2 windows)")
        with pytest.raises(ValueError):
            ctx.filter_batch([p] * 17, [ids] * 17)
        # the context still filters, and the outputs of the last good batch survived the rejections
        for w in range(2):
            o = _out_buf(pkg, ps[w])
            ctx.download_batch_output(w, o)
            _assert_equal((_planes(o), want[1][w]), (want[0][w], want[1][w]), ("kept", w))
        again = _batch(pkg, ctx, ps, idss)
        for w in range(2):
            _assert_equal((again[0][w], again[1][w]), (want[0][w], want[1][w]), ("after", w))
    finally:
        ctx.close()


def test_filter_batch_tensors_equal_download(pkg, tfgpu):
    W, H, bd = 353, 289, 10
    frames = _clips.moving_texture(W, H, 7, bd, seed=61)
    p = _params.tf_params(W, H, 7, bit_depth=bd)
    ids = _cache(pkg, tfgpu, p, frames, 937001)
    try:
        wins = _windows(p, ids)
        ps, idss = [w[0] for w in wins], [w[1] for w in wins]
        res = tfgpu.filter_batch_tensors(ps, idss)
        for w, (planes, diff) in enumerate(res):
            o = _out_buf(pkg, ps[w])
            tfgpu.download_batch_output(w, o)
            _, diffs = tfgpu.filter_batch_result(len(ps))
            assert (diff == diffs[w]).all()
            for pl, t in enumerate(planes):
                g = t.cpu().numpy().view(np.uint16)
                assert g.shape == (((H + 1) >> 1, (W + 1) >> 1) if pl else (H, W))
                assert (g == o.plane(pl)[:g.shape[0], :g.shape[1]]).all(), (w, pl)
    finally:
        for i in ids:
            tfgpu.evict_frame(i)


_PEER_CHILD = r"""
import sys
sys.path[:0] = [sys.argv[1], sys.argv[1] + "/tests"]
import conftest, _clips, _params
pkg = conftest.load_package()
handle, off, pitch = bytes.fromhex(sys.argv[2]), int(sys.argv[3]), int(sys.argv[4])
ctx = pkg.TemporalFilterGpu(device=0)
p = _params.tf_params(352, 288, 3)
ids = []
for i, planes in enumerate(_clips.moving_texture(352, 288, 3, 8, seed=71)):
    b = pkg.Yv12Buffer(352, 288, 1, 1, False, p["border"], frame_id=938001 + i)
    b.set_planes(*planes, extend=False)
    ctx.cache_frame(b)
    ids.append(938001 + i)
ctx.filter_batch([p], [ids])
ctx.output_ipc_import(0, handle, off, pitch)
try:
    ctx.filter_batch([p], [ids])
    print("accepted")
except pkg.TfGpuError as e:
    print("rejected", e.code, e)
ctx.output_ipc_import(0, None)
print("after", ctx.filter_batch([p], [ids])[1].tolist())
ctx.close()
"""


def test_batch_rejects_imported_peer_output(pkg):
    """An output plane imported from another process (slab mode over peer memory) is refused by a batch, which writes
    only its own outputs.  CUDA IPC handles cannot be opened in the process that exported them, so the importing
    context lives in a child process on the same GPU."""
    import os
    import subprocess
    import sys
    W, H = 352, 288
    owner = pkg.TemporalFilterGpu(device=0)
    try:
        p = _params.tf_params(W, H, 3)
        ids = _cache(pkg, owner, p, _clips.moving_texture(W, H, 3, 8, seed=71), 938001)
        owner.filter_resident(p, ids)  # the owner's output planes exist
        handle, off, pitch = owner.output_ipc_export(0)
        root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
        r = subprocess.run([sys.executable, "-c", _PEER_CHILD, root, handle.hex(), str(off), str(pitch)],
                           capture_output=True, text=True, timeout=300)
        assert r.returncode == 0, r.stderr[-2000:]
        lines = r.stdout.strip().splitlines()
        assert lines[0].startswith("rejected -1"), lines
        assert "imported from another rank" in lines[0], lines
        assert lines[1].startswith("after"), lines
        _, diff = owner.filter_resident(p, ids)
        assert lines[1] == "after " + str([diff.tolist()])
    finally:
        owner.close()


def test_luma_only_window_exposes_only_its_plane(pkg, tfgpu):
    """A window with num_planes = 1 over 4:2:0 frames writes luma only: its output has no chroma plane to hand out,
    and its luma equals the single-window call.  filter_batch_result never reads past the last batch's windows."""
    W, H, bd = 352, 288, 8
    frames = _clips.moving_texture(W, H, 5, bd, seed=81)
    p = _params.tf_params(W, H, 5, bit_depth=bd)
    ids = _cache(pkg, tfgpu, p, frames, 939001)
    try:
        lp = pkg.make_params(p)
        lp.num_planes = 1
        _, diffs = tfgpu.filter_batch([p, lp], [ids, ids])
        assert tfgpu.batch_output_device_plane(1, 0)[0]
        for pl in (1, 2):
            assert tfgpu.batch_output_device_plane(0, pl)[0]
            with pytest.raises(pkg.TfGpuError, match=f"window 1 filters 1 plane\\(s\\): no plane {pl}"):
                tfgpu.batch_output_device_plane(1, pl)
        y = pkg.Yv12Buffer(W, H, 1, 1, False, p["border"], monochrome=True)
        tfgpu.download_batch_output(1, y)
        _, single_diff = tfgpu.filter_resident(lp, ids)
        full = _out_buf(pkg, p)  # the single-window output holds every plane of the frames
        tfgpu.download_output(full)
        assert (y.full_blocks(0) == full.full_blocks(0)).all()
        assert (diffs[1] == single_diff).all()
        _, first = tfgpu.filter_batch_result(1)
        assert first.shape == (1, 2) and (first[0] == diffs[0]).all()
    finally:
        for i in ids:
            tfgpu.evict_frame(i)
