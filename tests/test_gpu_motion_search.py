"""GPU: tf_gpu_motion_search_batch -- tf_motion_search()'s per-block search (av1_full_pixel_search, then
find_fractional_mv_step to 1/8 pel, or the variance at the full-pel MV under force_integer_mv) over resident frames
against several references in one launch -- equal on all six result fields to the oracle's tfo_motion_search (tests/_oracle_motion.c),
which is composed of the pinned full-pel and sub-pel searches (test_oracle_motion_search.py).  Also equal to the library's
own paths: the full-pel fields to tf_gpu_fullpel_search_batch, the results on 32x32 blocks and their 16x16
sub-blocks to what the temporal filter records for the first frame of a window.  Then the call's own properties:
several references in one call, tensor-ingested frames, repeatability, launch count, and the rejections."""
import ctypes as C

import numpy as np
import pytest

import _clips
import _content
import _oracle_motion
import _params

pytestmark = pytest.mark.gpu

MAX_ORACLE_ITEMS = 300  # the oracle runs one block at a time on the CPU


def _bufs(pkg, p, frames, id_base):
    return [pkg.Yv12Buffer(p["width"], p["height"], p["ss_x"], p["ss_y"], p["use_hbd"], p["border"],
                           frame_id=id_base + i).set_planes(*f) for i, f in enumerate(frames)]


def _items(rng, W, H, bsize, motions, cap=MAX_ORACLE_ITEMS):
    """Every block of the bsize grid (16x16 on 16-px steps, 32x32 on 32-px steps; frame edges included), each with a
    start (zero, near the true motion of its reference, random in +-40) and a reference drawn at random."""
    aw, ah = -(-W // 8) * 8, -(-H // 8) * 8
    items = []
    for y in range(0, ah, bsize):
        for x in range(0, aw, bsize):
            ref = int(rng.integers(0, len(motions)))
            kind = int(rng.integers(0, 3))
            if kind == 0:
                sr, sc = 0, 0
            elif kind == 1:
                sr, sc = (int(round(m)) + int(rng.integers(-2, 3)) for m in motions[ref])
            else:
                sr, sc = int(rng.integers(-40, 41)), int(rng.integers(-40, 41))
            items.append((x, y, sr, sc, ref))
    if len(items) > cap:
        keep = sorted(set(rng.choice(len(items), cap, replace=False).tolist()) | {0, len(items) - 1})
        items = [items[i] for i in keep]
    return np.array(items, np.int64)


def _compare_with_oracle(pkg, tfgpu, p, frames, bsize, items, id_base):
    """frames[0] is the source, frames[1:] the references; items' ref indexes frames[1:]."""
    bufs = _bufs(pkg, p, frames, id_base)
    for b in bufs:
        tfgpu.cache_frame(b)
    try:
        got = tfgpu.motion_search_batch(p, bufs[0].frame_id, [b.frame_id for b in bufs[1:]], bsize, items)
    finally:
        for b in bufs:
            tfgpu.evict_frame(b.frame_id)
    o = _oracle_motion.MotionOracle(dict(p, num_frames=len(frames), filter_frame_idx=0), frames)
    bad = []
    for it, g in zip(items.tolist(), got.tolist()):
        want = o.motion_search(0, 1 + it[4], bsize, *it[:4])
        if tuple(g) != want:
            bad.append((it, tuple(g), want))
    o.close()
    assert not bad, (len(bad), len(items), bad[:5])
    return got


# name, W, H, bit depth, high-bitdepth container, speed, allow_hp, force_integer_mv
CASES = [
    ("cif8_s4", 352, 288, 8, 0, 4, 0, 0),
    ("cif10_s2_hp", 352, 288, 10, 1, 2, 1, 0),
    ("cif12_s0_hp", 352, 288, 12, 1, 0, 1, 0),      # TREE, 2 iterations per step
    ("cif8in16_s3", 352, 288, 8, 1, 3, 1, 0),       # 8-bit samples in a 16-bit container; PRUNED
    ("hd8_s4_hp", 1280, 720, 8, 0, 4, 1, 0),        # >= 720p: skip-row SAD and its audit
    ("hd10_s0", 1280, 720, 10, 1, 0, 0, 0),
    ("hd12_s2_hp", 1280, 720, 12, 1, 2, 1, 0),
    ("odd8_s2_hp", 200, 136, 8, 0, 2, 1, 0),
    ("odd10_s4", 216, 120, 10, 1, 4, 0, 0),
    ("cif8_fim", 352, 288, 8, 0, 4, 0, 1),
    ("hd10_s0_fim", 1280, 720, 10, 1, 0, 1, 1),
]
MOTION = (2, 3)  # per frame of _clips.moving_texture: the source is frame 1, the references frames 0, 2 and 3


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
@pytest.mark.parametrize("bsize", [16, 32])
def test_equals_oracle(pkg, tfgpu, case, bsize):
    name, W, H, bd, hbd, speed, hp, fim = case
    # whole-pixel motion plus per-frame noise (sub-pel motion: the content cases below)
    clip = _clips.moving_texture(W, H, 4, bd, motion=MOTION)
    frames = [clip[1], clip[0], clip[2], clip[3]]
    p = _params.tf_params(W, H, 4, bit_depth=bd, use_hbd=hbd, speed=speed, allow_hp=hp, force_integer_mv=fim)
    rng = np.random.default_rng(10 * CASES.index(case) + bsize)
    items = _items(rng, W, H, bsize, [((1 - k) * MOTION[0], (1 - k) * MOTION[1]) for k in (0, 2, 3)])
    got = _compare_with_oracle(pkg, tfgpu, p, frames, bsize, items, 910000 + 100 * CASES.index(case) + bsize)
    if fim:
        assert (got[:, 3] == 8 * got[:, 0]).all() and (got[:, 4] == 8 * got[:, 1]).all()


# class, W, H, bit depth, content options, parameter options, frame indices (source first)
CONTENT = [
    ("subpel_pan", 352, 288, 8, dict(velocity=(0.25, 0.5)), dict(speed=2, allow_hp=1), (2, 0, 1, 3)),
    ("subpel_pan", 352, 288, 10, dict(velocity=(1.375, -0.75)), dict(speed=0, allow_hp=1), (2, 0, 1, 3)),
    ("subpel_pan", 352, 288, 12, dict(velocity=(0.75, 0.25)), dict(speed=4, allow_hp=1), (2, 0, 1, 4)),
    ("periodic", 176, 144, 8, dict(kind="checker", period=8), {}, (2, 0, 1, 4)),
    ("periodic", 176, 144, 10, dict(kind="tile", period=12, motion=(3, 12)), dict(speed=0), (2, 0, 1, 4)),
    ("periodic", 176, 144, 12, dict(kind="grid", period=6), dict(speed=3), (2, 0, 1, 4)),
    ("tap_pattern", 176, 144, 10, dict(kind="columns"), dict(allow_hp=1), (1, 0, 2, 3)),
    ("tap_pattern", 176, 144, 12, dict(kind="noise"), dict(speed=2), (1, 0, 2, 3)),
    ("sharp_edges", 352, 288, 8, {}, dict(allow_hp=1), (2, 0, 1, 4)),
    ("sharp_edges", 352, 288, 12, {}, dict(speed=0), (2, 0, 1, 4)),
]


@pytest.mark.parametrize("t", CONTENT, ids=[f"{t[0]}-{t[3]}-{i}" for i, t in enumerate(CONTENT)])
@pytest.mark.parametrize("bsize", [16, 32])
def test_adversarial_content_equals_oracle(pkg, tfgpu, t, bsize):
    cls, W, H, bd, ckw, pkw, order = t
    clip = _content.make(cls, W, H, max(order) + 1, bd, **ckw)
    frames = [clip[i] for i in order]
    p = _params.tf_params(W, H, len(frames), bit_depth=bd, **pkw)
    v = ckw.get("velocity") or ckw.get("motion") or (0, 0)
    motions = [(-(i - order[0]) * v[0], -(i - order[0]) * v[1]) for i in order[1:]]
    rng = np.random.default_rng(CONTENT.index(t) * 10 + bsize)
    items = _items(rng, W, H, bsize, motions)
    got = _compare_with_oracle(pkg, tfgpu, p, frames, bsize, items, 920000 + 100 * CONTENT.index(t) + bsize)
    if cls == "subpel_pan":
        assert len(set((got[:, 3:5] & 7).ravel().tolist()) & {2, 4, 6}) >= 2  # quarter / half / 3/4-pel MVs


def test_large_motion_reaches_the_mv_clamp(pkg, tfgpu):
    """1080p pan of 150 px per frame: against frames 7..9 the true offset is 1050..1350 px, beyond the +-1023 clamp
    of the MV limits; items start near the true motion (clamped to int16 range) so the search ends on the clamp."""
    W, H, v = 1920, 1080, (2, 150)
    clip = _content.large_motion(W, H, 10, 10, velocity=v)
    order = (0, 7, 8, 9)
    frames = [clip[i] for i in order]
    p = _params.tf_params(W, H, 4, bit_depth=10)
    rng = np.random.default_rng(5)
    for bsize in (16, 32):
        items = _items(rng, W, H, bsize, [(-k * v[0], -k * v[1]) for k in order[1:]], cap=200)
        got = _compare_with_oracle(pkg, tfgpu, p, frames, bsize, items, 930000 + bsize)
        assert (np.abs(got[:, 1]) == 1023).any() and (np.abs(got[:, 4]) == 8 * 1023).any()


def test_fullpel_fields_equal_fullpel_search_batch(pkg, tfgpu):
    W, H = 640, 360
    frames = _clips.moving_texture(W, H, 4, 10, motion=(2, 3))
    p = _params.tf_params(W, H, 4, bit_depth=10, speed=2, allow_hp=1)
    bufs = _bufs(pkg, p, frames, 940000)
    for b in bufs:
        tfgpu.cache_frame(b)
    for bsize in (16, 32):
        items = _items(np.random.default_rng(bsize), W, H, bsize, [(-2 * k, -3 * k) for k in (1, 2, 3)], cap=10 ** 6)
        got = tfgpu.motion_search_batch(p, bufs[0].frame_id, [b.frame_id for b in bufs[1:]], bsize, items)
        for r in range(3):
            sel = items[:, 4] == r
            fp = tfgpu.fullpel_search_batch(p, bufs[0], bufs[1 + r], bsize, items[sel, :4].tolist())
            assert (got[sel, :3] == fp).all(), r
    for b in bufs:
        tfgpu.evict_frame(b.frame_id)


def _limits(x, y, bsize, mi_rows, mi_cols, border):
    """av1_set_mv_{row,col}_limits + the +-1023 clamp of a bsize block at (x, y) (tf_gpu.h, full-pel rule)."""
    mr, mc, m = y >> 2, x >> 2, bsize >> 2
    return (max(-(mr * 4 + border - 8), -((mr + m) * 4 + 8), -1023),
            min((mi_rows - mr - m) * 4 + border - 8, (mi_rows - mr) * 4 + 8, 1023),
            max(-(mc * 4 + border - 8), -((mc + m) * 4 + 8), -1023),
            min((mi_cols - mc - m) * 4 + border - 8, (mi_cols - mc) * 4 + 8, 1023))


def _rawpel(v):
    return (v + 3 + (v >= 0)) >> 3


def test_equals_temporal_filter_first_frame(pkg, tfgpu):
    """4K 8-bit window of three frames filtering frame 1 (sub-pel pan: the partition decision keeps some blocks
    whole and splits others): frame 0 is searched first, from a zero ref_mv.  Its 32x32
    blocks are motion searches from (0, 0), and each 16x16 sub-block a motion search from the full-pel rounding of
    its block's MV -- with the block's MV limits, which are the sub-block's own where the +-1023 clamp sets all four
    (at 4K the centre: 983 <= x, y and x, y <= size - 1015, 224 blocks).  There the recorded MVs / MSEs follow the
    partition decision (temporal_filter.c:270-292) exactly; every other block whose four records are one (MV, MSE)
    holds the 32x32 result, or is a split of four equal sub-blocks that the decision explains."""
    W, H = 3840, 2160
    frames = _content.subpel_pan(W, H, 3, 8, velocity=(0.75, -1.25))
    p = _params.tf_params(W, H, 3, filter_frame_idx=1, speed=2, allow_hp=1)
    bufs = _bufs(pkg, p, frames, 950000)
    out = pkg.Yv12Buffer(W, H, 1, 1, False, p["border"])
    dump = tfgpu.temporal_filter(p, bufs, out, dump=True)
    mvs, mses = dump["mvs"][:, 0], dump["mses"][:, 0]
    mb_cols = (W + 31) // 32
    cp = pkg.make_params(p)
    b32 = [(bc * 32, br * 32) for br in range((H + 31) // 32) for bc in range(mb_cols)]
    # blocks whose four sub-blocks have the block's own MV limits
    full = [b for b, (x, y) in enumerate(b32)
            if all(_limits(x + dx, y + dy, 16, cp.mi_rows, cp.mi_cols, p["border"])
                   == _limits(x, y, 32, cp.mi_rows, cp.mi_cols, p["border"]) for dy in (0, 16) for dx in (0, 16))]
    assert len(full) >= 200, len(full)
    r32 = tfgpu.motion_search_batch(p, bufs[1].frame_id, [bufs[0].frame_id], 32, [(x, y, 0, 0, 0) for x, y in b32])
    subs = [(b32[b][0] + dx, b32[b][1] + dy, _rawpel(int(r32[b, 3])), _rawpel(int(r32[b, 4])), 0)
            for b in full for dy in (0, 16) for dx in (0, 16)]
    r16 = tfgpu.motion_search_batch(p, bufs[1].frame_id, [bufs[0].frame_id], 16, subs).reshape(len(full), 4, 6)
    nosplit = bad = 0
    for k, b in enumerate(full):
        block_mv, block_mse = tuple(r32[b, 3:5]), (int(r32[b, 5]) + 512) // 1024
        sub_mv, sub_mse = r16[k, :, 3:5], (r16[k, :, 5] + 128) // 256
        s, lo, hi = int(sub_mse.sum()), int(sub_mse.min()), int(sub_mse.max())
        keep = (block_mse * 15 < s * 4 and hi - lo < 48) or (block_mse * 14 < s * 4 and hi - lo < 24)
        nosplit += keep
        want_mv = np.array([block_mv] * 4) if keep else sub_mv
        want_mse = np.array([block_mse] * 4) if keep else sub_mse
        bad += not ((mvs[b] == want_mv).all() and (mses[b] == want_mse).all())
    assert bad == 0, (bad, len(full))
    assert 0 < nosplit < len(full), (nosplit, len(full))
    fullset, same32 = set(full), 0
    for b in range(len(b32)):
        if b in fullset or not ((mvs[b] == mvs[b, :1]).all() and (mses[b] == mses[b, 0]).all()):
            continue
        block_mse = (int(r32[b, 5]) + 512) // 1024
        if tuple(mvs[b, 0]) == tuple(r32[b, 3:5]) and mses[b, 0] == block_mse:
            same32 += 1
        else:
            assert block_mse * 15 >= 16 * int(mses[b, 0]), (b, mvs[b], mses[b], r32[b])
    assert same32 > 0, (same32, len(b32))
    for b in bufs:
        tfgpu.evict_frame(b.frame_id)


@pytest.fixture(scope="module")
def resident(pkg, tfgpu):
    """A 640x360 8-bit source and three references, resident under ids 960000..960003."""
    W, H = 640, 360
    frames = _clips.moving_texture(W, H, 4, 8, motion=(1, 2))
    p = _params.tf_params(W, H, 4, speed=2, allow_hp=1)
    bufs = _bufs(pkg, p, frames, 960000)
    for b in bufs:
        tfgpu.cache_frame(b)
    yield p, frames, [b.frame_id for b in bufs]
    for b in bufs:
        tfgpu.evict_frame(b.frame_id)


def test_several_references_equal_one_call_per_reference(tfgpu, resident):
    p, _, ids = resident
    for bsize in (16, 32):
        items = _items(np.random.default_rng(bsize), 640, 360, bsize, [(-k, -2 * k) for k in (1, 2, 3)], cap=10 ** 6)
        got = tfgpu.motion_search_batch(p, ids[0], ids[1:], bsize, items)
        for r in range(3):
            sel = items[:, 4] == r
            one = items[sel].copy()
            one[:, 4] = 0
            assert (tfgpu.motion_search_batch(p, ids[0], [ids[1 + r]], bsize, one) == got[sel]).all(), r
        # a repeated reference, and the source as its own reference
        same = items.copy()
        same[:, 4] = 0
        a = tfgpu.motion_search_batch(p, ids[0], [ids[2], ids[0], ids[2]], bsize, same)
        same[:, 4] = 2
        assert (tfgpu.motion_search_batch(p, ids[0], [ids[2], ids[0], ids[2]], bsize, same) == a).all()
        zero = np.array([(x, y, 0, 0, 1) for x, y, *_ in items.tolist()])
        z = tfgpu.motion_search_batch(p, ids[0], [ids[2], ids[0], ids[2]], bsize, zero)
        assert (z[:, 3:5] == 0).all() and (z[:, 5] == 0).all()  # a block matches itself exactly at MV 0


def test_tensor_ingested_frames_equal_host_frames(pkg, tfgpu, resident):
    import torch
    p, frames, ids = resident
    tids = [961000 + i for i in range(4)]
    for fid, (y, u, v) in zip(tids, frames):
        tfgpu.cache_frame_tensor(fid, *(torch.from_numpy(np.ascontiguousarray(a)).cuda() for a in (y, u, v)))
    try:
        for bsize in (16, 32):
            items = _items(np.random.default_rng(7 + bsize), 640, 360, bsize, [(-k, -2 * k) for k in (1, 2, 3)],
                           cap=10 ** 6)
            host = tfgpu.motion_search_batch(p, ids[0], ids[1:], bsize, items)
            dev = tfgpu.motion_search_batch(p, tids[0], tids[1:], bsize, items)
            assert (host == dev).all()
    finally:
        for fid in tids:
            tfgpu.evict_frame(fid)


def test_repeatable_and_one_launch(tfgpu, resident):
    p, _, ids = resident
    items = _items(np.random.default_rng(3), 640, 360, 16, [(-k, -2 * k) for k in (1, 2, 3)], cap=10 ** 6)
    a = tfgpu.motion_search_batch(p, ids[0], ids[1:], 16, items)
    launches, ms = tfgpu.last_stats()
    assert launches == 1 and ms > 0
    for _ in range(3):
        assert (tfgpu.motion_search_batch(p, ids[0], ids[1:], 16, items) == a).all()
    assert tfgpu.motion_search_batch(p, ids[0], ids[1:], 16, []).shape == (0, 6)


def _raw_call(pkg, tfgpu, cp, src_id, ref_ids, num_refs, bsize, items, n, results=True):
    """tf_gpu_motion_search_batch without the Python-side checks; None stands for a NULL pointer."""
    ids = None if ref_ids is None else (C.c_uint64 * max(len(ref_ids), 1))(*ref_ids)
    arr = None if items is None else (pkg.MotionItem * max(len(items), 1))(*[pkg.MotionItem(*it) for it in items])
    res = (pkg.MotionResult * max(n, 1))() if results else None
    return tfgpu.lib.tf_gpu_motion_search_batch(tfgpu.h, None if cp is None else C.byref(cp), src_id, ids, num_refs,
                                                bsize, arr, n, res)


def test_rejections_leave_the_context_usable(pkg, tfgpu, resident):
    p, frames, ids = resident
    cp = pkg.make_params(p)
    ok = [(0, 0, 0, 0, 0)]
    assert _raw_call(pkg, tfgpu, cp, ids[0], ids[1:], 3, 16, ok, 1) == 0
    other = pkg.Yv12Buffer(352, 288, 1, 1, False, p["border"], frame_id=962000).set_planes(
        *_clips.moving_texture(352, 288, 1, 8)[0])
    tfgpu.cache_frame(other)
    bad = [
        (None, ids[0], ids[1:], 3, 16, ok, 1, True),             # NULL params
        (cp, ids[0], None, 3, 16, ok, 1, True),                  # NULL ref_ids
        (cp, ids[0], ids[1:], 3, 16, None, 1, True),             # NULL items
        (cp, ids[0], ids[1:], 3, 16, ok, 1, False),              # NULL results
        (cp, ids[0], ids[1:], 3, 24, ok, 1, True),               # block size
        (cp, ids[0], ids[1:], 3, 8, ok, 1, True),
        (cp, ids[0], ids[1:], 3, 16, ok, -1, True),              # n < 0
        (cp, ids[0], ids[1:], 0, 16, ok, 1, True),               # num_refs
        (cp, ids[0], list(range(1, 25)), 24, 16, ok, 1, True),
        (cp, 123456789, ids[1:], 3, 16, ok, 1, True),            # source not resident
        (cp, ids[0], [ids[1], 123456789], 2, 16, ok, 1, True),   # reference not resident
        (cp, ids[0], [ids[1], 0], 2, 16, ok, 1, True),           # id 0 is never resident
        (cp, ids[0], [ids[1], other.frame_id], 2, 16, ok, 1, True),  # mixed geometry
        (cp, ids[0], ids[1:], 3, 16, [(8, 0, 0, 0, 0)], 1, True),    # x not a multiple of 16
        (cp, ids[0], ids[1:], 3, 16, [(0, 2, 0, 0, 0)], 1, True),    # y not a multiple of 4
        (cp, ids[0], ids[1:], 3, 16, [(-16, 0, 0, 0, 0)], 1, True),
        (cp, ids[0], ids[1:], 3, 16, [(640, 0, 0, 0, 0)], 1, True),  # outside the mi grid
        (cp, ids[0], ids[1:], 3, 16, [(0, 360, 0, 0, 0)], 1, True),
        (cp, ids[0], ids[1:], 3, 16, [(0, 0, 0, 0, 3)], 1, True),    # ref out of [0, num_refs)
        (cp, ids[0], ids[1:], 3, 16, [(0, 0, 0, 0, 0), (0, 0, 0, 0, -1)], 2, True),
    ]
    for k, args in enumerate(bad):
        assert _raw_call(pkg, tfgpu, *args) == -1, k
    assert _raw_call(pkg, tfgpu, cp, ids[0], ids[1:], 3, 16, ok, 0) == 0  # n == 0
    tfgpu.evict_frame(other.frame_id)
    # the context filters as a fresh one does
    W, H = 352, 288
    clip = _clips.moving_texture(W, H, 3, 8)
    fp = _params.tf_params(W, H, 3)
    outs = []
    for ctx in (tfgpu, pkg.TemporalFilterGpu()):
        bufs = _bufs(pkg, fp, clip, 963000)
        out = pkg.Yv12Buffer(W, H, 1, 1, False, fp["border"])
        r = ctx.temporal_filter(fp, bufs, out, dump=True)
        outs.append((r, [out.full_blocks(pl).copy() for pl in range(3)]))
        for b in bufs:
            ctx.evict_frame(b.frame_id)
        if ctx is not tfgpu:
            ctx.close()
    (ra, oa), (rb, ob) = outs
    assert all((a == b).all() for a, b in zip(oa, ob))
    assert all((ra[k] == rb[k]).all() for k in ("diff", "mvs", "mses"))
