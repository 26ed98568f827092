"""GPU: tf_gpu_predict_device / TemporalFilterGpu.predict_tensors -- the temporal filter's 12-tap predictor at caller
MVs over resident frames, in device memory, on the caller's stream.  Equal to the filter's own predictor (the dump)
over the parity window cases and the adversarial content of test_gpu_motion_search.py; equal to the oracle's
tfo_predict_block at caller MVs up to the int16 extremes; chained on the device behind motion_search_tensors; the
source at MV 0 is the source block; stream order and slot lifetime; per-item rejection; host rejections."""
import ctypes as C

import numpy as np
import pytest

import _clips
import _content
import _gpu
import _oracle_predict
import _params
import test_gpu_motion_search as ms
from test_oracle_predict import _quadrant

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

SLEEP_CYCLES = 1_000_000_000  # torch.cuda._sleep: about half a second at B200 clocks


def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _flat(planes):
    """predict_tensors' planes -> uint16 numpy (n, num_pels) in the pred layout."""
    parts = [t.reshape(t.shape[0], -1).cpu().numpy() for t in planes]
    return np.concatenate([a.view(np.uint16) if a.dtype == np.int16 else a.astype(np.uint16) for a in parts], axis=1)


def _predict(tfgpu, p, ref_ids, bsize, items):
    planes, status = tfgpu.predict_tensors(p, ref_ids, bsize, _cuda(np.asarray(items, np.int64).reshape(-1, 5)))
    assert status.dtype == torch.int32 and len(planes) == (1 if p["monochrome"] else 3)
    assert tfgpu.last_stats() == (1, 0.0)
    return _flat(planes), status.cpu().numpy()


# name, W, H, N, bit depth, clip options, params options (the window cases of test_gpu_parity.py)
WINDOWS = [
    ("cif8", 352, 288, 5, 8, {}, {}),
    ("cif10_hp", 352, 288, 3, 10, dict(motion=(2, 1)), dict(allow_hp=1, speed=0)),
    ("bd12", 128, 96, 3, 12, {}, dict(speed=3, q_factor=15)),
    ("hbd8", 128, 96, 3, 8, {}, dict(use_hbd=1, allow_hp=1)),
    ("i444_8", 130, 70, 3, 8, {}, dict(ss_x=0, ss_y=0)),
    ("i422_10", 130, 70, 3, 10, {}, dict(ss_x=1, ss_y=0, speed=1)),
    ("mono8", 131, 77, 4, 8, {}, dict(monochrome=1, filter_frame_idx=3)),
    ("odd200x136_8", 200, 136, 3, 8, dict(motion=(3, 5)), dict(speed=2, allow_hp=1)),
    ("odd216x120_10", 216, 120, 3, 10, dict(motion=(1, 3)), dict(allow_hp=1)),
]


def _check_against_dump(pkg, tfgpu, p, frames, id_base):
    """Filter with the dump, then predict every (block, frame, quadrant) at the dumped MV from the frames the filter
    cached, and every block whose four MVs agree as one 32-item."""
    g = _gpu.run_gpu(pkg, tfgpu, p, frames, frame_id_base=id_base)
    N, fi = p["num_frames"], p["filter_frame_idx"]
    ids = [id_base + 1 + i for i in range(N)]
    mb_cols = (p["width"] + 31) // 32
    mi_rows, mi_cols = -(-p["height"] // 8) * 2, -(-p["width"] // 8) * 2
    np_ = 1 if p["monochrome"] else 3
    i16, want16, i32, want32 = [], [], [], []
    for blk in range(g["mvs"].shape[0]):
        by, bx = 32 * (blk // mb_cols), 32 * (blk % mb_cols)
        for f in range(N):
            mvs = g["mvs"][blk, f]
            entry = g["pred"][blk, f]
            if f == fi:  # the dump holds no predictor for the frame being filtered: its block at MV 0 is itself
                parts = []
                for pl in range(np_):
                    sx, sy = (p["ss_x"], p["ss_y"]) if pl else (0, 0)
                    parts.append(g["bufs"][f].plane(pl)[by >> sy:(by + 32) >> sy, bx >> sx:(bx + 32) >> sx].ravel())
                entry = np.concatenate(parts).astype(np.uint16)
                assert (mvs == 0).all()
            for q in range(4):
                x, y = bx + 16 * (q & 1), by + 16 * (q >> 1)
                if x < mi_cols * 4 and y < mi_rows * 4:  # the position rule; the 32-items cover the rest
                    i16.append((x, y, int(mvs[q, 0]), int(mvs[q, 1]), f))
                    want16.append(_quadrant(p, entry, np_, q))
            if (mvs == mvs[0]).all():
                i32.append((bx, by, int(mvs[0, 0]), int(mvs[0, 1]), f))
                want32.append(entry)
    try:
        got16, st16 = _predict(tfgpu, p, ids, 16, i16)
        got32, st32 = _predict(tfgpu, p, ids, 32, i32)
    finally:
        for i in ids:
            tfgpu.evict_frame(i)
    assert (st16 == 0).all() and (st32 == 0).all()
    bad = np.nonzero((got16 != np.array(want16)).any(axis=1))[0]
    assert len(bad) == 0, (len(bad), len(i16), [i16[k] for k in bad[:5]])
    bad = np.nonzero((got32 != np.array(want32)).any(axis=1))[0]
    assert len(bad) == 0, (len(bad), len(i32), [i32[k] for k in bad[:5]])
    return np.array(i16)


@pytest.mark.parametrize("case", WINDOWS, ids=[c[0] for c in WINDOWS])
def test_equals_the_filter_predictor(pkg, tfgpu, case):
    name, W, H, N, bd, ckw, pkw = case
    frames = _clips.moving_texture(W, H, N, bd, ss_x=pkw.get("ss_x", 1), ss_y=pkw.get("ss_y", 1),
                                   monochrome=pkw.get("monochrome", 0), **ckw)
    p = _params.tf_params(W, H, N, bit_depth=bd, **pkw)
    _check_against_dump(pkg, tfgpu, p, frames, 2_100_000 + 100 * WINDOWS.index(case))


@pytest.mark.parametrize("t", ms.CONTENT, ids=[f"{t[0]}-{t[3]}-{i}" for i, t in enumerate(ms.CONTENT)])
def test_adversarial_content_equals_the_filter_predictor(pkg, tfgpu, t):
    cls, W, H, bd, ckw, pkw, order = t
    clip = _content.make(cls, W, H, max(order) + 1, bd, **ckw)
    frames = [clip[i] for i in sorted(order)]
    p = _params.tf_params(W, H, len(frames), bit_depth=bd, **pkw)
    _check_against_dump(pkg, tfgpu, p, frames, 2_200_000 + 100 * ms.CONTENT.index(t))


def test_large_motion_to_the_clamp_equals_the_filter_predictor(pkg, tfgpu):
    W, H, v = 1920, 1080, (2, 150)
    clip = _content.large_motion(W, H, 10, 10, velocity=v)
    frames = [clip[i] for i in (0, 7, 8)]
    p = _params.tf_params(W, H, 3, bit_depth=10, filter_frame_idx=0)
    _check_against_dump(pkg, tfgpu, p, frames, 2_300_000)


# caller MVs: every 1/8 phase near the block, +-1 px .. +-4095.875 px, and origins between the device border (80)
# and the reference clamp (284) on every side
PHASES = [(r, c) for r in range(-4, 4) for c in range(-4, 4)]
FAR = [(8, -8), (-8, 8), (-800, 3), (5, -800), (-1600, -1601), (-2200, 13), (11, -2250), (800, 7), (6, 1600),
       (2200, 2201), (-32768, -32768), (32767, 32767), (-32768, 32767), (32767, -32768), (-23000, 900), (901, 31000)]


def _oracle_items(rng, W, H, bsize, num_refs):
    aw, ah = -(-W // 8) * 8, -(-H // 8) * 8
    last_x, last_y = (aw - 1) // 16 * 16, (ah - 1) // 4 * 4  # the last grid positions: the block runs past the frame
    pos = [(0, 0), (last_x, 0), (0, last_y), (last_x, last_y), (16, 4), (aw // 2 // 16 * 16, ah // 2 // 4 * 4)]
    mvs = PHASES + FAR + [tuple(int(v) for v in rng.integers(-32768, 32768, 2)) for _ in range(24)]
    return np.array([(x, y, r, c, int(rng.integers(0, num_refs))) for x, y in pos for r, c in mvs], np.int64)


# content, bit depth, subsampling, monochrome
ORACLE_CASES = [
    ("texture", 8, (1, 1), 0),
    ("texture", 10, (1, 0), 0),
    ("columns", 12, (1, 1), 0),  # int16 wrap of the 2-D intermediate
    ("noise", 12, (0, 0), 0),    # full-range binary noise: clipped predictor samples at both ends
    ("noise", 10, (1, 1), 1),
]


@pytest.mark.parametrize("case", ORACLE_CASES, ids=[f"{c[0]}{c[1]}-{c[2][0]}{c[2][1]}-m{c[3]}" for c in ORACLE_CASES])
@pytest.mark.parametrize("bsize", [16, 32])
def test_equals_the_oracle_at_caller_mvs(pkg, tfgpu, case, bsize):
    kind, bd, (ssx, ssy), mono = case
    W, H = 200, 136
    if kind == "texture":
        frames = _clips.moving_texture(W, H, 2, bd, ss_x=ssx, ss_y=ssy, monochrome=mono, motion=(2, 3))
    else:
        frames = _content.tap_pattern(W, H, 2, bd, ss_x=ssx, ss_y=ssy, monochrome=mono, kind=kind)
    p = _params.tf_params(W, H, 2, bit_depth=bd, ss_x=ssx, ss_y=ssy, monochrome=mono)
    bufs = [pkg.Yv12Buffer(W, H, ssx, ssy, p["use_hbd"], p["border"], mono, frame_id=2_400_000 + 10 * bsize + i)
            .set_planes(*f) for i, f in enumerate(frames)]
    for b in bufs:
        tfgpu.cache_frame(b)
    items = _oracle_items(np.random.default_rng(bd * 100 + bsize), W, H, bsize, 2)
    try:
        for num_planes in ((1,) if mono else (1, 3)):
            pp = dict(p, monochrome=int(num_planes == 1))
            got, status = _predict(tfgpu, pp, [b.frame_id for b in bufs], bsize, items)
            assert (status == 0).all()
            o = _oracle_predict.PredictOracle(p, frames)
            _oracle_predict.reset_stats()
            want = np.array([o.predict_block(int(it[4]), bsize, *map(int, it[:4]), num_planes) for it in items])
            st = _oracle_predict.get_stats()
            o.close()
            bad = np.nonzero((got != want).any(axis=1))[0]
            assert len(bad) == 0, (len(bad), len(items), items[bad[:5]])
    finally:
        for b in bufs:
            tfgpu.evict_frame(b.frame_id)
    if kind == "columns":
        assert st["conv_im_overflow"] > 0, st
    if kind == "noise" and bd == 12:
        assert st["pred_clip_lo"] > 0 and st["pred_clip_hi"] > 0, st


def test_chain_on_the_device(pkg, tfgpu):
    """A 32x32 motion search and the predictor at its MVs, enqueued on one stream behind a sleep with no host
    synchronise between them; equal to motion_search_batch followed by the oracle's predictor."""
    W, H = 640, 360
    clip = _content.subpel_pan(W, H, 3, 10, velocity=(0.75, -1.25))
    p = _params.tf_params(W, H, 3, bit_depth=10, speed=2, allow_hp=1)
    bufs = ms._bufs(pkg, p, [clip[1], clip[0], clip[2]], 2_500_000)
    for b in bufs:
        tfgpu.cache_frame(b)
    src, refs = bufs[0].frame_id, [bufs[1].frame_id, bufs[2].frame_id]
    ah = -(-H // 8) * 8
    items = np.array([(x, y, 0, 0, r) for r in (0, 1) for y in range(0, ah, 32) for x in range(0, W, 32)], np.int64)
    try:
        host = tfgpu.motion_search_batch(p, src, refs, 32, items)
        d_items = _cuda(items)
        side = torch.cuda.Stream()
        for sleep in (False, True):  # the first pass loads every kernel
            torch.cuda.synchronize()
            with torch.cuda.stream(side):
                if sleep:
                    torch.cuda._sleep(SLEEP_CYCLES)
                res = tfgpu.motion_search_tensors(p, src, refs, 32, d_items)
                pitems = d_items.clone()
                pitems[:, 2:4] = res[:, 3:5]
                planes, status = tfgpu.predict_tensors(p, refs, 32, pitems)
                assert not (sleep and side.query()), "the sleep was over before the chain was enqueued"
            side.synchronize()
            got = _flat(planes)
            assert (status.cpu().numpy() == 0).all()
            assert (res.cpu().numpy() == host).all()
    finally:
        for b in bufs:
            tfgpu.evict_frame(b.frame_id)
    o = _oracle_predict.PredictOracle(p, [clip[1], clip[0], clip[2]])
    want = np.array([o.predict_block(1 + int(it[4]), 32, int(it[0]), int(it[1]), int(h[3]), int(h[4]), 3)
                     for it, h in zip(items, host)])
    o.close()
    assert (got == want).all()
    assert (host[:, 3:5] & 7 != 0).any()


def test_source_at_mv_zero_is_the_source_block(pkg, tfgpu):
    W, H = 216, 120
    frames = _clips.moving_texture(W, H, 1, 10, ss_x=1, ss_y=0)
    p = _params.tf_params(W, H, 1, bit_depth=10, ss_x=1, ss_y=0)
    b = pkg.Yv12Buffer(W, H, 1, 0, True, p["border"], frame_id=2_600_000).set_planes(*frames[0])
    tfgpu.cache_frame(b)
    try:
        for bsize in (16, 32):
            items = np.array([(x, y, 0, 0, 0) for y in range(0, H, 4) for x in range(0, W, 16)], np.int64)
            got, status = _predict(tfgpu, p, [b.frame_id], bsize, items)
            assert (status == 0).all()
            for (x, y, *_), g in zip(items.tolist(), got):
                want = np.concatenate([b.plane(pl)[y:y + bsize, (x >> (pl > 0)):(x >> (pl > 0)) + (bsize >> (pl > 0))]
                                       .ravel() for pl in range(3)])
                assert (g == want).all(), (bsize, x, y)
    finally:
        tfgpu.evict_frame(b.frame_id)


@pytest.fixture(scope="module")
def resident(pkg, tfgpu):
    """A 640x360 8-bit clip of three frames, resident under ids 2700000..2700002."""
    W, H = 640, 360
    frames = _clips.moving_texture(W, H, 3, 8, motion=(1, 2))
    p = _params.tf_params(W, H, 3)
    bufs = ms._bufs(pkg, p, frames, 2_700_000)
    for b in bufs:
        tfgpu.cache_frame(b)
    yield p, frames, [b.frame_id for b in bufs]
    for b in bufs:
        tfgpu.evict_frame(b.frame_id)


def _items(seed, n=400, W=640, H=360, refs=3):
    rng = np.random.default_rng(seed)
    return np.stack([rng.integers(0, W // 16, n) * 16, rng.integers(0, H // 4, n) * 4, rng.integers(-300, 300, n),
                     rng.integers(-300, 300, n), rng.integers(0, refs, n)], axis=1)


def test_stream_order_and_no_host_block(pkg, tfgpu, resident):
    p, frames, ids = resident
    items_np = _items(1)
    want, _ = _predict(tfgpu, p, ids, 16, items_np)
    final = _cuda(items_np)
    side = torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        torch.cuda._sleep(SLEEP_CYCLES)
        items = torch.zeros_like(final)
        items.add_(final)  # written on this stream behind the sleep: the predictor has to come after
        planes, status = tfgpu.predict_tensors(p, ids, 16, items)
        consumed = [t + 0 for t in planes]
        assert not side.query(), "the call blocked until the stream was idle"
    side.synchronize()
    assert (_flat(consumed) == want).all() and (status.cpu().numpy() == 0).all()


def test_slots_evicted_behind_a_queued_predict(pkg):
    W, H = 640, 360
    clip = _clips.moving_texture(W, H, 5, 8, motion=(1, 2))
    p = _params.tf_params(W, H, 2)
    ctx = pkg.TemporalFilterGpu(max_cached_frames=2)
    try:
        old = ms._bufs(pkg, p, clip[:2], 2_710_000)
        for b in old:
            ctx.cache_frame(b)
        ids = [b.frame_id for b in old]
        items_np = _items(3, refs=2)
        want, _ = _predict(ctx, p, ids, 32, items_np)
        items = _cuda(items_np)
        new_planes = [[_cuda(a) for a in f] for f in clip[2:4]]
        warm = pkg.TemporalFilterGpu()  # load the ingest kernels before the timed part
        warm.cache_frame_tensor(2_710_030, *new_planes[0])
        warm.close()
        side = torch.cuda.Stream()
        torch.cuda.synchronize()
        with torch.cuda.stream(side):
            torch.cuda._sleep(SLEEP_CYCLES)
            planes, _ = ctx.predict_tensors(p, ids, 32, items)
            for i in ids:
                ctx.evict_frame(i)
            ctx.cache_frame_tensor(2_710_020, *new_planes[0])
            ctx.cache_frame_tensor(2_710_021, *new_planes[1])
            assert not side.query(), "the sleep was over before the slots were refilled: nothing is shown"
        ctx.synchronize()
        side.synchronize()
        assert (_flat(planes) == want).all()
        now, _ = _predict(ctx, p, [2_710_020, 2_710_021], 32, items_np)
        assert (now != want).any()
    finally:
        ctx.close()


def test_rejected_items_get_status_and_zeros(pkg, tfgpu, resident):
    p, _, ids = resident
    aw, ah = 640, 360
    bad = [(8, 0, 3, 5, 0), (0, 2, 0, 0, 1), (-16, 0, 0, 0, 0), (0, -4, 0, 0, 0), (aw, 16, 0, 0, 2), (16, ah, 3, 3, 0),
           (32, 32, 0, 0, -1), (32, 32, 0, 0, 3), (48, 16, 0, 0, 22)]
    good = _items(4, n=40)
    for bsize in (16, 32):
        rows, is_bad = [], []
        for k, g in enumerate(good.tolist()):
            rows.append(g)
            is_bad.append(False)
            if k < len(bad):
                rows.append(bad[k])
                is_bad.append(True)
        items, is_bad = np.array(rows, np.int64), np.array(is_bad)
        got, status = _predict(tfgpu, p, ids, bsize, items)
        assert (status[is_bad] == pkg.TF_GPU_MOTION_REJECTED).all() and (got[is_bad] == 0).all()
        assert (status[~is_bad] == 0).all()
        want, _ = _predict(tfgpu, p, ids, bsize, items[~is_bad])
        assert (got[~is_bad] == want).all()


def _mapped_bytes_from(ptr):
    """Bytes of device memory mapped contiguously from ptr on (the walk of the library's extent check)."""
    cuda = C.CDLL("libcuda.so.1")
    base, size = C.c_uint64(), C.c_size_t()
    assert cuda.cuMemGetAddressRange_v2(C.byref(base), C.byref(size), C.c_uint64(ptr)) == 0
    end = base.value + size.value
    while cuda.cuMemGetAddressRange_v2(C.byref(base), C.byref(size), C.c_uint64(end)) == 0 and base.value == end \
            and size.value:
        end += size.value
    return end - ptr


def _raw(tfgpu, cp, ref_ids, num_refs, bsize, items, n, pred, status, stream=None):
    ids = None if ref_ids is None else (C.c_uint64 * max(len(ref_ids), 1))(*ref_ids)
    return tfgpu.lib.tf_gpu_predict_device(tfgpu.h, None if cp is None else C.byref(cp), ids, num_refs, bsize, items,
                                           n, pred, status, stream)


def test_host_rejections_leave_the_context_usable(pkg, tfgpu, resident):
    p, frames, ids = resident
    cp = pkg.make_params(p)
    dev = torch.device("cuda", torch.cuda.current_device())
    items_np = _items(5, n=8)
    want, _ = _predict(tfgpu, p, ids, 16, items_np)
    it = pkg.pack_motion_items(_cuda(items_np))
    pred = torch.zeros((8, 384), dtype=torch.uint8, device=dev)
    st = torch.zeros(8, dtype=torch.int32, device=dev)
    big = torch.zeros(1 << 16, dtype=torch.int32, device=dev)
    ok_i, ok_p, ok_s = it.data_ptr(), pred.data_ptr(), st.data_ptr()
    other = pkg.Yv12Buffer(352, 288, 1, 1, False, p["border"], frame_id=2_720_000).set_planes(
        *_clips.moving_texture(352, 288, 1, 8)[0])
    mono = pkg.Yv12Buffer(640, 360, 1, 1, False, p["border"], monochrome=True, frame_id=2_720_001).set_planes(
        _clips.moving_texture(640, 360, 1, 8)[0][0])
    for b in (other, mono):
        tfgpu.cache_frame(b)
    cp10 = pkg.make_params(dict(p, bit_depth=10))
    cp1 = pkg.make_params(dict(p, monochrome=1))
    host = np.zeros(4096, np.int32)
    B = big.data_ptr()
    torch.cuda.synchronize()
    bad = [
        (None, ids, 3, 16, ok_i, 8, ok_p, ok_s),                 # NULL params
        (cp, None, 3, 16, ok_i, 8, ok_p, ok_s),                  # NULL ref_ids
        (cp, ids, 3, 16, None, 8, ok_p, ok_s),                   # NULL items
        (cp, ids, 3, 16, ok_i, 8, None, ok_s),                   # NULL pred
        (cp, ids, 3, 16, ok_i, 8, ok_p, None),                   # NULL status
        (cp, ids, 3, 8, ok_i, 8, ok_p, ok_s),                    # block size
        (cp, ids, 3, 64, ok_i, 8, ok_p, ok_s),
        (cp, ids, 3, 16, ok_i, -1, ok_p, ok_s),                  # n < 0
        (cp, ids, 0, 16, ok_i, 8, ok_p, ok_s),                   # num_refs
        (cp, list(range(1, 25)), 24, 16, ok_i, 8, ok_p, ok_s),
        (cp, [ids[0], 123456789], 2, 16, ok_i, 8, ok_p, ok_s),   # not resident
        (cp, [ids[0], other.frame_id], 2, 16, ok_i, 8, ok_p, ok_s),  # mixed geometry
        (cp, [ids[0], mono.frame_id], 2, 16, ok_i, 8, ok_p, ok_s),   # (a monochrome slot differs too)
        (cp, [mono.frame_id], 1, 16, ok_i, 8, ok_p, ok_s),       # num_planes 3 on a frame without chroma
        (cp10, ids, 3, 16, ok_i, 8, ok_p, ok_s),                 # bit depth 10 in an 8-bit container
        (cp, ids, 3, 16, host.ctypes.data, 8, ok_p, ok_s),       # host memory
        (cp, ids, 3, 16, ok_i, 8, host.ctypes.data, ok_s),
        (cp, ids, 3, 16, ok_i, 8, ok_p, host.ctypes.data),
        (cp, ids, 3, 16, ok_i + 2, 7, ok_p, ok_s),               # misaligned
        (cp, ids, 3, 16, ok_i, 8, ok_p, ok_s + 2),
        (cp, ids, 3, 16, ok_i, _mapped_bytes_from(ok_i) // 16 + 1, ok_p, ok_s),  # extents past the allocation
        (cp, ids, 3, 16, ok_i, 8, B + _mapped_bytes_from(B) - 384 * 8 + 1, ok_s),
        (cp, ids, 3, 16, ok_i, 8, ok_p, B + _mapped_bytes_from(B) - 28),
        (cp, ids, 3, 16, B, 8, B + 64, ok_s),                    # overlaps
        (cp, ids, 3, 16, B, 8, ok_p, B + 124),
        (cp, ids, 3, 16, ok_i, 8, B, B + 384 * 8 - 4),
    ]
    before = tfgpu.last_stats()
    for k, args in enumerate(bad):
        assert _raw(tfgpu, *args) == -1, k
    assert tfgpu.last_stats() == before
    hbd_pred = torch.zeros(384 * 8 + 1, dtype=torch.int16, device=dev)
    hbd = pkg.Yv12Buffer(640, 360, 1, 1, True, p["border"], frame_id=2_720_002).set_planes(
        *_clips.moving_texture(640, 360, 1, 10)[0])
    tfgpu.cache_frame(hbd)
    cph = pkg.make_params(dict(p, bit_depth=10))
    assert _raw(tfgpu, cph, [hbd.frame_id], 1, 16, ok_i, 8, hbd_pred.data_ptr() + 1, ok_s) == -1  # sample alignment
    assert _raw(tfgpu, cph, [hbd.frame_id], 1, 16, ok_i, 8, hbd_pred.data_ptr() + 2, ok_s) == 0
    torch.cuda.synchronize()
    with pytest.raises(ValueError, match="the context on cuda:1"):
        pkg.predict_device_args([1], 16, torch.zeros((1, 5), dtype=torch.int32, device="cuda:0"),
                                torch.device("cuda", 1))
    # n == 0 enqueues nothing
    sleeper, idle = torch.cuda.Stream(), torch.cuda.Stream()
    with torch.cuda.stream(sleeper):
        torch.cuda._sleep(SLEEP_CYCLES)
        assert _raw(tfgpu, cp, ids, 3, 16, ok_i, 8, ok_p, ok_s, sleeper.cuda_stream) == 0
    assert _raw(tfgpu, cp1, ids, 3, 16, ok_i, 0, ok_p, ok_s, idle.cuda_stream) == 0
    assert idle.query()
    torch.cuda.synchronize()
    for b in (other, mono, hbd):
        tfgpu.evict_frame(b.frame_id)
    got, status = _predict(tfgpu, p, ids, 16, items_np)  # the next valid call gives the same result
    assert (got == want).all() and (status == 0).all()
    assert (pred.cpu().numpy() == want).all()
