"""GPU: tf_gpu_motion_search_device / TemporalFilterGpu.motion_search_tensors -- the motion search of
tf_gpu_motion_search_batch with items and results in device memory, ordered on the caller's stream.  Equal on all six
fields to the synchronous call (and on a sample to the oracle) over the case lists of test_gpu_motion_search.py;
stream order in both directions; the call does not block the host; slots evicted behind a queued search keep their
frames until it has run; a two-stage 32x32 -> 16x16 chain on the device; per-item rejection in the kernel; host
rejections that leave the context usable; tensors of torch's chunked allocators."""
import ctypes as C
import os
import subprocess
import sys

import numpy as np
import pytest

import _clips
import _content
import _oracle_motion
import _params
import test_gpu_motion_search as ms

pytestmark = pytest.mark.gpu
torch = pytest.importorskip("torch")

HERE = os.path.dirname(os.path.abspath(__file__))
SLEEP_CYCLES = 1_000_000_000  # torch.cuda._sleep: about half a second at B200 clocks, far longer than the host work
ORACLE_SAMPLE = 12
REJECTED = [0, 0, -1, 0, 0, 2 ** 32 - 1]


def _cuda(a):
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


def _planes(frame):
    """CUDA tensors of a frame of _clips / _content (uint16 samples as int16)."""
    return [_cuda(a.view(np.int16) if a.dtype == np.uint16 else a) for a in frame]


def _check_against_sync(pkg, tfgpu, p, frames, bsize, items, id_base, ref_order=None, oracle=True):
    """frames[0] the source, frames[1:] the references (or the frames ref_order indexes, source included)."""
    bufs = ms._bufs(pkg, p, frames, id_base)
    for b in bufs:
        tfgpu.cache_frame(b)
    order = ref_order or list(range(1, len(frames)))
    ref_ids = [bufs[i].frame_id for i in order]
    try:
        want = tfgpu.motion_search_batch(p, bufs[0].frame_id, ref_ids, bsize, items)
        got = tfgpu.motion_search_tensors(p, bufs[0].frame_id, ref_ids, bsize, _cuda(items))
        assert got.dtype == torch.int64 and got.is_cuda and got.shape == (len(items), 6)
        got = got.cpu().numpy()
        launches, ms_ = tfgpu.last_stats()
        assert (launches, ms_) == (1, 0.0)
    finally:
        for b in bufs:
            tfgpu.evict_frame(b.frame_id)
    bad = np.nonzero((got != want).any(axis=1))[0]
    assert len(bad) == 0, (len(bad), len(items), items[bad[:5]], got[bad[:5]], want[bad[:5]])
    if oracle:
        o = _oracle_motion.MotionOracle(dict(p, num_frames=len(frames), filter_frame_idx=0), frames)
        pick = np.random.default_rng(id_base).choice(len(items), min(ORACLE_SAMPLE, len(items)), replace=False)
        for k in pick.tolist():
            it = items[k].tolist()
            assert tuple(got[k]) == o.motion_search(0, order[it[4]], bsize, *it[:4]), (it, got[k])
        o.close()
    return got


@pytest.mark.parametrize("case", ms.CASES, ids=[c[0] for c in ms.CASES])
@pytest.mark.parametrize("bsize", [16, 32])
def test_equals_synchronous_call(pkg, tfgpu, case, bsize):
    name, W, H, bd, hbd, speed, hp, fim = case
    clip = _clips.moving_texture(W, H, 4, bd, motion=ms.MOTION)
    frames = [clip[1], clip[0], clip[2], clip[3]]
    p = _params.tf_params(W, H, 4, bit_depth=bd, use_hbd=hbd, speed=speed, allow_hp=hp, force_integer_mv=fim)
    rng = np.random.default_rng(20 * ms.CASES.index(case) + bsize)
    motions = [((1 - k) * ms.MOTION[0], (1 - k) * ms.MOTION[1]) for k in (0, 2, 3)]
    items = ms._items(rng, W, H, bsize, motions, cap=10 ** 6)
    _check_against_sync(pkg, tfgpu, p, frames, bsize, items, 1_100_000 + 100 * ms.CASES.index(case) + bsize)


@pytest.mark.parametrize("t", ms.CONTENT, ids=[f"{t[0]}-{t[3]}-{i}" for i, t in enumerate(ms.CONTENT)])
@pytest.mark.parametrize("bsize", [16, 32])
def test_adversarial_content_equals_synchronous_call(pkg, tfgpu, t, bsize):
    cls, W, H, bd, ckw, pkw, order = t
    clip = _content.make(cls, W, H, max(order) + 1, bd, **ckw)
    frames = [clip[i] for i in order]
    p = _params.tf_params(W, H, len(frames), bit_depth=bd, **pkw)
    v = ckw.get("velocity") or ckw.get("motion") or (0, 0)
    motions = [(-(i - order[0]) * v[0], -(i - order[0]) * v[1]) for i in order[1:]]
    items = ms._items(np.random.default_rng(ms.CONTENT.index(t) * 20 + bsize), W, H, bsize, motions, cap=10 ** 6)
    _check_against_sync(pkg, tfgpu, p, frames, bsize, items, 1_200_000 + 100 * ms.CONTENT.index(t) + bsize)


def test_repeated_reference_and_source_as_reference(pkg, tfgpu):
    W, H = 640, 360
    clip = _clips.moving_texture(W, H, 3, 10, motion=(1, 2))
    p = _params.tf_params(W, H, 3, bit_depth=10, speed=2, allow_hp=1)
    for bsize in (16, 32):
        items = ms._items(np.random.default_rng(bsize), W, H, bsize, [(-1, -2), (0, 0), (-1, -2)], cap=10 ** 6)
        got = _check_against_sync(pkg, tfgpu, p, clip[1:2] + clip[0:1], bsize, items, 1_300_000 + bsize,
                                  ref_order=[1, 0, 1])
        same = (items[:, 4] == 1) & (items[:, 2] == 0) & (items[:, 3] == 0)
        assert (got[same, 3:6] == 0).all() and same.any()  # a block matches itself at MV 0


def test_large_motion_reaches_the_mv_clamp(pkg, tfgpu):
    W, H, v = 1920, 1080, (2, 150)
    clip = _content.large_motion(W, H, 10, 10, velocity=v)
    order = (0, 7, 8, 9)
    frames = [clip[i] for i in order]
    p = _params.tf_params(W, H, 4, bit_depth=10)
    rng = np.random.default_rng(6)
    for bsize in (16, 32):
        items = ms._items(rng, W, H, bsize, [(-k * v[0], -k * v[1]) for k in order[1:]], cap=10 ** 6)
        got = _check_against_sync(pkg, tfgpu, p, frames, bsize, items, 1_400_000 + bsize)
        assert (np.abs(got[:, 1]) == 1023).any() and (np.abs(got[:, 4]) == 8 * 1023).any()


@pytest.fixture(scope="module")
def resident(pkg, tfgpu):
    """A 640x360 8-bit source and three references, resident under ids 1500000..1500003."""
    W, H = 640, 360
    frames = _clips.moving_texture(W, H, 4, 8, motion=(1, 2))
    p = _params.tf_params(W, H, 4, speed=2, allow_hp=1)
    bufs = ms._bufs(pkg, p, frames, 1_500_000)
    for b in bufs:
        tfgpu.cache_frame(b)
    yield p, frames, [b.frame_id for b in bufs]
    for b in bufs:
        tfgpu.evict_frame(b.frame_id)


def _items16(seed, W=640, H=360):
    return ms._items(np.random.default_rng(seed), W, H, 16, [(-1, -2), (1, 2), (2, 4)], cap=10 ** 6)


def test_stream_order_in(pkg, tfgpu, resident):
    """On a side stream, after a sleep: torch ops write the items and the pixels of the frames, the frames are
    ingested, the search runs and a torch op consumes its result -- no host synchronise until the end."""
    p, frames, ids = resident
    items_np = _items16(1)
    want = tfgpu.motion_search_batch(p, ids[0], ids[1:], 16, items_np)
    final = [_planes(f) for f in frames]
    items_final = _cuda(items_np)
    side = torch.cuda.Stream()
    for sleep in (False, True):  # the first pass loads every kernel: a first launch may synchronise the device
        tids = [1_510_000 + 10 * sleep + i for i in range(4)]
        torch.cuda.synchronize()
        with torch.cuda.stream(side):
            if sleep:
                torch.cuda._sleep(SLEEP_CYCLES)
            for fid, f in zip(tids, final):
                planes = [torch.zeros_like(t) for t in f]
                for dst, src in zip(planes, f):
                    dst.add_(src)  # written on this stream; the ingest has to come after
                tfgpu.cache_frame_tensor(fid, *planes)
            items = torch.zeros_like(items_final)
            items.add_(items_final)
            res = tfgpu.motion_search_tensors(p, tids[0], tids[1:], 16, items)
            consumed = res + 0
            assert not (sleep and side.query()), "the sleep was over before the chain was enqueued"
        side.synchronize()
        try:
            assert (consumed.cpu().numpy() == want).all(), sleep
        finally:
            for fid in tids:
                tfgpu.evict_frame(fid)


def test_does_not_block_the_host(pkg, tfgpu, resident):
    p, _, ids = resident
    items = _cuda(_items16(2))
    want = tfgpu.motion_search_batch(p, ids[0], ids[1:], 16, items.cpu().numpy())
    tfgpu.motion_search_tensors(p, ids[0], ids[1:], 16, items)  # warm: allocations of the wrapper
    side = torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(side):
        torch.cuda._sleep(SLEEP_CYCLES)
        got = tfgpu.motion_search_tensors(p, ids[0], ids[1:], 16, items)
        assert not side.query()
    side.synchronize()
    assert (got.cpu().numpy() == want).all()


def test_slots_evicted_behind_a_queued_search(pkg):
    """A context of three slots holds the three frames a search reads.  With the search queued behind a sleep, all
    three are evicted and their slots refilled with other frames (tensor ingest, then a host upload); the search
    still sees the frames that were resident at the call."""
    W, H = 640, 360
    clip = _clips.moving_texture(W, H, 6, 8, motion=(1, 2))
    p = _params.tf_params(W, H, 3, speed=2, allow_hp=1)
    ctx = pkg.TemporalFilterGpu(max_cached_frames=3)
    try:
        old = ms._bufs(pkg, p, clip[:3], 1_520_000)
        for b in old:
            ctx.cache_frame(b)
        items_np = ms._items(np.random.default_rng(3), W, H, 16, [(-1, -2), (1, 2)], cap=10 ** 6)
        want = ctx.motion_search_batch(p, old[0].frame_id, [old[1].frame_id, old[2].frame_id], 16, items_np)
        items = _cuda(items_np)
        new_planes = [_planes(f) for f in clip[3:5]]
        new_host = ms._bufs(pkg, p, clip[5:6], 1_520_010)[0]
        # load every kernel the queued work launches first: a first launch may synchronise the device
        ctx.motion_search_tensors(p, old[0].frame_id, [old[1].frame_id, old[2].frame_id], 16, items)
        warm = pkg.TemporalFilterGpu()
        warm.cache_frame_tensor(1_520_030, *new_planes[0])
        warm.close()
        side = torch.cuda.Stream()
        torch.cuda.synchronize()
        with torch.cuda.stream(side):
            torch.cuda._sleep(SLEEP_CYCLES)
            got = ctx.motion_search_tensors(p, old[0].frame_id, [old[1].frame_id, old[2].frame_id], 16, items)
            for b in old:
                ctx.evict_frame(b.frame_id)
            ctx.cache_frame_tensor(1_520_020, *new_planes[0])
            ctx.cache_frame_tensor(1_520_021, *new_planes[1])
            assert not side.query(), "the sleep was over before the slots were refilled: nothing is shown"
            ctx.cache_frame_async(new_host)
        ctx.synchronize()
        side.synchronize()
        assert (got.cpu().numpy() == want).all()
        for b in old:  # every slot now holds a new frame
            with pytest.raises(pkg.TfGpuError):
                ctx.motion_search_batch(p, b.frame_id, [b.frame_id], 16, [(0, 0, 0, 0, 0)])
        now = ctx.motion_search_batch(p, 1_520_020, [1_520_021, new_host.frame_id], 16, items_np)
        assert (now != want).any()
    finally:
        ctx.close()


def test_two_stage_chain_on_the_device(pkg, tfgpu):
    """1080p: a 32x32 search of every block against two references, torch ops turning its 1/8-pel MVs into full-pel
    starts (GET_MV_RAWPEL) of the four 16x16 blocks of each 32x32 block, then the 16x16 search -- both calls enqueued
    behind a sleep on one stream.  Equal to the same chain driven through motion_search_batch on the host."""
    W, H = 1920, 1080
    clip = _content.subpel_pan(W, H, 3, 8, velocity=(0.75, -1.25))
    p = _params.tf_params(W, H, 3, speed=2, allow_hp=1)
    bufs = ms._bufs(pkg, p, [clip[1], clip[0], clip[2]], 1_530_000)
    for b in bufs:
        tfgpu.cache_frame(b)
    src, refs = bufs[0].frame_id, [bufs[1].frame_id, bufs[2].frame_id]
    aw, ah = W, -(-H // 8) * 8
    i32 = np.array([(x, y, 0, 0, r) for r in (0, 1) for y in range(0, ah, 32) for x in range(0, aw, 32)], np.int64)
    offs = [(0, 0), (16, 0), (0, 16), (16, 16)]
    try:
        h32 = tfgpu.motion_search_batch(p, src, refs, 32, i32)
        subs = [(x + dx, y + dy, ms._rawpel(int(m[3])), ms._rawpel(int(m[4])), r)
                for (x, y, _, _, r), m in zip(i32.tolist(), h32) for dx, dy in offs]
        h16 = tfgpu.motion_search_batch(p, src, refs, 16, subs)

        d32_items = _cuda(i32)
        d_offs = _cuda(np.array(offs, np.int64))
        side = torch.cuda.Stream()

        def rawpel(v):
            return torch.bitwise_right_shift(v + 3 + (v >= 0).to(torch.int64), 3)

        for sleep in (False, True):  # the first pass loads every kernel: a first launch may synchronise the device
            torch.cuda.synchronize()
            with torch.cuda.stream(side):
                if sleep:
                    torch.cuda._sleep(SLEEP_CYCLES)
                d32 = tfgpu.motion_search_tensors(p, src, refs, 32, d32_items)
                sub = torch.empty((len(i32), 4, 5), dtype=torch.int64, device=d32.device)
                sub[:, :, 0] = d32_items[:, 0:1] + d_offs[:, 0]
                sub[:, :, 1] = d32_items[:, 1:2] + d_offs[:, 1]
                sub[:, :, 2] = rawpel(d32[:, 3:4])
                sub[:, :, 3] = rawpel(d32[:, 4:5])
                sub[:, :, 4] = d32_items[:, 4:5]
                d16 = tfgpu.motion_search_tensors(p, src, refs, 16, sub.reshape(-1, 5))
                assert not (sleep and side.query()), "the sleep was over before both stages were enqueued"
            side.synchronize()
            assert (d32.cpu().numpy() == h32).all(), sleep
            assert (d16.cpu().numpy() == h16).all(), sleep
        assert (h16[:, 3:5] & 7 != 0).any()  # sub-pel MVs: the chain carries real 1/8-pel information
    finally:
        for b in bufs:
            tfgpu.evict_frame(b.frame_id)


def _invalid_items(W, H, num_refs):
    aw, ah = -(-W // 8) * 8, -(-H // 8) * 8
    return [(8, 0, 1, -1, 0), (0, 2, 0, 0, 1), (-16, 0, 0, 0, 0), (aw, 16, 0, 0, 2), (16, ah, 3, 3, 0),
            (32, 32, 0, 0, -1)] + [(48, 16, 0, 0, r) for r in range(num_refs, 23)]


@pytest.mark.parametrize("bsize", [16, 32])
def test_rejected_items_get_the_sentinel(pkg, tfgpu, resident, bsize):
    p, _, ids = resident
    W, H, db = 640, 360, tfgpu.device_border()
    cp = pkg.make_params(p)
    bad = _invalid_items(W, H, 3)
    # Were the kernel's check missing, every read of these items would stay inside the slot allocation (pixel (0, 0)
    # has db samples of border on every side, plus slack rows): the reference block moves inside the MV limits of
    # item_full_pixel_search, and the sub-pel filter taps, the 16-byte loads of the SAD engine and the sub-pel
    # stage add less than `margin` samples.  So a broken check shows up as a wrong result, not as a fault.
    margin = 24
    for x, y, *_ in bad:
        rmin, rmax, cmin, cmax = ms._limits(x, y, bsize, cp.mi_rows, cp.mi_cols, p["border"])
        assert x + cmin - margin >= -db and x + cmax + bsize + margin <= cp.mi_cols * 4 + db, (x, y)
        assert y + rmin - margin >= -db and y + rmax + bsize + margin <= cp.mi_rows * 4 + db, (x, y)
    good = ms._items(np.random.default_rng(30 + bsize), W, H, bsize, [(-1, -2), (1, 2), (2, 4)], cap=40)
    rows, is_bad = [], []
    for k, g in enumerate(good.tolist()):
        rows.append(g)
        is_bad.append(False)
        if k < len(bad):
            rows.append(bad[k])
            is_bad.append(True)
    rows += bad[len(good):]
    is_bad += [True] * len(bad[len(good):])
    items, is_bad = np.array(rows, np.int64), np.array(is_bad)
    assert is_bad.sum() == len(bad)
    got = tfgpu.motion_search_tensors(p, ids[0], ids[1:], bsize, _cuda(items)).cpu().numpy()
    assert (got[is_bad] == REJECTED).all(), got[is_bad]
    assert (got[is_bad, 2] == pkg.TF_GPU_MOTION_REJECTED).all()
    want = tfgpu.motion_search_batch(p, ids[0], ids[1:], bsize, items[~is_bad])
    assert (got[~is_bad] == want).all()
    assert (want[:, 2] >= 0).all()


def _raw(pkg, tfgpu, cp, src_id, ref_ids, num_refs, bsize, items, n, results, stream=None):
    """tf_gpu_motion_search_device without the Python-side checks; None stands for a NULL pointer."""
    ids = None if ref_ids is None else (C.c_uint64 * max(len(ref_ids), 1))(*ref_ids)
    return tfgpu.lib.tf_gpu_motion_search_device(tfgpu.h, None if cp is None else C.byref(cp), src_id, ids, num_refs,
                                                 bsize, items, n, results, stream)


def _mapped_bytes_from(ptr):
    """Bytes of device memory mapped contiguously from ptr on (the walk tf_gpu_motion_search_device makes)."""
    cuda = C.CDLL("libcuda.so.1")
    base, size = C.c_uint64(), C.c_size_t()
    assert cuda.cuMemGetAddressRange_v2(C.byref(base), C.byref(size), C.c_uint64(ptr)) == 0
    end = base.value + size.value
    while cuda.cuMemGetAddressRange_v2(C.byref(base), C.byref(size), C.c_uint64(end)) == 0 and base.value == end \
            and size.value:
        end += size.value
    return end - ptr


def test_host_rejections_leave_the_context_usable(pkg, tfgpu, resident):
    p, frames, ids = resident
    cp = pkg.make_params(p)
    it = pkg.pack_motion_items(_cuda(np.zeros((1, 5), np.int64)))
    res = torch.empty((1, 4), dtype=torch.int32, device=it.device)
    ok, out = it.data_ptr(), res.data_ptr()
    torch.cuda.synchronize()
    assert _raw(pkg, tfgpu, cp, ids[0], ids[1:], 3, 16, ok, 1, out) == 0
    tfgpu.synchronize()
    assert tfgpu.last_stats() == (1, 0.0)
    other = pkg.Yv12Buffer(352, 288, 1, 1, False, p["border"], frame_id=1_540_000).set_planes(
        *_clips.moving_texture(352, 288, 1, 8)[0])
    tfgpu.cache_frame(other)
    host = np.zeros((4, 4), np.int32)
    pinned = torch.zeros((4, 4), dtype=torch.int32).pin_memory()
    big = torch.zeros((8, 4), dtype=torch.int32, device=it.device)
    # extents: n items of a large buffer with `out` as results (larger than what is mapped from `out`, which grows
    # when the buffer lands right after it), and n one item past the memory mapped from `ok`
    for _ in range(4):
        large = torch.empty((max(1 << 20, _mapped_bytes_from(out) // 16 + 1), 4), dtype=torch.int32, device=it.device)
        if _mapped_bytes_from(out) < large.numel() * 4:
            break
    assert _mapped_bytes_from(out) < large.numel() * 4 <= _mapped_bytes_from(large.data_ptr())
    n_past = _mapped_bytes_from(ok) // 16 + 1
    assert n_past < 2 ** 31
    bad = [
        (None, ids[0], ids[1:], 3, 16, ok, 1, out),                 # NULL params
        (cp, ids[0], None, 3, 16, ok, 1, out),                      # NULL ref_ids
        (cp, ids[0], ids[1:], 3, 16, None, 1, out),                 # NULL items
        (cp, ids[0], ids[1:], 3, 16, ok, 1, None),                  # NULL results
        (cp, ids[0], ids[1:], 3, 24, ok, 1, out),                   # block size
        (cp, ids[0], ids[1:], 3, 8, ok, 1, out),
        (cp, ids[0], ids[1:], 3, 16, ok, -1, out),                  # n < 0
        (cp, ids[0], ids[1:], 0, 16, ok, 1, out),                   # num_refs
        (cp, ids[0], list(range(1, 25)), 24, 16, ok, 1, out),
        (cp, 123456789, ids[1:], 3, 16, ok, 1, out),                # source not resident
        (cp, ids[0], [ids[1], 123456789], 2, 16, ok, 1, out),       # reference not resident
        (cp, ids[0], [ids[1], other.frame_id], 2, 16, ok, 1, out),  # mixed geometry
        (cp, ids[0], ids[1:], 3, 16, host.ctypes.data, 1, out),     # host memory
        (cp, ids[0], ids[1:], 3, 16, ok, 1, host.ctypes.data),
        (cp, ids[0], ids[1:], 3, 16, pinned.data_ptr(), 1, out),    # pinned host memory
        (cp, ids[0], ids[1:], 3, 16, ok, 1, pinned.data_ptr()),
        (cp, ids[0], ids[1:], 3, 16, ok + 2, 1, out),               # misaligned
        (cp, ids[0], ids[1:], 3, 16, ok, 1, out + 2),
        (cp, ids[0], ids[1:], 3, 16, ok, n_past, big.data_ptr()),   # extent past the allocation
        (cp, ids[0], ids[1:], 3, 16, large.data_ptr(), large.shape[0], out),
        (cp, ids[0], ids[1:], 3, 16, big.data_ptr(), 2, big.data_ptr() + 16),  # overlap
        (cp, ids[0], ids[1:], 3, 16, big.data_ptr() + 16, 2, big.data_ptr()),
        (cp, ids[0], ids[1:], 3, 16, big.data_ptr(), 1, big.data_ptr()),
    ]
    before = tfgpu.last_stats()
    for k, args in enumerate(bad):
        assert _raw(pkg, tfgpu, *args) == -1, k
    assert tfgpu.last_stats() == before  # a rejected call leaves the context as it was
    with pytest.raises(ValueError, match="the context on cuda:1"):
        pkg.motion_search_device_args([1], 16, torch.zeros((1, 5), dtype=torch.int32, device="cuda:0"),
                                      torch.device("cuda", 1))
    # n == 0 enqueues nothing: with the context's stream held behind a sleep (a search queued on a sleeping stream),
    # a call with n == 0 leaves an idle stream idle, where a call with n == 1 makes it wait
    sleeper, idle = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(sleeper):
        torch.cuda._sleep(SLEEP_CYCLES)
        assert _raw(pkg, tfgpu, cp, ids[0], ids[1:], 3, 16, ok, 1, out, sleeper.cuda_stream) == 0
    assert _raw(pkg, tfgpu, cp, ids[0], ids[1:], 3, 16, ok, 0, out, idle.cuda_stream) == 0
    assert idle.query()
    assert _raw(pkg, tfgpu, cp, ids[0], ids[1:], 3, 16, big.data_ptr(), 1, out, idle.cuda_stream) == 0
    assert not idle.query()
    torch.cuda.synchronize()
    tfgpu.evict_frame(other.frame_id)
    # the context filters as a fresh one does
    W, H = 352, 288
    clip = _clips.moving_texture(W, H, 3, 8)
    fp = _params.tf_params(W, H, 3)
    outs = []
    for ctx in (tfgpu, pkg.TemporalFilterGpu()):
        bufs = ms._bufs(pkg, fp, clip, 1_541_000)
        o = pkg.Yv12Buffer(W, H, 1, 1, False, fp["border"])
        r = ctx.temporal_filter(fp, bufs, o, dump=True)
        outs.append((r, [o.full_blocks(pl).copy() for pl in range(3)]))
        for b in bufs:
            ctx.evict_frame(b.frame_id)
        if ctx is not tfgpu:
            ctx.close()
    (ra, oa), (rb, ob) = outs
    assert all((a == b).all() for a, b in zip(oa, ob))
    assert all((ra[k] == rb[k]).all() for k in ("diff", "mvs", "mses"))


ALLOCATOR_SCRIPT = r"""
import sys
import numpy as np, torch
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[2])
import conftest, _clips, _params
pkg = conftest.load_package()
ctx = pkg.TemporalFilterGpu(device=0)
W, H = 3840, 2160
p = _params.tf_params(W, H, 3, bit_depth=10, speed=4)
for i, planes in enumerate(_clips.moving_texture(W, H, 3, 10, motion=(1, 2))):
    ctx.cache_frame(pkg.Yv12Buffer(W, H, 1, 1, True, p["border"], frame_id=100 + i).set_planes(*planes))
items = np.array([(x, y, 0, 0, r) for r in (0, 1) for y in range(0, H, 16) for x in range(0, W, 16)], np.int64)
want = ctx.motion_search_batch(p, 100, [101, 102], 16, items)
keep = []
for pad_mb in (0, 1, 3, 7, 19):  # shift where the item and result tensors land in the allocator's chunks
    keep.append(torch.empty(pad_mb << 20, dtype=torch.uint8, device="cuda"))
    d_items = torch.from_numpy(items).cuda()
    got = ctx.motion_search_tensors(p, 100, [101, 102], 16, d_items)
    assert (got.cpu().numpy() == want).all(), pad_mb
ctx.close()
print("ok")
"""


@pytest.mark.parametrize("conf", ["expandable_segments:True", "backend:cudaMallocAsync"])
def test_tensors_of_chunked_allocators(conf):
    env = dict(os.environ, PYTORCH_CUDA_ALLOC_CONF=conf)
    r = subprocess.run([sys.executable, "-c", ALLOCATOR_SCRIPT, HERE, os.path.dirname(HERE)], env=env,
                       capture_output=True, text=True, timeout=600)
    print(r.stdout)
    assert r.returncode == 0 and "ok" in r.stdout, r.stderr[-3000:]
