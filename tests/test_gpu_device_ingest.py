"""GPU: frames that enter the device frame cache from device memory (tf_gpu_cache_frame_device, through
TemporalFilterGpu.cache_frame_tensor).  The ingest kernel must leave slots sample-identical to the host upload
(copy + extend_borders_kernel) over the whole defined region -- the search and filter kernels only read slots, so
that is the whole parity contract -- and the calls on top (filter_tensors, estimate_noise_tensor) must equal the
host path and the oracle.  Also: stream ordering against a producer's stream, cache semantics, and rejection of
bad descriptors before anything is launched."""
import ctypes as C

import numpy as np
import pytest
import torch

import _clips
import _gpu
import _oracle
import _params

pytestmark = pytest.mark.gpu


def _cuda(a, dev="cuda"):
    """numpy plane -> CUDA tensor (uint16 samples as int16, the dtype torch handles everywhere)."""
    return None if a is None else torch.from_numpy(a.view(np.int16) if a.dtype == np.uint16 else a).to(dev)


def _host_buffer(pkg, W, H, bd, sx, sy, mono, planes, fid):
    b = pkg.Yv12Buffer(W, H, sx, sy, bd > 8, 160, mono, frame_id=fid)
    return b.set_planes(*planes, extend=False)


def _read(ctx, fid, dtype, pl, x0, y0, w, h):
    dst = np.zeros((h, w), dtype)
    ctx._check(ctx.lib.tf_gpu_debug_read_plane(ctx.h, fid, pl, dst.ctypes.data, w, x0, y0, w, h))
    return dst


def _defined_region(ctx, b, fid, pl):
    """[-bx, aligned_w + bx) x [-by, aligned_h + by) of slot `fid`, the rectangle both load paths define."""
    k = 1 if pl else 0
    db = ctx.device_border()
    bx, by = (db >> b.ss_x, db >> b.ss_y) if k else (db, db)
    aw, ah = b.aligned[k]
    return _read(ctx, fid, b.dtype, pl, -bx, -by, aw + 2 * bx, ah + 2 * by)


# (W, H, bit depth, ss_x, ss_y, monochrome, column offset of the source in a wider tensor, extra columns)
SLOT_CASES = {
    "8bit_420": (352, 288, 8, 1, 1, False, 0, 0),
    "10bit_420": (352, 288, 10, 1, 1, False, 0, 0),
    "12bit_444": (200, 136, 12, 0, 0, False, 0, 0),
    "8bit_422": (352, 288, 8, 1, 0, False, 0, 0),
    "mono": (200, 136, 8, 1, 1, True, 0, 0),
    "odd_353x289_8": (353, 289, 8, 1, 1, False, 0, 0),
    "odd_353x289_10": (353, 289, 10, 1, 1, False, 0, 0),
    "odd_200x136_10": (200, 136, 10, 1, 1, False, 0, 0),
    "slice_8_off3": (352, 288, 8, 1, 1, False, 3, 45),     # base 3 bytes off 16-byte alignment: single samples
    "slice_8_off4": (353, 289, 8, 1, 1, False, 4, 27),     # 4-byte loads
    "slice_8_off8": (353, 289, 8, 1, 1, False, 8, 40),     # 8-byte loads
    "slice_10_off1": (352, 288, 10, 1, 1, False, 1, 13),   # 2 bytes off
    "slice_10_off2": (353, 289, 10, 1, 1, False, 2, 30),   # 4-byte loads
    "slice_12_off4_444": (200, 136, 12, 0, 0, False, 4, 9),  # 8-byte loads
}


@pytest.mark.parametrize("case", sorted(SLOT_CASES))
def test_ingested_slot_equals_host_upload(pkg, tfgpu, case):
    W, H, bd, sx, sy, mono, off, pad = SLOT_CASES[case]
    planes = _clips.moving_texture(W, H, 1, bd, ss_x=sx, ss_y=sy, monochrome=mono)[0]
    b = _host_buffer(pkg, W, H, bd, sx, sy, mono, planes, 910001)
    tfgpu.cache_frame(b)
    tens = []
    for a in planes:
        if a is None:
            continue
        t = _cuda(a)
        if pad:  # a column slice of a wider tensor: padded row stride, base not 16-byte aligned
            fill = 255 if t.dtype == torch.uint8 else -1
            wide = torch.full((t.shape[0], t.shape[1] + pad), fill, dtype=t.dtype, device=t.device)
            wide[:, off:off + t.shape[1]] = t
            t = wide[:, off:off + t.shape[1]]
            assert t.stride(0) == a.shape[1] + pad and (t.data_ptr() % 16) != 0
        tens.append(t)
    tfgpu.cache_frame_tensor(910002, *tens)
    try:
        for pl in range(b.num_planes):
            want = _defined_region(tfgpu, b, 910001, pl)
            got = _defined_region(tfgpu, b, 910002, pl)
            assert (got == want).all(), (pl, int((got != want).sum()))
    finally:
        tfgpu.evict_frame(910001)
        tfgpu.evict_frame(910002)


FILTER_CASES = {"cif8_n5": (352, 288, 8, 5, (0, 4, 8)), "1080p10_n5": (1920, 1080, 10, 5, (0, 17, 33)),
                "4k10_n5": (3840, 2160, 10, 5, (0, 67))}


@pytest.mark.parametrize("case", sorted(FILTER_CASES))
def test_filter_tensors_equals_host_filter_and_oracle(pkg, case):
    W, H, bd, N, rows = FILTER_CASES[case]
    ctx = pkg.TemporalFilterGpu(device=0)
    try:
        frames = _clips.moving_texture(W, H, N, bd)
        p = _params.tf_params(W, H, N, bit_depth=bd)
        host = _gpu.run_gpu(pkg, ctx, p, frames, dump=False)  # tf_gpu_filter over host frames
        ids = [920001 + i for i in range(N)]
        for i, planes in zip(ids, frames):
            ctx.cache_frame_tensor(i, *[_cuda(a) for a in planes])
        outs, diff = ctx.filter_tensors(p, ids)
        assert (diff == host["diff"]).all()
        got = [o.cpu().numpy().view(np.uint16) if bd > 8 else o.cpu().numpy() for o in outs]
        for pl, g in enumerate(got):
            assert g.shape == (((H + 1) >> 1, (W + 1) >> 1) if pl else (H, W))
            assert (g == host["out"][pl][:g.shape[0], :g.shape[1]]).all(), pl
        o = _oracle.OracleFilter(p, frames)
        for r in rows:
            ref = o.run(record=False, rows=(r, r + 1))
            for pl, g in enumerate(got):
                bh = 32 >> (1 if pl else 0)
                gs = g[r * bh:(r + 1) * bh]  # the last block row may end below the crop area
                want = ref["out"][pl][r * bh:r * bh + gs.shape[0], :gs.shape[1]]
                assert (gs.astype(np.uint16) == want).all(), (r, pl)
        o.close()
    finally:
        ctx.close()


def test_ingest_is_ordered_on_the_producer_stream(pkg, tfgpu):
    """The producer writes the planes on a side stream behind a long sleep and ingests there without a host
    sync; overwriting the source on the same stream right after the call must not reach the slot."""
    W, H = 352, 288
    planes = _clips.moving_texture(W, H, 1, 10)[0]
    b = _host_buffer(pkg, W, H, 10, 1, 1, False, planes, 930001)
    tfgpu.cache_frame(b)
    final = [_cuda(a) for a in planes]
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    with torch.cuda.stream(side):
        src = [torch.zeros_like(t) for t in final]
        torch.cuda._sleep(200_000_000)  # a few tens of ms: the ingest must not start before the copies below
        for s, t in zip(src, final):
            s.copy_(t)
        tfgpu.cache_frame_tensor(930002, *src)
        for s in src:
            s.fill_(-1)
    try:
        for pl in range(3):
            assert (_defined_region(tfgpu, b, 930002, pl) == _defined_region(tfgpu, b, 930001, pl)).all(), pl
        side.synchronize()
        assert all(bool((s == -1).all()) for s in src)
    finally:
        tfgpu.evict_frame(930001)
        tfgpu.evict_frame(930002)


def test_cache_semantics_and_mixed_window(pkg, tfgpu):
    W, H, N = 352, 288, 5
    frames = _clips.moving_texture(W, H, N, 8)
    p = _params.tf_params(W, H, N)
    host = _gpu.run_gpu(pkg, tfgpu, p, frames, dump=False)
    ids = [940001 + i for i in range(N)]
    try:
        for i, (fid, planes) in enumerate(zip(ids, frames)):
            if i % 2:  # odd frames from the host, even frames from device memory
                tfgpu.cache_frame(_host_buffer(pkg, W, H, 8, 1, 1, False, planes, fid))
            else:
                tens = [_cuda(a) for a in planes]
                tfgpu.cache_frame_tensor(fid, *tens)
                assert tfgpu.last_stats()[0] == 3  # one ingest launch per plane
                for t in tens:  # a resident id is not re-read: nothing is launched, the slot keeps its pixels
                    t.zero_()
                tfgpu.cache_frame_tensor(fid, *tens)
                assert tfgpu.last_stats()[0] == 0
        _, diff = tfgpu.filter_resident(p, ids)
        assert (diff == host["diff"]).all()
        out = pkg.Yv12Buffer(W, H, 1, 1, False, p["border"])
        tfgpu.download_output(out)
        for pl in range(3):
            assert (out.full_blocks(pl) == host["out"][pl]).all()
    finally:
        for fid in ids:
            tfgpu.evict_frame(fid)


@pytest.mark.parametrize("bd", [8, 10])
def test_estimate_noise_tensor_equals_host(pkg, tfgpu, bd):
    W, H = 352, 288
    planes = _clips.moving_texture(W, H, 1, bd)[0]
    b = _host_buffer(pkg, W, H, bd, 1, 1, False, planes, 0)
    tens = tuple(_cuda(a) for a in planes)
    try:
        for pl in range(3):
            want = tfgpu.estimate_noise_from_single_plane(b, pl, bd)
            assert tfgpu.estimate_noise_tensor(950001, tens, pl, bd) == want
    finally:
        tfgpu.evict_frame(950001)


def _rejected(pkg, ctx, f):
    rc = ctx.lib.tf_gpu_cache_frame_device(ctx.h, C.byref(f), None)
    assert rc == -1, ctx.lib.tf_gpu_last_error(ctx.h)
    assert ctx.last_stats()[0] == 0  # nothing launched
    with pytest.raises(pkg.TfGpuError):
        _read(ctx, f.frame_id or 1, np.uint8, 0, 0, 0, 1, 1)


def test_abi_rejects_bad_device_frames_before_any_launch(pkg):
    ctx = pkg.TemporalFilterGpu(device=0)
    try:
        W, H = 64, 48
        planes = [torch.zeros(s, dtype=torch.uint8, device="cuda:0") for s in ((H, W), (H // 2, W // 2), (H // 2, W // 2))]
        host = np.zeros((H, W), np.uint8)
        f, _ = pkg.tensor_frame(960001, *planes)
        f.plane[0] = host.ctypes.data  # a host (numpy) pointer
        _rejected(pkg, ctx, f)
        f, _ = pkg.tensor_frame(0, *planes)  # frame_id 0
        _rejected(pkg, ctx, f)
        f, _ = pkg.tensor_frame(960001, *planes)
        f.plane[0] = None  # a NULL plane
        _rejected(pkg, ctx, f)
        f, _ = pkg.tensor_frame(960001, *planes)
        f.plane[2] = None  # a NULL chroma plane of a three-plane frame
        _rejected(pkg, ctx, f)
        f, _ = pkg.tensor_frame(960001, *planes)
        f.aligned_w[0] = W - 8  # bad geometry (aligned smaller than crop)
        _rejected(pkg, ctx, f)
        if torch.cuda.device_count() >= 2:  # a plane on another device
            f, _ = pkg.tensor_frame(960001, *[t.to("cuda:1") for t in planes])
            _rejected(pkg, ctx, f)
        # the context stays usable, and the same descriptor with valid planes is accepted
        f, _ = pkg.tensor_frame(960001, *planes)
        assert ctx.lib.tf_gpu_cache_frame_device(ctx.h, C.byref(f), None) == 0
        torch.cuda.synchronize()
    finally:
        ctx.close()


def test_python_rejects_malformed_tensors(pkg, tfgpu):
    y = torch.zeros((48, 64), dtype=torch.uint8, device="cuda")
    u = torch.zeros((24, 32), dtype=torch.uint8, device="cuda")
    bad = {
        "cpu": (y.cpu(), u.cpu(), u.cpu()),
        "dtype": (y.float(), u.float(), u.float()),
        "chroma_shape": (y, u[:, :20], u[:, :20]),
        "mixed_dtypes": (y, u.to(torch.int16), u),
        # one uv stride in tf_gpu_frame: u contiguous, v a column slice of a wider tensor (and the reverse)
        "uv_row_strides": (y, u, torch.zeros((24, 48), dtype=torch.uint8, device="cuda")[:, 8:40]),
        "vu_row_strides": (y, torch.zeros((24, 48), dtype=torch.uint8, device="cuda")[:, 8:40], u),
    }
    for name, planes in bad.items():
        with pytest.raises(ValueError):
            tfgpu.cache_frame_tensor(970001, *planes)
        with pytest.raises(pkg.TfGpuError):  # nothing reached the cache
            _read(tfgpu, 970001, np.uint8, 0, 0, 0, 1, 1)
