"""GPU: the row-sum lower bound of the 16x16 search.  Every cached frame carries a plane of 16-sample luma row sums
(read back through tf_gpu_debug_read_plane with TF_GPU_DEBUG_ROWSUM_PLANE), and the 16x16 diamond search skips
sites whose bound sum_k |S_k - R_k(mv)| already rules them out.  The plane must equal the row sums of the
replicated-border frame for both cache routes, the skip must leave every result bit-exact (also where the bound
equals the SAD), and it must actually skip sites on moving content."""
import numpy as np
import pytest
import torch

import _clips
import _gpu
import _params

pytestmark = pytest.mark.gpu

ROWSUM_PLANE = 3  # TF_GPU_DEBUG_ROWSUM_PLANE


def _read(ctx, fid, dtype, pl, x0, y0, w, h):
    dst = np.zeros((h, w), dtype)
    ctx._check(ctx.lib.tf_gpu_debug_read_plane(ctx.h, fid, pl, dst.ctypes.data, w, x0, y0, w, h))
    return dst


def _check_rowsums(ctx, b, fid):
    """The plane over its whole defined region against numpy row sums of the slot's own luma plane."""
    db = ctx.device_border()
    aw, ah = b.aligned[0]
    luma = _read(ctx, fid, b.dtype, 0, -db, -db, aw + 2 * db, ah + 2 * db).astype(np.int64)
    c = np.concatenate([np.zeros((luma.shape[0], 1), np.int64), np.cumsum(luma, axis=1)], axis=1)
    want = c[:, 16:] - c[:, :-16]  # want[:, j] = sum of luma[:, j .. j + 15]
    got = _read(ctx, fid, np.uint16, ROWSUM_PLANE, -db, -db, want.shape[1], want.shape[0])
    assert (got.astype(np.int64) == want).all(), int((got != want).sum())
    return want


# (W, H, bit depth, content): "texture" is the moving-texture clip, "max" every sample at full range
CASES = {"8bit": (352, 288, 8, "texture"), "10bit": (353, 289, 10, "texture"), "12bit": (200, 136, 12, "texture"),
         "12bit_full_range": (200, 136, 12, "max")}


@pytest.mark.parametrize("case", sorted(CASES))
@pytest.mark.parametrize("route", ["host", "device"])
def test_rowsum_plane_equals_numpy(pkg, tfgpu, case, route):
    W, H, bd, content = CASES[case]
    planes = _clips.moving_texture(W, H, 1, bd)[0]
    if content == "max":
        planes = tuple(np.full_like(a, (1 << bd) - 1) for a in planes)
    fid = 930001
    if route == "host":
        b = pkg.Yv12Buffer(W, H, 1, 1, bd > 8, 160, False, frame_id=fid).set_planes(*planes, extend=False)
        tfgpu.cache_frame(b)
    else:
        b = pkg.Yv12Buffer(W, H, 1, 1, bd > 8, 160, False, frame_id=fid)
        tens = [torch.from_numpy(a.view(np.int16) if a.dtype == np.uint16 else a).cuda() for a in planes]
        tfgpu.cache_frame_tensor(fid, *tens)
        torch.cuda.synchronize()
    try:
        want = _check_rowsums(tfgpu, b, fid)
        if content == "max":
            assert (want == 16 * 4095).all()  # 65,520: the top of the uint16 range the plane relies on
    finally:
        tfgpu.evict_frame(fid)


def _constant_rows(W, H, N, bd, seed):
    """Every luma row constant (a random level per row, shifted down by one row per frame): the row sums of a
    candidate are 16 x its rows' levels, so the bound equals the skip-row SAD at every site."""
    r = np.random.default_rng(seed)
    maxv = (1 << bd) - 1
    dt = np.uint8 if bd == 8 else np.uint16
    levels = r.integers(0, maxv + 1, H + N)
    frames = []
    for f in range(N):
        y = np.repeat(levels[N - f:N - f + H, None], W, axis=1).astype(dt)
        u = np.full(((H + 1) // 2, (W + 1) // 2), maxv // 2, dt)
        frames.append((y, u, u.copy()))
    return frames


@pytest.mark.parametrize("bd", [8, 10])
def test_constant_rows_bound_equals_sad_matches_oracle(pkg, tfgpu, bd):
    W, H, N = 352, 288, 5
    # skip-row SAD (the path the bound serves) at this size too
    p = _params.tf_params(W, H, N, bit_depth=bd, use_downsampled_sad=1)
    frames = _constant_rows(W, H, N, bd, 40 + bd)
    g = _gpu.run_gpu(pkg, tfgpu, p, frames)
    o = _gpu.oracle_run(p, frames)
    rep = _gpu.compare(g, o, p, tol_out=1)
    assert rep["mvs"] == 0 and rep["mses"] == 0 and rep["pred"] == 0, rep
    assert rep["out_bad"] == 0 and rep["diff_equal"], rep


def test_bound_skips_sites_and_counters_change_nothing(pkg):
    W, H, N, bd = 1280, 720, 5, 10
    frames = _clips.moving_texture(W, H, N, bd)
    p = _params.tf_params(W, H, N, bit_depth=bd)
    ctx = pkg.TemporalFilterGpu(device=0)
    try:
        plain = _gpu.run_gpu(pkg, ctx, p, frames)
        ctx.collect_counters(True)
        counted = _gpu.run_gpu(pkg, ctx, p, frames)
        ctr = ctx.read_counters()
        ctx.collect_counters(False)
    finally:
        ctx.close()
    assert ctr[0] > 0 and ctr[3] > 0, ctr
    for k in ("mvs", "mses", "pred", "diff"):
        assert (plain[k] == counted[k]).all(), k
    for a, b in zip(plain["out"], counted["out"]):
        assert (a == b).all()
