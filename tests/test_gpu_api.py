"""GPU: the C ABI beyond the plain filter call -- reference fixtures, device frame cache,
resident variant, slab (row-range) mode, async submit/wait, error behaviour."""
import os

import numpy as np
import pytest

import _clips
import _gpu
import _params
from golden.make_golden import PIPELINE_CASES, make_frames

pytestmark = pytest.mark.gpu
G = np.load(os.path.join(os.path.dirname(__file__), "golden", "golden_r01.npz"))


@pytest.mark.parametrize("case", PIPELINE_CASES, ids=[c[0] for c in PIPELINE_CASES])
def test_gpu_matches_reference_fixture(pkg, tfgpu, case):
    """CUDA path vs outputs of the unmodified reference (no oracle in between)."""
    name, W, H, N, bd, kind, ckw, pkw = case
    frames = make_frames(kind, W, H, N, bd, ckw, pkw)
    p = _params.tf_params(W, H, N, bit_depth=bd, **pkw)
    b = pkg.Yv12Buffer(W, H, p["ss_x"], p["ss_y"], p["use_hbd"], p["border"], p["monochrome"])
    b.set_planes(*frames[p["filter_frame_idx"]])
    noise = [tfgpu.estimate_noise_from_single_plane(b, pl, bd) for pl in range(b.num_planes)]
    assert noise == list(G[f"{name}/noise"][: len(noise)])
    p["noise_levels"] = tuple(G[f"{name}/noise"])
    g = _gpu.run_gpu(pkg, tfgpu, p, frames)
    sel = [f for f in range(N) if f != p["filter_frame_idx"]]
    assert (g["mvs"][:, sel] == G[f"{name}/mvs"][:, sel]).all()
    assert (g["mses"][:, sel] == G[f"{name}/mses"][:, sel]).all()
    w = np.arange(1, g["pred"].shape[2] + 1, dtype=np.uint64)
    assert (g["pred"].astype(np.uint64).sum(axis=2)[:, sel] == G[f"{name}/pred_sum"][:, sel]).all()
    assert ((g["pred"].astype(np.uint64) * w).sum(axis=2)[:, sel] == G[f"{name}/pred_wsum"][:, sel]).all()
    bad = 0
    for i, out in enumerate(g["out"]):
        d = np.abs(out.astype(np.int32) - G[f"{name}/out{i}"].astype(np.int32))
        assert d.max() <= 1  # +-1 LSB bar for the float-weighted output
        bad += int((d > 0).sum())
    assert bad == 0, f"{bad} pixels differ by 1 LSB"  # in practice bit-exact
    assert (g["diff"] == G[f"{name}/diff"]).all()


def _bufs(pkg, p, frames, id_base):
    out = []
    for i, (y, u, v) in enumerate(frames):
        b = pkg.Yv12Buffer(p["width"], p["height"], p["ss_x"], p["ss_y"], p["use_hbd"], p["border"],
                           p["monochrome"], frame_id=id_base + i if id_base else 0)
        out.append(b.set_planes(y, u, v, extend=False))
    return out


def test_frame_cache_and_resident_call(pkg, tfgpu):
    W, H, N = 352, 288, 5
    frames = _clips.moving_texture(W, H, N, 10)
    p = _params.tf_params(W, H, N, bit_depth=10)
    ref = _gpu.run_gpu(pkg, tfgpu, p, frames, dump=False)
    bufs = _bufs(pkg, p, frames, 5000)
    for b in bufs:
        tfgpu.cache_frame(b)
    ms, diff = tfgpu.filter_resident(p, [b.frame_id for b in bufs])
    assert ms > 0 and (diff == ref["diff"]).all()
    out = pkg.Yv12Buffer(W, H, 1, 1, True, p["border"])
    tfgpu.download_output(out)
    for pl in range(3):
        assert (out.full_blocks(pl) == ref["out"][pl]).all()
    # cached ids are reused: overwrite the host copies, the result must not change
    for b in bufs:
        for a in b.alloc:
            a[:] = 0
    out2 = pkg.Yv12Buffer(W, H, 1, 1, True, p["border"])
    r2 = tfgpu.temporal_filter(p, bufs, out2)
    assert (r2["diff"] == ref["diff"]).all()
    tfgpu.evict_frame(bufs[0].frame_id)
    with pytest.raises(pkg.TfGpuError):
        tfgpu.filter_resident(p, [b.frame_id for b in bufs])
    for b in bufs:
        tfgpu.evict_frame(b.frame_id)


def test_slab_rows_equal_full_frame(pkg, tfgpu):
    """Slab mode (4K config): disjoint block-row ranges computed separately equal the full run;
    FRAME_DIFF adds up."""
    W, H, N = 352, 288, 3
    frames = _clips.moving_texture(W, H, N, 8)
    p = _params.tf_params(W, H, N)
    full = _gpu.run_gpu(pkg, tfgpu, p, frames, dump=False)
    mb_rows = (H + 31) // 32
    out = pkg.Yv12Buffer(W, H, 1, 1, False, p["border"])
    diff = np.zeros(2, np.int64)
    for b, e in ((0, 4), (4, mb_rows)):
        q = dict(p, out_row_begin=b, out_row_end=e)
        r = tfgpu.temporal_filter(q, _bufs(pkg, p, frames, 0), out)
        diff += r["diff"]
    for pl in range(3):
        assert (out.full_blocks(pl) == full["out"][pl]).all()
    assert (diff == full["diff"]).all()


def test_async_submit_wait(pkg, tfgpu):
    W, H, N = 176, 144, 3
    frames = _clips.moving_texture(W, H, N, 8)
    p = _params.tf_params(W, H, N)
    full = _gpu.run_gpu(pkg, tfgpu, p, frames, dump=False)
    outs = [pkg.Yv12Buffer(W, H, 1, 1, False, p["border"]) for _ in range(3)]
    bufs = _bufs(pkg, p, frames, 0)
    tickets = [tfgpu.submit(p, bufs, o) for o in outs]
    for (t, diff, _keep), o in zip(tickets, outs):
        tfgpu.wait(t)
        assert [diff[0], diff[1]] == list(full["diff"])
        assert (o.full_blocks(0) == full["out"][0]).all()


@pytest.mark.parametrize("slots", [0, 24], ids=["default-cache", "smallest-cache"])
def test_pipelined_submits_of_different_windows(pkg, slots):
    """Several different windows submitted back to back on one context (uploads of window k+1
    overlap the kernels of window k; uncached frames, id 0).  With the smallest cache (24 slots,
    15-frame windows) the second window has to reuse slots of the window still in flight, which
    must wait for it."""
    W, H, N = 320, 192, 15
    ctx = pkg.TemporalFilterGpu(max_cached_frames=slots)
    try:
        p = _params.tf_params(W, H, N, bit_depth=10)
        wins = [_clips.moving_texture(W, H, N, 10, seed=900 + k, motion=(k % 3, 1 + k % 4)) for k in range(5)]
        want = [_gpu.run_gpu(pkg, ctx, p, fr, dump=False) for fr in wins]
        bufs = [_bufs(pkg, p, fr, 0) for fr in wins]
        for rep in range(2):
            outs = [pkg.Yv12Buffer(W, H, 1, 1, True, p["border"]) for _ in wins]
            tickets = [ctx.submit(p, b, o) for b, o in zip(bufs, outs)]
            for (t, diff, _keep), o, w in zip(tickets, outs, want):
                ctx.wait(t)
                assert [diff[0], diff[1]] == list(w["diff"])
                for pl in range(3):
                    assert (o.full_blocks(pl) == w["out"][pl]).all()
    finally:
        ctx.close()


def test_invalid_arguments_return_errors(pkg, tfgpu):
    W, H, N = 64, 64, 3
    frames = _clips.moving_texture(W, H, N, 8)
    p = _params.tf_params(W, H, N)
    bufs = _bufs(pkg, p, frames, 0)
    out = pkg.Yv12Buffer(W, H, 1, 1, False, p["border"])
    for bad in (dict(num_frames=0), dict(num_frames=99), dict(filter_frame_idx=7), dict(bit_depth=9),
                dict(subpel_method=5), dict(filter_strength=9)):
        with pytest.raises(pkg.TfGpuError) as e:
            tfgpu.temporal_filter(dict(p, **bad), bufs, out)
        assert e.value.code == -1
    with pytest.raises(pkg.TfGpuError):  # 8-bit container with bit_depth 10
        tfgpu.temporal_filter(dict(p, bit_depth=10), bufs, out)
    # the context stays usable after an error
    tfgpu.temporal_filter(p, bufs, out)


def test_single_frame_window_is_identity(pkg, tfgpu):
    """arnr_max_frames = 1 disables filtering (temporal_filter.c:995-997): only the self term."""
    W, H = 96, 64
    frames = _clips.moving_texture(W, H, 1, 8)
    p = _params.tf_params(W, H, 1)
    g = _gpu.run_gpu(pkg, tfgpu, p, frames, dump=False)
    assert (g["out"][0][:H, :W] == frames[0][0]).all()
    assert (g["diff"] == 0).all()


@pytest.mark.parametrize("case", [(352, 288, 8, 96), (200, 120, 10, 160), (131, 77, 8, 160)])
def test_output_border_extension_matches_reference(pkg, tfgpu, case):
    """SURVEY 8a row 13 / 8f rank 2: aom_extend_frame_borders (yv12extend.c:221), which the caller runs
    right after av1_temporal_filter (temporal_filter.c:1372), done on the device; the whole extended
    allocation must equal the reference's (the oracle's where oracle/_ref is not built)."""
    import _ref
    W, H, bd, border = case
    N = 3
    frames = _clips.moving_texture(W, H, N, bd)
    p = _params.tf_params(W, H, N, bit_depth=bd, border=border)
    r = _ref.reference_or_oracle(p, frames)
    p["noise_levels"] = tuple(r.estimate_noise())
    r.close()
    r = _ref.reference_or_oracle(p, frames)
    r.run(record=False)
    r.extend_output_borders()
    out = pkg.Yv12Buffer(W, H, 1, 1, p["use_hbd"], border)
    tfgpu.temporal_filter(dict(p, extend_output_borders=1), _bufs(pkg, p, frames, 0), out)
    for pl in range(3):
        ref_plane, _ = r.plane_with_border(-1, pl)
        assert ref_plane.shape == out.alloc[pl].shape
        assert (ref_plane == out.alloc[pl]).all(), pl
    r.close()


@pytest.mark.parametrize("dims", [(352, 288, 8, 1, 1, 96), (131, 77, 10, 1, 1, 160), (130, 70, 8, 0, 0, 160), (1920, 1080, 10, 1, 1, 160)],
                         ids=["cif8", "odd10", "odd_i444", "1080p10"])
def test_device_input_plane_border_equals_copy_and_extend_frame(pkg, tfgpu, dims):
    """SURVEY 8a row 2, read back directly: only the crop area of a host frame crosses PCIe and
    extend_borders_kernel rebuilds the replication; the device plane -- border included, as far as the device
    border reaches -- must be sample-identical to what the reference's av1_copy_and_extend_frame
    (av1/encoder/extend.c:113-163) leaves in the lookahead slot (the oracle's copy where oracle/_ref is not built)."""
    import _ref
    W, H, bd, sx, sy, border = dims
    frames = _clips.moving_texture(W, H, 1, bd, ss_x=sx, ss_y=sy)
    p = _params.tf_params(W, H, 1, bit_depth=bd, ss_x=sx, ss_y=sy, border=border)
    r = _ref.reference_or_oracle(p, frames)
    # host frame WITHOUT borders: whatever lies outside the crop area on the device was built there
    b = pkg.Yv12Buffer(W, H, sx, sy, bd > 8, border, frame_id=777000 + W).set_planes(*frames[0], extend=False)
    tfgpu.cache_frame(b)
    db = tfgpu.device_border()
    for pl in range(3):
        k = 1 if pl else 0
        ref_plane, info = r.plane_with_border(0, pl)
        hb_x, hb_y = b.borders[k]
        aw, ah = b.aligned[k]
        ex = min(db >> (sx if pl else 0), hb_x)
        ey = min(db >> (sy if pl else 0), hb_y)
        got = tfgpu.debug_read_plane(b, pl, -ex, -ey, aw + 2 * ex, ah + 2 * ey)
        want = ref_plane[hb_y - ey:hb_y + ah + ey, hb_x - ex:hb_x + aw + ex]
        assert got.shape == want.shape
        assert (got.astype(np.uint16) == want).all(), (pl, int((got.astype(np.uint16) != want).sum()))
    tfgpu.evict_frame(b.frame_id)
    r.close()
