"""CPU: the content generators of _content.py reach what they target, shown by the oracle's event counters
(oracle/tf_oracle.h, tfo_stats), and a seed fixes every sample.  A class that reaches nothing would make its
GPU parity cases (test_gpu_content_parity.py) vacuous."""
import hashlib

import numpy as np
import pytest

import _content
import _oracle
import _params


def _stats(cls, W, H, N, bd, ckw=None, pkw=None, rows=None):
    pkw = dict(pkw or {})
    frames = _content.make(cls, W, H, N, bd, ss_x=pkw.get("ss_x", 1), ss_y=pkw.get("ss_y", 1),
                           monochrome=pkw.get("monochrome", 0), **(ckw or {}))
    p = _params.tf_params(W, H, N, bit_depth=bd, **pkw)
    o = _oracle.OracleFilter(p, frames)
    _oracle.reset_stats()
    r = o.run(record=rows is None, rows=rows)
    st = _oracle.get_stats()
    o.close()
    return st, r


# (class, bit depth, content options, parameter options, counters that must be > 0)
TARGETS = [
    ("periodic", 8, dict(kind="checker", period=8), {}, ("diamond_ties", "mesh_ties", "subpel_ties", "mesh_searches")),
    ("periodic", 10, dict(kind="tile", period=12, motion=(3, 12)), dict(speed=0),
     ("diamond_ties", "mesh_ties", "subpel_ties", "mesh_searches")),
    ("periodic", 12, dict(kind="grid", period=6), dict(speed=3), ("diamond_ties", "mesh_ties", "subpel_ties")),
    ("tap_pattern", 10, dict(kind="columns"), dict(filter_frame_idx=1), ("conv_im_overflow", "pred_clip_hi")),
    ("tap_pattern", 12, dict(kind="columns"), dict(filter_frame_idx=1), ("conv_im_overflow", "pred_clip_hi")),
    ("tap_pattern", 10, dict(kind="noise"), dict(filter_frame_idx=1), ("conv_im_overflow",)),
    ("tap_pattern", 12, dict(kind="noise"), dict(filter_frame_idx=1), ("conv_im_overflow", "sad_peak_groups")),
    ("sharp_edges", 8, {}, {}, ("pred_clip_lo", "pred_clip_hi")),
    ("sharp_edges", 10, {}, {}, ("pred_clip_lo", "pred_clip_hi")),
    ("sharp_edges", 12, {}, dict(speed=0), ("pred_clip_lo", "pred_clip_hi")),
    ("subpel_pan", 8, dict(velocity=(0.25, 0.5)), {}, ("subpel_ties",)),
    ("subpel_pan", 10, dict(velocity=(1.375, -0.75)), dict(speed=0, allow_hp=1), ("subpel_ties",)),
    ("large_motion", 10, dict(velocity=(6, 40)), {}, ("mesh_searches", "mesh_ties", "ref_mv_resets")),
    ("scene_cut", 8, {}, {}, ("ref_mv_resets", "mesh_searches")),
    ("fade", 10, {}, {}, ("ref_mv_resets",)),
]


@pytest.mark.parametrize("t", TARGETS, ids=[f"{t[0]}-{t[1]}-{i}" for i, t in enumerate(TARGETS)])
def test_class_reaches_its_target(t):
    cls, bd, ckw, pkw, want = t
    W, H = (320, 180) if cls == "large_motion" else (176, 144)
    N = 4 if cls == "tap_pattern" else 5
    st, _ = _stats(cls, W, H, N, bd, ckw, pkw)
    assert all(st[k] > 0 for k in want), (t, st)


def test_int16_wrap_changes_the_predictor():
    """The 12-periodic column pattern at phase (8, 8): the oracle's 2-D convolve narrows the intermediate to
    int16 as the reference does (convolve.c:96), and the wrap turns a max sample into 0."""
    for bd in (10, 12):
        maxv = (1 << bd) - 1
        col = _content._tap_columns(64, 20) * maxv
        src = np.ascontiguousarray(np.tile(col, (64, 1)).astype(np.uint16))
        dst = np.zeros((8, 8), np.uint16)
        _oracle.reset_stats()
        _oracle.lib().tfo_convolve12(src.ctypes.data + (20 * 64 + 20) * 2, 64, dst.ctypes.data, 8, 8, 8, 8, 8, bd, 1)
        assert _oracle.get_stats()["conv_im_overflow"] > 0
        assert src[20, 20] == maxv and dst[0, 0] == 0, (bd, dst[0, 0])


def test_subpel_pan_moves_by_fractions_of_a_pixel():
    """subpel_pan's MVs carry quarter-, half- and three-quarter-pel parts, and chroma moves with luma."""
    _, r = _stats("subpel_pan", 176, 144, 5, 8, dict(velocity=(0.25, 0.5)), dict(speed=0, allow_hp=1))
    sel = [f for f in range(5) if f != 2]
    frac = np.unique(r["mvs"][:, sel] & 7)
    assert {2, 4, 6} <= set(frac.tolist()), frac
    f = _content.subpel_pan(64, 64, 3, 8, velocity=(0.0, 1.0))
    assert (f[1][1][:, :-1] != f[0][1][:, :-1]).any()  # chroma changes with the pan


def test_large_motion_reaches_the_mv_clamp_at_1080p():
    """150 px per frame over 15 frames at 1080p: MVs of the top and bottom block rows stop on the +-1023
    clamp (the frame-edge limit is below -1023 there)."""
    hits = 0
    for row in (0, 33):
        st, _ = _stats("large_motion", 1920, 1080, 15, 10, dict(velocity=(0, 150), seed=11), {}, rows=(row, row + 1))
        hits += st["mv_on_clamp"]
        assert st["mesh_searches"] > 0
    assert hits > 0


def test_ref_mv_reset_boundary_is_reached():
    """block_mse == thresh exactly happens, so `>` vs `>=` in the ref_mv reset is observable."""
    st, _ = _stats("large_motion", 320, 180, 7, 10, dict(velocity=(6, 40)))
    assert st["block_mse_at_thresh"] > 0 and st["ref_mv_resets"] > 0, st


def test_edge_ramp_reaches_the_noise_estimate_minus_one_branch():
    """Fewer than 16 smooth pixels -> -1.0 (temporal_filter.c:1150-1194) at edge_thresh 16; 0.0 at 50 (all smooth)."""
    frames = _content.edge_ramp(64, 48, 10, slope=9)
    o = _oracle.OracleFilter(_params.tf_params(64, 48, 1, bit_depth=10), frames)
    assert o.estimate_noise(0, edge_thresh=16) == [-1.0] * 3
    assert o.estimate_noise(0, edge_thresh=50) == [0.0] * 3
    o.close()


def test_counters_only_observe():
    """Resetting and reading the counters leaves the oracle's results unchanged."""
    _, a = _stats("periodic", 96, 64, 3, 8, dict(kind="checker", period=4))
    _, b = _stats("periodic", 96, 64, 3, 8, dict(kind="checker", period=4))
    for k in ("mvs", "mses", "pred", "accum", "count", "diff"):
        assert (a[k] == b[k]).all()


# sha256 over every plane of every frame, per class at (72, 40, 3 frames, 10-bit, 4:2:0, seed 7)
HASHES = {
    "periodic": "e1b8cba551a19f2e765cd78e796ba49fcac28d161cb820739cb7bb0c06b10191",
    "tap_pattern": "ae6f1214cfba35a7d34c001deb97df0226aa388033f07dcbc9f9ea2555ab4780",
    "sharp_edges": "a101cf0dc3b50717dd6db734960189b69ce2fd7214d72c5e9f50c3ae627f393c",
    "subpel_pan": "7b95f3a6e61c724910eda8fbfb21b9c9b58b2ea28f263d87d3aee0a00ec33d55",
    "large_motion": "ac8945978c0a2d690bf75d819a80d1ec13c17ad6dfaf590e89c382ee94d1a037",
    "scene_cut": "2687f78a05dfd52eca7e5995178856683f3c58f7aba42d215b75d9c906dbca49",
    "fade": "6a81ecfd9529fd2d833e223100c1ab0e6f59222b83e2df02d0ba6dc0efe453a9",
}


def _digest(frames):
    h = hashlib.sha256()
    for planes in frames:
        for a in planes:
            if a is not None:
                h.update(str(a.dtype).encode() + str(a.shape).encode())
                h.update(np.ascontiguousarray(a).tobytes())
    return h.hexdigest()


@pytest.mark.parametrize("cls", sorted(HASHES))
def test_generator_is_deterministic(cls):
    a = _content.make(cls, 72, 40, 3, 10, seed=7)
    b = _content.make(cls, 72, 40, 3, 10, seed=7)
    assert _digest(a) == _digest(b)
    assert _digest(a) == HASHES[cls]
    for y, u, v in a:
        assert y.dtype == np.uint16 and y.shape == (40, 72) and u.shape == (20, 36) and v.shape == (20, 36)
        assert int(y.max()) <= 1023
    assert _content.make(cls, 72, 40, 1, 8, seed=7)[0][0].dtype == np.uint8
    assert _content.make(cls, 72, 40, 1, 8, seed=7, monochrome=True)[0][1] is None
