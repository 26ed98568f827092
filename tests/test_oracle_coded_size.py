"""CPU: the oracle on coded sizes and mi grids that differ from the crop size (superres, spatial resize) and on
border_in_pixels values where the border term of the MV limits binds.

tf_motion_search() takes the MV cost class and the ref_mv reset threshold from AOMMIN(cm->width, cm->height)
(temporal_filter.c:99-100,119-122,249-250) and the MV limits from cm->mi_params and oxcf.border_in_pixels
(mcomp.h:216-240); step_param (av1_init_search_range) and the weight's distance threshold (:603) use the size of
the frames.  These tests pin the oracle's restatement of that split, show that each case of
test_gpu_coded_size.py reaches the regime it is there for (oracle event counters, as test_content_coverage.py
does for content), and check the binding's new keys."""
import numpy as np
import pytest

import _clips
import _coded
import _oracle
import _oracle_motion
import _params
from test_gpu_fuzz import _case


def _fuzz(seed):
    W, H, N, bd, kw, clip, random_frames = _case(seed)
    fk = dict(ss_x=kw["ss_x"], ss_y=kw["ss_y"], monochrome=kw["monochrome"])
    frames = (_clips.random_frames(W, H, N, bd, seed=clip["seed"], **fk) if random_frames
              else _clips.moving_texture(W, H, N, bd, **fk, **clip))
    return _params.tf_params(W, H, N, bit_depth=bd, **kw), frames


def _run(p, frames, rows=None):
    o = _oracle.OracleFilter(p, frames)
    _oracle.reset_stats()
    r = o.run(rows=rows)
    st = _oracle.get_stats()
    o.close()
    return r, st


def _same(a, b):
    keys = ("mvs", "mses", "pred", "accum", "count", "diff")
    return all((a[k] == b[k]).all() for k in keys) and all((x == y).all() for x, y in zip(a["out"], b["out"]))


@pytest.mark.parametrize("seed", [0, 3, 7, 115, 426])
def test_zero_or_derived_values_keep_todays_results(seed):
    """The four fields at 0, or equal to what the oracle derives from the crop size, change nothing."""
    p, frames = _fuzz(seed)
    base, _ = _run(p, frames)
    zero, _ = _run(dict(p, mi_rows=0, mi_cols=0, cm_width=0, cm_height=0), frames)
    derived, _ = _run(dict(p, mi_rows=_coded.align8(p["height"]) // 4, mi_cols=_coded.align8(p["width"]) // 4,
                           cm_width=p["width"], cm_height=p["height"]), frames)
    assert _same(base, zero) and _same(base, derived), seed


def _limits_oracle(W, H, border, mi_rows=0, mi_cols=0):
    p = _params.tf_params(W, H, 1, border=border, mi_rows=mi_rows, mi_cols=mi_cols)
    return _oracle_motion.MotionOracle(p, _clips.random_frames(W, H, 1, 8))


# (frame W, H), border, (mi_rows, mi_cols) or None for the frame's grid, block size, (x, y)
#   -> (row_min, row_max, col_min, col_max), worked out by hand from av1_set_mv_{row,col}_limits and the +-1023 clamp
LIMITS = [
    # 4K, superres denominator 16: grid 540 x 480.  Rows as for the frame's own grid; columns inverted
    ((3840, 2160), 288, (540, 480), 32, (3808, 0), (-40, 1023, -1023, -1880)),
    ((3840, 2160), 288, None, 32, (3808, 0), (-40, 1023, -1023, 40)),
    ((3840, 2160), 288, (540, 480), 32, (3808, 1024), (-1023, 1023, -1023, -1880)),
    ((3840, 2160), 288, (540, 480), 32, (2944, 0), (-40, 1023, -1023, -1016)),   # the last column not inverted
    ((3840, 2160), 288, (540, 480), 32, (2976, 0), (-40, 1023, -1023, -1048)),   # the first inverted column
    # 1080p, denominator 9 (coded width 1707, grid 270 x 428): a non-empty range left of the block
    ((1920, 1080), 288, (270, 428), 32, (1888, 0), (-40, 1023, -1023, -168)),
    ((1920, 1080), 288, (270, 428), 16, (1696, 1072), (-1023, 16, -1023, 24)),
    # 720p resized to 640x360 (grid 90 x 160): both ranges lie above and left of the block
    ((1280, 720), 160, (90, 160), 32, (1248, 704), (-744, -336, -1023, -600)),
    # 640x360, 32x32 block at (320, 160): the border term binds below 48 ...
    ((640, 360), 40, None, 32, (320, 160), (-192, 200, -352, 320)),
    ((640, 360), 44, None, 32, (320, 160), (-196, 204, -356, 324)),
    ((640, 360), 47, None, 32, (320, 160), (-199, 207, -359, 327)),
    # ... and from 48 on the +-8 term sets every limit
    ((640, 360), 48, None, 32, (320, 160), (-200, 208, -360, 328)),
    ((640, 360), 288, None, 32, (320, 160), (-200, 208, -360, 328)),
    ((640, 360), 1024, None, 32, (320, 160), (-200, 208, -360, 328)),
    # a 16x16 block: the +-8 term binds at every border the library accepts
    ((640, 360), 40, None, 16, (320, 160), (-184, 208, -344, 328)),
    ((640, 360), 1024, None, 16, (320, 160), (-184, 208, -344, 328)),
]


@pytest.mark.parametrize("t", LIMITS, ids=[f"{t[0][0]}x{t[0][1]}-b{t[1]}-{t[3]}-{t[4][0]}_{t[4][1]}" for t in LIMITS])
def test_limit_table(t):
    (W, H), border, grid, bsize, (x, y), want = t
    mi_rows, mi_cols = grid or (0, 0)
    o = _limits_oracle(W, H, border, mi_rows, mi_cols)
    _oracle_motion.reset_stats()
    assert o.mv_limits(bsize, x, y) == want
    st = _oracle_motion.get_stats()
    assert (st["lim_inverted"] > 0) == (want[0] > want[1] or want[2] > want[3])
    assert (st["lim_border_bound"] > 0) == (bsize == 32 and border < 48)
    o.close()


def test_4k_start_is_clamped_onto_the_inverted_limit():
    """The 32x32 block at x = 3808 of a 4K frame coded at 1920 wide: the start MV 0 is clamped to col_max = -1880
    (clamp() tests the low bound first), no diamond or mesh site is in range, and the sub-pel range is empty, so the
    result is the clamped start, -15040 in 1/8 pel."""
    W, H = 3840, 2160
    frames = _coded.frames("large_motion", W, H, 2, 10)
    for speed in (0, 4):
        p = _coded.coded_params(W, H, 1920, 2160, 2, border=288, bit_depth=10, speed=speed)
        o = _oracle_motion.MotionOracle(p, frames)
        _oracle_motion.reset_stats()
        r = o.motion_search(0, 1, 32, 3808, 0, 0, 0)
        st = _oracle_motion.get_stats()
        assert r[:2] == (0, -1880) and r[3:5] == (0, -15040), (speed, r)
        assert st["lim_inverted"] > 0 and st["start_clamped"] > 0, st
        assert st["diamond_ties"] == 0 and st["subpel_ties"] == 0  # no candidate was ever evaluated
        o.close()


def _case_stats(case, N=_coded.N):
    p = _coded.case_params(case, N)
    frames = _coded.case_frames(case, N)
    rows = case[10]
    st = {k: 0 for k in _oracle.STAT_FIELDS}
    for rr in (rows or [None]):
        _, s = _run(p, frames, rows=rr)
        for k in st:
            st[k] += s[k]
    return st


@pytest.mark.parametrize("case", _coded.CASES, ids=[c[0] for c in _coded.CASES])
def test_gpu_case_reaches_its_target(case):
    st = _case_stats(case)
    assert all(st[k] > 0 for k in case[11]), (case[0], st)
    # border 288 and the all-intra border 64 never bind on their own
    assert st["lim_border_bound"] == 0, (case[0], st)


@pytest.mark.parametrize("border", _coded.BORDERS)
@pytest.mark.parametrize("size", _coded.BORDER_SIZES, ids=[f"{s[0]}x{s[1]}" for s in _coded.BORDER_SIZES])
def test_border_term_binds_only_below_48(size, border):
    W, H, rows = size
    p = _coded.border_params(W, H, border, 3)
    frames = _coded.frames("large_motion", W, H, 3, 8)
    st = {k: 0 for k in _oracle.STAT_FIELDS}
    for rr in (rows or [None]):
        _, s = _run(p, frames, rows=rr)
        for k in st:
            st[k] += s[k]
    assert (st["lim_border_bound"] > 0) == (border < 48), (border, st)


def test_border_below_48_changes_results_on_limit_content():
    """large_motion at 640x360: with border 40 the searches that stop on a frame-edge limit stop elsewhere than at
    border 48 (so a kernel that ignores P.border shows), and borders 48 and 1024 give identical results."""
    W, H, N = 640, 360, 3
    frames = _coded.frames("large_motion", W, H, N, 8)
    res = {b: _run(_coded.border_params(W, H, b, N), frames)[0] for b in (40, 48, 1024)}
    assert _same(res[48], res[1024])
    assert not (res[40]["mvs"] == res[48]["mvs"]).all()


def test_coded_size_selects_cost_class_and_threshold():
    """The same 1280x720 frames (large_motion, five frames, so the ref_mv chain carries a reset into the next
    search) coded at 640x360 (low-res class, threshold 3), 960x540 (medium class) and 1280x479 (low-res class) give
    MVs that differ from the crop size's (HD class, threshold 12) and, between the two classes, from each other.
    cm_width / cm_height at the crop size change nothing: the weights' distance threshold and step_param keep the
    crop size in every case."""
    W, H, N = 1280, 720, 5
    frames = _coded.frames("large_motion", W, H, N, 10)
    p = _params.tf_params(W, H, N, bit_depth=10, speed=4)
    rows = (10, 12)
    sel = slice(10 * 40, 12 * 40)
    res = {}
    for cw, ch in ((0, 0), (1280, 720), (640, 360), (960, 540), (1280, 479)):
        r, st = _run(dict(p, cm_width=cw, cm_height=ch), frames, rows)
        res[(cw, ch)] = (r["mvs"][sel], r["diff"], st["ref_mv_resets"])
    base = res[(0, 0)]
    assert (res[(1280, 720)][0] == base[0]).all() and (res[(1280, 720)][1] == base[1]).all()
    for k in ((640, 360), (960, 540), (1280, 479)):
        assert (res[k][0] != base[0]).any(), k
    assert (res[(640, 360)][0] != res[(960, 540)][0]).any()
    assert (res[(640, 360)][0] == res[(1280, 479)][0]).all()  # the class follows min(cm_width, cm_height)
    assert res[(640, 360)][2] > base[2]  # threshold 3 resets more often than 12


# ---- the binding's new keys (make_params) ------------------------------------------------------------------------
def test_make_params_coded_keys(pkg):
    p = _params.tf_params(1280, 720, 3)
    c = pkg.make_params(p)
    assert (c.mi_rows, c.mi_cols, c.cm_width, c.cm_height) == (180, 320, 0, 0)
    c = pkg.make_params(dict(p, mi_rows=90, mi_cols=160, cm_width=640, cm_height=360))
    assert (c.mi_rows, c.mi_cols, c.cm_width, c.cm_height) == (90, 160, 640, 360)
    c = pkg.make_params(dict(p, mi_rows=np.int64(135), mi_cols=None, cm_width=0))
    assert (c.mi_rows, c.mi_cols, c.cm_width) == (135, 320, 0)
    # the oracle receives the same values (tfo_set_coded)
    assert _oracle.coded_values(dict(p, mi_rows=90, mi_cols=160, cm_width=640, cm_height=360)) == (90, 160, 640, 360)
    assert _oracle.coded_values(p) == (0, 0, 0, 0)


@pytest.mark.parametrize("bad", [
    dict(mi_rows=0), dict(mi_cols=-4), dict(mi_rows=1.5), dict(mi_cols="160"), dict(mi_rows=True),
    dict(mi_rows=2 ** 31), dict(cm_width=-1), dict(cm_height=360.0), dict(cm_width=False), dict(cm_height=2 ** 40),
])
def test_make_params_rejects_bad_coded_keys(pkg, bad):
    with pytest.raises(ValueError):
        pkg.make_params(dict(_params.tf_params(1280, 720, 3), **bad))
