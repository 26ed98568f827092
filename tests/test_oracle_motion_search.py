"""CPU: the oracle's per-block motion search (tests/_oracle_motion.c, tfo_motion_search: tf_motion_search()'s
full-pel search, then its sub-pel search or, under force_integer_mv, the variance at the full-pel MV) is composed of
the pinned pieces: its full-pel part equals the pinned library's tfo_full_pixel_search, and on the 32x32 blocks the
pinned library's tfo_run leaves unsplit it reproduces what tfo_run recorded for them."""
import ctypes as C

import numpy as np
import pytest

import _clips
import _content
import _oracle
import _oracle_motion
import _params

W, H = 256, 192


def _items(bsize, rng, n=40):
    out = [(0, 0, 0, 0), (W - bsize, H - bsize, 0, 0)]  # frame corners
    while len(out) < n:
        x = int(rng.integers(0, W // 16)) * 16
        y = int(rng.integers(0, H // 4)) * 4
        if x + bsize > W or y + bsize > H:
            continue
        out.append((x, y, int(rng.integers(-40, 41)), int(rng.integers(-40, 41))))
    return out


@pytest.mark.parametrize("bd, speed", [(8, 4), (10, 2), (12, 0), (8, 3)])
@pytest.mark.parametrize("bsize", [16, 32])
def test_fullpel_part_equals_full_pixel_search(bd, speed, bsize):
    frames = _content.subpel_pan(W, H, 2, bd, velocity=(0.75, -1.5))
    p = _params.tf_params(W, H, 2, bit_depth=bd, speed=speed, allow_hp=1)
    o = _oracle.OracleFilter(p, frames)
    om = _oracle_motion.MotionOracle(p, frames)
    # the sub-pel stage starts at the full-pel MV; each of its rounds (step 4, 2, 1) moves a component by at most
    # one step, or two with the second-level check of subpel_iters_per_step 2
    reach = 7 * p["subpel_iters_per_step"]
    for x, y, sr, sc in _items(bsize, np.random.default_rng(bd * 100 + speed + bsize)):
        m = om.motion_search(0, 1, bsize, x, y, sr, sc)
        assert m[:3] == o.full_pixel_search(0, 1, bsize, x, y, sr, sc), (x, y, sr, sc)
        assert abs(m[3] - 8 * m[0]) <= reach and abs(m[4] - 8 * m[1]) <= reach, m
    o.close()
    om.close()


@pytest.mark.parametrize("bd, kw, noisy", [(8, {}, False), (10, dict(speed=2, allow_hp=1), True), (8, dict(speed=0), False)])
def test_unsplit_blocks_match_tfo_run(bd, kw, noisy):
    """Frame 0 of a window whose filter frame is 1 or later is searched first, so its ref_mv chain starts at zero:
    the 32x32 search of every block there is motion_search from (0, 0).  Where the partition decision kept the
    32x32 result, all four recorded sub-blocks hold its MV and (err + 512) / 1024.  (At 10 bit the smooth sub-pel pan
    leaves block errors that round to an MSE of 0, which always splits: that case uses textured noise.)"""
    n = 3
    if noisy:
        frames = _clips.moving_texture(W, H, n, bd, motion=(1, 2))
    else:
        frames = _content.subpel_pan(W, H, n, bd, velocity=(0.25, 0.75))
    p = _params.tf_params(W, H, n, filter_frame_idx=1, bit_depth=bd, **kw)
    o = _oracle.OracleFilter(p, frames)
    om = _oracle_motion.MotionOracle(p, frames)
    r = o.run()
    mvs, mses = r["mvs"][:, 0], r["mses"][:, 0]
    # four equal records with a nonzero MSE: the decision kept the 32x32 result (an MSE of 0 always splits)
    unsplit = [b for b in range(len(mvs))
               if (mvs[b] == mvs[b, :1]).all() and (mses[b] == mses[b, 0]).all() and mses[b, 0] > 0]
    assert len(unsplit) >= len(mvs) // 4, (len(unsplit), len(mvs))
    for b in unsplit:
        br, bc = divmod(b, o.mb_cols)
        m = om.motion_search(1, 0, 32, bc * 32, br * 32, 0, 0)
        assert (m[3], m[4]) == tuple(int(v) for v in mvs[b, 0]), (b, m, mvs[b])
        assert (m[5] + 512) // 1024 == mses[b, 0], (b, m, mses[b])
    o.close()
    om.close()


@pytest.mark.parametrize("bd, hbd", [(8, 0), (10, 1), (8, 1)])
@pytest.mark.parametrize("bsize", [16, 32])
def test_force_integer_mv(bd, hbd, bsize):
    frames = _content.subpel_pan(W, H, 2, bd, velocity=(0.5, 1.25))
    base = _params.tf_params(W, H, 2, bit_depth=bd, use_hbd=hbd, speed=2)
    o = _oracle_motion.MotionOracle(base, frames)
    oi = _oracle_motion.MotionOracle(dict(base, force_integer_mv=1), frames)
    planes = _oracle.OracleFilter(base, frames)
    y0, info = planes.plane_with_border(1, 0)   # source
    y1, _ = planes.plane_with_border(0, 0)      # reference
    bw, bh = info["bw"], info["bh"]
    lib = _oracle.lib()
    for x, y, sr, sc in _items(bsize, np.random.default_rng(7 + bsize + bd), n=24):
        m = oi.motion_search(1, 0, bsize, x, y, sr, sc)
        assert m[:3] == o.motion_search(1, 0, bsize, x, y, sr, sc)[:3]  # the full-pel stage does not change
        assert (m[3], m[4]) == (8 * m[0], 8 * m[1])
        src = np.ascontiguousarray(y0[bh + y:bh + y + bsize, bw + x:bw + x + bsize])
        ref = np.ascontiguousarray(y1[bh + y + m[0]:bh + y + m[0] + bsize, bw + x + m[1]:bw + x + m[1] + bsize])
        sse = C.c_uint()
        var = lib.tfo_variance(ref.ctypes.data, bsize, src.ctypes.data, bsize, bsize, bsize, bd, hbd, C.byref(sse))
        assert m[5] == var, (x, y, m, var)
    o.close()
    oi.close()
    planes.close()


def test_periodic_content_reaches_subpel_ties():
    """Every block of the grid, the ones that stick out of the frame included, of a moving checkerboard searched
    against three frames: some sub-pel candidates tie with the incumbent exactly, so the strict comparison of the
    sub-pel search is exercised (the GPU parity cases on periodic content rely on it)."""
    w, h = 176, 144
    frames = _content.periodic(w, h, 5, 8, kind="checker", period=8)
    o = _oracle_motion.MotionOracle(_params.tf_params(w, h, 5), frames)
    _oracle_motion.reset_stats()
    for ref in (0, 1, 4):
        for bsize in (16, 32):
            for y in range(0, h, bsize):
                for x in range(0, w, bsize):
                    o.motion_search(2, ref, bsize, x, y, 0, 0)
    assert _oracle_motion.get_stats()["subpel_ties"] > 0
    o.close()
