"""CPU: tfo_predict_block (tests/_oracle_predict.c), the oracle of tf_gpu_predict_device.  It equals tfo_run's pred
recorder at the MVs tfo_run records, which pins it to the oracle already pinned to the reference, and at far MVs it
equals tfo_convolve12 on an edge-padded copy of the crop area with a 320-sample border (wider than any read)."""
import numpy as np
import pytest

import _clips
import _oracle
import _oracle_predict
import _params

PAD = 320


def _plane_shape(p, plane, B):
    return (B >> p["ss_y"], B >> p["ss_x"]) if plane else (B, B)


def _quadrant(p, entry, num_planes, q, B=32):
    """Quadrant q of a 32x32 pred entry as the pred layout of a 16-item."""
    parts, off = [], 0
    for pl in range(num_planes):
        h, w = _plane_shape(p, pl, B)
        a = entry[off:off + h * w].reshape(h, w)
        parts.append(a[(q >> 1) * h // 2:((q >> 1) + 1) * h // 2, (q & 1) * w // 2:((q & 1) + 1) * w // 2].ravel())
        off += h * w
    return np.concatenate(parts)


CASES = [  # name, W, H, N, bit depth, clip options, params options
    ("i420_8", 176, 144, 3, 8, dict(motion=(2, 3)), dict(allow_hp=1)),
    ("i420_10_odd", 200, 136, 3, 10, dict(motion=(3, 1)), dict(speed=0, allow_hp=1)),
    ("i422_12", 216, 120, 3, 12, dict(motion=(1, 2), ss_x=1, ss_y=0), dict(ss_x=1, ss_y=0, speed=2)),
    ("i444_8in16", 96, 64, 3, 8, dict(motion=(2, 1), ss_x=0, ss_y=0), dict(ss_x=0, ss_y=0, use_hbd=1)),
    ("mono10", 131, 77, 3, 10, dict(monochrome=True), dict(monochrome=1)),
]


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_equals_the_pred_recorder(case):
    name, W, H, N, bd, ckw, pkw = case
    frames = _clips.moving_texture(W, H, N, bd, **ckw)
    p = _params.tf_params(W, H, N, bit_depth=bd, **pkw)
    o = _oracle.OracleFilter(p, frames)
    r = o.run()
    o.close()
    m = _oracle_predict.PredictOracle(p, frames)
    np_ = 1 if p["monochrome"] else 3
    checked = whole = 0
    for blk in range(r["mvs"].shape[0]):
        by, bx = 32 * (blk // o.mb_cols), 32 * (blk % o.mb_cols)
        for f in range(N):
            if f == p["filter_frame_idx"]:
                continue
            mvs = r["mvs"][blk, f]
            for q in range(4):
                got = m.predict_block(f, 16, bx + 16 * (q & 1), by + 16 * (q >> 1), int(mvs[q, 0]), int(mvs[q, 1]), np_)
                assert (got == _quadrant(p, r["pred"][blk, f], np_, q)).all(), (name, blk, f, q)
                checked += 1
            if (mvs == mvs[0]).all():
                got = m.predict_block(f, 32, bx, by, int(mvs[0, 0]), int(mvs[0, 1]), np_)
                assert (got == r["pred"][blk, f]).all(), (name, blk, f)
                whole += 1
    m.close()
    assert checked and whole
    assert (r["mvs"] & 7 != 0).any() or p["bit_depth"] == 12  # sub-pel MVs among those checked


def _padded_reference(plane, x0, y0, w, h, mv_row, mv_col, ssy, ssx, ah, aw, bd, hbd, lib):
    """build_predictor's position rule restated, and tfo_convolve12 on np.pad(mode="edge") of the crop plane."""
    pos_y = ((y0 << 4) + mv_row * (1 << (1 - ssy))) * 64 + 32
    pos_x = ((x0 << 4) + mv_col * (1 << (1 - ssx))) * 64 + 32
    pos_y = min(max(pos_y, -(((288 >> ssy) - 4) << 10)), (ah + 4) << 10)
    pos_x = min(max(pos_x, -(((288 >> ssx) - 4) << 10)), (aw + 4) << 10)
    oy, ox = pos_y >> 10, pos_x >> 10
    padded = np.ascontiguousarray(np.pad(plane.astype(np.uint16), PAD, mode="edge"))
    assert PAD + oy - 5 >= 0 and PAD + ox - 5 >= 0
    assert PAD + oy + h + 6 <= padded.shape[0] and PAD + ox + w + 6 <= padded.shape[1]
    dst = np.zeros((h, w), np.uint16)
    st = padded.shape[1]
    lib.tfo_convolve12(padded.ctypes.data + 2 * ((PAD + oy) * st + PAD + ox), st, dst.ctypes.data, w, w, h,
                       (pos_x & 1023) >> 6, (pos_y & 1023) >> 6, bd, hbd)
    return dst


FAR_MVS = [(-32768, -32768), (32767, 32767), (-32768, 32767), (32767, -32768), (-2296, 5), (3, -2290), (-8, 8),
           (-300 * 8 + 3, 17), (9, 4000 * 8 + 5), (-2000, -2001), (2001, 1999)]


@pytest.mark.parametrize("bd, ss", [(8, (1, 1)), (10, (1, 0)), (12, (1, 1)), (12, (0, 0))])
def test_far_mvs_equal_the_padded_convolve(bd, ss):
    W, H = 72, 40
    frames = _clips.random_frames(W, H, 1, bd, seed=bd, ss_x=ss[0], ss_y=ss[1])
    p = _params.tf_params(W, H, 1, bit_depth=bd, ss_x=ss[0], ss_y=ss[1])
    m = _oracle_predict.PredictOracle(p, frames)
    lib = _oracle_predict.lib()
    rng = np.random.default_rng(bd)
    mvs = FAR_MVS + [tuple(int(v) for v in rng.integers(-32768, 32768, 2)) for _ in range(20)]
    mvs += [(int(r), int(c)) for r in range(8) for c in range(8)]  # every 1/8-pel phase, near the frame
    _oracle_predict.reset_stats()
    aw, ah = -(-W // 8) * 8, -(-H // 8) * 8
    for bsize in (16, 32):
        for x, y in ((0, 0), (aw - 16, ah - 4) if bsize == 16 else (aw - 32, ah - 8), (16, 8)):
            for mv in mvs:
                got = m.predict_block(0, bsize, x, y, mv[0], mv[1], 3)
                parts = []
                for pl in range(3):
                    ssy, ssx = (ss[1], ss[0]) if pl else (0, 0)
                    k = 1 if pl else 0
                    h, w = 16 >> ssy, 16 >> ssx
                    blk = np.zeros((bsize >> ssy, bsize >> ssx), np.uint16)
                    for q in range(4 if bsize == 32 else 1):
                        i, j = (q >> 1) * h, (q & 1) * w
                        blk[i:i + h, j:j + w] = _padded_reference(
                            frames[0][pl], (x >> ssx) + j, (y >> ssy) + i, w, h, mv[0], mv[1], ssy, ssx,
                            ah >> ssy if k else ah, aw >> ssx if k else aw, bd, p["use_hbd"], lib)
                    parts.append(blk.ravel())
                assert (got == np.concatenate(parts)).all(), (bsize, x, y, mv)
    st = _oracle_predict.get_stats()
    m.close()
    assert st["pred_clip_lo"] > 0 and st["pred_clip_hi"] > 0, st
