"""CPU: the oracle (oracle/tf_oracle.c) against fixtures generated from the unmodified
reference (tests/golden/make_golden.py).  Bit-exact on everything, including the
float-weighted output (same libm on both sides)."""
import ctypes as C
import os

import numpy as np
import pytest

import _oracle
import _params
from golden.make_golden import PIPELINE_CASES, make_frames

G = np.load(os.path.join(os.path.dirname(__file__), "golden", "golden_r01.npz"))


@pytest.mark.parametrize("case", PIPELINE_CASES, ids=[c[0] for c in PIPELINE_CASES])
def test_pipeline_matches_reference_fixture(case):
    name, W, H, N, bd, kind, ckw, pkw = case
    frames = make_frames(kind, W, H, N, bd, ckw, pkw)
    p = _params.tf_params(W, H, N, bit_depth=bd, **pkw)
    o = _oracle.OracleFilter(p, frames)
    noise = o.estimate_noise()
    assert list(G[f"{name}/noise"][: len(noise)]) == noise
    p["noise_levels"] = tuple(G[f"{name}/noise"])
    o.close()
    o = _oracle.OracleFilter(p, frames)
    r = o.run()
    o.close()
    assert (r["mvs"] == G[f"{name}/mvs"]).all()
    assert (r["mses"] == G[f"{name}/mses"]).all()
    assert (r["diff"] == G[f"{name}/diff"]).all()
    for i, out in enumerate(r["out"]):
        assert (out == G[f"{name}/out{i}"]).all()
    w = np.arange(1, r["pred"].shape[2] + 1, dtype=np.uint64)
    assert (r["pred"].astype(np.uint64).sum(axis=2) == G[f"{name}/pred_sum"]).all()
    assert ((r["pred"].astype(np.uint64) * w).sum(axis=2) == G[f"{name}/pred_wsum"]).all()


@pytest.mark.parametrize("bd", [8, 10])
@pytest.mark.parametrize("ss", [(1, 1), (1, 0), (0, 0)])
@pytest.mark.parametrize("extreme", [None, 0, 1])
def test_apply_filter_block_vectors(bd, ss, extreme):
    """The fixed-parameter block test of test/temporal_filter_test.cc:130-260 (seed 0xbaba,
    sigma 2.1002103677063437, mvs {0,0},{5,5},{7,8},{2,10}, mses 15..18, q 12, strength 5)."""
    sx, sy = ss
    rng = np.random.default_rng(0xbaba)
    use_hbd = bd > 8
    dt = np.uint16 if use_hbd else np.uint8
    maxv = (1 << bd) - 1
    cw, ch = 32 >> sx, 32 >> sy
    stride, uvstride = 64, 64 >> sx

    def mk(h, w, st):
        buf = np.zeros((h, st), dt)
        buf[:, :w] = rng.integers(0, maxv + 1, size=(h, w)) if extreme is None else (maxv if extreme else 0)
        return buf
    y, u, v = mk(32, 32, stride), mk(ch, cw, uvstride), mk(ch, cw, uvstride)
    num_pels = 1024 + 2 * cw * ch
    pred = (rng.integers(0, maxv + 1, size=num_pels) if extreme is None
            else np.full(num_pels, 0 if extreme else maxv)).astype(dt)
    noise = np.array([2.1002103677063437] * 3)
    mvs = np.array([[0, 0], [5, 5], [7, 8], [2, 10]], np.int16)
    mses = np.array([15, 16, 17, 18], np.int32)
    accum = np.zeros(num_pels, np.uint32)
    count = np.zeros(num_pels, np.uint16)
    ptr = lambda a: a.ctypes.data_as(C.c_void_p)
    _oracle.lib().tfo_apply_block(540, 360, sx, sy, 3, bd, int(use_hbd), ptr(y), ptr(u), ptr(v), stride, uvstride,
                                  0, 0, ptr(noise), ptr(mvs), ptr(mses), 12, 5, ptr(pred), ptr(accum), ptr(count))
    key = f"apply/bd{bd}_ss{sx}{sy}_ex{extreme}"
    assert (accum == G[key + "/accum"]).all()
    assert (count == G[key + "/count"]).all()


def test_full_pixel_search_matches_reference_fixture():
    """With force_integer_mv the filter's MV of a block is its 32x32 full-pel search from a zero start
    (temporal_filter.c:94-176), so the reference's stored MVs of that case pin the oracle's per-block
    av1_full_pixel_search entry point (tfo_full_pixel_search) on every block, frame edges included."""
    name, W, H, N, bd, kind, ckw, pkw = next(c for c in PIPELINE_CASES if c[0] == "intmv8")
    frames = make_frames(kind, W, H, N, bd, ckw, pkw)
    p = _params.tf_params(W, H, N, bit_depth=bd, **pkw)
    o = _oracle.OracleFilter(p, frames)
    fi, mb_cols = p["filter_frame_idx"], (W + 31) // 32
    mvs = G[f"{name}/mvs"]
    for b in range(mvs.shape[0]):
        y, x = (b // mb_cols) * 32, (b % mb_cols) * 32
        for f in (f for f in range(N) if f != fi):
            row, col, _ = o.full_pixel_search(fi, f, 32, x, y, 0, 0)
            assert (row * 8, col * 8) == tuple(mvs[b, f, 0]), (b, f)
    o.close()


def test_od_divu_is_plain_division():
    # the exhaustive proof against the reference's table lives in test_oracle_vs_ref.py
    assert _oracle.lib().tfo_od_divu(21000 * 4095 + 10500, 21000) == (21000 * 4095 + 10500) // 21000
