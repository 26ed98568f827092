"""CPU: oracle vs the compiled, unmodified reference (oracle/_ref/libtf_ref.so, built by
oracle/Makefile from /root/reference).  Skipped where the .so is absent."""
import ctypes as C

import numpy as np
import pytest

import _clips
import _oracle
import _params
import _ref

pytestmark = pytest.mark.skipif(not _ref.available(), reason="oracle/_ref/libtf_ref.so not built")

CASES = [
    ("cif8", 352, 288, 7, 8, "m", {}, {}),
    ("cif10", 352, 288, 5, 10, "m", {}, {}),
    ("qcif8_s0", 176, 144, 3, 8, "m", {}, dict(speed=0)),
    ("qcif10_s1_hp", 176, 144, 3, 10, "m", {}, dict(speed=1, allow_hp=1)),
    ("s2_motion", 200, 120, 4, 8, "m", dict(motion=(3, 5)), dict(speed=2)),
    ("s3_q15", 128, 96, 3, 12, "m", {}, dict(speed=3, q_factor=15)),
    ("hbd8_q200", 128, 96, 3, 8, "m", {}, dict(use_hbd=1, q_factor=200, filter_strength=2)),
    ("i444", 130, 70, 3, 8, "m", {}, dict(ss_x=0, ss_y=0)),
    ("i422_10", 130, 70, 3, 10, "m", {}, dict(ss_x=1, ss_y=0, speed=1)),
    ("mono_last", 131, 77, 4, 8, "m", {}, dict(monochrome=1, filter_frame_idx=3)),
    ("intmv", 128, 96, 3, 10, "m", {}, dict(force_integer_mv=1, speed=0)),
    ("rand8", 160, 96, 3, 8, "r", {}, {}),
    ("rand10_s0", 160, 96, 3, 10, "r", {}, dict(speed=0)),
    ("extreme", 96, 64, 3, 8, "r", dict(extreme=0), {}),
    ("hd_skip", 1280, 720, 2, 8, "m", {}, {}),
    ("hd_skip_rand_kf", 1280, 720, 2, 8, "r", {}, dict(filter_frame_idx=0)),
    ("speed4_hp_8", 176, 144, 3, 8, "m", dict(motion=(1, 3)), dict(allow_hp=1)),
    ("speed4_hp_10", 176, 144, 3, 10, "m", dict(motion=(2, 1)), dict(allow_hp=1)),
    ("speed1_tree_iters2_8", 176, 144, 3, 8, "m", dict(motion=(2, 3)), dict(speed=1)),
    ("pruned_iters2_hp", 176, 144, 3, 8, "m", dict(motion=(1, 2)), dict(speed=3, subpel_iters_per_step=2, allow_hp=1)),
    ("pruned_more_iters2_10", 176, 144, 3, 10, "m", dict(motion=(3, 1)), dict(subpel_iters_per_step=2)),
    ("strength0_q5", 128, 96, 3, 8, "m", {}, dict(filter_strength=0, q_factor=5)),
    ("strength6_q255", 128, 96, 3, 10, "m", {}, dict(filter_strength=6, q_factor=255)),
    ("long_window_21", 96, 64, 21, 8, "m", dict(motion=(0, 1)), dict(filter_frame_idx=10)),
    ("tiny_17x33_10", 17, 33, 3, 10, "m", {}, dict(speed=1)),
]


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
def test_oracle_equals_reference(case):
    name, W, H, N, bd, kind, ckw, pkw = case
    kw = dict(ss_x=pkw.get("ss_x", 1), ss_y=pkw.get("ss_y", 1), monochrome=pkw.get("monochrome", 0))
    frames = (_clips.moving_texture(W, H, N, bd, **kw, **ckw) if kind == "m"
              else _clips.random_frames(W, H, N, bd, seed=3, **kw, **ckw))
    p = _params.tf_params(W, H, N, bit_depth=bd, **pkw)
    r, o = _ref.RefFilter(p, frames), _oracle.OracleFilter(p, frames)
    assert r.estimate_noise() == o.estimate_noise()
    a, b = r.run(), o.run()
    for k in ("mvs", "mses", "pred", "diff"):
        assert (a[k] == b[k]).all(), k
    for x, y in zip(a["out"], b["out"]):
        assert (x == y).all()
    # replicated borders equal the reference's av1_copy_and_extend_frame
    pb, info = r.plane_with_border(0, 0)
    ob, oinfo = o.plane_with_border(0, 0)
    assert pb.shape == ob.shape and (pb == ob).all()
    r.close()
    o.close()


# coded size and grid decoupled from the crop size (superres / resize): name, W, H, coded W, coded H, N, bit depth,
# border, parameter options
CODED_CASES = [
    ("half_720_lowres", 1280, 720, 640, 360, 5, 10, 160, dict(speed=4)),
    ("sr9_wide_mid", 704, 544, 626, 544, 4, 8, 288, dict(speed=2, allow_hp=1)),
    ("half_width_inverted", 2816, 64, 1408, 64, 3, 8, 288, dict(speed=0)),  # column limits invert for x > 2439
]
# (no border below 64 here: the reference's frames are allocated with border_in_pixels, and a chroma predictor at
# such a border's MV limit reads past them; the oracle's frames have a border of at least 64)


@pytest.mark.parametrize("case", CODED_CASES, ids=[c[0] for c in CODED_CASES])
def test_oracle_equals_reference_on_coded_sizes(case):
    """cm->width / cm->height and cm->mi_params set apart from the crop size: the cost class, the ref_mv reset
    threshold and the MV limits (inverted ones included) follow them in both."""
    name, W, H, cw, ch, N, bd, border, pkw = case
    frames = _clips.moving_texture(W, H, N, bd, motion=(2, 9))
    p = _params.tf_params(W, H, N, bit_depth=bd, border=border, **pkw)
    p.update(cm_width=cw, cm_height=ch, mi_rows=(ch + 7) // 8 * 2, mi_cols=(cw + 7) // 8 * 2)
    r, o = _ref.RefFilter(p, frames), _oracle.OracleFilter(p, frames)
    a, b = r.run(), o.run()
    for k in ("mvs", "mses", "pred", "diff"):
        assert (a[k] == b[k]).all(), k
    for x, y in zip(a["out"], b["out"]):
        assert (x == y).all()
    r.close()
    o.close()


def test_od_divu_equals_division_exhaustive():
    """OD_DIVU (aom_dsp/odintrin.h:30-42) uses a multiply-shift table for d < 1024; the product
    and the oracle use plain division.  Proven equal for every count in [1000,1023] and every
    accum + count/2 a 21-frame window of 12-bit samples can reach."""
    lib = _ref.lib()
    lib.tfref_od_divu_mismatches.restype = C.c_longlong
    assert lib.tfref_od_divu_mismatches(1000, 1023, 21000 * 4095 + 10500) == 0
