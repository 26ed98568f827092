"""GPU: tf_gpu_fullpel_search_batch -- the full-pixel search engine as a batch call (SURVEY 8f rank 4: the first
consumer beyond the temporal filter) -- against the reference's own av1_full_pixel_search() (mcomp.c:1693-1832) run
per block through the compiled, unmodified reference (oracle/_ref, tfref_full_pixel_search: configured as
tf_motion_search() configures it, the same NSTEP search first_pass_motion_search(), firstpass.c:261-300, and TPL's
motion_estimation(), tpl_model.c:285, run per 16x16 / 32x32 block); where oracle/_ref is not built, the oracle's
restatement of that search (tfo_full_pixel_search).  Best MV and returned variance cost must be equal for every
block: 16x16 and 32x32 blocks on the macroblock grid, zero and random start MVs, frame edges."""
import numpy as np
import pytest

import _clips
import _params
import _ref

pytestmark = pytest.mark.gpu

CASES = [  # name, W, H, bit depth, clip motion, params
    ("cif8_s4", 352, 288, 8, (1, 2), {}),
    ("cif10_s4", 352, 288, 10, (2, 3), {}),
    ("hd8_skip", 1280, 720, 8, (3, 5), {}),                  # >= 720p: skip-row SAD + audit, HDRES cost class
    ("hd10_skip", 1280, 720, 10, (4, 7), {}),
    ("qcif8_s0_mesh", 176, 144, 8, (6, 9), dict(speed=0)),  # mesh search never pruned
    ("vga8_s3", 640, 480, 8, (0, 11), dict(speed=3, q_factor=12)),  # MIDRES cost class, LVL_1 pruning off (q <= 20)
    ("odd8", 200, 136, 8, (1, 1), {}),
]


@pytest.mark.parametrize("case", CASES, ids=[c[0] for c in CASES])
@pytest.mark.parametrize("bsize", [16, 32])
def test_batch_search_equals_reference_full_pixel_search(pkg, tfgpu, case, bsize):
    name, W, H, bd, motion, pkw = case
    frames = _clips.moving_texture(W, H, 2, bd, motion=motion)
    p = _params.tf_params(W, H, 2, bit_depth=bd, **pkw)
    r = _ref.reference_or_oracle(p, frames)
    bufs = [pkg.Yv12Buffer(W, H, 1, 1, bd > 8, p["border"], frame_id=880000 + 10 * CASES.index(case) + i).set_planes(*f, extend=False)
            for i, f in enumerate(frames)]
    rng = np.random.default_rng(1234 + bsize)
    aw, ah = bufs[0].aligned[0]
    items = []
    for y in range(0, ah, bsize):
        for x in range(0, aw, 16 if bsize == 16 else 32):
            kind = rng.integers(0, 4)
            if kind == 0:
                sr, sc = 0, 0
            elif kind == 1:  # near the true motion
                sr, sc = -motion[0] + int(rng.integers(-2, 3)), -motion[1] + int(rng.integers(-2, 3))
            else:
                sr, sc = int(rng.integers(-40, 41)), int(rng.integers(-40, 41))
            items.append((x, y, sr, sc))
    if len(items) > 400:  # the reference runs one block at a time on the CPU
        keep = sorted(set(rng.choice(len(items), 400, replace=False).tolist()) | {0, len(items) - 1})
        items = [items[i] for i in keep]
    got = tfgpu.fullpel_search_batch(p, bufs[0], bufs[1], bsize, items)
    bad = []
    for i, (x, y, sr, sc) in enumerate(items):
        want = r.full_pixel_search(0, 1, bsize, x, y, sr, sc)
        if tuple(int(v) for v in got[i]) != tuple(want):
            bad.append((items[i], tuple(int(v) for v in got[i]), want))
    assert not bad, (len(bad), len(items), bad[:5])
    for b in bufs:
        tfgpu.evict_frame(b.frame_id)
    r.close()


def test_batch_search_rejects_bad_items(pkg, tfgpu):
    W, H = 352, 288
    frames = _clips.moving_texture(W, H, 2, 8)
    p = _params.tf_params(W, H, 2)
    bufs = [pkg.Yv12Buffer(W, H, 1, 1, False, p["border"]).set_planes(*f) for f in frames]
    for item in [(8, 0, 0, 0), (0, 2, 0, 0), (-16, 0, 0, 0), (352, 0, 0, 0), (0, 288, 0, 0)]:
        with pytest.raises(pkg.TfGpuError) as e:
            tfgpu.fullpel_search_batch(p, bufs[0], bufs[1], 16, [item])
        assert e.value.code == -1
    with pytest.raises(pkg.TfGpuError):
        tfgpu.fullpel_search_batch(p, bufs[0], bufs[1], 24, [(0, 0, 0, 0)])
    assert tfgpu.fullpel_search_batch(p, bufs[0], bufs[1], 16, []).shape == (0, 3)
