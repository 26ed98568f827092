"""GPU: CUDA path vs oracle on adversarial content (tests/_content.py) -- exact ties in the diamond, mesh and
sub-pel stages, the int16 wrap of the 12-tap predictor's 2-D intermediate, full-range edges that clamp the
predictor at both ends, sub-pel and large motion up to the +-1023 MV clamp, scene cuts and fades, windows of 22
to 24 frames, 12-bit extremes and the noise estimate.  The bar is test_gpu_fuzz's: MVs, MSEs, predictors, accum
and count bit-exact, output within 1 LSB, FRAME_DIFF equal."""
import os

import numpy as np
import pytest

import _clips
import _content
import _gpu
import _oracle
import _params

pytestmark = pytest.mark.gpu

CLASSES = tuple(_content.CLASSES)
# 8hbd: 8-bit samples in 16-bit containers (use_hbd = 1)
DEPTHS = (("8", 8, 0), ("10", 10, 1), ("12", 12, 1), ("8hbd", 8, 1))
SPEEDS = (0, 2, 3, 4)  # TREE / TREE / PRUNED / PRUNED_MORE, mesh prune levels 0 / 0 / 1 / 2
SIZES = ((176, 144), (200, 120), (257, 161), (320, 180), (189, 99), (352, 288))


def content_kwargs(cls, r):
    """Seeded options of one content class (r: numpy Generator)."""
    if cls == "periodic":
        p = int(r.choice([4, 6, 8, 12, 16]))
        kind = str(r.choice(["checker", "hstripes", "vstripes", "grid", "tile"]))
        my = int(r.integers(0, p))
        mx = int(r.choice([p, -p, int(r.integers(1, p)), 0]))
        return dict(kind=kind, period=p, motion=(my, mx), seed=int(r.integers(0, 1 << 20)))
    if cls == "tap_pattern":
        return dict(kind=str(r.choice(["columns", "noise"])),
                    motion=(float(r.choice([0.5, -0.5, 1.5])), float(r.choice([0.5, -0.5, 2.5]))),
                    seed=int(r.integers(0, 1 << 20)))
    if cls == "sharp_edges":
        return dict(motion=(float(r.choice([0.5, 0.25, -0.75, 1.0])), float(r.choice([1.25, -0.5, 0.375, 2.0]))),
                    seed=int(r.integers(0, 1 << 20)))
    if cls == "subpel_pan":
        return dict(velocity=(float(r.choice([0.25, 0.5, -0.75, 1.375])), float(r.choice([0.5, -0.75, 0.125, 2.25]))),
                    seed=int(r.integers(0, 1 << 20)))
    if cls == "large_motion":
        return dict(velocity=(int(r.integers(-8, 9)), int(r.choice([20, -24, 36, -48, 64]))),
                    seed=int(r.integers(0, 1 << 20)))
    if cls == "scene_cut":
        return dict(motion=(int(r.integers(0, 3)), int(r.integers(-3, 4))), seed=int(r.integers(0, 1 << 20)))
    if cls == "fade":
        g1 = float(r.choice([0.05, 0.6, 0.9, 0.97]))
        return dict(motion=(int(r.integers(0, 3)), int(r.integers(-2, 3))), gain=(1.0, g1),
                    seed=int(r.integers(0, 1 << 20)))
    raise ValueError(cls)


def fixed_cases():
    """Every class x bit depth x speed at 4:2:0, plus 4:4:4, 4:2:2 and mono per class; seeded options."""
    cases = []
    for ci, cls in enumerate(CLASSES):
        for di, (dname, bd, hbd) in enumerate(DEPTHS):
            for si, speed in enumerate(SPEEDS):
                k = ci * 16 + di * 4 + si
                r = np.random.default_rng(5000 + k)
                W, H = SIZES[k % len(SIZES)]
                N = 3 + k % 3
                pkw = dict(speed=speed, use_hbd=hbd, filter_frame_idx=(N // 2 if k % 4 else 1))
                if cls == "tap_pattern":  # the filtered frame sits half a period between two binary frames
                    pkw["filter_frame_idx"] = 1
                cases.append((f"{cls}-{dname}-s{speed}", cls, W, H, N, bd, content_kwargs(cls, r), pkw))
        for fi, (fname, fmt) in enumerate((("444", (0, 0, 0)), ("422", (1, 0, 0)), ("mono", (1, 1, 1)))):
            k = ci * 3 + fi
            r = np.random.default_rng(6000 + k)
            dname, bd, hbd = DEPTHS[k % 4]
            W, H = SIZES[(k + 1) % len(SIZES)]
            pkw = dict(speed=SPEEDS[k % 4], use_hbd=hbd, ss_x=fmt[0], ss_y=fmt[1], monochrome=fmt[2], filter_frame_idx=1)
            cases.append((f"{cls}-{fname}-{dname}", cls, W, H, 3, bd, content_kwargs(cls, r), pkw))
    cases.append(("periodic-640x360-10", "periodic", 640, 360, 3, 10, dict(kind="tile", period=16, motion=(3, 16)),
                  dict(speed=4)))
    cases.append(("tap_pattern-640x360-12", "tap_pattern", 640, 360, 3, 12, dict(kind="columns"),
                  dict(speed=3, filter_frame_idx=1)))
    return cases


FIXED = fixed_cases()


def frames_of(cls, W, H, N, bd, ckw, pkw):
    return _content.make(cls, W, H, N, bd, ss_x=pkw.get("ss_x", 1), ss_y=pkw.get("ss_y", 1),
                         monochrome=pkw.get("monochrome", 0), **ckw)


def assert_parity(pkg, tfgpu, p, frames, what):
    g = _gpu.run_gpu(pkg, tfgpu, p, frames)
    o = _gpu.oracle_run(p, frames)
    rep = _gpu.compare(g, o, p, tol_out=1)
    assert rep["mvs"] == 0 and rep["mses"] == 0 and rep["pred"] == 0, (what, rep)
    assert rep["accum"] == 0 and rep["count"] == 0, (what, rep)
    assert rep["out_bad"] == 0 and rep["diff_equal"], (what, rep)


@pytest.mark.parametrize("case", FIXED, ids=[c[0] for c in FIXED])
def test_content_matrix(pkg, tfgpu, case):
    name, cls, W, H, N, bd, ckw, pkw = case
    p = _params.tf_params(W, H, N, bit_depth=bd, **pkw)
    assert_parity(pkg, tfgpu, p, frames_of(cls, W, H, N, bd, ckw, pkw), case)


def sweep_case(seed):
    """test_gpu_fuzz's parameter sampler with the content class drawn as well."""
    from test_gpu_fuzz import _case
    W, H, N, bd, kw, _, _ = _case(seed)
    r = np.random.default_rng(7000 + seed)
    cls = CLASSES[int(r.integers(0, len(CLASSES)))]
    W, H = max(W, 48), max(H, 40)
    if cls == "tap_pattern":
        N = max(N, 3)
        kw["filter_frame_idx"] = min(kw["filter_frame_idx"], N - 1)
    return W, H, N, bd, kw, cls, content_kwargs(cls, r)


_SEEDS = range(int(os.environ.get("TF_FUZZ_SEEDS", "100")))


@pytest.mark.parametrize("seed", _SEEDS)
def test_content_sweep(pkg, tfgpu, seed):
    W, H, N, bd, kw, cls, ckw = sweep_case(seed)
    p = _params.tf_params(W, H, N, bit_depth=bd, **kw)
    assert_parity(pkg, tfgpu, p, frames_of(cls, W, H, N, bd, ckw, kw), (seed, cls, W, H, N, bd, kw, ckw))


# large motion at full size: 150 px per frame along x, so the outer frames of the 15-frame window lie over
# 1000 px away and the rightward / leftward blocks stop on the +-1023 clamp.  Rows: top, bottom and rows whose
# blocks the oracle's counters show on a limit.
LARGE = [("1080p10", 1920, 1080, (0, 16, 33)), ("4k10", 3840, 2160, (0, 40, 67))]


@pytest.mark.parametrize("wl", LARGE, ids=[w[0] for w in LARGE])
def test_large_motion_full_size_rows(pkg, tfgpu, wl):
    _, W, H, rows = wl
    N, bd = 15, 10
    frames = _content.large_motion(W, H, N, bd, velocity=(0, 150), seed=11)
    p = _params.tf_params(W, H, N, bit_depth=bd, q_factor=32, filter_strength=5)
    bufs = []
    for (y, u, v) in frames:
        bufs.append(pkg.Yv12Buffer(W, H, 1, 1, True, p["border"]).set_planes(y, u, v, extend=False))
    full_out = pkg.Yv12Buffer(W, H, 1, 1, True, p["border"])
    full = tfgpu.temporal_filter(p, bufs, full_out)
    planes = [full_out.full_blocks(pl).copy() for pl in range(3)]
    o = _oracle.OracleFilter(p, frames)
    slab_out = pkg.Yv12Buffer(W, H, 1, 1, True, p["border"])
    clamped = 0
    for b in rows:
        _oracle.reset_stats()
        ref = o.run(record=False, rows=(b, b + 1))
        clamped += _oracle.get_stats()["mv_on_clamp"]
        got = tfgpu.temporal_filter(dict(p, out_row_begin=b, out_row_end=b + 1), bufs, slab_out)
        assert (got["diff"] == ref["diff"]).all(), b
        for pl in range(3):
            bh = 32 >> (1 if pl else 0)
            want = ref["out"][pl][b * bh:(b + 1) * bh]
            have = planes[pl][b * bh:(b + 1) * bh].astype(np.uint16)
            assert (want == have).all(), (pl, b, int((want != have).sum()))
    o.close()
    assert clamped > 0  # the rows compared hold MVs stopped by the +-1023 clamp
    assert full["diff"][0] > 0


LONG = [(N, fi) for N in (22, 23, 24) for fi in (0, N // 2, N - 1)]


@pytest.mark.parametrize("nf", LONG, ids=[f"n{n}_f{f}" for n, f in LONG])
def test_long_windows(pkg, tfgpu, nf):
    """Windows of 22 to 24 frames (the library's maximum is 24) under a fast pan."""
    N, fi = nf
    W, H, bd = 96, 64, 10 if N % 2 else 8
    frames = _content.large_motion(W, H, N, bd, velocity=(1, 20), seed=N)
    p = _params.tf_params(W, H, N, bit_depth=bd, filter_frame_idx=fi, speed=2 + (N % 3))
    assert_parity(pkg, tfgpu, p, frames, nf)


EXTREME12 = [(0, "speed4"), (1, "speed4"), (0, "speed0"), (1, "speed0")]


@pytest.mark.parametrize("ex", EXTREME12, ids=[f"parity{e}_{s}" for e, s in EXTREME12])
def test_extreme_12bit(pkg, tfgpu, ex):
    """Flat frames alternating 0 / 4095 (test/temporal_filter_test.cc:165-187) at 12 bit, both parities."""
    extreme, speed = ex
    W, H, N = 96, 64, 3
    frames = _clips.random_frames(W, H, N, 12, seed=3, extreme=extreme)
    p = _params.tf_params(W, H, N, bit_depth=12, speed=int(speed[-1]))
    assert_parity(pkg, tfgpu, p, frames, ex)


NOISE = [(cls, bd) for cls in CLASSES for bd in (8, 10, 12)]


@pytest.mark.parametrize("cb", NOISE, ids=[f"{c}-{b}" for c, b in NOISE])
def test_noise_estimate(pkg, tfgpu, cb):
    cls, bd = cb
    W, H = 200, 120
    r = np.random.default_rng(bd)
    frames = _content.make(cls, W, H, 1, bd, **content_kwargs(cls, r))
    p = _params.tf_params(W, H, 1, bit_depth=bd)
    b = pkg.Yv12Buffer(W, H, 1, 1, p["use_hbd"], p["border"]).set_planes(*frames[0])
    o = _oracle.OracleFilter(p, frames)
    for thr in (50, 16):
        exp = o.estimate_noise(0, edge_thresh=thr)
        got = [tfgpu.estimate_noise_from_single_plane(b, pl, bd, edge_thresh=thr) for pl in range(3)]
        assert got == exp, (cls, bd, thr, got, exp)
    o.close()


def test_noise_estimate_too_few_smooth_pixels(pkg, tfgpu):
    """Ramps of slope 9 at 10 bit: the rounded gradient magnitude (72 >> 2 = 18) is at or above an edge_thresh
    of 16 at every pixel, no pixel is counted and the estimate is -1.0 on the GPU as in the oracle; at
    edge_thresh 50 every pixel counts."""
    W, H, bd = 64, 48, 10
    frames = _content.edge_ramp(W, H, bd, slope=9)
    p = _params.tf_params(W, H, 1, bit_depth=bd)
    b = pkg.Yv12Buffer(W, H, 1, 1, True, p["border"]).set_planes(*frames[0])
    o = _oracle.OracleFilter(p, frames)
    for thr in (16, 50):
        exp = o.estimate_noise(0, edge_thresh=thr)
        got = [tfgpu.estimate_noise_from_single_plane(b, pl, bd, edge_thresh=thr) for pl in range(3)]
        assert got == exp, (thr, got, exp)
        assert (exp == [-1.0] * 3) == (thr == 16), (thr, exp)
    o.close()
