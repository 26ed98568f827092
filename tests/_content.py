"""Seeded, deterministic adversarial content for the parity tests.

The clips of _clips.py are textured noise kept inside [0.11, 0.89] * max and moving by whole pixels. The
generators here produce what real frames have and those clips never do: exact ties in the motion search
(periodic patterns), the samples that push the 12-tap predictor's 2-D intermediate out of int16 (tap_pattern),
full-range edges that make the predictor clamp at both ends (sharp_edges), sub-pel motion with chroma moving
along (subpel_pan), pans far beyond the search window and onto the MV limits (large_motion), scene cuts and
fades (scene_cut, fade).

Every generator has the signature gen(width, height, num_frames, bit_depth=8, ss_x=1, ss_y=1, monochrome=False,
seed=0, **options) and returns [(y, u, v)] in the container dtype (u8 for 8-bit, u16 above; u and v are None when
monochrome).  Frames are rendered in float64, then rounded and clipped; only numpy and scipy.ndimage are used, so
a seed fixes every sample.
"""
import numpy as np
from scipy import ndimage

# MULTITAP_SHARP2 phase 8 (half pel), av1/common/filter.h:159-177 -- its positive taps
_K12_HALF = (-2, 4, -7, 13, -25, 81, 81, -25, 13, -7, 4, -2)


def _maxv(bd):
    return (1 << bd) - 1


def _dtype(bd):
    return np.uint8 if bd == 8 else np.uint16


def _q(a, bd):
    return np.clip(np.rint(a), 0, _maxv(bd)).astype(_dtype(bd))


def _chroma(a, ss_x, ss_y):
    """Average (1 << ss_y) x (1 << ss_x) luma-resolution samples into one chroma sample (edge-padded)."""
    h, w = a.shape
    ch, cw = (h + ss_y) >> ss_y, (w + ss_x) >> ss_x
    a = np.pad(a, ((0, (ch << ss_y) - h), (0, (cw << ss_x) - w)), mode="edge")
    return a.reshape(ch, 1 << ss_y, cw, 1 << ss_x).mean(axis=(1, 3))


def _frames(planes, bd, ss_x, ss_y, monochrome):
    """planes: per frame (Y, U, V) float64 at luma resolution -> [(y, u, v)] quantised, chroma subsampled."""
    out = []
    for y, u, v in planes:
        if monochrome:
            out.append((_q(y, bd), None, None))
        else:
            out.append((_q(y, bd), _q(_chroma(u, ss_x, ss_y), bd), _q(_chroma(v, ss_x, ss_y), bd)))
    return out


def _texture(rng, h, w, lo=0.2, hi=0.8, coarse=0.0, cell=32):
    """Box-blurred uniform noise rescaled to [lo, hi] (fractions of max); `coarse` mixes in a smooth field of
    `cell`-pixel features, which gives the diamond search a wide basin to descend far."""
    t = ndimage.uniform_filter(rng.random((h, w)), size=5, mode="wrap")
    if coarse:
        g = rng.random((h // cell + 3, w // cell + 3))
        t = (1 - coarse) * t + coarse * ndimage.zoom(g, cell, order=3, mode="nearest")[:h, :w]
    t = (t - t.min()) / (t.max() - t.min())
    return lo + (hi - lo) * t


def _shift(a, dy, dx, order=1):
    """a sampled at (y + dy, x + dx): exact slicing for whole pixels, scipy spline interpolation otherwise."""
    if float(dy).is_integer() and float(dx).is_integer():
        return np.roll(a, (-int(dy), -int(dx)), axis=(0, 1))
    return ndimage.shift(a, (-dy, -dx), order=order, mode="grid-wrap")


def _pan(canvases, n, velocity, height, width, order=1, origin=(0, 0)):
    """Frame n of a pan over the (periodic) canvases: each canvas sampled at origin + n * velocity, cropped."""
    dy, dx = origin[0] + n * velocity[0], origin[1] + n * velocity[1]
    return tuple(_shift(c, dy, dx, order)[:height, :width] for c in canvases)


def _uv_from(y, maxv):
    """Chroma that moves with luma: an affine image of it, one plane inverted."""
    return 0.25 * maxv + 0.5 * y, maxv - y


# ----------------------------------------------------------------------------------------------------------
def periodic(width, height, num_frames, bit_depth=8, ss_x=1, ss_y=1, monochrome=False, seed=0, kind="checker",
             period=8, motion=None, lo=0.0, hi=1.0):
    """Checkerboards, stripes, grids and random tiles of period `period` (4..16) moving by whole pixels.
    Motion defaults to one period along x plus a non-multiple along y.  kind: checker, hstripes, vstripes,
    grid (1-px lines every period), tile (a random period x period tile: 2-D periodic, so shifts by (+-p, 0)
    and (0, +-p) tie exactly).  Samples are lo / hi (fractions of max) except for tile."""
    rng = np.random.default_rng(seed)
    maxv = _maxv(bit_depth)
    p = int(period)
    if motion is None:
        motion = (int(rng.integers(1, p)), p)
    H = -(-(height + abs(motion[0]) * num_frames + p) // p) * p
    W = -(-(width + abs(motion[1]) * num_frames + p) // p) * p
    yy, xx = np.mgrid[0:H, 0:W]
    if kind == "checker":
        b = ((yy // (p // 2)) + (xx // (p // 2))) % 2
    elif kind == "hstripes":
        b = (yy % p) < p // 2
    elif kind == "vstripes":
        b = (xx % p) < p // 2
    elif kind == "grid":
        b = ((yy % p) == 0) | ((xx % p) == 0)
    elif kind == "tile":
        t = rng.random((p, p))
        b = t[yy % p, xx % p]
    else:
        raise ValueError(kind)
    y = maxv * (lo + (hi - lo) * b.astype(np.float64))
    planes = [(y, *_uv_from(y, maxv))]
    return _frames([_pan(planes[0], n, motion, height, width) for n in range(num_frames)],
                   bit_depth, ss_x, ss_y, monochrome)


def _tap_columns(n, x0=0):
    """1.0 where the half-pel 12-tap filter centred on column x0 (mod 12) has a positive tap, else 0.0."""
    k = (np.arange(n) - x0 + 5) % 12
    return (np.asarray(_K12_HALF)[k] > 0).astype(np.float64)


def tap_pattern(width, height, num_frames, bit_depth=8, ss_x=1, ss_y=1, monochrome=False, seed=0,
                kind="columns", motion=(0.5, 0.5)):
    """Binary {0, max} content that maximises the 12-tap predictor's horizontal sum, moving with a half-pel
    component (rendered by area coverage, i.e. linear interpolation of the binary pattern).
    kind "columns": the 12-periodic column pattern that is max under the positive taps of phase 8, XORed
    with the same pattern along rows (so vertical motion is visible).  At phase (8, 8) its 2-D intermediate
    reaches (max * 196 + 2^(bd+6)) >> r0, above int16 at 10 and 12 bit.
    kind "noise": uniform binary {0, max} noise; at 12 bit its SADs reach 16 differences of 4095 per group."""
    rng = np.random.default_rng(seed)
    maxv = _maxv(bit_depth)
    pad = int(np.ceil(max(abs(motion[0]), abs(motion[1])) * num_frames)) + 24
    H, W = height + pad, width + pad
    if kind == "columns":
        H, W = -(-H // 12) * 12, -(-W // 12) * 12
        a = _tap_columns(W, int(rng.integers(0, 12)))[None, :]
        b = _tap_columns(H, int(rng.integers(0, 12)))[:, None]
        y = maxv * (a + b - 2 * a * b)
    elif kind == "noise":
        y = maxv * rng.integers(0, 2, size=(H, W)).astype(np.float64)
    else:
        raise ValueError(kind)
    canv = (y, *_uv_from(y, maxv))
    return _frames([_pan(canv, n, motion, height, width) for n in range(num_frames)],
                   bit_depth, ss_x, ss_y, monochrome)


def sharp_edges(width, height, num_frames, bit_depth=8, ss_x=1, ss_y=1, monochrome=False, seed=0,
                motion=(0.5, 1.25), bar=None):
    """A textured background with full-range rectangles (0 and max), thin text-like strokes at max and 0,
    panning at a sub-pel velocity (linear interpolation), under static letterbox bars of exact 0 at the top
    and bottom (`bar` rows each, default height // 8)."""
    rng = np.random.default_rng(seed)
    maxv = _maxv(bit_depth)
    pad = int(np.ceil(max(abs(motion[0]), abs(motion[1])) * num_frames)) + 16
    H, W = height + pad, width + pad
    y = _texture(rng, H, W, 0.25, 0.75)
    for _ in range(max(4, H * W // 2000)):
        r0, c0 = int(rng.integers(0, H)), int(rng.integers(0, W))
        y[r0:r0 + int(rng.integers(3, 24)), c0:c0 + int(rng.integers(3, 24))] = float(rng.integers(0, 2))
    for _ in range(max(4, H * W // 1500)):  # strokes: 1-2 px wide, horizontal or vertical
        r0, c0, ln, wd = int(rng.integers(0, H)), int(rng.integers(0, W)), int(rng.integers(4, 16)), int(rng.integers(1, 3))
        v = float(rng.random() < 0.7)
        if rng.random() < 0.5:
            y[r0:r0 + wd, c0:c0 + ln] = v
        else:
            y[r0:r0 + ln, c0:c0 + wd] = v
    y *= maxv
    canv = (y, *_uv_from(y, maxv))
    bar = height // 8 if bar is None else bar
    planes = []
    for n in range(num_frames):
        fy, fu, fv = _pan(canv, n, motion, height, width)
        for f, val in ((fy, 0.0), (fu, 0.0), (fv, 0.0)):
            f[:bar] = val
            f[height - bar:] = val
        planes.append((fy, fu, fv))
    return _frames(planes, bit_depth, ss_x, ss_y, monochrome)


def subpel_pan(width, height, num_frames, bit_depth=8, ss_x=1, ss_y=1, monochrome=False, seed=0,
               velocity=(0.25, 0.5)):
    """A band-limited canvas (Gaussian-blurred noise) panned at a non-integer velocity in px per frame,
    resampled with cubic splines (scipy.ndimage.shift, order 3, periodic).  Chroma is derived from a second
    field of the same canvas and moves with luma."""
    rng = np.random.default_rng(seed)
    maxv = _maxv(bit_depth)
    pad = int(np.ceil(max(abs(velocity[0]), abs(velocity[1])) * num_frames)) + 16
    H, W = height + pad, width + pad

    def field():
        f = ndimage.gaussian_filter(rng.standard_normal((H, W)), 1.2, mode="wrap")
        return (f - f.mean()) / f.std()
    a, b = field(), field()
    y = maxv * np.clip(0.5 + 0.16 * a, 0.02, 0.98)
    u = maxv * np.clip(0.5 + 0.08 * b + 0.04 * a, 0.0, 1.0)
    v = maxv * np.clip(0.5 - 0.08 * b + 0.04 * a, 0.0, 1.0)
    return _frames([_pan((y, u, v), n, velocity, height, width, order=3) for n in range(num_frames)],
                   bit_depth, ss_x, ss_y, monochrome)


def large_motion(width, height, num_frames, bit_depth=8, ss_x=1, ss_y=1, monochrome=False, seed=0,
                 velocity=(6, 40)):
    """A fast pan (whole pixels, 20..150 px per frame), so that the outer frames of a window are hundreds of
    pixels away.  The canvas is a ramp along the motion plus a smooth field of 64-pixel features plus fine
    texture: the SAD falls steadily towards the true offset, so the diamond and mesh searches walk far and,
    where the true offset lies beyond the search range, stop on the frame-edge limits or, at >= 1080p with
    >= 74 px per frame over 15 frames, on the +-1023 clamp."""
    rng = np.random.default_rng(seed)
    maxv = _maxv(bit_depth)
    H = height + abs(int(velocity[0])) * num_frames + 8
    W = width + abs(int(velocity[1])) * num_frames + 8
    yy, xx = np.mgrid[0:H, 0:W] / float(max(H, W))
    sy, sx = np.sign(velocity[0]), np.sign(velocity[1])
    ramp = sy * yy + sx * xx
    ramp = (ramp - ramp.min()) / max(1e-9, ramp.max() - ramp.min())
    y = maxv * (0.05 + 0.55 * ramp + 0.3 * _texture(rng, H, W, 0.0, 1.0, coarse=0.9, cell=64)
                + 0.05 * _texture(rng, H, W, 0.0, 1.0))
    canv = (y, *_uv_from(y, maxv))
    origin = tuple(max(0, -int(v) * (num_frames - 1)) for v in velocity)  # every crop inside the canvas
    return _frames([_pan(canv, n, velocity, height, width, origin=origin) for n in range(num_frames)],
                   bit_depth, ss_x, ss_y, monochrome)


def scene_cut(width, height, num_frames, bit_depth=8, ss_x=1, ss_y=1, monochrome=False, seed=0, cut=None,
              motion=(1, 2)):
    """Frames [0, cut) pan over one texture, frames [cut, N) over an unrelated one (default cut = N // 2 + 1,
    just after the middle frame): the blocks' errors against the other scene exceed the ref_mv reset threshold
    and their weights go to near zero."""
    cut = num_frames // 2 + 1 if cut is None else cut
    rng = np.random.default_rng(seed)
    maxv = _maxv(bit_depth)
    H, W = height + abs(motion[0]) * num_frames + 8, width + abs(motion[1]) * num_frames + 8
    scenes = []
    for lo, hi in ((0.1, 0.9), (0.0, 1.0)):
        y = maxv * _texture(rng, H, W, lo, hi)
        scenes.append((y, *_uv_from(y, maxv)))
    return _frames([_pan(scenes[n >= cut], n, motion, height, width) for n in range(num_frames)],
                   bit_depth, ss_x, ss_y, monochrome)


def fade(width, height, num_frames, bit_depth=8, ss_x=1, ss_y=1, monochrome=False, seed=0, motion=(1, 1),
         gain=(1.0, 0.05)):
    """A pan whose brightness ramps linearly from gain[0] to gain[1] (a fade to black): growing block errors,
    ref_mv resets and small weights, with the darkest frames close to 0."""
    rng = np.random.default_rng(seed)
    maxv = _maxv(bit_depth)
    H, W = height + abs(motion[0]) * num_frames + 8, width + abs(motion[1]) * num_frames + 8
    y = maxv * _texture(rng, H, W, 0.1, 1.0)
    canv = (y, *_uv_from(y, maxv))
    planes = []
    for n in range(num_frames):
        g = gain[0] + (gain[1] - gain[0]) * n / max(1, num_frames - 1)
        fy, fu, fv = _pan(canv, n, motion, height, width)
        mid = 0.5 * maxv  # chroma fades towards grey
        planes.append((g * fy, mid + g * (fu - mid), mid + g * (fv - mid)))
    return _frames(planes, bit_depth, ss_x, ss_y, monochrome)


def edge_ramp(width, height, bit_depth=10, slope=9):
    """One 4:2:0 frame of horizontal ramps rising by `slope` per sample (V falling): the Sobel magnitude is
    8 * slope at every interior pixel, so with slope 9 at 10 bit ((72 + 2) >> 2 = 18) no pixel is below an edge
    threshold of 16 and the noise estimate has nothing to count (its -1.0 branch), while every pixel is below 50."""
    cw, ch = (width + 1) >> 1, (height + 1) >> 1
    y = np.tile(np.arange(width) * slope, (height, 1)).astype(_dtype(bit_depth))
    u = np.tile(np.arange(cw) * slope, (ch, 1)).astype(_dtype(bit_depth))
    return [(y, u, u[:, ::-1].copy())]


CLASSES = {
    "periodic": periodic,
    "tap_pattern": tap_pattern,
    "sharp_edges": sharp_edges,
    "subpel_pan": subpel_pan,
    "large_motion": large_motion,
    "scene_cut": scene_cut,
    "fade": fade,
}


def make(cls, width, height, num_frames, bit_depth=8, **kw):
    return CLASSES[cls](width, height, num_frames, bit_depth, **kw)
