"""Coded-size cases shared by test_oracle_coded_size.py (CPU) and test_gpu_coded_size.py (GPU).

Under superres or spatial resize the encoder's coded size (cm->width / cm->height) and its mi grid
(cm->mi_params) differ from the crop size of the frames the temporal filter reads.  The library takes them from
tf_gpu_params (mi_rows, mi_cols, cm_width, cm_height, border_in_pixels); the oracle from the same-named keys of the
params dict.  A case names a frame size, a coded size, the grid align8(coded) / 4, a border and the content."""
import _clips
import _content
import _params


def align8(v):
    return (v + 7) // 8 * 8


def coded_params(W, H, cw, ch, num_frames, border=None, **kw):
    """tf_params for a W x H frame whose coded size is cw x ch and whose mi grid is align8(coded) / 4."""
    p = _params.tf_params(W, H, num_frames, border=border, **kw)
    p.update(cm_width=cw, cm_height=ch, mi_rows=align8(ch) // 4, mi_cols=align8(cw) // 4)
    return p


def frames(content, W, H, N, bd, seed=0):
    if content == "random":
        return _clips.random_frames(W, H, N, bd, seed=seed)
    if content == "texture":
        return _clips.moving_texture(W, H, N, bd, seed=seed, motion=(2, 3))
    if content == "large_motion":
        return _content.large_motion(W, H, N, bd, seed=seed, velocity=(6, 40))
    return _content.make(content, W, H, N, bd, seed=seed)


# name, (W, H), (coded W, coded H), border, bit depth, use_hbd, speed, allow_hp, force_integer_mv, content,
# oracle block rows (None: the whole frame), oracle counters that must be > 0
CASES = [  # oracle and GPU windows have five frames, so a ref_mv reset reaches a later search
    # superres denominator 16 at 4K: the right half's 32x32 blocks have inverted column limits, the start is clamped
    ("a_4k_sr16_10", (3840, 2160), (1920, 2160), 288, 10, 1, 4, 0, 0, "large_motion", ((0, 1), (40, 41), (67, 68)),
     ("lim_inverted", "start_clamped", "mv_on_limit")),
    # superres denominator 9: the grid ends 208 px before the frame edge; starts clamped into non-empty ranges
    ("b_1080_sr9_8", (1920, 1080), (1707, 1080), 288, 8, 0, 2, 1, 0, "sharp_edges", ((0, 1), (33, 34)),
     ("start_clamped", "mv_on_limit")),
    # resize 1/2: both grids shrink, low-res cost class and threshold 3 on an HD frame
    ("c_720_half_12", (1280, 720), (640, 360), None, 12, 1, 0, 1, 0, "texture", ((0, 2), (11, 12), (22, 23)),
     ("start_clamped", "mv_on_limit")),
    # resize 3/4: medium cost class, 8-bit samples in a 16-bit container
    ("d_720_3q_8in16", (1280, 720), (960, 540), None, 8, 1, 3, 1, 0, "large_motion", ((0, 1), (16, 17), (22, 23)),
     ("start_clamped", "mv_on_limit")),
    # low-res class on a frame whose crop size is HD; integer MVs
    ("e_768_half_10_fim", (768, 768), (384, 768), None, 10, 1, 2, 0, 1, "texture", None,
     ("start_clamped", "mv_on_limit")),
    # small frame, the all-intra border
    ("f_cif_half_8", (352, 288), (176, 288), 64, 8, 0, 4, 1, 0, "random", None, ("start_clamped", "mv_on_limit")),
]

# coded = frame; av1_set_mv_{row,col}_limits' border term binds for a 32x32 block only below 48
BORDERS = (40, 44, 47, 48, 64, 96, 160, 288, 1024)
BORDER_SIZES = ((640, 360, None), (1920, 1080, ((0, 1), (17, 18), (33, 34))))


N = 5  # frames per window: the ref_mv chain carries a reset past the centre frame


def case_params(case, N=N):
    name, (W, H), (cw, ch), border, bd, hbd, speed, hp, fim, content, rows, _ = case
    return coded_params(W, H, cw, ch, N, border=border, bit_depth=bd, use_hbd=hbd, speed=speed, allow_hp=hp,
                        force_integer_mv=fim)


def case_frames(case, N=N):
    name, (W, H), _, _, bd, *_rest = case
    return frames(case[9], W, H, N, bd, seed=CASES.index(case) + 1 if case in CASES else 1)


def border_params(W, H, border, N, bd=8, speed=4):
    p = _params.tf_params(W, H, N, bit_depth=bd, speed=speed, border=border)
    return p
