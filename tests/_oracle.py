"""ctypes binding for oracle/libtf_oracle.so (our C restatement of the reference
algorithm).  TEST INFRASTRUCTURE ONLY -- never imported by the product."""
import ctypes as C
import os
import subprocess
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE_DIR = os.path.normpath(os.path.join(HERE, "..", "oracle"))
LIB = os.path.join(ORACLE_DIR, "libtf_oracle.so")


class OParams(C.Structure):
    _fields_ = [
        ("width", C.c_int), ("height", C.c_int),
        ("ss_x", C.c_int), ("ss_y", C.c_int), ("monochrome", C.c_int),
        ("bit_depth", C.c_int), ("use_hbd", C.c_int),
        ("border", C.c_int),
        ("num_frames", C.c_int), ("filter_frame_idx", C.c_int),
        ("noise_levels", C.c_double * 3),
        ("q_factor", C.c_int), ("filter_strength", C.c_int),
        ("force_integer_mv", C.c_int), ("allow_hp", C.c_int),
        ("subpel_method", C.c_int), ("subpel_iters_per_step", C.c_int),
        ("prune_mesh_level", C.c_int),
        ("mesh", (C.c_int * 2) * 4),
        ("use_downsampled_sad", C.c_int),
        ("compute_frame_diff", C.c_int),
    ]


BASE_STAT_FIELDS = ("mesh_searches", "diamond_ties", "mesh_ties", "subpel_ties", "conv_im_overflow", "pred_clip_lo",
                    "pred_clip_hi", "mv_on_limit", "mv_on_clamp", "ref_mv_resets", "block_mse_at_thresh",
                    "sad_peak_groups")
LIMIT_STAT_FIELDS = ("lim_inverted", "start_clamped", "lim_border_bound")
STAT_FIELDS = BASE_STAT_FIELDS + LIMIT_STAT_FIELDS

# optional keys of the params dict: the coded grid and size the encoder passes (0 or absent: the crop size's),
# handed to tfo_set_coded in this order
CODED_KEYS = ("mi_rows", "mi_cols", "cm_width", "cm_height")


class OStats(C.Structure):  # tfo_stats
    _fields_ = [(k, C.c_int64) for k in BASE_STAT_FIELDS]


class OLimitStats(C.Structure):  # tfo_limit_stats
    _fields_ = [(k, C.c_int64) for k in LIMIT_STAT_FIELDS]


def coded_values(p):
    """The tfo_set_coded arguments of a params dict: mi_rows, mi_cols, cm_width, cm_height (0 where absent)."""
    return tuple(int(p.get(k) or 0) for k in CODED_KEYS)


def bind_common(l):
    """argtypes of the entry points the filter oracle and the motion oracle library share."""
    l.tfo_create.restype = C.c_void_p
    l.tfo_create.argtypes = [C.POINTER(OParams)]
    l.tfo_set_coded.argtypes = [C.c_void_p] + [C.c_int] * 4
    l.tfo_set_coded.restype = None
    l.tfo_destroy.argtypes = [C.c_void_p]
    l.tfo_set_frame.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    l.tfo_reset_stats.argtypes = []
    l.tfo_reset_stats.restype = None
    l.tfo_get_stats.argtypes = [C.POINTER(OStats)]
    l.tfo_get_stats.restype = None
    l.tfo_get_limit_stats.argtypes = [C.POINTER(OLimitStats)]
    l.tfo_get_limit_stats.restype = None


def create(l, p):
    """tfo_create + tfo_set_coded for a params dict; returns (handle, OParams kept alive)."""
    cp = make_params(p)
    h = l.tfo_create(C.byref(cp))
    l.tfo_set_coded(h, *coded_values(p))
    return h, cp


def read_stats(l):
    st, ls = OStats(), OLimitStats()
    l.tfo_get_stats(C.byref(st))
    l.tfo_get_limit_stats(C.byref(ls))
    return {**{k: int(getattr(st, k)) for k in BASE_STAT_FIELDS}, **{k: int(getattr(ls, k)) for k in LIMIT_STAT_FIELDS}}


_lib = None


def build():
    if not os.path.exists(LIB) or os.path.getmtime(LIB) < os.path.getmtime(os.path.join(ORACLE_DIR, "tf_oracle.c")):
        subprocess.check_call(["make", "-C", ORACLE_DIR, "oracle"], stdout=subprocess.DEVNULL)


def lib():
    global _lib
    if _lib is None:
        build()
        l = C.CDLL(LIB)
        bind_common(l)
        l.tfo_estimate_noise.restype = C.c_double
        l.tfo_estimate_noise.argtypes = [C.c_void_p, C.c_int, C.c_int]
        l.tfo_estimate_noise_thresh.restype = C.c_double
        l.tfo_estimate_noise_thresh.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_int]
        l.tfo_run.argtypes = [C.c_void_p, C.c_int, C.c_int] + [C.c_void_p] * 6
        l.tfo_get_output.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int]
        l.tfo_get_plane_with_border.restype = C.c_int
        l.tfo_get_plane_with_border.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p] + [C.POINTER(C.c_int)] * 3
        l.tfo_plane_alloc_size.argtypes = [C.c_void_p, C.c_int]
        l.tfo_extend_output_borders.argtypes = [C.c_void_p]
        l.tfo_full_pixel_search.argtypes = [C.c_void_p] + [C.c_int] * 7 + [C.POINTER(C.c_int)]
        l.tfo_apply_block.argtypes = (
            [C.c_int] * 7 + [C.c_void_p] * 3 + [C.c_int] * 4 + [C.c_void_p] * 3 + [C.c_int] * 2 + [C.c_void_p] * 3)
        l.tfo_sad.restype = C.c_uint
        l.tfo_sad.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int] + [C.c_int] * 5
        l.tfo_variance.restype = C.c_uint
        l.tfo_variance.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int] + [C.c_int] * 4 + [C.POINTER(C.c_uint)]
        l.tfo_subpel_variance.restype = C.c_uint
        l.tfo_subpel_variance.argtypes = ([C.c_void_p, C.c_int, C.c_int, C.c_int, C.c_void_p, C.c_int]
                                          + [C.c_int] * 4 + [C.POINTER(C.c_uint)])
        l.tfo_convolve12.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int] + [C.c_int] * 6
        l.tfo_od_divu.argtypes = [C.c_uint, C.c_uint]
        _lib = l
    return _lib


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def reset_stats():
    """Zero the oracle's event counters (process-wide)."""
    lib().tfo_reset_stats()


def get_stats():
    """The oracle's event counters since the last reset_stats(), as a dict (tfo_stats and tfo_limit_stats in
    tf_oracle.h)."""
    return read_stats(lib())


def make_params(p):
    c = OParams()
    for k in ("width", "height", "ss_x", "ss_y", "monochrome", "bit_depth", "use_hbd", "border",
              "num_frames", "filter_frame_idx", "q_factor", "filter_strength", "force_integer_mv",
              "allow_hp", "subpel_method", "subpel_iters_per_step", "prune_mesh_level",
              "use_downsampled_sad", "compute_frame_diff"):
        setattr(c, k, int(p[k]))
    for i in range(3):
        c.noise_levels[i] = float(p["noise_levels"][i])
    for i in range(4):
        c.mesh[i][0], c.mesh[i][1] = p["mesh"][i]
    return c


class OracleFilter:
    def __init__(self, p, frames):
        self.p = dict(p)
        self.h, self.cp = create(lib(), p)
        self.num_planes = 1 if p["monochrome"] else 3
        self.mb_rows = (p["height"] + 31) // 32
        self.mb_cols = (p["width"] + 31) // 32
        self.num_pels = 1024 + (0 if p["monochrome"] else 2 * (1024 >> (p["ss_x"] + p["ss_y"])))
        dt = np.uint16 if p["use_hbd"] else np.uint8
        for i, (y, u, v) in enumerate(frames):
            ys = np.ascontiguousarray(y.astype(dt))
            us = None if u is None else np.ascontiguousarray(u.astype(dt))
            vs = None if v is None else np.ascontiguousarray(v.astype(dt))
            lib().tfo_set_frame(self.h, i, _ptr(ys), _ptr(us), _ptr(vs))

    def estimate_noise(self, idx=None, edge_thresh=50):
        idx = self.p["filter_frame_idx"] if idx is None else idx
        return [lib().tfo_estimate_noise_thresh(self.h, idx, pl, edge_thresh) for pl in range(self.num_planes)]

    def run(self, record=True, rows=None):
        nb = self.mb_rows * self.mb_cols
        nf = self.p["num_frames"]
        mvs = np.zeros((nb, nf, 4, 2), np.int16) if record else None
        mses = np.zeros((nb, nf, 4), np.int32) if record else None
        pred = np.zeros((nb, nf, self.num_pels), np.uint16) if record else None
        accum = np.zeros((nb, self.num_pels), np.uint32) if record else None
        count = np.zeros((nb, self.num_pels), np.uint16) if record else None
        diff = np.zeros(2, np.int64)
        r0, r1 = (0, self.mb_rows) if rows is None else rows
        lib().tfo_run(self.h, r0, r1, _ptr(mvs), _ptr(mses), _ptr(pred), _ptr(accum), _ptr(count), _ptr(diff))
        out = []
        for pl in range(self.num_planes):
            w = self.mb_cols * 32 >> (self.p["ss_x"] if pl else 0)
            h = self.mb_rows * 32 >> (self.p["ss_y"] if pl else 0)
            o = np.zeros((h, w), np.uint16)
            lib().tfo_get_output(self.h, pl, _ptr(o), w, h)
            out.append(o)
        return dict(mvs=mvs, mses=mses, pred=pred, accum=accum, count=count, out=out, diff=diff)

    def plane_with_border(self, idx, plane):
        n = lib().tfo_plane_alloc_size(self.h, plane)
        rows, bw, bh = C.c_int(), C.c_int(), C.c_int()
        stride = lib().tfo_get_plane_with_border(self.h, idx, plane, None, rows, bw, bh)
        buf = np.zeros((rows.value, stride), np.uint16)
        assert buf.size == n
        lib().tfo_get_plane_with_border(self.h, idx, plane, _ptr(buf), rows, bw, bh)
        return buf, dict(stride=stride, bw=bw.value, bh=bh.value)

    def extend_output_borders(self):
        """aom_extend_frame_borders on the output frame; plane_with_border(-1, plane) reads it back."""
        lib().tfo_extend_output_borders(self.h)

    def full_pixel_search(self, src_idx, ref_idx, bsize, x, y, start_row, start_col):
        """av1_full_pixel_search() on one block as tf_motion_search() configures it -> (row, col, var)."""
        out = (C.c_int * 3)()
        lib().tfo_full_pixel_search(self.h, src_idx, ref_idx, bsize, x, y, start_row, start_col, out)
        return out[0], out[1], out[2]

    def close(self):
        if self.h:
            lib().tfo_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
