"""ctypes binding for oracle/_ref/libtf_ref.so (the UNMODIFIED reference compiled
from the upstream source tree by oracle/Makefile).  TEST INFRASTRUCTURE ONLY."""
import ctypes as C
import os
import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
LIB = os.path.join(HERE, "..", "oracle", "_ref", "libtf_ref.so")
# same harness built around temporal_filter.c + integration/tf_gpu_seam.patch, linked to libtf_gpu.so
SEAM_LIB = os.path.join(HERE, "..", "oracle", "_ref", "libtf_ref_seam.so")


class RefCfg(C.Structure):
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
# same harness with the hot-path rtcd names bound to the reference's AVX2 intrinsics (CPU timing baseline)
AVX2_LIB = os.path.join(HERE, "..", "oracle", "_ref", "libtf_ref_avx2.so")


def avx2_available():
    try:
        flags = open("/proc/cpuinfo").read()
    except OSError:
        return False
    return os.path.exists(AVX2_LIB) and " avx2" in flags


_avx2 = None


def avx2_lib():
    global _avx2
    if _avx2 is None:
        _avx2 = _bind(C.CDLL(AVX2_LIB))
    return _avx2


# the upstream source tree oracle/Makefile compiles oracle/_ref from (make REF=<dir>); unset: not available
SOURCE_DIR = os.environ.get("REF", "")


def available():
    return os.path.exists(LIB)


def reference_or_oracle(p, frames):
    """The compiled reference where oracle/_ref is built, else the oracle (oracle/tf_oracle.c).  Both give
    estimate_noise, run, extend_output_borders, plane_with_border(idx, plane)[0] (the whole padded plane, same
    layout) and full_pixel_search.  tests/golden/ holds reference outputs of the filter pipeline only: the
    oracle's per-block search and border extension are pinned to them only where the pipeline exercises them
    (tests/test_oracle_golden.py), so where oracle/_ref is built these tests compare with the reference."""
    if available():
        return RefFilter(p, frames)
    import _oracle
    return _oracle.OracleFilter(p, frames)


def seam_available():
    return os.path.exists(SEAM_LIB)


_lib = None
_seam = None


def seam_lib():
    """The reference + CONFIG_TF_GPU seam; needs libtf_gpu.so and a GPU at call time."""
    global _seam
    if _seam is None:
        _seam = _bind(C.CDLL(SEAM_LIB))
        _seam.tfref_run_gpu_seam.argtypes = [C.c_void_p, C.c_void_p]
        _seam.tfref_gpu_noise_levels.argtypes = [C.c_void_p, C.c_int, C.POINTER(C.c_double)]
        _seam.tfref_gpu_estimate_noise.restype = C.c_double
        _seam.tfref_gpu_estimate_noise.argtypes = [C.c_void_p] + [C.c_int] * 4
        _seam.tfref_run_gpu_seam_async.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.POINTER(C.c_int)]
        _seam.tfref_gpu_push_window.argtypes = [C.c_void_p]
        _seam.tfref_gpu_last_launches.argtypes = [C.c_void_p]
        _seam.tfref_gpu_num_pinned.argtypes = [C.c_void_p]
        _seam.tfref_gpu_has_context.argtypes = [C.c_void_p]
        _seam.tfref_gpu_release.argtypes = [C.c_void_p]
    return _seam


def _bind(l):
    l.tfref_create.restype = C.c_void_p
    l.tfref_create.argtypes = [C.POINTER(RefCfg)]
    l.tfref_set_frame.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
    l.tfref_run.argtypes = [C.c_void_p, C.c_int, C.c_int] + [C.c_void_p] * 6
    l.tfref_get_output.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int]
    l.tfref_destroy.argtypes = [C.c_void_p]
    l.tfref_estimate_noise.restype = C.c_double
    l.tfref_estimate_noise.argtypes = [C.c_void_p, C.c_int, C.c_int]
    l.tfref_frame_info.argtypes = [C.c_void_p] + [C.POINTER(C.c_int)] * 5
    l.tfref_get_plane_with_border.restype = C.c_int
    l.tfref_get_plane_with_border.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.POINTER(C.c_int)]
    l.tfref_extend_output_borders.argtypes = [C.c_void_p]
    l.tfref_full_pixel_search.argtypes = [C.c_void_p] + [C.c_int] * 7 + [C.POINTER(C.c_int)]
    return l


def lib():
    global _lib
    if _lib is None:
        _lib = C.CDLL(LIB)
        _lib.tfref_create.restype = C.c_void_p
        _lib.tfref_create.argtypes = [C.POINTER(RefCfg)]
        _lib.tfref_set_frame.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_void_p, C.c_void_p]
        _lib.tfref_run.argtypes = [C.c_void_p, C.c_int, C.c_int] + [C.c_void_p] * 6
        _lib.tfref_get_output.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int, C.c_int]
        _lib.tfref_estimate_noise.restype = C.c_double
        _lib.tfref_estimate_noise.argtypes = [C.c_void_p, C.c_int, C.c_int]
        _lib.tfref_destroy.argtypes = [C.c_void_p]
        _lib.tfref_frame_info.argtypes = [C.c_void_p] + [C.POINTER(C.c_int)] * 5
        _lib.tfref_get_plane_with_border.restype = C.c_int
        _lib.tfref_get_plane_with_border.argtypes = [C.c_void_p, C.c_int, C.c_int, C.c_void_p, C.POINTER(C.c_int)]
        _lib.tfref_extend_output_borders.argtypes = [C.c_void_p]
        _lib.tfref_apply_block.argtypes = (
            [C.c_int] * 7 + [C.c_void_p] * 3 + [C.c_int] * 4 + [C.c_void_p] * 3 + [C.c_int] * 2 + [C.c_void_p] * 3)
    return _lib


def _ptr(a):
    return None if a is None else a.ctypes.data_as(C.c_void_p)


def make_cfg(p):
    """p: dict with the tf params (see tests/_params.py)."""
    c = RefCfg()
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


class RefFilter:
    def __init__(self, p, frames, seam=False, avx2=False):
        self.p = dict(p)
        self.cfg = make_cfg(p)
        self.L = seam_lib() if seam else avx2_lib() if avx2 else lib()
        self.h = self.L.tfref_create(C.byref(self.cfg))
        assert self.h
        coded = tuple(int(p.get(k) or 0) for k in ("mi_rows", "mi_cols", "cm_width", "cm_height"))
        if any(coded):  # the coded grid and size, where they differ from the crop size's
            self.L.tfref_set_coded.argtypes = [C.c_void_p] + [C.c_int] * 4
            self.L.tfref_set_coded(self.h, *coded)
        self.num_planes = 1 if p["monochrome"] else 3
        self.mb_rows = (p["height"] + 31) // 32
        self.mb_cols = (p["width"] + 31) // 32
        self.num_pels = 1024 + (0 if p["monochrome"] else 2 * (1024 >> (p["ss_x"] + p["ss_y"])))
        self._keep = []
        for i, (y, u, v) in enumerate(frames):
            dt = np.uint16 if p["use_hbd"] else np.uint8
            ys = np.ascontiguousarray(y.astype(dt))
            us = None if u is None else np.ascontiguousarray(u.astype(dt))
            vs = None if v is None else np.ascontiguousarray(v.astype(dt))
            self._keep.append((ys, us, vs))
            self.L.tfref_set_frame(self.h, i, _ptr(ys), _ptr(us), _ptr(vs))

    def estimate_noise(self, idx=None):
        idx = self.p["filter_frame_idx"] if idx is None else idx
        return [self.L.tfref_estimate_noise(self.h, idx, pl) for pl in range(self.num_planes)]

    def run(self, record=True, rows=None):
        nb = self.mb_rows * self.mb_cols
        nf = self.p["num_frames"]
        mvs = np.zeros((nb, nf, 4, 2), np.int16) if record else None
        mses = np.zeros((nb, nf, 4), np.int32) if record else None
        pred = np.zeros((nb, nf, self.num_pels), np.uint16) if record else None
        diff = np.zeros(2, np.int64)
        r0, r1 = (0, self.mb_rows) if rows is None else rows
        self.L.tfref_run(self.h, r0, r1, _ptr(mvs), _ptr(mses), _ptr(pred), None, None, _ptr(diff))
        return dict(mvs=mvs, mses=mses, pred=pred, out=self._outputs(), diff=diff)

    def _outputs(self):
        out = []
        for pl in range(self.num_planes):
            w = self.mb_cols * 32 >> (self.p["ss_x"] if pl else 0)
            h = self.mb_rows * 32 >> (self.p["ss_y"] if pl else 0)
            o = np.zeros((h, w), np.uint16)
            self.L.tfref_get_output(self.h, pl, _ptr(o), w, h)
            out.append(o)
        return out

    def gpu_noise_levels(self, idx=None):
        """The CONFIG_TF_GPU replacement of the noise loop in tf_setup_filtering_buffer()."""
        idx = self.p["filter_frame_idx"] if idx is None else idx
        out = (C.c_double * 3)(0.0, 0.0, 0.0)
        self.L.tfref_gpu_noise_levels(self.h, idx, out)
        return [out[i] for i in range(self.num_planes)]

    def run_gpu_seam(self):
        """av1_temporal_filter()'s CONFIG_TF_GPU branch: the reference-side shim calls libtf_gpu.so."""
        diff = np.zeros(2, np.int64)
        self.L.tfref_run_gpu_seam(self.h, _ptr(diff))
        return dict(out=self._outputs(), diff=diff)

    def run_gpu_seam_async(self, copies=2):
        """av1_tf_info_filtering()'s CONFIG_TF_GPU branch: `copies` windows submitted back to back and waited
        for together; the output frame comes back with its borders extended on the device."""
        diff = np.zeros(2, np.int64)
        eq = C.c_int(0)
        self.L.tfref_run_gpu_seam_async(self.h, copies, _ptr(diff), C.byref(eq))
        return dict(out=self._outputs(), diff=diff, all_equal=bool(eq.value))

    def gpu_push_window(self):
        """Real lookahead + the av1_receive_raw_frame() hunk: every pushed frame is uploaded at push time."""
        rc = self.L.tfref_gpu_push_window(self.h)
        assert rc == 0, rc

    def gpu_estimate_noise(self, idx, in_lookahead, plane, edge_thresh=50):
        return self.L.tfref_gpu_estimate_noise(self.h, idx, int(in_lookahead), plane, edge_thresh)

    def extend_output_borders(self):
        self.L.tfref_extend_output_borders(self.h)

    def full_pixel_search(self, src_idx, ref_idx, bsize, x, y, start_row, start_col):
        """av1_full_pixel_search() on one block as tf_motion_search() configures it -> (row, col, var)."""
        out = (C.c_int * 3)()
        self.L.tfref_full_pixel_search(self.h, src_idx, ref_idx, bsize, x, y, start_row, start_col, out)
        return out[0], out[1], out[2]

    def plane_with_border(self, idx, plane):
        ys, uvs, b, aw, ah = (C.c_int() for _ in range(5))
        self.L.tfref_frame_info(self.h, ys, uvs, b, aw, ah)
        stride = uvs.value if plane else ys.value
        bh = b.value >> (self.p["ss_y"] if plane else 0)
        ph = (ah.value >> (self.p["ss_y"] if plane else 0)) + 2 * bh
        buf = np.zeros((ph, stride), np.uint16)
        rows = C.c_int()
        s = self.L.tfref_get_plane_with_border(self.h, idx, plane, _ptr(buf), C.byref(rows))
        assert s == stride and rows.value == ph
        return buf, dict(y_stride=ys.value, uv_stride=uvs.value, border=b.value,
                         aligned_w=aw.value, aligned_h=ah.value)

    def close(self):
        if self.h:
            self.L.tfref_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
