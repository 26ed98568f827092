"""aom-av1-psy_b200: host-side mirror of the reference's temporal-filter interface
on top of the C ABI of libtf_gpu.so (include/tf_gpu.h).

The reference is C; the product's host side is the C++ inside libtf_gpu.so.
This module is only the thin ctypes binding used by tests, bench.py and
__graft_entry__: it names things the way av1/encoder/temporal_filter.{c,h} does
(YV12 buffers, TemporalFilterCtx fields, av1_temporal_filter,
av1_estimate_noise_from_single_plane, FRAME_DIFF) so parity tests read like the
reference's own.  There is no CPU fallback: importing works anywhere, but every
call raises TfGpuError unless libtf_gpu.so is built and a CUDA device exists.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libtf_gpu.so")
# development only: point at another build of the same library (A/B runs of two kernels on one box)
LIB_PATH = os.environ.get("TF_GPU_LIB", LIB_PATH)

TF_GPU_MAX_FRAMES = 24
TF_GPU_MAX_BATCH = 16
NOISE_ESTIMATION_EDGE_THRESHOLD = 50  # temporal_filter.h:79
TF_BLOCK = 32  # TF_BLOCK_SIZE = BLOCK_32X32, temporal_filter.h:31

ERRORS = {0: "OK", -1: "INVALID", -2: "MEM", -3: "CUDA", -4: "NO_DEVICE", -5: "UNSUPPORTED"}

EXPORTS = [
    "tf_gpu_abi_version", "tf_gpu_create", "tf_gpu_destroy", "tf_gpu_last_error", "tf_gpu_estimate_noise",
    "tf_gpu_filter", "tf_gpu_filter_dump", "tf_gpu_submit", "tf_gpu_wait", "tf_gpu_cache_frame",
    "tf_gpu_evict_frame", "tf_gpu_filter_resident", "tf_gpu_download_output", "tf_gpu_output_device_plane",
    "tf_gpu_host_register", "tf_gpu_host_unregister", "tf_gpu_last_stats", "tf_gpu_event_record",
    "tf_gpu_event_elapsed_ms", "tf_gpu_synchronize", "tf_gpu_microbench", "tf_gpu_last_kernel_times", "tf_gpu_filter_resident_async", "tf_gpu_filter_resident_result", "tf_gpu_collect_counters", "tf_gpu_read_counters",
    "tf_gpu_cache_frame_async", "tf_gpu_debug_read_plane", "tf_gpu_device_border", "tf_gpu_fullpel_search_batch",
    "tf_gpu_output_ipc_export", "tf_gpu_output_ipc_import", "tf_gpu_cache_frame_device",
    "tf_gpu_filter_batch_async", "tf_gpu_filter_batch_result", "tf_gpu_download_batch_output",
    "tf_gpu_batch_output_device_plane", "tf_gpu_motion_search_batch", "tf_gpu_motion_search_device",
]


class TfGpuError(RuntimeError):
    def __init__(self, code, msg=""):
        super().__init__(f"tf_gpu error {code} ({ERRORS.get(code, '?')}): {msg}")
        self.code = code


class DeviceCfg(C.Structure):
    _fields_ = [("device", C.c_int), ("max_cached_frames", C.c_int), ("reserved", C.c_int * 6)]


class Frame(C.Structure):
    """tf_gpu_frame: POD mirror of YV12_BUFFER_CONFIG (aom_scale/yv12config.h:43-123)."""
    _fields_ = [
        ("plane", C.c_void_p * 3), ("stride", C.c_int * 2), ("crop_w", C.c_int * 2), ("crop_h", C.c_int * 2),
        ("aligned_w", C.c_int * 2), ("aligned_h", C.c_int * 2), ("border", C.c_int), ("ss_x", C.c_int),
        ("ss_y", C.c_int), ("is_hbd", C.c_int), ("frame_id", C.c_uint64),
    ]


class Params(C.Structure):
    """tf_gpu_params: TemporalFilterCtx (temporal_filter.h:93-144) + the speed features the search reads."""
    _fields_ = [
        ("num_frames", C.c_int), ("filter_frame_idx", C.c_int), ("num_planes", C.c_int), ("bit_depth", C.c_int),
        ("noise_levels", C.c_double * 3), ("q_factor", C.c_int), ("filter_strength", C.c_int),
        ("mi_rows", C.c_int), ("mi_cols", C.c_int), ("border_in_pixels", C.c_int), ("force_integer_mv", C.c_int),
        ("allow_hp", C.c_int), ("subpel_method", C.c_int), ("subpel_iters_per_step", C.c_int),
        ("prune_mesh_level", C.c_int), ("mesh_patterns", (C.c_int * 2) * 4), ("use_downsampled_sad", C.c_int),
        ("compute_frame_diff", C.c_int), ("out_row_begin", C.c_int), ("out_row_end", C.c_int),
        ("extend_output_borders", C.c_int), ("cm_width", C.c_int), ("cm_height", C.c_int),
        ("reserved", C.c_int * 5),
    ]


class SearchItem(C.Structure):
    _fields_ = [("x", C.c_int), ("y", C.c_int), ("start_row", C.c_int16), ("start_col", C.c_int16)]


class SearchResult(C.Structure):
    _fields_ = [("row", C.c_int16), ("col", C.c_int16), ("var", C.c_int32)]


class MotionItem(C.Structure):
    """tf_gpu_motion_item: one block of the source searched against references[ref]."""
    _fields_ = [("x", C.c_int), ("y", C.c_int), ("start_row", C.c_int16), ("start_col", C.c_int16),
                ("ref", C.c_int32)]


class MotionResult(C.Structure):
    """tf_gpu_motion_result: the full-pel result and the final 1/8-pel MV with its error."""
    _fields_ = [("fullpel_row", C.c_int16), ("fullpel_col", C.c_int16), ("fullpel_var", C.c_int32),
                ("row", C.c_int16), ("col", C.c_int16), ("err", C.c_uint32)]


# numpy views of the two structs above, so that large batches are packed and unpacked without a Python loop
_MOTION_ITEM_DTYPE = np.dtype([("x", "<i4"), ("y", "<i4"), ("start_row", "<i2"), ("start_col", "<i2"),
                               ("ref", "<i4")])
_MOTION_RESULT_DTYPE = np.dtype([("fullpel_row", "<i2"), ("fullpel_col", "<i2"), ("fullpel_var", "<i4"),
                                 ("row", "<i2"), ("col", "<i2"), ("err", "<u4")])
assert _MOTION_ITEM_DTYPE.itemsize == C.sizeof(MotionItem) == 16
assert _MOTION_RESULT_DTYPE.itemsize == C.sizeof(MotionResult) == 16
TF_GPU_MOTION_REJECTED = -1  # fullpel_var of an item tf_gpu_motion_search_device rejected (tf_gpu.h)


class Dump(C.Structure):
    _fields_ = [("subblock_mvs", C.c_void_p), ("subblock_mses", C.c_void_p), ("pred", C.c_void_p),
                ("accum", C.c_void_p), ("count", C.c_void_p)]


_lib = None


def load_library():
    """dlopen libtf_gpu.so; fails loudly when the CUDA extension is missing."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise TfGpuError(-4, f"{LIB_PATH} is not built (run __graft_entry__.build()); there is no CPU fallback")
    lib = C.CDLL(LIB_PATH)
    vp, i, u64 = C.c_void_p, C.c_int, C.c_uint64
    lib.tf_gpu_abi_version.restype = i
    lib.tf_gpu_create.argtypes = [C.POINTER(vp), C.POINTER(DeviceCfg)]
    lib.tf_gpu_destroy.argtypes = [vp]
    lib.tf_gpu_destroy.restype = None
    lib.tf_gpu_last_error.argtypes = [vp]
    lib.tf_gpu_last_error.restype = C.c_char_p
    lib.tf_gpu_estimate_noise.argtypes = [vp, C.POINTER(Frame), i, i, i, C.POINTER(C.c_double)]
    lib.tf_gpu_filter.argtypes = [vp, C.POINTER(Params), C.POINTER(Frame), C.POINTER(Frame), C.POINTER(C.c_int64)]
    lib.tf_gpu_filter_dump.argtypes = lib.tf_gpu_filter.argtypes + [C.POINTER(Dump)]
    lib.tf_gpu_submit.argtypes = lib.tf_gpu_filter.argtypes + [C.POINTER(u64)]
    lib.tf_gpu_wait.argtypes = [vp, u64]
    lib.tf_gpu_cache_frame.argtypes = [vp, C.POINTER(Frame)]
    lib.tf_gpu_evict_frame.argtypes = [vp, u64]
    lib.tf_gpu_cache_frame_async.argtypes = [vp, C.POINTER(Frame)]
    lib.tf_gpu_cache_frame_device.argtypes = [vp, C.POINTER(Frame), vp]
    lib.tf_gpu_debug_read_plane.argtypes = [vp, u64, i, vp, i, i, i, i, i]
    lib.tf_gpu_device_border.restype = i
    lib.tf_gpu_output_ipc_export.argtypes = [vp, i, C.c_char_p, C.POINTER(C.c_size_t), C.POINTER(C.c_size_t)]
    lib.tf_gpu_output_ipc_import.argtypes = [vp, i, C.c_char_p, C.c_size_t, C.c_size_t]
    lib.tf_gpu_fullpel_search_batch.argtypes = [vp, C.POINTER(Params), C.POINTER(Frame), C.POINTER(Frame), i,
                                                C.POINTER(SearchItem), i, C.POINTER(SearchResult)]
    lib.tf_gpu_motion_search_batch.argtypes = [vp, C.POINTER(Params), u64, C.POINTER(u64), i, i,
                                               C.POINTER(MotionItem), i, C.POINTER(MotionResult)]
    lib.tf_gpu_motion_search_device.argtypes = [vp, C.POINTER(Params), u64, C.POINTER(u64), i, i, vp, i, vp, vp]
    lib.tf_gpu_filter_resident.argtypes = [vp, C.POINTER(Params), C.POINTER(u64), C.POINTER(C.c_int64),
                                           C.POINTER(C.c_float)]
    lib.tf_gpu_download_output.argtypes = [vp, C.POINTER(Frame), i, i]
    lib.tf_gpu_filter_resident_async.argtypes = [vp, C.POINTER(Params), C.POINTER(u64)]
    lib.tf_gpu_filter_resident_result.argtypes = [vp, C.POINTER(C.c_int64), C.POINTER(C.c_float)]
    lib.tf_gpu_output_device_plane.argtypes = [vp, i, C.POINTER(vp), C.POINTER(C.c_size_t), C.POINTER(i),
                                               C.POINTER(i)]
    lib.tf_gpu_host_register.argtypes = [vp, vp, C.c_size_t]
    lib.tf_gpu_host_unregister.argtypes = [vp, vp]
    lib.tf_gpu_last_stats.argtypes = [vp, C.POINTER(i), C.POINTER(C.c_float)]
    lib.tf_gpu_event_record.argtypes = [vp, i]
    lib.tf_gpu_event_elapsed_ms.argtypes = [vp, i, i, C.POINTER(C.c_float)]
    lib.tf_gpu_synchronize.argtypes = [vp]
    lib.tf_gpu_microbench.argtypes = [vp, i, C.POINTER(C.c_double)]
    lib.tf_gpu_last_kernel_times.argtypes = [vp, C.POINTER(C.c_float)]
    lib.tf_gpu_collect_counters.argtypes = [vp, i]
    lib.tf_gpu_filter_batch_async.argtypes = [vp, i, C.POINTER(Params), C.POINTER(C.POINTER(u64))]
    lib.tf_gpu_filter_batch_result.argtypes = [vp, C.POINTER(C.c_int64 * 2), C.POINTER(C.c_float)]
    lib.tf_gpu_download_batch_output.argtypes = [vp, i, C.POINTER(Frame)]
    lib.tf_gpu_batch_output_device_plane.argtypes = [vp, i, i, C.POINTER(vp), C.POINTER(C.c_size_t), C.POINTER(i),
                                                     C.POINTER(i)]
    lib.tf_gpu_read_counters.argtypes = [vp, C.POINTER(u64)]
    _lib = lib
    return lib


def _align(v, n):
    return (v + n - 1) // n * n


class Yv12Buffer:
    """Host frame with the reference's YV12_BUFFER_CONFIG layout
    (aom_realloc_frame_buffer, aom_scale/generic/yv12config.c:223-258): 8-aligned
    sizes, stride = align32(aligned_w + 2*border), planes at border*stride+border."""

    def __init__(self, width, height, ss_x=1, ss_y=1, use_hbd=False, border=160, monochrome=False, frame_id=0):
        self.width, self.height, self.ss_x, self.ss_y = width, height, ss_x, ss_y
        self.use_hbd, self.border, self.monochrome, self.frame_id = bool(use_hbd), border, bool(monochrome), frame_id
        self.dtype = np.uint16 if use_hbd else np.uint8
        aw, ah = _align(width, 8), _align(height, 8)
        self.aligned = [(aw, ah), (aw >> ss_x, ah >> ss_y)]
        self.crop = [(width, height), ((width + ss_x) >> ss_x, (height + ss_y) >> ss_y)]
        self.stride = [_align(aw + 2 * border, 32), _align(aw + 2 * border, 32) >> ss_x]
        self.borders = [(border, border), (border >> ss_x, border >> ss_y)]
        self.num_planes = 1 if monochrome else 3
        self.alloc = []
        for p in range(self.num_planes):
            k = 1 if p else 0
            rows = self.aligned[k][1] + 2 * self.borders[k][1]
            self.alloc.append(np.zeros((rows, self.stride[k]), self.dtype))

    def plane(self, p):
        """View whose [0,0] is pixel (0,0) (y_buffer / u_buffer / v_buffer)."""
        k = 1 if p else 0
        bx, by = self.borders[k]
        return self.alloc[p][by:, bx:]

    def set_planes(self, y, u=None, v=None, extend=True):
        """Copy crop-sized planes in; with extend, replicate edges with the extents of
        av1_copy_and_extend_frame (extend.c:113-131): top/left = border, right/bottom =
        max(aligned + border, align64(aligned)) - crop (chroma: luma extents >> ss)."""
        aw, ah = self.aligned[0]
        er_y = max(aw + self.border, _align(aw, 64)) - self.width
        eb_y = max(ah + self.border, _align(ah, 64)) - self.height
        for p, src in enumerate((y, u, v)[: self.num_planes]):
            k = 1 if p else 0
            cw, ch = self.crop[k]
            bx, by = self.borders[k]
            er = er_y >> self.ss_x if p else er_y
            eb = eb_y >> self.ss_y if p else eb_y
            a = self.alloc[p]
            a[by:by + ch, bx:bx + cw] = src
            if extend:
                x1 = min(bx + cw + er, a.shape[1])
                y1 = min(by + ch + eb, a.shape[0])
                a[by:by + ch, :bx] = a[by:by + ch, bx:bx + 1]
                a[by:by + ch, bx + cw:x1] = a[by:by + ch, bx + cw - 1:bx + cw]
                a[:by, :x1] = a[by:by + 1, :x1]
                a[by + ch:y1, :x1] = a[by + ch - 1:by + ch, :x1]
        return self

    def c_frame(self):
        f = Frame()
        for p in range(self.num_planes):
            k = 1 if p else 0
            bx, by = self.borders[k]
            f.plane[p] = self.alloc[p].ctypes.data + (by * self.stride[k] + bx) * self.alloc[p].itemsize
        for k in range(2):
            f.stride[k] = self.stride[k]
            f.crop_w[k], f.crop_h[k] = self.crop[k]
            f.aligned_w[k], f.aligned_h[k] = self.aligned[k]
        f.border, f.ss_x, f.ss_y = self.border, self.ss_x, self.ss_y
        f.is_hbd, f.frame_id = int(self.use_hbd), self.frame_id
        return f

    def full_blocks(self, p):
        """Plane region covered by whole 32x32 blocks (what temporal_filter.c:740-777 writes)."""
        k = 1 if p else 0
        w = _align(self.width, 32) >> (self.ss_x if p else 0)
        h = _align(self.height, 32) >> (self.ss_y if p else 0)
        return self.plane(p)[:h, :w]


def tensor_frame(frame_id, y, u=None, v=None):
    """tf_gpu_frame over 2-D CUDA tensors (the descriptor tf_gpu_cache_frame_device reads): uint8 for 8-bit,
    int16 / uint16 for high bit depth, unit column stride, any row stride.  The geometry is derived as Yv12Buffer
    derives it: crop = tensor shape, aligned = align8(luma) >> ss, ss_x / ss_y from the chroma shapes (no chroma:
    monochrome).  Returns (Frame, torch.device).  Malformed input raises ValueError."""
    import torch
    if (u is None) != (v is None):
        raise ValueError("give both chroma planes or neither")
    planes = [y] if u is None else [y, u, v]
    for t in planes:
        if not isinstance(t, torch.Tensor) or t.dim() != 2 or t.numel() == 0:
            raise ValueError("planes must be non-empty 2-D torch tensors")
    hbd_types = (torch.int16, getattr(torch, "uint16", torch.int16))
    if y.dtype == torch.uint8:
        hbd = False
    elif y.dtype in hbd_types:
        hbd = True
    else:
        raise ValueError(f"luma dtype {y.dtype}: uint8 for 8-bit, int16 or uint16 for high bit depth")
    if any(t.dtype != y.dtype for t in planes):
        raise ValueError(f"planes of one frame must share a dtype, got {[str(t.dtype) for t in planes]}")
    H, W = y.shape
    ss_x = ss_y = 1
    if u is not None:
        if u.shape != v.shape:
            raise ValueError(f"chroma planes differ in shape: {tuple(u.shape)} vs {tuple(v.shape)}")
        ch, cw = u.shape
        ss_x = next((s for s in (1, 0) if (W + s) >> s == cw), None)
        ss_y = next((s for s in (1, 0) if (H + s) >> s == ch), None)
        if ss_x is None or ss_y is None:
            raise ValueError(f"chroma shape {tuple(u.shape)} matches no subsampling of a {H}x{W} luma plane")
    def row_stride(t):
        return t.stride(0) if t.shape[0] > 1 else t.shape[1]

    for t in planes:
        if t.shape[1] > 1 and t.stride(1) != 1:
            raise ValueError("planes need a unit column stride (rows may have any stride)")
    if u is not None and row_stride(u) != row_stride(v):
        # tf_gpu_frame has one uv stride: the kernel would read one chroma plane with the other's row stride
        raise ValueError(f"the chroma planes differ in row stride ({row_stride(u)} vs {row_stride(v)} samples); "
                         "tf_gpu_frame has one uv stride: give them the same layout (e.g. .contiguous() both)")
    for t in planes:
        if not t.is_cuda:
            raise ValueError("planes must be CUDA tensors (host frames go through Yv12Buffer / cache_frame)")
        if t.device != y.device:
            raise ValueError("planes of one frame must be on one device")
    aw, ah = _align(W, 8), _align(H, 8)
    f = Frame()
    for p, t in enumerate(planes):
        f.plane[p] = t.data_ptr()
    for k, (t, sx, sy) in enumerate(((y, 0, 0), (planes[-1], ss_x, ss_y))):
        f.stride[k] = row_stride(t)
        f.crop_w[k], f.crop_h[k] = (W + sx) >> sx, (H + sy) >> sy
        f.aligned_w[k], f.aligned_h[k] = aw >> sx, ah >> sy
    f.border, f.ss_x, f.ss_y, f.is_hbd, f.frame_id = 0, ss_x, ss_y, int(hbd), frame_id
    return f, y.device


def _coded_value(p, key, lo):
    """Optional integer key of make_params' dict, >= lo; absent or None: None."""
    v = p.get(key)
    if v is None:
        return None
    if isinstance(v, bool) or not isinstance(v, (int, np.integer)):
        raise ValueError(f"{key} must be an integer, got {v!r}")
    if not lo <= int(v) <= np.iinfo(np.int32).max:
        raise ValueError(f"{key} must be in [{lo}, 2**31), got {v}")
    return int(v)


def make_params(p):
    """dict (tests/_params.tf_params) -> tf_gpu_params.  Optional keys carry the encoder's coded geometry where it
    differs from the frames' crop size (superres, resize): mi_rows / mi_cols (cm->mi_params; default the frame's own
    grid, align8(size) / 4) and cm_width / cm_height (cm->width / height; default 0, the crop size).  Raises
    ValueError for a value of these keys that is not an integer, a grid below 1 or a coded size below 0; the library
    checks the grid against the frames."""
    c = Params()
    c.num_frames, c.filter_frame_idx = p["num_frames"], p["filter_frame_idx"]
    c.num_planes = 1 if p["monochrome"] else 3
    c.bit_depth = p["bit_depth"]
    for i in range(3):
        c.noise_levels[i] = float(p["noise_levels"][i])
    c.q_factor, c.filter_strength = p["q_factor"], p["filter_strength"]
    mi_rows, mi_cols = _coded_value(p, "mi_rows", 1), _coded_value(p, "mi_cols", 1)
    cm_w, cm_h = _coded_value(p, "cm_width", 0), _coded_value(p, "cm_height", 0)
    c.mi_rows = _align(p["height"], 8) // 4 if mi_rows is None else mi_rows
    c.mi_cols = _align(p["width"], 8) // 4 if mi_cols is None else mi_cols
    c.border_in_pixels = p["border"]
    c.force_integer_mv, c.allow_hp = p["force_integer_mv"], p["allow_hp"]
    c.subpel_method, c.subpel_iters_per_step = p["subpel_method"], p["subpel_iters_per_step"]
    c.prune_mesh_level = p["prune_mesh_level"]
    for i in range(4):
        c.mesh_patterns[i][0], c.mesh_patterns[i][1] = p["mesh"][i]
    c.use_downsampled_sad, c.compute_frame_diff = p["use_downsampled_sad"], p["compute_frame_diff"]
    c.out_row_begin, c.out_row_end = p.get("out_row_begin", 0), p.get("out_row_end", 0)
    c.extend_output_borders = p.get("extend_output_borders", 0)
    c.cm_width, c.cm_height = cm_w or 0, cm_h or 0
    return c


def batch_args(params_list, frame_ids_list):
    """Arguments of tf_gpu_filter_batch_async for a list of windows: (n, tf_gpu_params[n], uint64_t *[n], keep-alive).
    params_list holds dicts (tests/_params.tf_params) or Params; frame_ids_list one id list per window.  Raises
    ValueError, before anything reaches the library, for lists of different lengths, an empty batch or one of more
    than TF_GPU_MAX_BATCH windows, and a window whose id count differs from its num_frames."""
    params_list, frame_ids_list = list(params_list), list(frame_ids_list)
    if len(params_list) != len(frame_ids_list):
        raise ValueError(f"{len(params_list)} params for {len(frame_ids_list)} id lists")
    n = len(params_list)
    if not 1 <= n <= TF_GPU_MAX_BATCH:
        raise ValueError(f"a batch holds 1 to {TF_GPU_MAX_BATCH} windows, got {n}")
    cps = [make_params(p) if isinstance(p, dict) else p for p in params_list]
    ids = []
    for w, (cp, fl) in enumerate(zip(cps, frame_ids_list)):
        fl = [int(i) for i in fl]
        if len(fl) != cp.num_frames:
            raise ValueError(f"window {w}: {len(fl)} frame ids for num_frames {cp.num_frames}")
        ids.append((C.c_uint64 * len(fl))(*fl))
    params = (Params * n)(*cps)
    ptrs = (C.POINTER(C.c_uint64) * n)(*[C.cast(a, C.POINTER(C.c_uint64)) for a in ids])
    return n, params, ptrs, ids


def motion_search_args(ref_ids, block_size, items):
    """Arguments of tf_gpu_motion_search_batch: (uint64_t ref_ids[num_refs], num_refs, items, n), items packed as
    tf_gpu_motion_item[n] in a numpy array.  items: integer array-like of shape (n, 5) = x, y, start_row, start_col,
    ref (an empty sequence is n = 0).  Raises ValueError, before anything reaches the library, for items of another
    shape or a non-integer dtype, x / y outside int32, starts outside int16, a ref outside [0, num_refs), 0 or more
    than TF_GPU_MAX_FRAMES - 1 references, and a block size other than 16 or 32.  The block positions are checked by
    the library, which knows the frame size."""
    if block_size not in (16, 32):
        raise ValueError(f"block_size must be 16 or 32, got {block_size}")
    ids = [int(r) for r in ref_ids]
    if not 1 <= len(ids) <= TF_GPU_MAX_FRAMES - 1:
        raise ValueError(f"1 to {TF_GPU_MAX_FRAMES - 1} reference frames, got {len(ids)}")
    a = np.asarray(items)
    if a.ndim == 1 and a.size == 0:
        a = a.reshape(0, 5).astype(np.int64)
    if a.ndim != 2 or a.shape[1] != 5:
        raise ValueError(f"items must have shape (n, 5) (x, y, start_row, start_col, ref), got {a.shape}")
    if not np.issubdtype(a.dtype, np.integer):
        raise ValueError(f"items must be integers, got dtype {a.dtype}")
    a = a.astype(np.int64)
    i16, i32 = np.iinfo(np.int16), np.iinfo(np.int32)
    if ((a[:, 0:2] < i32.min) | (a[:, 0:2] > i32.max)).any():
        raise ValueError("item positions must fit in int32")
    if ((a[:, 2:4] < i16.min) | (a[:, 2:4] > i16.max)).any():
        raise ValueError("start MVs must fit in int16")
    if ((a[:, 4] < 0) | (a[:, 4] >= len(ids))).any():
        raise ValueError(f"item ref out of [0, {len(ids)})")
    packed = np.zeros(len(a), _MOTION_ITEM_DTYPE)
    for k, name in enumerate(_MOTION_ITEM_DTYPE.names):
        packed[name] = a[:, k]
    return (C.c_uint64 * len(ids))(*ids), len(ids), packed, len(a)


def motion_search_device_args(ref_ids, block_size, items, device):
    """Arguments of tf_gpu_motion_search_device that can be checked without reading the items (which would
    synchronise): (uint64_t ref_ids[num_refs], num_refs, n).  items: an integer CUDA tensor of shape (n, 5) = x, y,
    start_row, start_col, ref on `device`, the context's torch.device.  Raises ValueError, before anything reaches
    the library, for items that are not such a tensor, 0 or more than TF_GPU_MAX_FRAMES - 1 references, and a block
    size other than 16 or 32.  Positions and refs are checked per item by the kernel (tf_gpu.h)."""
    import torch
    if block_size not in (16, 32):
        raise ValueError(f"block_size must be 16 or 32, got {block_size}")
    ids = [int(r) for r in ref_ids]
    if not 1 <= len(ids) <= TF_GPU_MAX_FRAMES - 1:
        raise ValueError(f"1 to {TF_GPU_MAX_FRAMES - 1} reference frames, got {len(ids)}")
    if not isinstance(items, torch.Tensor):
        raise ValueError(f"items must be a torch tensor, got {type(items).__name__}")
    if items.dim() != 2 or items.shape[1] != 5:
        raise ValueError(f"items must have shape (n, 5) (x, y, start_row, start_col, ref), got {tuple(items.shape)}")
    if items.dtype.is_floating_point or items.dtype.is_complex or items.dtype == torch.bool:
        raise ValueError(f"items must be integers, got dtype {items.dtype}")
    if not items.is_cuda:
        raise ValueError(f"items must be a CUDA tensor, got one on {items.device}")
    if items.device != torch.device(device):
        raise ValueError(f"items are on {items.device}, the context on {torch.device(device)}")
    return (C.c_uint64 * len(ids))(*ids), len(ids), items.shape[0]


def pack_motion_items(items):
    """(n, 5) integer tensor (x, y, start_row, start_col, ref) -> (n, 4) int32 tensor whose rows are
    tf_gpu_motion_item, by torch ops on the tensor's device (and current stream).  Values are converted as the C
    struct holds them: x, y and ref to int32, the starts to int16 (each modulo its type's range)."""
    import torch
    out = torch.empty((items.shape[0], 4), dtype=torch.int32, device=items.device)
    out[:, 0] = items[:, 0]
    out[:, 1] = items[:, 1]
    out[:, 3] = items[:, 4]
    half = out.view(torch.int16)  # (n, 8): start_row, start_col are halves 4 and 5 (bytes 8..11)
    half[:, 4] = items[:, 2]
    half[:, 5] = items[:, 3]
    return out


def unpack_motion_results(res):
    """(n, 4) int32 tensor of tf_gpu_motion_result rows -> int64 tensor (n, 6) = fullpel_row, fullpel_col,
    fullpel_var, row, col, err (err unsigned), by torch ops on the tensor's device (and current stream)."""
    import torch
    half = res.view(torch.int16)
    cols = (half[:, 0], half[:, 1], res[:, 1], half[:, 4], half[:, 5], res[:, 3].to(torch.int64) & 0xFFFFFFFF)
    return torch.stack([c.to(torch.int64) for c in cols], dim=1)


class TemporalFilterGpu:
    """One tf_gpu_ctx (CUDA device + stream + frame cache)."""

    def __init__(self, device=-1, max_cached_frames=0):
        self.lib = load_library()
        self.device = device
        self.h = C.c_void_p()
        cfg = DeviceCfg(device=device, max_cached_frames=max_cached_frames)
        rc = self.lib.tf_gpu_create(C.byref(self.h), C.byref(cfg))
        if rc:
            self.h = None
            raise TfGpuError(rc, "tf_gpu_create failed (no CUDA device? there is no CPU fallback)")

    def _check(self, rc):
        if rc:
            raise TfGpuError(rc, (self.lib.tf_gpu_last_error(self.h) or b"").decode())

    def close(self):
        if getattr(self, "h", None):
            self.lib.tf_gpu_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    # av1_estimate_noise_from_single_plane (temporal_filter.c:1150-1194)
    def estimate_noise_from_single_plane(self, frame, plane, bit_depth, edge_thresh=NOISE_ESTIMATION_EDGE_THRESHOLD):
        out = C.c_double()
        cf = frame.c_frame()
        self._check(self.lib.tf_gpu_estimate_noise(self.h, C.byref(cf), plane, bit_depth, edge_thresh, C.byref(out)))
        return out.value

    # av1_temporal_filter (temporal_filter.c:1276-1312)
    def temporal_filter(self, params, frames, out, dump=False):
        """frames: list of Yv12Buffer; out: Yv12Buffer.  Returns dict(diff=[sum, sse], mvs, mses, pred, accum, count)."""
        cp = make_params(params) if isinstance(params, dict) else params
        n = cp.num_frames
        arr = (Frame * max(len(frames), 1))(*[f.c_frame() for f in frames])
        co = out.c_frame()
        diff = (C.c_int64 * 2)()
        res = {}
        if dump:
            n = max(n, 1)
            mb_rows, mb_cols = (out.height + 31) // 32, (out.width + 31) // 32
            nb = mb_rows * mb_cols
            num_pels = 1024 + (0 if cp.num_planes == 1 else 2 * (1024 >> (out.ss_x + out.ss_y)))
            res["mvs"] = np.zeros((nb, n, 4, 2), np.int16)
            res["mses"] = np.zeros((nb, n, 4), np.int32)
            res["pred"] = np.zeros((nb, n, num_pels), np.uint16)
            res["accum"] = np.zeros((nb, num_pels), np.uint32)
            res["count"] = np.zeros((nb, num_pels), np.uint16)
            d = Dump(*[res[k].ctypes.data for k in ("mvs", "mses", "pred", "accum", "count")])
            self._check(self.lib.tf_gpu_filter_dump(self.h, C.byref(cp), arr, C.byref(co), diff, C.byref(d)))
        else:
            self._check(self.lib.tf_gpu_filter(self.h, C.byref(cp), arr, C.byref(co), diff))
        res["diff"] = np.array([diff[0], diff[1]], np.int64)
        return res

    def submit(self, params, frames, out):
        cp = make_params(params) if isinstance(params, dict) else params
        arr = (Frame * max(len(frames), 1))(*[f.c_frame() for f in frames])
        co = out.c_frame()
        diff = (C.c_int64 * 2)()
        t = C.c_uint64()
        self._check(self.lib.tf_gpu_submit(self.h, C.byref(cp), arr, C.byref(co), diff, C.byref(t)))
        return t.value, diff, (arr, co)

    def wait(self, ticket):
        self._check(self.lib.tf_gpu_wait(self.h, ticket))

    def cache_frame(self, frame):
        cf = frame.c_frame()
        self._check(self.lib.tf_gpu_cache_frame(self.h, C.byref(cf)))

    def cache_frame_async(self, frame):
        """Upload without waiting (at most one outstanding; see tf_gpu.h)."""
        cf = frame.c_frame()
        self._check(self.lib.tf_gpu_cache_frame_async(self.h, C.byref(cf)))

    # ---- frames that already live in device memory (torch CUDA tensors) ---------------------------------------
    def cache_frame_tensor(self, frame_id, y, u=None, v=None):
        """Put a frame held in CUDA tensors into the device cache (tf_gpu_cache_frame_device): see tensor_frame()
        for what the tensors may be.  Ordered on the tensors' current torch stream: the ingest runs after what is
        already enqueued there, and later work on that stream runs after the ingest, so the tensors may be
        overwritten on that stream right after the call.  They may also be freed: the tensors are recorded as in use
        on that stream (Tensor.record_stream), so the caching allocator does not hand their memory out again, on
        the stream they were allocated on or any other, before the ingest has read it.  Does not block the host."""
        import torch
        f, dev = tensor_frame(frame_id, y, u, v)
        s = torch.cuda.current_stream(dev)
        self._check(self.lib.tf_gpu_cache_frame_device(self.h, C.byref(f), s.cuda_stream))
        for t in (y, u, v):
            if t is not None:
                t.record_stream(s)

    def _torch_device(self, torch):
        return torch.device("cuda", self.device if self.device >= 0 else torch.cuda.current_device())

    def filter_tensors(self, params, frame_ids):
        """filter_resident() over cached frames, returning the crop area of every output plane as new CUDA tensors
        (uint8 for 8-bit, int16 for high bit depth) and FRAME_DIFF.  params: the dict form (_params.tf_params),
        which carries the crop size.  The copies out of the library's output planes (the zero-copy views
        sharding.SlabWindow.device_planes builds) run on the current torch stream and have finished on return,
        so the next filter call of this context may overwrite the planes."""
        import torch
        _, diff = self.filter_resident(params, frame_ids)
        out = self._clone_planes(torch, params, self.output_device_plane)
        torch.cuda.current_stream(self._torch_device(torch)).synchronize()
        return out, diff

    def _clone_planes(self, torch, params, device_plane):
        """Crop area of every output plane that device_plane(plane) describes, cloned on the current torch stream."""
        dev = self._torch_device(torch)
        W, H = params["width"], params["height"]
        out = []
        for pl in range(1 if params["monochrome"] else 3):
            sx, sy = (params["ss_x"], params["ss_y"]) if pl else (0, 0)
            es = 2 if params["use_hbd"] else 1
            ptr, pitch, rows, _ = device_plane(pl)

            class _View:  # __cuda_array_interface__ holder
                pass
            view = _View()
            view.__cuda_array_interface__ = {"shape": (rows, pitch), "typestr": "|u1", "data": (ptr, False),
                                             "version": 3}
            t = torch.as_tensor(view, device=dev)[:(H + sy) >> sy, :((W + sx) >> sx) * es]
            out.append(t.view(torch.int16).clone() if es == 2 else t.clone())
        return out

    # ---- several windows over one frame cache in one call (tf_gpu_filter_batch_async) -------------------------
    def filter_batch_async(self, params_list, frame_ids_list):
        """Enqueue a batch of windows over resident frames (see batch_args for the checks made here)."""
        n, params, ptrs, _ = batch_args(params_list, frame_ids_list)
        self._check(self.lib.tf_gpu_filter_batch_async(self.h, n, params, ptrs))
        self._batch_n = n
        return n

    def filter_batch_result(self, n=None):
        """Wait for the last batch: (kernel ms, FRAME_DIFF int64[n, 2]), n = its window count unless given (at most
        that).  The library writes one entry per window of the last batch, so the buffer holds TF_GPU_MAX_BATCH."""
        last = getattr(self, "_batch_n", 0)
        n = last if n is None else min(int(n), last)
        diffs = (C.c_int64 * 2 * TF_GPU_MAX_BATCH)()
        ms = C.c_float()
        self._check(self.lib.tf_gpu_filter_batch_result(self.h, diffs, C.byref(ms)))
        return ms.value, np.array([[d[0], d[1]] for d in diffs[:n]], np.int64).reshape(n, 2)

    def filter_batch(self, params_list, frame_ids_list):
        """Filter several windows over cached frames in one call: (kernel ms, FRAME_DIFF int64[n, 2]).  Each window's
        output stays on the device (download_batch_output, batch_output_device_plane) until the next batch."""
        return self.filter_batch_result(self.filter_batch_async(params_list, frame_ids_list))

    def download_batch_output(self, window, out):
        co = out.c_frame()
        self._check(self.lib.tf_gpu_download_batch_output(self.h, window, C.byref(co)))

    def batch_output_device_plane(self, window, plane):
        p, pitch, rows, rb = C.c_void_p(), C.c_size_t(), C.c_int(), C.c_int()
        self._check(self.lib.tf_gpu_batch_output_device_plane(self.h, window, plane, C.byref(p), C.byref(pitch),
                                                              C.byref(rows), C.byref(rb)))
        return p.value, pitch.value, rows.value, rb.value

    def filter_batch_tensors(self, params_list, frame_ids_list):
        """filter_batch() returning, per window, (output planes as new CUDA tensors, FRAME_DIFF) as filter_tensors
        does.  params_list: dicts (_params.tf_params).  The copies run on the current torch stream and have
        finished on return."""
        import torch
        _, diffs = self.filter_batch(params_list, frame_ids_list)
        res = []
        for w, p in enumerate(params_list):
            res.append((self._clone_planes(torch, p, lambda pl, w=w: self.batch_output_device_plane(w, pl)), diffs[w]))
        torch.cuda.current_stream(self._torch_device(torch)).synchronize()
        return res

    def estimate_noise_tensor(self, frame_id, tensors, plane, bit_depth,
                              edge_thresh=NOISE_ESTIMATION_EDGE_THRESHOLD):
        """av1_estimate_noise_from_single_plane on a frame held in CUDA tensors (y,) or (y, u, v): ingests it under
        frame_id (nothing is read when that id is resident), then estimates from the cached slot."""
        y, u, v = (tuple(tensors) + (None, None))[:3]
        self.cache_frame_tensor(frame_id, y, u, v)
        f, _ = tensor_frame(frame_id, y, u, v)
        out = C.c_double()
        self._check(self.lib.tf_gpu_estimate_noise(self.h, C.byref(f), plane, bit_depth, edge_thresh, C.byref(out)))
        return out.value

    def debug_read_plane(self, frame, plane, x0, y0, w, h):
        """Rectangle of a cached device plane, border included (test hook for the upload path)."""
        dst = np.zeros((h, w), frame.dtype)
        self._check(self.lib.tf_gpu_debug_read_plane(self.h, frame.frame_id, plane, dst.ctypes.data, w, x0, y0, w, h))
        return dst

    def fullpel_search_batch(self, params, src, ref, block_size, items):
        """items: sequence of (x, y, start_row, start_col); returns an int array [n, 3] of (row, col, var) --
        av1_full_pixel_search() as tf_motion_search() configures it, per block (see tf_gpu.h)."""
        cp = make_params(params) if isinstance(params, dict) else params
        n = len(items)
        arr = (SearchItem * max(n, 1))(*[SearchItem(*map(int, it)) for it in items])
        res = (SearchResult * max(n, 1))()
        cs, cr = src.c_frame(), ref.c_frame()
        self._check(self.lib.tf_gpu_fullpel_search_batch(self.h, C.byref(cp), C.byref(cs), C.byref(cr), block_size, arr, n, res))
        return np.array([(r.row, r.col, r.var) for r in res[:n]], np.int64).reshape(n, 3)

    def motion_search_batch(self, params, src_id, ref_ids, block_size, items):
        """tf_motion_search()'s search of many blocks of the resident frame src_id against the resident frames
        ref_ids (uploaded or ingested from tensors) in one call: see tf_gpu_motion_search_batch in tf_gpu.h and
        motion_search_args for items.  Returns an int64 array (n, 6): fullpel_row, fullpel_col, fullpel_var, row,
        col (1/8 pel), err."""
        cp = make_params(params) if isinstance(params, dict) else params
        ids, num_refs, packed, n = motion_search_args(ref_ids, block_size, items)
        res = np.zeros(max(n, 1), _MOTION_RESULT_DTYPE)
        self._check(self.lib.tf_gpu_motion_search_batch(
            self.h, C.byref(cp), int(src_id), ids, num_refs, block_size,
            C.cast(packed.ctypes.data, C.POINTER(MotionItem)), n, C.cast(res.ctypes.data, C.POINTER(MotionResult))))
        return np.stack([res[k][:n].astype(np.int64) for k in _MOTION_RESULT_DTYPE.names], axis=1).reshape(n, 6)

    def motion_search_tensors(self, params, src_id, ref_ids, block_size, items):
        """motion_search_batch() with items and results on the GPU (tf_gpu_motion_search_device): items is an integer
        CUDA tensor (n, 5) on the context's device (see motion_search_device_args); returns a new int64 CUDA tensor
        (n, 6) with the columns of motion_search_batch.  Packing, search and unpacking run in order on the current
        torch stream of that device, after what is already enqueued there, and the call does not synchronise: read
        the result on that stream (or after synchronising it).  The starts are taken as int16, as the C struct holds
        them, without a range check (which would need a synchronise); the full-pel search clamps its start into the
        block's MV limits, so any start is safe.  An item whose position or ref the kernel rejects gets
        fullpel_var = TF_GPU_MOTION_REJECTED, MVs 0 and err = 2**32 - 1.  The input buffers need no record_stream:
        the library makes the stream wait for the search before the call returns."""
        import torch
        cp = make_params(params) if isinstance(params, dict) else params
        dev = self._torch_device(torch)
        ids, num_refs, n = motion_search_device_args(ref_ids, block_size, items, dev)
        with torch.cuda.device(dev):
            packed = pack_motion_items(items) if n else torch.zeros((1, 4), dtype=torch.int32, device=dev)
            res = torch.empty((max(n, 1), 4), dtype=torch.int32, device=dev)
            s = torch.cuda.current_stream(dev)
            self._check(self.lib.tf_gpu_motion_search_device(self.h, C.byref(cp), int(src_id), ids, num_refs,
                                                             block_size, packed.data_ptr(), n, res.data_ptr(),
                                                             s.cuda_stream))
            return unpack_motion_results(res[:n])

    def device_border(self):
        return self.lib.tf_gpu_device_border()

    def evict_frame(self, frame_id):
        self._check(self.lib.tf_gpu_evict_frame(self.h, frame_id))

    def filter_resident(self, params, frame_ids):
        cp = make_params(params) if isinstance(params, dict) else params
        ids = (C.c_uint64 * len(frame_ids))(*frame_ids)
        diff = (C.c_int64 * 2)()
        ms = C.c_float()
        self._check(self.lib.tf_gpu_filter_resident(self.h, C.byref(cp), ids, diff, C.byref(ms)))
        return ms.value, np.array([diff[0], diff[1]], np.int64)

    def filter_resident_async(self, params, frame_ids):
        cp = make_params(params) if isinstance(params, dict) else params
        ids = (C.c_uint64 * len(frame_ids))(*frame_ids)
        self._check(self.lib.tf_gpu_filter_resident_async(self.h, C.byref(cp), ids))

    def filter_resident_result(self):
        diff = (C.c_int64 * 2)()
        ms = C.c_float()
        self._check(self.lib.tf_gpu_filter_resident_result(self.h, diff, C.byref(ms)))
        return ms.value, np.array([diff[0], diff[1]], np.int64)

    def download_output(self, out, row_begin=0, row_end=0):
        co = out.c_frame()
        self._check(self.lib.tf_gpu_download_output(self.h, C.byref(co), row_begin, row_end))

    def output_device_plane(self, plane):
        p, pitch, rows, rb = C.c_void_p(), C.c_size_t(), C.c_int(), C.c_int()
        self._check(self.lib.tf_gpu_output_device_plane(self.h, plane, C.byref(p), C.byref(pitch), C.byref(rows),
                                                        C.byref(rb)))
        return p.value, pitch.value, rows.value, rb.value

    def output_ipc_export(self, plane):
        """(handle bytes, byte offset of pixel (0,0), pitch bytes) of an output plane, for another rank's import."""
        buf = C.create_string_buffer(64)
        off, pitch = C.c_size_t(), C.c_size_t()
        self._check(self.lib.tf_gpu_output_ipc_export(self.h, plane, buf, C.byref(off), C.byref(pitch)))
        return buf.raw, off.value, pitch.value

    def output_ipc_import(self, plane, handle, offset=0, pitch=0):
        """Store this context's output rows into another rank's plane (handle=None: back to its own planes)."""
        self._check(self.lib.tf_gpu_output_ipc_import(self.h, plane, handle, offset, pitch))

    def host_register(self, arr):
        self._check(self.lib.tf_gpu_host_register(self.h, arr.ctypes.data, arr.nbytes))

    def host_unregister(self, arr):
        self._check(self.lib.tf_gpu_host_unregister(self.h, arr.ctypes.data))

    def event_record(self, slot):
        self._check(self.lib.tf_gpu_event_record(self.h, slot))

    def event_elapsed_ms(self, a, b):
        ms = C.c_float()
        self._check(self.lib.tf_gpu_event_elapsed_ms(self.h, a, b, C.byref(ms)))
        return ms.value

    def synchronize(self):
        self._check(self.lib.tf_gpu_synchronize(self.h))

    def microbench(self, kind):
        v = C.c_double()
        self._check(self.lib.tf_gpu_microbench(self.h, kind, C.byref(v)))
        return v.value

    def collect_counters(self, enable):
        self._check(self.lib.tf_gpu_collect_counters(self.h, int(enable)))

    def read_counters(self):
        c = (C.c_uint64 * 4)()
        self._check(self.lib.tf_gpu_read_counters(self.h, c))
        return [int(x) for x in c]

    def last_kernel_times(self):
        ms = (C.c_float * 3)()
        self._check(self.lib.tf_gpu_last_kernel_times(self.h, ms))
        return [ms[0], ms[1], ms[2]]

    def last_stats(self):
        n, ms = C.c_int(), C.c_float()
        self._check(self.lib.tf_gpu_last_stats(self.h, C.byref(n), C.byref(ms)))
        return n.value, ms.value
