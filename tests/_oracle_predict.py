"""ctypes binding for the oracle's block predictor at caller MVs (tests/_oracle_predict.c: tf_build_predictor's
position rule for one block and the pinned tfo_convolve12 of oracle/tf_oracle.c, which that unit compiles unchanged).
The library is built on first use into a temporary directory, named by a hash of its sources, so the tree stays
read-only.  TEST INFRASTRUCTURE ONLY -- never imported by the product."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

import _oracle

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = (os.path.join(HERE, "_oracle_predict.c"), os.path.join(_oracle.ORACLE_DIR, "tf_oracle.c"),
           os.path.join(_oracle.ORACLE_DIR, "tf_oracle.h"))

_lib = None


def build():
    h = hashlib.sha256()
    for s in SOURCES:
        with open(s, "rb") as f:
            h.update(f.read())
    out = os.path.join(tempfile.gettempdir(), f"tf_oracle_predict_{h.hexdigest()[:16]}.so")
    if not os.path.exists(out):
        tmp = f"{out}.{os.getpid()}.tmp"
        subprocess.check_call([os.environ.get("CC", "gcc"), "-O2", "-fPIC", "-shared", "-std=c11", "-Wall", "-o", tmp,
                               SOURCES[0], "-lm"])
        os.replace(tmp, out)
    return out


def lib():
    global _lib
    if _lib is None:
        l = C.CDLL(build())
        _oracle.bind_common(l)
        l.tfo_predict_block.argtypes = [C.c_void_p] + [C.c_int] * 7 + [C.c_void_p]
        l.tfo_predict_block.restype = None
        l.tfo_convolve12.argtypes = [C.c_void_p, C.c_int, C.c_void_p, C.c_int] + [C.c_int] * 6
        l.tfo_convolve12.restype = None
        _lib = l
    return _lib


def reset_stats():
    """Zero the event counters of this library's copy of the oracle (separate from _oracle's)."""
    lib().tfo_reset_stats()


def get_stats():
    return _oracle.read_stats(lib())


class PredictOracle:
    """Frames as for _oracle.OracleFilter (params dict of tests/_params.tf_params, list of (y, u, v))."""

    def __init__(self, p, frames):
        self.p = dict(p)
        self.h, self.cp = _oracle.create(lib(), p)
        dt = np.uint16 if p["use_hbd"] else np.uint8
        for i, planes in enumerate(frames):  # tfo_set_frame copies the samples
            arrs = [None if a is None else np.ascontiguousarray(a.astype(dt)) for a in planes]
            lib().tfo_set_frame(self.h, i, *[_oracle._ptr(a) for a in arrs])

    def predict_block(self, ref_idx, bsize, x, y, mv_row, mv_col, num_planes):
        """The filter's predictor of the bsize block at (x, y) of frame ref_idx at MV (mv_row, mv_col), 1/8 pel: a
        uint16 array of num_pels samples in the layout of tfo_run's pred recorder."""
        ss_x, ss_y = self.p["ss_x"], self.p["ss_y"]
        n = bsize * bsize + (2 * (bsize >> ss_x) * (bsize >> ss_y) if num_planes == 3 else 0)
        out = np.zeros(n, np.uint16)
        lib().tfo_predict_block(self.h, ref_idx, bsize, x, y, mv_row, mv_col, num_planes, out.ctypes.data)
        return out

    def close(self):
        if self.h:
            lib().tfo_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
