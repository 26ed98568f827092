"""ctypes binding for the oracle's per-block motion search (tests/_oracle_motion.c: tf_motion_search()'s search of
one block composed from the pinned routines of oracle/tf_oracle.c, which that unit compiles unchanged).  The library
is built on first use into a temporary directory, named by a hash of its sources, so the tree stays read-only.
TEST INFRASTRUCTURE ONLY -- never imported by the product."""
import ctypes as C
import hashlib
import os
import subprocess
import tempfile

import numpy as np

import _oracle

HERE = os.path.dirname(os.path.abspath(__file__))
SOURCES = (os.path.join(HERE, "_oracle_motion.c"), os.path.join(_oracle.ORACLE_DIR, "tf_oracle.c"),
           os.path.join(_oracle.ORACLE_DIR, "tf_oracle.h"))

_lib = None


def build():
    h = hashlib.sha256()
    for s in SOURCES:
        with open(s, "rb") as f:
            h.update(f.read())
    out = os.path.join(tempfile.gettempdir(), f"tf_oracle_motion_{h.hexdigest()[:16]}.so")
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
        l.tfo_motion_search.argtypes = [C.c_void_p] + [C.c_int] * 7 + [C.POINTER(C.c_int)]
        l.tfo_mv_limits.argtypes = [C.c_void_p] + [C.c_int] * 3 + [C.POINTER(C.c_int)]
        _lib = l
    return _lib


def reset_stats():
    """Zero the event counters of this library's copy of the oracle (separate from _oracle's)."""
    lib().tfo_reset_stats()


def get_stats():
    return _oracle.read_stats(lib())


class MotionOracle:
    """Frames as for _oracle.OracleFilter (params dict of tests/_params.tf_params, list of (y, u, v))."""

    def __init__(self, p, frames):
        self.h, self.cp = _oracle.create(lib(), p)
        dt = np.uint16 if p["use_hbd"] else np.uint8
        for i, planes in enumerate(frames):  # tfo_set_frame copies the samples
            arrs = [None if a is None else np.ascontiguousarray(a.astype(dt)) for a in planes]
            lib().tfo_set_frame(self.h, i, *[_oracle._ptr(a) for a in arrs])

    def motion_search(self, src_idx, ref_idx, bsize, x, y, start_row, start_col):
        """-> (full row, full col, full var cost, row (1/8 pel), col (1/8 pel), err)."""
        out = (C.c_int * 6)()
        lib().tfo_motion_search(self.h, src_idx, ref_idx, bsize, x, y, start_row, start_col, out)
        return tuple(int(v) for v in out[:5]) + (out[5] & 0xffffffff,)

    def mv_limits(self, bsize, x, y):
        """The full-pel MV limits of a bsize block at (x, y): (row_min, row_max, col_min, col_max)."""
        out = (C.c_int * 4)()
        lib().tfo_mv_limits(self.h, bsize, x, y, out)
        return tuple(out)

    def close(self):
        if self.h:
            lib().tfo_destroy(self.h)
            self.h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
