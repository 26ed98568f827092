"""GPU: device ingest of tensors from torch's other allocator back ends.  With expandable segments (virtual-memory
mappings) or the stream-ordered cudaMallocAsync pool, cuMemGetAddressRange may report one mapped chunk rather than
the whole tensor; the extent check of tf_gpu_cache_frame_device follows contiguous chunks, so 4K 10-bit planes
allocated back to back (some crossing chunk boundaries) must be accepted, and their slots must equal the host
upload.  Each back end runs in a fresh interpreter, because the allocator is chosen when torch initialises CUDA."""
import os
import subprocess
import sys

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
pytestmark = pytest.mark.gpu

SCRIPT = r"""
import ctypes as C, sys
import numpy as np, torch
sys.path.insert(0, sys.argv[1]); sys.path.insert(0, sys.argv[2])
import conftest, _clips
pkg = conftest.load_package()
ctx = pkg.TemporalFilterGpu(device=0)
W, H = 3840, 2160
frames = _clips.moving_texture(W, H, 3, 10)
cuda = C.CDLL("libcuda.so.1")
spans = 0
for i, planes in enumerate(frames):
    b = pkg.Yv12Buffer(W, H, 1, 1, True, 160, frame_id=100 + i).set_planes(*planes, extend=False)
    ctx.cache_frame(b)
    tens = [torch.from_numpy(a.view(np.int16)).cuda() for a in planes]
    for t in tens:  # does the range the driver reports for the tensor's first byte cover the whole tensor?
        base, size = C.c_uint64(), C.c_size_t()
        assert cuda.cuMemGetAddressRange_v2(C.byref(base), C.byref(size), C.c_uint64(t.data_ptr())) == 0
        spans += base.value + size.value < t.data_ptr() + t.numel() * 2
    ctx.cache_frame_tensor(200 + i, *tens)
    db = ctx.device_border()
    for pl in range(3):
        bx = db >> 1 if pl else db
        aw, ah = b.aligned[1 if pl else 0]
        got, want = (np.zeros((ah + 2 * bx, aw + 2 * bx), np.uint16) for _ in range(2))
        for fid, dst in ((100 + i, want), (200 + i, got)):
            ctx._check(ctx.lib.tf_gpu_debug_read_plane(ctx.h, fid, pl, dst.ctypes.data, dst.shape[1], -bx, -bx,
                                                       dst.shape[1], dst.shape[0]))
        assert (got == want).all(), (i, pl)
ctx.close()
print("planes crossing a reported range:", spans)
"""


@pytest.mark.parametrize("conf", ["expandable_segments:True", "backend:cudaMallocAsync"])
def test_ingest_accepts_tensors_of_chunked_allocators(conf):
    env = dict(os.environ, PYTORCH_CUDA_ALLOC_CONF=conf)
    r = subprocess.run([sys.executable, "-c", SCRIPT, HERE, os.path.dirname(HERE)], env=env, capture_output=True,
                       text=True, timeout=600)
    print(r.stdout)
    assert r.returncode == 0, r.stderr[-3000:]
