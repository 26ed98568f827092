"""CPU: the checks of TemporalFilterGpu.predict_tensors made before the C call (predict_device_args), and
pack_motion_items read back as tf_gpu_predict_item."""
import ctypes as C

import numpy as np
import pytest
import torch


@pytest.mark.parametrize("ref_ids, bsize, items, msg", [
    ([1], 16, np.zeros((1, 5), np.int32), "must be a torch tensor"),
    ([1], 16, torch.zeros((1, 5), dtype=torch.int32), "must be a CUDA tensor"),
    ([1], 16, torch.zeros((3, 4), dtype=torch.int32), r"shape \(n, 5\)"),
    ([1], 16, torch.zeros((2, 5), dtype=torch.float32), "must be integers"),
    ([], 16, torch.zeros((1, 5), dtype=torch.int32), "1 to 23 reference frames, got 0"),
    (list(range(1, 25)), 32, torch.zeros((1, 5), dtype=torch.int32), "1 to 23 reference frames, got 24"),
    ([1], 8, torch.zeros((1, 5), dtype=torch.int32), "block_size must be 16 or 32"),
    ([1], 64, torch.zeros((1, 5), dtype=torch.int32), "block_size must be 16 or 32"),
])
def test_rejects(pkg, ref_ids, bsize, items, msg):
    with pytest.raises(ValueError, match=msg):
        pkg.predict_device_args(ref_ids, bsize, items, torch.device("cuda", 0))


def test_packed_items_read_back_as_predict_items(pkg):
    rng = np.random.default_rng(7)
    n = 129
    items = np.stack([rng.integers(-2 ** 31, 2 ** 31, n), rng.integers(-2 ** 31, 2 ** 31, n),
                      rng.integers(-2 ** 15, 2 ** 15, n), rng.integers(-2 ** 15, 2 ** 15, n),
                      rng.integers(-2 ** 31, 2 ** 31, n)], axis=1)
    items[:2] = [[0, 4, -32768, 32767, 22], [1904, 1076, -7, 13, 0]]
    packed = pkg.pack_motion_items(torch.from_numpy(items))
    got = (pkg.PredictItem * n).from_buffer_copy(packed.numpy().tobytes())
    assert C.sizeof(pkg.PredictItem) == 16
    assert [(g.x, g.y, g.row, g.col, g.ref) for g in got] == [tuple(r) for r in items.tolist()]


def test_predict_tensors_needs_the_dict_params(pkg):
    class _Ctx(pkg.TemporalFilterGpu):
        def __init__(self):  # no device: only the argument check runs
            self.device = 0

    with pytest.raises(ValueError, match="dict form"):
        _Ctx().predict_tensors(pkg.Params(), [1], 16, torch.zeros((1, 5), dtype=torch.int32))
