"""CPU: the checks of TemporalFilterGpu.motion_search_tensors made before the C call (motion_search_device_args), and
the torch packing of tf_gpu_motion_item / unpacking of tf_gpu_motion_result against the numpy views of the structs."""
import numpy as np
import pytest
import torch


@pytest.mark.parametrize("ref_ids, bsize, items, msg", [
    ([1], 16, np.zeros((1, 5), np.int32), "must be a torch tensor"),
    ([1], 16, [[0, 0, 0, 0, 0]], "must be a torch tensor"),
    ([1], 16, torch.zeros((1, 5), dtype=torch.int32), "must be a CUDA tensor"),
    ([1], 16, torch.zeros((1, 5), dtype=torch.int32, device="meta"), "must be a CUDA tensor"),
    ([1], 16, torch.zeros((3, 4), dtype=torch.int32), r"shape \(n, 5\)"),
    ([1], 16, torch.zeros(5, dtype=torch.int32), r"shape \(n, 5\)"),
    ([1], 16, torch.zeros((1, 5, 1), dtype=torch.int32), r"shape \(n, 5\)"),
    ([1], 16, torch.zeros((2, 5), dtype=torch.float32), "must be integers"),
    ([1], 16, torch.zeros((2, 5), dtype=torch.bool), "must be integers"),
    ([1], 16, torch.zeros((2, 5), dtype=torch.complex64), "must be integers"),
    ([], 16, torch.zeros((1, 5), dtype=torch.int32), "1 to 23 reference frames, got 0"),
    (list(range(1, 25)), 16, torch.zeros((1, 5), dtype=torch.int32), "1 to 23 reference frames, got 24"),
    ([1], 8, torch.zeros((1, 5), dtype=torch.int32), "block_size must be 16 or 32"),
    ([1], 24, torch.zeros((1, 5), dtype=torch.int32), "block_size must be 16 or 32"),
])
def test_rejects(pkg, ref_ids, bsize, items, msg):
    with pytest.raises(ValueError, match=msg):
        pkg.motion_search_device_args(ref_ids, bsize, items, torch.device("cuda", 0))


def test_round_trip_against_the_struct_dtypes(pkg):
    rng = np.random.default_rng(1)
    n = 257
    items = np.stack([rng.integers(-2 ** 31, 2 ** 31, n), rng.integers(-2 ** 31, 2 ** 31, n),
                      rng.integers(-2 ** 15, 2 ** 15, n), rng.integers(-2 ** 15, 2 ** 15, n),
                      rng.integers(-2 ** 31, 2 ** 31, n)], axis=1)
    items[:3] = [[0, 0, -32768, 32767, 0], [16, 4, -3, 7, 22], [-16, 2 ** 31 - 1, -1, 1, -1]]
    for dtype in (torch.int64, torch.int32):
        packed = pkg.pack_motion_items(torch.from_numpy(items).to(dtype))
        assert packed.dtype == torch.int32 and packed.shape == (n, 4)
        want = np.zeros(n, pkg._MOTION_ITEM_DTYPE)
        for k, name in enumerate(pkg._MOTION_ITEM_DTYPE.names):
            want[name] = items[:, k]
        assert packed.numpy().tobytes() == want.tobytes()
    small = torch.tensor([[16, 8, -5, 6, 1]], dtype=torch.int16)  # narrower integer inputs widen
    assert pkg.pack_motion_items(small).numpy().view(pkg._MOTION_ITEM_DTYPE).ravel()[0].tolist() == (16, 8, -5, 6, 1)

    res = np.zeros(n, pkg._MOTION_RESULT_DTYPE)
    fields = [rng.integers(-2 ** 15, 2 ** 15, n), rng.integers(-2 ** 15, 2 ** 15, n),
              rng.integers(-2 ** 31, 2 ** 31, n), rng.integers(-2 ** 15, 2 ** 15, n),
              rng.integers(-2 ** 15, 2 ** 15, n), rng.integers(0, 2 ** 32, n)]
    for name, f in zip(pkg._MOTION_RESULT_DTYPE.names, fields):
        res[name] = f
    res[0] = (0, 0, pkg.TF_GPU_MOTION_REJECTED, 0, 0, 2 ** 32 - 1)  # a rejected item
    res[1] = (-1023, 1023, 2 ** 31 - 1, -8184, 8184, 2 ** 31)      # err >= 2**31 stays unsigned
    got = pkg.unpack_motion_results(torch.from_numpy(res.view(np.int32).reshape(n, 4).copy()))
    assert got.dtype == torch.int64 and got.shape == (n, 6)
    want = np.stack([res[k].astype(np.int64) for k in pkg._MOTION_RESULT_DTYPE.names], axis=1)
    assert (got.numpy() == want).all()
    assert got[0].tolist() == [0, 0, -1, 0, 0, 2 ** 32 - 1] and got[1, 5] == 2 ** 31


def test_empty(pkg):
    assert pkg.pack_motion_items(torch.zeros((0, 5), dtype=torch.int64)).shape == (0, 4)
    assert pkg.unpack_motion_results(torch.zeros((0, 4), dtype=torch.int32)).shape == (0, 6)
