"""CPU: argument packing and checks of TemporalFilterGpu.motion_search_batch (motion_search_args), made before the C
call."""
import numpy as np
import pytest


def test_packs_items_in_field_order(pkg):
    items = np.array([[0, 0, 0, 0, 0], [16, 4, -3, 7, 2], [32, 8, -32768, 32767, 1]], np.int32)
    ids, num_refs, packed, n = pkg.motion_search_args([11, 12, 13], 16, items)
    assert (n, num_refs) == (3, 3)
    assert [ids[i] for i in range(3)] == [11, 12, 13]
    assert packed.dtype.itemsize == 16 and packed.flags.c_contiguous
    assert packed[1].tolist() == (16, 4, -3, 7, 2)
    assert packed[2].tolist() == (32, 8, -32768, 32767, 1)


@pytest.mark.parametrize("items", [[[0, 0, 0, 0, 0]], ((16, 0, 1, 2, 0),), np.zeros((4, 5), np.uint8),
                                   np.zeros((2, 5), np.int64)])
def test_accepts_integer_array_likes(pkg, items):
    _, _, packed, n = pkg.motion_search_args([5], 32, items)
    assert n == len(packed) == len(items)


@pytest.mark.parametrize("items", [[], np.zeros((0, 5), np.int32)])
def test_empty_batch(pkg, items):
    _, _, packed, n = pkg.motion_search_args([5], 16, items)
    assert n == 0 and len(packed) == 0


def test_most_references(pkg):
    m = pkg.TF_GPU_MAX_FRAMES - 1
    assert m == 23
    _, num_refs, _, _ = pkg.motion_search_args(range(1, m + 1), 16, [[0, 0, 0, 0, m - 1]])
    assert num_refs == m


@pytest.mark.parametrize("ref_ids, bsize, items, msg", [
    ([1], 16, np.zeros((3, 4), np.int32), r"shape \(n, 5\)"),
    ([1], 16, np.zeros(5, np.int32), r"shape \(n, 5\)"),
    ([1], 16, np.zeros((1, 5, 1), np.int32), r"shape \(n, 5\)"),
    ([1], 16, np.zeros((2, 5), np.float32), "must be integers"),
    ([1], 16, [[0, 0, 0.5, 0, 0]], "must be integers"),
    ([1], 16, np.zeros((2, 5), bool), "must be integers"),
    ([1], 16, [[0, 0, 32768, 0, 0]], "int16"),
    ([1], 16, [[0, 0, 0, -32769, 0]], "int16"),
    ([1], 16, [[2 ** 31, 0, 0, 0, 0]], "int32"),
    ([1, 2], 16, [[0, 0, 0, 0, 2]], r"ref out of \[0, 2\)"),
    ([1, 2], 16, [[0, 0, 0, 0, -1]], r"ref out of \[0, 2\)"),
    ([], 16, np.zeros((1, 5), np.int32), "1 to 23 reference frames, got 0"),
    (list(range(1, 25)), 16, np.zeros((1, 5), np.int32), "1 to 23 reference frames, got 24"),
    ([1], 8, np.zeros((1, 5), np.int32), "block_size must be 16 or 32"),
    ([1], 24, np.zeros((1, 5), np.int32), "block_size must be 16 or 32"),
])
def test_rejects(pkg, ref_ids, bsize, items, msg):
    with pytest.raises(ValueError, match=msg):
        pkg.motion_search_args(ref_ids, bsize, items)
