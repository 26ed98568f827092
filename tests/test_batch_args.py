"""CPU: argument building and checks of TemporalFilterGpu.filter_batch* (batch_args), made before the C call."""
import ctypes as C

import pytest

import _params


def _p(n, **kw):
    return _params.tf_params(352, 288, n, **kw)


def test_batch_args_builds_one_id_array_per_window(pkg):
    n, params, ptrs, _ = pkg.batch_args([_p(3), _p(1), _p(5, filter_frame_idx=0)], [[1, 2, 3], [7], [4, 5, 6, 7, 8]])
    assert n == 3
    assert [params[w].num_frames for w in range(3)] == [3, 1, 5]
    assert params[2].filter_frame_idx == 0
    assert [ptrs[1][0]] == [7]
    assert [ptrs[2][i] for i in range(5)] == [4, 5, 6, 7, 8]
    assert C.sizeof(params) == 3 * C.sizeof(pkg.Params)


def test_batch_args_accepts_params_structs(pkg):
    cp = pkg.make_params(_p(2))
    n, params, _, _ = pkg.batch_args([cp], [(11, 12)])
    assert n == 1 and params[0].num_frames == 2


def test_batch_args_full_batch(pkg):
    m = pkg.TF_GPU_MAX_BATCH
    assert m == 16
    n, _, _, _ = pkg.batch_args([_p(1)] * m, [[i + 1] for i in range(m)])
    assert n == m


@pytest.mark.parametrize("params_list, ids_list, msg", [
    ([_p(2), _p(2)], [[1, 2]], "2 params for 1 id lists"),
    ([], [], "1 to 16 windows, got 0"),
    ([_p(1)] * 17, [[1]] * 17, "1 to 16 windows, got 17"),
    ([_p(3)], [[1, 2]], "window 0: 2 frame ids for num_frames 3"),
    ([_p(1), _p(2)], [[1], [1, 2, 3]], "window 1: 3 frame ids for num_frames 2"),
])
def test_batch_args_rejects(pkg, params_list, ids_list, msg):
    with pytest.raises(ValueError, match=msg):
        pkg.batch_args(params_list, ids_list)
