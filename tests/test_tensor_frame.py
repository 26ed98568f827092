"""CPU: the frame descriptor built over torch tensors (tensor_frame, used by cache_frame_tensor) -- malformed planes
raise ValueError before the C ABI is called; the checks run in an order that lets host tensors reach each of them."""
import pytest
import torch


def _planes(W, H, dt, cw=None, ch=None):
    cw = (W + 1) >> 1 if cw is None else cw
    ch = (H + 1) >> 1 if ch is None else ch
    return torch.zeros((H, W), dtype=dt), torch.zeros((ch, cw), dtype=dt), torch.zeros((ch, cw), dtype=dt)


@pytest.mark.parametrize("bad", ["dtype", "mixed", "chroma_shape", "u_only", "uv_differ", "column_stride", "cpu", "3d",
                                 "uv_row_stride", "vu_row_stride"])
def test_malformed_planes_raise_value_error(pkg, bad):
    y, u, v = _planes(64, 48, torch.uint8)
    if bad == "dtype":
        y, u, v = _planes(64, 48, torch.int32)
    elif bad == "mixed":
        u = u.to(torch.int16)
    elif bad == "chroma_shape":
        y, u, v = _planes(64, 48, torch.uint8, cw=20, ch=24)
    elif bad == "u_only":
        v = None
    elif bad == "uv_differ":
        v = torch.zeros((24, 31), dtype=torch.uint8)
    elif bad == "column_stride":
        y = torch.zeros((48, 128), dtype=torch.uint8)[:, ::2]
    elif bad == "3d":
        y = y[None]
    elif bad in ("uv_row_stride", "vu_row_stride"):  # tf_gpu_frame has one uv stride
        wide = torch.zeros((24, 40), dtype=torch.uint8)[:, 3:35]
        u, v = (u, wide) if bad == "uv_row_stride" else (wide, v)
    with pytest.raises(ValueError, match="row stride" if bad.endswith("row_stride") else None):
        pkg.tensor_frame(7, y, u, v)


def test_cpu_tensor_passes_every_check_but_the_device(pkg):
    for dt in (torch.uint8, torch.int16):
        with pytest.raises(ValueError, match="CUDA"):
            pkg.tensor_frame(7, *_planes(353, 289, dt))
        with pytest.raises(ValueError, match="CUDA"):
            pkg.tensor_frame(7, torch.zeros((17, 9), dtype=dt))
    for cw, ch in ((64, 24), (32, 48), (64, 48)):  # 4:2:2-like, 4:4:0, 4:4:4
        with pytest.raises(ValueError, match="CUDA"):
            pkg.tensor_frame(7, *_planes(64, 48, torch.uint8, cw=cw, ch=ch))


def test_chroma_planes_with_one_padded_stride_pass_to_the_device_check(pkg):
    """Both chroma planes column slices of wider tensors with the same row stride: one uv stride describes them."""
    y = torch.zeros((48, 64), dtype=torch.int16)
    u = torch.zeros((24, 45), dtype=torch.int16)[:, 5:37]
    v = torch.zeros((24, 45), dtype=torch.int16)[:, 1:33]
    with pytest.raises(ValueError, match="CUDA"):
        pkg.tensor_frame(7, y, u, v)
