"""CPU: host-side logic -- parameter presets, YV12 layout mirror, clip generator, sharding."""
import os

import numpy as np
import pytest

import _clips
import _params
import _ref


def test_speed_presets_follow_speed_features():
    p = _params.tf_params(1920, 1080, 7, speed=4)
    assert (p["subpel_method"], p["subpel_iters_per_step"], p["prune_mesh_level"], p["use_downsampled_sad"]) == (2, 1, 2, 1)
    assert p["mesh"] == [(64, 16), (24, 8), (12, 4), (7, 1)] and p["border"] == 160
    p = _params.tf_params(352, 288, 7, speed=0)
    assert (p["subpel_method"], p["subpel_iters_per_step"], p["prune_mesh_level"], p["use_downsampled_sad"]) == (0, 2, 0, 0)
    assert p["mesh"][2] == (15, 1) and p["border"] == 160
    p = _params.tf_params(352, 288, 7, speed=3)
    assert (p["subpel_method"], p["prune_mesh_level"], p["border"]) == (1, 1, 96)


def test_clip_generator_is_deterministic():
    a = _clips.moving_texture(64, 48, 3, 10)
    b = _clips.moving_texture(64, 48, 3, 10)
    for (y0, u0, v0), (y1, u1, v1) in zip(a, b):
        assert (y0 == y1).all() and (u0 == u1).all() and (v0 == v1).all()
    assert a[0][0].dtype == np.uint16 and a[0][0].max() < 1024 and a[0][1].shape == (24, 32)


@pytest.mark.skipif(not _ref.available(), reason="oracle/_ref/libtf_ref.so not built")
@pytest.mark.parametrize("dims", [(352, 288, 1, 1, 0, 96), (1920, 1080, 1, 1, 1, 160), (131, 77, 0, 0, 0, 160)])
def test_yv12_mirror_matches_reference_layout(pkg, dims):
    """Yv12Buffer reproduces aom_realloc_frame_buffer's strides / aligned sizes and, with
    extend=True, the exact border contents av1_copy_and_extend_frame produces."""
    W, H, sx, sy, hbd, border = dims
    bd = 10 if hbd else 8
    frames = _clips.moving_texture(W, H, 1, bd, ss_x=sx, ss_y=sy)
    p = _params.tf_params(W, H, 1, bit_depth=bd, ss_x=sx, ss_y=sy, border=border)
    r = _ref.RefFilter(p, frames)
    b = pkg.Yv12Buffer(W, H, sx, sy, hbd, border).set_planes(*frames[0])
    for pl in range(3):
        ref_plane, info = r.plane_with_border(0, pl)
        assert info["y_stride"] == b.stride[0] and info["uv_stride"] == b.stride[1]
        assert (info["aligned_w"], info["aligned_h"]) == b.aligned[0]
        assert ref_plane.shape == b.alloc[pl].shape
        assert (ref_plane == b.alloc[pl]).all()
    r.close()


def test_slab_partition_covers_all_rows(pkg):
    import importlib
    sh = importlib.import_module("aom_av1_psy_b200.sharding")
    for mb_rows in (9, 34, 68):
        for world in (1, 2, 4, 8):
            ranges = [sh.slab_rows(mb_rows, world, r) for r in range(world)]
            assert ranges[0][0] == 0 and ranges[-1][1] == mb_rows
            assert all(ranges[i][1] == ranges[i + 1][0] for i in range(world - 1))
            sizes = [e - b for b, e in ranges]
            assert max(sizes) - min(sizes) <= 1 and max(sizes) == sh.max_slab_rows(mb_rows, world)
    assert [sh.window_owner(i, 8) for i in range(10)] == [0, 1, 2, 3, 4, 5, 6, 7, 0, 1]


def test_int_roofline_work_matches_survey():
    import bench
    w = bench.int_work_per_block_ref(allow_hp=1)
    assert w["sad"] == 144384 and w["var"] == 4096 and w["pred"] == 53760 and w["weights"] == 44544
    assert w["subpel"] == 16 * 2048 * 6


@pytest.mark.skipif(not (_ref.SOURCE_DIR and os.path.exists(os.path.join(_ref.SOURCE_DIR, "av1/encoder/temporal_filter.c"))),
                    reason="upstream source tree not given (REF=<dir>)")
def test_seam_patch_applies_to_the_reference(tmp_path):
    """integration/tf_gpu_seam.patch is a well-formed unified diff against the reference tree."""
    import re
    import shutil
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    patch = os.path.join(root, "integration", "tf_gpu_seam.patch")
    files = re.findall(r"^--- a/(\S+)$", open(patch).read(), re.M)
    assert sorted(files) == ["CMakeLists.txt", "av1/encoder/encode_strategy.c", "av1/encoder/encoder.c",
                             "av1/encoder/temporal_filter.c", "av1/encoder/temporal_filter.h",
                             "build/cmake/aom_config_defaults.cmake"]
    for rel in files:
        os.makedirs(os.path.dirname(tmp_path / rel), exist_ok=True)
        shutil.copyfile(os.path.join(_ref.SOURCE_DIR, rel), tmp_path / rel)
    r = subprocess.run(["patch", "-p1", "-s", "-i", patch], cwd=tmp_path, capture_output=True, text=True)
    assert r.returncode == 0, r.stdout + r.stderr
    patched = open(tmp_path / "av1/encoder/temporal_filter.c").read()
    assert "tf_gpu_do_filtering(cpi, frame_diff);" in patched and "tf_gpu_noise_levels(cpi, to_filter_buf, noise_levels);" in patched
    # every caller the seam covers (SURVEY 8f 1-3): submit/wait in av1_tf_info_filtering, context freed with the
    # TEMPORAL_FILTER_INFO, upload at lookahead push, the two other noise-estimate callers
    assert "tf_gpu_submit_filtering(cpi, gpu_diff[buf_idx]);" in patched and "tf_gpu_release(tf_info);" in patched
    assert "av1_tf_gpu_lookahead_push(cpi);" in open(tmp_path / "av1/encoder/encoder.c").read()
    assert "av1_tf_gpu_estimate_noise(cpi, sd, 0, 0," in open(tmp_path / "av1/encoder/encoder.c").read()
    assert "av1_tf_gpu_estimate_noise(" in open(tmp_path / "av1/encoder/encode_strategy.c").read()
    assert "struct tf_gpu_ctx *gpu;" in open(tmp_path / "av1/encoder/temporal_filter.h").read()
    assert "static tf_gpu_ctx *tf_gpu_instance" not in patched  # no process-wide context
