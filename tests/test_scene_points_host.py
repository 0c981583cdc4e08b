"""CPU tests of the scene's coloured point cloud (csrc/points.cu, fusion.compact_points, run_scene(images=)): malformed input
is rejected before any launch, the C-ABI validates its arguments, the fake implementations give the shapes, and the colour
rule restated in NumPy (`color_rule`, the reference of tests/test_gpu_scene_points.py) is NumPy's cast on [0,1] and returns
every byte of a u8 / 255 image."""
import ctypes

import numpy as np
import pytest
import torch

import effimvs_b200  # noqa: F401
from effimvs_b200 import capi, fusion, scene


def color_rule(x):
    """the library's colour byte: trunc(clamp(x * 255, 0, 255)), the product an IEEE float32 multiply, NaN giving 0"""
    p = np.asarray(x, dtype=np.float32) * np.float32(255)
    with np.errstate(invalid="ignore"):
        return np.trunc(np.clip(np.nan_to_num(p, nan=0.0, posinf=255.0, neginf=0.0), 0, 255)).astype(np.uint8)


def test_color_rule_is_numpys_cast_on_the_unit_interval():
    rng = np.random.default_rng(0)
    x = np.concatenate([np.linspace(0, 1, 1 << 20, dtype=np.float32), rng.random(1 << 20, dtype=np.float32),
                        np.float32([0, 1, np.nextafter(np.float32(1), np.float32(0))])])
    k = np.arange(256, dtype=np.float32) / np.float32(255)            # k/255 and its float32 neighbours
    x = np.concatenate([x, k, np.nextafter(k, np.float32(0)), np.clip(np.nextafter(k, np.float32(2)), 0, 1)])
    assert np.array_equal(color_rule(x), (x * 255).astype(np.uint8))


def test_color_rule_returns_every_byte_of_a_u8_image():
    u8 = np.arange(256, dtype=np.uint8)
    assert np.array_equal(color_rule(u8.astype(np.float32) / np.float32(255)), u8)


def test_color_rule_outside_the_unit_interval():
    x = np.float32([-1e30, -1, -1e-30, 1 + 1e-7, 2, 1e30, np.inf, -np.inf, np.nan])
    assert color_rule(x).tolist() == [0, 0, 0, 255, 255, 255, 255, 0, 0]


def _inputs(n=2, h=6, w=8, n_images=3):
    return torch.zeros(n, 1, h, w, dtype=torch.bool), torch.zeros(n, 3, h, w), torch.zeros(n_images, 3, h, w)


@pytest.mark.parametrize("case", ["mask_points_n", "mask_points_hw", "views_count", "images_hw", "images_channels", "image_row",
                                  "negative_row", "no_views"])
def test_compact_points_rejects_malformed_input(case):
    final, pts, imgs = _inputs()
    views = [0, 2]
    if case == "mask_points_n":
        pts = torch.zeros(3, 3, 6, 8)
    elif case == "mask_points_hw":
        pts = torch.zeros(2, 3, 6, 9)
    elif case == "views_count":
        views = [0]
    elif case == "images_hw":
        imgs = torch.zeros(3, 3, 8, 6)
    elif case == "images_channels":
        imgs = torch.zeros(3, 1, 6, 8)
    elif case == "image_row":
        views = [0, 3]
    elif case == "negative_row":
        views = [-1, 0]
    elif case == "no_views":
        final, pts, views = final[:0], pts[:0], []
    with pytest.raises(ValueError):
        fusion.compact_points(final, pts, views, imgs)


def test_compact_points_rejects_cpu_tensors():
    final, pts, imgs = _inputs()
    with pytest.raises(RuntimeError, match="CUDA-only"):
        fusion.compact_points(final, pts, [0, 1])
    with pytest.raises(RuntimeError, match="CUDA-only"):
        fusion.compact_points(final, pts, [0, 1], imgs)


def _never(*args):
    raise AssertionError("run_scene called infer / fuse before rejecting its images")


@pytest.mark.parametrize("shape", [(4, 3, 6, 8), (5, 1, 6, 8), (5, 3, 6)])
def test_run_scene_rejects_malformed_images_before_inference(shape):
    with pytest.raises(ValueError, match="images"):
        scene.run_scene(_never, _never, 5, [[1]] * 5, device="cpu", images=torch.zeros(shape))


def test_run_scene_rejects_cpu_images_before_inference():
    with pytest.raises(RuntimeError, match="CUDA-only"):
        scene.run_scene(_never, _never, 5, [[1]] * 5, device="cpu", images=torch.zeros(5, 3, 6, 8))


def test_c_abi_rejects_bad_arguments():
    lib = capi.lib
    P = ctypes.c_void_p
    a = P(1 << 20)                                          # 16-byte aligned dummy address; every call fails before a launch
    need = lib.effimvs_point_offsets_workspace_bytes(49, 1184, 1600)
    assert need == 49 * ((1184 * 1600 + 4095) // 4096) * 8
    assert lib.effimvs_point_offsets_workspace_bytes(1, 1, 1) == 8
    assert lib.effimvs_point_offsets_workspace_bytes(0, 8, 8) == 0 and lib.effimvs_point_offsets_workspace_bytes(1, -1, 8) == 0
    assert lib.effimvs_point_offsets(None, 1, 8, 8, a, 8, a, None) == capi.EINVAL
    assert "null pointer" in capi.last_error()
    assert lib.effimvs_point_offsets(a, 1, 8, 8, None, 8, a, None) == capi.EINVAL
    assert lib.effimvs_point_offsets(a, 1, 8, 8, a, 8, None, None) == capi.EINVAL
    assert lib.effimvs_point_offsets(a, 0, 8, 8, a, 8, a, None) == capi.EINVAL
    assert lib.effimvs_point_offsets(a, 1, 0, 8, a, 8, a, None) == capi.EINVAL
    assert lib.effimvs_point_offsets(a, 1, 8, 8, P((1 << 20) + 8), 8, a, None) == capi.EINVAL
    assert lib.effimvs_point_offsets(a, 2, 64, 128, a, 8, a, None) == capi.EWORKSPACE
    gather = lib.effimvs_gather_points_f32
    assert gather(None, a, None, 0, None, 1, 8, 8, a, 8, a, None, None) == capi.EINVAL
    assert gather(a, None, None, 0, None, 1, 8, 8, a, 8, a, None, None) == capi.EINVAL
    assert gather(a, a, None, 0, None, 1, 8, 8, None, 8, a, None, None) == capi.EINVAL
    assert gather(a, a, None, 0, None, 1, 8, 8, a, 8, None, None, None) == capi.EINVAL
    assert gather(a, a, a, 4, None, 1, 8, 8, a, 8, a, a, None) == capi.EINVAL              # images without rows
    assert gather(a, a, a, 4, a, 1, 8, 8, a, 8, a, None, None) == capi.EINVAL              # images without colours out
    assert gather(a, a, a, 0, a, 1, 8, 8, a, 8, a, a, None) == capi.EINVAL                 # no image rows to read
    assert gather(a, a, None, 0, None, 1, 8, -8, a, 8, a, None, None) == capi.EINVAL
    assert gather(a, a, None, 0, None, 1, 8, 8, a, 8, P((1 << 20) + 4), None, None) == capi.EINVAL
    assert "16-byte aligned" in capi.last_error()
    assert gather(a, a, a, 4, a, 1, 8, 8, a, 8, a, P((1 << 20) + 3), None) == capi.EINVAL
    assert gather(a, a, None, 0, None, 3, 64, 128, a, 16, a, None, None) == capi.EWORKSPACE


def test_fake_implementations_give_shapes_without_a_device():
    with torch.device("meta"):
        final = torch.empty(3, 37, 53, dtype=torch.uint8)
        offsets, ws = torch.ops.effimvs.point_offsets(final)
        assert offsets.shape == (4,) and offsets.dtype == torch.int64
        assert ws.shape == (3 * 8,) and ws.dtype == torch.uint8
        pts, cols = torch.ops.effimvs.gather_points(final, torch.empty(3, 3, 37, 53), torch.empty(5, 3, 37, 53),
                                                    torch.empty(3, dtype=torch.int32), ws, 1000)
        assert pts.shape == (1000, 3) and pts.dtype == torch.float32
        assert cols.shape == (1000, 3) and cols.dtype == torch.uint8
        pts, cols = torch.ops.effimvs.gather_points(final, torch.empty(3, 3, 37, 53), None, None, ws, 7)
        assert pts.shape == (7, 3) and cols.shape == (0, 3)
