"""CPU tests of the update block's fp32-grade (bf16x3) tensor-core convolutions: the effimvs_conv2d_bf16x3* entry points
validate on the host, their shape support and packed size, the precision argument of the ops, and how net.py chooses the
kernel and caches its packed weights per precision (nothing is launched)."""
import ctypes

import pytest
import torch

import effimvs_b200  # noqa: F401
from effimvs_b200 import capi, hotpath, net, ops

# every (cin, cout) of the update block at hidden size h = 16 and h = 32: cd2 / zr (2h -> 2h), dprime (2h -> h), head1 (h -> h),
# q (2h -> h, two segments), mask0 (h -> 2h)
BLOCK_SHAPES = [(32, 32), (32, 16), (16, 16), (16, 32), (64, 64), (64, 32), (32, 32), (32, 64)]


def test_bf16x3_supported_and_packed_bytes():
    lib = capi.lib
    for cin, cout in BLOCK_SHAPES:
        assert lib.effimvs_conv2d_bf16x3_supported(cin, cout) == 1, (cin, cout)
        assert ops.conv2d_tc_supported(cin, cout, "bf16x3")
    for cin in (16, 32, 48, 64, 96):
        for cout in (4, 16, 20, 32, 64, 96):
            coutp = (cout + 15) // 16 * 16
            assert lib.effimvs_conv2d_bf16x3_packed_bytes(cin, cout) == 36 * cin * coutp
            assert lib.effimvs_conv2d_bf16x3_packed_bytes(cin, cout) == 2 * lib.effimvs_conv2d_tf32_packed_bytes(cin, cout)
    assert lib.effimvs_conv2d_bf16x3_packed_bytes(0, 16) == 0
    # the 1/8 stage (h = 48): 96 -> 96 needs 332 KB of weight images, more than shared memory holds
    assert lib.effimvs_conv2d_bf16x3_supported(96, 96) == 0
    assert lib.effimvs_conv2d_tf32_supported(96, 96) == 1
    for cin, cout in ((12, 16), (24, 16), (16, 6), (16, 132), (0, 16)):
        assert lib.effimvs_conv2d_bf16x3_supported(cin, cout) == 0, (cin, cout)


def test_bf16x3_entry_points_validate_on_the_host():
    lib, a, mode = capi.lib, ctypes.c_void_p(1 << 20), capi.CONV2D_BIAS
    P = ctypes.c_void_p
    f = lib.effimvs_conv2d_bf16x3
    assert f(None, 32, 32, None, 0, 0, a, None, 32, 1, 8, 8, mode, a, 32, None, 0, None, 0, None) == capi.EINVAL
    assert "null pointer" in capi.last_error() and "bf16x3" in capi.last_error()
    assert f(a, 32, 32, None, 0, 0, None, None, 32, 1, 8, 8, mode, a, 32, None, 0, None, 0, None) == capi.EINVAL   # no weights
    assert f(a, 32, 32, None, 0, 0, a, None, 32, 1, 1, 8, mode, a, 32, None, 0, None, 0, None) == capi.EINVAL      # H < 2
    assert f(a, 32, 12, None, 0, 0, a, None, 32, 1, 8, 8, mode, a, 32, None, 0, None, 0, None) == capi.EINVAL      # segment % 8
    assert f(a, 32, 24, None, 0, 0, a, None, 32, 1, 8, 8, mode, a, 32, None, 0, None, 0, None) == capi.EUNSUPPORTED  # cin % 16
    assert f(a, 96, 96, None, 0, 0, a, None, 96, 1, 8, 8, mode, a, 96, None, 0, None, 0, None) == capi.EUNSUPPORTED  # 96 -> 96
    assert "not supported" in capi.last_error()
    assert f(P((1 << 20) + 16), 32, 32, None, 0, 0, a, None, 32, 1, 8, 8, mode, a, 32, None, 0, None, 0, None) == capi.EINVAL
    assert "aligned" in capi.last_error()
    assert f(a, 32, 32, None, 0, 0, P((1 << 20) + 8), None, 32, 1, 8, 8, mode, a, 32, None, 0, None, 0, None) == capi.EINVAL
    assert f(a, 36, 32, None, 0, 0, a, None, 32, 1, 8, 8, mode, a, 32, None, 0, None, 0, None) == capi.EINVAL      # stride % 8
    assert f(a, 32, 32, None, 0, 0, a, None, 32, 1, 8, 8, 9, a, 32, None, 0, None, 0, None) == capi.EINVAL         # mode
    assert "bad mode" in capi.last_error()
    assert f(a, 32, 32, None, 0, 0, a, None, 32, 1, 8, 8, -1, a, 32, None, 0, None, 0, None) == capi.EINVAL
    assert f(a, 32, 32, None, 0, 0, a, None, 32, 1, 8, 8, capi.CONV2D_ADD_RELU, a, 32, None, 0, None, 0, None) == capi.EINVAL
    assert "addend" in capi.last_error()
    assert f(a, 32, 32, None, 0, 0, a, None, 32, 1, 8, 8, capi.CONV2D_GRU_GATES, a, 16, a, 16, None, 0, None) == capi.EINVAL
    assert f(a, 32, 32, None, 0, 0, a, None, 32, 1, 8, 8, capi.CONV2D_GRU_UPDATE, a, 32, None, 0, None, 0, None) == capi.EINVAL
    assert lib.effimvs_conv2d_bf16x3_pack(None, 16, 16, a, None) == capi.EINVAL
    assert lib.effimvs_conv2d_bf16x3_pack(a, 16, 16, None, None) == capi.EINVAL
    assert lib.effimvs_conv2d_bf16x3_pack(a, 12, 16, a, None) == capi.EUNSUPPORTED
    assert lib.effimvs_conv2d_bf16x3_pack(a, 96, 96, a, None) == capi.EUNSUPPORTED


def test_ops_precision_argument():
    assert ops.conv2d_tc_supported(96, 96) and not ops.conv2d_tc_supported(96, 96, "bf16x3")
    with pytest.raises(ValueError, match="precision"):
        ops.conv2d_tc_supported(16, 16, "fp8")
    with pytest.raises(RuntimeError):      # CPU tensors are rejected, not emulated
        ops.conv2d_tc(torch.zeros(1, 16, 4, 4), None, torch.zeros(10), None, 16, capi.CONV2D_BIAS, torch.zeros(1, 16, 4, 4),
                      None, None, "bf16x3")
    with torch.device("meta"):
        w = torch.empty(20, 32, 3, 3)
        assert torch.ops.effimvs.conv2d_tc_pack(w).numel() * 4 == capi.lib.effimvs_conv2d_tf32_packed_bytes(32, 20)
        assert torch.ops.effimvs.conv2d_tc_pack(w, "bf16x3").numel() * 4 == capi.lib.effimvs_conv2d_bf16x3_packed_bytes(32, 20)


def test_hotpath_binds_the_bf16x3_kernel():
    hp, hp3 = hotpath.CudaHotPath(), hotpath.CudaHotPath("bf16x3", conv2d_precision="bf16x3")
    assert hp.conv2d_precision == "f16" and not hp.conv2d_fp32_grade
    assert hp3.conv2d_precision == "bf16x3" and hp3.conv2d_fp32_grade
    assert hp.conv2d_tc_supported(96, 96) and not hp3.conv2d_tc_supported(96, 96)
    assert hp3.conv2d_tc_pack.keywords == {"precision": "bf16x3"} and hp3.conv2d_tc.keywords == {"precision": "bf16x3"}
    with pytest.raises(ValueError):
        hotpath.CudaHotPath(conv2d_precision="f16")


class _Glue:
    """stand-in for the glue table: the kernel accepts every shape but 96 -> 96 (as the bf16x3 kernel does)"""
    conv2d_precision = "f16"

    def __init__(self):
        self.packed = []

    def conv2d_tc(self, *args):
        raise AssertionError("not launched here")

    def conv2d_tc_supported(self, cin, cout):
        return not (cin == 96 and cout == 96)

    def conv2d_tc_pack(self, weight):
        self.packed.append(self.conv2d_precision)
        return (self.conv2d_precision, weight)


class _Glue3(_Glue):
    conv2d_precision = "bf16x3"
    conv2d_fp32_grade = True


@pytest.mark.parametrize("allow_tf32", [False, True])
def test_conv_tc_enabled_follows_precision(allow_tf32, monkeypatch):
    monkeypatch.delenv("EFFIMVS_CONV2D", raising=False)
    monkeypatch.delenv("EFFIMVS_CONV2D_MIN_PIXELS", raising=False)
    monkeypatch.setattr(torch.backends.cudnn, "allow_tf32", allow_tf32)
    for glue in (_Glue3(), hotpath.CudaHotPath(conv2d_precision="bf16x3")):
        assert net._conv_tc_enabled(glue, 16, 592, 800)           # DTU stage 3
        assert net._conv_tc_enabled(glue, 32, 296, 400)           # DTU stage 2
        assert not net._conv_tc_enabled(glue, 48, 148, 200)       # the 1/8 stage: 96 -> 96 unsupported, below 100k pixels
        assert not net._conv_tc_enabled(glue, 16, 148, 200)       # below the minimum pixel count
    for glue in (_Glue(), hotpath.CudaHotPath()):                 # the default glue: as before, only with allow_tf32
        assert net._conv_tc_enabled(glue, 16, 592, 800) == allow_tf32
        assert net._conv_tc_enabled(glue, 32, 296, 400) == allow_tf32
        assert not net._conv_tc_enabled(glue, 16, 148, 200)
    assert net._conv_tc_enabled(hotpath.CudaHotPath(), 48, 148, 200) is False
    monkeypatch.setenv("EFFIMVS_CONV2D", "0")
    assert not net._conv_tc_enabled(_Glue3(), 16, 592, 800)


def test_packed_weights_are_cached_per_precision():
    block = net.UpdateBlock(16, 6, 2, 4).eval()
    w = net._fused_update_weights(block)
    g, g3 = _Glue(), _Glue3()
    tc = net._tc_update_weights(block, g, w)
    tc3 = net._tc_update_weights(block, g3, w)
    assert all(v[0] == "f16" for k, v in tc.items() if k != "b_zr")
    assert all(v[0] == "bf16x3" for k, v in tc3.items() if k != "b_zr")
    # each precision packs once; alternating reuses its own images
    assert net._tc_update_weights(block, g, w) is tc and net._tc_update_weights(block, g3, w) is tc3
    assert g.packed == ["f16"] * 6 and g3.packed == ["bf16x3"] * 6
