"""``torch.library`` custom ops ``effimvs::*`` over the C-ABI (device pointers only).

PyTorch is plumbing here: it owns the device buffers and the stream; every op forwards raw
pointers to libeffimvs.so.  Inference only (no autograd formula).  CPU tensors are rejected --
there is no fallback.
"""
from __future__ import annotations

import os
from typing import List, Optional, Tuple

import torch
from torch import Tensor

from . import capi

_lib = capi.lib
_NHWC_MAXC = int(os.environ.get("EFFIMVS_NHWC_MAXC", "32"))

# kernels of libeffimvs.so launched through this module since the caller last reset it (bench.py's
# `gpu_launches`); every op adds the number of launches its C entry point enqueues.
LAUNCHES = 0


def _count(n: int) -> None:
    global LAUNCHES
    LAUNCHES += n


def _dev(t: Tensor, name: str) -> Tensor:
    if not t.is_cuda:
        raise RuntimeError("effimvs::{} got a CPU tensor; the hot path is CUDA-only (no fallback)".format(name))
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous()


def _features(ref: Tensor, srcs: List[Tensor], name: str):
    """Feature maps as the kernels read them: all NCHW-contiguous or all channels-last (NHWC).
    Channels-last maps (what the channels_last FPN emits) are passed through without a copy."""
    for t in [ref] + list(srcs):
        if not t.is_cuda:
            raise RuntimeError("effimvs::{} got a CPU tensor; the hot path is CUDA-only (no fallback)".format(name))
    # channels-last maps go to the tiled kernel (csrc/warp_tile.cu: TMA-staged source tiles, any C in {8,16,32});
    # EFFIMVS_NHWC_MAXC caps the channel count that takes that path (wider maps are converted to planar once)
    nhwc = (ref.dim() == 4 and 1 < ref.shape[1] <= _NHWC_MAXC and not ref.is_contiguous()
            and ref.is_contiguous(memory_format=torch.channels_last))
    fmt = torch.channels_last if nhwc else torch.contiguous_format
    fix = lambda t: (t if t.dtype == torch.float32 else t.float()).contiguous(memory_format=fmt)   # noqa: E731
    return fix(ref), [fix(s) for s in srcs], (capi.FEA_NHWC if nhwc else capi.FEA_NCHW)


def _stream() -> int:
    # inside _on_tensor_device the current device is the tensors' device, so this is THEIR current stream
    return torch.cuda.current_stream().cuda_stream


def _on_tensor_device(fn):
    """Run an op body with the CUDA device of its tensor arguments current (so that the launch, the stream handed
    to the library and the output allocations all belong to that device, whatever torch's current device is), and
    reject tensors spread over several CUDA devices.  CPU tensors pass through: the body reports them by name."""
    import functools

    def tensors(args):
        for a in args:
            if isinstance(a, Tensor):
                yield a
            elif isinstance(a, (list, tuple)):
                for b in a:
                    if isinstance(b, Tensor):
                        yield b

    @functools.wraps(fn)
    def call(*args, **kw):
        devs = {t.device for t in tensors(list(args) + list(kw.values())) if t.is_cuda}
        if len(devs) > 1:
            raise RuntimeError("effimvs::{} got tensors on several devices: {}".format(fn.__name__, sorted(map(str, devs))))
        if not devs or next(iter(devs)).index == torch.cuda.current_device():
            return fn(*args, **kw)
        with torch.cuda.device(next(iter(devs))):
            return fn(*args, **kw)
    return call


def _opt(t: Optional[Tensor]):
    return t.data_ptr() if t is not None else None


# -------------------------------------------------------------------------------------------
@torch.library.custom_op("effimvs::relative_projection", mutates_args=())
@_on_tensor_device
def relative_projection(cams: Tensor) -> Tensor:
    cams = _dev(cams, "relative_projection")
    B, V = cams.shape[0], cams.shape[1]
    out = torch.empty(B, V - 1, 12, device=cams.device, dtype=torch.float32)
    _count(1)
    capi.check(_lib.effimvs_relative_projection_f32(cams.data_ptr(), B, V, out.data_ptr(), _stream()))
    return out


@relative_projection.register_fake
def _(cams):
    return cams.new_empty(cams.shape[0], cams.shape[1] - 1, 12)


# -------------------------------------------------------------------------------------------
@torch.library.custom_op("effimvs::homo_warp", mutates_args=())
@_on_tensor_device
def homo_warp(src_fea: Tensor, proj: Tensor, hyp: Tensor, hyp_mode: int, D: int) -> Tensor:
    src_fea, proj, hyp = _dev(src_fea, "homo_warp"), _dev(proj, "homo_warp"), _dev(hyp, "homo_warp")
    B, Cc, H, W = src_fea.shape
    out = torch.empty(B, Cc, D, H, W, device=src_fea.device, dtype=torch.float32)
    _count(1)
    capi.check(_lib.effimvs_homo_warp_f32(src_fea.data_ptr(), proj.data_ptr(), hyp.data_ptr(), hyp_mode, B, Cc, H, W, D,
                                          out.data_ptr(), _stream()))
    return out


@homo_warp.register_fake
def _(src_fea, proj, hyp, hyp_mode, D):
    B, Cc, H, W = src_fea.shape
    return src_fea.new_empty(B, Cc, D, H, W)


@torch.library.custom_op("effimvs::depth_ranges", mutates_args=())
@_on_tensor_device
def depth_ranges(depth_values: Tensor, ndepth1: int, ratios: List[float]) -> Tensor:
    """depth_values (B,Dv) -> a flat buffer of 8 B + B ndepth1 floats: 8 rows of B scalars [depth_far, depth_near, lo_disp, hi_disp,
    interval_1, interval_2, interval_3, 0] followed by the (B, ndepth1) plane-sweep hypotheses -- everything Effi_MVS_plus.forward
    derives from depth_values alone (Effi_MVS_plus.py:409-424, module.py:577-585), bit-identical to the torch expressions, in one launch."""
    import ctypes
    depth_values = _dev(depth_values, "depth_ranges")
    B, Dv = depth_values.shape
    if len(ratios) != 3:
        raise ValueError("depth_ranges: three interval ratios expected")
    out = torch.empty(B * (8 + ndepth1), device=depth_values.device, dtype=torch.float32)
    r3 = (ctypes.c_float * 3)(*[float(r) for r in ratios])
    _count(1)
    capi.check(_lib.effimvs_depth_ranges_f32(depth_values.data_ptr(), B, Dv, ndepth1, r3, out.data_ptr(), _stream()))
    return out


@depth_ranges.register_fake
def _(depth_values, ndepth1, ratios):
    return depth_values.new_empty(depth_values.shape[0] * (8 + ndepth1))


@torch.library.custom_op("effimvs::depth_range_samples", mutates_args=())
@_on_tensor_device
def depth_range_samples(cur: Tensor, interval: Tensor, ndepth: int) -> Tensor:
    cur, interval = _dev(cur, "depth_range_samples"), _dev(interval, "depth_range_samples")
    B, H, W = cur.shape
    out = torch.empty(B, ndepth, H, W, device=cur.device, dtype=torch.float32)
    _count(1)
    capi.check(_lib.effimvs_depth_range_samples_f32(cur.data_ptr(), interval.data_ptr(), B, ndepth, H, W, out.data_ptr(), _stream()))
    return out


@depth_range_samples.register_fake
def _(cur, interval, ndepth):
    B, H, W = cur.shape
    return cur.new_empty(B, ndepth, H, W)


@torch.library.custom_op("effimvs::fusion_masks", mutates_args=())
@_on_tensor_device
def fusion_masks(ref_depth: Tensor, reproj_xyd: Tensor, dist_base: float, rel_diff_base: float, thres_view: int,
                 relative: bool) -> Tensor:
    ref_depth, reproj_xyd = _dev(ref_depth, "fusion_masks"), _dev(reproj_xyd, "fusion_masks")
    n, v, _, h, w = reproj_xyd.shape
    K = v - thres_view + 1
    out = torch.empty(n, v, K, h, w, device=ref_depth.device, dtype=torch.uint8)
    _count(1)
    capi.check(_lib.effimvs_fusion_masks_f32(ref_depth.data_ptr(), reproj_xyd.data_ptr(), n, v, h, w, dist_base, rel_diff_base,
                                             thres_view, int(relative), out.data_ptr(), _stream()))
    return out


@fusion_masks.register_fake
def _(ref_depth, reproj_xyd, dist_base, rel_diff_base, thres_view, relative):
    n, v, _, h, w = reproj_xyd.shape
    return ref_depth.new_empty(n, v, v - thres_view + 1, h, w, dtype=torch.uint8)


# -------------------------------------------------------------------------------------------
@torch.library.custom_op("effimvs::warp_corr_agg", mutates_args=())
@_on_tensor_device
def warp_corr_agg(ref: Tensor, srcs: List[Tensor], proj: Tensor, hyp: Tensor, hyp_mode: int,
                  interval: Optional[Tensor], weights: Optional[Tensor], D: int, G: int,
                  want_hyp: bool) -> Tuple[Tensor, Tensor]:
    ref, srcs, layout = _features(ref, srcs, "warp_corr_agg")
    proj, hyp = _dev(proj, "warp_corr_agg"), _dev(hyp, "warp_corr_agg")
    interval = _dev(interval, "warp_corr_agg") if interval is not None else None
    weights = _dev(weights, "warp_corr_agg") if weights is not None else None
    B, Cc, H, W = ref.shape
    sim = torch.empty(B, G, D, H, W, device=ref.device, dtype=torch.float32)
    hyp_out = torch.empty(B, D, H, W, device=ref.device, dtype=torch.float32) if want_hyp else ref.new_empty(0)
    arr, keep = capi.ptr_array([s.data_ptr() for s in srcs])
    _count(1)
    capi.check(_lib.effimvs_warp_corr_agg_f32(ref.data_ptr(), arr, len(srcs), proj.data_ptr(), hyp.data_ptr(), hyp_mode,
                                              _opt(interval), _opt(weights), B, Cc, H, W, D, G, layout, sim.data_ptr(),
                                              hyp_out.data_ptr() if want_hyp else None, _stream()))
    del keep
    return sim, hyp_out


@warp_corr_agg.register_fake
def _(ref, srcs, proj, hyp, hyp_mode, interval, weights, D, G, want_hyp):
    B, _, H, W = ref.shape
    return ref.new_empty(B, G, D, H, W), (ref.new_empty(B, D, H, W) if want_hyp else ref.new_empty(0))


@torch.library.custom_op("effimvs::warp_corr_views", mutates_args=())
@_on_tensor_device
def warp_corr_views(ref: Tensor, srcs: List[Tensor], proj: Tensor, hyp: Tensor, hyp_mode: int, D: int) -> Tuple[Tensor, Tensor]:
    ref, srcs, layout = _features(ref, srcs, "warp_corr_views")
    proj, hyp = _dev(proj, "warp_corr_views"), _dev(hyp, "warp_corr_views")
    B, Cc, H, W = ref.shape
    n = len(srcs)
    sims = torch.empty(B, n, D, H, W, device=ref.device, dtype=torch.float32)
    ent = torch.empty(B, n, H, W, device=ref.device, dtype=torch.float32)
    arr, keep = capi.ptr_array([s.data_ptr() for s in srcs])
    _count(1)
    capi.check(_lib.effimvs_warp_corr_views_f32(ref.data_ptr(), arr, n, proj.data_ptr(), hyp.data_ptr(), hyp_mode,
                                                B, Cc, H, W, D, layout, sims.data_ptr(), ent.data_ptr(), _stream()))
    del keep
    return sims, ent


@warp_corr_views.register_fake
def _(ref, srcs, proj, hyp, hyp_mode, D):
    B, _, H, W = ref.shape
    return ref.new_empty(B, len(srcs), D, H, W), ref.new_empty(B, len(srcs), H, W)


@torch.library.custom_op("effimvs::weighted_agg", mutates_args=())
@_on_tensor_device
def weighted_agg(sims: Tensor, weights: Tensor) -> Tensor:
    sims, weights = _dev(sims, "weighted_agg"), _dev(weights, "weighted_agg")
    B, n, D, H, W = sims.shape
    out = torch.empty(B, D, H, W, device=sims.device, dtype=torch.float32)
    _count(1)
    capi.check(_lib.effimvs_weighted_agg_f32(sims.data_ptr(), weights.data_ptr(), B, n, D, H, W, out.data_ptr(), _stream()))
    return out


@weighted_agg.register_fake
def _(sims, weights):
    B, n, D, H, W = sims.shape
    return sims.new_empty(B, D, H, W)


# -------------------------------------------------------------------------------------------
def _range_mode(dmin: Tensor, B: int, H: int, W: int) -> int:
    if dmin.numel() == B:
        return capi.RANGE_SCALAR
    if dmin.numel() == B * H * W:
        return capi.RANGE_PIXEL
    raise ValueError("depth range must have B or B*H*W elements, got {}".format(tuple(dmin.shape)))


@torch.library.custom_op("effimvs::volume_lookup", mutates_args=())
@_on_tensor_device
def volume_lookup(volume: Tensor, depth_sample: Tensor, depth_min: Tensor, depth_max: Tensor, sample_stride: int) -> Tensor:
    volume, depth_sample = _dev(volume, "volume_lookup"), _dev(depth_sample, "volume_lookup")
    depth_min, depth_max = _dev(depth_min, "volume_lookup"), _dev(depth_max, "volume_lookup")
    B, D, H, W = volume.shape
    d = depth_sample.shape[1]
    if tuple(depth_sample.shape[2:]) != (H * sample_stride, W * sample_stride):
        raise ValueError("depth_sample {} does not match volume {} with stride {}".format(tuple(depth_sample.shape), tuple(volume.shape), sample_stride))
    mode = _range_mode(depth_min, B, H, W)
    if _range_mode(depth_max, B, H, W) != mode:
        raise ValueError("depth_min and depth_max must have the same shape")
    out = torch.empty(B, d, H, W, device=volume.device, dtype=torch.float32)
    _count(1)
    capi.check(_lib.effimvs_volume_lookup_f32(volume.data_ptr(), depth_sample.data_ptr(), depth_min.data_ptr(),
                                              depth_max.data_ptr(), mode, sample_stride, B, D, d, H, W, out.data_ptr(), _stream()))
    return out


@volume_lookup.register_fake
def _(volume, depth_sample, depth_min, depth_max, sample_stride):
    B, D, H, W = volume.shape
    return volume.new_empty(B, depth_sample.shape[1], H, W)


@torch.library.custom_op("effimvs::dynamic_cost", mutates_args=())
@_on_tensor_device
def dynamic_cost(cur_depth: Tensor, raw: Tensor, reg: Tensor, interval: Tensor, depth_min: Tensor, depth_max: Tensor,
                 ndepth: int) -> Tensor:
    cur_depth, raw, reg = _dev(cur_depth, "dynamic_cost"), _dev(raw, "dynamic_cost"), _dev(reg, "dynamic_cost")
    interval, depth_min, depth_max = _dev(interval, "dynamic_cost"), _dev(depth_min, "dynamic_cost"), _dev(depth_max, "dynamic_cost")
    B, D, H, W = raw.shape
    if reg.shape != raw.shape or cur_depth.numel() != B * H * W or interval.numel() != B:
        raise ValueError("dynamic_cost: inconsistent shapes")
    mode = _range_mode(depth_min, B, H, W)
    if _range_mode(depth_max, B, H, W) != mode:
        raise ValueError("depth_min and depth_max must have the same shape")
    out = torch.empty(B, 2 * ndepth, H, W, device=raw.device, dtype=torch.float32)
    _count(1)
    capi.check(_lib.effimvs_dynamic_cost_f32(cur_depth.data_ptr(), raw.data_ptr(), reg.data_ptr(), interval.data_ptr(),
                                             depth_min.data_ptr(), depth_max.data_ptr(), mode, ndepth, B, D, H, W,
                                             out.data_ptr(), _stream()))
    return out


@dynamic_cost.register_fake
def _(cur_depth, raw, reg, interval, depth_min, depth_max, ndepth):
    B, D, H, W = raw.shape
    return raw.new_empty(B, 2 * ndepth, H, W)


@torch.library.custom_op("effimvs::softmax_regress_conf", mutates_args=())
@_on_tensor_device
def softmax_regress_conf(prob_pre: Tensor, hyp: Tensor, hyp_mode: int) -> Tuple[Tensor, Tensor]:
    prob_pre, hyp = _dev(prob_pre, "softmax_regress_conf"), _dev(hyp, "softmax_regress_conf")
    B, D, H, W = prob_pre.shape
    depth = torch.empty(B, H, W, device=prob_pre.device, dtype=torch.float32)
    conf = torch.empty(B, H, W, device=prob_pre.device, dtype=torch.float32)
    _count(1)
    capi.check(_lib.effimvs_softmax_regress_conf_f32(prob_pre.data_ptr(), hyp.data_ptr(), hyp_mode, B, D, H, W,
                                                     depth.data_ptr(), conf.data_ptr(), _stream()))
    return depth, conf


@softmax_regress_conf.register_fake
def _(prob_pre, hyp, hyp_mode):
    B, D, H, W = prob_pre.shape
    return prob_pre.new_empty(B, H, W), prob_pre.new_empty(B, H, W)


# -------------------------------------------------------------------------------------------
@torch.library.custom_op("effimvs::conv3d", mutates_args=())
@_on_tensor_device
def conv3d(x: Tensor, weight: Tensor, bias: Optional[Tensor], residual: Optional[Tensor], stride: List[int],
           transposed: bool, relu: bool) -> Tensor:
    x, weight = _dev(x, "conv3d"), _dev(weight, "conv3d")
    bias = _dev(bias, "conv3d") if bias is not None else None
    residual = _dev(residual, "conv3d") if residual is not None else None
    B, Cin, D, H, W = x.shape
    Cout = weight.shape[1] if transposed else weight.shape[0]
    sd, sh, sw = stride
    if transposed:
        Do, Ho, Wo = D * sd, H * sh, W * sw
    else:
        Do, Ho, Wo = (D - 1) // sd + 1, (H - 1) // sh + 1, (W - 1) // sw + 1
    y = torch.empty(B, Cout, Do, Ho, Wo, device=x.device, dtype=torch.float32)
    _count(1)
    capi.check(_lib.effimvs_conv3d_f32(x.data_ptr(), weight.data_ptr(), _opt(bias), _opt(residual), B, Cin, Cout, D, H, W,
                                       sd, sh, sw, int(transposed), int(relu), y.data_ptr(), 0, Cout, _stream()))
    return y


@conv3d.register_fake
def _(x, weight, bias, residual, stride, transposed, relu):
    B, Cin, D, H, W = x.shape
    Cout = weight.shape[1] if transposed else weight.shape[0]
    sd, sh, sw = stride
    if transposed:
        return x.new_empty(B, Cout, D * sd, H * sh, W * sw)
    return x.new_empty(B, Cout, (D - 1) // sd + 1, (H - 1) // sh + 1, (W - 1) // sw + 1)


@torch.library.custom_op("effimvs::conv3d_bf16", mutates_args=())
@_on_tensor_device
def conv3d_bf16(x: Tensor, weight: Tensor, bias: Optional[Tensor], residual: Optional[Tensor], sd: int,
                transposed: bool, relu: bool, precision: int) -> Tensor:
    """One (de)conv layer on the tensor cores (tcgen05), fp32 NCDHW in/out.  Conv: stride sd in all
    dims (1 or 2); transposed conv: stride (sd,2,2)."""
    x, weight = _dev(x, "conv3d_bf16"), _dev(weight, "conv3d_bf16")
    bias = _dev(bias, "conv3d_bf16") if bias is not None else None
    residual = _dev(residual, "conv3d_bf16") if residual is not None else None
    B, Cin, D, H, W = x.shape
    Cout = weight.shape[1] if transposed else weight.shape[0]
    if transposed:
        Do, Ho, Wo = D * sd, H * 2, W * 2
    else:
        Do, Ho, Wo = D // sd, H // sd, W // sd
    need = _lib.effimvs_conv3d_bf16_workspace_bytes(B, Cin, Cout, D, H, W, sd, int(transposed), precision)
    ws = torch.empty(max(need, 256), device=x.device, dtype=torch.uint8)
    y = torch.empty(B, Cout, Do, Ho, Wo, device=x.device, dtype=torch.float32)
    _count(5)
    capi.check(_lib.effimvs_conv3d_bf16(x.data_ptr(), weight.data_ptr(), _opt(bias), _opt(residual), B, Cin, Cout, D, H, W,
                                        sd, int(transposed), int(relu), precision, ws.data_ptr(), ws.numel(), y.data_ptr(), _stream()))
    return y


@conv3d_bf16.register_fake
def _(x, weight, bias, residual, sd, transposed, relu, precision):
    B, Cin, D, H, W = x.shape
    Cout = weight.shape[1] if transposed else weight.shape[0]
    if transposed:
        return x.new_empty(B, Cout, D * sd, H * 2, W * 2)
    return x.new_empty(B, Cout, D // sd, H // sd, W // sd)


@torch.library.custom_op("effimvs::costreg_fpn3d", mutates_args=())
@_on_tensor_device
def costreg_fpn3d(x: Tensor, weights: List[Tensor], biases: List[Tensor], precision: int) -> Tensor:
    x = _dev(x, "costreg_fpn3d")
    weights = [_dev(w, "costreg_fpn3d") for w in weights]
    biases = [_dev(b, "costreg_fpn3d") for b in biases]
    if len(weights) != 9 or len(biases) != 8:
        raise ValueError("costreg_fpn3d wants 9 weights and 8 biases")
    B, _, D, H, W = x.shape
    need = _lib.effimvs_costreg_workspace_bytes(B, D, H, W, precision)
    ws = torch.empty(max(need, 256), device=x.device, dtype=torch.uint8)
    out = torch.empty(B, 1, D, H, W, device=x.device, dtype=torch.float32)
    wa, k1 = capi.ptr_array([w.data_ptr() for w in weights])
    ba, k2 = capi.ptr_array([b.data_ptr() for b in biases])
    _count(9 if precision == capi.PREC_F32 else 11)   # tensor-core modes: halo zeroing + weight pack + 1 CUDA-core conv + 8 tcgen05 layers
    capi.check(_lib.effimvs_costreg_fpn3d(x.data_ptr(), wa, ba, B, D, H, W, precision, ws.data_ptr(), ws.numel(),
                                          out.data_ptr(), _stream()))
    del k1, k2
    return out


@costreg_fpn3d.register_fake
def _(x, weights, biases, precision):
    return x.new_empty(x.shape)


@torch.library.custom_op("effimvs::cost_up_small", mutates_args=())
@_on_tensor_device
def cost_up_small(x: Tensor, prev: Tensor, weights: List[Tensor], biases: List[Tensor], precision: int) -> Tensor:
    x, prev = _dev(x, "cost_up_small"), _dev(prev, "cost_up_small")
    weights = [_dev(w, "cost_up_small") for w in weights]
    biases = [_dev(b, "cost_up_small") for b in biases]
    if len(weights) != 4 or len(biases) != 4:
        raise ValueError("cost_up_small wants 4 weights and 4 biases")
    B, _, D, H, W = x.shape
    if tuple(prev.shape) != (B, 1, D, H // 2, W // 2):
        raise ValueError("cost_up_small: prev {} does not match x {}".format(tuple(prev.shape), tuple(x.shape)))
    need = _lib.effimvs_cost_up_workspace_bytes(B, D, H, W, precision)
    ws = torch.empty(max(need, 256), device=x.device, dtype=torch.uint8)
    out = torch.empty(B, 1, D, H, W, device=x.device, dtype=torch.float32)
    wa, k1 = capi.ptr_array([w.data_ptr() for w in weights])
    ba, k2 = capi.ptr_array([b.data_ptr() for b in biases])
    _count(4 if precision == capi.PREC_F32 else 6)    # tensor-core modes: halo zeroing + weight pack + 2 CUDA-core convs + 2 tcgen05 layers
    capi.check(_lib.effimvs_cost_up_small(x.data_ptr(), prev.data_ptr(), wa, ba, B, D, H, W, precision, ws.data_ptr(),
                                          ws.numel(), out.data_ptr(), _stream()))
    del k1, k2
    return out


@cost_up_small.register_fake
def _(x, prev, weights, biases, precision):
    return x.new_empty(x.shape)


# ---- the same two networks against a caller-kept workspace (effimvs_*_ex: PREPARE once per weights and shape, then RUN) ----
def costreg_workspace_bytes(B: int, D: int, H: int, W: int, precision: int) -> int:
    return int(_lib.effimvs_costreg_workspace_bytes(B, D, H, W, precision))


def cost_up_workspace_bytes(B: int, D: int, H: int, W: int, precision: int) -> int:
    return int(_lib.effimvs_cost_up_workspace_bytes(B, D, H, W, precision))


def _wsbuf(ws: Tensor, what: str) -> Tensor:
    if not ws.is_cuda or ws.dtype != torch.uint8 or not ws.is_contiguous():
        raise RuntimeError("effimvs::{}: the workspace must be a contiguous CUDA uint8 tensor".format(what))
    return ws


def _reg_args(weights, biases, nw, nb, what):
    weights = [_dev(w, what) for w in weights]
    biases = [_dev(b, what) for b in biases]
    if len(weights) != nw or len(biases) != nb:
        raise ValueError("{} wants {} weights and {} biases".format(what, nw, nb))
    return capi.ptr_array([w.data_ptr() for w in weights]), capi.ptr_array([b.data_ptr() for b in biases])


@torch.library.custom_op("effimvs::costreg_prepare", mutates_args=("ws",))
@_on_tensor_device
def costreg_prepare(weights: List[Tensor], biases: List[Tensor], B: int, D: int, H: int, W: int, precision: int, ws: Tensor) -> None:
    (wa, k1), (ba, k2) = _reg_args(weights, biases, 9, 8, "costreg_prepare")
    ws = _wsbuf(ws, "costreg_prepare")
    _count(0 if precision == capi.PREC_F32 else 2)
    capi.check(_lib.effimvs_costreg_fpn3d_ex(None, wa, ba, B, D, H, W, precision, capi.WS_PREPARE, ws.data_ptr(), ws.numel(),
                                             None, _stream()))
    del k1, k2


@torch.library.custom_op("effimvs::costreg_run", mutates_args=("ws",))
@_on_tensor_device
def costreg_run(x: Tensor, weights: List[Tensor], biases: List[Tensor], precision: int, ws: Tensor) -> Tensor:
    """costreg_fpn3d on a workspace prepared by costreg_prepare for these weights and this shape."""
    x, ws = _dev(x, "costreg_run"), _wsbuf(ws, "costreg_run")
    (wa, k1), (ba, k2) = _reg_args(weights, biases, 9, 8, "costreg_run")
    B, _, D, H, W = x.shape
    out = torch.empty(B, 1, D, H, W, device=x.device, dtype=torch.float32)
    _count(9)
    capi.check(_lib.effimvs_costreg_fpn3d_ex(x.data_ptr(), wa, ba, B, D, H, W, precision, capi.WS_RUN, ws.data_ptr(), ws.numel(),
                                             out.data_ptr(), _stream()))
    del k1, k2
    return out


@costreg_run.register_fake
def _(x, weights, biases, precision, ws):
    return x.new_empty(x.shape)


@torch.library.custom_op("effimvs::cost_up_prepare", mutates_args=("ws",))
@_on_tensor_device
def cost_up_prepare(weights: List[Tensor], biases: List[Tensor], B: int, D: int, H: int, W: int, precision: int, ws: Tensor) -> None:
    (wa, k1), (ba, k2) = _reg_args(weights, biases, 4, 4, "cost_up_prepare")
    ws = _wsbuf(ws, "cost_up_prepare")
    _count(0 if precision == capi.PREC_F32 else 2)
    capi.check(_lib.effimvs_cost_up_small_ex(None, None, wa, ba, B, D, H, W, precision, capi.WS_PREPARE, ws.data_ptr(), ws.numel(),
                                             None, _stream()))
    del k1, k2


@torch.library.custom_op("effimvs::cost_up_run", mutates_args=("ws",))
@_on_tensor_device
def cost_up_run(x: Tensor, prev: Tensor, weights: List[Tensor], biases: List[Tensor], precision: int, ws: Tensor) -> Tensor:
    """cost_up_small on a workspace prepared by cost_up_prepare for these weights and this shape."""
    x, prev, ws = _dev(x, "cost_up_run"), _dev(prev, "cost_up_run"), _wsbuf(ws, "cost_up_run")
    (wa, k1), (ba, k2) = _reg_args(weights, biases, 4, 4, "cost_up_run")
    B, _, D, H, W = x.shape
    if tuple(prev.shape) != (B, 1, D, H // 2, W // 2):
        raise ValueError("cost_up_run: prev {} does not match x {}".format(tuple(prev.shape), tuple(x.shape)))
    out = torch.empty(B, 1, D, H, W, device=x.device, dtype=torch.float32)
    _count(4)
    capi.check(_lib.effimvs_cost_up_small_ex(x.data_ptr(), prev.data_ptr(), wa, ba, B, D, H, W, precision, capi.WS_RUN, ws.data_ptr(),
                                             ws.numel(), out.data_ptr(), _stream()))
    del k1, k2
    return out


@cost_up_run.register_fake
def _(x, prev, weights, biases, precision, ws):
    return x.new_empty(x.shape)


# -------------------------------------------------------------------------------------------
@torch.library.custom_op("effimvs::images_u8_to_f32", mutates_args=("out",))
@_on_tensor_device
def images_u8_to_f32(images: Tensor, out: Tensor) -> None:
    """out[i] = images[i] / 255 (IEEE division, upstream's loader arithmetic); images uint8, out fp32, same shape, both contiguous."""
    if not (images.is_cuda and out.is_cuda):
        raise RuntimeError("effimvs::images_u8_to_f32 got a CPU tensor; the hot path is CUDA-only (no fallback)")
    if images.dtype != torch.uint8 or out.dtype != torch.float32 or images.shape != out.shape or not (
            images.is_contiguous() and out.is_contiguous()):
        raise RuntimeError("effimvs::images_u8_to_f32: images must be uint8, out fp32, same shape, contiguous")
    _count(1)
    capi.check(_lib.effimvs_images_u8_to_f32(images.data_ptr(), images.numel(), out.data_ptr(), _stream()))


@torch.library.custom_op("effimvs::fusion_invert_cameras", mutates_args=())
@_on_tensor_device
def fusion_invert_cameras(ref_cam: Tensor, srcs_cam: Tensor) -> Tensor:
    ref_cam, srcs_cam = _dev(ref_cam, "fusion_invert_cameras"), _dev(srcs_cam, "fusion_invert_cameras")
    n, v = srcs_cam.shape[0], srcs_cam.shape[1]
    out = torch.empty(n, v + 1, 2, 4, 4, device=ref_cam.device, dtype=torch.float32)
    _count(1)
    capi.check(_lib.effimvs_fusion_invert_cameras_f32(ref_cam.data_ptr(), srcs_cam.data_ptr(), n, v, out.data_ptr(), _stream()))
    return out


@fusion_invert_cameras.register_fake
def _(ref_cam, srcs_cam):
    return ref_cam.new_empty(srcs_cam.shape[0], srcs_cam.shape[1] + 1, 2, 4, 4)


@torch.library.custom_op("effimvs::fusion_reproject", mutates_args=())
@_on_tensor_device
def fusion_reproject(ref_depth: Tensor, srcs_depth: Tensor, ref_cam: Tensor, srcs_cam: Tensor,
                     inv_cams: Optional[Tensor]) -> Tensor:
    ref_depth, srcs_depth = _dev(ref_depth, "fusion_reproject"), _dev(srcs_depth, "fusion_reproject")
    ref_cam, srcs_cam = _dev(ref_cam, "fusion_reproject"), _dev(srcs_cam, "fusion_reproject")
    inv_cams = _dev(inv_cams, "fusion_reproject") if inv_cams is not None else None
    n, v, _, h, w = srcs_depth.shape
    out = torch.empty(n, v, 3, h, w, device=ref_depth.device, dtype=torch.float32)
    _count(1)
    capi.check(_lib.effimvs_fusion_reproject_f32(ref_depth.data_ptr(), srcs_depth.data_ptr(), ref_cam.data_ptr(),
                                                 srcs_cam.data_ptr(), _opt(inv_cams), n, v, h, w, out.data_ptr(), _stream()))
    return out


@fusion_reproject.register_fake
def _(ref_depth, srcs_depth, ref_cam, srcs_cam, inv_cams):
    n, v, _, h, w = srcs_depth.shape
    return ref_depth.new_empty(n, v, 3, h, w)


@torch.library.custom_op("effimvs::fusion_filter", mutates_args=())
@_on_tensor_device
def fusion_filter(ref_depth: Tensor, srcs_depth: Tensor, conf: Tensor, ref_cam: Tensor, srcs_cam: Tensor,
                  inv_cams: Optional[Tensor], dist_base: float, rel_diff_base: float, thres_view: int,
                  prob_threshold: float, relative: bool, want_masks: bool) -> Tuple[Tensor, Tensor, Tensor, Tensor]:
    ref_depth, srcs_depth, conf = _dev(ref_depth, "fusion_filter"), _dev(srcs_depth, "fusion_filter"), _dev(conf, "fusion_filter")
    ref_cam, srcs_cam = _dev(ref_cam, "fusion_filter"), _dev(srcs_cam, "fusion_filter")
    inv_cams = _dev(inv_cams, "fusion_filter") if inv_cams is not None else None
    n, v, _, h, w = srcs_depth.shape
    hc, wc = conf.shape[-2:]
    dev = ref_depth.device
    final = torch.empty(n, 1, h, w, device=dev, dtype=torch.uint8)
    avg = torch.empty(n, 1, h, w, device=dev, dtype=torch.float32)
    pts = torch.empty(n, 3, h, w, device=dev, dtype=torch.float32)
    K = v - thres_view + 1
    masks = torch.empty((n, v, K, h, w) if want_masks else (0,), device=dev, dtype=torch.uint8)
    _count(1)
    capi.check(_lib.effimvs_fusion_filter_f32(ref_depth.data_ptr(), srcs_depth.data_ptr(), conf.data_ptr(), ref_cam.data_ptr(),
                                              srcs_cam.data_ptr(), _opt(inv_cams), n, v, h, w, hc, wc, dist_base, rel_diff_base,
                                              thres_view, prob_threshold, int(relative), final.data_ptr(), avg.data_ptr(),
                                              pts.data_ptr(), masks.data_ptr() if want_masks else None, _stream()))
    return final, avg, pts, masks


@fusion_filter.register_fake
def _(ref_depth, srcs_depth, conf, ref_cam, srcs_cam, inv_cams, dist_base, rel_diff_base, thres_view, prob_threshold,
      relative, want_masks):
    n, v, _, h, w = srcs_depth.shape
    K = v - thres_view + 1
    u8 = torch.uint8
    return (ref_depth.new_empty(n, 1, h, w, dtype=u8), ref_depth.new_empty(n, 1, h, w), ref_depth.new_empty(n, 3, h, w),
            ref_depth.new_empty((n, v, K, h, w) if want_masks else (0,), dtype=u8))


# -------------------------------------------------------------------------------------------
# SURVEY section 8(f) row 3: ConvGRU / convex-upsampling glue (csrc/update_glue.cu).  Multi-channel maps
# are channels-last; (B,1,H,W) maps are plain dense.
def _nhwc(t: Tensor, name: str) -> Tensor:
    if not t.is_cuda:
        raise RuntimeError("effimvs::{} got a CPU tensor; the hot path is CUDA-only (no fallback)".format(name))
    if t.dtype != torch.float32:
        t = t.float()
    return t.contiguous(memory_format=torch.channels_last)


@torch.library.custom_op("effimvs::gru_reset", mutates_args=())
@_on_tensor_device
def gru_reset(zr_pre: Tensor, bias_r: Tensor, hx: Tensor) -> Tensor:
    """zr_pre (B,2h,H,W) = [convz ; convr] without bias, hx (B,h+cx,H,W) = cat[h, x] -> cat[sigmoid(r) * h, x]."""
    zr_pre, hx, bias_r = _nhwc(zr_pre, "gru_reset"), _nhwc(hx, "gru_reset"), _dev(bias_r, "gru_reset")
    B, two_h, H, W = zr_pre.shape
    h = two_h // 2
    out = torch.empty_like(hx, memory_format=torch.channels_last)
    _count(1)
    capi.check(_lib.effimvs_gru_reset_f32(zr_pre.data_ptr(), bias_r.data_ptr(), hx.data_ptr(), B * H * W, h, hx.shape[1] - h,
                                          out.data_ptr(), _stream()))
    return out


@gru_reset.register_fake
def _(zr_pre, bias_r, hx):
    return torch.empty_like(hx, memory_format=torch.channels_last)


@torch.library.custom_op("effimvs::gru_update", mutates_args=("hx",))
@_on_tensor_device
def gru_update(zr_pre: Tensor, bias_z: Tensor, q_pre: Tensor, bias_q: Tensor, hx: Tensor) -> Tensor:
    """h' = (1 - z) * h + z * tanh(q_pre + bias_q); updates hx[:, :h] in place (hx must be channels-last) and
    returns h' as a dense channels-last (B,h,H,W) map."""
    zr_pre, q_pre = _nhwc(zr_pre, "gru_update"), _nhwc(q_pre, "gru_update")
    bias_z, bias_q = _dev(bias_z, "gru_update"), _dev(bias_q, "gru_update")
    if not (hx.is_cuda and hx.dtype == torch.float32 and hx.is_contiguous(memory_format=torch.channels_last)):
        raise RuntimeError("effimvs::gru_update needs hx as a channels-last fp32 CUDA tensor (it is updated in place)")
    B, h, H, W = q_pre.shape
    net = torch.empty_like(q_pre, memory_format=torch.channels_last)
    _count(1)
    capi.check(_lib.effimvs_gru_update_f32(zr_pre.data_ptr(), bias_z.data_ptr(), q_pre.data_ptr(), bias_q.data_ptr(), hx.data_ptr(),
                                           B * H * W, h, hx.shape[1] - h, net.data_ptr(), _stream()))
    return net


@gru_update.register_fake
def _(zr_pre, bias_z, q_pre, bias_q, hx):
    return torch.empty_like(q_pre, memory_format=torch.channels_last)


@torch.library.custom_op("effimvs::gru_delta", mutates_args=())
@_on_tensor_device
def gru_delta(pre: Optional[Tensor], bias: Optional[Tensor], inv: Tensor, lo_disp: Tensor, hi_disp: Tensor) -> Tuple[Tensor, Tensor]:
    """inv' = inv + tanh(pre + bias) (pre None: inv' = inv) and depth = 1 / clamp(lo + (hi - lo) * inv', 1e-4); all (B,1,H,W)."""
    inv, lo_disp, hi_disp = _dev(inv, "gru_delta"), _dev(lo_disp, "gru_delta"), _dev(hi_disp, "gru_delta")
    B, _, H, W = inv.shape
    if pre is not None:
        pre, bias = _dev(pre, "gru_delta"), _dev(bias, "gru_delta")
        inv_out = torch.empty_like(inv)
    else:
        inv_out = inv
    depth = torch.empty_like(inv)
    _count(1)
    capi.check(_lib.effimvs_gru_delta_f32(_opt(pre), _opt(bias), inv.data_ptr(), lo_disp.data_ptr(), hi_disp.data_ptr(), B, H * W,
                                          inv_out.data_ptr() if pre is not None else None, depth.data_ptr(), _stream()))
    return (inv_out if pre is not None else inv.clone()), depth


@gru_delta.register_fake
def _(pre, bias, inv, lo_disp, hi_disp):
    return torch.empty_like(inv), torch.empty_like(inv)


@torch.library.custom_op("effimvs::inv_init", mutates_args=())
@_on_tensor_device
def inv_init(cur_depth: Tensor, lo_disp: Tensor, hi_disp: Tensor) -> Tuple[Tensor, Tensor]:
    """cur_depth (B,1,H,W) -> (inv, depth): inv = (1 / cur_depth - lo) / ((hi - lo) + 1e-10) and depth = 1 / clamp(lo + (hi - lo) inv,
    1e-4): depth_to_disp followed by disp_to_depth (models/Effi_MVS_plus.py:138-164), bit-identical to the torch chain."""
    cur_depth, lo_disp, hi_disp = _dev(cur_depth, "inv_init"), _dev(lo_disp, "inv_init"), _dev(hi_disp, "inv_init")
    B, _, H, W = cur_depth.shape
    inv, depth = torch.empty_like(cur_depth), torch.empty_like(cur_depth)
    _count(1)
    capi.check(_lib.effimvs_inv_init_f32(cur_depth.data_ptr(), lo_disp.data_ptr(), hi_disp.data_ptr(), B, H * W, inv.data_ptr(),
                                         depth.data_ptr(), _stream()))
    return inv, depth


@inv_init.register_fake
def _(cur_depth, lo_disp, hi_disp):
    return torch.empty_like(cur_depth), torch.empty_like(cur_depth)


@torch.library.custom_op("effimvs::delta_head", mutates_args=())
@_on_tensor_device
def delta_head(t: Tensor, weight: Tensor, bias: Tensor, inv: Tensor, lo_disp: Tensor, hi_disp: Tensor) -> Tuple[Tensor, Tensor]:
    """t (B,h,H,W) = relu(depth_head.conv1(net)), weight (1,h,3,3), bias (1): inv' = inv + tanh(conv3x3(t) + bias) and
    depth = 1 / clamp(lo + (hi - lo) * inv', 1e-4), both (B,1,H,W) -- depth_head.conv2 and gru_delta in one pass."""
    t, weight, bias = _nhwc(t, "delta_head"), _dev(weight, "delta_head"), _dev(bias, "delta_head")
    inv, lo_disp, hi_disp = _dev(inv, "delta_head"), _dev(lo_disp, "delta_head"), _dev(hi_disp, "delta_head")
    B, h, H, W = t.shape
    if tuple(weight.shape) != (1, h, 3, 3) or inv.numel() != B * H * W:
        raise ValueError("delta_head: weight {} / inv {} do not match t {}".format(tuple(weight.shape), tuple(inv.shape), tuple(t.shape)))
    inv_out, depth = torch.empty_like(inv), torch.empty_like(inv)
    _count(1)
    capi.check(_lib.effimvs_delta_head_f32(t.data_ptr(), weight.data_ptr(), bias.data_ptr(), inv.data_ptr(), lo_disp.data_ptr(),
                                           hi_disp.data_ptr(), B, h, H, W, inv_out.data_ptr(), depth.data_ptr(), _stream()))
    return inv_out, depth


@delta_head.register_fake
def _(t, weight, bias, inv, lo_disp, hi_disp):
    return torch.empty_like(inv), torch.empty_like(inv)


@torch.library.custom_op("effimvs::convex_upsample", mutates_args=())
@_on_tensor_device
def convex_upsample(mask_pre: Tensor, mask_bias: Optional[Tensor], mask_scale: float, inv: Tensor, lo_disp: Tensor,
                    hi_disp: Tensor, ratio: int) -> Tuple[Tensor, Tensor]:
    """upsample_depth on mask = mask_scale * (mask_pre + mask_bias): (B,9*ratio^2,H,W), inv (B,1,H,W)
    -> up (B,ratio*H,ratio*W) and disp_to_depth(up)."""
    mask_pre, inv = _nhwc(mask_pre, "convex_upsample"), _dev(inv, "convex_upsample")
    lo_disp, hi_disp = _dev(lo_disp, "convex_upsample"), _dev(hi_disp, "convex_upsample")
    mask_bias = _dev(mask_bias, "convex_upsample") if mask_bias is not None else None
    B, _, H, W = inv.shape
    up = torch.empty(B, ratio * H, ratio * W, device=inv.device, dtype=torch.float32)
    depth = torch.empty_like(up)
    _count(1)
    capi.check(_lib.effimvs_convex_upsample_f32(mask_pre.data_ptr(), _opt(mask_bias), mask_scale, inv.data_ptr(), lo_disp.data_ptr(),
                                                hi_disp.data_ptr(), B, H, W, ratio, up.data_ptr(), depth.data_ptr(), _stream()))
    return up, depth


@convex_upsample.register_fake
def _(mask_pre, mask_bias, mask_scale, inv, lo_disp, hi_disp, ratio):
    B, _, H, W = inv.shape
    return inv.new_empty(B, ratio * H, ratio * W), inv.new_empty(B, ratio * H, ratio * W)


@torch.library.custom_op("effimvs::convex_upsample_conv", mutates_args=())
@_on_tensor_device
def convex_upsample_conv(t: Tensor, mask_w: Tensor, mask_bias: Optional[Tensor], mask_scale: float, inv: Tensor, lo_disp: Tensor,
                         hi_disp: Tensor, ratio: int) -> Tuple[Tensor, Tensor]:
    """convex_upsample with mask = mask_scale * (conv1x1(t, mask_w) + mask_bias) formed in the kernel: t (B,K,H,W) =
    relu(mask[0](net)), mask_w (9*ratio^2, K, 1, 1)."""
    t, mask_w, inv = _nhwc(t, "convex_upsample_conv"), _dev(mask_w, "convex_upsample_conv"), _dev(inv, "convex_upsample_conv")
    lo_disp, hi_disp = _dev(lo_disp, "convex_upsample_conv"), _dev(hi_disp, "convex_upsample_conv")
    mask_bias = _dev(mask_bias, "convex_upsample_conv") if mask_bias is not None else None
    B, K, H, W = t.shape
    if mask_w.numel() != 9 * ratio * ratio * K or inv.numel() != B * H * W:
        raise ValueError("convex_upsample_conv: shapes do not match")
    up = torch.empty(B, ratio * H, ratio * W, device=inv.device, dtype=torch.float32)
    depth = torch.empty_like(up)
    _count(1)
    capi.check(_lib.effimvs_convex_upsample_conv_f32(t.data_ptr(), K, mask_w.data_ptr(), _opt(mask_bias), mask_scale, inv.data_ptr(),
                                                     lo_disp.data_ptr(), hi_disp.data_ptr(), B, H, W, ratio, up.data_ptr(),
                                                     depth.data_ptr(), _stream()))
    return up, depth


@convex_upsample_conv.register_fake
def _(t, mask_w, mask_bias, mask_scale, inv, lo_disp, hi_disp, ratio):
    B, _, H, W = inv.shape
    return inv.new_empty(B, ratio * H, ratio * W), inv.new_empty(B, ratio * H, ratio * W)


# Host-side weight tables of encoder_head's constant-bank kernel (csrc/update_glue.cu: the weights travel as kernel parameters, so
# they must be in host memory when the kernel is launched).  One entry per set of weight tensors, found by object identity: the
# entry holds weak references and the versions / addresses it was built from, so an in-place update, a re-assigned .data or a
# recycled id() misses and rebuilds.  Building costs one synchronous device -> host copy of ~50 h floats; it cannot happen
# while the stream is being captured, where a miss falls back to the kernel that reads the weights from device memory.
_EH_TABLES: dict = {}


def _encoder_head_table(ws, CD: int, h: int):
    import weakref
    key = tuple(id(t) for t in ws)
    stamp = tuple((t.data_ptr(), t._version) for t in ws)
    hit = _EH_TABLES.get(key)
    if hit is not None and hit[1] == stamp and all(r() is t for r, t in zip(hit[0], ws)):
        return hit[2]
    if torch.cuda.is_current_stream_capturing():
        return None
    host = [t.detach().to("cpu", torch.float32).contiguous() for t in ws]
    table = torch.empty(_lib.effimvs_encoder_head_table_floats(h), dtype=torch.float32)
    capi.check(_lib.effimvs_encoder_head_pack_host(host[0].data_ptr(), host[1].data_ptr(), host[2].data_ptr(), host[3].data_ptr(), CD, h,
                                                   table.data_ptr()))
    if len(_EH_TABLES) >= 256:                     # temporaries (tests, one-off calls) would otherwise pile up as dead entries
        for k in [k for k, v in _EH_TABLES.items() if any(r() is None for r in v[0])]:
            del _EH_TABLES[k]
    try:
        _EH_TABLES[key] = (tuple(weakref.ref(t) for t in ws), stamp, table)
    except TypeError:                              # not weak-referenceable (never the case for torch.Tensor): use it uncached
        pass
    return table


@torch.library.custom_op("effimvs::encoder_head", mutates_args=())
@_on_tensor_device
def encoder_head(cost: Tensor, inv: Tensor, wc1: Tensor, bc1: Tensor, wd1: Tensor, bd1: Tensor) -> Tensor:
    """cat[relu(convc1(cost)), relu(convd1(inv))] as one channels-last (B,2h,H,W) map (models/update.py:88-91)."""
    cost, inv = _dev(cost, "encoder_head"), _dev(inv, "encoder_head")
    wc1, bc1, wd1, bd1 = _dev(wc1, "encoder_head"), _dev(bc1, "encoder_head"), _dev(wd1, "encoder_head"), _dev(bd1, "encoder_head")
    B, CD, H, W = cost.shape
    h = wc1.shape[0]
    out = torch.empty(B, 2 * h, H, W, device=cost.device, dtype=torch.float32, memory_format=torch.channels_last)
    # measured on B200 (tools/eh_time.py, DTU stage shapes): h = 16 at 800 x 592 40.0 us against 47.1 from device-memory weights,
    # h = 32 at 400 x 296 31.7 / 32.8 (two launches), h = 48 at 200 x 148 33.8 / 20.4 (three launches of a grid that no longer
    # fills the machine): by default only the single-launch case.  EFFIMVS_EH_CONST = 1 / 0 forces it on / off.
    mode = os.environ.get("EFFIMVS_EH_CONST", "auto")
    use_const = 1 <= CD <= 8 and h % 16 == 0 and 16 <= h <= 128 and (mode == "1" or (mode != "0" and h == 16))
    table = _encoder_head_table((wc1, bc1, wd1, bd1), CD, h) if use_const else None
    if table is not None:          # weights as kernel parameters: h / 16 launches, no staging prologue, no shared-memory weight reads
        _count(h // 16)
        capi.check(_lib.effimvs_encoder_head_hostw_f32(cost.data_ptr(), inv.data_ptr(), table.data_ptr(), B, CD, h, H, W, out.data_ptr(),
                                                       _stream()))
        return out
    _count(1)
    capi.check(_lib.effimvs_encoder_head_f32(cost.data_ptr(), inv.data_ptr(), wc1.data_ptr(), bc1.data_ptr(), wd1.data_ptr(), bd1.data_ptr(),
                                             B, CD, h, H, W, out.data_ptr(), _stream()))
    return out


@encoder_head.register_fake
def _(cost, inv, wc1, bc1, wd1, bd1):
    B, _, H, W = cost.shape
    return torch.empty((B, 2 * wc1.shape[0], H, W), device=cost.device, dtype=cost.dtype, memory_format=torch.channels_last)


@torch.library.custom_op("effimvs::encoder_tail", mutates_args=("hx",))
@_on_tensor_device
def encoder_tail(m: Tensor, w: Tensor, ctx_term: Tensor, hx: Tensor) -> None:
    """hx[:, h:] = relu(conv1x1(m, w) + ctx_term) in place; m (B,hm,H,W), ctx_term (B,h,H,W), hx (B,2h,H,W) channels-last."""
    m, ctx_term, w = _nhwc(m, "encoder_tail"), _nhwc(ctx_term, "encoder_tail"), _dev(w, "encoder_tail")
    if not (hx.is_cuda and hx.dtype == torch.float32 and hx.is_contiguous(memory_format=torch.channels_last)):
        raise RuntimeError("effimvs::encoder_tail needs hx as a channels-last fp32 CUDA tensor (it is updated in place)")
    B, hm, H, W = m.shape
    h = ctx_term.shape[1]
    if hx.shape[1] != 2 * h or w.shape[0] != h or w.shape[1] != hm:
        raise ValueError("encoder_tail: shapes do not match")
    _count(1)
    capi.check(_lib.effimvs_encoder_tail_f32(m.data_ptr(), w.data_ptr(), ctx_term.data_ptr(), B * H * W, hm, h, hx.data_ptr(), _stream()))


@torch.library.custom_op("effimvs::encoder_tail_ctx", mutates_args=("hx",))
@_on_tensor_device
def encoder_tail_ctx(m: Tensor, w_m: Tensor, ctx: Tensor, ctx_offset: int, cx: int, ctx_relu: bool, w_ctx: Tensor, bias: Tensor,
                     hx: Tensor) -> None:
    """hx[:, h:] = relu(conv1x1(m, w_m) + conv1x1(act(ctx[:, ctx_offset:ctx_offset+cx]), w_ctx) + bias) in place;
    m (B,hm,H,W), ctx (B,*,H,W), hx (B,2h,H,W) channels-last; act = relu if ctx_relu else identity."""
    m, ctx = _nhwc(m, "encoder_tail_ctx"), _nhwc(ctx, "encoder_tail_ctx")
    w_m, w_ctx, bias = _dev(w_m, "encoder_tail_ctx"), _dev(w_ctx, "encoder_tail_ctx"), _dev(bias, "encoder_tail_ctx")
    if not (hx.is_cuda and hx.dtype == torch.float32 and hx.is_contiguous(memory_format=torch.channels_last)):
        raise RuntimeError("effimvs::encoder_tail_ctx needs hx as a channels-last fp32 CUDA tensor (it is updated in place)")
    B, hm, H, W = m.shape
    h = w_m.shape[0]
    ct = ctx.shape[1]
    if (hx.shape[1] != 2 * h or w_m.numel() != h * hm or w_ctx.numel() != h * cx or bias.numel() != h or ctx_offset < 0
            or ctx_offset + cx > ct or ctx_offset % 4 or tuple(ctx.shape[2:]) != (H, W)):
        raise ValueError("encoder_tail_ctx: shapes do not match")
    _count(1)
    capi.check(_lib.effimvs_encoder_tail_ctx_f32(m.data_ptr(), w_m.data_ptr(), ctx.data_ptr() + 4 * ctx_offset, ct, cx, int(ctx_relu),
                                                 w_ctx.data_ptr(), bias.data_ptr(), B * H * W, hm, h, hx.data_ptr(), _stream()))


# -------------------------------------------------------------------------------------------
# SURVEY section 8(f) row 3, the convolutions: 3x3 convolutions of the update block on the tensor cores (csrc/conv2d_tc.cu)
# precision "f16": operands rounded to fp16 (TF32's 11 significant bits, saturating at +-65504), the effimvs_conv2d_tf32 family;
# "bf16x3": operands as hi + lo bf16 pairs, three products, fp32 range (fp32-grade), the effimvs_conv2d_bf16x3 family
def _conv2d_fns(precision: str):
    if precision == "f16":
        return (_lib.effimvs_conv2d_tf32_supported, _lib.effimvs_conv2d_tf32_packed_bytes, _lib.effimvs_conv2d_tf32_pack,
                _lib.effimvs_conv2d_tf32)
    if precision == "bf16x3":
        return (_lib.effimvs_conv2d_bf16x3_supported, _lib.effimvs_conv2d_bf16x3_packed_bytes, _lib.effimvs_conv2d_bf16x3_pack,
                _lib.effimvs_conv2d_bf16x3)
    raise ValueError("conv2d_tc: precision must be 'f16' or 'bf16x3', got {!r}".format(precision))


def conv2d_tc_supported(cin: int, cout: int, precision: str = "f16") -> bool:
    return bool(_conv2d_fns(precision)[0](int(cin), int(cout)))


def _cl_view(t: Tensor, name: str):
    """(pointer, pixel stride) of a channels-last map or of a channel slice of one: dims (B,C,H,W), element strides
    (H*W*ps, 1, W*ps, ps)."""
    if not t.is_cuda or t.dtype != torch.float32 or t.dim() != 4:
        raise RuntimeError("effimvs::conv2d_tc needs 4-D fp32 CUDA tensors ({})".format(name))
    B, C, H, W = t.shape
    ps = t.stride(3)
    if t.stride(1) != 1 or t.stride(2) != W * ps or (B > 1 and t.stride(0) != H * W * ps) or ps < C:
        raise RuntimeError("effimvs::conv2d_tc: {} must be a channels-last map or a channel slice of one, got strides {}".format(name, t.stride()))
    return t.data_ptr(), ps


@torch.library.custom_op("effimvs::conv2d_tc_pack", mutates_args=())
@_on_tensor_device
def conv2d_tc_pack(weight: Tensor, precision: str = "f16") -> Tensor:
    """(cout, cin, 3, 3) fp32 -> the kernel's packed weight image for `precision` (once per weight tensor): fp16, or the
    bf16 hi image followed by the lo image for "bf16x3"."""
    supported, packed_bytes, pack, _ = _conv2d_fns(precision)
    weight = _dev(weight, "conv2d_tc_pack")
    cout, cin = weight.shape[:2]
    if tuple(weight.shape[2:]) != (3, 3) or not supported(cin, cout):
        raise ValueError("conv2d_tc_pack: unsupported weight shape {} for precision {}".format(tuple(weight.shape), precision))
    packed = torch.empty(packed_bytes(cin, cout) // 4, device=weight.device, dtype=torch.float32)
    _count(1)
    capi.check(pack(weight.data_ptr(), cin, cout, packed.data_ptr(), _stream()))
    return packed


@conv2d_tc_pack.register_fake
def _(weight, precision="f16"):
    copies = 2 if precision == "bf16x3" else 1
    return weight.new_empty(copies * 9 * weight.shape[1] * ((weight.shape[0] + 15) // 16 * 16) // 2)


@torch.library.custom_op("effimvs::conv2d_tc", mutates_args=("out", "aux1"))
@_on_tensor_device
def conv2d_tc(in0: Tensor, in1: Optional[Tensor], packed: Tensor, bias: Optional[Tensor], cout: int, mode: int, out: Tensor,
              aux0: Optional[Tensor], aux1: Optional[Tensor], precision: str = "f16") -> None:
    """3x3 / stride 1 / padding 1 convolution of cat[in0, in1] (channels-last maps or channel slices of such maps, read and
    written in place) with the epilogue `mode` (capi.CONV2D_*): BIAS / BIAS_RELU -> out; ADD_RELU: out = relu(acc + aux0);
    GRU_GATES: aux1 = z, out = r * aux0 (aux0 = h); GRU_UPDATE: out = (1 - aux0) * out + aux0 * tanh(acc + bias) (aux0 = z).  `packed` from conv2d_tc_pack with the same
    precision."""
    _, packed_bytes, _, conv = _conv2d_fns(precision)
    B, c0, H, W = in0.shape
    p0, ps0 = _cl_view(in0, "in0")
    p1, ps1, c1 = None, 0, 0
    if in1 is not None:
        p1, ps1 = _cl_view(in1, "in1")
        c1 = in1.shape[1]
        if tuple(in1.shape) != (B, c1, H, W):
            raise ValueError("conv2d_tc: in1 {} does not match in0 {}".format(tuple(in1.shape), tuple(in0.shape)))
    po, pso = _cl_view(out, "out")
    h = cout // 2 if mode == capi.CONV2D_GRU_GATES else cout
    if tuple(out.shape) != (B, h, H, W):
        raise ValueError("conv2d_tc: out {} should be {}".format(tuple(out.shape), (B, h, H, W)))
    pa0, psa0 = _cl_view(aux0, "aux0") if aux0 is not None else (None, 0)
    pa1, psa1 = _cl_view(aux1, "aux1") if aux1 is not None else (None, 0)
    for a in (aux0, aux1):
        if a is not None and tuple(a.shape) != (B, h, H, W):
            raise ValueError("conv2d_tc: aux map {} should be {}".format(tuple(a.shape), (B, h, H, W)))
    if packed.numel() * 4 != packed_bytes(c0 + c1, cout):
        raise ValueError("conv2d_tc: packed weights do not match cin = {} cout = {} ({})".format(c0 + c1, cout, precision))
    bias = _dev(bias, "conv2d_tc") if bias is not None else None
    _count(1)
    capi.check(conv(p0, ps0, c0, p1, ps1, c1, packed.data_ptr(), _opt(bias), cout, B, H, W, mode,
                    po, pso, pa0, psa0, pa1, psa1, _stream()))


@conv2d_tc.register_fake
def _(in0, in1, packed, bias, cout, mode, out, aux0, aux1, precision="f16"):
    return None


@torch.library.custom_op("effimvs::gru_init", mutates_args=())
@_on_tensor_device
def gru_init(ctx_map: Tensor, h: int) -> Tensor:
    """ctx_map (B,h+cx,H,W) -> hx (B,2h,H,W) channels-last with hx[:, :h] = tanh(ctx_map[:, :h]) (the x half is left for
    encoder_tail to fill)."""
    ctx_map = _nhwc(ctx_map, "gru_init")
    B, ct, H, W = ctx_map.shape
    if h <= 0 or h % 4 or ct < h or (ct - h) % 4:
        raise ValueError("gru_init: hidden {} / map channels {} must be multiples of 4".format(h, ct))
    hx = torch.empty(B, 2 * h, H, W, device=ctx_map.device, dtype=torch.float32, memory_format=torch.channels_last)
    _count(1)
    capi.check(_lib.effimvs_gru_init_f32(ctx_map.data_ptr(), B * H * W, h, ct - h, hx.data_ptr(), _stream()))
    return hx


@gru_init.register_fake
def _(ctx_map, h):
    B, _, H, W = ctx_map.shape
    return torch.empty((B, 2 * h, H, W), device=ctx_map.device, dtype=ctx_map.dtype, memory_format=torch.channels_last)


@torch.library.custom_op("effimvs::gru_init_ctx", mutates_args=())
@_on_tensor_device
def gru_init_ctx(ctx_map: Tensor, h: int, w_ctx: Tensor, bias: Tensor) -> Tuple[Tensor, Tensor]:
    """gru_init plus the iteration-invariant context term of the encoder tail in the same pass over the context map:
    returns (hx (B,2h,H,W) with hx[:, :h] = tanh(ctx_map[:, :h]), ctx_term (B,h,H,W) = conv1x1(relu(ctx_map[:, h:]), w_ctx) + bias),
    both channels-last; w_ctx (h, cx[, 1, 1]) = convc.weight[:, hm:], bias (h) (models/update.py:93-95, Effi_MVS_plus.py:464-466)."""
    ctx_map = _nhwc(ctx_map, "gru_init_ctx")
    B, ct, H, W = ctx_map.shape
    cx = ct - h
    if h <= 0 or h % 4 or h > 128 or cx < 4 or cx % 4 or cx > 64:
        raise ValueError("gru_init_ctx: hidden {} (<= 128) / context {} (4..64) channels must be multiples of 4".format(h, cx))
    w2 = w_ctx.detach().reshape(w_ctx.shape[0], -1).contiguous().float()
    if tuple(w2.shape) != (h, cx) or bias.numel() != h:
        raise ValueError("gru_init_ctx: w_ctx {} / bias {} do not match h={}, cx={}".format(tuple(w_ctx.shape), tuple(bias.shape), h, cx))
    bias = bias.detach().contiguous().float()
    hx = torch.empty(B, 2 * h, H, W, device=ctx_map.device, dtype=torch.float32, memory_format=torch.channels_last)
    term = torch.empty(B, h, H, W, device=ctx_map.device, dtype=torch.float32, memory_format=torch.channels_last)
    _count(1)
    capi.check(_lib.effimvs_gru_init_ctx_f32(ctx_map.data_ptr(), B * H * W, h, cx, w2.data_ptr(), bias.data_ptr(), hx.data_ptr(),
                                             term.data_ptr(), _stream()))
    return hx, term


@gru_init_ctx.register_fake
def _(ctx_map, h, w_ctx, bias):
    B, _, H, W = ctx_map.shape
    mk = lambda c: torch.empty((B, c, H, W), device=ctx_map.device, dtype=ctx_map.dtype, memory_format=torch.channels_last)   # noqa: E731
    return mk(2 * h), mk(h)


# -------------------------------------------------------------------------------------------
# SURVEY section 8(f) row 2: DTU geometric filter (csrc/dtu_filter.cu)
@torch.library.custom_op("effimvs::dtu_filter", mutates_args=())
@_on_tensor_device
def dtu_filter(ref_depth: Tensor, srcs_depth: Tensor, conf: Tensor, mats: Tensor, thr_dist: List[float], thr_diff: List[float],
               first_rung: int, full_count: int, conf_thres: float, conf_keep: float, want_masks: bool) -> Tuple[Tensor, Tensor, Tensor, Tensor, Tensor, Tensor]:
    """-> final (h,w) u8, geo (h,w) u8, depth_avg (h,w), points (3,h,w), masks (v,K,h,w) u8, reproj_depth (v,h,w)
    (the last two empty unless want_masks)."""
    import ctypes
    ref_depth, srcs_depth, conf, mats = (_dev(ref_depth, "dtu_filter"), _dev(srcs_depth, "dtu_filter"), _dev(conf, "dtu_filter"),
                                         _dev(mats, "dtu_filter"))
    v, h, w = srcs_depth.shape
    K = len(thr_dist)
    dev = ref_depth.device
    final = torch.empty(h, w, device=dev, dtype=torch.uint8)
    geo = torch.empty(h, w, device=dev, dtype=torch.uint8)
    avg = torch.empty(h, w, device=dev, dtype=torch.float32)
    pts = torch.empty(3, h, w, device=dev, dtype=torch.float32)
    masks = torch.empty((v, K, h, w) if want_masks else (0,), device=dev, dtype=torch.uint8)
    rep = torch.empty((v, h, w) if want_masks else (0,), device=dev, dtype=torch.float32)
    td = (ctypes.c_double * K)(*thr_dist)
    tf = (ctypes.c_float * K)(*thr_diff)
    _count(1)
    capi.check(_lib.effimvs_dtu_filter_f32(ref_depth.data_ptr(), srcs_depth.data_ptr(), conf.data_ptr(), mats.data_ptr(), td, tf, K,
                                           first_rung, full_count, conf_thres, conf_keep, v, h, w, final.data_ptr(), geo.data_ptr(),
                                           avg.data_ptr(), pts.data_ptr(), masks.data_ptr() if want_masks else None,
                                           rep.data_ptr() if want_masks else None, _stream()))
    return final, geo, avg, pts, masks, rep


@dtu_filter.register_fake
def _(ref_depth, srcs_depth, conf, mats, thr_dist, thr_diff, first_rung, full_count, conf_thres, conf_keep, want_masks):
    v, h, w = srcs_depth.shape
    K = len(thr_dist)
    u8 = torch.uint8
    return (ref_depth.new_empty(h, w, dtype=u8), ref_depth.new_empty(h, w, dtype=u8), ref_depth.new_empty(h, w),
            ref_depth.new_empty(3, h, w), ref_depth.new_empty((v, K, h, w) if want_masks else (0,), dtype=u8),
            ref_depth.new_empty((v, h, w) if want_masks else (0,)))
