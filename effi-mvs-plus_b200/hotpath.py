"""CudaHotPath: the hot-path table (stage1 / local_volume / volume_lookup / cross_scale /
dynamic_cost) backed by the hand-written sm_100a kernels through ``effimvs::*`` custom ops.

The same table shape is implemented by the test oracle; ``net.EffiMVSPlus`` and the upstream
drop-ins in ``dropin.py`` are written against it.  Nothing here falls back to PyTorch math: if
libeffimvs.so is missing the import of ``capi`` raises.
"""
from __future__ import annotations

import collections
import functools
import os
import weakref

import torch

from . import capi, ops


def fold_bn(block, transposed: bool):
    """Eval-mode BatchNorm folded into the preceding bias-free (de)conv
    (upstream models/module.py:146-160, 189-203).  Returns fp32 (weight, bias)."""
    bn = block.bn
    scale = bn.weight / torch.sqrt(bn.running_var + bn.eps)
    shift = bn.bias - bn.running_mean * scale
    w = block.conv.weight
    w = w * (scale.reshape(1, -1, 1, 1, 1) if transposed else scale.reshape(-1, 1, 1, 1, 1))
    return w.detach().float().contiguous(), shift.detach().float().contiguous()


class _FoldCache:
    """Folded weights per module, invalidated when a parameter / buffer is replaced or updated in place.  Keyed by the
    module object itself through a weak reference: an entry dies with its module, so a recycled id() cannot serve
    another module's weights."""

    def __init__(self):
        self._store = weakref.WeakKeyDictionary()

    def get(self, net, build):
        stamp = tuple((id(t), t._version, t.device) for t in list(net.parameters()) + list(net.buffers()))
        hit = self._store.get(net)
        if hit is None or hit[0] != stamp:
            hit = (stamp, build(net))
            self._store[net] = hit
        return hit[1]


def _inference_only(*tensors):
    """The effimvs:: ops carry no autograd formula: refuse to drop gradients silently."""
    if torch.is_grad_enabled() and any(torch.is_tensor(t) and t.requires_grad for t in tensors):
        raise RuntimeError("the CUDA hot path is inference only (no autograd formula): run it under torch.no_grad(), "
                           "or use upstream's PyTorch path for training / test-time adaptation")


class _WorkspaceCache:
    """One regularization workspace per (network, shape, precision, device), kept across calls so that its
    preparation (halo clearing + weight packing, effimvs_*_ex PREPARE) runs once per weights instead of once
    per forward.  ``stamp`` is the folded-weight list the workspace was prepared for (held, so its identity
    cannot be recycled).  Least-recently-used entries are dropped beyond ``cap``."""

    def __init__(self, cap: int = 24):
        self._store = collections.OrderedDict()
        self.cap = cap

    def get(self, key, nbytes, device):
        """A workspace that was handed out while its stream was being captured is baked into a CUDA graph by raw
        pointer: it is pinned and never evicted or reallocated (the graph owner may replay it at any time)."""
        capturing = torch.cuda.is_current_stream_capturing() if torch.device(device).type == "cuda" else False
        ent = self._store.get(key)
        if ent is not None and ent["ws"].numel() < nbytes:
            if ent["pinned"]:
                raise RuntimeError("a regularization workspace captured in a CUDA graph is too small for this call")
            ent = None
        if ent is None:
            if capturing:
                raise RuntimeError("regularization workspace requested for the first time during CUDA-graph capture: "
                                   "run one eager forward of this shape before capturing")
            ent = {"ws": torch.empty(max(nbytes, 256), device=device, dtype=torch.uint8), "stamp": None, "pinned": False}
            self._store[key] = ent
            evictable = [k for k, e in self._store.items() if not e["pinned"] and k != key]
            while len(self._store) > self.cap and evictable:
                del self._store[evictable.pop(0)]
        ent["pinned"] = ent["pinned"] or capturing
        self._store.move_to_end(key)
        return ent

    def drop(self, owner_id):
        for k in [k for k in self._store if k[1] == owner_id]:
            del self._store[k]


def _is_planes(hyp: torch.Tensor) -> bool:
    return hyp.dim() == 2 or (hyp.dim() == 4 and (hyp.shape[2:] == (1, 1) or (hyp.stride(2) == 0 and hyp.stride(3) == 0)))


def _forget(hp_ref, owner_id):
    hp = hp_ref()
    if hp is not None:
        hp._tracked.discard(owner_id)
        hp._workspaces.drop(owner_id)


class CudaHotPath:
    name = "cuda"
    fused_update = True      # net.UpdateBlock.forward_fused: GRU / upsampling glue kernels (SURVEY section 8(f) row 3)

    def __init__(self, precision: str = "f32", native_projection: bool = False, persistent_workspaces: bool = True,
                 parallel_branches: bool = False, conv2d_precision=None):
        """precision of the 3-D regularization: 'f32' (CUDA-core direct convs), 'bf16' (tcgen05 implicit
        GEMM, one bf16 MMA per product) or 'bf16x3' (tcgen05, hi/lo split operands, fp32-grade).
        native_projection: compute P_src @ inverse(P_ref) with the library's fp64 kernel instead
        of torch (needed under CUDA-graph capture; torch.linalg.inv may synchronise).
        persistent_workspaces: keep one prepared workspace per regularization network and shape (tensor-core
        precisions) instead of clearing halos and packing weights in every call; an instance must then not run
        the same network on two streams at once.
        parallel_branches: offer a side stream for the independent cross-scale branches (net.EffiMVSPlus).  Off by
        default: measured on B200 the forked graph is slower (7.00 vs 6.91 ms per DTU depth map) -- the persistent
        tensor-core kernels of the two branches cannot co-reside, and the fork / join costs more than the small
        CUDA-core layers gain.
        conv2d_precision: arithmetic of the update block's tensor-core 3x3 convolutions (csrc/conv2d_tc.cu).  None: operands
        rounded to fp16 (TF32's 11 significant bits), used only while torch.backends.cudnn.allow_tf32 is on -- with it off
        those layers stay on cuDNN's fp32 kernels.  'bf16x3': operands as hi + lo bf16 pairs, three products, fp32
        accumulation and range (~2^-16 relative, fp32-grade), so the kernel also runs with allow_tf32 off."""
        self.precision = {"f32": capi.PREC_F32, "bf16": capi.PREC_BF16, "bf16x3": capi.PREC_BF16X3}[precision]
        self.native_projection = native_projection
        self.persistent_workspaces = persistent_workspaces and os.environ.get("EFFIMVS_PERSISTENT_WS", "1") != "0"
        self.parallel_branches = parallel_branches or os.environ.get("EFFIMVS_PARALLEL_BRANCHES", "0") == "1"
        self._folds = _FoldCache()
        self._workspaces = _WorkspaceCache()
        self._side_streams = {}
        self._tracked = set()
        if conv2d_precision not in (None, "bf16x3"):
            raise ValueError("conv2d_precision must be None or 'bf16x3', got {!r}".format(conv2d_precision))
        if conv2d_precision == "bf16x3":
            # the table's conv2d_tc* entries bound to the bf16x3 kernel; net.py keys its packed weight images by
            # conv2d_precision and runs fp32-grade convolutions whatever allow_tf32 says
            self.conv2d_precision = "bf16x3"
            self.conv2d_fp32_grade = True
            self.conv2d_tc = functools.partial(ops.conv2d_tc, precision="bf16x3")
            self.conv2d_tc_pack = functools.partial(ops.conv2d_tc_pack, precision="bf16x3")
            self.conv2d_tc_supported = functools.partial(ops.conv2d_tc_supported, precision="bf16x3")

    def side_stream(self, device):
        """Stream for work that is independent of the caller's current stream (None: run it in line)."""
        if not self.parallel_branches:
            return None
        key = torch.device(device).index
        if key not in self._side_streams:
            self._side_streams[key] = torch.cuda.Stream(device=device)
        return self._side_streams[key]

    # -- a1 + module.py:314 -------------------------------------------------------------------
    def relative_projection(self, cams: torch.Tensor) -> torch.Tensor:
        """cams (B,V,2,4,4) -> (B,V-1,12) rot|trans of P_src @ inverse(P_ref)."""
        if self.native_projection:
            return ops.relative_projection(cams)
        # the same torch calls, with the same operand shapes, as upstream issues per source view
        # (Effi_MVS_plus.py:34-37, module.py:314): a batched formulation can differ from it by an ulp in
        # the entries of proj, which is 1e-4 px at 1600-pixel coordinates
        B, V = cams.shape[:2]

        def compose(c):
            P = c[:, 0].clone()
            P[:, :3, :4] = torch.matmul(c[:, 1, :3, :3], c[:, 0, :3, :4])
            return P
        inv_ref = torch.linalg.inv_ex(compose(cams[:, 0]))[0]       # torch.inverse minus the host-side error check
        rows = []
        for v in range(1, V):
            rel = torch.matmul(compose(cams[:, v]), inv_ref)
            rows.append(torch.cat([rel[:, :3, :3].reshape(B, 9), rel[:, :3, 3]], dim=-1))
        return torch.stack(rows, dim=1).contiguous()

    # -- a2-a4, a9, a11, a12 ---------------------------------------------------------------------
    def stage1(self, features, cams, depth_hyp, pixel_wise_net, reg_net, G):
        if G != 1:
            raise ValueError("stage-1 view weighting requires G == 1 (upstream squeezes the group axis, Effi_MVS_plus.py:43)")
        _inference_only(*features)
        ref, srcs = features[0], list(features[1:])
        B, _, H, W = ref.shape
        D = depth_hyp.shape[1]
        proj = self.relative_projection(cams)
        if _is_planes(depth_hyp):
            hyp, mode = depth_hyp.reshape(B, D, -1)[:, :, 0].contiguous(), capi.HYP_PLANES
        else:
            hyp, mode = depth_hyp, capi.HYP_TENSOR
        sims, ent = ops.warp_corr_views(ref, srcs, proj, hyp, mode, D)
        n = len(srcs)
        vw = pixel_wise_net(ent.reshape(B * n, 1, H, W)).reshape(B, n, H, W)
        sim = ops.weighted_agg(sims, vw)
        prob_pre = self.cost_regularization(reg_net, sim.unsqueeze(1)).squeeze(1)
        depth, conf = ops.softmax_regress_conf(prob_pre, hyp, mode)
        return {"depth": depth, "photometric_confidence": conf, "view_weights": vw,
                "reg_volume": prob_pre, "volume": sim.unsqueeze(1)}

    # -- a5 ---------------------------------------------------------------------------------------
    def local_volume(self, cur_depth, features, cams, interval, view_weights, ndepth, G):
        _inference_only(cur_depth, *features)
        ref, srcs = features[0], list(features[1:])
        B, _, H, W = ref.shape
        proj = self.relative_projection(cams)
        iv = interval.reshape(-1).expand(B) if torch.is_tensor(interval) else torch.full((B,), float(interval), device=ref.device)
        sim, hyp = ops.warp_corr_agg(ref, srcs, proj, cur_depth, capi.HYP_LOCAL, iv.float().contiguous(), view_weights, ndepth, G, True)
        return sim.reshape(B, G * ndepth, H, W), hyp

    # -- a2 + a3 + aggregation with explicit hypotheses (config-2 microbench form) --------------------
    def warp_corr_agg(self, features, cams, hyp, view_weights, G):
        ref, srcs = features[0], list(features[1:])
        D = hyp.shape[1]
        proj = self.relative_projection(cams)
        if _is_planes(hyp):
            hyp, mode = hyp.reshape(hyp.shape[0], D, -1)[:, :, 0].contiguous(), capi.HYP_PLANES
        else:
            mode = capi.HYP_TENSOR
        return ops.warp_corr_agg(ref, srcs, proj, hyp, mode, None, view_weights, D, G, False)[0]

    # -- a6 / a8 ----------------------------------------------------------------------------------
    def volume_lookup(self, volume, depth_sample, depth_min, depth_max):
        """depth_sample may be a [::2, ::2] view of a full-resolution tensor (Effi_MVS_plus.py:514);
        the stride-2 read is then fused into the kernel instead of materialising the view."""
        B, D, H, W = volume.shape
        base = getattr(depth_sample, "_base", None)
        if (not depth_sample.is_contiguous() and base is not None and base.is_contiguous() and base.dim() == 4
                and tuple(base.shape) == (B, depth_sample.shape[1], 2 * H, 2 * W)
                and depth_sample.stride() == (base.stride(0), base.stride(1), 2 * base.stride(2), 2)
                and depth_sample.storage_offset() == base.storage_offset()):
            return ops.volume_lookup(volume, base, self._range(depth_min, B), self._range(depth_max, B), 2)
        return ops.volume_lookup(volume, depth_sample, self._range(depth_min, B), self._range(depth_max, B), 1)

    @staticmethod
    def _range(t, B):
        t = t.reshape(B, -1)
        return t.contiguous()

    # -- a7 ---------------------------------------------------------------------------------------
    def dynamic_cost(self, cur_depth, raw_volume, reg_volume, interval, vmin, vmax, ndepth):
        B = raw_volume.shape[0]
        iv = interval.reshape(-1).expand(B) if torch.is_tensor(interval) else torch.full((B,), float(interval), device=raw_volume.device)
        return ops.dynamic_cost(cur_depth, raw_volume, reg_volume, iv.float().contiguous(), self._range(vmin, B), self._range(vmax, B), ndepth)

    # -- a9 / a10 ---------------------------------------------------------------------------------
    def _reg_weights(self, net):
        def build(n):
            ws, bs = [], []
            for name, tr in (("conv0", False), ("conv1", False), ("conv2", False), ("conv3", False), ("conv4", False),
                             ("conv5", False), ("conv6", True), ("conv7", True)):
                w, b = fold_bn(getattr(n, name), tr)
                ws.append(w)
                bs.append(b)
            ws.append(n.prob.weight.detach().float().contiguous())
            return ws, bs
        return self._folds.get(net, build)

    def _csp_weights(self, net):
        def build(n):
            pairs = [fold_bn(n.conv0, False), fold_bn(n.conv_cost, False), fold_bn(n.conv1, False), fold_bn(n.conv2, True)]
            return [p[0] for p in pairs], [p[1] for p in pairs]
        return self._folds.get(net, build)

    def _track(self, net):
        """workspaces are keyed by id(net): drop them when the network dies so that a recycled id starts clean"""
        if id(net) not in self._tracked:
            self._tracked.add(id(net))
            weakref.finalize(net, _forget, weakref.ref(self), id(net))

    def cost_regularization(self, net, x):
        """x (B,1,D,H,W) -> prob_pre (B,1,D,H,W)   (upstream models/module.py:453-463)."""
        ws, bs = self._reg_weights(net)
        if self.precision == capi.PREC_F32 or not self.persistent_workspaces:
            return ops.costreg_fpn3d(x, ws, bs, self.precision)
        B, _, D, H, W = x.shape
        self._track(net)
        ent = self._workspaces.get(("costreg", id(net), B, D, H, W, self.precision, x.device),
                                   ops.costreg_workspace_bytes(B, D, H, W, self.precision), x.device)
        if ent["stamp"] is not ws:
            ops.costreg_prepare(ws, bs, B, D, H, W, self.precision, ent["ws"])
            ent["stamp"] = ws
        return ops.costreg_run(x, ws, bs, self.precision, ent["ws"])

    def cross_scale(self, net, cur_volume, prev_resampled):
        """cur (B,1,D,H,W), prev (B,1,D,H/2,W/2) -> (B,1,D,H,W)   (upstream models/module.py:509-516)."""
        ws, bs = self._csp_weights(net)
        if self.precision == capi.PREC_F32 or not self.persistent_workspaces:
            return ops.cost_up_small(cur_volume, prev_resampled, ws, bs, self.precision)
        B, _, D, H, W = cur_volume.shape
        self._track(net)
        ent = self._workspaces.get(("cost_up", id(net), B, D, H, W, self.precision, cur_volume.device),
                                   ops.cost_up_workspace_bytes(B, D, H, W, self.precision), cur_volume.device)
        if ent["stamp"] is not ws:
            ops.cost_up_prepare(ws, bs, B, D, H, W, self.precision, ent["ws"])
            ent["stamp"] = ws
        return ops.cost_up_run(cur_volume, prev_resampled, ws, bs, self.precision, ent["ws"])

    # -- section 8(f) row 3: update-block glue (upstream models/update.py:33-49, 114-127; Effi_MVS_plus.py:138-178) ---
    gru_reset = staticmethod(ops.gru_reset)
    gru_update = staticmethod(ops.gru_update)
    gru_delta = staticmethod(ops.gru_delta)
    inv_init = staticmethod(ops.inv_init)
    depth_ranges = staticmethod(ops.depth_ranges)
    delta_head = staticmethod(ops.delta_head)
    convex_upsample = staticmethod(ops.convex_upsample)
    convex_upsample_conv = staticmethod(ops.convex_upsample_conv)
    encoder_head = staticmethod(ops.encoder_head)
    encoder_tail = staticmethod(ops.encoder_tail)
    encoder_tail_ctx = staticmethod(ops.encoder_tail_ctx)
    gru_init = staticmethod(ops.gru_init)
    gru_init_ctx = staticmethod(ops.gru_init_ctx)
    # the block's 3x3 convolutions on the tensor cores, gate arithmetic as epilogues (csrc/conv2d_tc.cu); fp16 operands unless
    # the instance was built with conv2d_precision='bf16x3'
    conv2d_precision = "f16"
    conv2d_fp32_grade = False
    conv2d_tc = staticmethod(ops.conv2d_tc)
    conv2d_tc_pack = staticmethod(ops.conv2d_tc_pack)
    conv2d_tc_supported = staticmethod(ops.conv2d_tc_supported)

    # -- a11 / a12 --------------------------------------------------------------------------------
    def softmax_regress_conf(self, prob_pre, hyp):
        if _is_planes(hyp):
            B, D = prob_pre.shape[:2]
            return ops.softmax_regress_conf(prob_pre, hyp.reshape(B, D, -1)[:, :, 0].contiguous(), capi.HYP_PLANES)
        return ops.softmax_regress_conf(prob_pre, hyp, capi.HYP_TENSOR)
