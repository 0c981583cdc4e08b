"""Host-side network around the hot path (stock PyTorch), checkpoint-compatible
with upstream ``Effi_MVS_plus`` (models/Effi_MVS_plus.py:315-568).

Only the *callers* of the hot path live here: the 2-D feature pyramid
(models/module.py:346-412), the ConvGRU update block (models/update.py:10-141),
the convex upsampling (Effi_MVS_plus.py:167-178) and the three-stage cascade that
strings them together.  They stay stock PyTorch (BASELINE.json north_star).  All
cost-volume work is delegated to a *hot-path table* -- by default
``hotpath.CudaHotPath`` (hand-written sm_100a kernels behind the C-ABI); tests and
the CPU-baseline leg of bench.py inject the oracle's table instead.

Parameter names reproduce upstream's ``state_dict`` layout (including the
duplicate registrations ``update_block_depth1`` / ``update_block.0`` etc.) so that
``model_dtu.ckpt`` / ``model_tank.ckpt`` load with ``strict=True``.
"""
from __future__ import annotations

import os

import torch
import torch.nn as nn
import torch.nn.functional as F

# cuDNN's fused convolution + bias + ReLU (aten::cudnn_convolution_relu, stock PyTorch) for the
# inference path on CUDA; EFFIMVS_FUSED_CONV_RELU=0 falls back to conv2d followed by relu_.
_FUSED_CONV_RELU = os.environ.get("EFFIMVS_FUSED_CONV_RELU", "1") == "1"


def conv_relu(x, weight, bias, stride=(1, 1), padding=(0, 0)):
    """relu(conv2d(x) + bias) -- one fused cuDNN call on CUDA in no-grad mode."""
    if _FUSED_CONV_RELU and x.is_cuda and bias is not None and not torch.is_grad_enabled():
        return torch.cudnn_convolution_relu(x, weight, bias, stride, padding, (1, 1), 1)
    return F.relu(F.conv2d(x, weight, bias, stride, padding), inplace=True)


def _conv_relu_mod(conv: nn.Conv2d, x):
    return conv_relu(x, conv.weight, conv.bias, conv.stride, conv.padding)


# ----------------------------------------------------------------------------
# building blocks (attribute names .conv / .bn are the checkpoint format)
# ----------------------------------------------------------------------------
class ConvBNReLU2d(nn.Module):
    """conv2d(bias-free) + BatchNorm2d + ReLU  (upstream Conv2d / ConvBnReLU).

    In eval mode the BatchNorm is folded into the convolution (the standard PyTorch inference
    fusion, cf. torch.nn.utils.fusion.fuse_conv_bn_eval): one cuDNN convolution with bias instead
    of convolution + a separate normalisation pass over the full-resolution map.  The fold is
    cached and rebuilt when a parameter or buffer changes.
    """

    def __init__(self, cin, cout, k, stride=1, padding=0):
        super().__init__()
        self.conv = nn.Conv2d(cin, cout, k, stride=stride, padding=padding, bias=False)
        self.bn = nn.BatchNorm2d(cout)
        self._fold = None

    def _folded(self):
        bn = self.bn
        ts = (self.conv.weight, bn.weight, bn.bias, bn.running_mean, bn.running_var)
        stamp = tuple((id(t), t._version, t.device) for t in ts)
        if self._fold is None or self._fold[0] != stamp:
            scale = bn.weight / torch.sqrt(bn.running_var + bn.eps)
            w = (self.conv.weight * scale.reshape(-1, 1, 1, 1)).detach()
            b = (bn.bias - bn.running_mean * scale).detach()
            if w.is_cuda:
                w = w.contiguous(memory_format=torch.channels_last)
            self._fold = (stamp, w, b)
        return self._fold[1], self._fold[2]

    def forward(self, x):
        if self.training or torch.is_grad_enabled():
            # the fold below is detached: with autograd on (frozen-BN fine-tuning, test-time adaptation) keep the plain
            # expression so that the convolution's parameters receive gradients, as in upstream
            return F.relu(self.bn(self.conv(x)), inplace=True)
        w, b = self._folded()
        return conv_relu(x, w, b, self.conv.stride, self.conv.padding)


class ConvBN3d(nn.Module):
    """Parameter holder for one 3-D (de)conv + BN layer of the regularization nets.

    The arithmetic runs inside the hot-path table (CUDA kernels with the BN folded in),
    so this module has no forward of its own.
    """

    def __init__(self, cin, cout, transposed=False):
        super().__init__()
        if transposed:
            self.conv = nn.ConvTranspose3d(cin, cout, 3, bias=False)
        else:
            self.conv = nn.Conv3d(cin, cout, 3, bias=False)
        self.bn = nn.BatchNorm3d(cout)
        self.transposed = transposed


class RegNet3D(nn.Module):
    """Weights of CostRegNet_2_sample_FPN3D_Fast (models/module.py:435-452)."""

    def __init__(self, cin=1, base=8):
        super().__init__()
        self.conv0 = ConvBN3d(cin, base)
        self.conv1 = ConvBN3d(base, base)
        self.conv2 = ConvBN3d(base, base * 2)
        self.conv3 = ConvBN3d(base * 2, base * 2)
        self.conv4 = ConvBN3d(base * 2, base * 4)
        self.conv5 = ConvBN3d(base * 4, base * 4)
        self.conv6 = ConvBN3d(base * 4, base * 2, transposed=True)
        self.conv7 = ConvBN3d(base * 2, base, transposed=True)
        self.prob = nn.Conv3d(base, 1, 3, stride=1, padding=1, bias=False)


class CrossScaleNet3D(nn.Module):
    """Weights of cost_up_small (models/module.py:501-508)."""

    def __init__(self, cin=1, base=8):
        super().__init__()
        self.conv0 = ConvBN3d(cin, base)
        self.conv_cost = ConvBN3d(1, base)
        self.conv1 = ConvBN3d(base * 2, base)
        self.conv2 = ConvBN3d(base, 1, transposed=True)


def _upsample2_nearest(t):
    """Nearest x2 of a channels-last map as one strided copy (F.interpolate's NHWC kernel is ~4x slower)."""
    N, C, h, w = t.shape
    v = t.permute(0, 2, 3, 1)
    v = v[:, :, None, :, None, :].expand(N, h, 2, w, 2, C).reshape(N, 2 * h, 2 * w, C)
    return v.permute(0, 3, 1, 2)


class FeaturePyramid(nn.Module):
    """P_1to8_FeatureNet_Fast (models/module.py:346-412): strides 1,2,4,8; heads at 1/8, 1/4, 1/2.

    Inference on CUDA runs an algebraically identical top-down path that never materialises the
    64-channel half-resolution map (upstream: nearest x2, 1x1 lateral conv, bias add, sum, 3x3 head =
    five passes over 600 MB at the DTU shape).  The head is linear, so
        out3(up(t) + inner2(l1)) = out3(up(t)) + (out3 o inner2)(l1) + out3(bias),
    where out3(up(t)) is four phase-specific 3x3 convolutions on the quarter-resolution map (sub-pixel
    form of a 3x3 convolution over a nearest-upsampled image; zero padding carries over exactly),
    out3 o inner2 is one composed 16->8 3x3 convolution on l1 and out3(bias) is a constant map.
    The quarter-resolution level adds the lateral 1x1 conv as one in-place addmm on the NHWC view.
    """

    def __init__(self, chans, heads):
        super().__init__()
        c0, c1, c2, c3 = chans
        self.conv0 = nn.Sequential(ConvBNReLU2d(3, c0, 3, 1, 1), ConvBNReLU2d(c0, c0, 3, 1, 1))
        self.conv1 = nn.Sequential(ConvBNReLU2d(c0, c1, 5, 2, 2), ConvBNReLU2d(c1, c1, 3, 1, 1), ConvBNReLU2d(c1, c1, 3, 1, 1))
        self.conv2 = nn.Sequential(ConvBNReLU2d(c1, c2, 5, 2, 2), ConvBNReLU2d(c2, c2, 3, 1, 1), ConvBNReLU2d(c2, c2, 3, 1, 1))
        self.conv3 = nn.Sequential(ConvBNReLU2d(c2, c3, 5, 2, 2), ConvBNReLU2d(c3, c3, 3, 1, 1), ConvBNReLU2d(c3, c3, 3, 1, 1))
        self.out1 = nn.Conv2d(c3, heads[0], 1, bias=False)
        self.inner1 = nn.Conv2d(c2, c3, 1, bias=True)
        self.inner2 = nn.Conv2d(c1, c3, 1, bias=True)
        self.out2 = nn.Conv2d(c3, heads[1], 3, padding=1, bias=False)
        self.out3 = nn.Conv2d(c3, heads[2], 3, padding=1, bias=False)
        self.fused_topdown = None     # None: on CUDA in eval mode; True / False force it
        self._heads = None
        self._bias_maps = {}

    def _head_weights(self):
        ts = (self.out3.weight, self.inner2.weight, self.inner2.bias, self.inner1.weight, self.inner1.bias)
        stamp = tuple((id(t), t._version, t.device) for t in ts)
        if self._heads is None or self._heads[0] != stamp:
            w3 = self.out3.weight.detach()                      # (O, M, 3, 3)
            O, M = w3.shape[:2]
            lateral = torch.einsum("omyx,mi->oiyx", w3, self.inner2.weight.detach()[:, :, 0, 0]).contiguous()
            # output row 2i+p reads input rows i-1, i, i+1 of the low-resolution map through kernel rows:
            #   p = 0: {ky 0 -> i-1, ky 1 -> i, ky 2 -> i};   p = 1: {ky 0 -> i, ky 1 -> i, ky 2 -> i+1}
            taps = {0: ((0, 0), (1, 1), (2, 1)), 1: ((0, 1), (1, 1), (2, 2))}
            phase = w3.new_zeros(2, 2, O, M, 3, 3)
            for py in (0, 1):
                for px in (0, 1):
                    for ky, dy in taps[py]:
                        for kx, dx in taps[px]:
                            phase[py, px, :, :, dy, dx] += w3[:, :, ky, kx]
            phase = phase.reshape(4 * O, M, 3, 3)
            w1t = self.inner1.weight.detach()[:, :, 0, 0].t().contiguous()      # (C2, M)
            if w3.is_cuda:
                lateral = lateral.contiguous(memory_format=torch.channels_last)
                phase = phase.contiguous(memory_format=torch.channels_last)
            self._heads = (stamp, lateral, phase, w1t)
            self._bias_maps = {}
        return self._heads[1:]

    def _bias_map(self, H, W):
        """out3 applied to the constant lateral bias: (1, O, H, W), differs from a constant only on the border."""
        key = (H, W)
        if key not in self._bias_maps:
            b = self.inner2.bias.detach().reshape(1, -1, 1, 1).expand(1, -1, H, W)
            self._bias_maps[key] = F.conv2d(b, self.out3.weight.detach(), padding=1)
        return self._bias_maps[key]

    def _topdown_fused(self, l1, l2, top):
        lateral, phase, w1t = self._head_weights()
        s1 = self.out1(top)
        # 1/4 level: up(top) + inner1(l2) = up(top + bias) + l2 @ W1^T, accumulated in place on the NHWC view
        t2 = _upsample2_nearest(top + self.inner1.bias.reshape(1, -1, 1, 1))
        N, M, h, w = t2.shape
        t2_rows = t2.permute(0, 2, 3, 1).reshape(-1, M)
        t2_rows.addmm_(l2.permute(0, 2, 3, 1).reshape(-1, l2.shape[1]), w1t)
        s2 = self.out2(t2)
        # 1/2 level, never materialised
        O = self.out3.weight.shape[0]
        a = F.conv2d(t2, phase, padding=1)                               # (N, 4*O, h, w), channel = (py, px, o)
        s3 = F.conv2d(l1, lateral, padding=1)                            # (N, O, 2h, 2w)
        s3_view = s3.permute(0, 2, 3, 1).reshape(N, h, 2, w, 2, O)       # (n, i, py, j, px, o)
        if s3_view.data_ptr() != s3.data_ptr():                          # not a view (unexpected layout): plain path
            return None
        s3_view += a.permute(0, 2, 3, 1).reshape(N, h, w, 2, 2, O).permute(0, 1, 3, 2, 4, 5)
        s3 += self._bias_map(2 * h, 2 * w)
        return [s1, s2, s3]

    def forward(self, x):
        l1 = self.conv1(self.conv0(x))
        l2 = self.conv2(l1)
        top = self.conv3(l2)
        fused = self.fused_topdown
        if fused is None:
            fused = x.is_cuda and not self.training and not torch.is_grad_enabled()
        if fused and l1.shape[2] == 2 * l2.shape[2] and l1.shape[3] == 2 * l2.shape[3]:
            out = self._topdown_fused(l1, l2, top)
            if out is not None:
                return out
        s1 = self.out1(top)
        top = F.interpolate(top, scale_factor=2, mode="nearest") + self.inner1(l2)
        s2 = self.out2(top)
        top = F.interpolate(top, scale_factor=2, mode="nearest") + self.inner2(l1)
        s3 = self.out3(top)
        return [s1, s2, s3]


class CostEncoder(nn.Module):
    """ProjectionInput (models/update.py:69-99)."""

    def __init__(self, cost_dim, hidden, context_dim):
        super().__init__()
        self.convc1 = nn.Conv2d(cost_dim, hidden, 1)
        self.convc2 = nn.Conv2d(hidden, hidden, 3, padding=1)
        self.convd1 = nn.Conv2d(1, hidden, 7, padding=3)
        self.convd2 = nn.Conv2d(hidden, hidden, 3, padding=1)
        self.convd = nn.Conv2d(2 * hidden, hidden - context_dim, 3, padding=1)
        self.convc = nn.Conv2d(hidden, hidden, 1)

    def forward(self, inv_depth, cost, context):
        c = _conv_relu_mod(self.convc2, _conv_relu_mod(self.convc1, cost))
        d = _conv_relu_mod(self.convd2, _conv_relu_mod(self.convd1, inv_depth))
        m = self.convd(torch.cat([c, d], dim=1))
        return _conv_relu_mod(self.convc, torch.cat([m, context], dim=1))


class GRUCell2d(nn.Module):
    """ConvGRU (models/update.py:33-49)."""

    def __init__(self, hidden, inp):
        super().__init__()
        self.convz = nn.Conv2d(hidden + inp, hidden, 3, padding=1)
        self.convr = nn.Conv2d(hidden + inp, hidden, 3, padding=1)
        self.convq = nn.Conv2d(hidden + inp, hidden, 3, padding=1)

    def forward(self, h, x):
        hx = torch.cat([h, x], dim=1)
        z = torch.sigmoid(self.convz(hx))
        r = torch.sigmoid(self.convr(hx))
        q = torch.tanh(self.convq(torch.cat([r * h, x], dim=1)))
        return (1 - z) * h + z * q


class DeltaHead(nn.Module):
    """DepthHead (models/update.py:10-27), eval mode: tanh(conv2(relu(conv1)))."""

    def __init__(self, hidden):
        super().__init__()
        self.conv1 = nn.Conv2d(hidden, hidden, 3, padding=1)
        self.conv2 = nn.Conv2d(hidden, 1, 3, padding=1)

    def forward(self, x):
        return torch.tanh(self.conv2(_conv_relu_mod(self.conv1, x)))


class UpdateBlock(nn.Module):
    """BasicUpdateBlock (models/update.py:101-141): GRU iterations that query the
    dynamic cost volume through ``cost_fn(depth)`` (the a7 hot-path row)."""

    def __init__(self, hidden, cost_dim, ratio, context_dim):
        super().__init__()
        self.encoder = CostEncoder(cost_dim, hidden, context_dim)
        self.depth_gru = GRUCell2d(hidden, hidden)
        self.depth_head = DeltaHead(hidden)
        self.mask = nn.Sequential(nn.Conv2d(hidden, hidden * 2, 3, padding=1), nn.ReLU(inplace=True),
                                  nn.Conv2d(hidden * 2, ratio * ratio * 9, 1))

    def forward(self, net, cost_fn, inv_depth, context, iters, to_depth):
        inv_seq = []
        for _ in range(iters):
            inv_depth = inv_depth.detach()
            x = self.encoder(inv_depth, cost_fn(to_depth(inv_depth)), context)
            net = self.depth_gru(net, x)
            inv_depth = inv_depth + self.depth_head(net)
            inv_seq.append(inv_depth)
        return net, 0.25 * self.mask[2](_conv_relu_mod(self.mask[0], net)), inv_seq

    def forward_fused(self, glue, net, cost_fn, inv_depth, context, iters, lo_disp, hi_disp, ctx_map=None, want_mask=True, cur_depth=None):
        return update_block_forward_fused(self, glue, net, cost_fn, inv_depth, context, iters, lo_disp, hi_disp, ctx_map, want_mask, cur_depth)


# ---- inference on CUDA: cuDNN convolutions + the glue kernels of the hot-path table ------------------
# Written against the attribute names of upstream's BasicUpdateBlock (encoder.convc1 ... mask[2]), which
# UpdateBlock shares, so that dropin.patch() can run an upstream instance through the same code.
def _fused_update_weights(block):
    g, e = block.depth_gru, block.encoder
    ts = (g.convz.weight, g.convz.bias, g.convr.weight, g.convr.bias, e.convd.bias, e.convc.weight, e.convc.bias,
          e.convc2.weight, e.convc2.bias, e.convd2.weight, e.convd2.bias, block.depth_head.conv2.weight,
          e.convd.weight, g.convq.weight, block.depth_head.conv1.weight, block.mask[0].weight)
    stamp = tuple((id(t), t._version, t.device) for t in ts)
    hit = getattr(block, "_effimvs_fused", None)
    if hit is None or hit[0] != stamp:
        cl = lambda w: w.detach().contiguous(memory_format=torch.channels_last)   # noqa: E731
        h = g.convz.out_channels
        hm = e.convd.out_channels                       # hidden - context_dim
        wc = e.convc.weight.detach()
        # convc(cat[m + b_d, context]) = Wc[:, :hm] m + (Wc[:, hm:] context + b_c + Wc[:, :hm] b_d): the second
        # term does not change over the GRU iterations
        bias_c = e.convc.bias.detach() + wc[:, :hm, 0, 0] @ e.convd.bias.detach()
        w_cd2 = wc.new_zeros(2 * h, 2 * h, 3, 3)        # block-diagonal second encoder layer: [convc2 0; 0 convd2]
        w_cd2[:h, :h] = e.convc2.weight.detach()
        w_cd2[h:, h:] = e.convd2.weight.detach()
        hit = (stamp, {
            "w_cd2": cl(w_cd2), "b_cd2": torch.cat([e.convc2.bias.detach(), e.convd2.bias.detach()]).contiguous(),
            "wzr": cl(torch.cat([g.convz.weight, g.convr.weight], dim=0)),      # one convolution for both gates
            "wc_m": cl(wc[:, :hm]), "wc_ctx": cl(wc[:, hm:]), "bias_c": bias_c.contiguous(),
            # (1, h, 3, 3) in its planar order for delta_head: a channels-last module would otherwise be re-laid out per call
            "w_d2": block.depth_head.conv2.weight.detach().contiguous()})
        object.__setattr__(block, "_effimvs_fused", hit)
    return hit[1]


def _conv_tc_enabled(glue, h, H, W):
    """Whether the update block's 3x3 convolutions run on the library's tensor-core kernel (csrc/conv2d_tc.cu: operands with
    the 11 significant bits of TF32, fp32 accumulation, gate arithmetic as epilogues) instead of cuDNN.  Follows PyTorch's own
    switch for that arithmetic class: with torch.backends.cudnn.allow_tf32 = False (fp32 products wanted) cuDNN's fp32 kernels
    stay -- unless the glue's convolutions are fp32-grade (glue.conv2d_fp32_grade: CudaHotPath(conv2d_precision='bf16x3'), hi/lo
    bf16 operands), which run either way.  EFFIMVS_CONV2D = 0 / 1 forces it off / on; by default maps below
    EFFIMVS_CONV2D_MIN_PIXELS pixels (the 1/8-resolution stage, where launch and prologue latency dominate and cuDNN is faster)
    stay on cuDNN as well."""
    env = os.environ.get("EFFIMVS_CONV2D", "auto")
    if env == "0" or not hasattr(glue, "conv2d_tc") or h % 16 != 0:
        return False
    if env != "1" and not torch.backends.cudnn.allow_tf32 and not getattr(glue, "conv2d_fp32_grade", False):
        return False
    sup = glue.conv2d_tc_supported
    if not (sup(2 * h, 2 * h) and sup(2 * h, h) and sup(h, h) and sup(h, 2 * h)):
        return False
    return env == "1" or H * W >= int(os.environ.get("EFFIMVS_CONV2D_MIN_PIXELS", "100000"))


def _tc_update_weights(block, glue, w):
    """Packed weight images of the block's six 3x3 convolutions for conv2d_tc, built once per weight set (they live in the
    dict _fused_update_weights caches, so they are rebuilt when a parameter changes).  Keyed by the glue's operand precision:
    one model may run under hot paths of different precisions, and each kernel reads only its own image format."""
    key = ("tc", getattr(glue, "conv2d_precision", "f16"))
    tc = w.get(key)
    if tc is None:
        g, e, hd = block.depth_gru, block.encoder, block.depth_head
        hm = e.convd.out_channels
        # convc (1x1, no nonlinearity in between) composed with convd: one 3x3 convolution 2h -> h
        d_prime = torch.einsum("om,miyx->oiyx", e.convc.weight.detach()[:, :hm, 0, 0], e.convd.weight.detach())
        tc = {"cd2": glue.conv2d_tc_pack(w["w_cd2"]), "dprime": glue.conv2d_tc_pack(d_prime.contiguous()),
              "zr": glue.conv2d_tc_pack(w["wzr"]), "q": glue.conv2d_tc_pack(g.convq.weight.detach()),
              "head1": glue.conv2d_tc_pack(hd.conv1.weight.detach()), "mask0": glue.conv2d_tc_pack(block.mask[0].weight.detach()),
              "b_zr": torch.cat([g.convz.bias.detach(), g.convr.bias.detach()]).contiguous()}
        w[key] = tc
    return tc


def _start_inverse_depth(glue, inv_depth, cur_depth, lo_disp, hi_disp):
    """(inv, depth) the first iteration starts from: from the stage's depth estimate in one kernel (glue.inv_init: depth_to_disp +
    disp_to_depth, Effi_MVS_plus.py:138-164) when the caller passes it, else from the normalised inverse depth it computed."""
    if cur_depth is not None and hasattr(glue, "inv_init") and os.environ.get("EFFIMVS_INV_INIT", "1") != "0":
        return glue.inv_init(cur_depth, lo_disp, hi_disp)
    if inv_depth is None:
        lo, hi = lo_disp.reshape(-1, 1, 1, 1), hi_disp.reshape(-1, 1, 1, 1)
        inv_depth = (cur_depth.reciprocal() - lo) / ((hi - lo) + 1e-10)
    return glue.gru_delta(None, None, inv_depth, lo_disp, hi_disp)


def _update_block_forward_tc(block, glue, w, hx, ctx_term, cost_fn, inv_depth, iters, lo_disp, hi_disp, want_mask, cur_depth=None):
    """The iterations of update_block_forward_fused with every 3x3 convolution on glue.conv2d_tc: encoder tail, GRU gates and
    state update are epilogues (no encoder_tail / gru_reset / gru_update launches, cat[h, x] and cat[r * h, x] never
    materialised).  hx (B,2h,H,W) channels-last holds [h ; x]; ctx_term (B,h,H,W) = convc's context half + bias."""
    from . import capi
    g, e, hd = block.depth_gru, block.encoder, block.depth_head
    tc = _tc_update_weights(block, glue, w)
    B, two_h, H, W = hx.shape
    h = two_h // 2
    ratio = int(round((block.mask[2].out_channels / 9) ** 0.5))
    mk = lambda c: torch.empty(B, c, H, W, device=hx.device, dtype=torch.float32, memory_format=torch.channels_last)   # noqa: E731
    cd, z, rh, t1 = mk(two_h), mk(h), mk(h), mk(h)
    net_v, x_v = hx[:, :h], hx[:, h:]
    # the one layer without an epilogue to fuse (block-diagonal convc2 | convd2 + relu) can stay on cuDNN: EFFIMVS_CONV2D_CD2=cudnn
    cd2_cudnn = os.environ.get("EFFIMVS_CONV2D_CD2", "own") == "cudnn"
    inv, depth = _start_inverse_depth(glue, inv_depth, cur_depth, lo_disp, hi_disp)
    inv_seq, depth_seq = [], []
    for it in range(iters):
        c1d1 = glue.encoder_head(cost_fn(depth, it), inv, e.convc1.weight, e.convc1.bias, e.convd1.weight, e.convd1.bias)
        if cd2_cudnn:
            cd = conv_relu(c1d1, w["w_cd2"], w["b_cd2"], (1, 1), (1, 1))
        else:
            glue.conv2d_tc(c1d1, None, tc["cd2"], w["b_cd2"], two_h, capi.CONV2D_BIAS_RELU, cd, None, None)
        glue.conv2d_tc(cd, None, tc["dprime"], None, h, capi.CONV2D_ADD_RELU, x_v, ctx_term, None)          # x = relu(convc(cat[convd(cd), ctx]))
        glue.conv2d_tc(hx, None, tc["zr"], tc["b_zr"], two_h, capi.CONV2D_GRU_GATES, rh, net_v, z)          # z, r * h
        glue.conv2d_tc(rh, x_v, tc["q"], g.convq.bias, h, capi.CONV2D_GRU_UPDATE, net_v, z, None)           # h = (1 - z) h + z tanh(q)
        glue.conv2d_tc(net_v, None, tc["head1"], hd.conv1.bias, h, capi.CONV2D_BIAS_RELU, t1, None, None)
        inv, depth = glue.delta_head(t1, w["w_d2"], hd.conv2.bias, inv, lo_disp, hi_disp)
        inv_seq.append(inv)
        depth_seq.append(depth)
    m0 = mk(two_h)
    glue.conv2d_tc(net_v, None, tc["mask0"], block.mask[0].bias, two_h, capi.CONV2D_BIAS_RELU, m0, None, None)
    mask_pre = F.conv2d(m0, block.mask[2].weight, None)
    up, depth_up = glue.convex_upsample(mask_pre, block.mask[2].bias, 0.25, inv, lo_disp, hi_disp, ratio)
    return net_v, inv_seq, depth_seq, up, depth_up, (mask_pre if want_mask else None)


def update_block_forward_fused(block, glue, net, cost_fn, inv_depth, context, iters, lo_disp, hi_disp, ctx_map=None, want_mask=True,
                               cur_depth=None):
    """Same arithmetic as BasicUpdateBlock.forward (models/update.py:114-141) + upsample_depth + disp_to_depth
    (Effi_MVS_plus.py:138-178), with the elementwise chains between the convolutions replaced by
    glue.encoder_head / gru_reset / gru_update / gru_delta / convex_upsample.  cost_fn(depth, iteration).
    ctx_map (B,h+cx,H,W): the context network's raw output map; when given, net = tanh(ctx_map[:, :h]) and
    context = relu(ctx_map[:, h:]) (Effi_MVS_plus.py:464-466) are formed inside the glue kernels and the net / context
    arguments are ignored.
    Returns (net, inv_seq, depth_seq, inv_up (B,rH,rW), depth_up (B,rH,rW), mask_pre (B,9rr,H,W) without bias; None
    unless want_mask)."""
    w = _fused_update_weights(block)
    g, e, hd = block.depth_gru, block.encoder, block.depth_head
    ratio = int(round((block.mask[2].out_channels / 9) ** 0.5))
    h = g.convz.out_channels
    cx = e.convc.in_channels - e.convd.out_channels                  # context channels
    tail_ctx = hasattr(glue, "encoder_tail_ctx") and cx in (4, 8, 12) and os.environ.get("EFFIMVS_TAIL_CTX", "1") != "0"
    fused_start = ctx_map is not None and tail_ctx and hasattr(glue, "gru_init") and ctx_map.shape[1] == h + cx and h % 4 == 0
    Hm, Wm = (ctx_map if ctx_map is not None else net).shape[2:]
    tc_path = _conv_tc_enabled(glue, h, Hm, Wm) and tuple(hd.conv2.weight.shape) == (1, h, 3, 3) and h <= 128
    if fused_start and tc_path and hasattr(glue, "gru_init_ctx") and os.environ.get("EFFIMVS_INIT_CTX", "1") != "0":
        # start state and the iteration-invariant context term of the encoder tail in one pass over the context map
        hx, ctx_term = glue.gru_init_ctx(ctx_map, h, w["wc_ctx"], w["bias_c"])
        return _update_block_forward_tc(block, glue, w, hx, ctx_term, cost_fn, inv_depth, iters, lo_disp, hi_disp, want_mask, cur_depth)
    if fused_start:
        hx = glue.gru_init(ctx_map, h)                               # hx[:, :h] = tanh(hidden half)
        net = hx[:, :h]
        ctx_src, ctx_off, ctx_relu = ctx_map, h, True
    else:
        if ctx_map is not None:
            hidden, context = torch.split(ctx_map, [h, ctx_map.shape[1] - h], dim=1)
            net, context = torch.tanh(hidden), torch.relu(context)
        B, _, H, W = net.shape
        hx = torch.empty(B, 2 * h, H, W, device=net.device, dtype=net.dtype, memory_format=torch.channels_last)
        hx[:, :h] = net
        ctx_src = context.contiguous(memory_format=torch.channels_last) if (tail_ctx and context.is_cuda) else context
        ctx_off, ctx_relu = 0, False
    if tc_path:
        ctx_in = torch.relu(ctx_src[:, ctx_off:ctx_off + cx]) if ctx_relu else (ctx_src if ctx_src.shape[1] == cx else ctx_src[:, ctx_off:ctx_off + cx])
        ctx_term = F.conv2d(ctx_in, w["wc_ctx"], w["bias_c"]).contiguous(memory_format=torch.channels_last)
        return _update_block_forward_tc(block, glue, w, hx, ctx_term, cost_fn, inv_depth, iters, lo_disp, hi_disp, want_mask, cur_depth)
    if not tail_ctx:
        ctx_term = F.conv2d(context, w["wc_ctx"], w["bias_c"])
    inv, depth = _start_inverse_depth(glue, inv_depth, cur_depth, lo_disp, hi_disp)
    inv_seq, depth_seq = [], []
    head_fused = (hasattr(glue, "delta_head") and h % 16 == 0 and h <= 128 and tuple(hd.conv2.weight.shape) == (1, h, 3, 3)
                  and os.environ.get("EFFIMVS_DELTA_HEAD", "1") != "0")
    for it in range(iters):
        c1d1 = glue.encoder_head(cost_fn(depth, it), inv, e.convc1.weight, e.convc1.bias, e.convd1.weight, e.convd1.bias)
        cd = conv_relu(c1d1, w["w_cd2"], w["b_cd2"], (1, 1), (1, 1))
        m = F.conv2d(cd, e.convd.weight, None, padding=1)
        if tail_ctx:       # hx[:, h:] = relu(Wm m + Wctx context + bias): the context term is formed in the kernel
            glue.encoder_tail_ctx(m, w["wc_m"], ctx_src, ctx_off, cx, ctx_relu, w["wc_ctx"], w["bias_c"], hx)
        else:
            glue.encoder_tail(m, w["wc_m"], ctx_term, hx)      # hx[:, h:] = relu(conv1x1(m) + ctx_term)
        zr_pre = F.conv2d(hx, w["wzr"], None, padding=1)
        rhx = glue.gru_reset(zr_pre, g.convr.bias, hx)
        q_pre = F.conv2d(rhx, g.convq.weight, None, padding=1)
        net = glue.gru_update(zr_pre, g.convz.bias, q_pre, g.convq.bias, hx)
        if head_fused:     # depth_head.conv2 (h -> 1) + tanh + step + disp_to_depth: one streaming kernel
            inv, depth = glue.delta_head(_conv_relu_mod(hd.conv1, net), w["w_d2"], hd.conv2.bias, inv, lo_disp, hi_disp)
        else:
            pre = F.conv2d(_conv_relu_mod(hd.conv1, net), hd.conv2.weight, None, padding=1)
            inv, depth = glue.gru_delta(pre, hd.conv2.bias, inv, lo_disp, hi_disp)
        inv_seq.append(inv)
        depth_seq.append(depth)
    m0 = _conv_relu_mod(block.mask[0], net)
    if (not want_mask and hasattr(glue, "convex_upsample_conv") and tuple(block.mask[2].kernel_size) == (1, 1) and m0.shape[1] % 4 == 0
            and os.environ.get("EFFIMVS_UPSAMPLE_CONV", "0") == "1"):
        # mask[2] (1x1) folded into the upsampling kernel: the 9 r^2-channel mask map is never materialised.  Opt-in:
        # measured on B200 the thread-per-pixel K x 36 product is shared-memory bound (one broadcast LDS.128 per four
        # FMAs) and the fused kernel loses 0.06 ms per DTU depth map against cuDNN's 1x1 convolution + the plain kernel.
        up, depth_up = glue.convex_upsample_conv(m0, block.mask[2].weight, block.mask[2].bias, 0.25, inv, lo_disp, hi_disp, ratio)
        return net, inv_seq, depth_seq, up, depth_up, None
    mask_pre = F.conv2d(m0, block.mask[2].weight, None)
    up, depth_up = glue.convex_upsample(mask_pre, block.mask[2].bias, 0.25, inv, lo_disp, hi_disp, ratio)
    return net, inv_seq, depth_seq, up, depth_up, mask_pre


def convex_upsample(x, mask, ratio):
    """upsample_depth (Effi_MVS_plus.py:167-178): softmax-weighted 3x3 upsampling."""
    N, _, H, W = x.shape
    m = torch.softmax(mask.view(N, 1, 9, ratio, ratio, H, W), dim=2)
    nb = F.unfold(x, [3, 3], padding=1).view(N, 1, 9, 1, 1, H, W)
    up = torch.sum(m * nb, dim=2).permute(0, 1, 4, 2, 5, 3)
    return up.reshape(N, ratio * H, ratio * W)


# ----------------------------------------------------------------------------
# the cascade
# ----------------------------------------------------------------------------
class EffiMVSPlus(nn.Module):
    """Three-stage Effi-MVS+ cascade; same constructor fields and forward contract as
    upstream (``args.ndepths``, ``args.GRUiters``, ``args.CostNum``; forward(imgs
    (B,V,3,H,W), proj_matrices {"stage1".."stage3": (B,V,2,4,4)}, depth_values (B,Dv))
    -> {"depth": 13 maps, "photometric_confidence"})."""

    RATIOS = (4, 2, 1)           # depth_interals_ratio, Effi_MVS_plus.py:316
    HIDDEN = (48, 32, 16)        # :337
    CONTEXT = (12, 8, 4)         # :338
    FEAT = (32, 16, 8)           # :350
    G = 1                        # :349

    def __init__(self, args, hotpath=None):
        super().__init__()
        self.ndepths = [int(e) for e in str(args.ndepths).split(",")]
        self.iters = [int(e) for e in str(args.GRUiters).split(",")]
        self.cost_num = int(args.CostNum)
        self.PixelwiseNet = nn.Sequential(ConvBNReLU2d(1, 16, 3, 1, 1), ConvBNReLU2d(16, 16, 3, 1, 1),
                                          ConvBNReLU2d(16, 8, 3, 1, 1), nn.Conv2d(8, 1, 1), nn.Sigmoid())
        self.feature = FeaturePyramid((8, 16, 32, 64), self.FEAT)
        self.cnet_depth = FeaturePyramid((4, 8, 16, 32), (60, 40, 20))
        blocks = [UpdateBlock(self.HIDDEN[i], self.G * self.cost_num * 2, 2, self.CONTEXT[i]) for i in range(3)]
        self.update_block_depth1, self.update_block_depth2, self.update_block_depth3 = blocks
        self.update_block = nn.ModuleList(blocks)
        self.CSP_R1, self.CSP_R2 = CrossScaleNet3D(self.G), CrossScaleNet3D(self.G)
        self.CSP_R = nn.ModuleList([self.CSP_R1, self.CSP_R2])
        self.CSP_C1, self.CSP_C2 = CrossScaleNet3D(self.G), CrossScaleNet3D(self.G)
        self.CSP_C = nn.ModuleList([self.CSP_C1, self.CSP_C2])
        self.cost_regularization = RegNet3D(self.G, 8)
        object.__setattr__(self, "_hotpath", hotpath)

    # the table is not a submodule: keep it out of state_dict / .to()
    @property
    def hotpath(self):
        hp = self._hotpath
        if hp is None:
            from .hotpath import CudaHotPath      # raises if libeffimvs.so is missing
            hp = CudaHotPath()
            object.__setattr__(self, "_hotpath", hp)
        return hp

    def set_hotpath(self, hp):
        object.__setattr__(self, "_hotpath", hp)

    def encode(self, imgs):
        """FPN over all V views in one batch -> per stage a list of V (B,C,h,w) maps."""
        B, V = imgs.shape[:2]
        x = imgs.reshape(B * V, *imgs.shape[2:])
        if x.is_cuda:
            x = x.contiguous(memory_format=torch.channels_last)   # cuDNN NHWC kernels, no layout round trips
        pyr = self.feature(x)
        return [[p.reshape(B, V, *p.shape[1:])[:, v] for v in range(V)] for p in pyr]

    def forward(self, imgs, proj_matrices, depth_values):
        return self.forward_from_features(self.encode(imgs), imgs[:, 0], proj_matrices, depth_values)

    def forward_from_features(self, feats, ref_img, proj_matrices, depth_values):
        """The cascade on already encoded views (SURVEY section 8(f) row 1: per-scene feature cache -- upstream
        re-encodes every image for each reference view that lists it as a source, Effi_MVS_plus.py:432-435).
        feats: per stage a list of V maps (B,C,h,w), the reference view first (what ``encode`` returns);
        ref_img (B,3,H,W) feeds the context network."""
        hp = self.hotpath
        imgs = ref_img
        B = imgs.shape[0]
        disp_min = depth_values[:, 0].reshape(B, 1, 1, 1)
        disp_max = depth_values[:, -1].reshape(B, 1, 1, 1)
        # x.reciprocal() is what torch evaluates for 1.0 / x (followed by a multiplication by 1.0): same bits, one
        # launch instead of two.  Everything that depends on depth_values only is formed once, here.
        planes = None
        if (hasattr(hp, "depth_ranges") and depth_values.is_cuda and not torch.is_grad_enabled()
                and os.environ.get("EFFIMVS_DEPTH_RANGES", "1") != "0"):
            # the same numbers from one kernel (bit-identical; ~16 single-element launches otherwise)
            R = hp.depth_ranges(depth_values, self.ndepths[0], [float(r) for r in self.RATIOS])
            row = lambda i: R[i * B:(i + 1) * B].reshape(B, 1, 1, 1)      # noqa: E731
            depth_far, depth_near, lo_disp, hi_disp = row(0), row(1), row(2), row(3)
            intervals = [row(4), row(5), row(6)]
            planes = R[8 * B:].reshape(B, self.ndepths[0])
        else:
            depth_far, depth_near = disp_min.reciprocal(), disp_max.reciprocal()
            unit = (disp_max - disp_min) / depth_values.size(1)
            intervals = [unit * r for r in self.RATIOS]
            lo_disp, hi_disp = depth_far.reciprocal(), depth_near.reciprocal()   # double reciprocal, as upstream rounds it

        def to_depth(inv):                      # disp_to_depth, Effi_MVS_plus.py:138-148
            return 1.0 / (lo_disp + (hi_disp - lo_disp) * inv).clamp(min=1e-4)

        ctx_pyr = self.cnet_depth(ref_img.contiguous(memory_format=torch.channels_last) if ref_img.is_cuda else ref_img)

        preds = []
        conf = None
        view_w = raw_vol = reg_vol = None
        vol_near, vol_far = depth_near, depth_far        # range of the volume the GRU reads
        for s in range(3):
            f = feats[s]
            cams = proj_matrices["stage{}".format(s + 1)]
            glue = hp if (getattr(hp, "fused_update", False) and imgs.is_cuda and not torch.is_grad_enabled()) else None
            if glue is None:
                hidden, context = torch.split(ctx_pyr[s], [self.HIDDEN[s], self.CONTEXT[s]], dim=1)
                hidden, context = torch.tanh(hidden), torch.relu(context)
            H, W = f[0].shape[2:]
            if s == 0:
                D = self.ndepths[0]
                if planes is None:
                    k = torch.arange(D, device=imgs.device, dtype=imgs.dtype).reshape(1, D)
                    inv_s = disp_min.reshape(B, 1) + k * ((disp_max - disp_min).reshape(B, 1) / (D - 1))
                    planes = inv_s.reciprocal()
                hyp = planes.reshape(B, D, 1, 1).expand(B, D, H, W)   # plane sweep: stride-0 view
                out = hp.stage1(f, cams, hyp, self.PixelwiseNet, self.cost_regularization, self.G)
                conf = F.interpolate(out["photometric_confidence"].unsqueeze(1), [H * 4, W * 4], mode="nearest").squeeze(1)
                view_w = out["view_weights"]
                raw_vol = out["volume"].squeeze(1)
                reg_vol = out["reg_volume"]
                cur_depth = out["depth"].unsqueeze(1)
                preds.append(out["depth"])
            else:
                cur_depth = preds[-1].unsqueeze(1).detach()
                view_w = F.interpolate(view_w, scale_factor=2, mode="nearest")
                D = self.ndepths[s]
                loc, hyp = hp.local_volume(cur_depth, f, cams, intervals[s], view_w, D, self.G)
                hyp_low = hyp[:, :, ::2, ::2]                 # nearest x1/2 (Effi_MVS_plus.py:514)
                loc5 = loc.reshape(B, self.G, D, H, W)
                # the two cross-scale branches (regularized / raw volume) are independent: the raw one runs on a side
                # stream when the table offers one (a parallel branch of the CUDA graph under capture)
                side = hp.side_stream(loc.device) if hasattr(hp, "side_stream") else None
                if side is not None:
                    main = torch.cuda.current_stream(loc.device)
                    side.wait_stream(main)
                    with torch.cuda.stream(side):
                        raw_prev = hp.volume_lookup(raw_vol, hyp_low, vol_near, vol_far)
                        raw_vol = hp.cross_scale(self.CSP_C[s - 1], loc5, raw_prev.unsqueeze(1)).squeeze(1)
                reg_prev = hp.volume_lookup(reg_vol, hyp_low, vol_near, vol_far)
                reg_vol = hp.cross_scale(self.CSP_R[s - 1], loc5, reg_prev.unsqueeze(1)).squeeze(1)
                if side is not None:
                    main.wait_stream(side)
                else:
                    raw_prev = hp.volume_lookup(raw_vol, hyp_low, vol_near, vol_far)
                    raw_vol = hp.cross_scale(self.CSP_C[s - 1], loc5, raw_prev.unsqueeze(1)).squeeze(1)
                vol_far, vol_near = hyp[:, 0:1], hyp[:, -1:]

            interval = intervals[s]

            def cost_fn(depth, _it=0, _raw=raw_vol, _reg=reg_vol, _iv=interval, _n=vol_near, _f=vol_far):
                return hp.dynamic_cost(depth, _raw, _reg, _iv, _n, _f, self.cost_num)

            if glue is not None:     # tanh / relu of the context map and depth_to_disp happen inside the glue kernels
                _, _, depth_seq, _, depth_up, _ = self.update_block[s].forward_fused(
                    glue, None, cost_fn, None, None, self.iters[s], lo_disp.reshape(B), hi_disp.reshape(B), ctx_pyr[s], False, cur_depth)
                preds.extend(d.squeeze(1) for d in depth_seq)
                preds.append(depth_up)
                continue
            inv0 = (cur_depth.reciprocal() - lo_disp) / ((hi_disp - lo_disp) + 1e-10)     # depth_to_disp, Effi_MVS_plus.py:151-164
            _, mask, inv_seq = self.update_block[s](hidden, cost_fn, inv0, context, self.iters[s], to_depth)
            for inv in inv_seq:
                preds.append(to_depth(inv).squeeze(1))
            up = convex_upsample(inv_seq[-1], mask, 2).unsqueeze(1)
            preds.append(to_depth(up).squeeze(1))
        return {"depth": preds, "photometric_confidence": conf}
