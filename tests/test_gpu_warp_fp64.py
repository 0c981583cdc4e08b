"""The warp + correlation kernels (csrc/warp_corr.cu, csrc/warp_tile.cu) element by element against fp64 restatements of the
operations they replace (``-m gpu``).

The kernels claim sample coordinates bit-identical to upstream's on a CUDA device (csrc/warp_coords.cuh).  So the reference
restates the coordinate chain in fp32, operation for operation: the ray rot @ (x, y, 1) in the order cuBLAS uses for the map
size (ray_unfused_for), p = ray * d + t with two roundings, the z == 0 nudge, IEEE division, u * fl(1 / fl((W-1)/2)) - 1 and
(g + 1) * (W-1)/2.  Torch's fp32 elementwise operations round as IEEE does on the CPU and on the device; the one fused
multiply-add of the chain (fma(r1, y, r0 x) in the fused ray) goes through fma32(), an exact helper.  The local hypotheses
are restated the same way from local_hypothesis().  Everything after the coordinates -- the bilinear weights of upstream's
grid_sample, zero padding, the group mean, the (weighted) mean over views, the softmax entropy -- is fp64.

Every bar is a per-element bound derived from the kernels' fp32 arithmetic (sample_bar(), agg_bar(); the entropy through
softmax_bar / entropy_bar of tests/test_gpu_glue_fp64.py), never fitted to observed error.  The bars assume exact coordinates:
a coordinate one ulp off moves a similarity by far more than they allow, so a coordinate mismatch fails.  Where a result must
be bit-identical (the hypotheses written back, forced gathers against staged samples, the restated ray against torch.matmul)
the check is exact.

The case matrix (module-level lists) covers the cascade's own calls at the DTU and Tanks & Temples stage shapes with up to 8
reference views, all 12 (C, G) instantiations of the tile, the channels-last generic and the planar aggregation kernels, the
stage-1 views kernels at every entropy branch, homo_warp, weighted_agg and geometric edge cases.  tests/test_warp_cases_host.py
restates the launch rules and the tile kernel's staging decisions on the CPU and asserts that these lists reach every branch.
Case inputs come from CPU generators, so that the host test sees the same data.
"""
import math
import zlib
from collections import namedtuple

import numpy as np
import pytest
import torch

from test_gpu_glue_fp64 import U, _planted, check, entropy_bar, gamma, softmax_bar, worst_ratio  # noqa: F401

pytestmark = pytest.mark.gpu
DEV = "cuda"

HYP_TENSOR, HYP_PLANES, HYP_LOCAL = 0, 1, 2          # include/effimvs.h (capi.HYP_*)
MODE_NAMES = {HYP_TENSOR: "tensor", HYP_PLANES: "planes", HYP_LOCAL: "local"}
RAY_UNFUSED_MAX_PIXELS = 220000                      # kRayUnfusedMaxPixels, csrc/warp_coords.cuh


def ray_unfused_for(H, W):
    """csrc/warp_coords.cuh: maps of at most 220,000 pixels form the ray without contraction, (r0 x + r1 y) + r2"""
    return H * W <= RAY_UNFUSED_MAX_PIXELS


# ---- case matrix ---------------------------------------------------------------------------------------------------
# kind: "agg" (warp_corr_agg) or "views" (warp_corr_views; at stage shapes followed by weighted_agg)
# layout: "tile" (channels-last, 32-byte aligned), "nhwc" (channels-last, source 0 offset by 4 floats: the generic kernel),
#         "planar" (NCHW)
# geom: how the cameras and hypotheses are built (make_inputs)
Case = namedtuple("Case", "kind H W B n C G D mode weighted layout geom")


def case_id(c):
    return "{}-{}x{}-B{}-n{}-C{}G{}-D{}-{}{}-{}-{}".format(c.kind, c.H, c.W, c.B, c.n, c.C, c.G, c.D, MODE_NAMES[c.mode],
                                                         "-w" if c.weighted else "", c.layout, c.geom)


LAYOUTS = ("tile", "nhwc", "planar")
BATCHES = (1, 2, 8)
# the cascade's calls: (kind, H, W, n, C, D, mode); stage 1 = views + weighted_agg, stages 2 / 3 = local hypotheses, G = 1
STAGES = {"dtu": [("views", 148, 200, 4, 32, 48, HYP_PLANES), ("agg", 296, 400, 4, 16, 8, HYP_LOCAL),
                  ("agg", 592, 800, 4, 8, 8, HYP_LOCAL)],
          "tanks": [("views", 132, 240, 6, 32, 96, HYP_PLANES), ("agg", 264, 480, 6, 16, 8, HYP_LOCAL),
                    ("agg", 528, 960, 6, 8, 8, HYP_LOCAL)]}
STAGE_CASES = [Case(k, H, W, B, n, C, 1, D, mode, True, layout, "normal") for ds in ("dtu", "tanks")
               for (k, H, W, n, C, D, mode) in STAGES[ds] for B in BATCHES for layout in ("tile", "planar")]


def _instance_cases():
    """all 12 (C, G) pairs on each aggregation path at 37 x 53 (partial 32 x 4 tiles and 128-pixel blocks), rotating through
    the hypothesis modes, with and without weights; D % 8 != 0 and D % 4 != 0, or D = 1 (not for LOCAL, which needs D > 1)"""
    out, i = [], 0
    for layout in LAYOUTS:
        for C in (8, 16, 32):
            for G in (1, 2, 4, 8):
                mode = (HYP_TENSOR, HYP_PLANES, HYP_LOCAL)[i % 3]
                D = 1 if (mode != HYP_LOCAL and i % 4 == 0) else (5, 11, 13, 7)[i % 4]
                out.append(Case("agg", 37, 53, 2, 3, C, G, D, mode, (i // 3) % 2 == 0, layout, "normal"))
                i += 1
    return out


INSTANCE_CASES = _instance_cases()
# (H, W, B, n, C, G, D, mode, weighted, geom) -- run on every layout
_EDGE = [(2, 131, 2, 3, 8, 1, 7, HYP_TENSOR, True, "normal"),
         (131, 2, 2, 3, 16, 2, 7, HYP_PLANES, False, "normal"),
         (2, 2, 2, 3, 8, 2, 5, HYP_LOCAL, True, "normal"),
         (37, 53, 2, 1, 16, 1, 9, HYP_PLANES, True, "normal"),
         (37, 53, 2, 16, 8, 1, 8, HYP_TENSOR, True, "normal"),
         (37, 53, 8, 3, 8, 1, 8, HYP_LOCAL, True, "normal"),
         (37, 53, 2, 2, 16, 4, 8, HYP_PLANES, True, "identity"),
         (37, 53, 2, 3, 8, 1, 16, HYP_PLANES, True, "both_sides"),
         (37, 53, 2, 2, 8, 1, 8, HYP_PLANES, False, "z0"),
         (37, 53, 2, 3, 8, 1, 8, HYP_TENSOR, True, "offimage"),
         (37, 53, 2, 4, 16, 1, 16, HYP_PLANES, True, "offimage"),
         (37, 53, 2, 3, 16, 1, 16, HYP_PLANES, True, "wide"),
         (96, 160, 2, 4, 8, 1, 16, HYP_TENSOR, True, "wide"),
         (37, 53, 2, 3, 32, 4, 8, HYP_TENSOR, True, "special"),
         (37, 53, 2, 3, 8, 2, 8, HYP_PLANES, False, "special"),
         (37, 53, 2, 3, 16, 1, 8, HYP_LOCAL, True, "special"),
         (37, 53, 2, 3, 16, 2, 16, HYP_TENSOR, True, "unordered")]
EDGE_CASES = [Case("agg", H, W, B, n, C, G, D, mode, wt, layout, geom) for (H, W, B, n, C, G, D, mode, wt, geom) in _EDGE
              for layout in LAYOUTS]
VIEWS_D = (1, 7, 48, 49, 96, 97, 385, 1024)
VIEWS_CASES = [Case("views", 37, 53, 2, 2, C, 1, D, HYP_TENSOR if D % 2 else HYP_PLANES, False, layout, "normal")
               for C in (8, 16, 32) for layout in LAYOUTS for D in VIEWS_D] + \
              [Case("views", H, W, B, n, C, 1, D, mode, False, layout, geom)
               for (H, W, B, n, C, D, mode, geom) in ((2, 131, 2, 3, 8, 9, HYP_TENSOR, "normal"),
                                                      (37, 53, 8, 3, 16, 16, HYP_TENSOR, "special"),
                                                      (37, 53, 2, 16, 8, 8, HYP_PLANES, "normal"),
                                                      (37, 53, 2, 3, 8, 16, HYP_PLANES, "both_sides"),
                                                      (37, 53, 2, 3, 32, 16, HYP_PLANES, "wide"),
                                                      (37, 53, 2, 3, 8, 8, HYP_TENSOR, "offimage"))
               for layout in LAYOUTS]
AGG_CASES = [c for c in STAGE_CASES if c.kind == "agg"] + INSTANCE_CASES + EDGE_CASES
ALL_VIEWS_CASES = [c for c in STAGE_CASES if c.kind == "views"] + VIEWS_CASES
# homo_warp (C, mode, H, W, D): every channel count at B = 2, and the edge shapes
HOMO_CASES = [(C, mode, 37, 53, 7) for C in (1, 3, 8, 64) for mode in (HYP_TENSOR, HYP_PLANES)] + \
             [(3, HYP_TENSOR, H, W, 5) for (H, W) in ((2, 131), (131, 2), (2, 2))] + [(8, HYP_PLANES, 592, 800, 3)]
# weighted_agg (n_src, D): gridDim.y = min(D, 8), so D > 8 takes several passes over the planes
WAGG_CASES = [(n, D) for n in (1, 4, 6, 16) for D in (1, 5, 8, 48, 96)]


# ---- the fp32 restatement of the coordinates -----------------------------------------------------------------------
def fma32(a, b, c):
    """fma(a, b, c) of fp32 tensors rounded once to fp32.  a * b is exact in fp64 (24 + 24 bits); s = fl64(a b + c) and the
    exact residual r = (a b + c) - s (TwoSum) describe the exact sum.  Rounding s to fp32 is correct unless s lies exactly
    halfway between two fp32 neighbours and r != 0: then the exact sum lies on the side of r."""
    a, b, c = a.double(), b.double(), c.double()
    p = a * b
    s = p + c
    bb = s - p
    r = (p - (s - bb)) + (c - bb)
    f = s.float()
    fd = f.double()
    nb = torch.nextafter(f, torch.where(s > fd, torch.full_like(f, math.inf), torch.full_like(f, -math.inf)))
    mid = (fd != s) & ((fd + nb.double()) * 0.5 == s)
    fix = mid & (r != 0) & ((r > 0) == (nb.double() > fd))
    return torch.where(fix, nb, f)


def pixel_grid(H, W, device):
    k = torch.arange(H * W, device=device)
    return (k % W).float(), torch.div(k, W, rounding_mode="floor").float()


def restate_rays(proj, H, W):
    """rot @ (x, y, 1) of every (batch, view, pixel) as the kernels form it (make_ray): (B, V, 3, HW) fp32"""
    x, y = pixel_grid(H, W, proj.device)
    rows = []
    for r in range(3):
        p0, p1, p2 = (proj[:, :, 3 * r + i].unsqueeze(-1) for i in range(3))
        if ray_unfused_for(H, W):
            rows.append(((p0 * x) + (p1 * y)) + p2)
        else:
            rows.append(fma32(p1, y, p0 * x) + p2)
    return torch.stack(rows, 2)


def inv_half(n):
    """fl(1 / fl((n - 1) / 2)) (an IEEE single division, as the kernels' __fdiv_rn and the host's WarpConsts)"""
    return float(np.float32(1.0) / np.float32((n - 1) / 2.0))


def restate_coords(ray, trans, depth, H, W):
    """sample_coords(): ray (B, 3, HW) and trans (B, 3) of one view, depth (B, Dc, HW) -> (ix, iy), each (B, Dc, HW) fp32"""
    r = [ray[:, i].unsqueeze(1) for i in range(3)]
    t = [trans[:, i].reshape(-1, 1, 1) for i in range(3)]
    px, py, pz = ((r[i] * depth) + t[i] for i in range(3))
    pz = torch.where(pz == 0, pz + 1e-8, pz)
    u, v = px / pz, py / pz
    gx, gy = (u * inv_half(W)) - 1.0, (v * inv_half(H)) - 1.0
    return (gx + 1.0) * (0.5 * (W - 1)), (gy + 1.0) * (0.5 * (H - 1))


def restate_local(cur, interval, D):
    """local_hypothesis() for every plane: cur (B, H, W), interval (B,) -> (B, D, HW) fp32 (fmaxf / fminf ignore NaN, as
    torch.fmax / fmin do)"""
    B = cur.shape[0]
    c = cur.reshape(B, 1, -1)
    one = torch.ones_like(c)
    inv = one / c
    half = interval.reshape(B, 1, 1) * float(D // 2)
    lo = torch.fmax(inv - half, torch.full_like(c, 1e-4))
    hi = torch.fmin(torch.fmax(inv + half, torch.full_like(c, 1e-4)), torch.full_like(c, 1e4))
    step = (hi - lo) * float(np.float32(1.0) / np.float32(D - 1))
    d = torch.arange(D, device=cur.device, dtype=torch.float32).reshape(1, D, 1)
    s = torch.fmax(lo + (d * step), torch.full_like(lo + d, 1e-5))
    return torch.ones_like(s) / s


def restate_depth(c, hyp, interval):
    """the hypotheses the kernels read (fetch_hypothesis), (B, D, HW) fp32"""
    HW = c.H * c.W
    if c.mode == HYP_TENSOR:
        return hyp.reshape(c.B, c.D, HW)
    if c.mode == HYP_PLANES:
        return hyp.reshape(c.B, c.D, 1).expand(c.B, c.D, HW)
    return restate_local(hyp, interval, c.D)


def same(a, b):
    """bit-level agreement up to the NaN payload"""
    return a.shape == b.shape and bool(((a == b) | (torch.isnan(a) & torch.isnan(b))).all())


# ---- the fp64 reference after the coordinates ------------------------------------------------------------------------
def interp(flat, b_off, ix, iy, H, W):
    """grid_sample (bilinear, zeros, align_corners=True) of channels-last rows flat (B*HW, C) fp64 at fp32 positions:
    upstream's weights (x1 - ix)(y1 - iy), ... in fp64, taps outside the image (and NaN / inf positions) contribute 0.
    Returns (value, sum |w v|), each (B, Dc, HW, C)."""
    ix, iy = ix.double(), iy.double()
    fx, fy = torch.floor(ix), torch.floor(iy)
    wx = ((fx + 1) - ix, ix - fx)
    wy = ((fy + 1) - iy, iy - fy)
    val, aval = 0.0, 0.0
    for dy in (0, 1):
        for dx in (0, 1):
            xx, yy = fx + dx, fy + dy
            ok = (xx >= 0) & (xx <= W - 1) & (yy >= 0) & (yy <= H - 1)
            idx = torch.where(ok, b_off + yy * W + xx, torch.zeros_like(xx)).long()
            w = torch.where(ok, wx[dx] * wy[dy], torch.zeros_like(xx)).unsqueeze(-1)
            v = flat[idx]
            val = val + w * v
            aval = aval + w.abs() * v.abs()
    return val, aval


def _chunk(B, HW, C):
    return max(1, (1 << 24) // (B * HW * C))


def sample_bar(abs_terms, CG):
    """One sample's group correlation (1/CG) sum_c ref_c sum_tap w_tap v_tap,c.  The tap weights are products of two axis
    weights, each of which may round once (fl(fl(x0 + 1) - ix), fl(ix - x0)): 3 roundings.  Then the longest path over the
    three kernel orders:
      tile (warp_tile.cu)      4-tap FMA chain (4), packed per-pair FMA chain over CG/2 channels (CG/2), lo + hi (1);
      planar (warp_corr.cu)    4-tap FMA chain (4), per-channel FMA chain over CG channels (CG);
      NHWC generic             per-tap dot over CG channels (CG), FMA with the tap weight over the 4 taps (4);
    at most 3 + 4 + CG = CG + 7 roundings (CG >= 1); the scaling by 1/CG is exact.  |err| <= gamma_{CG+7} sum |w v ref| / CG."""
    return gamma(CG + 7) * abs_terms


def view_sims(c, ref, srcs, proj, depth):
    """per source view: (sim, bar), each (B, G, D, HW) fp64"""
    B, C, H, W, G, D = c.B, c.C, c.H, c.W, c.G, c.D
    HW, CG = H * W, C // G
    rays = restate_rays(proj, H, W)
    refd = ref.double().permute(0, 2, 3, 1).reshape(B, 1, HW, C)
    b_off = (torch.arange(B, device=ref.device, dtype=torch.float64) * HW).reshape(B, 1, 1)
    dc = _chunk(B, HW, C)
    for v in range(len(srcs)):
        flat = srcs[v].double().permute(0, 2, 3, 1).reshape(B * HW, C)
        sim = torch.empty(B, G, D, HW, dtype=torch.float64, device=ref.device)
        bar = torch.empty_like(sim)
        for d0 in range(0, D, dc):
            ix, iy = restate_coords(rays[:, v], proj[:, v, 9:], depth[:, d0:d0 + dc], H, W)
            val, aval = interp(flat, b_off, ix, iy, H, W)
            n = val.shape[1]
            s = (val * refd).reshape(B, n, HW, G, CG).sum(-1) / CG
            a = (aval * refd.abs()).reshape(B, n, HW, G, CG).sum(-1) / CG
            sim[:, :, d0:d0 + n] = s.permute(0, 3, 1, 2)
            bar[:, :, d0:d0 + n] = sample_bar(a, CG).permute(0, 3, 1, 2)
        yield sim, bar


def agg_bar(num, err_num, abs_num, den, abs_den, n, weighted):
    """the aggregation over n views of similarities known to within err_v each.  Weighted: sum fl(fl(sim_v w_v) + num) over
    the views (a product and n - 1 additions: gamma_n sum |sim_v w_v|, plus sum |w_v| err_v carried by the products, with
    gamma_n on it too), the denominator sum w_v + 1e-6 (n additions: gamma_n (sum |w_v| + 1e-6)), one division (u);
    first order in the quotient, 1 % margin.  Unweighted: n - 1 additions, division by n.
    num, den: fp64 sums; err_num = sum |w_v| err_v; abs_num = sum |w_v sim_v|; abs_den = sum |w_v|."""
    if weighted:
        dd = den + 1e-6
        q = num / dd
        e_num = err_num * (1 + gamma(n)) + gamma(n) * abs_num
        e_den = gamma(n) * (abs_den + 1e-6)
        return q, 1.01 * ((e_num + q.abs() * e_den) / dd.abs()) + 1.01 * U * q.abs()
    q = num / n
    return q, 1.01 * (err_num * (1 + gamma(n)) + gamma(max(n - 1, 0)) * abs_num) / n + U * q.abs()


def agg_reference(c, ref, srcs, proj, depth, weights):
    """warp_corr_agg in fp64: (B, G, D, HW) value and bar"""
    HW = c.H * c.W
    num = err = absn = 0.0
    den = absd = 0.0
    for v, (s, e) in enumerate(view_sims(c, ref, srcs, proj, depth)):
        w = weights[:, v].double().reshape(c.B, 1, 1, HW) if weights is not None else 1.0
        wa = w.abs() if weights is not None else 1.0
        num = num + s * w
        err = err + e * wa
        absn = absn + (s * w).abs()
        den = den + w
        absd = absd + wa
    return agg_bar(num, err, absn, den, absd, len(srcs), weights is not None)


# ---- inputs ----------------------------------------------------------------------------------------------------------
def _rotation(a):
    k = torch.zeros(3, 3, dtype=torch.float64)
    k[0, 1], k[0, 2], k[1, 2] = -a[2], a[1], -a[0]
    return torch.linalg.matrix_exp(k - k.T)


def make_proj(g, geom, B, n, H, W):
    """(B, n, 12) fp32: rot = K R K^-1 (row major) and trans = K t of source cameras around a reference camera with focal
    length 1.2 max(H, W), different for every (batch entry, view).  Depths are DTU-like (425 .. 935).
      normal     baselines of 40, rotations of ~0.02 rad
      wide       baselines of 300: tile footprints beyond the staged box, staged and gathered samples mixed
      identity   the reference camera as source: samples at the pixel centres
      both_sides the source camera 650 in front of the reference: planes on both sides of it (z changes sign)
      z0         rz = 1, tz = -650, tiny rx, ry: z is exactly 0 on the 650 plane and the 1e-8 nudge decides the sample
      offimage   source view 1 moved ten widths to the right of the image: a round that stages nothing"""
    if geom == "identity":
        return torch.tensor([1, 0, 0, 0, 1, 0, 0, 0, 1, 0, 0, 0], dtype=torch.float32).repeat(B, n, 1)
    if geom == "z0":
        a = float(np.float32(0.5 / (650.0 * 1e8)))
        return torch.tensor([a, 0, 0, 0, a, 0, 0, 0, 1, 0, 0, -650.0], dtype=torch.float32).repeat(B, n, 1)
    f = 1.2 * max(H, W)
    K = torch.tensor([[f, 0, (W - 1) / 2], [0, f, (H - 1) / 2], [0, 0, 1]], dtype=torch.float64)
    Ki = torch.linalg.inv(K)
    base = 300.0 if geom == "wide" else 40.0
    P = torch.empty(B, n, 12, dtype=torch.float64)
    for b in range(B):
        for v in range(n):
            r = torch.randn(6, generator=g, dtype=torch.float64)
            R = _rotation(0.02 * r[:3])
            t = base * torch.stack([(-1.0) ** v * (1 + 0.2 * r[3]), 0.3 * r[4], 0.05 * r[5]])
            if geom == "both_sides":
                t[2] = -650.0
            rot, tr = K @ R @ Ki, K @ t
            if geom == "offimage" and v == 1:
                rot[0] += 10 * W * rot[2]
                tr[0] += 10 * W * tr[2]
            P[b, v, :9], P[b, v, 9:] = rot.reshape(9), tr
    return P.float()


def _planes(B, D):
    """(B, D) depths uniform in inverse depth over a range that differs per batch entry"""
    dmin = 425.0 - 10.0 * torch.arange(B, dtype=torch.float64)
    dmax = 935.0 + 25.0 * torch.arange(B, dtype=torch.float64)
    if D == 1:
        return (0.5 * (dmin + dmax)).reshape(B, 1)
    k = torch.arange(D, dtype=torch.float64) / (D - 1)
    return 1.0 / (1.0 / dmax.reshape(B, 1) + k * (1.0 / dmin - 1.0 / dmax).reshape(B, 1))


def make_hyp(g, c):
    """(hyp, interval) as the kernels read them; geom "special" plants NaN, +-inf, 0, negative and tiny hypotheses, "unordered"
    permutes the planes of every pixel, "z0" puts a plane exactly at 650"""
    B, D, H, W = c.B, c.D, c.H, c.W
    planes = _planes(B, D)
    if c.mode == HYP_PLANES:
        hyp = planes.float()
        if c.geom == "z0":
            hyp[:, D // 2] = 650.0
        if c.geom == "special":
            hyp[0, 1], hyp[-1, 2], hyp[0, 3], hyp[-1, 4], hyp[0, 5] = 0.0, -500.0, math.nan, math.inf, -math.inf
        return hyp.contiguous(), None
    if c.mode == HYP_TENSOR:
        hyp = (planes.reshape(B, D, 1, 1) * (1 + 0.02 * torch.randn(B, D, H, W, generator=g, dtype=torch.float64))).float()
        hyp = _planted(hyp).abs()
        if c.geom == "unordered":
            hyp = hyp.gather(1, torch.argsort(torch.rand(B, D, H, W, generator=g), dim=1))
        if c.geom == "special":
            vals = torch.tensor([math.nan, math.inf, -math.inf, 0.0, -600.0, -1.0, 1e-30, 1e30])
            hyp[:, 0, 0, :8] = vals
            hyp[:, D - 1, 1, 3:11] = vals
            hyp[:, D // 2, H - 1, W - 8:] = vals
        return hyp.contiguous(), None
    cur = _planted(425.0 + 510.0 * torch.rand(B, H, W, generator=g)).abs()
    if c.geom == "special":
        cur[:, 0, :6] = torch.tensor([0.0, -500.0, math.nan, math.inf, 1e-30, -math.inf])
    interval = ((1 / 425.0 - 1 / 935.0) / (4 * D)) * (1 + 0.1 * torch.arange(B, dtype=torch.float32))
    return cur.contiguous(), interval.float()


def make_inputs(c):
    """(ref, srcs, proj, hyp, interval, weights) of a case on the CPU, from a generator seeded by the case"""
    g = torch.Generator().manual_seed(zlib.crc32(repr(tuple(c)).encode()))
    ref = _planted(torch.randn(c.B, c.C, c.H, c.W, generator=g))
    srcs = [_planted(torch.randn(c.B, c.C, c.H, c.W, generator=g)) for _ in range(c.n)]
    proj = make_proj(g, c.geom, c.B, c.n, c.H, c.W)
    hyp, interval = make_hyp(g, c)
    weights = (0.1 + torch.rand(c.B, c.n, c.H, c.W, generator=g)) if c.weighted else None
    return ref, srcs, proj, hyp, interval, weights


def to_layout(t, layout, offset=False):
    """planar (NCHW), channels-last, or channels-last starting 4 floats (16 bytes) into a buffer: 16- but not 32-byte aligned"""
    if layout == "planar":
        return t.contiguous()
    if not offset:
        return t.contiguous(memory_format=torch.channels_last)
    B, C, H, W = t.shape
    buf = torch.empty(B * C * H * W + 4, device=t.device)
    out = buf[4:].view(B, H, W, C).permute(0, 3, 1, 2)
    out.copy_(t)
    return out


def feature_maps(c, ref, srcs):
    """the maps in the case's layout; "nhwc" offsets source 0 so that the dispatcher takes the generic channels-last kernel"""
    r = to_layout(ref, c.layout)
    s = [to_layout(t, c.layout, offset=(c.layout == "nhwc" and i == 0)) for i, t in enumerate(srcs)]
    if c.layout != "planar":
        assert all(t.is_contiguous(memory_format=torch.channels_last) and not t.is_contiguous() for t in [r] + s)
        assert r.data_ptr() % 32 == 0 and all(t.data_ptr() % 32 == (16 if c.layout == "nhwc" and i == 0 else 0)
                                             for i, t in enumerate(s))
    return r, s


# ---- fixtures --------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module", autouse=True)
def _strict_fp32():
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.set_grad_enabled(False)
    yield


@pytest.fixture
def record(record_property):
    return lambda name, ratio: record_property("ratio:" + name, "{:.4g}".format(ratio))


def _device(inputs):
    ref, srcs, proj, hyp, interval, weights = inputs
    mv = lambda t: t.to(DEV) if t is not None else None    # noqa: E731
    return mv(ref), [mv(s) for s in srcs], mv(proj), mv(hyp), mv(interval), mv(weights)


def _check_ray_vs_matmul(c, proj):
    """at B = 1: the restated ray equals upstream's torch.matmul(rot, xyz) on the device bit for bit (cuBLAS's order)"""
    x, y = pixel_grid(c.H, c.W, proj.device)
    xyz = torch.stack((x, y, torch.ones_like(x))).unsqueeze(0)
    rays = restate_rays(proj, c.H, c.W)
    for v in range(c.n):
        want = torch.matmul(proj[:, v, :9].reshape(1, 3, 3), xyz)
        assert torch.equal(rays[:, v], want), ("ray order", ray_unfused_for(c.H, c.W), v)


# ---- warp_corr_agg ---------------------------------------------------------------------------------------------------
def _agg(c, ref, srcs, proj, hyp, interval, weights):
    from effimvs_b200 import ops
    return ops.warp_corr_agg(ref, srcs, proj, hyp, c.mode, interval, weights, c.D, c.G, True)


@pytest.mark.parametrize("c", AGG_CASES, ids=[case_id(c) for c in AGG_CASES])
def test_warp_corr_agg_vs_fp64(c, record, monkeypatch):
    """warp_corr_agg (tile, NHWC generic or planar kernel by layout) against the fp64 aggregation of the restated samples;
    the hypotheses it writes back bit for bit; on the tile path, every sample gathered from global memory
    (EFFIMVS_WARP_FORCE_GATHER=1, read per call) bit for bit equal to the staged run."""
    monkeypatch.delenv("EFFIMVS_WARP_FORCE_GATHER", raising=False)
    ref, srcs, proj, hyp, interval, weights = _device(make_inputs(c))
    r, s = feature_maps(c, ref, srcs)
    HW = c.H * c.W
    # a run with different data first: an element the kernel skips then holds a stale, wrong value
    _agg(c, to_layout(-r + 0.5, c.layout), s[::-1], proj, hyp, interval, weights)
    sim, hyp_out = _agg(c, r, s, proj, hyp, interval, weights)
    depth = restate_depth(c, hyp, interval)
    assert same(hyp_out.reshape(c.B, c.D, HW), depth), "hypotheses written back"
    want, bar = agg_reference(c, ref, srcs, proj, depth, weights)
    check("warp_corr_agg." + c.layout, sim.reshape(c.B, c.G, c.D, HW), want, bar, record)
    if c.layout == "tile":
        monkeypatch.setenv("EFFIMVS_WARP_FORCE_GATHER", "1")
        sim_g, hyp_g = _agg(c, r, s, proj, hyp, interval, weights)
        monkeypatch.delenv("EFFIMVS_WARP_FORCE_GATHER")
        assert same(sim_g, sim) and same(hyp_g, hyp_out), "gathered samples differ from staged ones"
    if c.B == 1 and c in STAGE_CASES:
        _check_ray_vs_matmul(c, proj)


# ---- warp_corr_views (+ weighted_agg at the stage shapes) --------------------------------------------------------------
def _views(c, ref, srcs, proj, hyp):
    from effimvs_b200 import ops
    return ops.warp_corr_views(ref, srcs, proj, hyp, c.mode, c.D)


@pytest.mark.parametrize("c", ALL_VIEWS_CASES, ids=[case_id(c) for c in ALL_VIEWS_CASES])
def test_warp_corr_views_vs_fp64(c, record, monkeypatch):
    """warp_corr_views: every view's similarities against fp64 and their softmax entropy over D (the tile path's reg48 /
    reg96 / generic entropy kernels, the generic kernel's in-kernel entropy, whose shared memory exceeds 48 KB above D = 384)
    through softmax_bar / entropy_bar with the similarity bar as the logits' error.  At the stage shapes the cascade's
    weighted_agg of those similarities follows, against fp64 on the kernel's own similarities."""
    from effimvs_b200 import ops
    monkeypatch.delenv("EFFIMVS_WARP_FORCE_GATHER", raising=False)
    ref, srcs, proj, hyp, _, weights = _device(make_inputs(c))
    r, s = feature_maps(c, ref, srcs)
    HW = c.H * c.W
    _views(c, to_layout(-r + 0.5, c.layout), s[::-1], proj, hyp)
    sims, ent = _views(c, r, s, proj, hyp)
    depth = restate_depth(c, hyp, None)
    pairs = list(view_sims(c, ref, srcs, proj, depth))
    want = torch.stack([p[0][:, 0] for p in pairs], 1)          # (B, n, D, HW)
    bar = torch.stack([p[1][:, 0] for p in pairs], 1)
    del pairs
    check("warp_corr_views." + c.layout, sims.reshape(c.B, c.n, c.D, HW), want, bar, record)
    p, dp = softmax_bar(want, bar, 2)
    check("softmax_entropy." + c.layout, ent.reshape(c.B, c.n, HW), -(p * torch.log(p + 1e-7)).sum(2), entropy_bar(p, dp, 2),
          record)
    del p, dp, want, bar
    if c.layout == "tile":
        monkeypatch.setenv("EFFIMVS_WARP_FORCE_GATHER", "1")
        sims_g, ent_g = _views(c, r, s, proj, hyp)
        monkeypatch.delenv("EFFIMVS_WARP_FORCE_GATHER")
        assert same(sims_g, sims) and same(ent_g, ent), "gathered samples differ from staged ones"
    if c in STAGE_CASES:
        if c.B == 1:
            _check_ray_vs_matmul(c, proj)
        ops.weighted_agg(-sims, weights.flip(1).contiguous())
        got = ops.weighted_agg(sims, weights)
        _check_weighted_agg(sims, weights, got, record)


# ---- weighted_agg ----------------------------------------------------------------------------------------------------
def _check_weighted_agg(sims, weights, got, record):
    B, n, D, H, W = sims.shape
    w = weights.double().unsqueeze(2)
    s = sims.double()
    want, bar = agg_bar((s * w).sum(1), 0.0, (s * w).abs().sum(1), w.sum(1), w.abs().sum(1), n, True)
    check("weighted_agg", got, want, bar, record)


@pytest.mark.parametrize("n,D", WAGG_CASES, ids=["n{}-D{}".format(n, D) for n, D in WAGG_CASES])
def test_weighted_agg_vs_fp64(n, D, record):
    from effimvs_b200 import ops
    B, H, W = 2, 37, 53
    g = torch.Generator().manual_seed(zlib.crc32(repr(("wagg", n, D)).encode()))
    sims = _planted(torch.randn(B, n, D, H, W, generator=g)).to(DEV)
    weights = (0.1 + torch.rand(B, n, H, W, generator=g)).to(DEV)
    ops.weighted_agg(-sims + 0.5, weights.flip(1).contiguous())
    _check_weighted_agg(sims, weights, ops.weighted_agg(sims, weights), record)


# ---- homo_warp -------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("C,mode,H,W,D", HOMO_CASES, ids=["C{}-{}-{}x{}-D{}".format(C, MODE_NAMES[m], H, W, D)
                                                          for (C, m, H, W, D) in HOMO_CASES])
def test_homo_warp_vs_fp64(C, mode, H, W, D, record):
    """homo_warp (homo_warping_new, the materialised (B, C, D, H, W) volume): each value is the 4-tap FMA chain of fp32 tap
    weights, gamma_7 sum |w v| (3 roundings in the weights, 4 in the chain)"""
    from effimvs_b200 import ops
    B = 2
    c = Case("homo", H, W, B, 1, C, 1, D, mode, False, "planar", "normal")
    g = torch.Generator().manual_seed(zlib.crc32(repr(tuple(c)).encode()))
    src = _planted(torch.randn(B, C, H, W, generator=g)).to(DEV)
    proj = make_proj(g, "normal", B, 1, H, W).to(DEV)
    hyp = make_hyp(g, c)[0].to(DEV)
    ops.homo_warp(-src + 0.5, proj.flip(0).contiguous(), hyp, mode, D)
    got = ops.homo_warp(src, proj.reshape(B, 12), hyp, mode, D)
    HW = H * W
    depth = restate_depth(c, hyp, None)
    rays = restate_rays(proj, H, W)
    flat = src.double().permute(0, 2, 3, 1).reshape(B * HW, C)
    b_off = (torch.arange(B, device=DEV, dtype=torch.float64) * HW).reshape(B, 1, 1)
    ix, iy = restate_coords(rays[:, 0], proj[:, 0, 9:], depth, H, W)
    val, aval = interp(flat, b_off, ix, iy, H, W)                    # (B, D, HW, C)
    check("homo_warp", got.reshape(B, C, D, HW), val.permute(0, 3, 1, 2), gamma(7) * aval.permute(0, 3, 1, 2), record)
