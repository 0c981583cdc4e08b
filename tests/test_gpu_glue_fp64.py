"""The update block's glue kernels (csrc/update_glue.cu) and the per-pixel cost kernels (csrc/lookup.cu, the softmax entropy of
csrc/warp_tile.cu) element by element against fp64 restatements of the operations they replace (``-m gpu``).

Every reference is the upstream expression evaluated in float64 on the fp32 operands the kernel reads.  Every bar is a per-element
bound derived from the kernel's fp32 arithmetic (the bar functions below, each with its derivation), never from observed error,
so that an error in one element -- a partial tile, the second grid-stride pass, batch index b >= 1 -- cannot hide behind the
magnitude of the rest of the tensor.  Where the source claims bit-identity with a torch fp32 expression, the check is torch.equal.

The case matrix (module-level lists) runs each kernel at the DTU and Tanks & Temples stage shapes with each stage's hidden and
context sizes, with up to 8 reference views per batch, and at edge shapes; tests/test_glue_cases_host.py restates the host-side
launch rules and asserts that these lists reach every launch branch, and that the bars reject small corruptions.
"""
import math
import os
import subprocess
import sys
import zlib

import pytest
import torch
import torch.nn.functional as F

from effimvs_b200 import net

pytestmark = pytest.mark.gpu
DEV = "cuda"

U = 2.0 ** -24              # unit roundoff of fp32, round to nearest
ULP = 2.0 * U               # one ulp of a normal fp32 value x is at most ULP * |x|
DENORM = 2.0 ** -149        # the fp32 denormal spacing: the absolute error floor of expf in its underflow range
TANHF_ULPS, EXPF_ULPS, LOGF_ULPS = 2, 2, 1    # CUDA C Programming Guide, maximum ulp errors of the single-precision functions

# ---- case matrix ---------------------------------------------------------------------------------------------------
HIDDEN, CONTEXT = net.EffiMVSPlus.HIDDEN, net.EffiMVSPlus.CONTEXT
COST_DIM = net.EffiMVSPlus.G * 3 * 2           # G * cost_num * 2 cost channels (cost_num = 3)
STAGE_HW = {"dtu": ((148, 200), (296, 400), (592, 800)), "tanks": ((132, 240), (264, 480), (528, 960))}
BATCHES = {0: (1, 2, 4, 8), 1: (1, 2, 4, 8), 2: (1, 2, 8)}     # reference views per CUDA-graph replay, trimmed at full size
# (H, W, h, cx, B): every stage shape with its own hidden / context sizes
STAGE_CASES = [(H, W, HIDDEN[s], CONTEXT[s], B) for ds in ("dtu", "tanks") for s, (H, W) in enumerate(STAGE_HW[ds])
               for B in BATCHES[s]]
# maps that end in a partial tile of every kernel (delta_head: 64 x 4, encoder_head: 64 x 4 / 64 x 8, 128 / 256-thread blocks),
# 1-pixel-high and 1-pixel-wide maps
EDGE_HW = ((1, 1), (1, 131), (131, 1), (5, 65), (9, 63), (37, 53))
EDGE_CASES = [(H, W, h, max(4, h // 4), 3) for (H, W) in EDGE_HW for h in (16, 48)] + \
             [(37, 53, h, 4, 2) for h in (32, 64, 96, 128)]
# inv_init / gru_delta: HW > 148 * 16 * 256 = 606,208 takes a second grid-stride pass
HUGE_HW = ((1, 700001), (781, 800))
# encoder_head (CD, h, const, H, W, B): both kernels, every hidden size, 1 / 6 / 8 cost channels
EH_CASES = [(CD, h, const, H, W, 2) for CD in (1, 6, 8) for h in (16, 32, 48, 64, 128) for const in (False, True)
            for (H, W) in ((37, 53), (5, 65))]
# the per-process instantiations: tile rows 8 (<8,0>) and hidden 48 without the threadIdx.z chunks (<4,0>)
EH_ENV_CASES = [({"EFFIMVS_EH_TY": "8"}, (16, 48, 128)), ({"EFFIMVS_EH_ZCHUNKS": "0"}, (48,))]
UPSAMPLE_K = (4, 32, 96, 256)
SOFTMAX_D = (8, 48, 49, 96, 97, 192)
# (D, B, H, W): every D at a small map, plus the stage-1 shapes the cascade regresses at
SOFTMAX_CASES = [(D, 2, 37, 53) for D in SOFTMAX_D] + [(48, 8, 148, 200), (96, 2, 132, 240)]
ENTROPY_CASES = [(D, 37, 53) for D in SOFTMAX_D] + [(48, 148, 200), (96, 132, 240)]
# volume_lookup (B, D, d, H, W, per_pixel_range, sample_stride); H, W are the volume's
LOOKUP_CASES = [(2, 8, 3, 37, 53, True, 1), (3, 16, 8, 37, 53, False, 1), (2, 48, 16, 37, 53, True, 1),
                (2, 8, 16, 148, 200, False, 1), (8, 8, 8, 148, 200, True, 1), (4, 48, 8, 148, 200, False, 2),
                (2, 8, 3, 296, 400, True, 2)]
# dynamic_cost (B, D, ndepth, H, W, per_pixel_range)
DYNCOST_CASES = [(2, 8, 3, 37, 53, True), (2, 8, 8, 37, 53, False), (2, 16, 16, 37, 53, True), (8, 8, 3, 148, 200, True),
                 (2, 8, 3, 592, 800, True), (4, 8, 3, 264, 480, False)]


def _ids(cases):
    return ["-".join(str(v) for v in c) for c in cases]


# ---- bars ----------------------------------------------------------------------------------------------------------
def gamma(n):
    """gamma_n = n u / (1 - n u): the relative error bound of n successive fp32 roundings (Higham, Lemma 3.1)."""
    return n * U / (1.0 - n * U)


def dot_bar(abs_terms, n):
    """An fp32 dot product / convolution in which every term passes through at most n roundings (an FMA chain of n products
    started from the bias, or a summation tree of depth n): |err| <= gamma_n * sum |w_i x_i| (+ |bias|).  relu and clamp are
    1-Lipschitz, so the bound carries through them."""
    return gamma(n) * abs_terms


def libm_bar(value, ulps):
    """A libdevice function with a documented maximum error of `ulps` ulps at an exact argument: ulps * ULP * |f(x)|."""
    return ulps * ULP * value.abs()


def tanh_bar(x, dx):
    """tanhf of an fp32 argument within dx of x: tanh' = 1 - tanh^2 is largest where |x| is smallest, so the argument's error
    moves the result by at most (1 - tanh^2(max(|x| - dx, 0))) dx; plus TANHF_ULPS ulps of the result."""
    slope = 1.0 - torch.tanh((x.abs() - dx).clamp(min=0.0)) ** 2
    return slope * dx + libm_bar(torch.tanh(x), TANHF_ULPS) * (1 + 4 * U)


def sigmoid_bar(x, dx):
    """1 / (1 + expf(-x)) (the kernels' sigmoid) with the argument within dx of x: with e = exp(-x) and s = 1 / (1 + e),
    ds / s = -de / (1 + e), so expf's relative error (EXPF_ULPS ulps) and the argument's (|de| / e = dx, to first order, 1 %
    margin) enter scaled by e / (1 + e) <= 1; the addition and the division add u each."""
    e = torch.exp(-x)
    s = 1.0 / (1.0 + e)
    rel = (e / (1.0 + e)) * (EXPF_ULPS * ULP + 1.01 * dx) + 2 * U
    return s, s * rel * 1.01


def to_depth_bar(inv, dinv, lo, hi):
    """disp_to_depth, 1 / max(lo + (hi - lo) inv, 1e-4), on an inverse depth within dinv of inv: the kernel's s carries the
    roundings of hi - lo, of the product and of the sum (u each, on their own magnitudes) plus (hi - lo) dinv; clamp is
    1-Lipschitz and 1 / s moves by ds / (s (s - ds)); the division adds u.  Returns (depth, bar)."""
    span = hi - lo
    s = lo + span * inv
    ds = U * (span.abs() * inv.abs() * 2 + s.abs()) + span.abs() * dinv
    sc = s.clamp(min=1e-4)
    depth = 1.0 / sc
    return depth, ds / (sc * (sc - ds).clamp(min=1e-300)) * 1.001 + U * depth


def softmax_bar(x, dx, dim):
    """The kernels' softmax, p = expf(x - max) / sum: per logit the relative error of e is EXPF_ULPS ulps plus the subtraction's
    rounding u |x - m| and the logits' own error dx + max(dx) (|de| / e = d(arg), first order, 1 % margin); the sequential sum
    adds gamma_{D-1} and the quotient u.  An expf result in the underflow range is off by at most 2 denormal spacings, which the
    division by z >= 1 does not enlarge.  Returns (p, dp) with dp an absolute bound."""
    m = x.amax(dim=dim, keepdim=True)
    e = torch.exp(x - m)
    z = e.sum(dim=dim, keepdim=True)
    p = e / z
    eps = EXPF_ULPS * ULP + 1.01 * (U * (x - m).abs() + dx + dx.amax(dim=dim, keepdim=True))
    eps_z = (p * eps).sum(dim=dim, keepdim=True) + gamma(x.shape[dim])
    return p, (p * (eps + eps_z + U) * 1.01 + 2 * EXPF_ULPS * DENORM)


def weighted_sum_bar(p, dp, v, dim, n=None):
    """sum_k p_k v_k in fp32 (products rounded, sequential sum): sum |v_k| dp_k for the weights' error, plus gamma_{n} sum
    |p_k v_k| with n = D + 1 roundings on the longest path."""
    n = p.shape[dim] + 1 if n is None else n
    return (v.abs() * dp).sum(dim=dim) + gamma(n) * (p * v).abs().sum(dim=dim)


def entropy_bar(p, dp, dim):
    """-sum p log(p + 1e-7) with p within dp: |d(p log(p + 1e-7)) / dp| <= |log(p + 1e-7)| + 1; the rounding of p + 1e-7 moves
    the log by u, logf adds LOGF_ULPS ulps, the product u of the term, the D-term sum gamma_D of sum |terms|."""
    lg = torch.log(p + 1e-7)
    t = p * lg
    own = p * (U + LOGF_ULPS * ULP * lg.abs()) + U * t.abs()
    return ((lg.abs() + 1.0) * dp + own).sum(dim=dim) + gamma(p.shape[dim]) * t.abs().sum(dim=dim)


def worst_ratio(got, ref, bar):
    """max |got - ref| / bar over the elements (0 where both are 0); NaN / inf must sit where the reference has them."""
    got = got.double()
    same_nonfinite = (~torch.isfinite(ref)) & (got == ref) | (torch.isnan(ref) & torch.isnan(got))
    err = (got - ref).abs()
    err = torch.where(same_nonfinite, torch.zeros_like(err), err)
    err = torch.where(torch.isnan(err), torch.full_like(err, math.inf), err)
    r = err / bar.clamp(min=1e-300)
    r = torch.where(err == 0, torch.zeros_like(r), r)
    return float(r.max()) if r.numel() else 0.0


def within(got, ref, bar):
    return worst_ratio(got, ref, bar) <= 1.0


def check(name, got, ref, bar, record=None):
    """element-wise |got - ref| <= bar; the worst ratio goes into the test report under `name`."""
    assert got.shape == ref.shape, (name, tuple(got.shape), tuple(ref.shape))
    r = worst_ratio(got, ref, bar.expand_as(ref))
    if record is not None:
        record(name, r)
    if r > 1.0:
        err = (got.double() - ref).abs() / bar.expand_as(ref).clamp(min=1e-300)
        idx = torch.nonzero(err == err.max())[0].tolist()
        raise AssertionError("{}: |got - ref| / bar = {:.3g} at {} (got {!r}, ref {!r}, bar {!r})".format(
            name, r, idx, float(got[tuple(idx)]), float(ref[tuple(idx)]), float(bar.expand_as(ref)[tuple(idx)])))
    return r


# ---- fixtures and generators ---------------------------------------------------------------------------------------
@pytest.fixture(scope="module", autouse=True)
def _strict_fp32():
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.set_grad_enabled(False)
    yield


@pytest.fixture
def record(record_property):
    return lambda name, ratio: record_property("ratio:" + name, "{:.4g}".format(ratio))


def _gen(*key):
    return torch.Generator(device=DEV).manual_seed(zlib.crc32(repr(key).encode()))


def _planted(t):
    """t with a structure no other position shares: the last batch entry negated and shifted, the last row and column scaled
    and shifted, so that a skipped, stale or misindexed element of them cannot agree with the reference by chance."""
    t = t.clone()
    t[-1] = -t[-1] + 0.125
    t[..., -1, :] = 1.5 * t[..., -1, :] - 0.25
    t[..., :, -1] = 0.75 * t[..., :, -1] + 0.375
    return t


def _randn(g, *shape, scale=1.0):
    return _planted(torch.randn(*shape, device=DEV, generator=g) * scale)


def _cl(t):
    return t.contiguous(memory_format=torch.channels_last)


def _ranges(B):
    """per-batch inverse-depth ranges (lo, hi) as the cascade forms them, different for every batch entry"""
    dmin = 425.0 - 10.0 * torch.arange(B, device=DEV, dtype=torch.float32)
    dmax = 935.0 + 25.0 * torch.arange(B, device=DEV, dtype=torch.float32)
    return dmax.reciprocal(), dmin.reciprocal()


def _d(t):
    return t.double()


def _conv_abs(x, w, b, padding=0):
    """(fp64 convolution, fp64 sum of |w x| + |b|) of fp32 operands"""
    x, w = _d(x), _d(w)
    b = _d(b) if b is not None else None
    return F.conv2d(x, w, b, padding=padding), F.conv2d(x.abs(), w.abs(), b.abs() if b is not None else None, padding=padding)


# ---- GRU gates ----------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("H,W,h,cx,B", STAGE_CASES + EDGE_CASES, ids=_ids(STAGE_CASES + EDGE_CASES))
def test_gru_reset_and_update_vs_fp64(H, W, h, cx, B, record):
    """gru_reset (sigmoid(r + b_r) * h written beside x) and gru_update ((1 - z) h + z tanh(q + b_q), in place and out), upstream
    models/update.py:41-48; hx = cat[h, x] has 2h channels as in the update block."""
    from effimvs_b200 import ops
    g = _gen("gru", H, W, h, B)
    zr_pre, q_pre = _cl(_randn(g, B, 2 * h, H, W, scale=2.0)), _cl(_randn(g, B, h, H, W, scale=2.0))
    hv, x = torch.tanh(_randn(g, B, h, H, W)), torch.relu(_randn(g, B, h, H, W))
    bz, br, bq = (torch.randn(h, device=DEV, generator=g) for _ in range(3))
    hx = _cl(torch.cat([hv, x], dim=1))
    out = ops.gru_reset(zr_pre, br, hx)
    arg = _d(zr_pre[:, h:]) + _d(br).reshape(1, -1, 1, 1)
    s, ds = sigmoid_bar(arg, U * arg.abs())
    ref = s * _d(hv)
    check("gru_reset", out[:, :h], ref, _d(hv).abs() * ds + U * ref.abs(), record)
    assert torch.equal(out[:, h:], x)
    hx2 = hx.clone()
    got = ops.gru_update(zr_pre, bz, q_pre, bq, hx2)
    za = _d(zr_pre[:, :h]) + _d(bz).reshape(1, -1, 1, 1)
    z, dz = sigmoid_bar(za, U * za.abs())
    qa = _d(q_pre) + _d(bq).reshape(1, -1, 1, 1)
    q, dq = torch.tanh(qa), tanh_bar(qa, U * qa.abs())
    h64 = _d(hv)
    a, b = (1 - z) * h64, z * q
    bar = h64.abs() * (dz + U * (1 - z).abs()) + U * a.abs() + q.abs() * dz + z * dq + U * b.abs() + U * (a + b).abs()
    check("gru_update", got, a + b, bar * (1 + 8 * U), record)
    assert torch.equal(hx2[:, :h], got) and torch.equal(hx2[:, h:], x)


# ---- inverse-depth steps ----------------------------------------------------------------------------------------------
DELTA_CASES = [(H, W, B) for (H, W, _, _, B) in STAGE_CASES] + [(H, W, 3) for (H, W) in EDGE_HW] + [(H, W, 2) for (H, W) in HUGE_HW]


@pytest.mark.parametrize("H,W,B", DELTA_CASES, ids=_ids(DELTA_CASES))
def test_inv_init_and_gru_delta(H, W, B, record):
    """inv_init and gru_delta without a residual bit for bit against torch's fp32 depth_to_disp / disp_to_depth chain
    (models/Effi_MVS_plus.py:138-164); gru_delta with a residual, inv + tanh(pre + b), against fp64."""
    from effimvs_b200 import ops
    g = _gen("delta", H, W, B)
    lo, hi = _ranges(B)
    l4, h4 = lo.reshape(B, 1, 1, 1), hi.reshape(B, 1, 1, 1)
    cur = _planted(425.0 + 510.0 * torch.rand(B, 1, H, W, device=DEV, generator=g))
    inv, depth = ops.inv_init(cur, lo, hi)
    want_inv = (cur.reciprocal() - l4) / ((h4 - l4) + 1e-10)
    want_depth = 1.0 / (l4 + (h4 - l4) * want_inv).clamp(min=1e-4)
    assert torch.equal(inv, want_inv) and torch.equal(depth, want_depth)
    inv0, dep0 = ops.gru_delta(None, None, want_inv, lo, hi)
    assert torch.equal(inv0, want_inv) and torch.equal(dep0, want_depth)
    pre, bias = _randn(g, B, 1, H, W), torch.randn(1, device=DEV, generator=g)
    inv2, dep2 = ops.gru_delta(pre, bias, inv, lo, hi)
    arg = _d(pre) + _d(bias)
    ref = _d(inv) + torch.tanh(arg)
    dinv = tanh_bar(arg, U * arg.abs()) + U * ref.abs()
    check("gru_delta.inv", inv2, ref, dinv, record)
    dref, dbar = to_depth_bar(ref, dinv, _d(l4), _d(h4))
    check("gru_delta.depth", dep2, dref, dbar, record)


DH_CASES = [(H, W, h, B) for (H, W, h, _, B) in STAGE_CASES + EDGE_CASES]


@pytest.mark.parametrize("H,W,h,B", DH_CASES, ids=_ids(DH_CASES))
def test_delta_head_vs_fp64(H, W, h, B, record):
    """delta_head: inv + tanh(conv3x3(t) + b) (DepthHead.conv2, zero padding) and its depth, upstream models/update.py:19-27,
    121-125.  The convolution's 9h products reach the pixel through 9h/16 FMAs of one of 16 partial sums, two adds, two shuffle
    adds and the bias add: a summation tree of depth 9h/16 + 5."""
    from effimvs_b200 import ops
    g = _gen("dh", H, W, h, B)
    t = torch.relu(_randn(g, B, h, H, W))
    w, bias = torch.randn(1, h, 3, 3, device=DEV, generator=g) * 0.1, torch.randn(1, device=DEV, generator=g) * 0.1
    inv = _planted(torch.rand(B, 1, H, W, device=DEV, generator=g))
    lo, hi = _ranges(B)
    got_inv, got_depth = ops.delta_head(_cl(t), w, bias, inv, lo, hi)
    c, ca = _conv_abs(t, w, bias, padding=1)
    dc = dot_bar(ca, 9 * h // 16 + 5)
    ref = _d(inv) + torch.tanh(c)
    dinv = tanh_bar(c, dc) + U * ref.abs()
    check("delta_head.inv", got_inv, ref, dinv, record)
    dref, dbar = to_depth_bar(ref, dinv, _d(lo).reshape(B, 1, 1, 1), _d(hi).reshape(B, 1, 1, 1))
    check("delta_head.depth", got_depth, dref, dbar, record)


# ---- convex upsampling --------------------------------------------------------------------------------------------
def _upsample_ref(inv, m, dm, lo, hi):
    """upsample_depth (net.convex_upsample, models/Effi_MVS_plus.py:167-178) in fp64 on logits m (B,36,H,W) known to within dm,
    with its bar, and disp_to_depth of it: returns (up, up_bar, depth, depth_bar)."""
    B, _, H, W = inv.shape
    up = net.convex_upsample(_d(inv), m, 2)
    x = m.view(B, 9, 4, H, W)
    p, dp = softmax_bar(x, dm.reshape(B, 9, 4, H, W), 1)
    nb = F.unfold(_d(inv), [3, 3], padding=1).view(B, 9, 1, H, W)
    bar = weighted_sum_bar(p, dp, nb.expand_as(p), 1, n=10)                 # (B, 4, H, W), channel = 2 ry + rx
    bar = bar.view(B, 2, 2, H, W).permute(0, 3, 1, 4, 2).reshape(B, 2 * H, 2 * W)
    lo3, hi3 = _d(lo).reshape(B, 1, 1), _d(hi).reshape(B, 1, 1)
    depth, dbar = to_depth_bar(up, bar, lo3, hi3)
    return up, bar, depth, dbar


UP_CASES = [(H, W, h, B) for (H, W, h, _, B) in STAGE_CASES if B <= 4] + [(H, W, h, B) for (H, W, h, _, B) in EDGE_CASES]


@pytest.mark.parametrize("H,W,h,B", UP_CASES, ids=_ids(UP_CASES))
def test_convex_upsample_vs_fp64(H, W, h, B, record):
    """convex_upsample on mask = 0.25 (mask_pre + b) and convex_upsample_conv with the mask head's 1x1 convolution (2h -> 36)
    formed in the kernel, against net.convex_upsample on double tensors; the logits' own errors propagate through the softmax."""
    from effimvs_b200 import ops
    g = _gen("up", H, W, h, B)
    inv = _planted(torch.rand(B, 1, H, W, device=DEV, generator=g))
    lo, hi = _ranges(B)
    mask_pre, mb = _cl(_randn(g, B, 36, H, W, scale=3.0)), torch.randn(36, device=DEV, generator=g)
    up, dup = ops.convex_upsample(mask_pre, mb, 0.25, inv, lo, hi, 2)
    s = (_d(mask_pre) + _d(mb).reshape(1, -1, 1, 1)).contiguous()
    m = 0.25 * s
    ref, bar, dref, dbar = _upsample_ref(inv, m, 0.25 * U * s.abs() + U * m.abs(), lo, hi)
    check("convex_upsample", up, ref, bar, record)
    check("convex_upsample.depth", dup, dref, dbar, record)
    _check_upsample_conv(g, inv, lo, hi, 2 * h, "convex_upsample_conv", record)


def _check_upsample_conv(g, inv, lo, hi, K, name, record):
    from effimvs_b200 import ops
    B, _, H, W = inv.shape
    t = torch.relu(_randn(g, B, K, H, W))
    mw, mb = torch.randn(36, K, 1, 1, device=DEV, generator=g) * (1.5 / math.sqrt(K)), torch.randn(36, device=DEV, generator=g)
    up, dup = ops.convex_upsample_conv(_cl(t), mw, mb, 0.25, inv, lo, hi, 2)
    c, ca = _conv_abs(t, mw, mb)
    m = (0.25 * c).contiguous()
    ref, bar, dref, dbar = _upsample_ref(inv, m, 0.25 * dot_bar(ca, K + 1) + U * m.abs(), lo, hi)
    check(name, up, ref, bar, record)
    check(name + ".depth", dup, dref, dbar, record)


UPK_CASES = [(K, H, W) for K in UPSAMPLE_K for (H, W) in ((37, 53), (1, 131), (131, 1))]


@pytest.mark.parametrize("K,H,W", UPK_CASES, ids=_ids(UPK_CASES))
def test_convex_upsample_conv_every_k(K, H, W, record):
    g = _gen("upk", K, H, W)
    B = 2
    lo, hi = _ranges(B)
    _check_upsample_conv(g, _planted(torch.rand(B, 1, H, W, device=DEV, generator=g)), lo, hi, K, "convex_upsample_conv", record)


# ---- cost encoder ----------------------------------------------------------------------------------------------------
def _encoder_head_check(CD, h, H, W, B, record, name="encoder_head"):
    """relu(convc1(cost)) (1x1, CD products after the bias) beside relu(convd1(inv)) (7x7, 49 products), upstream
    models/update.py:88-91."""
    from effimvs_b200 import ops
    g = _gen("eh", CD, h, H, W, B)
    cost, inv = _randn(g, B, CD, H, W), _planted(torch.rand(B, 1, H, W, device=DEV, generator=g))
    wc1, bc1 = torch.randn(h, CD, 1, 1, device=DEV, generator=g) * 0.3, torch.randn(h, device=DEV, generator=g)
    wd1, bd1 = torch.randn(h, 1, 7, 7, device=DEV, generator=g) * 0.2, torch.randn(h, device=DEV, generator=g)
    got = ops.encoder_head(cost, inv, wc1, bc1, wd1, bd1)
    assert got.is_contiguous(memory_format=torch.channels_last)
    c, ca = _conv_abs(cost, wc1, bc1)
    d, da = _conv_abs(inv, wd1, bd1, padding=3)
    ref = torch.cat([torch.relu(c), torch.relu(d)], dim=1)
    bar = torch.cat([dot_bar(ca, CD), dot_bar(da, 49)], dim=1)
    return check(name, got, ref, bar, record)


EH_STAGE_CASES = [(H, W, h, B) for (H, W, h, _, B) in STAGE_CASES] + [(H, W, h, B) for (H, W, h, _, B) in EDGE_CASES]


@pytest.mark.parametrize("H,W,h,B", EH_STAGE_CASES, ids=_ids(EH_STAGE_CASES))
def test_encoder_head_stage_shapes(H, W, h, B, record):
    _encoder_head_check(COST_DIM, h, H, W, B, record)


@pytest.mark.parametrize("CD,h,const,H,W,B", EH_CASES, ids=_ids(EH_CASES))
def test_encoder_head_every_kernel(CD, h, const, H, W, B, record, monkeypatch):
    from effimvs_b200 import ops
    monkeypatch.setenv("EFFIMVS_EH_CONST", "1" if const else "0")
    before = ops.LAUNCHES
    _encoder_head_check(CD, h, H, W, B, record)
    assert ops.LAUNCHES - before == (h // 16 if const else 1)


_EH_SCRIPT = r"""
import os, sys
sys.path.insert(0, {root!r}); sys.path.insert(0, os.path.join({root!r}, "tests"))
import torch
import test_gpu_glue_fp64 as t
torch.backends.cudnn.allow_tf32 = False
os.environ["EFFIMVS_EH_CONST"] = "0"
ratios = {{}}
with torch.no_grad():
    for h in {hs!r}:
        for CD in (1, 6, 8):
            for (H, W, B) in ((37, 53, 2), (9, 63, 3), (148, 200, 4)):
                key = "encoder_head.h{{}}.cd{{}}.{{}}x{{}}x{{}}".format(h, CD, B, H, W)
                ratios[key] = t._encoder_head_check(CD, h, H, W, B, None, key)
torch.save(ratios, sys.argv[1])
"""


@pytest.mark.parametrize("env,hs", EH_ENV_CASES, ids=["-".join(e) for e, _ in EH_ENV_CASES])
def test_encoder_head_per_process_switches(env, hs, tmp_path, record):
    """EFFIMVS_EH_TY and EFFIMVS_EH_ZCHUNKS are read once per process: the instantiations they select run in a fresh
    interpreter, which holds them to the same fp64 bars itself and returns the worst ratios."""
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    script = tmp_path / "eh_run.py"
    script.write_text(_EH_SCRIPT.format(root=root, hs=tuple(hs)))
    out = tmp_path / "eh.pt"
    res = subprocess.run([sys.executable, str(script), str(out)], env=dict(os.environ, **env), timeout=600,
                         capture_output=True, text=True)
    assert res.returncode == 0, res.stderr[-4000:]
    ratios = torch.load(out)
    assert len(ratios) == 9 * len(hs)
    for k, r in ratios.items():
        record(k, r)
        assert r <= 1.0, (k, r)


TAIL_CASES = STAGE_CASES + [(H, W, h, cx, B) for (H, W, h, cx, B) in EDGE_CASES if h - cx >= 8 and (h - cx) % 4 == 0 and h - cx <= 48
                            and cx in (4, 8, 12)]


@pytest.mark.parametrize("H,W,h,cx,B", TAIL_CASES, ids=_ids(TAIL_CASES))
def test_encoder_tail_and_gru_init_vs_fp64(H, W, h, cx, B, record):
    """gru_init (tanh of the hidden half of the context map), gru_init_ctx (that plus the context term
    w_ctx relu(context) + b), encoder_tail (relu(w m + term)) and encoder_tail_ctx (relu(w_m m + w_ctx relu(context) + b)),
    upstream models/update.py:93-95 and models/Effi_MVS_plus.py:464-466; hm = h - cx channels of m."""
    from effimvs_b200 import ops
    g = _gen("tail", H, W, h, cx, B)
    hm = h - cx
    ctx_map = _cl(_randn(g, B, h + cx, H, W))
    w_m, w_ctx = torch.randn(h, hm, 1, 1, device=DEV, generator=g) * 0.3, torch.randn(h, cx, 1, 1, device=DEV, generator=g) * 0.3
    bias = torch.randn(h, device=DEV, generator=g) * 0.1
    m = _cl(_randn(g, B, hm, H, W))
    th = torch.tanh(_d(ctx_map[:, :h]))
    hx0 = ops.gru_init(ctx_map, h)
    check("gru_init", hx0[:, :h], th, libm_bar(th, TANHF_ULPS), record)
    hx, term = ops.gru_init_ctx(ctx_map, h, _cl(w_ctx), bias)
    assert torch.equal(hx[:, :h], hx0[:, :h])
    ctx = torch.relu(ctx_map[:, h:])
    t64, ta = _conv_abs(ctx, w_ctx, bias)
    check("gru_init_ctx.term", term, t64, dot_bar(ta, cx), record)
    keep = hx[:, :h].clone()
    ops.encoder_tail_ctx(m, w_m, ctx_map, h, cx, True, w_ctx, bias, hx)
    mm, ma = _conv_abs(m, w_m, None)
    check("encoder_tail_ctx", hx[:, h:], torch.relu(mm + t64), dot_bar(ma + ta, cx + hm), record)
    assert torch.equal(hx[:, :h], keep)
    hx2 = _cl(torch.zeros(B, 2 * h, H, W, device=DEV))
    ops.encoder_tail(m, w_m, term, hx2)
    tt = _d(term)
    check("encoder_tail", hx2[:, h:], torch.relu(mm + tt), dot_bar(ma + tt.abs(), hm), record)
    assert not hx2[:, :h].any()


# ---- softmax regression, entropy --------------------------------------------------------------------------------------
def _planted_logits(g, B, D, H, W):
    """3 randn logits, with planted rows: uniform logits, one-hot at d = 0 and at d = D-1 (the clamped 4-bin window), and
    logits of +-80 (expf underflows)"""
    x = 3.0 * torch.randn(B, D, H, W, device=DEV, generator=g)
    x[-1] = -x[-1]
    x[:, :, -1, :] = 0.0
    x[:, :, -2, :] = -80.0
    x[:, 0, -2, : W // 2] = 80.0
    x[:, D - 1, -2, W // 2:] = 80.0
    x[:, :, -3, :] = 80.0 * torch.sign(torch.randn(B, D, W, device=DEV, generator=g))
    x[:, :, :, -1] = 5.0 * x[:, :, :, -1] + 0.5
    return x


@pytest.mark.parametrize("D,B,H,W", SOFTMAX_CASES, ids=_ids(SOFTMAX_CASES))
def test_softmax_regress_conf_vs_fp64(D, B, H, W, record):
    """softmax over D, sum p h, and the confidence sum of p over [idx-1, idx+2], idx = trunc(sum p d) clamped (upstream
    models/Effi_MVS_plus.py:78-88, models/module.py:518-524).  Where idx is within its error bound of an integer either window
    is accepted.  HYP_PLANES gives the same bits as the expanded HYP_TENSOR."""
    from effimvs_b200 import capi, ops
    g = _gen("smx", D, B, H, W)
    x = _planted_logits(g, B, D, H, W)
    planes = 425.0 + 510.0 * torch.rand(B, D, device=DEV, generator=g)
    hyp = _planted(425.0 + 510.0 * torch.rand(B, D, H, W, device=DEV, generator=g)).abs()
    depth, conf = ops.softmax_regress_conf(x, hyp, capi.HYP_TENSOR)
    p, dp = softmax_bar(_d(x), torch.zeros_like(_d(x)), 1)
    h64 = _d(hyp)
    check("softmax_regress_conf.depth", depth, (p * h64).sum(1), weighted_sum_bar(p, dp, h64, 1), record)
    dd = torch.arange(D, device=DEV, dtype=torch.float64).reshape(1, D, 1, 1)
    idxf = (p * dd).sum(1)
    didx = weighted_sum_bar(p, dp, dd.expand_as(p), 1)
    taps = torch.arange(-1, 3, device=DEV).reshape(1, 4, 1, 1)

    def window(idx):
        """sum of p over [idx-1, idx+2] inside [0, D-1] (the zero-padded 4-bin window) and its bar: the weights' own errors
        plus the kernel's sequential sum of at most 4 terms"""
        k = idx.long().clamp(0, D - 1).unsqueeze(1) + taps
        ok = (k >= 0) & (k < D)
        kc = k.clamp(0, D - 1)
        zero = torch.zeros((), dtype=torch.float64, device=DEV)
        s = torch.where(ok, p.gather(1, kc), zero).sum(1)
        return s, torch.where(ok, dp.gather(1, kc), zero).sum(1) + gamma(3) * s

    def ratio(s, e):
        err = (conf.double() - s).abs()
        return torch.where(err == 0, torch.zeros_like(err), err / e)

    # where idx = trunc(E[d]) is within its error bound of an integer, the kernel may take either window
    r = float(torch.minimum(ratio(*window(torch.trunc((idxf - didx).clamp(min=0)))),
                            ratio(*window(torch.trunc(idxf + didx)))).max())
    record("softmax_regress_conf.conf", r)
    assert r <= 1.0, r
    pd, pc = ops.softmax_regress_conf(x, planes, capi.HYP_PLANES)
    td, tc = ops.softmax_regress_conf(x, planes.reshape(B, D, 1, 1).expand(B, D, H, W).contiguous(), capi.HYP_TENSOR)
    assert torch.equal(pd, td) and torch.equal(pc, tc)


@pytest.mark.parametrize("D,H,W", ENTROPY_CASES, ids=_ids(ENTROPY_CASES))
def test_softmax_entropy_vs_fp64(D, H, W, record):
    """the softmax entropy of each view's similarities, -sum p log(p + 1e-7) (upstream models/Effi_MVS_plus.py:43-44), computed
    by the kernel after the tile warp kernel wrote the similarities (channels-last maps), against fp64 on those similarities.
    Source view 0 has zero features (uniform logits), view 2 features scaled so that the logits reach the expf underflow."""
    from effimvs_b200 import capi, hotpath, ops, synthetic
    feats, cams, hyp, _ = synthetic.microbench_inputs(16, D, H, W, views=4, seed=D + W, device=DEV)
    feats[1] = torch.zeros_like(feats[1])
    feats[3] = feats[3] * 200.0
    feats = [_cl(torch.cat([f, f.flip(-1)])) for f in feats]      # B = 2, the second entry different
    cams = cams.repeat(2, 1, 1, 1, 1)
    hyp = hyp.repeat(2, 1, 1, 1).contiguous()
    proj = hotpath.CudaHotPath().relative_projection(cams)
    sims, ent = ops.warp_corr_views(feats[0], feats[1:], proj, hyp, capi.HYP_TENSOR, D)
    p, dp = softmax_bar(_d(sims), torch.zeros_like(_d(sims)), 2)
    ref = -(p * torch.log(p + 1e-7)).sum(2)
    check("softmax_entropy", ent, ref, entropy_bar(p, dp, 2), record)
    assert float(sims[:, 0].abs().max()) == 0.0 and float(sims[:, 2].abs().max()) > 110.0


# ---- volume lookup / dynamic cost ----------------------------------------------------------------------------------
def lookup_ix_bar(depth, ddepth, dmin, dmax, D):
    """lookup_1d's sampling coordinate ix = (1/depth - 1/dmax) / ((1/dmin - 1/dmax) + 1e-10) (D-1), through bilinear_sampler's
    normalise / un-normalise round trip, in fp64, and a bound on the kernel's error in it: every one of its IEEE operations
    adds u times its result, propagated forward to first order (1 % margin).  The depth itself is known to within ddepth."""
    ia, ic, r = 1.0 / dmax, 1.0 / dmin, 1.0 / depth
    e_ia, e_ic = U * ia.abs(), U * ic.abs()
    e_r = U * r.abs() + ddepth * r * r
    num = r - ia
    e_num = e_r + e_ia + U * num.abs()
    den = (ic - ia) + 1e-10
    e_den = e_ic + e_ia + 2 * U * den.abs()
    q = num / den
    e_q = (e_num + q.abs() * e_den) / den.abs() + U * q.abs()
    t = q * (D - 1)
    e_t = e_q * (D - 1) + U * t.abs()
    rinv = 1.0 / (D - 1)
    g2 = 2 * t * rinv
    e_g = 2 * e_t * rinv + 2 * t.abs() * U * rinv + U * g2.abs() + U * (g2 - 1).abs()
    e_ix = (e_g + U * g2.abs()) * 0.5 * (D - 1) + U * t.abs()
    return t, e_ix * 1.01


def lookup_bar(vol, ix, e_ix, dim):
    """linear interpolation of vol along `dim` at ix with zero padding (grid_sample, padding_mode zeros, align_corners True):
    continuous and piecewise linear, so the coordinate's error moves it by at most e_ix times the largest neighbouring slope;
    the two weights (f + 1 - ix, ix - f), the product and the FMA round once each.  Returns (value, bar)."""
    D = vol.shape[dim]
    shape = [1] * vol.dim()
    shape[dim] = 2
    z = torch.zeros([2 if i == dim else s for i, s in enumerate(vol.shape)], dtype=vol.dtype, device=vol.device)
    vext = torch.cat([z, vol, z], dim=dim)                                   # vext[k + 2] = vol[k], zero for k < 0 or k >= D
    f = torch.floor(ix).clamp(-2, D).long()
    inside = (ix >= -1) & (ix <= D)
    take = lambda k: vext.gather(dim, (k + 2).clamp(0, D + 3))              # noqa: E731
    v0, v1 = take(f), take(f + 1)
    w1 = ix - f
    w0 = 1.0 - w1
    val = torch.where(inside, v0 * w0 + v1 * w1, torch.zeros_like(ix))
    slope = torch.maximum(torch.maximum((v1 - v0).abs(), (v0 - take(f - 1)).abs()), (take(f + 2) - v1).abs())
    own = 2 * U * ((v0 * w0).abs() + (v1 * w1).abs()) + U * val.abs()
    return val, slope * e_ix + torch.where(inside, own, torch.zeros_like(own))


def _sample_depths(g, B, d, H, W, dmin, dmax):
    """depths in the range, with planted samples exactly at dmin and dmax, just outside them (taps f = -1 and f = D-1) and far
    outside"""
    u = torch.rand(B, d, H, W, device=DEV, generator=g)
    s = 1.0 / (1.0 / dmax + u * (1.0 / dmin - 1.0 / dmax))
    lo_, hi_ = dmin.expand(B, 1, H, W)[:, 0], dmax.expand(B, 1, H, W)[:, 0]
    for r in (-1, -2):                       # two rows / columns, so that a [::2, ::2] view keeps one of each
        s[:, 0, r, :] = lo_[:, r, :]
        s[:, -1, r, :] = hi_[:, r, :]
        s[:, 0, :, r] = hi_[:, :, r] * (1 + 1e-4)
        s[:, -1, :, r] = lo_[:, :, r] * (1 - 1e-4)
    s[:, 0, 0, 0], s[:, -1, 0, 0] = 3 * hi_[:, 0, 0], 0.3 * lo_[:, 0, 0]
    return s


def _range_tensors(g, B, H, W, per_pixel):
    if per_pixel:
        dmin = 425.0 + 100.0 * torch.rand(B, 1, H, W, device=DEV, generator=g)
        return dmin, dmin + 200.0 + 300.0 * torch.rand(B, 1, H, W, device=DEV, generator=g)
    return (425.0 - 10 * torch.arange(B, device=DEV, dtype=torch.float32)).reshape(B, 1, 1, 1), \
        (935.0 + 20 * torch.arange(B, device=DEV, dtype=torch.float32)).reshape(B, 1, 1, 1)


@pytest.mark.parametrize("B,D,d,H,W,per_pixel,stride", LOOKUP_CASES, ids=_ids(LOOKUP_CASES))
def test_volume_lookup_vs_fp64(B, D, d, H, W, per_pixel, stride, record):
    """volume_lookup (pro_bilinear_sampler, upstream models/Effi_MVS_plus.py:102-134) against fp64 interpolation; stride 2
    reads the [::2, ::2] view of full-resolution samples in the kernel."""
    from effimvs_b200 import hotpath
    g = _gen("look", B, D, d, H, W, per_pixel, stride)
    vol = _randn(g, B, D, H, W)
    dmin, dmax = _range_tensors(g, B, H, W, per_pixel)
    full = _sample_depths(g, B, d, H * stride, W * stride,
                          dmin.repeat_interleave(stride, 2).repeat_interleave(stride, 3) if per_pixel else dmin,
                          dmax.repeat_interleave(stride, 2).repeat_interleave(stride, 3) if per_pixel else dmax)
    samples = full[:, :, ::stride, ::stride]
    got = hotpath.CudaHotPath("f32").volume_lookup(vol, samples, dmin, dmax)
    ix, e_ix = lookup_ix_bar(_d(samples), 0.0, _d(dmin), _d(dmax), D)
    vals, bars = [], []
    for k in range(d):
        v, b = lookup_bar(_d(vol), ix[:, k:k + 1].expand(B, 1, H, W), e_ix[:, k:k + 1].expand(B, 1, H, W), 1)
        vals.append(v)
        bars.append(b)
    check("volume_lookup", got, torch.cat(vals, 1), torch.cat(bars, 1), record)


def local_hypothesis_bar(cur, interval, nd, k):
    """get_cur_depth_range_samples of one plane on 1 / cur, as dynamic_cost's local_hypothesis forms it, in fp64, with a forward
    bound of its fp32 roundings (u per operation, first order, clamps 1-Lipschitz): returns (depth, bound)."""
    inv = 1.0 / cur
    half = (nd // 2) * interval
    e_inv, e_half = U * inv.abs(), U * half.abs()
    lo = (inv - half).clamp(min=1e-4)
    e_lo = e_inv + e_half + U * lo.abs()
    hi = (inv + half).clamp(min=1e-4).clamp(max=1e4)
    e_hi = e_inv + e_half + U * hi.abs()
    rinv = 1.0 / (nd - 1)
    step = (hi - lo) * rinv
    e_step = (e_hi + e_lo + U * (hi - lo).abs()) * rinv + 2 * U * step.abs()
    s = (lo + k * step).clamp(min=1e-5)
    e_s = e_lo + k * e_step + U * (k * step).abs() + U * s.abs()
    depth = 1.0 / s
    return depth, 1.01 * (e_s / (s * s) + U * depth)


@pytest.mark.parametrize("B,D,nd,H,W,per_pixel", DYNCOST_CASES, ids=_ids(DYNCOST_CASES))
def test_dynamic_cost_vs_fp64(B, D, nd, H, W, per_pixel, record):
    """dynamic_cost (GetCost.forward, upstream models/Effi_MVS_plus.py:257-303): nd local hypotheses around each pixel's depth
    looked up in the raw and the regularised volume."""
    from effimvs_b200 import hotpath
    g = _gen("dyn", B, D, nd, H, W, per_pixel)
    raw, reg = _randn(g, B, D, H, W), _randn(g, B, D, H, W)
    dmin, dmax = _range_tensors(g, B, H, W, per_pixel)
    cur = _planted(_sample_depths(g, B, 1, H, W, dmin, dmax)).abs()
    cur[:, :, 0, 1] = dmin.expand(B, 1, H, W)[:, :, 0, 1]
    interval = 1e-4 * (1 + torch.rand(B, device=DEV, generator=g))
    got = hotpath.CudaHotPath("f32").dynamic_cost(cur, raw, reg, interval, dmin, dmax, nd)
    vals, bars = [], []
    for vol in (raw, reg):
        for k in range(nd):
            dep, e_dep = local_hypothesis_bar(_d(cur), _d(interval).reshape(B, 1, 1, 1), nd, k)
            ix, e_ix = lookup_ix_bar(dep, e_dep, _d(dmin), _d(dmax), D)
            v, b = lookup_bar(_d(vol), ix, e_ix, 1)
            vals.append(v)
            bars.append(b)
    check("dynamic_cost", got, torch.cat(vals, 1), torch.cat(bars, 1), record)


# ---- bit-exact helpers of the cascade --------------------------------------------------------------------------------
RANGE_CASES = [(B, nd, H, W) for (H, W, _, _, B) in STAGE_CASES if B in (1, 8) for nd in (8,)] + [(3, 5, 1, 131), (2, 16, 131, 1)]


@pytest.mark.parametrize("B,nd,H,W", RANGE_CASES, ids=_ids(RANGE_CASES))
def test_range_samples_bit_exact(B, nd, H, W):
    """depth_range_samples (get_cur_depth_range_samples, upstream models/module.py:554-570) bit for bit against the torch
    expression on the device (a tensor divided by a Python scalar is a multiplication by the fp32 reciprocal there too)."""
    from effimvs_b200 import ops
    g = _gen("rs", B, nd, H, W)
    cur = _planted(1.0 / (425.0 + 510.0 * torch.rand(B, H, W, device=DEV, generator=g))).abs()
    cur[0, 0, 0] = 1e-6
    iv = 1e-4 * (1 + torch.rand(B, device=DEV, generator=g))
    got = ops.depth_range_samples(cur, iv, nd)
    half = (nd // 2) * iv.reshape(B, 1, 1)
    lo = (cur - half).clamp(min=1e-4)
    hi = (cur + half).clamp(min=1e-4).clamp(max=1e4)
    step = (hi - lo) / (nd - 1)
    k = torch.arange(nd, device=DEV, dtype=torch.float32).reshape(1, nd, 1, 1)
    want = (lo.unsqueeze(1) + k * step.unsqueeze(1)).clamp(min=1e-5)
    assert torch.equal(got, want)


def test_relative_projection_vs_fp64_and_singular_reference():
    """P_src inverse(P_ref) with P = [K E[:3]; E[3]] formed in fp32 as upstream's matmul does: fp64 inversion, rounded once; a
    singular reference camera gives NaN for all of its source views and leaves the other batch entries alone."""
    from effimvs_b200 import ops, synthetic
    B, V = 8, 5
    _, cams, _, _ = synthetic.microbench_inputs(8, 4, 32, 40, views=V, seed=3, device=DEV)
    cams = cams.repeat(B, 1, 1, 1, 1).clone()
    cams[:, :, 0, :3, 3] += torch.arange(B, device=DEV, dtype=torch.float32).reshape(B, 1, 1) * 3.0
    cams[B - 1, 0, 0] = 0.0                                                  # the last batch entry's reference extrinsic
    got = ops.relative_projection(cams)
    E, K = _d(cams[:B - 1, :, 0]), _d(cams[:B - 1, :, 1])
    P = E.clone()
    P[:, :, :3, :4] = torch.matmul(K[:, :, :3, :3], E[:, :, :3, :4])
    Pi = torch.linalg.inv(P[:, :1])
    R = torch.matmul(P[:, 1:], Pi)
    # the kernel rounds each entry of K E[:3] once per product of its 3-term FMA chain (gamma_3 relative); to first order a
    # perturbation dP_src dP_ref moves R by dP_src Pi - R dP_ref Pi, bounded entrywise by gamma_3 (|P_src| |Pi| + |R| |P_ref| |Pi|);
    # the fp64 inversion and products add a few 2^-53 of the same magnitudes; the result is rounded to fp32 once
    sens = torch.matmul(P[:, 1:].abs(), Pi.abs()) + torch.matmul(torch.matmul(R.abs(), P[:, :1].abs()), Pi.abs())
    bar = U * R.abs() + (1.01 * gamma(3) + 2.0 ** -45) * sens
    flat = lambda t: torch.cat([t[:, :, :3, :3].reshape(B - 1, V - 1, 9), t[:, :, :3, 3]], dim=2)    # noqa: E731
    check("relative_projection", got[:B - 1], flat(R), flat(bar))
    assert torch.isnan(got[B - 1]).all()
