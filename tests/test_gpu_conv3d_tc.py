"""The tensor-core 3-D nets (csrc/conv3d_tc.cu: costreg_bf16, cost_up_bf16) layer by layer, in bf16x3.

Every layer of the two nets is held to an fp64 restatement of its own arithmetic, computed from the layer's decoded input
as the net left it in the caller's workspace, so that errors do not compound from layer to layer:

  - activations are stored as a bf16 pair hi = RN(v), lo = RN(v - hi); weights are packed the same way;
  - a tensor-core layer forms xhi*whi + xlo*whi + xhi*wlo (the z-sweep programs also xlo*wlo), all exact in fp32, and only
    the order of the fp32 accumulation is free; the CUDA-core layers (1 -> 8, 8 -> 1) are fp32 FMAs on fp32 weights;
  - so per voxel |got - ref| <= 2^-17 |ref| (the hi/lo storage, absent for fp32 outputs) + C_ACC 2^-23 S, where S is the
    same restatement on absolute values plus |bias| and |residual|.

The workspace is filled with 0xFF bytes (NaN as bf16 and as fp32) before PREPARE, so the tests also see which interior
voxels a layer failed to write, and every store into a halo or guard voxel (the next layer reads those as its zero padding).

The CPU part checks the test-side decoder of the workspace layout against the library's workspace sizes and against the
ported index function, and the fp64 restatements against brute-force loops.
"""
import os
from typing import NamedTuple

import pytest
import torch
import torch.nn.functional as F

DEV = "cuda"
# accumulation-order term of the bound, in units of 2^-23 S.  Calibrated on a B200 (1000 W): the worst voxel of all layers,
# shapes and weights needed 13.1 (cross-scale conv1, 16 -> 8 z-sweep, CSP_C weights), the other layers 0.6 - 9.6.
C_ACC = 16.0
STORE = 2.0 ** -17          # hi/lo storage: |hi + lo - v| <= 2^-17 |v|
ULP23 = 2.0 ** -23

# ------------------------------------------------------------------------------------------------
# workspace layout: a port of make_layout / act_index / layout_bytes and of the Carver order (csrc/conv3d_tc.cu)
# ------------------------------------------------------------------------------------------------
L_REG, L_SPLIT = 0, 1
W_SLOT = 128 * 1024
WS_SLACK = 4096


class Layout(NamedTuple):
    kind: int
    C: int
    planes: int       # hi and lo halves counted
    D: int
    H: int
    W: int
    lo_off: int       # plane offset of the lo half (0: plain bf16)
    Py: int
    Px: int
    guard: int
    zstride: int
    vs: int           # voxels per (sub-)volume including both guards
    batch_stride: int


def make_layout(kind, C, D, H, W, hilo):
    lo_off = C // 8 if hilo else 0
    planes = (C // 8) * (2 if hilo else 1)
    d, h, w = (D // 2, H // 2, W // 2) if kind == L_SPLIT else (D, H, W)
    Py, Px = h + 2, w + 2
    guard = Px + 136
    zstride = Py * Px
    vs = (d + 2) * zstride + 2 * guard
    return Layout(kind, C, planes, D, H, W, lo_off, Py, Px, guard, zstride, vs, vs * planes * (8 if kind == L_SPLIT else 1))


def layout_bytes(L, B):
    return (L.batch_stride * B * 16 + 255) & ~255


def act_index(L, b, plane, z, y, x):
    """voxel (16-byte unit) index of (b, plane, z, y, x); works on ints and on int64 tensors"""
    if L.kind == L_REG:
        return b * L.batch_stride + plane * L.vs + L.guard + (z + 1) * L.zstride + (y + 1) * L.Px + (x + 1)
    sub = ((z & 1) << 2) | ((y & 1) << 1) | (x & 1)
    return (b * L.batch_stride + (plane * 8 + sub) * L.vs + L.guard + ((z >> 1) + 1) * L.zstride + ((y >> 1) + 1) * L.Px +
            ((x >> 1) + 1))


class Buf(NamedTuple):
    name: str
    L: Layout
    off: int          # byte offset in the workspace
    raw: bool         # raw fp32 pair: channels 0-3 in the "hi" voxel, 4-7 in the "lo" voxel


class WsLayout(NamedTuple):
    B: int
    bufs: dict        # name -> Buf, in carve order
    act_bytes: int    # end of the activations (the packed weight slots follow)
    total: int        # the library's workspace size


def _carve(B, named, n_slots, raw=()):
    off, bufs = 0, {}
    for name, L in named:
        bufs[name] = Buf(name, L, off, name in raw)
        off += (layout_bytes(L, B) + 255) & ~255
    return WsLayout(B, bufs, off, off + n_slots * W_SLOT + WS_SLACK)


def costreg_layout(B, D, H, W, hilo=True, raw_c7=False):
    L0, L1 = make_layout(L_REG, 8, D, H, W, hilo), make_layout(L_SPLIT, 8, D, H, W, hilo)
    L2, L3 = make_layout(L_REG, 16, D // 2, H // 2, W // 2, hilo), make_layout(L_SPLIT, 16, D // 2, H // 2, W // 2, hilo)
    L4 = make_layout(L_REG, 32, D // 4, H // 4, W // 4, hilo)
    named = [("c0", L0), ("c7", L0), ("c1", L1), ("c2", L2), ("c6", L2), ("c3", L3), ("c4", L4), ("c5", L4)]
    return _carve(B, named, 8, ("c7",) if raw_c7 else ())


def cost_up_layout(B, D, H, W, hilo=True, raw_c1=True):
    """cat: planes [conv0 hi, conv_cost hi, conv0 lo, conv_cost lo], i.e. channels 0-7 conv0, 8-15 conv_cost"""
    named = [("cat", make_layout(L_REG, 16, D, H // 2, W // 2, hilo)), ("c1", make_layout(L_REG, 8, D, H // 2, W // 2, hilo))]
    return _carve(B, named, 2, ("c1",) if raw_c1 else ())


def _region(ws, buf, B, dtype):
    """(B, volumes, vs, lanes) view of one buffer; lanes = 16 bytes as `dtype`"""
    L = buf.L
    nvol = L.planes * (8 if L.kind == L_SPLIT else 1)
    lanes = 16 // torch.empty((), dtype=dtype).element_size()
    return ws[buf.off: buf.off + L.batch_stride * B * 16].view(dtype).view(B, nvol, L.vs, lanes)


def _interior(ws, buf, B, dtype):
    """view (B, planes, D, H, W, lanes) of the interior voxels, in logical coordinates (split layouts interleaved back)"""
    L = buf.L
    r = _region(ws, buf, B, dtype)
    lanes = r.shape[-1]
    d = L.D // 2 if L.kind == L_SPLIT else L.D
    v = r[:, :, L.guard: L.guard + (d + 2) * L.zstride].view(B, r.shape[1], d + 2, L.Py, L.Px, lanes)[:, :, 1:-1, 1:-1, 1:-1]
    if L.kind == L_REG:
        return v
    v = v.reshape(B, L.planes, 2, 2, 2, d, L.Py - 2, L.Px - 2, lanes)     # volume = plane * 8 + (sz, sy, sx)
    return v.permute(0, 1, 5, 2, 6, 3, 7, 4, 8)        # (B, P, d, sz, h, sy, w, sx, lanes): z = 2 * zz + sz


def _split_interior(ws, buf, B, dtype):
    """writable form of _interior for split layouts: the 8 sub-volume views (sub -> (B, P, d, h, w, lanes))"""
    L = buf.L
    r = _region(ws, buf, B, dtype)
    d = L.D // 2
    v = r[:, :, L.guard: L.guard + (d + 2) * L.zstride].view(B, L.planes, 8, d + 2, L.Py, L.Px, r.shape[-1])
    return [v[:, :, s, 1:-1, 1:-1, 1:-1] for s in range(8)]


def _to_nc(v, groups, B, D, H, W):
    """(B, groups, D, H, W, lanes) -> (B, groups * lanes, D, H, W)"""
    return v.reshape(B, groups, D, H, W, v.shape[-1]).permute(0, 1, 5, 2, 3, 4).reshape(B, -1, D, H, W)


def decode(ws, lay):
    """every activation of the workspace as fp32 (B, C, D, H, W): {name: {"hi", "lo", "val", "raw"}}"""
    out = {}
    for name, buf in lay.bufs.items():
        L, B = buf.L, lay.B
        if buf.raw:
            v = _interior(ws, buf, B, torch.float32)
            val = _to_nc(v, 2, B, L.D, L.H, L.W)            # plane 0: channels 0-3, plane 1 (the "lo" voxel): 4-7
            out[name] = {"hi": val, "lo": torch.zeros_like(val), "val": val, "raw": True}
            continue
        v = _interior(ws, buf, B, torch.bfloat16)
        g = L.C // 8
        hi = _to_nc(v[:, :g], g, B, L.D, L.H, L.W).float()
        lo = _to_nc(v[:, L.lo_off:L.lo_off + g], g, B, L.D, L.H, L.W).float() if L.lo_off else torch.zeros_like(hi)
        out[name] = {"hi": hi, "lo": lo, "val": hi + lo, "raw": False}
    return out


def encode(ws, lay, values):
    """inverse of decode (values: {name: fp32 (B, C, D, H, W)}): hi = RN(v), lo = RN(v - hi), or the raw fp32 pair"""
    for name, buf in lay.bufs.items():
        L, B, v = buf.L, lay.B, values[name]
        if buf.raw:
            planes = [(v[:, :4], 0), (v[:, 4:8], 1)]
            dtype = torch.float32
        else:
            hi = v.to(torch.bfloat16)
            lo = (v - hi.float()).to(torch.bfloat16)
            g = L.C // 8
            planes = [(hi[:, 8 * i:8 * i + 8], i) for i in range(g)]
            if L.lo_off:
                planes += [(lo[:, 8 * i:8 * i + 8], L.lo_off + i) for i in range(g)]
            dtype = torch.bfloat16
        for t, p in planes:
            t = t.permute(0, 2, 3, 4, 1)                     # (B, D, H, W, lanes)
            if L.kind == L_REG:
                _interior(ws, buf, B, dtype)[:, p].copy_(t)
            else:
                subs = _split_interior(ws, buf, B, dtype)
                for s in range(8):
                    subs[s][:, p].copy_(t[:, (s >> 2)::2, ((s >> 1) & 1)::2, (s & 1)::2])


def halo_mask(L):
    """(vs,) bool: True at every guard and halo voxel of one (sub-)volume (the same for every plane, sub-volume and item)"""
    d = L.D // 2 if L.kind == L_SPLIT else L.D
    m = torch.ones(L.vs, dtype=torch.bool)
    m[L.guard: L.guard + (d + 2) * L.zstride].view(d + 2, L.Py, L.Px)[1:-1, 1:-1, 1:-1] = False
    return m


def halos(ws, lay):
    """{name: uint8 (B, volumes, n_halo, 16)} -- the bytes of every guard and halo voxel"""
    out = {}
    for name, buf in lay.bufs.items():
        m = halo_mask(buf.L).to(ws.device)
        out[name] = _region(ws, buf, lay.B, torch.uint8)[:, :, m]
    return out


# ------------------------------------------------------------------------------------------------
# fp64 restatement of each layer kind
# ------------------------------------------------------------------------------------------------
def split_w(w):
    """the packed weight pair as pack_weights_kernel forms it: hi = RN_bf16(w), lo = RN_bf16(w - hi)"""
    hi = w.to(torch.bfloat16)
    return hi.double(), (w - hi.float()).to(torch.bfloat16).double()


def _conv(kind, x, w):
    if kind == "s1":
        return F.conv3d(x, w, stride=1, padding=1)
    if kind == "s2":
        return F.conv3d(x, w, stride=2, padding=1)
    if kind == "cin1_s2":
        return F.conv3d(x, w, stride=(1, 2, 2), padding=1)
    if kind == "t222":
        return F.conv_transpose3d(x, w, stride=2, padding=1, output_padding=1)
    if kind == "t122":
        return F.conv_transpose3d(x, w, stride=(1, 2, 2), padding=1, output_padding=(0, 1, 1))
    raise ValueError(kind)


def _epilogue(acc, S, bias, relu, res):
    if bias is not None:
        b = bias.double().reshape(1, -1, 1, 1, 1)
        acc, S = acc + b, S + b.abs()
    if relu:
        acc = acc.relu()
    if res is not None:
        acc, S = acc + res, S + res.abs()
    return acc, S


def tc_layer(xhi, xlo, w, bias, kind, zsweep, relu=True, res=None):
    """a tensor-core layer: xhi*whi + xlo*whi + xhi*wlo (+ xlo*wlo in the z-sweep programs), then bias, ReLU, residual.
    x*: fp64 (B, Cin, D, H, W); w: fp32 in the ATen layout of the layer; res: fp64 output-shaped or None -> (ref, S)"""
    whi, wlo = split_w(w)
    x, ww = xhi + xlo, whi + wlo
    acc = _conv(kind, x, ww)                          # all four products
    if not zsweep:
        acc = acc - _conv(kind, xlo, wlo)
    S = _conv(kind, x.abs(), ww.abs())
    return _epilogue(acc, S, bias, relu, res)


def fma_layer(x, w, bias, kind, relu):
    """a CUDA-core layer: fp32 input, fp32 weights, fp32 FMAs (conv_cin1, conv_cout1, deconv_cout1)"""
    wd = w.double()
    return _epilogue(_conv(kind, x, wd), _conv(kind, x.abs(), wd.abs()), bias, relu, None)


def bound_ratio(got, ref, S, stored):
    """the accumulation constant this voxel needs: (|got - ref| - storage term) / (2^-23 S), maximum over the tensor"""
    err = (got.double() - ref).abs()
    if stored:
        err = (err - STORE * ref.abs()).clamp(min=0)
    assert bool(torch.isfinite(got).all())
    need = torch.where(err > 0, err / (ULP23 * S), torch.zeros_like(err))
    return float(need.max())


# ------------------------------------------------------------------------------------------------
# CPU: the decoder against the library, the restatements against brute force
# ------------------------------------------------------------------------------------------------
SIZE_SHAPES = [(1, 48, 148, 200), (1, 96, 132, 240), (2, 48, 36, 52), (1, 4, 4, 4), (1, 4, 8, 12), (3, 8, 20, 28)]
UP_SIZE_SHAPES = [(1, 8, 296, 400), (1, 8, 592, 800), (1, 8, 298, 402), (2, 6, 40, 56), (1, 8, 2, 2), (3, 5, 14, 22)]


@pytest.mark.parametrize("prec", ["bf16", "bf16x3"])
def test_decoder_sizes_match_library(prec):
    from effimvs_b200 import capi
    p = {"bf16": capi.PREC_BF16, "bf16x3": capi.PREC_BF16X3}[prec]
    for B, D, H, W in SIZE_SHAPES:
        assert costreg_layout(B, D, H, W, prec == "bf16x3").total == capi.lib.effimvs_costreg_workspace_bytes(B, D, H, W, p)
    for B, D, H, W in UP_SIZE_SHAPES:
        assert cost_up_layout(B, D, H, W, prec == "bf16x3").total == capi.lib.effimvs_cost_up_workspace_bytes(B, D, H, W, p)


@pytest.mark.parametrize("which,shape,hilo,raw", [
    ("costreg", (2, 8, 12, 16), True, False), ("costreg", (1, 4, 8, 12), True, True), ("costreg", (2, 4, 4, 8), False, False),
    ("cost_up", (2, 6, 10, 14), True, True), ("cost_up", (1, 4, 6, 8), True, False), ("cost_up", (2, 4, 2, 2), False, False)])
def test_decoder_round_trip(which, shape, hilo, raw):
    B, D, H, W = shape
    lay = costreg_layout(B, D, H, W, hilo, raw) if which == "costreg" else cost_up_layout(B, D, H, W, hilo, raw)
    gen = torch.Generator().manual_seed(sum(shape))
    vals = {n: torch.randn(B, b.L.C, b.L.D, b.L.H, b.L.W, generator=gen) * 10 for n, b in lay.bufs.items()}
    ws = torch.zeros(lay.total, dtype=torch.uint8)
    encode(ws, lay, vals)
    dec = decode(ws, lay)
    for n, b in lay.bufs.items():
        v = vals[n]
        if b.raw:
            assert torch.equal(dec[n]["val"], v)
            continue
        hi = v.to(torch.bfloat16).float()
        assert torch.equal(dec[n]["hi"], hi)
        if hilo:
            assert torch.equal(dec[n]["lo"], (v - hi).to(torch.bfloat16).float())
            assert float((dec[n]["val"] - v).abs().max()) <= STORE * float(v.abs().max())
        else:
            assert not bool(dec[n]["lo"].any())
    # every byte is either a halo byte (still zero) or an interior byte of exactly one buffer
    hal = halos(ws, lay)
    assert all(not bool(h.any()) for h in hal.values())
    n_interior = sum(b.L.planes * b.L.D * b.L.H * b.L.W * B for b in lay.bufs.values())
    n_halo = sum(h.shape[0] * h.shape[1] * h.shape[2] for h in hal.values())
    assert n_interior + n_halo == sum(b.L.batch_stride * B for b in lay.bufs.values())
    # the vectorised decoder against the ported scalar act_index, voxel by voxel
    for n, b in lay.bufs.items():
        L = b.L
        vox = ws[b.off:].view(-1, 16)
        for _ in range(40):
            bb, c = int(torch.randint(B, (1,), generator=gen)), int(torch.randint(L.C, (1,), generator=gen))
            z, y, x = (int(torch.randint(n_, (1,), generator=gen)) for n_ in (L.D, L.H, L.W))
            if b.raw:
                got = vox[act_index(L, bb, c // 4, z, y, x)].view(torch.float32)[c % 4]
                assert float(got) == float(dec[n]["val"][bb, c, z, y, x])
            else:
                i = act_index(L, bb, c // 8, z, y, x)
                assert float(vox[i].view(torch.bfloat16)[c % 8]) == float(dec[n]["hi"][bb, c, z, y, x])
                if L.lo_off:
                    j = act_index(L, bb, c // 8 + L.lo_off, z, y, x)
                    assert float(vox[j].view(torch.bfloat16)[c % 8]) == float(dec[n]["lo"][bb, c, z, y, x])


def _brute_conv(x, w, stride):
    B, Ci, D, H, W = x.shape
    Co = w.shape[0]
    Do, Ho, Wo = ((n - 1) // s + 1 for n, s in zip((D, H, W), stride))
    out = torch.zeros(B, Co, Do, Ho, Wo, dtype=torch.float64)
    for oz in range(Do):
        for oy in range(Ho):
            for ox in range(Wo):
                for a in range(3):
                    for b in range(3):
                        for c in range(3):
                            iz, iy, ix = oz * stride[0] + a - 1, oy * stride[1] + b - 1, ox * stride[2] + c - 1
                            if 0 <= iz < D and 0 <= iy < H and 0 <= ix < W:
                                out[:, :, oz, oy, ox] += x[:, :, iz, iy, ix] @ w[:, :, a, b, c].T
    return out


def _brute_deconv(x, w, stride):
    """out[s*i + k - 1] += x[i] * w[k] (padding 1, output size s * n)"""
    B, Ci, D, H, W = x.shape
    Co = w.shape[1]
    out = torch.zeros(B, Co, D * stride[0], H * stride[1], W * stride[2], dtype=torch.float64)
    for iz in range(D):
        for iy in range(H):
            for ix in range(W):
                for a in range(3):
                    for b in range(3):
                        for c in range(3):
                            oz, oy, ox = iz * stride[0] + a - 1, iy * stride[1] + b - 1, ix * stride[2] + c - 1
                            if 0 <= oz < out.shape[2] and 0 <= oy < out.shape[3] and 0 <= ox < out.shape[4]:
                                out[:, :, oz, oy, ox] += x[:, :, iz, iy, ix] @ w[:, :, a, b, c]
    return out


@pytest.mark.parametrize("kind,zsweep", [("s1", True), ("s1", False), ("s2", False), ("cin1_s2", False), ("t222", False),
                                         ("t122", False)])
def test_restatement_vs_brute_force(kind, zsweep):
    """the fp64 restatement of each layer kind against the definition on a 3x4x5 volume (for the transposed kinds: every
    output parity class), with the term set of the program written out product by product"""
    gen = torch.Generator().manual_seed(len(kind) + zsweep)
    cin, cout = (1, 3) if kind.startswith("cin1") else (2, 3)
    transposed = kind.startswith("t")
    x = torch.randn(2, cin, 3, 4, 5, generator=gen, dtype=torch.float64)
    w = torch.randn((cin, cout, 3, 3, 3) if transposed else (cout, cin, 3, 3, 3), generator=gen)
    bias = torch.randn(cout, generator=gen)
    xhi = x.to(torch.bfloat16).double()
    xlo = (x - xhi).to(torch.bfloat16).double()
    stride = {"s1": (1, 1, 1), "s2": (2, 2, 2), "cin1_s2": (1, 2, 2), "t222": (2, 2, 2), "t122": (1, 2, 2)}[kind]
    brute = _brute_deconv if transposed else _brute_conv
    whi, wlo = split_w(w)
    terms = brute(xhi, whi, stride) + brute(xlo, whi, stride) + brute(xhi, wlo, stride)
    if zsweep:
        terms = terms + brute(xlo, wlo, stride)
    res = torch.randn(terms.shape, generator=gen, dtype=torch.float64)
    want = (terms + bias.double().reshape(1, -1, 1, 1, 1)).relu() + res
    ref, S = tc_layer(xhi, xlo, w, bias, kind, zsweep, relu=True, res=res)
    assert ref.shape == want.shape
    assert float((ref - want).abs().max()) < 1e-12
    absS = brute((xhi + xlo).abs(), (whi + wlo).abs(), stride) + bias.double().abs().reshape(1, -1, 1, 1, 1) + res.abs()
    assert float((S - absS).abs().max()) < 1e-12
    # the CUDA-core form: fp32 weights, one product per tap
    ref1, _ = fma_layer(x, w, bias, kind, relu=False)
    assert float((ref1 - brute(x, w.double(), stride) - bias.double().reshape(1, -1, 1, 1, 1)).abs().max()) < 1e-12
    # and the term set matters: dropping xhi*wlo is visible at the bound's scale
    assert float(((ref - res) - (terms - brute(xhi, wlo, stride) + bias.double().reshape(1, -1, 1, 1, 1)).relu()).abs().max()) > \
        C_ACC * ULP23 * float(S.max())


def test_bound_ratio_and_canonical_pairs_on_cpu():
    v = torch.randn(1000, generator=torch.Generator().manual_seed(1), dtype=torch.float64)
    S = v.abs() + 1
    assert bound_ratio(v.float(), v, S, stored=False) <= 1.0            # fp32 rounding: half an ulp of |v| <= S
    assert bound_ratio(v.float(), v, S, stored=True) == 0.0
    hi = v.float().to(torch.bfloat16).float()
    lo = (v.float() - hi).to(torch.bfloat16).float()
    assert canonical_violations(hi, lo) == 0
    assert canonical_violations(hi, torch.roll(lo, 1)) > 0               # a lo plane taken from another voxel
    assert canonical_violations(hi, lo * 300) > 0


def canonical_violations(hi, lo):
    """count of voxels whose pair is not (RN(v), RN(v - RN(v))): |lo| <= half an ulp of hi, and hi = RN(hi + lo) except
    when lo is exactly that half ulp (a tie that RN-even may resolve away from hi)"""
    _, e = torch.frexp(hi)                                  # |hi| in [2^(e-1), 2^e): bf16 ulp 2^(e-8)
    half = torch.ldexp(torch.ones_like(hi), e - 9)
    half = torch.where(hi == 0, torch.zeros_like(hi), half)
    ok = lo.abs() <= half
    ok &= ((hi + lo).to(torch.bfloat16).float() == hi) | (lo.abs() == half)
    return int((~ok).sum())


# ------------------------------------------------------------------------------------------------
# GPU: every layer of the nets on a poisoned workspace
# ------------------------------------------------------------------------------------------------
def _switches():
    env = os.environ
    return {"no_zsweep": "EFFIMVS_TC_NO_ZSWEEP" in env, "raw_prob": env.get("EFFIMVS_PROB_PATH") == "raw",
            "cuda_core_prob": "EFFIMVS_CUDA_CORE_PROB" in env, "tc_cout1": "EFFIMVS_TC_COUT1" in env,
            "no_raw": "EFFIMVS_NO_RAW_F32" in env}


def _zsweep(D, cin, sw):
    return D % 4 == 0 and cin in (8, 16) and not sw["no_zsweep"]


def _ws_checks(ws, lay, tag):
    """poison left in the interior, stores into halos and guards, and non-canonical hi/lo pairs"""
    dec = decode(ws, lay)
    for name, h in halos(ws, lay).items():
        assert not bool(h.any()), "{} {}: {} halo/guard bytes written".format(tag, name, int((h != 0).sum()))
    for name, d in dec.items():
        bad = (~torch.isfinite(d["hi"])) | (~torch.isfinite(d["lo"]))
        assert not bool(bad.any()), "{} {}: {} interior values never written".format(tag, name, int(bad.sum()))
        if not d["raw"]:
            n = canonical_violations(d["hi"], d["lo"])
            assert n == 0, "{} {}: {} non-canonical hi/lo pairs".format(tag, name, n)
    return dec


def _poisoned(nbytes):
    return torch.full((nbytes,), 0xFF, dtype=torch.uint8, device=DEV)


def run_costreg(ws_, bs, x):
    from effimvs_b200 import capi, ops
    B, _, D, H, W = x.shape
    lay = costreg_layout(B, D, H, W, True, _switches()["raw_prob"])
    assert lay.total == ops.costreg_workspace_bytes(B, D, H, W, capi.PREC_BF16X3)
    ws = _poisoned(lay.total)
    ops.costreg_prepare(ws_, bs, B, D, H, W, capi.PREC_BF16X3, ws)
    out = ops.costreg_run(x, ws_, bs, capi.PREC_BF16X3, ws)
    return ws, lay, out


def run_cost_up(ws_, bs, x, prev):
    from effimvs_b200 import capi, ops
    B, _, D, H, W = x.shape
    sw = _switches()
    lay = cost_up_layout(B, D, H, W, True, not (sw["tc_cout1"] or sw["no_raw"]))
    assert lay.total == ops.cost_up_workspace_bytes(B, D, H, W, capi.PREC_BF16X3)
    ws = _poisoned(lay.total)
    ops.cost_up_prepare(ws_, bs, B, D, H, W, capi.PREC_BF16X3, ws)
    out = ops.cost_up_run(x, prev, ws_, bs, capi.PREC_BF16X3, ws)
    return ws, lay, out


def check_costreg(ws_, bs, x, tag):
    """-> the workspace and its layout; asserts the workspace checks and every layer's bound"""
    sw = _switches()
    ws, lay, out = run_costreg(ws_, bs, x)
    dec = _ws_checks(ws, lay, tag)
    D, D2 = x.shape[2], x.shape[2] // 2
    hl = lambda n: (dec[n]["hi"].double(), dec[n]["lo"].double())      # noqa: E731
    val = lambda n: dec[n]["val"].double()                               # noqa: E731
    layers = [  # name, got, (ref, S), stored as a hi/lo pair
        ("conv0 cin1", dec["c0"]["val"], fma_layer(x.double(), ws_[0], bs[0], "s1", True), True),
        ("conv1 s1->split", dec["c1"]["val"], tc_layer(*hl("c0"), ws_[1], bs[1], "s1", _zsweep(D, 8, sw)), True),
        ("conv2 s2", dec["c2"]["val"], tc_layer(*hl("c1"), ws_[2], bs[2], "s2", False), True),
        ("conv3 s1->split", dec["c3"]["val"], tc_layer(*hl("c2"), ws_[3], bs[3], "s1", _zsweep(D2, 16, sw)), True),
        ("conv4 s2", dec["c4"]["val"], tc_layer(*hl("c3"), ws_[4], bs[4], "s2", False), True),
        ("conv5 s1", dec["c5"]["val"], tc_layer(*hl("c4"), ws_[5], bs[5], "s1", False), True),
        ("conv6 t222+c3", dec["c6"]["val"], tc_layer(*hl("c5"), ws_[6], bs[6], "t222", False, res=val("c3")), True),
        ("conv7 t222+c1", dec["c7"]["val"], tc_layer(*hl("c6"), ws_[7], bs[7], "t222", False, res=val("c1")),
         not dec["c7"]["raw"]),
    ]
    if sw["raw_prob"] or sw["cuda_core_prob"]:
        layers.append(("prob cuda-core", out, fma_layer(val("c7"), ws_[8], None, "s1", False), False))
    else:
        layers.append(("prob tc", out, tc_layer(*hl("c7"), ws_[8], None, "s1", _zsweep(D, 8, sw), relu=False), False))
    _check_layers(layers, tag)
    return ws, lay


def check_cost_up(ws_, bs, x, prev, tag):
    sw = _switches()
    ws, lay, out = run_cost_up(ws_, bs, x, prev)
    dec = _ws_checks(ws, lay, tag)
    D = x.shape[2]
    cat = dec["cat"]["val"]
    c1 = dec["c1"]
    layers = [
        ("conv0 cin1 s(1,2,2)", cat[:, :8], fma_layer(x.double(), ws_[0], bs[0], "cin1_s2", True), True),
        ("conv_cost cin1", cat[:, 8:], fma_layer(prev.double(), ws_[1], bs[1], "s1", True), True),
        ("conv1 s1", c1["val"], tc_layer(dec["cat"]["hi"].double(), dec["cat"]["lo"].double(), ws_[2], bs[2], "s1",
                                         _zsweep(D, 16, sw)), not c1["raw"]),
    ]
    if sw["tc_cout1"]:
        layers.append(("conv2 t122 tc", out, tc_layer(c1["hi"].double(), c1["lo"].double(), ws_[3], bs[3], "t122", False),
                       False))
    else:
        layers.append(("conv2 t122 cuda-core", out, fma_layer(c1["val"].double(), ws_[3], bs[3], "t122", True), False))
    _check_layers(layers, tag)
    return ws, lay


def _check_layers(layers, tag):
    need = {}
    for name, got, (ref, S), stored in layers:
        assert got.shape == ref.shape, (name, got.shape, ref.shape)
        need[name] = bound_ratio(got, ref, S, stored)
    print("{}: accumulation constant needed per layer (bar {}): {}".format(
        tag, C_ACC, ", ".join("{} {:.2f}".format(k, v) for k, v in need.items())))
    bad = {k: v for k, v in need.items() if not v <= C_ACC}
    assert not bad, "{}: {}".format(tag, bad)
    return need


@pytest.fixture(scope="module")
def _gpu_env():
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    prev = torch.is_grad_enabled()
    torch.set_grad_enabled(False)
    yield
    torch.set_grad_enabled(prev)


@pytest.fixture(scope="module")
def nets(_gpu_env):
    """folded fp32 weights as CudaHotPath passes them: the DTU checkpoint's nets and the golden fixture's"""
    from effimvs_b200 import hotpath
    from util import cspnet, dtu_model, golden, regnet
    hp = hotpath.CudaHotPath("bf16x3")
    m = dtu_model(hp, DEV)
    g = golden("regnets", DEV)
    return {"hp": hp, "model": m,
            "costreg": {"dtu": hp._reg_weights(m.cost_regularization), "golden": hp._reg_weights(regnet(g, DEV))},
            "cost_up": {"dtu_R0": hp._csp_weights(m.CSP_R[0]), "dtu_C1": hp._csp_weights(m.CSP_C[1]),
                        "golden": hp._csp_weights(cspnet(g, DEV))}}


COSTREG_SHAPES = [(1, 48, 148, 200), (1, 96, 132, 240), (2, 48, 36, 52), (1, 4, 4, 4), (1, 4, 8, 12)]
COST_UP_SHAPES = [(1, 8, 296, 400), (1, 8, 592, 800), (1, 8, 264, 480), (1, 8, 528, 960), (1, 8, 298, 402), (2, 6, 40, 56),
                  (1, 8, 2, 2)]


@pytest.mark.gpu
@pytest.mark.parametrize("weights", ["dtu", "golden"])
@pytest.mark.parametrize("shape", COSTREG_SHAPES)
def test_costreg_layers_vs_fp64(nets, shape, weights):
    B, D, H, W = shape
    gen = torch.Generator(device=DEV).manual_seed(D * H + W)
    ws_, bs = nets["costreg"][weights]
    x = torch.randn(B, 1, D, H, W, device=DEV, generator=gen) * 2
    ws, lay = check_costreg(ws_, bs, x, "costreg {} {}".format(weights, shape))
    # the same prepared workspace, other activations: still nothing outside the interiors
    from effimvs_b200 import capi, ops
    ops.costreg_run(torch.randn(B, 1, D, H, W, device=DEV, generator=gen) * 20, ws_, bs, capi.PREC_BF16X3, ws)
    _ws_checks(ws, lay, "costreg second run")


@pytest.mark.gpu
@pytest.mark.parametrize("weights", ["dtu_R0", "dtu_C1", "golden"])
@pytest.mark.parametrize("shape", COST_UP_SHAPES)
def test_cost_up_layers_vs_fp64(nets, shape, weights):
    B, D, H, W = shape
    gen = torch.Generator(device=DEV).manual_seed(D * H + W + len(weights))
    ws_, bs = nets["cost_up"][weights]
    x = torch.randn(B, 1, D, H, W, device=DEV, generator=gen)
    prev = torch.randn(B, 1, D, H // 2, W // 2, device=DEV, generator=gen) * 3
    ws, lay = check_cost_up(ws_, bs, x, prev, "cost_up {} {}".format(weights, shape))
    from effimvs_b200 import capi, ops
    ops.cost_up_run(x * -4, prev * 0.5, ws_, bs, capi.PREC_BF16X3, ws)
    _ws_checks(ws, lay, "cost_up second run")


@pytest.fixture(scope="module")
def recorded(nets):
    """the volumes a synthetic DTU forward (1600 x 1184, 5 views) feeds the regularization nets"""
    from effimvs_b200 import synthetic
    hp, m = nets["hp"], nets["model"]
    calls = {"costreg": [], "cost_up": []}
    reg, up = hp.cost_regularization, hp.cross_scale

    def rec_reg(net, x):
        calls["costreg"].append((net, x.clone()))
        return reg(net, x)

    def rec_up(net, cur, prev):
        calls["cost_up"].append((net, cur.clone(), prev.clone()))
        return up(net, cur, prev)

    hp.cost_regularization, hp.cross_scale = rec_reg, rec_up
    try:
        s = synthetic.make_sample("dtu", seed=11, device=DEV)
        m(s["imgs"], s["proj_matrices"], s["depth_values"])
    finally:
        del hp.cost_regularization, hp.cross_scale
    assert len(calls["costreg"]) == 1 and len(calls["cost_up"]) >= 4
    return calls


@pytest.mark.gpu
def test_layers_vs_fp64_on_forward_volumes(nets, recorded):
    hp = nets["hp"]
    net, x = recorded["costreg"][0]
    assert tuple(x.shape) == (1, 1, 48, 148, 200)
    ws_, bs = hp._reg_weights(net)
    check_costreg(ws_, bs, x, "costreg forward volume {}".format(tuple(x.shape)))
    seen = set()
    for net, cur, prev in recorded["cost_up"]:
        key = (id(net), tuple(cur.shape))
        if key in seen:
            continue
        seen.add(key)
        ws_, bs = hp._csp_weights(net)
        check_cost_up(ws_, bs, cur, prev, "cost_up forward volume {}".format(tuple(cur.shape)))


# ------------------------------------------------------------------------------------------------
# GPU: the shipped switches of conv3d_tc.cu (EFFIMVS_TC_DEBUG is profiling only and deliberately wrong: not here)
# ------------------------------------------------------------------------------------------------
SAME_RESULT = [("EFFIMVS_TC_MAXCTA", "1"), ("EFFIMVS_TC_TWO_TMEM_STAGES", "1")]
COSTREG_TERMS = [("EFFIMVS_TC_NO_ZSWEEP", "1"), ("EFFIMVS_PROB_PATH", "raw"), ("EFFIMVS_CUDA_CORE_PROB", "1")]
COST_UP_TERMS = [("EFFIMVS_TC_NO_ZSWEEP", "1"), ("EFFIMVS_TC_COUT1", "1"), ("EFFIMVS_NO_RAW_F32", "1")]
_ALL_SWITCHES = [k for k, _ in SAME_RESULT + COSTREG_TERMS + COST_UP_TERMS]


@pytest.fixture
def clean_env(monkeypatch):
    for k in _ALL_SWITCHES + ["EFFIMVS_TC_DEBUG"]:
        monkeypatch.delenv(k, raising=False)
    return monkeypatch


def _same_bits(run, monkeypatch, key, value):
    ws0, lay, out0 = run()
    monkeypatch.setenv(key, value)
    ws1, _, out1 = run()
    assert torch.equal(out0, out1), key
    assert torch.equal(ws0[:lay.act_bytes], ws1[:lay.act_bytes]), key


@pytest.mark.gpu
@pytest.mark.parametrize("key,value", SAME_RESULT + COSTREG_TERMS)
def test_costreg_switches(nets, clean_env, key, value):
    ws_, bs = nets["costreg"]["dtu"]
    x = torch.randn(1, 1, 48, 148, 200, device=DEV, generator=torch.Generator(device=DEV).manual_seed(7))
    if (key, value) in SAME_RESULT:
        _same_bits(lambda: run_costreg(ws_, bs, x), clean_env, key, value)
    else:
        clean_env.setenv(key, value)
        check_costreg(ws_, bs, x, "costreg {}={}".format(key, value))


@pytest.mark.gpu
@pytest.mark.parametrize("key,value", SAME_RESULT + COST_UP_TERMS)
@pytest.mark.parametrize("shape", [(1, 8, 296, 400), (1, 8, 592, 800)])
def test_cost_up_switches(nets, clean_env, shape, key, value):
    B, D, H, W = shape
    ws_, bs = nets["cost_up"]["dtu_R0"]
    gen = torch.Generator(device=DEV).manual_seed(H)
    x, prev = torch.randn(B, 1, D, H, W, device=DEV, generator=gen), torch.randn(B, 1, D, H // 2, W // 2, device=DEV, generator=gen)
    if (key, value) in SAME_RESULT:
        _same_bits(lambda: run_cost_up(ws_, bs, x, prev), clean_env, key, value)
    else:
        clean_env.setenv(key, value)
        check_cost_up(ws_, bs, x, prev, "cost_up {} {}={}".format(shape, key, value))


# ------------------------------------------------------------------------------------------------
# GPU: the fp32 CUDA-core nets at the stage shapes against the oracle's nets in fp64
# ------------------------------------------------------------------------------------------------
def _f64(net):
    import copy
    return copy.deepcopy(net).double()


def _rel_to_S(got, ref, S):
    err = (got.double() - ref).abs()
    return float(torch.where(err > 0, err / S, torch.zeros_like(err)).max())


@pytest.mark.gpu
def test_f32_nets_vs_fp64_oracle(nets):
    from effimvs_b200 import hotpath
    from oracle import hotpath as ohp
    hpf, m = hotpath.CudaHotPath("f32"), nets["model"]
    gen = torch.Generator(device=DEV).manual_seed(5)
    x = torch.randn(1, 1, 48, 148, 200, device=DEV, generator=gen) * 2
    got = hpf.cost_regularization(m.cost_regularization, x)
    net64 = _f64(m.cost_regularization)
    ref, pro = ohp.cost_regularization(net64, x.double())
    S = F.conv3d(pro.abs(), net64.prob.weight.abs(), padding=1)
    r = _rel_to_S(got, ref, S)
    print("costreg f32 {}: max |got - ref| / S = {:.2e}".format(tuple(x.shape), r))
    assert r < 1e-5
    for shape, csp in (((1, 1, 8, 296, 400), m.CSP_R[0]), ((1, 1, 8, 592, 800), m.CSP_C[1])):
        x = torch.randn(shape, device=DEV, generator=gen)
        prev = torch.randn(shape[:3] + (shape[3] // 2, shape[4] // 2), device=DEV, generator=gen) * 3
        got = hpf.cross_scale(csp, x, prev)
        net64 = _f64(csp)
        ref, c1 = ohp.cross_scale_net(net64, x.double(), prev.double())
        w, b = hotpath.fold_bn(net64.conv2, True)
        S = _conv("t122", c1.abs(), w.double().abs()) + b.double().abs().reshape(1, -1, 1, 1, 1)
        r = _rel_to_S(got, ref, S)
        print("cost_up f32 {}: max |got - ref| / S = {:.2e}".format(shape, r))
        assert r < 1e-5
