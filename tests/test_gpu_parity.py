"""GPU parity tests (``-m gpu``): the CUDA path, called through the C-ABI (ctypes ->
torch.library ops), against (a) the oracle on the same seeded inputs on the same device and
(b) the golden fixtures produced by upstream itself (tests/golden/make_golden.py).

Tolerances (BASELINE.json north_star): fp32 cost volumes max|d| <= 1e-4 * max|ref|; depth maps
|d depth| <= 1e-3 * (depth_max - depth_min) on >= 99.9 % of pixels; fusion masks identical except
within 1e-5 (relative) of a threshold.
"""
import os

import pytest
import torch

from util import cspnet, dtu_model, golden, pixelwise, regnet, rel_max

pytestmark = pytest.mark.gpu
DEV = "cuda"
DEPTH_RANGE = 935.0 - 425.0


@pytest.fixture(scope="module", autouse=True)
def _strict_fp32():
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.set_grad_enabled(False)
    yield


@pytest.fixture(scope="module")
def hp():
    from effimvs_b200 import hotpath
    return hotpath.CudaHotPath("f32")


@pytest.fixture(scope="module")
def ohp():
    from oracle import hotpath as o
    return o


def frac_within(a, b, tol):
    return float(((a - b).abs() <= tol).float().mean())


# ------------------------------------------------------------------------------------------
# warp + correlation + aggregation
# ------------------------------------------------------------------------------------------
def test_warp_corr_agg_golden(hp):
    g = golden("warp_corr", DEV)
    feats = list(g["feats"])
    got = hp.warp_corr_agg(feats, g["cams"], g["hyp"], g["wts"], g["G"])
    assert rel_max(got, g["agg"]) < 1e-4


@pytest.mark.parametrize("C,G,D,H,W", [(8, 1, 8, 37, 53), (8, 8, 16, 64, 80), (16, 4, 8, 40, 64), (16, 1, 48, 32, 40),
                                       (32, 1, 48, 37, 50), (32, 8, 8, 64, 96), (32, 2, 3, 20, 31)])
@pytest.mark.parametrize("weighted", [True, False])
@pytest.mark.parametrize("channels_last", [False, True])
def test_warp_corr_agg_vs_oracle(hp, ohp, C, G, D, H, W, weighted, channels_last):
    from effimvs_b200 import synthetic
    feats, cams, hyp, wts = synthetic.microbench_inputs(C, D, H, W, views=5, seed=C + D, device=DEV)
    if channels_last:          # NHWC kernels: the maps are read in place, as a channels_last FPN emits them
        feats = [f.contiguous(memory_format=torch.channels_last) for f in feats]
    got = hp.warp_corr_agg(feats, cams, hyp, wts if weighted else None, G)
    sims = [ohp.view_similarity(feats[0], feats[v], cams[:, 0], cams[:, v], hyp, G) for v in range(1, 5)]
    want = ohp.weighted_aggregate(sims, [wts[:, i:i + 1] for i in range(4)]) if weighted else sum(sims) / 4
    assert rel_max(got, want) < 1e-4


def test_warp_corr_agg_per_pixel_hypotheses_and_edge_cases(hp, ohp):
    """Per-pixel hypotheses (HYP_TENSOR), out-of-frustum planes, negative / zero / NaN depths, batch of 2."""
    from effimvs_b200 import synthetic
    gen = torch.Generator().manual_seed(7)
    C, D, H, W = 16, 8, 36, 44
    feats, cams, hyp, wts = synthetic.microbench_inputs(C, D, H, W, views=4, seed=11)
    feats = [torch.cat([f, torch.randn(1, C, H, W, generator=gen)]).to(DEV) for f in feats]
    cams = cams.repeat(2, 1, 1, 1, 1).to(DEV)
    hyp = (hyp.repeat(2, 1, 1, 1) * (0.8 + 0.4 * torch.rand(2, D, H, W, generator=gen))).to(DEV)
    hyp[0, 0] = 30.0
    hyp[1, 1, :5] = -400.0
    hyp[0, 2, 3, 3] = 0.0
    hyp[1, 3, 4, 4] = float("nan")
    wts = wts.repeat(2, 1, 1, 1).to(DEV)
    got = hp.warp_corr_agg(feats, cams, hyp, wts, 2)
    sims = [ohp.view_similarity(feats[0], feats[v], cams[:, 0], cams[:, v], hyp, 2) for v in range(1, 4)]
    want = ohp.weighted_aggregate(sims, [wts[:, i:i + 1] for i in range(3)])
    assert torch.isfinite(got).all()           # NaN coordinates contribute zero, like ATen's CUDA kernel
    ok = torch.isfinite(want)
    assert ok.float().mean() > 0.99
    assert rel_max(got[ok], want[ok]) < 1e-4
    # the same through the tiled (TMA-staged) kernel: channels-last maps, batch of 2, staged and gathered samples mixed
    got_cl = hp.warp_corr_agg([f.contiguous(memory_format=torch.channels_last) for f in feats], cams, hyp, wts, 2)
    assert torch.isfinite(got_cl).all()
    assert rel_max(got_cl[ok], want[ok]) < 1e-4


def test_local_volume_golden_and_oracle(hp, ohp):
    g = golden("local_volume", DEV)
    feats = list(g["feats"])
    sim, hyp = hp.local_volume(g["cur"], feats, g["cams"], g["interval"], g["wts"], 8, 1)
    assert float(((hyp - g["samples"]).abs() / g["samples"]).max()) < 1e-6
    assert rel_max(sim, g["sim"]) < 1e-4
    sim2, _ = hp.local_volume(g["cur"], feats, g["cams"], g["interval"], None, 8, 1)
    assert rel_max(sim2, g["sim_noweights"]) < 1e-4
    o_sim, o_hyp = ohp.local_volume(g["cur"], feats, g["cams"], g["interval"], g["wts"], 8, 1)
    assert torch.equal(hyp, o_hyp)             # hypothesis generation is bit-exact against torch on the device
    assert rel_max(sim, o_sim) < 1e-4


def test_native_projection_matches_torch(hp):
    from effimvs_b200 import hotpath, synthetic
    s = synthetic.make_sample("plumbing", seed=3)
    cams = s["proj_matrices"]["stage2"].to(DEV)
    a = hp.relative_projection(cams)
    b = hotpath.CudaHotPath("f32", native_projection=True).relative_projection(cams)
    assert float(((a - b).abs() / a.abs().clamp(min=1.0)).max()) < 1e-5


# ------------------------------------------------------------------------------------------
# stage 1 (per-view sims + entropy, weighted aggregation, regularization, regression)
# ------------------------------------------------------------------------------------------
def test_stage1_golden(hp):
    g, r = golden("stage1", DEV), golden("regnets", DEV)
    out = hp.stage1(list(g["feats"]), g["cams"], g["hyp"], pixelwise(g, DEV), regnet(r, DEV), 1)
    assert rel_max(out["volume"], g["volume"]) < 1e-4
    assert rel_max(out["view_weights"], g["view_weights"]) < 1e-4
    assert rel_max(out["reg_volume"], g["reg_volume"]) < 1e-4
    assert frac_within(out["depth"], g["depth"], 1e-3 * DEPTH_RANGE) >= 0.999
    assert float((out["photometric_confidence"] - g["conf"]).abs().max()) < 1e-4


def test_stage1_views_entropy_vs_oracle(ohp):
    from effimvs_b200 import capi, ops, synthetic, hotpath
    feats, cams, hyp, _ = synthetic.microbench_inputs(32, 96, 33, 47, views=7, seed=5, device=DEV)
    feats = [f * 0.4 for f in feats]
    proj = hotpath.CudaHotPath().relative_projection(cams)
    sims, ent = ops.warp_corr_views(feats[0], feats[1:], proj, hyp, capi.HYP_TENSOR, 96)
    cl = [f.contiguous(memory_format=torch.channels_last) for f in feats]
    sims_cl, ent_cl = ops.warp_corr_views(cl[0], cl[1:], proj, hyp, capi.HYP_TENSOR, 96)
    assert rel_max(sims_cl, sims) < 1e-5 and float((ent_cl - ent).abs().max()) < 1e-5
    planes = hyp[:, :, 0, 0].contiguous()
    sims_p, ent_p = ops.warp_corr_views(feats[0], feats[1:], proj, planes, capi.HYP_PLANES, 96)
    assert torch.equal(sims, sims_p) and torch.equal(ent, ent_p)
    for v in range(6):
        want = ohp.view_similarity(feats[0], feats[v + 1], cams[:, 0], cams[:, v + 1], hyp, 1)
        assert rel_max(sims[:, v], want[:, 0]) < 1e-4
        assert float((ent[:, v:v + 1] - ohp.similarity_entropy(want)).abs().max()) < 1e-4


def test_softmax_regress_conf_vs_oracle(hp, ohp):
    gen = torch.Generator().manual_seed(3)
    for D in (8, 48, 96):
        logits = (3 * torch.randn(2, D, 19, 23, generator=gen)).to(DEV)
        hyp = (425 + 510 * torch.rand(2, D, 19, 23, generator=gen)).to(DEV)
        d, c = hp.softmax_regress_conf(logits, hyp)
        od, oc = ohp.softmax_regress_confidence(logits, hyp)
        assert float((d - od).abs().max()) < 1e-3 and float((c - oc).abs().max()) < 1e-5
    # peaked distributions at the volume borders exercise the zero-padded 4-bin window
    logits = torch.full((1, 8, 4, 4), -20.0, device=DEV)
    logits[:, 0, :2] = 20.0
    logits[:, 7, 2:] = 20.0
    hyp = torch.linspace(500, 900, 8, device=DEV).reshape(1, 8, 1, 1).expand(1, 8, 4, 4)
    d, c = hp.softmax_regress_conf(logits, hyp)
    od, oc = ohp.softmax_regress_confidence(logits, hyp.contiguous())
    assert float((d - od).abs().max()) < 1e-3 and float((c - oc).abs().max()) < 1e-5


# ------------------------------------------------------------------------------------------
# volume lookup / dynamic cost
# ------------------------------------------------------------------------------------------
def test_lookup_golden_and_oracle(hp, ohp):
    g = golden("lookup", DEV)
    out = hp.dynamic_cost(g["cur"], g["vol_raw"], g["vol_reg"], g["interval"], g["vmin"], g["vmax"], 3)
    assert rel_max(out, g["out6"]) < 1e-4
    gmin, gmax = torch.full((1, 1, 1, 1), 425.0, device=DEV), torch.full((1, 1, 1, 1), 935.0, device=DEV)
    out = hp.dynamic_cost(g["cur"], g["vol_raw"], g["vol_reg"], g["interval"] * 6, gmin, gmax, 3)
    assert rel_max(out, g["out6_global"]) < 1e-4
    look = hp.volume_lookup(g["vol_raw"], g["samples"], gmin, gmax)
    assert rel_max(look, g["look_global"]) < 1e-4
    # samples far outside the volume's range -> zero contribution from out-of-range taps
    far = torch.cat([g["samples"] * 3.0, g["samples"] * 0.3], dim=1)
    assert rel_max(hp.volume_lookup(g["vol_raw"], far, gmin, gmax), ohp.volume_lookup(g["vol_raw"], far, gmin, gmax)) < 1e-4


def test_lookup_fused_half_resolution_view(hp, ohp):
    gen = torch.Generator().manual_seed(5)
    vol = torch.randn(2, 48, 20, 28, generator=gen).to(DEV)
    full = (450 + 450 * torch.rand(2, 8, 40, 56, generator=gen)).to(DEV)
    gmin, gmax = torch.full((2, 1, 1, 1), 425.0, device=DEV), torch.full((2, 1, 1, 1), 935.0, device=DEV)
    low = full[:, :, ::2, ::2]
    got = hp.volume_lookup(vol, low, gmin, gmax)                 # takes the fused stride-2 path
    want = ohp.volume_lookup(vol, low.contiguous(), gmin, gmax)
    assert rel_max(got, want) < 1e-4
    assert torch.equal(got, hp.volume_lookup(vol, low.contiguous(), gmin, gmax))


# ------------------------------------------------------------------------------------------
# 3-D regularization nets, fp32 path
# ------------------------------------------------------------------------------------------
def test_regnets_golden(hp):
    g = golden("regnets", DEV)
    y = hp.cost_regularization(regnet(g, DEV), g["x"])
    assert rel_max(y, g["y"]) < 1e-4
    up = hp.cross_scale(cspnet(g, DEV), g["xs"], g["prev"])
    assert rel_max(up, g["up"]) < 1e-4


@pytest.mark.parametrize("cin,cout,stride,transposed", [(1, 8, (1, 1, 1), False), (8, 16, (2, 2, 2), False), (16, 16, (1, 1, 1), False),
                                                        (32, 32, (1, 1, 1), False), (1, 8, (1, 2, 2), False), (32, 16, (2, 2, 2), True),
                                                        (8, 1, (1, 2, 2), True), (8, 1, (1, 1, 1), False)])
def test_conv3d_layer_vs_aten(cin, cout, stride, transposed):
    import torch.nn.functional as F
    from effimvs_b200 import ops
    gen = torch.Generator().manual_seed(cin * 100 + cout)
    x = torch.randn(2, cin, 8, 10, 12, generator=gen).to(DEV)
    w = (torch.randn((cin, cout, 3, 3, 3) if transposed else (cout, cin, 3, 3, 3), generator=gen) * 0.2).to(DEV)
    b = torch.randn(cout, generator=gen).to(DEV)
    if transposed:
        ref = F.conv_transpose3d(x, w, b, stride=stride, padding=1, output_padding=tuple(s - 1 for s in stride))
    else:
        ref = F.conv3d(x, w, b, stride=stride, padding=1)
    res = torch.randn(ref.shape, generator=gen).to(DEV)
    got = ops.conv3d(x, w, b, res, list(stride), transposed, True)
    assert rel_max(got, torch.relu(ref) + res) < 1e-5


# ------------------------------------------------------------------------------------------
# whole cascade
# ------------------------------------------------------------------------------------------
def test_model_forward_golden(hp):
    from effimvs_b200 import synthetic
    g = golden("model_forward")
    s = synthetic.make_sample("plumbing", seed=g["seed"], width=g["width"], height=g["height"], device=DEV)
    out = dtu_model(hp, DEV)(s["imgs"], s["proj_matrices"], s["depth_values"])
    for i, d in enumerate(out["depth"]):
        assert frac_within(d.cpu(), g["depth{:02d}".format(i)], 1e-3 * DEPTH_RANGE) >= 0.999, i
    assert frac_within(out["photometric_confidence"].cpu(), g["conf"], 1e-3) >= 0.999


@pytest.mark.parametrize("shape,ndepths,size", [("plumbing", "48,8,8", None), ("tanks", "96,8,8", (480, 288))])
def test_model_forward_vs_oracle_on_device(hp, ohp, shape, ndepths, size):
    """640x512 x 5 views (config 1) and a Tanks&Temples-like case: 7 views, 96 stage-1 planes."""
    from effimvs_b200 import synthetic
    kw = {} if size is None else {"width": size[0], "height": size[1]}
    s = synthetic.make_sample(shape, seed=1, device=DEV, **kw)
    cuda_model = dtu_model(hp, DEV, ndepths)
    want = dtu_model(ohp.OracleHotPath(), DEV, ndepths)(s["imgs"], s["proj_matrices"], s["depth_values"])
    got = cuda_model(s["imgs"], s["proj_matrices"], s["depth_values"])
    for i, (a, b) in enumerate(zip(got["depth"], want["depth"])):
        assert frac_within(a, b, 1e-3 * DEPTH_RANGE) >= 0.999, i


# ------------------------------------------------------------------------------------------
# fusion
# ------------------------------------------------------------------------------------------
def _near_threshold(xyd, ref_depth, cx, cy, ks, dist_base, rel_base, rel=1e-5):
    """Pixels whose reprojection distance / depth error lies within `rel` of a ladder threshold,
    `rel` taken relative to the magnitude of the quantities that are subtracted to form the error
    (pixel coordinates up to w, depths up to depth_max): 1e-5 * 1600 px = 0.016 px and
    1e-5 * 935 mm = 0.009 mm at the DTU shape, i.e. ~100 fp32 ulps of those magnitudes -- the
    reprojection is a chain of six fp32 matrix products, so a band in ulps of the operands is the
    tightest statement of the north_star's "identical except within 1e-5 of the thresholds"."""
    e_xy = ((xyd[:, :, 0] - cx) ** 2 + (xyd[:, :, 1] - cy) ** 2).sqrt()
    e_d = (ref_depth - xyd[:, :, 2]).abs()
    band_xy = rel * max(float(cx.max()), float(cy.max()))
    band_d = rel * float(ref_depth.abs().max())
    near = torch.zeros_like(e_xy, dtype=torch.bool)
    for k in ks:
        near |= ((e_xy - k / dist_base).abs() <= band_xy) | ((e_d - k / rel_base).abs() <= band_d)
    return near.any(dim=1, keepdim=True)


@pytest.mark.parametrize("tag", ["mm", "tank"])
@pytest.mark.parametrize("torch_inverse", [True, False])
def test_fusion_golden(tag, torch_inverse):
    from effimvs_b200 import fusion
    g = golden("fusion_" + tag, DEV)
    xyd, _, _ = fusion.get_reproj_dynamic(g["ref_depth"], g["srcs_depth"], g["ref_cam"], g["srcs_cam"], torch_inverse)
    want = g["reproj_xyd"]
    sane = torch.isfinite(want) & (want.abs() < 1e6)
    assert rel_max(xyd[sane], want[sane]) < 1e-4
    out = fusion.filter_view(g["ref_depth"], g["conf"], g["srcs_depth"], g["ref_cam"], g["srcs_cam"], g["dist_base"],
                             g["rel_diff_base"], g["thres_view"], g["prob_threshold"], want_masks=True, torch_inverse=torch_inverse)
    n, v, _, h, w = g["srcs_depth"].shape
    cx = (torch.arange(w, device=DEV) + 0.5).reshape(1, 1, 1, w)
    cy = (torch.arange(h, device=DEV) + 0.5).reshape(1, 1, h, 1)
    near = _near_threshold(want, g["ref_depth"], cx, cy, range(g["thres_view"], v + 1), g["dist_base"], g["rel_diff_base"])
    gm = g["masks"].bool()
    diff = (out["masks"] != gm).any(dim=2).any(dim=1, keepdim=True)
    assert not (diff & ~near).any(), "masks differ away from thresholds"
    keep = ~near
    assert torch.equal(out["final"][keep], g["final"].bool()[keep])
    same = ~diff
    assert rel_max(out["depth_avg"][same], g["depth_avg"][same]) < 1e-5
    assert rel_max(out["points"][same.expand(-1, 3, -1, -1)], g["points"][same.expand(-1, 3, -1, -1)]) < 1e-4


def test_fusion_vs_oracle_full_size():
    """1600x1184 with 10 source views against the oracle on the device (size-independent property:
    identical final masks away from thresholds, averaged depth equal where masks agree)."""
    from effimvs_b200 import fusion, synthetic
    from oracle import fusion as ofu
    h, w, v = 1184, 1600, 10
    E, K = synthetic.camera_ring(v + 1, w, h)
    depths = synthetic.render_plane_scene(E, K, w, h, noise=0.15, seed=4).to(DEV)
    cams = synthetic.stage_cameras(E, K, 1)["stage4"].to(DEV)
    conf = torch.rand(1, h // 2, w // 2, device=DEV)
    args = (depths[0][None, None], conf, depths[1:][None, :, None], cams[:, 0], cams[:, 1:], 2, 6, 2, 0.3)
    got = fusion.filter_view(*args)
    want = ofu.fuse_view(*args)
    cx = (torch.arange(w, device=DEV) + 0.5).reshape(1, 1, 1, w)
    cy = (torch.arange(h, device=DEV) + 0.5).reshape(1, 1, h, 1)
    near = _near_threshold(want["reproj_xyd"], args[0], cx, cy, range(2, v + 1), 2, 6)
    # the band must leave most pixels to compare: measured 0.132 of the pixels have at least one of their 10 views x 9 rungs x 2
    # quantities inside it (1.6e-2 px / 9e-3 mm around each threshold), i.e. 1.9 % of the (pixel, view) pairs
    print("fusion band: {:.4f} of the pixels are excluded".format(float(near.float().mean())))
    assert float(near.float().mean()) < 0.15, float(near.float().mean())
    assert torch.equal(got["final"][~near], want["final"][~near])
    # averaged depth wherever every per-view mask of the ladder agrees (a flipped view changes the average)
    got_m = fusion.filter_view(*args, want_masks=True)["masks"]
    agree = ~(got_m != want["masks"]).any(dim=2).any(dim=1, keepdim=True)
    assert float(agree.float().mean()) > 0.98
    d = (got["depth_avg"] - want["depth_avg"]).abs() * agree
    bad = d > 1e-5 * float(want["depth_avg"].abs().max())
    where = torch.nonzero(bad)[:5].tolist()
    info = [(w_, float(got["depth_avg"][tuple(w_)]), float(want["depth_avg"][tuple(w_)]), float(args[0][tuple(w_)]),
             want["reproj_xyd"][0, :, 2, w_[2], w_[3]].tolist()) for w_ in where]
    # a handful of border pixels may exceed it: where a source sample straddles the image edge the
    # zero-padded bilinear sample has a gradient of ~depth per pixel, which amplifies the 1e-4 px
    # fp32 coordinate noise to ~0.05 mm (observed: 5 of 1.9 M pixels, max 0.043 mm)
    assert int(bad.sum()) <= 1e-5 * bad.numel() and float(d.max()) < 1e-4 * float(want["depth_avg"].abs().max()), \
        (int(bad.sum()), float(d.max()), info)
    assert 0.3 < float(want["final"].float().mean()) < 0.99


# ------------------------------------------------------------------------------------------
# bf16 tensor-core (tcgen05) regularization path
# ------------------------------------------------------------------------------------------
def _bf16(t):
    return t.to(torch.bfloat16).float()


@pytest.mark.parametrize("cin,cout,sd,transposed,dims", [
    (8, 8, 1, False, (4, 6, 10)), (8, 8, 1, False, (8, 20, 36)), (16, 16, 1, False, (6, 12, 20)), (32, 32, 1, False, (4, 10, 14)),
    (16, 8, 1, False, (8, 18, 26)), (8, 1, 1, False, (8, 12, 20)),
    (8, 16, 2, False, (8, 12, 20)), (16, 32, 2, False, (8, 16, 24)),
    (32, 16, 2, True, (3, 5, 7)), (16, 8, 2, True, (4, 9, 13)), (8, 1, 1, True, (8, 10, 14))])
def test_conv3d_bf16_layer_vs_aten(cin, cout, sd, transposed, dims):
    """Every tcgen05 program builder against ATen fp32 on bf16-rounded operands (so that only the
    accumulation order and the final bf16 rounding of the output differ)."""
    import torch.nn.functional as F
    from effimvs_b200 import ops
    gen = torch.Generator().manual_seed(cin * 1000 + cout * 10 + sd)
    D, H, W = dims
    x = _bf16(torch.randn(2, cin, D, H, W, generator=gen)).to(DEV)
    w = _bf16(torch.randn((cin, cout, 3, 3, 3) if transposed else (cout, cin, 3, 3, 3), generator=gen) * 0.2).to(DEV)
    b = torch.randn(cout, generator=gen).to(DEV)
    if transposed:
        ref = F.conv_transpose3d(x, w, b, stride=(sd, 2, 2), padding=1, output_padding=(sd - 1, 1, 1))
    else:
        ref = F.conv3d(x, w, b, stride=sd, padding=1)
    res = _bf16(torch.randn(ref.shape, generator=gen)).to(DEV)
    from effimvs_b200 import capi
    got = ops.conv3d_bf16(x, w, b, res, sd, transposed, True, capi.PREC_BF16)
    want = torch.relu(ref) + res
    assert got.shape == want.shape
    assert rel_max(got, want) < 1e-2          # one bf16 rounding of the output (2^-8 relative)
    assert float((got - want).abs().mean() / want.abs().mean()) < 3e-3
    # hi/lo split operands, three MMAs per product: fp32-grade on un-rounded fp32 operands
    xf = torch.randn(2, cin, D, H, W, generator=gen).to(DEV)
    wf = (torch.randn(w.shape, generator=gen) * 0.2).to(DEV)
    rf = torch.randn(ref.shape, generator=gen).to(DEV)
    if transposed:
        ref3 = F.conv_transpose3d(xf, wf, b, stride=(sd, 2, 2), padding=1, output_padding=(sd - 1, 1, 1))
    else:
        ref3 = F.conv3d(xf, wf, b, stride=sd, padding=1)
    got3 = ops.conv3d_bf16(xf, wf, b, rf, sd, transposed, True, capi.PREC_BF16X3)
    assert rel_max(got3, torch.relu(ref3) + rf) < 1e-4


@pytest.mark.parametrize("prec,tol", [("bf16", 3e-2), ("bf16x3", 2e-4)])
def test_regnets_tensor_core_vs_fp32(prec, tol):
    from effimvs_b200 import hotpath
    g = golden("regnets", DEV)
    hb, hf = hotpath.CudaHotPath(prec), hotpath.CudaHotPath("f32")
    reg, csp = regnet(g, DEV), cspnet(g, DEV)
    y, yf = hb.cost_regularization(reg, g["x"]), hf.cost_regularization(reg, g["x"])
    assert rel_max(y, yf) < tol
    if prec == "bf16x3":
        assert rel_max(y, g["y"]) < 2e-4                               # against upstream's own output
    up, upf = hb.cross_scale(csp, g["xs"], g["prev"]), hf.cross_scale(csp, g["xs"], g["prev"])
    assert rel_max(up, upf) < tol
    gen = torch.Generator().manual_seed(9)
    x = torch.randn(1, 1, 48, 36, 52, generator=gen).to(DEV)          # D = 48 like stage 1
    assert rel_max(hb.cost_regularization(reg, x), hf.cost_regularization(reg, x)) < tol
    xs, prev = torch.randn(2, 1, 8, 40, 56, generator=gen).to(DEV), torch.randn(2, 1, 8, 20, 28, generator=gen).to(DEV)
    assert rel_max(hb.cross_scale(csp, xs, prev), hf.cross_scale(csp, xs, prev)) < tol


def test_regnets_persistent_workspace_equals_plain_call():
    """effimvs_*_ex phases: a workspace prepared once serves repeated runs (bit-identical to the plain
    PREPARE | RUN call, also after other shapes were run in between and with a dirty output buffer), and a
    change of the weights re-prepares it."""
    from effimvs_b200 import hotpath
    g = golden("regnets", DEV)
    keep, plain = hotpath.CudaHotPath("bf16x3"), hotpath.CudaHotPath("bf16x3", persistent_workspaces=False)
    assert keep.persistent_workspaces and not plain.persistent_workspaces
    reg, csp = regnet(g, DEV), cspnet(g, DEV)
    gen = torch.Generator().manual_seed(3)
    x2 = torch.randn(1, 1, 48, 36, 52, generator=gen).to(DEV)
    xs2, prev2 = torch.randn(2, 1, 8, 40, 56, generator=gen).to(DEV), torch.randn(2, 1, 8, 20, 28, generator=gen).to(DEV)
    want = [plain.cost_regularization(reg, g["x"]), plain.cost_regularization(reg, x2),
            plain.cross_scale(csp, g["xs"], g["prev"]), plain.cross_scale(csp, xs2, prev2)]
    for _ in range(3):      # runs 2 and 3 reuse the prepared workspaces; shapes interleaved
        got = [keep.cost_regularization(reg, g["x"]), keep.cost_regularization(reg, x2),
               keep.cross_scale(csp, g["xs"], g["prev"]), keep.cross_scale(csp, xs2, prev2)]
        for a, b in zip(got, want):
            assert torch.equal(a, b)
    assert len(keep._workspaces._store) == 4
    # different activations through the same prepared workspace: nothing of the previous run leaks (halos stay clean)
    x3 = torch.randn(1, 1, 48, 36, 52, generator=gen).to(DEV) * 50
    assert torch.equal(keep.cost_regularization(reg, x3), plain.cost_regularization(reg, x3))
    assert torch.equal(keep.cost_regularization(reg, x2), want[1])
    # new weights (in-place update bumps the version -> new fold -> new stamp -> PREPARE again)
    with torch.no_grad():
        reg.conv1.conv.weight.mul_(1.25)
        csp.conv1.conv.weight.mul_(0.75)
    assert torch.equal(keep.cost_regularization(reg, x2), plain.cost_regularization(reg, x2))
    assert not torch.equal(keep.cost_regularization(reg, x2), want[1])
    assert torch.equal(keep.cross_scale(csp, xs2, prev2), plain.cross_scale(csp, xs2, prev2))


def test_model_forward_tensor_core_tanks_shape():
    """7 views, 96 stage-1 planes through the tcgen05 (bf16x3) regularization against the fp32 CUDA-core nets."""
    from effimvs_b200 import hotpath, synthetic
    s = synthetic.make_sample("tanks", seed=2, device=DEV, width=480, height=288)
    want = dtu_model(hotpath.CudaHotPath("f32"), DEV, "96,8,8")(s["imgs"], s["proj_matrices"], s["depth_values"])
    got = dtu_model(hotpath.CudaHotPath("bf16x3"), DEV, "96,8,8")(s["imgs"], s["proj_matrices"], s["depth_values"])
    fr = [frac_within(a, b, 1e-3 * DEPTH_RANGE) for a, b in zip(got["depth"], want["depth"])]
    assert min(fr) >= 0.999, fr


def test_model_forward_tensor_core_depth_tolerance():
    """north_star: tensor-core (bf16 MMA) regularized depth maps within 1e-3 * (depth_max - depth_min)
    on >= 99.9 % of pixels -- met by the hi/lo split mode (bf16x3).  Plain bf16 operands are measured
    and reported but cannot meet the bound on ambiguous (synthetic, textureless-like) inputs: 2^-8
    relative activation error through nine layers moves the softmax expectation by millimetres."""
    from effimvs_b200 import hotpath, synthetic
    s = synthetic.make_sample("plumbing", seed=1, device=DEV)
    want = dtu_model(hotpath.CudaHotPath("f32"), DEV)(s["imgs"], s["proj_matrices"], s["depth_values"])
    got = dtu_model(hotpath.CudaHotPath("bf16x3"), DEV)(s["imgs"], s["proj_matrices"], s["depth_values"])
    fr = [frac_within(a, b, 1e-3 * DEPTH_RANGE) for a, b in zip(got["depth"], want["depth"])]
    print("bf16x3 vs f32 fraction within tolerance per output:", ["%.4f" % f for f in fr])
    assert min(fr) >= 0.999, fr
    low = dtu_model(hotpath.CudaHotPath("bf16"), DEV)(s["imgs"], s["proj_matrices"], s["depth_values"])
    fl = [frac_within(a, b, 1e-3 * DEPTH_RANGE) for a, b in zip(low["depth"], want["depth"])]
    err = float((low["depth"][-1] - want["depth"][-1]).abs().mean())
    print("plain bf16 vs f32 fraction within tolerance per output:", ["%.4f" % f for f in fl], "mean |d| final = %.3f mm" % err)
    assert err < 1e-2 * DEPTH_RANGE


def test_full_size_dtu_forward_precision_modes_and_graph_replay():
    """BASELINE's full DTU shape (1600x1184, 5 views, 48/8/8 planes): (a) the tensor-core (bf16x3) cascade stays within
    1e-3 * (depth_max - depth_min) of the fp32 CUDA-core cascade on >= 99.9 % of the pixels of every output; (b) the
    forward captured as a CUDA graph (persistent regularization workspaces prepared before capture) is idempotent:
    replaying it on sample A, then on sample B, then on A again gives A's depth maps bit for bit and they agree with the
    eager forward -- nothing of a previous sample survives in the kept workspaces."""
    from effimvs_b200 import hotpath, synthetic
    sa = synthetic.make_sample("dtu", seed=4, device=DEV)
    sb = synthetic.make_sample("dtu", seed=5, device=DEV)
    m3 = dtu_model(hotpath.CudaHotPath("bf16x3", native_projection=True), DEV)
    mf = dtu_model(hotpath.CudaHotPath("f32", native_projection=True), DEV)
    run = lambda m, s: m(s["imgs"], s["proj_matrices"], s["depth_values"])      # noqa: E731
    want, got = run(mf, sa), run(m3, sa)
    assert tuple(got["depth"][-1].shape) == (1, 1184, 1600)
    fr = [frac_within(a, b, 1e-3 * DEPTH_RANGE) for a, b in zip(got["depth"], want["depth"])]
    assert min(fr) >= 0.999, fr                                                                   # (a)
    del mf, want
    static = {"imgs": sa["imgs"].clone(), "depth_values": sa["depth_values"].clone(),
              "proj_matrices": {k: v.clone() for k, v in sa["proj_matrices"].items()}}

    def load(s):
        static["imgs"].copy_(s["imgs"])
        static["depth_values"].copy_(s["depth_values"])
        for k, v in static["proj_matrices"].items():
            v.copy_(s["proj_matrices"][k])
    torch.cuda.synchronize()
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        run(m3, static)
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = run(m3, static)
    snaps = []
    for s in (sa, sb, sa):
        load(s)
        g.replay()
        torch.cuda.synchronize()
        snaps.append(([d.clone() for d in out["depth"]], out["photometric_confidence"].clone()))
    for x, y in zip(snaps[0][0], snaps[2][0]):
        assert torch.equal(x, y)                                                                  # (b) idempotent
    assert torch.equal(snaps[0][1], snaps[2][1])
    assert not torch.equal(snaps[0][0][-1], snaps[1][0][-1])                                      # B really ran
    fg = [frac_within(a, b, 1e-3 * DEPTH_RANGE) for a, b in zip(snaps[0][0], got["depth"])]
    assert min(fg) >= 0.999, fg                                                                   # graph == eager (cuDNN may pick other algorithms)


# ------------------------------------------------------------------------------------------
# end-to-end pipeline (host in, host out; H2D of sample k+1 overlapped with the forward of sample k)
# ------------------------------------------------------------------------------------------
def test_pipeline_matches_direct_forward(hp):
    from effimvs_b200 import pipeline, synthetic
    model = dtu_model(hp, DEV)
    samples = [synthetic.make_sample("plumbing", seed=s, width=256, height=192) for s in (0, 1, 2)]
    host = [{"imgs": s["imgs"].pin_memory(), "depth_values": s["depth_values"].pin_memory(),
             "proj_matrices": {k: v.pin_memory() for k, v in s["proj_matrices"].items()}} for s in samples]
    pipe = pipeline.DepthMapPipeline(model, host[0], slots=2)
    tickets, got = [], []
    for i, h in enumerate(host):                       # 3 samples through 2 slots: slot 0 is reused
        tickets.append(pipe.submit(h))
        if i >= 1:
            d, c = pipe.result(tickets[i - 1])
            got.append((d.clone(), c.clone()))
    d, c = pipe.result(tickets[-1])
    got.append((d.clone(), c.clone()))
    for s, (d, c) in zip(samples, got):
        want = model(s["imgs"].to(DEV), {k: v.to(DEV) for k, v in s["proj_matrices"].items()}, s["depth_values"].to(DEV))
        assert frac_within(d, want["depth"][-1].cpu(), 1e-3 * DEPTH_RANGE) >= 0.999
        assert frac_within(c, want["photometric_confidence"].cpu(), 1e-3) >= 0.999


def test_pipeline_8bit_images_equal_fp32_images(hp):
    """8-bit host images (a quarter of the PCIe bytes) divided by 255 on the device give the depth maps of the fp32 host
    images upstream's loaders form (np.float32 / 255., datasets/general_eval.py:83-87) bit for bit; the conversion kernel
    itself equals the NumPy expression for all 256 values and for unaligned / ragged sizes."""
    import numpy as np
    from effimvs_b200 import ops, pipeline, synthetic
    for n, off in ((256, 0), (1000003, 0), (4099, 3), (7, 1)):
        u8 = torch.arange(n + off, dtype=torch.int64).remainder(256).to(torch.uint8)[off:]
        dev_u8 = torch.arange(n + off, device=DEV, dtype=torch.int64).remainder(256).to(torch.uint8)[off:]
        out = torch.empty(n, device=DEV)
        ops.images_u8_to_f32(dev_u8.contiguous(), out)
        assert np.array_equal(out.cpu().numpy(), u8.numpy().astype(np.float32) / np.float32(255.0))
    model = dtu_model(hp, DEV)
    s = synthetic.make_sample("plumbing", seed=3, width=256, height=192)
    u8 = (s["imgs"] * 255.0).round().clamp(0, 255).to(torch.uint8)
    f32 = torch.from_numpy(u8.numpy().astype(np.float32) / np.float32(255.0))
    rest = {"depth_values": s["depth_values"].pin_memory(), "proj_matrices": {k: v.pin_memory() for k, v in s["proj_matrices"].items()}}
    pipe = pipeline.DepthMapPipeline(model, dict(rest, imgs=f32.pin_memory()), slots=2)
    a = [t.clone() for t in pipe.result(pipe.submit(dict(rest, imgs=f32.pin_memory())))]
    b = [t.clone() for t in pipe.result(pipe.submit(dict(rest, imgs=u8.pin_memory())))]
    c = [t.clone() for t in pipe.result(pipe.submit(dict(rest, imgs=u8.pin_memory())))]       # the other slot
    assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1]) and torch.equal(b[0], c[0])
    assert pipe.h2d_bytes(dict(rest, imgs=u8)) < 0.27 * pipe.h2d_bytes(dict(rest, imgs=f32))
    pipe8 = pipeline.DepthMapPipeline(model, dict(rest, imgs=u8.pin_memory()), slots=1)       # a pipeline built from 8-bit images
    d = pipe8.result(pipe8.submit(dict(rest, imgs=u8.pin_memory())))
    assert torch.equal(d[0], a[0])


# ------------------------------------------------------------------------------------------
# remaining upstream-named call sites (SURVEY.md section 8(b)): homo_warping_new, get_depth_range_samples,
# vis_filter_dynamic
# ------------------------------------------------------------------------------------------
def test_homo_warping_new_dropin_golden_and_oracle(ohp):
    from effimvs_b200 import dropin
    g = golden("warp_corr", DEV)
    feats, cams, hyp = list(g["feats"]), g["cams"], g["hyp"]
    P = [ohp.compose_projection(cams[:, v]) for v in range(len(feats))]
    got = dropin.homo_warping_new(feats[1], P[1], P[0], hyp)
    assert got.shape == (1, 8, 6, 20, 28)
    assert rel_max(got.reshape(g["warped1"].shape), g["warped1"]) < 1e-4
    planes = (1.0 / torch.linspace(1 / 935.0, 1 / 425.0, 5, device=DEV)).reshape(1, 5)
    a = dropin.homo_warping_new(feats[2], P[2], P[0], planes)
    b = ohp.homo_warp(feats[2], P[2], P[0], planes.reshape(1, 5, 1, 1).expand(1, 5, 20, 28).contiguous())
    assert rel_max(a, b) < 1e-4


def test_get_depth_range_samples_dropin_bit_exact(ohp):
    from effimvs_b200 import dropin
    gen = torch.Generator().manual_seed(1)
    inv = (1.0 / (430 + 500 * torch.rand(2, 30, 44, generator=gen))).to(DEV)
    inv[0, 0, :3] = torch.tensor([1e-6, 2e4, 5e-5], device=DEV)            # exercise the clamps
    interval = torch.tensor([1e-5, 3e-6], device=DEV).reshape(2, 1, 1, 1)
    for nd in (3, 8):
        got = dropin.get_depth_range_samples(inv, nd, interval.squeeze(1), shape=[2, 30, 44])
        want = ohp.local_inverse_depth_samples(inv, nd, interval.squeeze(1))
        assert torch.equal(got, want)
    dv = torch.linspace(1 / 935.0, 1 / 425.0, 384, device=DEV).unsqueeze(0)
    assert torch.equal(dropin.get_depth_range_samples(dv, 48, None, shape=[1, 6, 7]), ohp.uniform_inverse_depth_samples(dv, 48, 6, 7))


@pytest.mark.parametrize("tag", ["mm", "tank"])
def test_vis_filter_dynamic_dropin_golden(tag):
    from effimvs_b200 import fusion
    g = golden("fusion_" + tag, DEV)
    masks, mask = fusion.vis_filter_dynamic(g["ref_depth"], g["reproj_xyd"], None, None, dist_base=g["dist_base"],
                                            rel_diff_base=g["rel_diff_base"], thres_view=g["thres_view"])
    assert torch.equal(masks, g["masks"].bool())          # same reproj_xyd in -> identical masks
    assert torch.equal(mask, g["masks"].bool()[:, :, -1:])


# ---- SURVEY section 8(f) row 3: update-block glue kernels ------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("h,cx,H,W", [(16, 4, 37, 53), (32, 8, 24, 40), (48, 12, 19, 25)])
def test_gru_init_and_encoder_tail_ctx_vs_torch(h, cx, H, W):
    """gru_init (tanh of the hidden half of the context map into hx) and the encoder tail with the context term
    formed in the kernel (relu on the fly, channel range of the map) against the torch chain
    (models/Effi_MVS_plus.py:464-466, models/update.py:93-95)."""
    import torch.nn.functional as F
    from effimvs_b200 import ops
    gen = torch.Generator(device=DEV).manual_seed(h)
    rnd = lambda *s: torch.randn(*s, device=DEV, generator=gen)      # noqa: E731
    B, hm = 2, h - cx
    ctx_map = rnd(B, h + cx, H, W).contiguous(memory_format=torch.channels_last)
    hx = ops.gru_init(ctx_map, h)
    assert hx.shape == (B, 2 * h, H, W) and hx.is_contiguous(memory_format=torch.channels_last)
    assert float((hx[:, :h] - torch.tanh(ctx_map[:, :h])).abs().max()) < 1e-6
    m, w_m, w_ctx, bias = rnd(B, hm, H, W), rnd(h, hm, 1, 1) * 0.2, rnd(h, cx, 1, 1) * 0.2, rnd(h) * 0.1
    context = torch.relu(ctx_map[:, h:])
    want = torch.relu(F.conv2d(m, w_m) + F.conv2d(context, w_ctx, bias))
    keep = hx[:, :h].clone()
    ops.encoder_tail_ctx(m, w_m, ctx_map, h, cx, True, w_ctx, bias, hx)           # channel range of the map, relu in the kernel
    assert rel_max(hx[:, h:], want) < 1e-5 and torch.equal(hx[:, :h], keep)
    hx2 = torch.zeros_like(hx)
    ops.encoder_tail_ctx(m, w_m, context.contiguous(), 0, cx, False, w_ctx, bias, hx2)   # an already activated planar context tensor
    assert rel_max(hx2[:, h:], want) < 1e-5
    ctx_term = F.conv2d(context, w_ctx, bias)
    hx3 = torch.zeros_like(hx)
    ops.encoder_tail(m, w_m, ctx_term, hx3)                                        # the precomputed-term form agrees
    assert rel_max(hx3[:, h:], hx2[:, h:]) < 1e-5


@pytest.mark.gpu
@pytest.mark.parametrize("B,Dv,D1", [(1, 48, 48), (3, 192, 48), (2, 7, 96)])
def test_depth_ranges_is_bit_identical_to_the_torch_expressions(B, Dv, D1):
    """depth_ranges: everything the cascade derives from depth_values alone (upstream models/Effi_MVS_plus.py:409-424 and the
    plane sweep of get_depth_range_samples, models/module.py:577-585) from one kernel, against the torch expressions of
    net.EffiMVSPlus.forward_from_features bit for bit."""
    from effimvs_b200 import ops
    gen = torch.Generator(device=DEV).manual_seed(Dv)
    lo = 1.0 / (900.0 + 100.0 * torch.rand(B, 1, device=DEV, generator=gen))
    hi = 1.0 / (400.0 + 50.0 * torch.rand(B, 1, device=DEV, generator=gen))
    depth_values = lo + (hi - lo) * torch.linspace(0, 1, Dv, device=DEV).reshape(1, Dv)
    R = ops.depth_ranges(depth_values, D1, [4.0, 2.0, 1.0])
    row = lambda i: R[i * B:(i + 1) * B]      # noqa: E731
    disp_min, disp_max = depth_values[:, 0], depth_values[:, -1]
    far, near = disp_min.reciprocal(), disp_max.reciprocal()
    unit = (disp_max - disp_min) / depth_values.size(1)
    want = [far, near, far.reciprocal(), near.reciprocal(), unit * 4, unit * 2, unit * 1, torch.zeros_like(far)]
    for i, w in enumerate(want):
        assert torch.equal(row(i), w), "row {}".format(i)
    assert torch.equal(far, 1.0 / disp_min)                         # what upstream writes (Effi_MVS_plus.py:413)
    k = torch.arange(D1, device=DEV, dtype=torch.float32).reshape(1, D1)
    inv_s = disp_min.reshape(B, 1) + k * ((disp_max - disp_min).reshape(B, 1) / (D1 - 1))
    assert torch.equal(R[8 * B:].reshape(B, D1), inv_s.reciprocal())


@pytest.mark.gpu
def test_inv_init_is_bit_identical_to_the_torch_chain():
    """inv_init = depth_to_disp + disp_to_depth of a stage's depth estimate (models/Effi_MVS_plus.py:138-164) in one kernel:
    the same bits as torch's reciprocal / sub / div / mul / add / clamp / reciprocal chain, per-batch ranges."""
    from effimvs_b200 import ops
    gen = torch.Generator(device=DEV).manual_seed(11)
    B, H, W = 2, 148, 201
    cur = 425.0 + 510.0 * torch.rand(B, 1, H, W, device=DEV, generator=gen)
    cur[0, 0, 0, :4] = torch.tensor([1e-3, 1e6, 425.0, 935.0], device=DEV)
    dmin, dmax = torch.tensor([425.0, 300.0], device=DEV), torch.tensor([935.0, 1200.0], device=DEV)
    far, near = dmin.reciprocal(), dmax.reciprocal()                 # the cascade's lo_disp / hi_disp: double reciprocals
    lo, hi = far.reciprocal().reshape(B, 1, 1, 1), near.reciprocal().reshape(B, 1, 1, 1)
    inv, depth = ops.inv_init(cur, lo.reshape(B), hi.reshape(B))
    want_inv = (cur.reciprocal() - lo) / ((hi - lo) + 1e-10)
    want_depth = 1.0 / (lo + (hi - lo) * want_inv).clamp(min=1e-4)
    assert torch.equal(inv, want_inv) and torch.equal(depth, want_depth)
    inv2, depth2 = ops.gru_delta(None, None, want_inv, lo.reshape(B), hi.reshape(B))     # the two-step form it replaces
    assert torch.equal(inv2, inv) and torch.equal(depth2, depth)


@pytest.mark.gpu
@pytest.mark.parametrize("h,cx,H,W", [(16, 4, 37, 53), (32, 8, 24, 40), (48, 12, 19, 25), (16, 4, 592, 800)])
def test_gru_init_ctx_vs_torch(h, cx, H, W):
    """gru_init_ctx: the GRU start state and the iteration-invariant context term of the encoder tail (the aux map of conv2d_tc's
    ADD_RELU epilogue) in one pass over the context map, against tanh / relu / conv1x1 + bias in torch with fp32 products
    (models/Effi_MVS_plus.py:464-466, models/update.py:93-95); the last case is the DTU stage-3 map."""
    import torch.nn.functional as F
    from effimvs_b200 import ops
    gen = torch.Generator(device=DEV).manual_seed(h + W)
    rnd = lambda *s: torch.randn(*s, device=DEV, generator=gen)      # noqa: E731
    B = 2 if H < 100 else 1
    ctx_map = rnd(B, h + cx, H, W).contiguous(memory_format=torch.channels_last)
    w_ctx, bias = rnd(h, cx, 1, 1) * 0.3, rnd(h) * 0.1
    hx, term = ops.gru_init_ctx(ctx_map, h, w_ctx.contiguous(memory_format=torch.channels_last), bias)
    assert hx.shape == (B, 2 * h, H, W) and hx.is_contiguous(memory_format=torch.channels_last)
    assert term.shape == (B, h, H, W) and term.is_contiguous(memory_format=torch.channels_last)
    assert torch.equal(hx[:, :h], ops.gru_init(ctx_map, h)[:, :h])
    saved = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False
    try:
        want = F.conv2d(torch.relu(ctx_map[:, h:]), w_ctx, bias)
    finally:
        torch.backends.cudnn.allow_tf32 = saved
    assert rel_max(term, want) < 1e-5


@pytest.mark.gpu
@pytest.mark.parametrize("h,B,H,W", [(16, 2, 37, 70), (32, 1, 24, 129), (48, 2, 19, 25), (16, 1, 3, 2), (64, 1, 9, 66)])
def test_delta_head_vs_torch(h, B, H, W):
    """DepthHead.conv2 + tanh + inverse-depth step + disp_to_depth in one kernel against the torch chain
    (upstream models/update.py:19-27, 121-125; Effi_MVS_plus.py:138-148): zero padding at every border, tile edges
    (64-column x 4-row blocks), planar and channels-last inputs."""
    import torch.nn.functional as F
    from effimvs_b200 import ops
    gen = torch.Generator(device=DEV).manual_seed(h + W)
    rnd = lambda *s: torch.randn(*s, device=DEV, generator=gen)      # noqa: E731
    t, w, bias = torch.relu(rnd(B, h, H, W)), rnd(1, h, 3, 3) * 0.1, rnd(1) * 0.1
    inv = torch.rand(B, 1, H, W, device=DEV, generator=gen)
    lo, hi = torch.full((B,), 1 / 935.0, device=DEV), torch.full((B,), 1 / 425.0, device=DEV)
    hi[-1] = 1 / 300.0
    want_inv = inv + torch.tanh(F.conv2d(t, w, bias, padding=1))
    want_depth = 1.0 / (lo.reshape(B, 1, 1, 1) + (hi - lo).reshape(B, 1, 1, 1) * want_inv).clamp(min=1e-4)
    for tt in (t, t.contiguous(memory_format=torch.channels_last)):
        got_inv, got_depth = ops.delta_head(tt, w, bias, inv, lo, hi)
        assert got_inv.shape == inv.shape and got_depth.shape == inv.shape
        assert float((got_inv - want_inv).abs().max()) < 2e-5
        assert rel_max(got_depth, want_depth) < 2e-5
    with pytest.raises(Exception):
        ops.delta_head(torch.relu(rnd(1, 24, 8, 8)), rnd(1, 24, 3, 3), bias, torch.rand(1, 1, 8, 8, device=DEV), lo[:1], hi[:1])


@pytest.mark.gpu
@pytest.mark.parametrize("h,H,W", [(16, 37, 53), (32, 24, 40), (48, 19, 25)])
def test_update_glue_kernels_vs_torch(h, H, W):
    """each glue kernel against the torch elementwise chain it replaces (upstream models/update.py:41-48, 27,
    121-125; Effi_MVS_plus.py:138-148, 167-178), same device, fp32"""
    from effimvs_b200 import ops, net
    gen = torch.Generator(device=DEV).manual_seed(h)
    B = 2
    cl = lambda t: t.contiguous(memory_format=torch.channels_last)   # noqa: E731
    rnd = lambda *s: torch.randn(*s, device=DEV, generator=gen)      # noqa: E731
    zr_pre, q_pre, hv, x = cl(rnd(B, 2 * h, H, W) * 2), cl(rnd(B, h, H, W) * 2), cl(torch.tanh(rnd(B, h, H, W))), cl(torch.relu(rnd(B, h, H, W)))
    bz, br, bq = rnd(h), rnd(h), rnd(h)
    hx = cl(torch.cat([hv, x], dim=1))
    z = torch.sigmoid(zr_pre[:, :h] + bz.reshape(1, -1, 1, 1))
    r = torch.sigmoid(zr_pre[:, h:] + br.reshape(1, -1, 1, 1))
    assert float((ops.gru_reset(zr_pre, br, hx) - torch.cat([r * hv, x], dim=1)).abs().max()) <= 2e-7
    want = (1 - z) * hv + z * torch.tanh(q_pre + bq.reshape(1, -1, 1, 1))
    got = ops.gru_update(zr_pre, bz, q_pre, bq, hx)
    assert float((got - want).abs().max()) <= 2e-7        # tanhf / expf: same libdevice functions, at most an ulp of the sum
    assert torch.equal(hx[:, :h], got) and torch.equal(hx[:, h:], x)
    # inverse-depth step + disp_to_depth
    lo, hi = torch.tensor([1 / 935.0, 1 / 1000.0], device=DEV), torch.tensor([1 / 425.0, 1 / 400.0], device=DEV)
    inv, pre, b1 = torch.rand(B, 1, H, W, device=DEV, generator=gen), rnd(B, 1, H, W), rnd(1)
    to_depth = lambda v: 1.0 / (lo.reshape(B, 1, 1, 1) + (hi - lo).reshape(B, 1, 1, 1) * v).clamp(min=1e-4)   # noqa: E731
    inv2, dep2 = ops.gru_delta(pre, b1, inv, lo, hi)
    want_inv = inv + torch.tanh(pre + b1)
    assert float((inv2 - want_inv).abs().max()) <= 2e-7
    assert rel_max(dep2, to_depth(inv2)) <= 2e-7
    inv0, dep0 = ops.gru_delta(None, None, inv, lo, hi)
    assert torch.equal(inv0, inv) and rel_max(dep0, to_depth(inv)) <= 2e-7
    # convex upsampling
    mask_pre, mb = cl(rnd(B, 36, H, W) * 3), rnd(36)
    up, dup = ops.convex_upsample(mask_pre, mb, 0.25, inv, lo, hi, 2)
    want_up = net.convex_upsample(inv, 0.25 * (mask_pre + mb.reshape(1, -1, 1, 1)), 2)
    assert float((up - want_up).abs().max()) <= 1e-6
    assert rel_max(dup, to_depth(up.unsqueeze(1)).squeeze(1)) <= 2e-7
    # the same with the mask head's 1x1 convolution folded into the kernel
    import torch.nn.functional as F
    t, mw = torch.relu(rnd(B, 2 * h, H, W)), rnd(36, 2 * h, 1, 1) * 0.3
    for tt in (t, cl(t)):
        up2, dup2 = ops.convex_upsample_conv(tt, mw, mb, 0.25, inv, lo, hi, 2)
        want2 = net.convex_upsample(inv, 0.25 * (F.conv2d(t, mw) + mb.reshape(1, -1, 1, 1)), 2)
        assert float((up2 - want2).abs().max()) <= 2e-6
        assert rel_max(dup2, to_depth(up2.unsqueeze(1)).squeeze(1)) <= 2e-7


@pytest.mark.gpu
def test_update_block_fused_golden(hp):
    """UpdateBlock.forward_fused (cuDNN convolutions + glue kernels) against upstream's BasicUpdateBlock,
    upsample_depth and disp_to_depth (tests/golden/update_block.npz)"""
    from test_net_host import load_update_block, _update_cost_fn
    g = golden("update_block", DEV)
    blk = load_update_block(g, DEV)
    B = g["inv0"].shape[0]
    lo, hi = (1.0 / g["dmax"]).reshape(B), (1.0 / g["dmin"]).reshape(B)
    with torch.no_grad():
        n, invs, deps, up, dup, _ = blk.forward_fused(hp, g["net0"], _update_cost_fn, g["inv0"], g["context"], 3, lo, hi)
    assert rel_max(n, g["net"]) < 1e-4
    for i in range(3):
        assert float((invs[i] - g["inv{}".format(i + 1)]).abs().max()) < 1e-4
        assert rel_max(deps[i], g["depth{}".format(i + 1)]) < 1e-4
    assert float((up - g["up"]).abs().max()) < 1e-4 and rel_max(dup, g["depth_up"]) < 1e-4


@pytest.mark.gpu
def test_update_block_fused_equals_plain_at_dtu_stage3(hp):
    """full DTU stage-3 size (800x592, hidden 16): fused and plain paths agree on the same device"""
    from test_net_host import _update_cost_fn
    from effimvs_b200 import net
    torch.manual_seed(3)
    blk = net.UpdateBlock(16, 6, 2, 4).to(DEV).eval()
    B, H, W = 1, 592, 800
    n0, ctx = torch.tanh(torch.randn(B, 16, H, W, device=DEV)), torch.relu(torch.randn(B, 4, H, W, device=DEV))
    inv0 = torch.rand(B, 1, H, W, device=DEV)
    lo, hi = torch.tensor([1 / 935.0], device=DEV), torch.tensor([1 / 425.0], device=DEV)
    to_depth = lambda v: 1.0 / (lo.reshape(B, 1, 1, 1) + (hi - lo).reshape(B, 1, 1, 1) * v).clamp(min=1e-4)   # noqa: E731
    with torch.no_grad():
        n, invs, deps, up, dup, _ = blk.forward_fused(hp, n0, _update_cost_fn, inv0, ctx, 3, lo, hi)
        n_p, mask_p, invs_p = blk(n0, _update_cost_fn, inv0, ctx, 3, to_depth)
        up_p = net.convex_upsample(invs_p[-1], mask_p, 2)
    assert rel_max(n, n_p) < 1e-4 and float((invs[-1] - invs_p[-1]).abs().max()) < 1e-4
    assert float((up - up_p).abs().max()) < 1e-4 and rel_max(dup, to_depth(up_p.unsqueeze(1)).squeeze(1)) < 1e-4


# ---- SURVEY section 8(f) row 2: DTU geometric filter -------------------------------------------------------
def _dtu_filter_compare(out, want_final, want_geo, want_avg, want_pts, dist_band, diff_band):
    """masks identical except where a rung is decided within the band (float64 rounding of the matrix
    products); averaged depth / points equal wherever the masks agree"""
    import numpy as np
    final, geo = out["final"].cpu().numpy(), out["geo"].cpu().numpy()
    bad_geo = float((geo != want_geo).mean())
    bad_final = float((final != want_final).mean())
    assert bad_geo <= dist_band and bad_final <= dist_band, (bad_geo, bad_final)
    same = geo == want_geo
    avg = out["depth_avg"].cpu().numpy()
    close = np.abs(avg - want_avg) <= 1e-6 * np.maximum(np.abs(want_avg), 1.0)
    assert float((close | ~same).mean()) >= 1.0 - diff_band
    pts = out["points"].cpu().numpy()
    ok = (np.abs(pts - want_pts).max(axis=0) <= 1e-3) | ~close
    assert float(ok.mean()) == 1.0


@pytest.mark.gpu
def test_dtu_filter_golden():
    """effimvs_dtu_filter_f32 against upstream's own functions + real cv2.remap (tests/golden/dtu_filter.npz)"""
    import numpy as np
    from effimvs_b200 import fusion
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "dtu_filter.npz"))
    d, K, E = z["depths"], z["K"], z["E"]
    v = d.shape[0] - 1
    dev_d = torch.from_numpy(d).to(DEV)
    out = fusion.dtu_filter_view(dev_d[0], torch.from_numpy(z["confidence"]).to(DEV), dev_d[1:], K, E[0], [K] * v, list(E[1:]),
                                 float(z["conf_thres"]), want_masks=True)
    masks = out["masks"].cpu().numpy()
    assert float((masks != z["masks"]).mean()) <= 1e-5           # a rung decided within ~1e-12 of its threshold
    rep = out["reproj_depth"].cpu().numpy()
    agree = (masks[:, -1] == z["masks"][:, -1])
    assert float(((np.abs(rep - z["reproj_depth"]) <= 1e-6 * np.maximum(z["reproj_depth"], 1.0)) | ~agree).mean()) == 1.0
    _dtu_filter_compare(out, z["final_mask"], z["geo_mask"], z["depth_avg"], z["points"], 1e-5, 1e-5)


@pytest.mark.gpu
def test_dtu_filter_vs_oracle_dtu_size():
    """a 1600x1184 reference view with 10 source views against the NumPy oracle (no cv2 needed on the GPU box)"""
    from effimvs_b200 import fusion, synthetic
    from oracle import dtu_filter as o
    h, w, v = 1184, 1600, 10
    E, K = synthetic.camera_ring(v + 1, w, h)
    depths = synthetic.render_plane_scene(E, K, w, h, noise=0.05, seed=2)
    depths[2, 100:300, 200:500] += 3.0
    conf = torch.rand(h // 2, w // 2, generator=torch.Generator().manual_seed(0))
    conf_full = torch.nn.functional.interpolate(conf[None, None], size=(h, w), mode="bilinear", align_corners=False)[0, 0]
    K32, E32 = K.numpy().astype("float32"), E.numpy().astype("float32")
    want = o.filter_view(depths[0].numpy(), conf_full.numpy(), depths[1:].numpy(), K32, E32[0], [K32] * v, list(E32[1:]), 0.5)
    out = fusion.dtu_filter_view(depths[0].to(DEV), conf.to(DEV), depths[1:].to(DEV), K32, E32[0], [K32] * v, list(E32[1:]), 0.5)
    assert 0.05 < want["final"].mean() < 0.95
    # the resized confidence is compared with a threshold too: allow pixels whose confidence sits within 1e-6 of 0.5 / 0.75
    _dtu_filter_compare(out, want["final"], want["geo"], want["depth_avg"], want["points"], 2e-5, 2e-5)


@pytest.mark.gpu
@pytest.mark.parametrize("h,H,W", [(16, 37, 53), (32, 24, 70), (48, 19, 25), (16, 148, 201)])
def test_encoder_head_vs_torch(h, H, W, monkeypatch):
    """effimvs_encoder_head_f32 against relu(conv2d) of upstream's ProjectionInput head (models/update.py:88-91)"""
    import torch.nn.functional as F
    from effimvs_b200 import ops
    gen = torch.Generator(device=DEV).manual_seed(h)
    rnd = lambda *s: torch.randn(*s, device=DEV, generator=gen)      # noqa: E731
    B, CD = 2, 6
    cost, inv = rnd(B, CD, H, W), torch.rand(B, 1, H, W, device=DEV, generator=gen)
    wc1, bc1, wd1, bd1 = rnd(h, CD, 1, 1) * 0.3, rnd(h), rnd(h, 1, 7, 7) * 0.2, rnd(h)
    monkeypatch.setenv("EFFIMVS_EH_CONST", "1")                        # (by default only h = 16 takes this path)
    before = ops.LAUNCHES
    got = ops.encoder_head(cost, inv, wc1, bc1, wd1, bd1)              # weights as kernel parameters: one launch per 16 channels
    assert ops.LAUNCHES - before == h // 16
    want = torch.cat([F.relu(F.conv2d(cost, wc1, bc1)), F.relu(F.conv2d(inv, wd1, bd1, padding=3))], dim=1)
    assert got.shape == want.shape and got.is_contiguous(memory_format=torch.channels_last)
    assert rel_max(got, want) < 1e-5
    assert torch.equal(ops.encoder_head(cost, inv, wc1, bc1, wd1, bd1), got)      # second call: the cached host tables
    wd1.mul_(2.0)                                                                  # in-place update: the tables are rebuilt
    want2 = torch.cat([F.relu(F.conv2d(cost, wc1, bc1)), F.relu(F.conv2d(inv, wd1, bd1, padding=3))], dim=1)
    assert rel_max(ops.encoder_head(cost, inv, wc1, bc1, wd1, bd1), want2) < 1e-5
    monkeypatch.setenv("EFFIMVS_EH_CONST", "0")                                    # the kernel that reads the weights from device memory
    before = ops.LAUNCHES
    dev_w = ops.encoder_head(cost, inv, wc1, bc1, wd1.clone(), bd1)
    assert ops.LAUNCHES - before == 1 and rel_max(dev_w, want2) < 1e-5


@pytest.mark.gpu
def test_update_block_dropin_golden(hp):
    """dropin.make_update_block_forward / make_upsample_depth called the way upstream's Effi_MVS_plus.forward calls
    BasicUpdateBlock.forward and upsample_depth (Effi_MVS_plus.py:552-564), against the upstream golden fixture"""
    import types
    from functools import partial
    from effimvs_b200 import dropin
    from test_net_host import load_update_block, _update_cost_fn
    g = golden("update_block", DEV)
    blk = load_update_block(g, DEV)
    blk.UpMask = True

    def disp_to_depth(disp, min_depth, max_depth):       # the signature dropin reads the range from
        raise AssertionError("the drop-in converts in-kernel")
    scale = partial(disp_to_depth, min_depth=g["dmin"], max_depth=g["dmax"])
    fwd = types.MethodType(dropin.make_update_block_forward(hp), blk)
    net_out, masks, invs = fwd(g["net0"], lambda depth, iter=0: _update_cost_fn(depth), g["inv0"], g["context"], seq_len=3,
                               scale_inv_depth=scale)
    assert rel_max(net_out, g["net"]) < 1e-4 and rel_max(masks[-1], g["mask"]) < 1e-4
    for i in range(3):
        assert float((invs[i] - g["inv{}".format(i + 1)]).abs().max()) < 1e-4
    up = dropin.make_upsample_depth(hp)(invs[-1], masks[-1], ratio=2)
    assert float((up - g["up"]).abs().max()) < 1e-4


@pytest.mark.gpu
@pytest.mark.parametrize("h,ctx,H,W", [(16, 4, 37, 53), (32, 8, 24, 70), (48, 12, 19, 25)])
def test_encoder_tail_vs_torch(h, ctx, H, W):
    """effimvs_encoder_tail_f32 against relu(convc(cat[m + b_d, context])) of upstream's ProjectionInput (models/update.py:93-95)"""
    import torch.nn.functional as F
    from effimvs_b200 import ops
    gen = torch.Generator(device=DEV).manual_seed(h)
    rnd = lambda *s: torch.randn(*s, device=DEV, generator=gen)      # noqa: E731
    cl = lambda t: t.contiguous(memory_format=torch.channels_last)   # noqa: E731
    B, hm = 2, h - ctx
    m, context, hprev = cl(rnd(B, hm, H, W)), cl(torch.relu(rnd(B, ctx, H, W))), cl(rnd(B, h, H, W))
    wc, bc, bd = rnd(h, h, 1, 1) * 0.3, rnd(h), rnd(hm)
    want = F.relu(F.conv2d(torch.cat([m + bd.reshape(1, -1, 1, 1), context], dim=1), wc, bc))
    ctx_term = F.conv2d(context, wc[:, hm:], bc + wc[:, :hm, 0, 0] @ bd)
    hx = cl(torch.cat([hprev, torch.zeros_like(hprev)], dim=1))
    ops.encoder_tail(m, wc[:, :hm].contiguous(), ctx_term, hx)
    assert torch.equal(hx[:, :h], hprev)
    assert rel_max(hx[:, h:], want) < 1e-5


# ---- size-independent properties at BASELINE's full stage sizes (no oracle needed at these sizes) -----------
@pytest.mark.gpu
@pytest.mark.parametrize("C,D,H,W,G", [(8, 8, 592, 800, 1), (16, 8, 296, 400, 1), (32, 48, 148, 200, 1), (8, 16, 592, 800, 8),
                                       (32, 8, 296, 400, 8), (16, 16, 592, 800, 4)])
def test_warp_corr_agg_properties_at_dtu_stage_sizes(hp, C, D, H, W, G):
    """DTU stage shapes: (a) channels-last (tiled TMA kernel) and planar (gather kernel) agree; (b) the similarity is
    linear in the reference features (exactly, for a power-of-two factor); (c) a source view with the reference camera
    samples pixel centres, so every plane holds mean_c(ref * src) whatever the hypothesis; (d) with equal features and
    weights the weighted aggregation of identical views is the single-view similarity."""
    from effimvs_b200 import synthetic
    feats, cams, hyp, wts = synthetic.microbench_inputs(C, D, H, W, views=5, seed=C + D, device=DEV)
    cl = [f.contiguous(memory_format=torch.channels_last) for f in feats]
    planar = hp.warp_corr_agg(feats, cams, hyp, wts, G)
    tiled = hp.warp_corr_agg(cl, cams, hyp, wts, G)
    assert rel_max(tiled, planar) < 1e-5                                                     # (a)
    doubled = hp.warp_corr_agg([cl[0] * 2.0] + cl[1:], cams, hyp, wts, G)
    assert torch.equal(doubled, tiled * 2.0)                                                 # (b)
    same_cam = cams[:, :1].repeat(1, 5, 1, 1, 1)
    for fs in (feats, cl):
        ident = hp.warp_corr_agg(fs, same_cam, hyp, None, G)                                 # (c)
        want = sum((fs[0] * fs[v]).reshape(1, G, C // G, H, W).mean(2) for v in range(1, 5)) / 4
        # upstream's coordinate chain ((x*d + t) / (z*d + t), normalise, un-normalise) lands within ~1e-4 px of the centre at
        # x ~ 800, i.e. a 1e-4 blend with the neighbouring pixel
        assert rel_max(ident, want.unsqueeze(2).expand(-1, -1, D, -1, -1)) < 1e-3
    rep = [cl[0]] + [cl[1]] * 4
    one = hp.warp_corr_agg(rep[:2], cams[:, :2], hyp, wts[:, :1], G)
    four = hp.warp_corr_agg(rep, cams[:, [0, 1, 1, 1, 1]], hyp, wts[:, :1].repeat(1, 4, 1, 1), G)
    w = wts[:, :1].unsqueeze(1)
    assert rel_max(four * (4 * w + 1e-6), one * (w + 1e-6) * 4) < 1e-5                        # (d)


@pytest.mark.gpu
def test_stage1_views_properties_at_dtu_size(hp):
    """stage-1 shape (C=32, D=48, 200x148): tiled and planar per-view similarities / entropies agree; the entropy of a
    view whose similarities do not depend on the plane is log(D) (reference camera as source)"""
    import math
    from effimvs_b200 import capi, ops, synthetic
    C, D, H, W = 32, 48, 148, 200
    feats, cams, hyp, _ = synthetic.microbench_inputs(C, D, H, W, views=5, seed=1, device=DEV)
    feats = [f * 0.3 for f in feats]
    cl = [f.contiguous(memory_format=torch.channels_last) for f in feats]
    planes = hyp[:, :, 0, 0].contiguous()
    proj = hp.relative_projection(cams)
    s_p, e_p = ops.warp_corr_views(feats[0], feats[1:], proj, planes, capi.HYP_PLANES, D)
    s_t, e_t = ops.warp_corr_views(cl[0], cl[1:], proj, planes, capi.HYP_PLANES, D)
    assert rel_max(s_t, s_p) < 1e-5 and float((e_t - e_p).abs().max()) < 1e-4
    proj_id = hp.relative_projection(cams[:, :1].repeat(1, 5, 1, 1, 1))
    _, e_id = ops.warp_corr_views(cl[0], cl[1:], proj_id, planes, capi.HYP_PLANES, D)
    assert float((e_id - math.log(D)).abs().max()) < 1e-3


@pytest.mark.gpu
def test_scene_runner_feature_cache_on_device(hp):
    """run_scene with the CUDA callables on a small 6-view scene: depth maps and fused point counts with the
    per-scene feature cache + block sharding, eager and as CUDA graphs, equal those of re-encoding every view
    (SURVEY section 8(f) row 1)"""
    from effimvs_b200 import scene, synthetic
    N, W, H = 6, 160, 128
    model = dtu_model(hp, DEV, ndepths="8,4,4")
    g = torch.Generator().manual_seed(0)
    imgs = torch.rand(N, 3, H, W, generator=g).to(DEV)
    E, K = synthetic.camera_arc(N, W, H)
    cams = {k: v[0].to(DEV) for k, v in synthetic.stage_cameras(E, K, 1).items()}
    dv = torch.linspace(1 / 935.0, 1 / 425.0, 384, device=DEV)
    pairs = [[(i + d) % N for d in (1, 2, N - 1, N - 2)] for i in range(N)]
    runs = {}
    for mode in ("plain", "cache", "graph"):
        infer, fuse = scene.cuda_scene_callables(model, imgs, cams, dv, 2.0, 6.0, 2, 0.3, feature_cache=mode != "plain",
                                                 graphed_src_views=4 if mode == "graph" else 0)
        runs[mode] = scene.run_scene(infer, fuse, N, pairs, 0, 1, DEV, sharding="round_robin" if mode == "plain" else "block")
    for i in range(N):
        for mode in ("cache", "graph"):
            d0, d1 = runs["plain"][i][1], runs[mode][i][1]
            assert frac_within(d1, d0, 1e-3 * DEPTH_RANGE) >= 0.999, mode
            n0, n1 = runs["plain"][i][0].shape[0], runs[mode][i][0].shape[0]
            assert abs(n0 - n1) <= 0.02 * H * W, mode


# ---- channels-last warp kernels (csrc/warp_tile.cu) against the oracle at the cascade's shapes ------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("C,D,H,W", [(8, 8, 592, 800), (16, 8, 296, 400), (8, 8, 97, 131), (16, 5, 64, 96), (32, 8, 40, 56), (8, 12, 50, 70)])
@pytest.mark.parametrize("depth_kind,ratio", [("smooth", 1), ("noise", 1), ("steps", 2), ("smooth", 12), ("near", 1)])
def test_local_volume_channels_last_vs_oracle(hp, ohp, C, D, H, W, depth_kind, ratio):
    """a5 on channels-last maps (the staged tile kernel) against the oracle on the device, with and without view weights.
    smooth / noise / steps: rendered surface, white-noise depth, depth discontinuities; ratio 12: planes several pixels
    apart; near: depths so close that most of the epipolar segments leave the source images (dead samples, clamped boxes,
    border cells)."""
    from effimvs_b200 import synthetic
    feats, cams, _, wts = synthetic.microbench_inputs(C, D, H, W, views=5, seed=C + D + H, device=DEV)
    gen = torch.Generator().manual_seed(H)
    if depth_kind == "smooth":
        E, K = synthetic.camera_ring(5, W, H)
        cur = synthetic.render_plane_scene(E[:1], K, W, H, noise=0.0)[0].reshape(1, 1, H, W).to(DEV)
    elif depth_kind == "noise":
        cur = (600 + 200 * torch.rand(1, 1, H, W, generator=gen)).to(DEV)
    elif depth_kind == "near":
        cur = (30 + 300 * torch.rand(1, 1, H, W, generator=gen)).to(DEV)
    else:
        cur = torch.full((1, 1, H, W), 500.0)
        cur[..., W // 3:] = 800.0
        cur[..., H // 2:, :] += 90.0
        cur = cur.to(DEV)
    iv = torch.full((1, 1, 1, 1), (1 / 425.0 - 1 / 935.0) / 384 * ratio, device=DEV)
    cl = [f.contiguous(memory_format=torch.channels_last) for f in feats]
    want, want_hyp = ohp.local_volume(cur, feats, cams, iv, wts, D, 1)
    got, hyp = hp.local_volume(cur, cl, cams, iv, wts, D, 1)
    assert torch.equal(hyp, want_hyp)
    assert rel_max(got, want) < 1e-4
    got_nw, _ = hp.local_volume(cur, cl, cams, iv, None, D, 1)
    want_nw, _ = ohp.local_volume(cur, feats, cams, iv, None, D, 1)
    assert rel_max(got_nw, want_nw) < 1e-4


@pytest.mark.gpu
@pytest.mark.parametrize("C,D,H,W,V", [(32, 48, 148, 200, 5), (32, 96, 132, 240, 7), (32, 48, 37, 53, 3), (16, 20, 64, 80, 5)])
def test_stage1_views_channels_last_vs_oracle(ohp, C, D, H, W, V):
    """a4 on channels-last maps (the staged per-view tile kernel) at the DTU and Tanks & Temples stage-1 shapes: per-view
    similarities and entropies against the oracle on the device."""
    from effimvs_b200 import capi, hotpath, ops, synthetic
    feats, cams, hyp, _ = synthetic.microbench_inputs(C, D, H, W, views=V, seed=D, device=DEV)
    feats = [f * 0.4 for f in feats]
    cl = [f.contiguous(memory_format=torch.channels_last) for f in feats]
    planes = hyp[:, :, 0, 0].contiguous()
    proj = hotpath.CudaHotPath().relative_projection(cams)
    sims, ent = ops.warp_corr_views(cl[0], cl[1:], proj, planes, capi.HYP_PLANES, D)
    for v in range(V - 1):
        want = ohp.view_similarity(feats[0], feats[v + 1], cams[:, 0], cams[:, v + 1], hyp, 1)
        assert rel_max(sims[:, v], want[:, 0]) < 1e-4
        assert float((ent[:, v:v + 1] - ohp.similarity_entropy(want)).abs().max()) < 1e-3


@pytest.mark.gpu
@pytest.mark.parametrize("C,D,H,W", [(8, 8, 296, 400), (16, 16, 148, 200), (32, 48, 74, 100)])
def test_plane_sweep_channels_last_vs_oracle(hp, ohp, C, D, H, W):
    """G = 1 plane sweeps over the whole depth range on channels-last maps (the staged tile kernel), with per-pixel
    hypotheses and with per-batch planes.  At 296 x 400 with 8 planes over the whole range nearly every block's footprint
    exceeds the staged box, so its samples take the global-gather path."""
    from effimvs_b200 import synthetic
    feats, cams, hyp, wts = synthetic.microbench_inputs(C, D, H, W, views=5, seed=C + D, device=DEV)
    cl = [f.contiguous(memory_format=torch.channels_last) for f in feats]
    sims = [ohp.view_similarity(feats[0], feats[v], cams[:, 0], cams[:, v], hyp, 1) for v in range(1, 5)]
    want = ohp.weighted_aggregate(sims, [wts[:, i:i + 1] for i in range(4)])
    got = hp.warp_corr_agg(cl, cams, hyp, wts, 1)
    got_planes = hp.warp_corr_agg(cl, cams, hyp[:, :, :1, :1].contiguous(), wts, 1)
    assert rel_max(got, want) < 1e-4 and rel_max(got_planes, want) < 1e-4


@pytest.mark.gpu
@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two CUDA devices")
def test_ops_run_on_the_tensors_device_not_the_current_one(ohp):
    """every effimvs:: op launches on the device (and that device's current stream) of its tensor arguments whatever torch's
    current device is, and rejects tensors spread over two devices"""
    from effimvs_b200 import hotpath, synthetic
    feats, cams, hyp, wts = synthetic.microbench_inputs(8, 4, 40, 56, views=3, seed=9, device="cuda:1")
    assert torch.cuda.current_device() == 0
    hp1 = hotpath.CudaHotPath("f32", native_projection=True)
    got = hp1.warp_corr_agg(feats, cams, hyp, wts, 1)
    assert got.device == torch.device("cuda:1") and torch.cuda.current_device() == 0
    sims = [ohp.view_similarity(feats[0], feats[v], cams[:, 0], cams[:, v], hyp, 1) for v in range(1, 3)]
    want = ohp.weighted_aggregate(sims, [wts[:, i:i + 1] for i in range(2)])
    assert rel_max(got, want) < 1e-4
    with pytest.raises(RuntimeError, match="several devices"):
        hp1.warp_corr_agg([feats[0].to("cuda:0")] + feats[1:], cams, hyp, wts, 1)
