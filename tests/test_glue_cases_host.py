"""CPU checks of tests/test_gpu_glue_fp64.py: its case matrix reaches every launch branch of the host code, and its bars are
tight enough to reject small corruptions.

The launch rules are restated here from the host functions of csrc/update_glue.cu, csrc/lookup.cu and csrc/warp_tile.cu
(grid_for, the encoder_tail(_ctx) grid, the encoder_head instantiation, delta_head's <J>, the entropy kernel chosen by D,
volume_lookup's gridDim.y); the case lists are imported from the GPU module, so the two cannot drift apart.
"""
import math

import pytest
import torch

import test_gpu_glue_fp64 as G

NUM_SMS = 148


# ---- launch rules --------------------------------------------------------------------------------------------------
def grid_for_passes(work, block=256):
    """grid_for: ceil(work / block) blocks capped at 148 * 16; the kernels stride over the rest.  -> grid-stride passes"""
    grid = min(max(-(-work // block), 1), NUM_SMS * 16)
    return -(-work // (grid * block))


def tail_ctx_launch(n_pix, h):
    """effimvs_encoder_tail_ctx_f32: (grid-stride passes, output-channel slices over gridDim.y)"""
    blocks = -(-n_pix // 256)
    h4 = h // 4
    slices = 1 if blocks >= NUM_SMS * 2 else (3 if h4 % 3 == 0 else (2 if h4 % 2 == 0 else 1))
    grid = min(blocks, NUM_SMS * 8)
    return -(-n_pix // (grid * 256)), slices


def encoder_head_kernel(h, const, ty="4", zchunks="1"):
    """ops.encoder_head (EFFIMVS_EH_CONST) and effimvs_encoder_head_f32 (EFFIMVS_EH_TY, EFFIMVS_EH_ZCHUNKS)"""
    if const:
        return "const"
    if ty == "8":
        return "<8,0>"
    if h == 16:
        return "<4,16>"
    if h == 48 and zchunks != "0":
        return "<4,48,zc>"
    if h == 32:
        return "<4,32>"
    return "<4,0>"


def entropy_kernel(D):
    return "reg48" if D <= 48 else ("reg96" if D <= 96 else "generic")


def reached():
    """every launch branch the GPU module's cases take"""
    got = set()
    for (H, W, h, cx, B) in G.STAGE_CASES + G.EDGE_CASES:
        n = B * H * W
        got.add(("gru_reset", grid_for_passes(n * (2 * h) // 4) > 1))
        got.add(("gru_update", grid_for_passes(n * h // 4) > 1))
        got.add(("delta_head", h // 16))
        got.add(("encoder_head", encoder_head_kernel(h, h == 16)))      # EFFIMVS_EH_CONST unset: constant bank for h = 16
    for (H, W, h, cx, B) in G.TAIL_CASES:
        n = B * H * W
        passes, slices = tail_ctx_launch(n, h)
        got.add(("encoder_tail_ctx.passes", passes > 1))
        got.add(("encoder_tail_ctx.slices", slices))
        got.add(("encoder_tail.passes", -(-n // (min(-(-n // 256), NUM_SMS * 8) * 256)) > 1))
        got.add(("gru_init_ctx", grid_for_passes(n * h // 4) > 1))
    for (H, W, B) in G.DELTA_CASES:
        got.add(("inv_init / gru_delta", grid_for_passes(H * W) > 1))
    for (CD, h, const, H, W, B) in G.EH_CASES:
        got.add(("encoder_head", encoder_head_kernel(h, const)))
        got.add(("encoder_head.cd", CD))
    for env, hs in G.EH_ENV_CASES:
        for h in hs:
            got.add(("encoder_head", encoder_head_kernel(h, False, env.get("EFFIMVS_EH_TY", "4"), env.get("EFFIMVS_EH_ZCHUNKS", "1"))))
    for K in G.UPSAMPLE_K:
        got.add(("convex_upsample_conv.K", K))
    for (D, *_rest) in G.ENTROPY_CASES:
        got.add(("softmax_entropy", entropy_kernel(D)))
    for (B, D, d, H, W, per_pixel, stride) in G.LOOKUP_CASES:
        gy = min(d, 8)
        got.add(("volume_lookup.gridDim.y", gy))
        got.add(("volume_lookup.sample passes > 1", -(-d // gy) > 1))
        got.add(("volume_lookup.range", per_pixel))
        got.add(("volume_lookup.stride", stride))
        got.add(("volume_lookup.batch > 1", B > 1))
    for (B, D, nd, H, W, per_pixel) in G.DYNCOST_CASES:
        got.add(("dynamic_cost.range", per_pixel))
        got.add(("dynamic_cost.ndepth", nd))
    return got


EXPECTED = (
    [("gru_reset", True), ("gru_reset", False), ("gru_update", True), ("gru_update", False),
     ("inv_init / gru_delta", True), ("inv_init / gru_delta", False), ("gru_init_ctx", True), ("gru_init_ctx", False)]
    + [("delta_head", J) for J in (1, 2, 3, 4, 6, 8)]
    + [("encoder_head", k) for k in ("const", "<4,16>", "<4,32>", "<4,48,zc>", "<4,0>", "<8,0>")]
    + [("encoder_head.cd", c) for c in (1, 6, 8)]
    + [("encoder_tail_ctx.passes", True), ("encoder_tail_ctx.passes", False), ("encoder_tail.passes", True),
       ("encoder_tail.passes", False)]
    + [("encoder_tail_ctx.slices", s) for s in (1, 2, 3)]
    + [("convex_upsample_conv.K", K) for K in (4, 32, 96, 256)]
    + [("softmax_entropy", k) for k in ("reg48", "reg96", "generic")]
    + [("volume_lookup.gridDim.y", 3), ("volume_lookup.gridDim.y", 8), ("volume_lookup.sample passes > 1", True),
       ("volume_lookup.range", True), ("volume_lookup.range", False), ("volume_lookup.stride", 1), ("volume_lookup.stride", 2),
       ("volume_lookup.batch > 1", True)]
    + [("dynamic_cost.range", True), ("dynamic_cost.range", False)] + [("dynamic_cost.ndepth", n) for n in (3, 8, 16)]
)


@pytest.mark.parametrize("branch", EXPECTED, ids=[" ".join(map(str, b)) for b in EXPECTED])
def test_case_matrix_reaches_every_launch_branch(branch):
    assert branch in reached()


def test_case_matrix_covers_the_stage_shapes_and_view_batches():
    stages = {(H, W, h, cx) for (H, W, h, cx, B) in G.STAGE_CASES}
    assert stages == {(H, W, G.HIDDEN[s], G.CONTEXT[s]) for hw in G.STAGE_HW.values() for s, (H, W) in enumerate(hw)}
    assert {B for (*_, B) in G.STAGE_CASES} == {1, 2, 4, 8}
    assert set(G.SOFTMAX_D) == {8, 48, 49, 96, 97, 192}
    assert {D for (D, *_r) in G.SOFTMAX_CASES} == set(G.SOFTMAX_D) == {D for (D, *_r) in G.ENTROPY_CASES}
    assert any(H == 1 for (H, W) in G.EDGE_HW) and any(W == 1 for (H, W) in G.EDGE_HW)
    assert any(W % 64 and H % 4 for (H, W) in G.EDGE_HW)                # a partial delta_head / encoder_head tile in both directions


def test_launch_rule_restatement_matches_the_documented_examples():
    """the numbers the sources and the issue of this test state: stage-3 GRU gates take several passes, gru_delta reaches a
    second pass only above 606,208 pixels, encoder_tail_ctx at stage 1 with h = 48 has 3 slices for K <= 2 and 1 for K >= 3"""
    assert grid_for_passes(592 * 800 * 32 // 4) == 7
    assert grid_for_passes(606208) == 1 and grid_for_passes(606209) == 2
    assert [tail_ctx_launch(k * 148 * 200, 48)[1] for k in (1, 2, 3, 8)] == [3, 3, 1, 1]
    assert tail_ctx_launch(592 * 800, 16)[0] == 2


# ---- sensitivity of the bars ----------------------------------------------------------------------------------------
def _gen(seed):
    return torch.Generator().manual_seed(seed)


def _scenario_dot():
    """a 1x1 convolution of 6 channels plus bias (convc1 with the cascade's cost channels): n = 6 roundings"""
    g = _gen(1)
    x, w, b = torch.randn(2, 6, 16, 24, generator=g), torch.randn(8, 6, 1, 1, generator=g), torch.randn(8, generator=g)
    c, ca = G._conv_abs(x, w, b)
    return c, G.dot_bar(ca, 6)


def _scenario_conv7():
    """convd1: a 7x7 convolution, 49 roundings"""
    g = _gen(2)
    x, w, b = torch.rand(2, 1, 16, 24, generator=g), torch.randn(4, 1, 7, 7, generator=g) * 0.2, torch.randn(4, generator=g)
    c, ca = G._conv_abs(x, w, b, padding=3)
    return torch.relu(c), G.dot_bar(ca, 49)


def _scenario_tanh():
    g = _gen(3)
    x = (2 * torch.randn(2, 4, 16, 24, generator=g)).double()
    return torch.tanh(x), G.tanh_bar(x, G.U * x.abs())


def _scenario_sigmoid():
    g = _gen(4)
    x = (2 * torch.randn(2, 4, 16, 24, generator=g)).double()
    s, ds = G.sigmoid_bar(x, G.U * x.abs())
    return s, ds


def _scenario_depth():
    g = _gen(5)
    inv = torch.rand(2, 1, 16, 24, generator=g).double()
    lo = torch.tensor([1 / 935.0, 1 / 1000.0], dtype=torch.float64).reshape(2, 1, 1, 1)
    hi = torch.tensor([1 / 425.0, 1 / 400.0], dtype=torch.float64).reshape(2, 1, 1, 1)
    return G.to_depth_bar(inv, G.U * inv.abs(), lo, hi)


def _scenario_regression():
    g = _gen(6)
    x = (3 * torch.randn(2, 48, 16, 24, generator=g)).double()
    hyp = (425 + 510 * torch.rand(2, 48, 16, 24, generator=g)).double()
    p, dp = G.softmax_bar(x, torch.zeros_like(x), 1)
    return (p * hyp).sum(1, keepdim=True), G.weighted_sum_bar(p, dp, hyp, 1).unsqueeze(1)


def _scenario_entropy():
    g = _gen(7)
    x = (3 * torch.randn(2, 48, 16, 24, generator=g)).double()
    p, dp = G.softmax_bar(x, torch.zeros_like(x), 1)
    return -(p * torch.log(p + 1e-7)).sum(1, keepdim=True), G.entropy_bar(p, dp, 1).unsqueeze(1)


def _scenario_lookup():
    g = _gen(8)
    vol = torch.randn(2, 8, 16, 24, generator=g).double()
    depth = (450 + 450 * torch.rand(2, 1, 16, 24, generator=g)).double()
    ix, e_ix = G.lookup_ix_bar(depth, 0.0, torch.tensor(425.0, dtype=torch.float64), torch.tensor(935.0, dtype=torch.float64), 8)
    return G.lookup_bar(vol, ix, e_ix, 1)


SCENARIOS = {"dot_bar": _scenario_dot, "dot_bar(49)": _scenario_conv7, "tanh_bar": _scenario_tanh, "sigmoid_bar": _scenario_sigmoid,
             "to_depth_bar": _scenario_depth, "weighted_sum_bar": _scenario_regression, "entropy_bar": _scenario_entropy,
             "lookup_bar": _scenario_lookup}
# an 8-ulp move of one element is rejected where the bound is narrower than 8 ulps: the elementwise bars and a short dot product.
# A sound bound of a long reduction (a 49-term convolution, a softmax over 48 planes, the entropy) or of an interpolation at a
# coordinate with rounding error (the lookup) is wider than that; those scenarios are held to the other three corruptions.
EIGHT_ULPS = ["dot_bar", "tanh_bar", "sigmoid_bar", "to_depth_bar"]


def _ulps(x32, k):
    """x32 moved by k ulps away from zero"""
    bits = x32.view(torch.int32)
    return (bits + k).view(torch.float32)


@pytest.mark.parametrize("name", list(SCENARIOS))
def test_bar_accepts_the_fp32_rounding_and_rejects_corruptions(name):
    ref, bar = SCENARIOS[name]()
    bar = bar.expand_as(ref)
    got = ref.float()
    assert G.within(got, ref, bar), "the fp32 rounding of the reference must pass"
    row = got.clone()
    row[..., -1, :] = row[..., -2, :]                   # one border row replaced by its neighbour
    assert not G.within(row, ref, bar)
    swap = got.clone()
    swap[0], swap[1] = got[1], got[0]                  # batch entries 0 and 1 swapped
    assert not G.within(swap, ref, bar)
    assert not G.within(got.bfloat16().float(), ref, bar)     # the result rounded through bf16
    if name in EIGHT_ULPS:
        ratio_ulp = bar / (got.double().abs() * G.ULP).clamp(min=1e-300)
        where = tuple(torch.nonzero(ratio_ulp == ratio_ulp.min())[0].tolist())
        moved = got.clone()
        moved[where] = _ulps(got[where].reshape(1), 8)[0]
        assert not G.within(moved, ref, bar), "one element moved by 8 ulps"
