"""CPU checks of tests/test_gpu_warp_fp64.py: its case matrix reaches every launch branch of the warp kernels and every kind of
round of the tile kernel's staging, its exact-FMA helper rounds as an FMA does, and its bars reject small corruptions.

The launch rules are restated from the host code of csrc/warp_corr.cu and csrc/warp_tile.cu (and ops._features); the staging
decisions from run_round() in csrc/warp_tile.cu.  The case lists and input generators are imported from the GPU module, so the
two cannot drift apart.
"""
import math
import random
from fractions import Fraction

import numpy as np
import pytest
import torch

import test_gpu_warp_fp64 as T

TW, TH = 32, 4                                        # reference tile of a tile-kernel block
BOX = {8: (64, 12), 16: (64, 12), 32: (64, 8)}        # Box<C>: staged source box in pixels


# ---- launch rules --------------------------------------------------------------------------------------------------
def agg_path(c):
    """effimvs_warp_corr_agg_f32 / effimvs_warp_corr_views_f32: channels-last maps with C in {8, 16, 32} whose pointers are all
    32-byte aligned take the tile kernels, other channels-last maps the generic kernel's NHWC form, NCHW maps the planar form.
    The GPU module's "nhwc" layout offsets source 0 by 16 bytes."""
    if c.layout == "planar":
        return "planar"
    return "tile" if c.C in (8, 16, 32) and c.layout == "tile" else "nhwc"


def planes_per_thread(G):
    """TilePlanes<G> (tile kernel) and PlanesPerThread<G> (generic kernel): 4 planes for G >= 4, else 8"""
    return 4 if G >= 4 else 8


def entropy_kernel(c):
    """tile path: launch_views picks the entropy kernel by D; the generic kernel reduces the entropy in itself"""
    if agg_path(c) != "tile":
        return "in-kernel"
    return "reg48" if c.D <= 48 else ("reg96" if c.D <= 96 else "generic")


def views_smem_attribute(c):
    """the generic views kernel asks for more than the default 48 KB of dynamic shared memory (D x 32 floats) above D = 384"""
    return agg_path(c) != "tile" and c.D * 32 * 4 > 48 * 1024


def reached():
    got = set()
    for c in T.AGG_CASES:
        p = agg_path(c)
        got.add(("agg", p, c.C, c.G))
        got.add(("agg.mode", p, c.mode))
        got.add(("agg.weighted", p, c.weighted))
        if c.D == 1:
            got.add(("agg.D = 1", p))
        dpt = planes_per_thread(c.G)
        if c.D % dpt:
            got.add(("agg.partial plane group", p, dpt))
        if p == "tile" and c.W % TW and c.H % TH:
            got.add(("agg.partial tile in both directions", p))
        if p != "tile" and (c.H * c.W) % 128:
            got.add(("agg.partial block", p))
        got.add(("agg.ray unfused", p, T.ray_unfused_for(c.H, c.W)))
        got.add(("agg.n_src", c.n))
        got.add(("agg.B", c.B))
        got.add(("agg.geom", c.geom))
        if min(c.H, c.W) == 2:
            got.add(("agg.2-pixel side", p, (c.H, c.W)))
    for c in T.ALL_VIEWS_CASES:
        p = agg_path(c)
        got.add(("views", p, c.C))
        got.add(("views.entropy", entropy_kernel(c)))
        got.add(("views.smem > 48 KB", views_smem_attribute(c)))
        got.add(("views.ray unfused", T.ray_unfused_for(c.H, c.W)))
        if c.D % 8:
            got.add(("views.partial plane group", p))
    for (C, mode, H, W, D) in T.HOMO_CASES:
        got.add(("homo_warp.C", C))
        got.add(("homo_warp.mode", mode))
        got.add(("homo_warp.ray unfused", T.ray_unfused_for(H, W)))
    for (n, D) in T.WAGG_CASES:
        got.add(("weighted_agg.n_src", n))
        got.add(("weighted_agg.plane passes > 1", -(-D // min(D, 8)) > 1))
    return got


PATHS = ("tile", "nhwc", "planar")
EXPECTED = (
    [("agg", p, C, G) for p in PATHS for C in (8, 16, 32) for G in (1, 2, 4, 8)]
    + [("agg.mode", p, m) for p in PATHS for m in (T.HYP_TENSOR, T.HYP_PLANES, T.HYP_LOCAL)]
    + [("agg.weighted", p, w) for p in PATHS for w in (True, False)]
    + [("agg.D = 1", p) for p in PATHS]
    + [("agg.partial plane group", p, dpt) for p in PATHS for dpt in (4, 8)]
    + [("agg.partial tile in both directions", "tile")] + [("agg.partial block", p) for p in ("nhwc", "planar")]
    + [("agg.ray unfused", p, u) for p in ("tile", "planar") for u in (True, False)]
    + [("agg.2-pixel side", p, hw) for p in PATHS for hw in ((2, 131), (131, 2), (2, 2))]
    + [("agg.n_src", n) for n in (1, 4, 6, 16)] + [("agg.B", B) for B in (1, 2, 8)]
    + [("agg.geom", gm) for gm in ("normal", "wide", "identity", "both_sides", "z0", "offimage", "special", "unordered")]
    + [("views", p, C) for p in PATHS for C in (8, 16, 32)]
    + [("views.entropy", k) for k in ("reg48", "reg96", "generic", "in-kernel")]
    + [("views.smem > 48 KB", True), ("views.smem > 48 KB", False), ("views.ray unfused", True)]
    + [("views.partial plane group", p) for p in PATHS]
    + [("homo_warp.C", C) for C in (1, 3, 8, 64)] + [("homo_warp.mode", m) for m in (T.HYP_TENSOR, T.HYP_PLANES)]
    + [("homo_warp.ray unfused", u) for u in (True, False)]
    + [("weighted_agg.n_src", n) for n in (1, 4, 6, 16)] + [("weighted_agg.plane passes > 1", v) for v in (True, False)]
)


@pytest.mark.parametrize("branch", EXPECTED, ids=[" ".join(map(str, b)) for b in EXPECTED])
def test_case_matrix_reaches_every_launch_branch(branch):
    assert branch in reached()


def test_case_matrix_covers_the_cascade_calls():
    """every stage call of both datasets at B = 1, 2 and 8 in both layouts; the stage shapes cover both ray orders, and the
    instantiation cases use D values that leave a partial plane group for both planes-per-thread counts"""
    stage = {(c.kind, c.H, c.W, c.n, c.C, c.D, c.mode) for c in T.STAGE_CASES}
    assert stage == {s for ds in T.STAGES.values() for s in ds}
    assert {(c.B, c.layout) for c in T.STAGE_CASES} == {(B, L) for B in (1, 2, 8) for L in ("tile", "planar")}
    assert {T.ray_unfused_for(c.H, c.W) for c in T.STAGE_CASES} == {True, False}
    assert all(c.D == 1 or (c.D % 8 and c.D % 4) for c in T.INSTANCE_CASES)
    assert not any(c.mode == T.HYP_LOCAL and c.D == 1 for c in T.AGG_CASES)
    assert set(T.VIEWS_D) == {1, 7, 48, 49, 96, 97, 385, 1024}


def test_ray_order_rule_matches_the_probed_sizes():
    """warp_coords.cuh: 400 x 512 (204,800 pixels) was probed unfused, 400 x 600 (240,000) fused"""
    assert T.ray_unfused_for(400, 512) and not T.ray_unfused_for(400, 600)
    assert T.ray_unfused_for(1, 220000) and not T.ray_unfused_for(1, 220001)


# ---- the tile kernel's staging decisions -----------------------------------------------------------------------------
def tile_rounds(c):
    """run_round() of every block and round of a tile-kernel case, restated: step 1 (the box of the end planes' cells, clamped
    to [-1, W-1] x [-1, H-1], over the block's 32 x 4 pixels) and step 4 (a live sample is staged when its cell lies in the
    BW x BH box anchored at the box's top-left corner).  Returns per (block, round) [any, live, staged] and the count of live,
    gathered samples on border cells (x0 or y0 at -1 or at the last column / row) and on the last row."""
    ref, srcs, proj, hyp, interval, _ = T.make_inputs(c)
    B, D, H, W = c.B, c.D, c.H, c.W
    BW, BH = BOX[c.C]
    dpt = planes_per_thread(c.G) if c.kind == "agg" else 8
    nG, tY, tX = -(-D // dpt), -(-H // TH), -(-W // TW)
    depth = T.restate_depth(c, hyp, interval)
    rays = T.restate_rays(proj, H, W)
    kl = torch.tensor([min(dpt, D - g * dpt) - 1 for g in range(nG)])
    rounds, border, bottom = [], 0, 0
    for v in range(c.n):
        ix, iy = T.restate_coords(rays[:, v], proj[:, v, 9:], depth, H, W)

        def blocks(t):
            p = torch.full((B, nG * dpt, tY * TH, tX * TW), math.nan)
            p[:, :D, :H, :W] = t.reshape(B, D, H, W)
            return p.reshape(B, nG, dpt, tY, TH, tX, TW).permute(0, 1, 3, 5, 2, 4, 6).reshape(B, nG, tY, tX, dpt, TH * TW)

        bx_, by_ = blocks(ix), blocks(iy)
        inimg = torch.zeros(tY * TH, tX * TW, dtype=torch.bool)
        inimg[:H, :W] = True
        inimg = inimg.reshape(tY, TH, tX, TW).permute(0, 2, 1, 3).reshape(1, 1, tY, tX, TH * TW)
        sel = kl.reshape(1, nG, 1, 1, 1, 1).expand(B, nG, tY, tX, 1, TH * TW)
        x0, y0 = bx_[..., 0, :], by_[..., 0, :]
        jx, jy = bx_.gather(4, sel)[..., 0, :], by_.gather(4, sel)[..., 0, :]
        lx, hx = torch.floor(torch.fmin(x0, jx)), torch.floor(torch.fmax(x0, jx))
        ly, hy = torch.floor(torch.fmin(y0, jy)), torch.floor(torch.fmax(y0, jy))
        on = inimg & (lx <= W - 1) & (hx >= -1) & (ly <= H - 1) & (hy >= -1) & \
            (lx.abs() < 1e9) & (hx.abs() < 1e9) & (ly.abs() < 1e9) & (hy.abs() < 1e9)
        big = 1e30
        mnx = torch.where(on, lx.clamp(min=-1), torch.full_like(lx, big)).amin(-1)
        mxx = torch.where(on, hx.clamp(max=W - 1), torch.full_like(hx, -big)).amax(-1)
        mny = torch.where(on, ly.clamp(min=-1), torch.full_like(ly, big)).amin(-1)
        anyr = mnx <= mxx
        fx, fy = torch.floor(bx_), torch.floor(by_)
        live = (fx >= -1) & (fx <= W - 1) & (fy >= -1) & (fy <= H - 1)
        ox, oy = fx - mnx[..., None, None], fy - mny[..., None, None]
        staged = live & anyr[..., None, None] & (ox >= 0) & (ox <= BW - 2) & (oy >= 0) & (oy <= BH - 2)
        gathered = live & ~staged
        border += int((gathered & ((fx == -1) | (fx == W - 1) | (fy == -1) | (fy == H - 1))).sum())
        bottom += int((gathered & (fy == H - 1)).sum())
        rounds.append(torch.stack([anyr.long(), live.sum((-1, -2)), staged.sum((-1, -2))], -1))
    return torch.stack(rounds, -2), border, bottom       # (B, nG, tY, tX, rounds, 3)


GEOMETRIC_CASES = [c for c in T.EDGE_CASES + T.VIEWS_CASES if c.layout == "tile" and c.geom != "normal"] + \
    [c for c in T.EDGE_CASES if c.layout == "tile" and min(c.H, c.W) == 2]


def staging_kinds():
    kinds = {}
    for c in GEOMETRIC_CASES:
        r, border, bottom = tile_rounds(c)
        anyr, live, staged = r[..., 0].bool(), r[..., 1], r[..., 2]
        found = set()
        if ((live > 0) & (staged == live)).any():
            found.add("every sample staged")
        if ((staged > 0) & (staged < live)).any():
            found.add("staged and gathered samples mixed")
        if (anyr & (staged == 0) & (live > 0)).any() or (~anyr & (live > 0)).any():
            found.add("a round that gathers every live sample")
        before = torch.cummax(anyr.long(), -1).values.roll(1, -1)
        before[..., 0] = 0
        after = torch.cummax(anyr.long().flip(-1), -1).values.flip(-1).roll(-1, -1)
        after[..., -1] = 0
        if (~anyr & before.bool() & after.bool()).any():
            found.add("a round that stages nothing between rounds that stage")
        if border:
            found.add("gathered samples on border cells")
        if bottom:
            found.add("gathered samples on last-row cells")
        kinds[T.case_id(c)] = found
    return kinds


STAGING_KINDS = ("every sample staged", "staged and gathered samples mixed", "a round that gathers every live sample",
                 "a round that stages nothing between rounds that stage", "gathered samples on border cells",
                 "gathered samples on last-row cells")


def test_tile_cases_reach_every_kind_of_round():
    """the geometric cases make the tile kernel stage whole rounds, mix staged and gathered samples, gather samples on the
    border cells that gather_cell() clamps, and leave a round without a box between rounds with one (the mbarrier phase and
    the double-buffered box reset)"""
    kinds = staging_kinds()
    union = set().union(*kinds.values())
    assert union >= set(STAGING_KINDS), sorted(set(STAGING_KINDS) - union)
    assert "a round that stages nothing between rounds that stage" in kinds[T.case_id(
        T.Case("agg", 37, 53, 2, 3, 8, 1, 8, T.HYP_TENSOR, True, "tile", "offimage"))]


def test_z0_case_hits_a_zero_depth_exactly():
    """the hand-built projection makes z exactly 0 on the 650 plane, so the 1e-8 nudge decides those samples"""
    c = [c for c in T.EDGE_CASES if c.geom == "z0"][0]
    _, _, proj, hyp, interval, _ = T.make_inputs(c)
    depth = T.restate_depth(c, hyp, interval)
    rays = T.restate_rays(proj, c.H, c.W)
    pz = (rays[:, 0, 2].unsqueeze(1) * depth) + proj[:, 0, 11].reshape(-1, 1, 1)
    assert bool((pz[:, c.D // 2] == 0).all())
    ix, _ = T.restate_coords(rays[:, 0], proj[:, 0, 9:], depth, c.H, c.W)
    assert bool(torch.isfinite(ix[:, c.D // 2]).all()) and float(ix[:, c.D // 2].amax()) > 10


def test_both_sides_case_puts_planes_on_both_sides_of_the_source_camera():
    c = [c for c in T.EDGE_CASES if c.geom == "both_sides"][0]
    _, _, proj, hyp, interval, _ = T.make_inputs(c)
    depth = T.restate_depth(c, hyp, interval)
    rays = T.restate_rays(proj, c.H, c.W)
    pz = (rays[:, :, 2].unsqueeze(2) * depth.unsqueeze(1)) + proj[:, :, 11].reshape(c.B, c.n, 1, 1)
    assert bool((pz < 0).any()) and bool((pz > 0).any())


# ---- the exact FMA helper ------------------------------------------------------------------------------------------
def round_f32(x):
    """a Fraction rounded to the nearest fp32 value, ties to even"""
    f = np.float32(float(x))
    cands = [f, np.nextafter(f, np.float32(-np.inf)), np.nextafter(f, np.float32(np.inf))]
    return min(cands, key=lambda v: (abs(Fraction(float(v)) - x), int(np.array(v).view(np.int32)) & 1))


def _midpoint_cases():
    """a b + c a hair off an fp32 midpoint, so that fp64 rounds it onto the midpoint: (1 + 2^-11)(1 - 2^-11 + 2^-22) = 1 + 2^-33
    and (1 - 2^-11)(1 + 2^-11 + 2^-22) = 1 - 2^-33 (exact fp32 factors), scaled by 2^-24 onto 1 and 1 + 2^-23"""
    p, q = 2.0 ** -11, 2.0 ** -22
    base = [((1 + p) * 2.0 ** -24, 1 - p + q, 1.0), ((1 - p) * 2.0 ** -24, 1 + p + q, 1.0 + 2.0 ** -23),
            ((1 + p) * 2.0 ** -24, 1 - p + q, 1.0 + 2.0 ** -23), ((1 - p) * 2.0 ** -24, 1 + p + q, 1.0)]
    out = []
    for (a, b, c) in base:
        for e in (-30, -3, 0, 7, 40):
            for s in (1.0, -1.0):
                out.append((s * a * 2.0 ** e, b, s * c * 2.0 ** e))
    return out


def test_fma32_rounds_as_one_fma():
    rng = random.Random(5)
    trip = [tuple(float(np.float32(rng.gauss(0, 1) * 2.0 ** rng.randint(-30, 30))) for _ in range(3)) for _ in range(3000)]
    trip += [(float(np.float32(rng.uniform(-2, 2))), float(rng.randint(0, 2000)), float(np.float32(rng.uniform(-1e3, 1e3))))
             for _ in range(2000)]                                  # the ray's operands: fma(r1, y, r0 * x)
    mids = _midpoint_cases()
    trip += mids
    a, b, c = (torch.tensor([t[i] for t in trip], dtype=torch.float32) for i in range(3))
    assert all(float(np.float32(v)) == v for t in trip for v in t)
    got = T.fma32(a, b, c)
    want = torch.tensor([float(round_f32(Fraction(x) * Fraction(y) + Fraction(z))) for (x, y, z) in trip], dtype=torch.float32)
    assert torch.equal(got.view(torch.int32), want.view(torch.int32))
    # the constructed cases are real double-rounding traps: fp64 then fp32 gets half of them wrong
    m = len(mids)
    naive = (a[-m:].double() * b[-m:].double() + c[-m:].double()).float()
    assert int((naive != want[-m:]).sum()) == m // 2


# ---- sensitivity of the bars -------------------------------------------------------------------------------------------
SMALL = T.Case("agg", 13, 21, 2, 3, 16, 2, 6, T.HYP_TENSOR, True, "planar", "normal")


def fp32_agg(c, ref, srcs, proj, depth, weights, shift_ix=False, src_map=None, drop_view=None, plane_from=None,
             last_row_dy=False, batch0=False):
    """the aggregation evaluated in fp32 without FMAs (mul then add: at most one more rounding per step than the planar
    kernel, inside the bar's path length), with corruptions: ix one ulp up, a channel permutation of the source maps, one
    view's term dropped from the numerator, plane 0 read at plane 1's depth, the weight of a cell on the last row taken
    from the wrong axis weight (dy for ey), batch entry 1 reading batch entry 0's source maps"""
    B, C, H, W, G = c.B, c.C, c.H, c.W, c.G
    HW, CG = H * W, C // G
    rays = T.restate_rays(proj, H, W)
    if plane_from is not None:
        depth = depth.clone()
        depth[:, 0] = depth[:, plane_from]
    refl = ref.permute(0, 2, 3, 1).reshape(B, 1, HW, C)
    num = torch.zeros(B, c.D, HW, G)
    den = torch.zeros(B, 1, HW)
    for v in range(c.n):
        src = srcs[v] if src_map is None else srcs[v][:, src_map]
        if batch0:
            src = src[[0] * B]
        flat = src.permute(0, 2, 3, 1).reshape(B * HW, C)
        ix, iy = T.restate_coords(rays[:, v], proj[:, v, 9:], depth, H, W)
        if shift_ix:
            ix = torch.nextafter(ix, torch.full_like(ix, math.inf))
        fx, fy = torch.floor(ix), torch.floor(iy)
        ex, dx, ey, dy = (fx + 1) - ix, ix - fx, (fy + 1) - iy, iy - fy
        wt = torch.where(fy == H - 1, dy, ey) if last_row_dy else ey
        taps = ((0, 0, ex * wt), (1, 0, dx * wt), (0, 1, ex * dy), (1, 1, dx * dy))
        val = None
        for (ox, oy, w) in taps:
            xx, yy = fx + ox, fy + oy
            ok = (xx >= 0) & (xx <= W - 1) & (yy >= 0) & (yy <= H - 1)
            b_off = (torch.arange(B) * HW).reshape(B, 1, 1)
            idx = torch.where(ok, b_off + yy * W + xx, torch.zeros_like(xx)).long()
            t = flat[idx] * torch.where(ok, w, torch.zeros_like(w)).unsqueeze(-1)
            val = t if val is None else val + t
        prod = val * refl
        acc = prod.reshape(B, c.D, HW, G, CG)[..., 0]
        for k in range(1, CG):
            acc = acc + prod.reshape(B, c.D, HW, G, CG)[..., k]
        sim = acc * (1.0 / CG)
        w = weights[:, v].reshape(B, 1, HW)
        if v != drop_view:
            num = num + sim * w.unsqueeze(-1)
        den = den + w
    out = num / (den + 1e-6).unsqueeze(-1)
    return out.permute(0, 3, 1, 2)


CORRUPTIONS = {
    "ix one ulp up": dict(shift_ix=True),
    "channels swapped across a group boundary": dict(src_map=[*range(7), 8, 7, *range(9, 16)]),
    "16-byte halves of a pixel swapped": dict(src_map=[4, 5, 6, 7, 0, 1, 2, 3, *range(8, 16)]),
    "one view's weight dropped": dict(drop_view=1),
    "plane 0 read as plane 1": dict(plane_from=1),
    "last-row cell weighted with dy": dict(last_row_dy=True),
    "batch entry 1 read as entry 0": dict(batch0=True),
}


def _small_case():
    c = SMALL
    ref, srcs, proj, hyp, interval, weights = T.make_inputs(c)
    depth = T.restate_depth(c, hyp, interval)
    want, bar = T.agg_reference(c, ref, srcs, proj, depth, weights)
    return c, (ref, srcs, proj, depth, weights), want, bar


def test_fp32_evaluation_passes_the_bar():
    c, args, want, bar = _small_case()
    got = fp32_agg(c, *args)
    assert T.worst_ratio(got.reshape(want.shape), want, bar) <= 1.0


@pytest.mark.parametrize("name", list(CORRUPTIONS))
def test_bar_rejects_corruption(name):
    c, args, want, bar = _small_case()
    got = fp32_agg(c, *args, **CORRUPTIONS[name])
    assert T.worst_ratio(got.reshape(want.shape), want, bar) > 1.0


def test_small_case_has_last_row_cells():
    """the last-row corruption only bites where samples fall on cells with y0 = H - 1"""
    c, (ref, srcs, proj, depth, weights), _, _ = _small_case()
    rays = T.restate_rays(proj, c.H, c.W)
    _, iy = T.restate_coords(rays[:, 0], proj[:, 0, 9:], depth, c.H, c.W)
    assert bool((torch.floor(iy) == c.H - 1).any())
