"""The dynamic filter for whole scenes on the device (``-m gpu``): effimvs_fusion_filter_views_f32 through
fusion.filter_views against fusion.filter_view(..., torch_inverse=False) per view (bit for bit: ragged source lists from
1 to 16, relative depth errors, confidences at half and full resolution, views out of scene order, a stack_rows mapping,
1600x1184), against upstream's golden file and the oracle at 1600x1184 (the bars of test_gpu_parity's single-view tests),
under CUDA-graph capture, one launch per rank through cuda_scene_callables' fuse, and run_scene with the graphed infer
end to end."""
import numpy as np
import pytest
import torch

from util import golden, rel_max

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t


def _assert_same(got, want, what):
    assert got.shape == want.shape and got.dtype == want.dtype, (what, got.shape, want.shape)
    assert torch.equal(_bits(got), _bits(want)), what


def _scene(n, w, h, seed=2, noise=0.05):
    """n views on a camera arc over the rendered surface: depth stack (n,h,w), stage-4 cameras (n,2,4,4), on the device"""
    from effimvs_b200 import synthetic
    E, K = synthetic.camera_arc(n, w, h)
    depths = synthetic.render_plane_scene(E, K, w, h, noise=noise, seed=seed)
    return depths.to(DEV), synthetic.stage_cameras(E, K, 1)["stage4"][0].to(DEV)


def _pairs(n, counts, seed):
    """a source list of each count for every view: distinct other views in a seeded order (ragged across views)"""
    rng = np.random.default_rng(seed)
    return [[int(j) for j in rng.permutation([j for j in range(n) if j != i])[:counts[i % len(counts)]]] for i in range(n)]


def _per_view(stack, confs, cams, views, pairs, args, relative=False):
    """filter_view per reference view on copies of its maps and cameras (what cuda_scene_callables' fuse does)"""
    from effimvs_b200 import fusion
    return [fusion.filter_view(stack[i][None, None], confs[b][None], stack[pairs[i]][None, :, None], cams[i][None],
                               cams[pairs[i]][None], *args, relative=relative, torch_inverse=False) for b, i in enumerate(views)]


# (scene views, width, height, reference views (in this order), their source counts, thres_view, relative, confidence
#  scale (2: half resolution), stack order reversed)
CASES = {"tv1_ragged": (20, 64, 48, [5, 0, 17, 3], [16, 1, 7, 2], 1, False, 2, False),
         "tv3_relative_fullconf": (20, 64, 48, [11, 2, 19], [3, 16, 9], 3, True, 1, False),
         "stack_rows": (20, 64, 48, [7, 13, 1], [4, 16, 2], 2, False, 2, True),
         "dtu": (11, 1600, 1184, [0, 6], [10, 10], 2, False, 2, False)}


@pytest.mark.parametrize("name", sorted(CASES))
def test_batched_equals_single_view(name):
    from effimvs_b200 import fusion
    n, w, h, views, counts, tv, relative, cs, reverse = CASES[name]
    stack, cams = _scene(n, w, h, noise=0.15 if name == "dtu" else 0.05)
    pairs = _pairs(n, [max(tv, 1)], 0)
    for i, c in zip(views, counts):
        pairs[i] = _pairs(n, [c], i)[i]
    if name == "dtu":
        pairs[0] = list(range(1, 11))
    table = fusion.dynamic_scene_cameras(cams, pairs)
    confs = torch.rand(len(views), h // cs, w // cs, generator=torch.Generator().manual_seed(1)).to(DEV)
    args = (2.0, 6.0, tv, 0.3)
    want = _per_view(stack, confs, cams, views, pairs, args, relative)
    if reverse:                                     # the maps in reverse order, read through stack_rows
        got = fusion.filter_views(stack.flip(0).contiguous(), views, confs, table, *args, relative=relative,
                                  stack_rows={i: n - 1 - i for i in range(n)})
    else:
        got = fusion.filter_views(stack, views, confs, table, *args, relative=relative)
    for b, i in enumerate(views):
        for key in ("final", "depth_avg", "points"):
            _assert_same(got[key][b:b + 1], want[b][key], (name, i, key))
    kept = [float(got["final"][b].float().mean()) for b in range(len(views))]
    print("{}: kept fraction per view {}".format(name, kept))
    if name == "dtu":
        assert 0.05 < kept[0] < 0.95        # view 0 with 10 sources keeps part of the view: the comparison is not vacuous


def _near_threshold(xyd, ref_depth, cx, cy, ks, dist_base, rel_base, rel=1e-5):
    """test_gpu_parity's band: pixels whose reprojection distance / depth error lies within `rel` of a ladder threshold"""
    e_xy = ((xyd[:, :, 0] - cx) ** 2 + (xyd[:, :, 1] - cy) ** 2).sqrt()
    e_d = (ref_depth - xyd[:, :, 2]).abs()
    band_xy = rel * max(float(cx.max()), float(cy.max()))
    band_d = rel * float(ref_depth.abs().max())
    near = torch.zeros_like(e_xy, dtype=torch.bool)
    for k in ks:
        near |= ((e_xy - k / dist_base).abs() <= band_xy) | ((e_d - k / rel_base).abs() <= band_d)
    return near.any(dim=1, keepdim=True)


def test_batched_golden():
    """view 0 of a launch that filters two views of a scene stack built from tests/golden/fusion_tank.npz, with the bars of
    test_fusion_golden (the per-rung masks, which the batched kernel does not write, from the single-view kernel)"""
    from effimvs_b200 import fusion
    g = golden("fusion_tank", DEV)
    n, v, _, h, w = g["srcs_depth"].shape
    stack = torch.cat([g["ref_depth"][0], g["srcs_depth"][0, :, 0]])
    cams = torch.cat([g["ref_cam"], g["srcs_cam"][0]])
    pairs = [list(range(1, v + 1))] + [[0] + [j for j in range(1, v + 1) if j != i][:2] for i in range(1, v + 1)]
    table = fusion.dynamic_scene_cameras(cams, pairs)
    conf = g["conf"][0]
    args = (g["dist_base"], g["rel_diff_base"], g["thres_view"], g["prob_threshold"])
    got = fusion.filter_views(stack, [0, 2], torch.stack([conf, conf]), table, *args)
    out = {k: got[k][:1] for k in got}
    single = fusion.filter_view(g["ref_depth"], g["conf"], g["srcs_depth"], g["ref_cam"], g["srcs_cam"], *args, want_masks=True,
                                torch_inverse=False)
    for key in out:
        _assert_same(out[key], single[key], key)
    want = g["reproj_xyd"]
    cx = (torch.arange(w, device=DEV) + 0.5).reshape(1, 1, 1, w)
    cy = (torch.arange(h, device=DEV) + 0.5).reshape(1, 1, h, 1)
    near = _near_threshold(want, g["ref_depth"], cx, cy, range(g["thres_view"], v + 1), g["dist_base"], g["rel_diff_base"])
    diff = (single["masks"] != g["masks"].bool()).any(dim=2).any(dim=1, keepdim=True)
    assert not (diff & ~near).any(), "masks differ away from thresholds"
    keep = ~near
    assert torch.equal(out["final"][keep], g["final"].bool()[keep])
    same = ~diff
    assert rel_max(out["depth_avg"][same], g["depth_avg"][same]) < 1e-5
    assert rel_max(out["points"][same.expand(-1, 3, -1, -1)], g["points"][same.expand(-1, 3, -1, -1)]) < 1e-4


def test_batched_vs_oracle_full_size():
    """a 1600x1184 reference view with 10 source views against oracle.fusion.fuse_view, filtered in one launch with a
    second view, with the bars of test_fusion_vs_oracle_full_size"""
    from effimvs_b200 import fusion, synthetic
    from oracle import fusion as ofu
    h, w, v = 1184, 1600, 10
    E, K = synthetic.camera_ring(v + 1, w, h)
    depths = synthetic.render_plane_scene(E, K, w, h, noise=0.15, seed=4).to(DEV)
    cams = synthetic.stage_cameras(E, K, 1)["stage4"].to(DEV)
    conf = torch.rand(1, h // 2, w // 2, device=DEV)
    args = (depths[0][None, None], conf, depths[1:][None, :, None], cams[:, 0], cams[:, 1:], 2, 6, 2, 0.3)
    pairs = [list(range(1, v + 1))] + [[0, (i % v) + 1] for i in range(1, v + 1)]
    table = fusion.dynamic_scene_cameras(cams[0], pairs)
    got = fusion.filter_views(depths, [0, 5], torch.cat([conf, conf]), table, 2, 6, 2, 0.3)
    got = {k: got[k][:1] for k in got}
    want = ofu.fuse_view(*args)
    cx = (torch.arange(w, device=DEV) + 0.5).reshape(1, 1, 1, w)
    cy = (torch.arange(h, device=DEV) + 0.5).reshape(1, 1, h, 1)
    near = _near_threshold(want["reproj_xyd"], args[0], cx, cy, range(2, v + 1), 2, 6)
    print("fusion band: {:.4f} of the pixels are excluded".format(float(near.float().mean())))
    assert float(near.float().mean()) < 0.15, float(near.float().mean())
    assert torch.equal(got["final"][~near], want["final"][~near])
    got_m = fusion.filter_view(*args, want_masks=True, torch_inverse=False)["masks"]
    agree = ~(got_m != want["masks"]).any(dim=2).any(dim=1, keepdim=True)
    assert float(agree.float().mean()) > 0.98
    d = (got["depth_avg"] - want["depth_avg"]).abs() * agree
    bad = d > 1e-5 * float(want["depth_avg"].abs().max())
    assert int(bad.sum()) <= 1e-5 * bad.numel() and float(d.max()) < 1e-4 * float(want["depth_avg"].abs().max()), \
        (int(bad.sum()), float(d.max()))
    assert 0.3 < float(want["final"].float().mean()) < 0.99


def test_cuda_graph_replay_equals_eager():
    """fusion.filter_views captured in a CUDA graph: a replay equals the eager call bit for bit, and a replay after the
    depth stack and confidences are overwritten in place equals the eager call on the new contents"""
    from effimvs_b200 import fusion
    n, w, h = 12, 160, 128
    stack, cams = _scene(n, w, h)
    other, _ = _scene(n, w, h, seed=5)
    pairs = _pairs(n, [6, 3, 9, 2], 7)
    table = fusion.dynamic_scene_cameras(cams, pairs)
    views = [1, 2, 3, 7, 11]
    g = torch.Generator().manual_seed(2)
    confs, confs2 = torch.rand(len(views), h // 2, w // 2, generator=g).to(DEV), torch.rand(len(views), h // 2, w // 2, generator=g).to(DEV)
    args = (2.0, 6.0, 2, 0.3)
    eager = fusion.filter_views(stack, views, confs, table, *args)          # also puts the table's rows on the device
    eager2 = fusion.filter_views(other, views, confs2, table, *args)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fusion.filter_views(stack, views, confs, table, *args)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = fusion.filter_views(stack, views, confs, table, *args)
    graph.replay()
    torch.cuda.synchronize()
    for key in eager:
        _assert_same(out[key], eager[key], key)
    stack.copy_(other)
    confs.copy_(confs2)
    graph.replay()
    torch.cuda.synchronize()
    for key in eager:
        _assert_same(out[key], eager2[key], key)


def test_one_launch_per_rank():
    """run_scene with cuda_scene_callables' fuse enqueues one filter launch for all of the rank's views once the scene's
    camera table exists (its inverse table is one more launch, once per scene); the per-view call stays filter_view"""
    from effimvs_b200 import ops, scene
    n, w, h = 9, 96, 64
    stack, cams = _scene(n, w, h)
    pairs = _pairs(n, [4, 2, 5], 3)
    _, fuse = scene.cuda_scene_callables(None, torch.zeros(n, 3, 8, 8, device=DEV), {"stage4": cams}, torch.zeros(4, device=DEV),
                                         2.0, 6.0, 2, 0.3)
    conf = torch.rand(n, h // 2, w // 2, generator=torch.Generator().manual_seed(4)).to(DEV)

    def infer(i, srcs):
        return stack[i], conf[i]
    before = ops.LAUNCHES
    first = scene.run_scene(infer, fuse, n, pairs, 0, 1, DEV)
    assert ops.LAUNCHES - before == 2                       # the inverse table, then the filter
    for sharding in ("round_robin", "block"):
        before = ops.LAUNCHES
        got = scene.run_scene(infer, fuse, n, pairs, 0, 1, DEV, sharding=sharding)
        assert ops.LAUNCHES - before == 1 and sorted(got) == list(range(n))
        for i in got:
            _assert_same(got[i][0], first[i][0], ("points", sharding, i))
    before = ops.LAUNCHES
    fuse(3, stack[3].reshape(1, 1, h, w), conf[3:4], pairs[3], stack[pairs[3]].reshape(1, -1, 1, h, w))
    assert ops.LAUNCHES - before == 2                       # filter_view: camera inversion + filter, as before


def test_run_scene_graphed_infer_and_batched_fuse_end_to_end():
    """an 8-view 160x128 scene through the graphed cascade (4 source views) and cuda_scene_callables' fuse, now batched:
    the depth map and the points of every view equal a hand-written per-view loop of filter_view over the gathered depth
    maps, and so do those of run_scene driving the per-view fuse call"""
    from util import dtu_model
    from effimvs_b200 import fusion, hotpath, scene, synthetic
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    n, W, H = 8, 160, 128
    model = dtu_model(hotpath.CudaHotPath("f32"), DEV, ndepths="8,4,4")
    imgs = torch.rand(n, 3, H, W, generator=torch.Generator().manual_seed(0)).to(DEV)
    E, K = synthetic.camera_arc(n, W, H)
    cams = {k: v[0].to(DEV) for k, v in synthetic.stage_cameras(E, K, 1).items()}
    dv = torch.linspace(1 / 935.0, 1 / 425.0, 384, device=DEV)
    nb = lambda i, m: [j for d in range(1, m // 2 + 1) for j in ((i - d) % n, (i + d) % n)]      # noqa: E731
    pairs = [nb(i, 4) for i in range(n)]
    fpairs = [nb(i, 6)[:4 + i % 3] for i in range(n)]
    with torch.no_grad():
        infer, fuse = scene.cuda_scene_callables(model, imgs, cams, dv, 2.0, 6.0, 2, 0.3, feature_cache=True, graphed_src_views=4)
        assert hasattr(fuse, "batch")
        maps = {}
        batch = infer.batch

        def recording_batch(items):
            res = batch(items)
            maps.update({i: dc for (i, _), dc in zip(items, res)})
            return res
        infer.batch = recording_batch
        got = scene.run_scene(infer, fuse, n, pairs, 0, 1, DEV, fuse_pairs=fpairs, sharding="block")
        plain = scene.run_scene(lambda i, s: maps[i], lambda *a: fuse(*a), n, pairs, 0, 1, DEV, fuse_pairs=fpairs)
    full = cams["stage4"]
    all_depths = torch.stack([maps[i][0] for i in range(n)])
    total = 0
    for i in range(n):
        src = fpairs[i]
        want = fusion.filter_view(all_depths[i][None, None], maps[i][1][None], all_depths[src][None, :, None], full[i][None],
                                  full[src][None], 2.0, 6.0, 2, 0.3, torch_inverse=False)
        pts = want["points"][0][:, want["final"][0, 0]].t().contiguous()
        for run in (got, plain):
            _assert_same(run[i][1], maps[i][0], ("depth", i))
            _assert_same(run[i][0], pts, ("points", i))
        total += pts.shape[0]
    assert total > 0
    print("run_scene with the batched dynamic fuse: {} points over {} views".format(total, n))
