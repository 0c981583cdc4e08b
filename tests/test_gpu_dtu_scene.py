"""The DTU filter for whole scenes on the device (``-m gpu``): effimvs_dtu_filter_views_f32 through fusion.dtu_filter_views
against fusion.dtu_filter_view per view (bit for bit, ragged source lists, up to the 31-source limit), against upstream's
golden file and the NumPy oracle at 1600x1184 (the bars of test_gpu_parity's single-view tests), under CUDA-graph
capture, one launch per rank, and run_scene with the graphed infer and cuda_dtu_fuse end to end."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
DEV = "cuda"


def _bits(t):
    return t.view(torch.int32) if t.dtype == torch.float32 else t


def _assert_same(got, want, what):
    assert got.shape == want.shape and got.dtype == want.dtype, (what, got.shape, want.shape)
    assert torch.equal(_bits(got), _bits(want)), what


def _scene(n, w, h, seed=2):
    """n views on a camera ring over the rendered surface: depth stack (n,h,w) on the device, K (n,3,3), E (n,4,4) float32"""
    from effimvs_b200 import synthetic
    E, K = synthetic.camera_ring(n, w, h)
    depths = synthetic.render_plane_scene(E, K, w, h, noise=0.05, seed=seed)
    return depths.to(DEV), np.repeat(K.numpy().astype(np.float32)[None], n, 0), E.numpy().astype(np.float32)


def _pairs(n, counts, seed):
    """a source list of each count for every view: distinct other views in a seeded order (ragged across views)"""
    rng = np.random.default_rng(seed)
    return [[int(j) for j in rng.permutation([j for j in range(n) if j != i])[:counts[i % len(counts)]]] for i in range(n)]


def _per_view(stack, confs, K, E, views, pairs):
    from effimvs_b200 import fusion
    return [fusion.dtu_filter_view(stack[i], confs[b], stack[pairs[i]], K[i], E[i], [K[j] for j in pairs[i]],
                                   [E[j] for j in pairs[i]], 0.5) for b, i in enumerate(views)]


# (scene views, width, height, reference views, their source counts)
CASES = {"small": (32, 64, 48, [0, 5, 17, 31], [31, 1, 9, 4]),
         "dtu": (11, 1600, 1184, [0, 4, 8], [10, 6, 3])}


@pytest.mark.parametrize("name", sorted(CASES))
def test_batched_equals_single_view(name):
    from effimvs_b200 import fusion
    n, w, h, views, counts = CASES[name]
    stack, K, E = _scene(n, w, h)
    pairs = _pairs(n, [1], 0)
    for i, c in zip(views, counts):
        pairs[i] = _pairs(n, [c], i)[i]
    table = fusion.dtu_scene_cameras(K, E, pairs)
    confs = torch.rand(len(views), h // 2, w // 2, generator=torch.Generator().manual_seed(1)).to(DEV)
    got = fusion.dtu_filter_views(stack, views, confs, table, 0.5)
    want = _per_view(stack, confs, K, E, views, pairs)
    for b, i in enumerate(views):
        for key in ("final", "geo", "depth_avg", "points"):
            _assert_same(got[key][b], want[b][key], (name, i, key))
    kept = [float(got["final"][b].float().mean()) for b in range(len(views))]
    print("{}: kept fraction per view {}".format(name, kept))
    if name == "dtu":
        assert 0.05 < kept[0] < 0.95        # view 0 with 10 sources keeps part of the view: the comparison is not vacuous


def _dtu_filter_compare(out, want_final, want_geo, want_avg, want_pts, dist_band, diff_band):
    """masks identical except where a rung is decided within the band (float64 rounding of the matrix
    products); averaged depth / points equal wherever the masks agree"""
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


def _view(out, b):
    return {k: out[k][b] for k in ("final", "geo", "depth_avg", "points")}


def test_batched_golden():
    """the batched kernel against upstream's own functions + real cv2.remap (tests/golden/dtu_filter.npz), view 0 of a
    launch that filters two views"""
    from effimvs_b200 import fusion
    z = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "dtu_filter.npz"))
    d, K, E = z["depths"], z["K"], z["E"]
    n = d.shape[0]
    pairs = [list(range(1, n))] + [[0]] * (n - 1)
    table = fusion.dtu_scene_cameras(np.repeat(K[None], n, 0), E, pairs)
    conf = torch.from_numpy(z["confidence"]).to(DEV)
    out = fusion.dtu_filter_views(torch.from_numpy(d).to(DEV), [0, 1], torch.stack([conf, conf]), table, float(z["conf_thres"]))
    _dtu_filter_compare(_view(out, 0), z["final_mask"], z["geo_mask"], z["depth_avg"], z["points"], 1e-5, 1e-5)


def test_batched_vs_oracle_dtu_size():
    """a 1600x1184 reference view with 10 source views against the NumPy oracle, filtered in one launch with a second view"""
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
    pairs = [list(range(1, v + 1))] + [[0, (i % v) + 1] for i in range(1, v + 1)]
    table = fusion.dtu_scene_cameras(np.repeat(K32[None], v + 1, 0), E32, pairs)
    out = fusion.dtu_filter_views(depths.to(DEV), [0, 5], torch.stack([conf, conf]).to(DEV), table, 0.5)
    assert 0.05 < want["final"].mean() < 0.95
    _dtu_filter_compare(_view(out, 0), want["final"], want["geo"], want["depth_avg"], want["points"], 2e-5, 2e-5)


def test_cuda_graph_replay_equals_eager():
    """fusion.dtu_filter_views captured in a CUDA graph: a replay equals the eager call bit for bit, and a replay after the
    depth stack and confidences are overwritten in place equals the eager call on the new contents"""
    from effimvs_b200 import fusion
    n, w, h = 12, 160, 128
    stack, K, E = _scene(n, w, h)
    other, _, _ = _scene(n, w, h, seed=5)
    pairs = _pairs(n, [6, 3, 9, 1], 7)
    table = fusion.dtu_scene_cameras(K, E, pairs)
    views = [1, 2, 3, 7, 11]
    g = torch.Generator().manual_seed(2)
    confs, confs2 = torch.rand(len(views), h // 2, w // 2, generator=g).to(DEV), torch.rand(len(views), h // 2, w // 2, generator=g).to(DEV)
    eager = fusion.dtu_filter_views(stack, views, confs, table)          # also puts the table's rows on the device
    eager2 = fusion.dtu_filter_views(other, views, confs2, table)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        fusion.dtu_filter_views(stack, views, confs, table)
    torch.cuda.current_stream().wait_stream(s)
    graph = torch.cuda.CUDAGraph()
    with torch.cuda.graph(graph):
        out = fusion.dtu_filter_views(stack, views, confs, table)
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
    """run_scene with cuda_dtu_fuse enqueues one filter launch for all of the rank's views"""
    from effimvs_b200 import ops, scene, synthetic
    n, w, h = 9, 96, 64
    stack, K, E = _scene(n, w, h)
    cams = synthetic.stage_cameras(torch.from_numpy(E).double(), torch.from_numpy(K[0]).double(), 1)["stage4"][0].to(DEV)
    pairs = _pairs(n, [4, 2, 5], 3)
    fuse = scene.cuda_dtu_fuse(cams, pairs)
    conf = torch.rand(n, h // 2, w // 2, generator=torch.Generator().manual_seed(4)).to(DEV)

    def infer(i, srcs):
        return stack[i], conf[i]
    for sharding in ("round_robin", "block"):
        before = ops.LAUNCHES
        got = scene.run_scene(infer, fuse, n, pairs, 0, 1, DEV, sharding=sharding)
        assert ops.LAUNCHES - before == 1 and sorted(got) == list(range(n))
    before = ops.LAUNCHES
    fuse(3, stack[3].reshape(1, 1, h, w), conf[3:4], pairs[3], stack[pairs[3]].reshape(1, -1, 1, h, w))
    assert ops.LAUNCHES - before == 1


def test_run_scene_graphed_infer_and_dtu_fuse_end_to_end():
    """an 8-view 160x128 scene through the graphed cascade (4 source views) and cuda_dtu_fuse: the depth map and the points
    of every view equal a hand-written per-view loop of dtu_filter_view over the gathered depth maps, and so do those of
    the per-view fuse call"""
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
        infer, _ = scene.cuda_scene_callables(model, imgs, cams, dv, 2.0, 6.0, 2, 0.3, feature_cache=True, graphed_src_views=4)
        fuse = scene.cuda_dtu_fuse(cams["stage4"], fpairs)
        maps = {}
        batch = infer.batch

        def recording_batch(items):
            res = batch(items)
            maps.update({i: dc for (i, _), dc in zip(items, res)})
            return res
        infer.batch = recording_batch
        got = scene.run_scene(infer, fuse, n, pairs, 0, 1, DEV, fuse_pairs=fpairs, sharding="block")
        plain = scene.run_scene(lambda i, s: maps[i], lambda *a: fuse(*a), n, pairs, 0, 1, DEV, fuse_pairs=fpairs)
    c = cams["stage4"].cpu()
    K32, E32 = c[:, 1, :3, :3].numpy(), c[:, 0].numpy()
    all_depths = torch.stack([maps[i][0] for i in range(n)])
    total = 0
    for i in range(n):
        src = fpairs[i]
        want = fusion.dtu_filter_view(all_depths[i], maps[i][1], all_depths[src], K32[i], E32[i], [K32[j] for j in src],
                                      [E32[j] for j in src], 0.5)
        pts = want["points"][:, want["final"]].t().contiguous()
        for run in (got, plain):
            _assert_same(run[i][1], maps[i][0], ("depth", i))
            _assert_same(run[i][0], pts, ("points", i))
        total += pts.shape[0]
    print("run_scene with cuda_dtu_fuse: {} points over {} views".format(total, n))
