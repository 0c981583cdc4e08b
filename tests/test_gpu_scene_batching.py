"""View batching in the scene runner on the device (``-m gpu``): GraphedViewRunner with K = views_per_replay reference
views per replay of the cascade graph against K = 1, the padded short last batch, the static index buffer across
replays, the layout of the gathered features, and run_scene through cuda_scene_callables end to end.

Bar (as the feature-cache test of test_gpu_parity): every depth map within 1e-3 * (935 - 425) mm on >= 99.9 % of its
pixels -- cuDNN may pick other algorithms at batch K, so batched and unbatched maps need not be bit-identical."""
import pytest
import torch

from util import dtu_model

pytestmark = pytest.mark.gpu
DEV = "cuda"
DEPTH_RANGE = 935.0 - 425.0
N_VIEWS = 9
SHAPES = {"small": (160, 128, "8,4,4"), "dtu": (1600, 1184, "48,8,8")}


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


def _neighbours(i, n, n_views=N_VIEWS):
    return [j for d in range(1, n // 2 + 1) for j in ((i - d) % n_views, (i + d) % n_views)]


@pytest.fixture(scope="module")
def scenes(hp):
    """per shape: (model, imgs, cams, depth values, pairs) of a 9-view scene, 4 source views per reference view"""
    from effimvs_b200 import synthetic
    out = {}
    for name, (W, H, nd) in SHAPES.items():
        model = dtu_model(hp, DEV, ndepths=nd)
        g = torch.Generator().manual_seed(0)
        imgs = torch.rand(N_VIEWS, 3, H, W, generator=g).to(DEV)
        E, K = synthetic.camera_arc(N_VIEWS, W, H)
        cams = {k: v[0].to(DEV) for k, v in synthetic.stage_cameras(E, K, 1).items()}
        dv = torch.linspace(1 / 935.0, 1 / 425.0, 384, device=DEV)
        out[name] = (model, imgs, cams, dv, [_neighbours(i, 4) for i in range(N_VIEWS)])
    return out


@pytest.fixture(scope="module")
def runner(scenes):
    """runner(shape, K): the GraphedViewRunner of that scene at K views per replay, captured once per module"""
    from effimvs_b200 import scene
    made = {}

    def get(name, k):
        if (name, k) not in made:
            model, imgs, cams, dv, _ = scenes[name]
            made[(name, k)] = scene.GraphedViewRunner(model, imgs, cams, dv, 4, views_per_replay=k)
        return made[(name, k)]
    yield get
    made.clear()
    torch.cuda.empty_cache()


def _all_views(runner, pairs):
    """every view of the scene through the runner in groups of K -> ({view: (depth, conf)}, results per replay)"""
    from effimvs_b200 import scene
    res, per_replay = {}, []
    for group, n in scene.view_groups(list(range(N_VIEWS)), runner.views_per_replay):
        got = runner.infer_batch([(i, pairs[i]) for i in group[:n]])
        per_replay.append(len(got))
        res.update(zip(group[:n], got))
    return res, per_replay


def frac_within(a, b, tol):
    return float(((a - b).abs() <= tol).float().mean())


@pytest.mark.parametrize("name", ["small", "dtu"])
@pytest.mark.parametrize("k", [2, 3, 4])
def test_batched_equals_unbatched(scenes, runner, name, k):
    pairs = scenes[name][4]
    one, _ = _all_views(runner(name, 1), pairs)
    got, per_replay = _all_views(runner(name, k), pairs)
    assert sorted(got) == list(range(N_VIEWS))
    # 9 views in groups of k: k = 4 gives 4 + 4 + 1, the padded rows' outputs are dropped
    assert per_replay == [min(k, N_VIEWS - a) for a in range(0, N_VIEWS, k)]
    worst = 0.0
    for i in range(N_VIEWS):
        d1, c1 = one[i]
        d, c = got[i]
        assert d.shape == d1.shape and c.shape == c1.shape
        worst = max(worst, float((d - d1).abs().max()))
        assert frac_within(d, d1, 1e-3 * DEPTH_RANGE) >= 0.999, (name, k, i)
    print("{} K={}: max |d depth| against K=1 over {} views: {:.3e} mm".format(name, k, N_VIEWS, worst))


def test_short_last_batch(scenes, runner):
    """9 views at K = 4: the tail replay holds one real view (view 8) and three padded copies of it; it returns one result,
    which meets the bar against K = 1, and padding rows never reach the caller"""
    pairs = scenes["small"][4]
    r4 = runner("small", 4)
    tail = r4.infer_batch([(8, pairs[8])])
    assert len(tail) == 1
    want = runner("small", 1).infer_batch([(8, pairs[8])])[0]
    assert frac_within(tail[0][0], want[0], 1e-3 * DEPTH_RANGE) >= 0.999
    # a tail that follows a full batch of other views: no stale rows leak into its result
    r4.infer_batch([(i, pairs[i]) for i in range(4)])
    again = r4.infer_batch([(8, pairs[8])])
    assert len(again) == 1 and torch.equal(again[0][0], tail[0][0]) and torch.equal(again[0][1], tail[0][1])
    with pytest.raises(ValueError):
        r4.infer_batch([(i, pairs[i]) for i in range(5)])
    with pytest.raises(ValueError):
        r4.infer_batch([(0, pairs[0][:3])])


def test_index_buffer_across_replays(scenes, runner):
    """two different batches alternated over four replays: each replay is bit-identical to the earlier replay of the same
    batch (the index buffer and the cache rows are current for every replay)"""
    pairs = scenes["small"][4]
    r2 = runner("small", 2)
    r2.clear_cache()
    a, b = [(0, pairs[0]), (1, pairs[1])], [(5, pairs[5]), (7, pairs[7])]
    outs = [r2.infer_batch(x) for x in (a, b, a, b)]
    for first, second in ((outs[0], outs[2]), (outs[1], outs[3])):
        for (d0, c0), (d1, c1) in zip(first, second):
            assert torch.equal(d0, d1) and torch.equal(c0, c1)
    assert not torch.equal(outs[0][0][0], outs[1][0][0])


@pytest.mark.parametrize("name", ["small", "dtu"])
def test_gathered_features_layout(runner, name):
    """the maps the cascade reads (gathered from the stacked cache) and every cache row are channels-last with 32-byte
    aligned data pointers: the condition of the TMA tile kernels of effimvs_warp_corr_agg_f32"""
    r3 = runner(name, 3)
    for stage in r3.feat_in:
        assert len(stage) == 5
        for t in stage:
            assert t.shape[0] == 3 and t.is_contiguous(memory_format=torch.channels_last) and not t.is_contiguous()
            assert t.data_ptr() % 32 == 0
    for c in r3.cache:
        rows = c.permute(0, 3, 1, 2)
        assert c.shape[0] == N_VIEWS
        for j in range(N_VIEWS):
            assert rows[j:j + 1].is_contiguous(memory_format=torch.channels_last) and rows[j].data_ptr() % 32 == 0


@pytest.mark.parametrize("k", [3, 4])
def test_run_scene_batched_end_to_end(scenes, k):
    from effimvs_b200 import scene
    model, imgs, cams, dv, pairs = scenes["small"]
    H, W = imgs.shape[2:]
    runs = {}
    for kk in (1, k):
        infer, fuse = scene.cuda_scene_callables(model, imgs, cams, dv, 2.0, 6.0, 2, 0.3, feature_cache=True,
                                                 graphed_src_views=4, views_per_replay=kk)
        runs[kk] = scene.run_scene(infer, fuse, N_VIEWS, pairs, 0, 1, DEV, sharding="block", views_per_batch=kk)
    assert sorted(runs[k]) == sorted(runs[1]) == list(range(N_VIEWS))
    worst = 0.0
    for i in range(N_VIEWS):
        d0, d1 = runs[1][i][1], runs[k][i][1]
        worst = max(worst, float((d1 - d0).abs().max()))
        assert frac_within(d1, d0, 1e-3 * DEPTH_RANGE) >= 0.999, i
        n0, n1 = runs[1][i][0].shape[0], runs[k][i][0].shape[0]
        assert abs(n0 - n1) <= 0.02 * H * W, i
    print("run_scene K={}: max |d depth| against K=1: {:.3e} mm".format(k, worst))
