"""View batching in the scene runner, host side (CPU): the grouping of a rank's views into batches, and run_scene with an
injected batched `infer` on 2 gloo ranks -- which must equal the unbatched single-rank run bit for bit.  The graphed
batched runner behind the same interface is covered by test_gpu_scene_batching."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import effimvs_b200  # noqa: F401
from effimvs_b200 import scene, synthetic

N_VIEWS, H, W = 7, 24, 32


@pytest.mark.parametrize("views,k,want", [
    ([0, 1, 2, 3, 4, 5, 6], 3, [([0, 1, 2], 3), ([3, 4, 5], 3), ([6, 6, 6], 1)]),
    ([4, 5, 6], 3, [([4, 5, 6], 3)]),
    ([2, 3, 4, 5], 1, [([2], 1), ([3], 1), ([4], 1), ([5], 1)]),
    ([1, 3, 5], 2, [([1, 3], 2), ([5, 5], 1)]),
    ([5], 4, [([5, 5, 5, 5], 1)]),              # fewer views than k
    ([], 4, []),                                # a rank without a view
])
def test_view_groups(views, k, want):
    got = scene.view_groups(views, k)
    assert got == want
    assert [v for g, n in got for v in g[:n]] == views          # every view once, in order; padding is never real


def test_view_groups_rejects_empty_groups():
    with pytest.raises(ValueError):
        scene.view_groups([0, 1], 0)


def _inputs(n_views=N_VIEWS):
    E, K = synthetic.camera_ring(n_views, W, H)
    depths = synthetic.render_plane_scene(E, K, W, H, noise=0.05, seed=1)
    cams = synthetic.stage_cameras(E, K, 1)["stage4"]
    pairs = [[(i + k) % n_views for k in range(1, min(4, n_views))] for i in range(n_views)]
    return depths, cams, pairs


def _run(rank, world, sharding="round_robin", k=None, n_views=N_VIEWS):
    """k None: the unbatched callable; else a callable with `batch` that records the groups it is given"""
    from oracle import fusion as ofu
    depths, cams, pairs = _inputs(n_views)
    thres_view = min(2, n_views - 1)

    def infer(i, srcs):
        return depths[i], torch.full((H // 2, W // 2), 0.9)

    calls = []
    if k is not None:
        def batch(items):
            calls.append([i for i, _ in items])
            assert all(list(s) == pairs[i] for i, s in items)
            return [infer(i, s) for i, s in items]
        infer.batch = batch
        infer.views_per_batch = k

    def fuse(i, ref_depth, conf, srcs, src_depths):
        return ofu.fuse_view(ref_depth, conf, src_depths, cams[:, i], cams[:, srcs], 1, 0.5, thres_view, 0.3)
    return scene.run_scene(infer, fuse, n_views, pairs, rank, world, device="cpu", sharding=sharding), calls


def _worker(rank, world, port, out_dir, sharding, k):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        res, calls = _run(rank, world, sharding, k)
        torch.save({"res": {i: (p, d) for i, (p, d) in res.items()}, "calls": calls}, os.path.join(out_dir, "rank{}.pt".format(rank)))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("k", [1, 2, 3])
@pytest.mark.parametrize("sharding", ["round_robin", "block"])
def test_two_ranks_batched_equal_one_unbatched(tmp_path, sharding, k):
    single, _ = _run(0, 1)
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_worker, args=(2, port, str(tmp_path), sharding, k), nprocs=2, join=True)
    merged = {}
    for r in range(2):
        part = torch.load(os.path.join(str(tmp_path), "rank{}.pt".format(r)))
        mine = scene.shard_views(N_VIEWS, r, 2, sharding)
        assert sorted(part["res"]) == mine
        # the rank's views in view order, in groups of at most k, every view exactly once
        assert part["calls"] == [g[:n] for g, n in scene.view_groups(mine, k)]
        merged.update(part["res"])
    assert sorted(merged) == list(range(N_VIEWS))
    for i in range(N_VIEWS):
        assert torch.equal(merged[i][0], single[i][0]) and torch.equal(merged[i][1], single[i][1])
    assert sum(v[0].shape[0] for v in single.values()) > 0.3 * N_VIEWS * H * W


def test_explicit_views_per_batch_overrides_the_callable_default():
    single, _ = _run(0, 1)
    from oracle import fusion as ofu
    depths, cams, pairs = _inputs()
    calls = []

    def infer(i, srcs):
        return depths[i], torch.full((H // 2, W // 2), 0.9)

    def batch(items):
        calls.append([i for i, _ in items])
        return [infer(i, s) for i, s in items]
    infer.batch, infer.views_per_batch = batch, 2

    def fuse(i, ref_depth, conf, srcs, src_depths):
        return ofu.fuse_view(ref_depth, conf, src_depths, cams[:, i], cams[:, srcs], 1, 0.5, 2, 0.3)
    got = scene.run_scene(infer, fuse, N_VIEWS, pairs, device="cpu", views_per_batch=4)
    assert calls == [[0, 1, 2, 3], [4, 5, 6]]
    for i in range(N_VIEWS):
        assert torch.equal(got[i][0], single[i][0]) and torch.equal(got[i][1], single[i][1])


def test_views_per_batch_without_a_batched_infer_is_rejected():
    with pytest.raises(ValueError):
        scene.run_scene(lambda i, s: None, None, 3, [[1], [2], [0]], device="cpu", views_per_batch=2)


def test_batched_callables_need_the_graphs():
    with pytest.raises(ValueError):
        scene.cuda_scene_callables(None, torch.zeros(2, 3, 8, 8), {}, torch.zeros(4), 1.0, 1.0, 1, 0.3,
                                   feature_cache=True, graphed_src_views=0, views_per_replay=2)
