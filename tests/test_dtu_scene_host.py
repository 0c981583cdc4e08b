"""The DTU filter as a fusion mode of the scene runner, host side (CPU): the scene camera table against dtu_camera_pack
bit for bit, the rows handed to the batched kernel, the argument checks, and run_scene with a batched `fuse` built on the
NumPy oracle (oracle/dtu_filter.py) -- on one rank and on 2 gloo ranks it must equal the per-view run bit for bit.  The
kernel behind the same interface is covered by test_gpu_dtu_scene."""
import os
import socket

import numpy as np
import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

import effimvs_b200  # noqa: F401
from effimvs_b200 import fusion, scene, synthetic

N_VIEWS, H, W = 9, 48, 64


def _cameras(n):
    E, K = synthetic.camera_arc(n, W, H)
    return np.repeat(K.numpy().astype(np.float32)[None], n, 0), E.numpy().astype(np.float32)


RAGGED = [[1, 2, 3], [0], [4, 6, 0, 1, 5], [2, 4], [3, 5, 6, 0, 1, 2], [6], [5, 4, 3]]     # source lists of a 7-view scene


def test_table_rows_equal_the_single_view_pack():
    K, E = _cameras(7)
    K = K * (1 + 0.01 * np.arange(7, dtype=np.float32))[:, None, None]   # a different K per view
    K[:, 2, 2] = 1
    table = fusion.dtu_scene_cameras(K, E, RAGGED)
    assert table.n_views == 7 and table.vmax == 6
    assert table.mats.dtype == torch.float32 and table.mats.shape == (7, 34 + 50 * 6)
    for i, p in enumerate(RAGGED):
        want = fusion.dtu_camera_pack(K[i], E[i], [K[j] for j in p], [E[j] for j in p])
        row = table.mats[i]
        assert torch.equal(row[:want.numel()].view(torch.int32), want.view(torch.int32)), i     # bit for bit
        assert not row[want.numel():].any()                                                      # zero padding
        assert table.src[i, :len(p)].tolist() == p and not table.src[i, len(p):].any()
        assert int(table.count[i]) == len(p)


def test_table_from_torch_cameras_matches_numpy():
    K, E = _cameras(7)
    a = fusion.dtu_scene_cameras(K, E, RAGGED)
    b = fusion.dtu_scene_cameras(torch.from_numpy(K), torch.from_numpy(E).double(), RAGGED)
    assert torch.equal(a.mats.view(torch.int32), b.mats.view(torch.int32))


def test_rows_in_scene_order_and_in_a_stack_of_its_own():
    K, E = _cameras(7)
    table = fusion.dtu_scene_cameras(K, E, RAGGED)
    ref, src, count, mats = table.rows([4, 1, 2], "cpu")
    assert ref.dtype == src.dtype == count.dtype == torch.int32 and mats.dtype == torch.float32
    assert ref.tolist() == [4, 1, 2] and count.tolist() == [6, 1, 5]
    assert src.tolist() == [table.src[i].tolist() for i in (4, 1, 2)]
    assert torch.equal(mats.view(torch.int32), table.mats[[4, 1, 2]].view(torch.int32))
    assert table.rows([4, 1, 2], "cpu")[0] is ref                      # built once per list
    # view 2 with its own maps stacked as [ref, sources in order]
    rows = {2: 0, 4: 1, 6: 2, 0: 3, 1: 4, 5: 5}
    ref, src, count, mats = table.rows([2], "cpu", rows)
    assert ref.tolist() == [0] and src[0, :5].tolist() == [1, 2, 3, 4, 5] and count.tolist() == [5]
    assert torch.equal(mats.view(torch.int32), table.mats[2:3].view(torch.int32))


def test_rejected_arguments():
    K, E = _cameras(40)
    with pytest.raises(ValueError):
        fusion.dtu_scene_cameras(K, E, [[j for j in range(40) if j != i][:32] for i in range(40)])    # 32 sources
    fusion.dtu_scene_cameras(K, E, [[j for j in range(40) if j != i][:31] for i in range(40)])        # 31 is the limit
    with pytest.raises(ValueError):
        fusion.dtu_scene_cameras(K, E, [[1]] * 39 + [[]])                                             # no source
    with pytest.raises(ValueError):
        fusion.dtu_scene_cameras(K, E, [[1]] * 39 + [[40]])                                           # outside the scene
    with pytest.raises(ValueError):
        fusion.dtu_scene_cameras(K, E, [[1]] * 39 + [[-1]])
    with pytest.raises(ValueError):
        fusion.dtu_scene_cameras(K, E, [[1]] * 39)                                                    # a list per view
    with pytest.raises(ValueError):
        fusion.dtu_scene_cameras(K[:39], E, [[1]] * 40)                                               # K and E disagree
    K, E = _cameras(7)
    table = fusion.dtu_scene_cameras(K, E, RAGGED)
    stack, confs = torch.ones(7, H, W), torch.ones(2, H // 2, W // 2)
    with pytest.raises(ValueError):
        fusion.dtu_filter_views(stack, [0, 7], confs, table)                                          # view outside the scene
    with pytest.raises(ValueError):
        fusion.dtu_filter_views(stack, [0, -1], confs, table)
    with pytest.raises(ValueError):
        fusion.dtu_filter_views(stack[:6], [0, 1], confs, table)                                      # stack != scene
    with pytest.raises(ValueError):
        fusion.dtu_filter_views(stack, [0, 1, 2], confs, table)                                       # 2 maps for 3 views
    with pytest.raises(ValueError):
        fusion.dtu_filter_views(stack[0], [0, 1], confs, table)                                       # not (N,h,w)
    with pytest.raises(ValueError):
        fusion.dtu_filter_views(stack[:3], [0], confs[:1], table, stack_rows={0: 0, 1: 1, 2: 2})      # a source not stacked
    with pytest.raises(ValueError):
        fusion.dtu_filter_views(stack[:3], [0], confs[:1], table, stack_rows={0: 0, 1: 1, 2: 2, 3: 3})  # beyond the stack
    with pytest.raises(ValueError):
        fusion.dtu_filter_views(stack, [], confs[:0], table)
    cams = torch.zeros(7, 2, 4, 4)
    cams[:, 0], cams[:, 1, :3, :3] = torch.from_numpy(E), torch.from_numpy(K)
    fuse = scene.cuda_dtu_fuse(cams, RAGGED)
    with pytest.raises(ValueError):
        fuse(0, stack[:1], confs[:1], [1, 2], stack[1:3])                                             # not the scene's list
    with pytest.raises(ValueError):
        fuse.batch([0, 1], stack, confs, [[1, 2]] + RAGGED[1:])


def _inputs(n_views=N_VIEWS):
    """a camera arc over the rendered surface; 2 source views for depth, 4 to 6 for fusion (the filter wants several
    consistent views before it keeps a pixel)"""
    E, K = synthetic.camera_arc(n_views, W, H)
    depths = synthetic.render_plane_scene(E, K, W, H, noise=0.01, seed=1)
    K32, E32 = _cameras(n_views)
    nb = lambda i, m: [j for d in range(1, m // 2 + 1) for j in ((i - d) % n_views, (i + d) % n_views)]   # noqa: E731
    pairs = [nb(i, 2) for i in range(n_views)]
    fuse_pairs = [nb(i, 6)[:4 + i % 3] for i in range(n_views)]                                          # ragged
    conf = 0.4 + 0.6 * torch.rand(n_views, H // 2, W // 2, generator=torch.Generator().manual_seed(3))
    return depths, conf, K32, E32, pairs, fuse_pairs


def _oracle_fuse(K, E, batched):
    """a CPU `fuse` on the NumPy restatement of upstream's filter; with `batch` when batched"""
    from oracle import dtu_filter as odtu

    def one(i, ref, conf, srcs, src_depths):
        conf = torch.nn.functional.interpolate(conf.reshape(1, 1, *conf.shape[-2:]), size=(H, W), mode="bilinear",
                                               align_corners=False).reshape(H, W)
        r = odtu.filter_view(ref.reshape(H, W).numpy(), conf.numpy(), src_depths.reshape(-1, H, W).numpy(), K[i], E[i],
                             [K[j] for j in srcs], [E[j] for j in srcs], 0.5)
        return torch.from_numpy(r["final"]), torch.from_numpy(r["points"].astype(np.float32))

    def fuse(i, ref_depth, conf, srcs, src_depths):
        final, pts = one(i, ref_depth, conf, srcs, src_depths)
        return {"final": final[None, None], "points": pts[None]}
    if batched:
        def batch(views, all_depths, confs, fuse_pairs):
            got = [one(i, all_depths[i], confs[b], fuse_pairs[i], all_depths[list(fuse_pairs[i])]) for b, i in enumerate(views)]
            batch.calls.append(list(views))
            return {"final": torch.stack([f for f, _ in got])[:, None], "points": torch.stack([p for _, p in got])}
        batch.calls = []
        fuse.batch = batch
    return fuse


def _run(rank, world, sharding="round_robin", batched=False):
    depths, conf, K, E, pairs, fuse_pairs = _inputs()

    def infer(i, srcs):
        return depths[i], conf[i]
    fuse = _oracle_fuse(K, E, batched)
    out = scene.run_scene(infer, fuse, N_VIEWS, pairs, rank, world, device="cpu", fuse_pairs=fuse_pairs, sharding=sharding)
    return out, (fuse.batch.calls if batched else None)


def _equal(a, b):
    assert sorted(a) == sorted(b)
    for i in a:
        assert torch.equal(a[i][0], b[i][0]) and torch.equal(a[i][1], b[i][1]), i


def test_run_scene_with_a_batched_fuse_equals_per_view():
    single, _ = _run(0, 1)
    got, calls = _run(0, 1, batched=True)
    assert calls == [list(range(N_VIEWS))]                 # one call for all of the rank's views, in view order
    _equal(got, single)
    assert sum(v[0].shape[0] for v in single.values()) > 0.2 * N_VIEWS * H * W


def _worker(rank, world, port, out_dir, sharding):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        res, calls = _run(rank, world, sharding, batched=True)
        torch.save({"res": {i: (p, d) for i, (p, d) in res.items()}, "calls": calls}, os.path.join(out_dir, "rank{}.pt".format(rank)))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("sharding", ["round_robin", "block"])
def test_two_ranks_batched_fuse_equal_one_per_view(tmp_path, sharding):
    single, _ = _run(0, 1)
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        port = s.getsockname()[1]
    mp.spawn(_worker, args=(2, port, str(tmp_path), sharding), nprocs=2, join=True)
    merged = {}
    for r in range(2):
        part = torch.load(os.path.join(str(tmp_path), "rank{}.pt".format(r)))
        mine = scene.shard_views(N_VIEWS, r, 2, sharding)
        assert sorted(part["res"]) == mine and part["calls"] == [mine]
        merged.update(part["res"])
    _equal(merged, single)


def test_c_abi_rejects_bad_sizes():
    """effimvs_dtu_filter_views_f32 checks its sizes and ladder on the host, before any launch"""
    import ctypes
    from effimvs_b200 import capi
    lib, one = capi.lib, ctypes.c_void_p(16)
    td, tf = (ctypes.c_double * 2)(0.5, 1.0), (ctypes.c_float * 2)(0.1, 0.2)

    def call(n_depths=8, vmax=10, n=3, h=8, w=8, td=td, tf=tf, depths=one, geo=None):
        return lib.effimvs_dtu_filter_views_f32(depths, n_depths, one, one, one, vmax, one, one, td, tf, 2, 1, 11, 0.5, 0.75,
                                                n, h, w, one, geo, one, one, None)
    assert call(vmax=32) == capi.EINVAL and "vmax=32" in capi.last_error()        # beyond the kernel's histogram limit
    assert call(vmax=0) == capi.EINVAL
    assert call(n=0) == capi.EINVAL
    assert call(n_depths=0) == capi.EINVAL
    assert call(h=1) == capi.EINVAL
    assert call(h=65536, w=65536) == capi.EINVAL                                 # h * w beyond int
    assert call(depths=None) == capi.EINVAL and "null" in capi.last_error()
    down = (ctypes.c_double * 2)(1.0, 0.5)
    assert call(td=down) == capi.EUNSUPPORTED and "non-decreasing" in capi.last_error()
