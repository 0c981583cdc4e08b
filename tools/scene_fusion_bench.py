"""Fusion of a whole scene, per-view loop against one batched launch, for either filter of the scene runner:
  --filter dtu      the per-view loop of fusion.dtu_filter_view (what a DTU user of run_scene wrote by hand) against
                    cuda_dtu_fuse's batched call (fusion.dtu_filter_views);
  --filter dynamic  the per-view `fuse` of cuda_scene_callables (fusion.filter_view), driven the way run_scene drove it
                    before that fuse had a `batch` method, against its fuse.batch (fusion.filter_views).
The batched calls filter all of a rank's views in one launch, depth maps read in place from the all-gathered tensor.

The scene is bench.py's `scene49` leg at the DTU shape: a 49-view camera arc, 10 fusion source views per view, one
rank.  Its depth maps are the rendered surface of synthetic.render_plane_scene (noise 0.05 mm) and its confidence maps
are uniform in [0.4, 1) at half resolution (resized inside the filter), so that the filter keeps most pixels.  The
dynamic filter runs with bench.py's parameters (dist_base 2.0, rel_diff_base 6.0, thres_view 2, prob_threshold 0.3).  The
depth phase is not timed here: infer returns the rendered maps.

Two timings per arm, CUDA events:
  fusion_ms  run_scene's own `fusion_ms` (the filter plus the per-view point extraction, which both arms share),
             with the wall clock of run_scene to a device synchronise as `scene_ms`;
  filter_ms  the filter alone over all 49 views (the per-view loop, or one fuse.batch), with the host time
             spent in those calls as `filter_host_ms`.
The rounds alternate the arms in one process after one untimed pass per arm; medians are reported.  Both arms' points
must be bit-identical.  The card's name, power limit and max SM clock are read in the same run.

    python tools/scene_fusion_bench.py [--filter dtu|dynamic] [--views 49] [--sources 10] [--rounds 7] [--out FILE]
"""
import argparse
import json
import os
import statistics
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

import torch  # noqa: E402

import effimvs_b200  # noqa: E402,F401
from effimvs_b200 import fusion, scene, synthetic  # noqa: E402


def parse(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--filter", default="dtu", choices=["dtu", "dynamic"])
    ap.add_argument("--views", type=int, default=49)
    ap.add_argument("--shape", default="dtu", choices=sorted(synthetic.SHAPES))
    ap.add_argument("--sources", type=int, default=10, help="fusion source views per reference view (even; at most 30, "
                                                             "16 for the dynamic filter)")
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--out", help="also write the JSON result to this file")
    a = ap.parse_args(argv)
    top = 30 if a.filter == "dtu" else 16
    if a.rounds < 1 or a.sources < 2 or a.sources % 2 or a.sources > top or a.views < a.sources + 1:
        ap.error("need --rounds >= 1, an even --sources in [2, {}] and --views > --sources".format(top))
    return a


def build_scene(n, n_src, W, H, dev):
    """depth stack (n,H,W), confidences (n,H/2,W/2), stage-4 cameras (n,2,4,4) on the device; source lists"""
    E, K = synthetic.camera_arc(n, W, H)
    depths = synthetic.render_plane_scene(E, K, W, H, noise=0.05, seed=0).to(dev)
    confs = (0.4 + 0.6 * torch.rand(n, H // 2, W // 2, generator=torch.Generator().manual_seed(1))).to(dev)
    cams = synthetic.stage_cameras(E, K, 1)["stage4"][0].to(dev)
    pairs = [[j for d in range(1, n_src // 2 + 1) for j in ((i - d) % n, (i + d) % n)] for i in range(n)]
    return depths, confs, cams, pairs


def per_view_fuse(cams):
    """the hand-written fuse of a DTU user before cuda_dtu_fuse: dtu_filter_view per reference view"""
    c = cams.cpu()
    K, E = c[:, 1, :3, :3].numpy(), c[:, 0].numpy()

    def fuse(i, ref_depth, conf, srcs, src_depths):
        h, w = ref_depth.shape[-2:]
        r = fusion.dtu_filter_view(ref_depth.reshape(h, w), conf[0], src_depths.reshape(-1, h, w), K[i], E[i],
                                   [K[j] for j in srcs], [E[j] for j in srcs], 0.5)
        return {"final": r["final"][None, None], "points": r["points"][None]}
    return fuse, K, E


def dynamic_arms(cams, dev):
    """cuda_scene_callables' fuse with bench.py's parameters: its per-view call, hidden from run_scene's batch protocol
    (the path run_scene took before), and the fuse itself, whose `batch` run_scene now calls"""
    _, fuse = scene.cuda_scene_callables(None, torch.zeros(1, 3, 8, 8, device=dev), {"stage4": cams}, torch.zeros(4, device=dev),
                                         2.0, 6.0, 2, 0.3)

    def per_view(*args):
        return fuse(*args)
    return {"per_view_loop": per_view, "batched": fuse}


def main(argv=None):
    a = parse(argv)
    assert torch.cuda.is_available(), "scene_fusion_bench.py measures on a CUDA device; there is no CPU path"
    from scene_batch_bench import card
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    cfg = synthetic.SHAPES[a.shape]
    W, H, N = cfg["width"], cfg["height"], a.views
    t = time.perf_counter()
    depths, confs, cams, pairs = build_scene(N, a.sources, W, H, dev)
    render_s = time.perf_counter() - t
    if a.filter == "dtu":
        arms = {"per_view_loop": per_view_fuse(cams)[0], "batched": scene.cuda_dtu_fuse(cams, pairs)}
    else:
        arms = dynamic_arms(cams, dev)
    views = list(range(N))

    def infer(i, srcs):
        return depths[i], confs[i]

    host = {"s": 0.0}

    def timed(fn):
        def call(*args):
            t = time.perf_counter()
            r = fn(*args)
            host["s"] += time.perf_counter() - t
            return r
        return call

    def filter_only(name):
        """the filter over every view, without run_scene's point extraction"""
        fuse = arms[name]
        ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
        torch.cuda.synchronize()
        host["s"] = 0.0
        ev[0].record()
        if name == "batched":
            timed(fuse.batch)(views, depths, confs, pairs)
        else:
            sel = torch.as_tensor([j for i in views for j in pairs[i]], device=dev)
            for i in views:
                src = sel[i * a.sources:(i + 1) * a.sources]
                timed(fuse)(i, depths[i].reshape(1, 1, H, W), confs[i:i + 1], pairs[i], depths.index_select(0, src)[None, :, None])
        ev[1].record()
        torch.cuda.synchronize()
        return {"filter_ms": ev[0].elapsed_time(ev[1]), "filter_host_ms": host["s"] * 1e3}

    def whole(name):
        fuse = arms[name]
        torch.cuda.synchronize()
        tm = {}
        t = time.perf_counter()
        out = scene.run_scene(infer, fuse, N, pairs, 0, 1, dev, timings=tm, sharding="block")
        torch.cuda.synchronize()
        return {"scene_ms": (time.perf_counter() - t) * 1e3, "fusion_ms": tm["fusion_ms"]}, out

    outs = {}
    for name in arms:                                   # untimed pass per arm: allocator pools, the table's device rows
        filter_only(name)
        _, outs[name] = whole(name)
    for i in views:                                     # both arms give the same points, bit for bit
        assert torch.equal(outs["batched"][i][0].view(torch.int32), outs["per_view_loop"][i][0].view(torch.int32)), i
    points = int(sum(v[0].shape[0] for v in outs["batched"].values()))
    del outs
    rounds = {name: [] for name in arms}
    for r in range(a.rounds):
        for name in (list(arms) if r % 2 == 0 else list(arms)[::-1]):
            res, _ = whole(name)
            res.update(filter_only(name))
            rounds[name].append(res)
    res = {}
    for name, rs in rounds.items():
        res[name] = {k: statistics.median(x[k] for x in rs) for k in rs[0]}
        res[name]["filter_ms_min"] = min(x["filter_ms"] for x in rs)
        res[name]["filter_ms_max"] = max(x["filter_ms"] for x in rs)
        res[name]["filter_ms_per_view"] = res[name]["filter_ms"] / N
    line = {"tool": "scene_fusion_bench", "filter": a.filter, "card": card(), "views": N, "shape": [W, H], "sources": a.sources,
            "rounds": a.rounds, "fused_points": points, "render_s": render_s, "arms": res,
            "note": "medians over rounds, arms alternated in one process after one untimed pass each; fusion_ms and "
                    "scene_ms include run_scene's per-view point extraction, filter_ms is the filter alone"}
    print(json.dumps(line), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(line, f, indent=1)


if __name__ == "__main__":
    main()
