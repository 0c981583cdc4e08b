"""View batching on the scene path: the 49-view DTU-shape scene of bench.py's `scene49` leg (camera arc, 4 source views
for depth and 10 for fusion, thresholds 2.0 / 6.0 / 2 / 0.3, feature cache + CUDA graphs, block sharding) with
K = views_per_replay reference views per replay of the cascade graph.  Every arm is captured up front; the rounds
alternate the arms in one process, after one untimed pass per arm, and the median of the rounds is reported.

Per arm: depth-phase ms per view (CUDA events around run_scene's depth maps), scene seconds (wall clock around run_scene
to a device synchronise), depth maps per second including fusion, host time per view spent enqueuing the depth phase
(inside infer.batch), and the peak of torch.cuda.max_memory_allocated over the arm's rounds.  The card's name, power
limit and max SM clock are read in the same run.

    python tools/scene_batch_bench.py [--ks 1,2,4,8] [--rounds 5] [--precision bf16x3] [--forced-conv2d-arm]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import effimvs_b200  # noqa: E402,F401
from effimvs_b200 import hotpath, scene, synthetic  # noqa: E402


def parse(argv=None):
    ap = argparse.ArgumentParser(description=__doc__.split("\n\n")[0])
    ap.add_argument("--views", type=int, default=49)
    ap.add_argument("--shape", default="dtu", choices=sorted(synthetic.SHAPES))
    ap.add_argument("--ks", default="1,2,4,8", help="comma-separated views per replay")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--precision", default="bf16x3", choices=["f32", "bf16", "bf16x3"])
    ap.add_argument("--forced-conv2d-arm", action="store_true",
                    help="one more arm at the largest K captured with EFFIMVS_CONV2D=1 (the 1/8 stage's update block on the "
                         "tensor-core kernel instead of cuDNN); information only")
    ap.add_argument("--out", help="also write the JSON result to this file")
    a = ap.parse_args(argv)
    a.ks = [int(k) for k in a.ks.split(",")]
    if a.rounds < 1 or a.views < 3 or any(k < 1 for k in a.ks):
        ap.error("need --rounds >= 1, --views >= 3 and every K >= 1")
    return a


def build_scene(n, shape, dev):
    """bench.py scene_leg's inputs: (imgs, cams, depth values, pairs for depth, pairs for fusion)"""
    cfg = synthetic.SHAPES[shape]
    W, H = cfg["width"], cfg["height"]
    g = torch.Generator().manual_seed(0)
    imgs = torch.rand(n, 3, H, W, generator=g).to(dev)
    E, K = synthetic.camera_arc(n, W, H)
    cams = {k: v[0].to(dev) for k, v in synthetic.stage_cameras(E, K, 1).items()}
    dv = torch.linspace(1 / 935.0, 1 / 425.0, 384, device=dev)
    nb = lambda i, m: [j for d in range(1, m // 2 + 1) for j in ((i - d) % n, (i + d) % n)]      # noqa: E731
    return imgs, cams, dv, [nb(i, 4) for i in range(n)], [nb(i, min(10, (n - 1) // 2 * 2)) for i in range(n)]


def card():
    """name, power limit and max SM clock of the GPU, as nvidia-smi reports them"""
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60).stdout.strip()
        name, power, clock = (x.strip() for x in q.split(","))
        return {"name": name, "power_limit": power, "max_sm_clock": clock}
    except (OSError, ValueError, subprocess.SubprocessError) as e:
        return {"name": torch.cuda.get_device_name(0), "power_limit": "unknown ({})".format(e), "max_sm_clock": "unknown"}


def main(argv=None):
    a = parse(argv)
    assert torch.cuda.is_available(), "scene_batch_bench.py measures on a CUDA device; there is no CPU path"
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    torch.backends.cudnn.benchmark = True
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from util import dtu_model
    model = dtu_model(hotpath.CudaHotPath(a.precision, native_projection=True), dev, synthetic.SHAPES[a.shape]["ndepths"])
    for m in model.modules():
        if isinstance(m, torch.nn.Conv2d):
            m.weight.data = m.weight.data.contiguous(memory_format=torch.channels_last)
    N = a.views
    imgs, cams, dv, pairs, fpairs = build_scene(N, a.shape, dev)
    arms = [("K={}".format(k), k, None) for k in a.ks]
    if a.forced_conv2d_arm:
        arms.append(("K={} EFFIMVS_CONV2D=1".format(max(a.ks)), max(a.ks), "1"))
    made = {}
    for name, k, conv2d in arms:
        saved = os.environ.get("EFFIMVS_CONV2D")
        if conv2d is not None:
            os.environ["EFFIMVS_CONV2D"] = conv2d       # read while the graphs are captured
        try:
            before = torch.cuda.memory_allocated()
            infer, fuse = scene.cuda_scene_callables(model, imgs, cams, dv, 2.0, 6.0, 2, 0.3, feature_cache=True,
                                                     graphed_src_views=4, views_per_replay=k)
            torch.cuda.synchronize()
            made[name] = (infer, fuse, k, (torch.cuda.memory_allocated() - before) / 1e9)
        finally:
            if conv2d is not None:
                if saved is None:
                    os.environ.pop("EFFIMVS_CONV2D", None)
                else:
                    os.environ["EFFIMVS_CONV2D"] = saved
    host = {"s": 0.0}

    def one_pass(name):
        infer, fuse, k, _ = made[name]
        batch = infer.batch

        def timed_batch(items):
            t = time.perf_counter()
            r = batch(items)
            host["s"] += time.perf_counter() - t
            return r
        infer.batch = timed_batch
        try:
            infer.clear_cache()                         # every pass encodes its images again
            torch.cuda.synchronize()
            host["s"] = 0.0
            torch.cuda.reset_peak_memory_stats()
            tm = {}
            t0 = time.perf_counter()
            out = scene.run_scene(infer, fuse, N, pairs, 0, 1, dev, fuse_pairs=fpairs, timings=tm, sharding="block")
            torch.cuda.synchronize()
            secs = time.perf_counter() - t0
        finally:
            infer.batch = batch
        return {"seconds": secs, "depth_ms_per_view": tm["depth_maps_ms"] / N, "host_ms_per_view": host["s"] * 1e3 / N,
                "fusion_ms": tm["fusion_ms"], "max_memory_allocated_GB": torch.cuda.max_memory_allocated() / 1e9,
                "fused_points": int(sum(v[0].shape[0] for v in out.values()))}

    for name, _, _ in arms:                             # untimed pass per arm: allocator pools, autotuned algorithms
        one_pass(name)
    rounds = {name: [] for name, _, _ in arms}
    for r in range(a.rounds):
        order = arms if r % 2 == 0 else arms[::-1]
        for name, _, _ in order:
            rounds[name].append(one_pass(name))
    med = lambda xs: statistics.median(xs)              # noqa: E731
    res = {}
    for name, k, _ in arms:
        rs = rounds[name]
        secs = med([x["seconds"] for x in rs])
        res[name] = {"views_per_replay": k, "seconds": secs, "seconds_min": min(x["seconds"] for x in rs),
                     "seconds_max": max(x["seconds"] for x in rs), "depth_maps_per_sec_incl_fusion": N / secs,
                     "depth_ms_per_view": med([x["depth_ms_per_view"] for x in rs]),
                     "host_ms_per_view": med([x["host_ms_per_view"] for x in rs]),
                     "fusion_ms": med([x["fusion_ms"] for x in rs]),
                     "max_memory_allocated_GB": max(x["max_memory_allocated_GB"] for x in rs),
                     "arm_resident_GB": made[name][3], "fused_points": rs[-1]["fused_points"]}
    cfg = synthetic.SHAPES[a.shape]
    line = {"tool": "scene_batch_bench", "card": card(), "views": N, "shape": [cfg["width"], cfg["height"]],
            "precision": a.precision, "rounds": a.rounds, "arms": res,
            "note": "median over rounds (arms alternated, one untimed pass each); max_memory_allocated is process-wide "
                    "(every arm's cache and graphs are resident), arm_resident_GB what capturing the arm allocated"}
    print(json.dumps(line), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(line, f, indent=1)


if __name__ == "__main__":
    main()
