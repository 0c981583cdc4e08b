"""The scene's point cloud, taken from the filters' dense outputs: run_scene's per-view boolean-index loop against
fusion.compact_points (csrc/points.cu: count, scan, gather -- three launches for all views), for either filter.

The scene is scene_fusion_bench's: bench.py's `scene49` leg at the DTU shape (49 views at 1600x1184 on a camera arc, 10
fusion source views per view, one rank), whose filters keep nearly every pixel.  The reference images are u8 / 255 from a
seeded generator.  Arms, all on the same filter output (fuse.batch over the 49 views, run once and untimed):
  index_loop       points[b][:, final[b]].t().contiguous() per view: run_scene's expression without images (one nonzero
                   and one host synchronisation per view)
  compact          compact_points without colours
  compact_colors   compact_points with colours
and run_scene itself, filter included: its `fusion_ms` and its wall clock to a device synchronise, without and with
images.  Each arm is timed with CUDA events from before its first launch to after its last, including its host
synchronisations.  The rounds alternate the arms in one process after one untimed pass each; medians over the rounds are
reported.  Every arm's points must be bit-identical to index_loop's, and run_scene's with images to those without.

Algorithmic bytes: the mask is read twice (2 B per pixel); each kept point reads 12 B of points and writes 12 B, and with
colours reads 12 B of image and writes 3 B more.  GB/s is those bytes over the arm's median time.  The card's name, power
limit and max SM clock are read in the same run.

    python tools/scene_points_bench.py [--filter dtu|dynamic|both] [--views 49] [--sources 10] [--rounds 7] [--out FILE]
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
    ap.add_argument("--filter", default="both", choices=["dtu", "dynamic", "both"])
    ap.add_argument("--views", type=int, default=49)
    ap.add_argument("--shape", default="dtu", choices=sorted(synthetic.SHAPES))
    ap.add_argument("--sources", type=int, default=10, help="fusion source views per reference view (even, at most 16)")
    ap.add_argument("--rounds", type=int, default=7)
    ap.add_argument("--out", help="also write the JSON result to this file")
    a = ap.parse_args(argv)
    if a.rounds < 1 or a.sources < 2 or a.sources % 2 or a.sources > 16 or a.views < a.sources + 1:
        ap.error("need --rounds >= 1, an even --sources in [2, 16] and --views > --sources")
    return a


def timed(fn):
    """fn() between two CUDA events, the host waiting for the second: (result, device ms, host ms)"""
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    torch.cuda.synchronize()
    t = time.perf_counter()
    ev[0].record()
    r = fn()
    ev[1].record()
    torch.cuda.synchronize()
    return r, ev[0].elapsed_time(ev[1]), (time.perf_counter() - t) * 1e3


def same_bits(a, b):
    return a.shape == b.shape and torch.equal(a.view(torch.int32), b.view(torch.int32))


def bench_filter(kind, depths, confs, cams, pairs, images, rounds):
    from scene_fusion_bench import dynamic_arms
    N, H, W = depths.shape
    views = list(range(N))
    fuse = scene.cuda_dtu_fuse(cams, pairs) if kind == "dtu" else dynamic_arms(cams, depths.device)["batched"]
    res = fuse.batch(views, depths, confs, pairs)
    final, points = res["final"], res["points"]

    def index_loop():
        return [points[b][:, final[b, 0]].t().contiguous() for b in views]

    def infer(i, srcs):
        return depths[i], confs[i]

    def run(imgs):
        tm = {}
        out = scene.run_scene(infer, fuse, N, pairs, 0, 1, depths.device, timings=tm, sharding="block", images=imgs)
        return out, tm["fusion_ms"]

    arms = {"index_loop": index_loop,
            "compact": lambda: fusion.compact_points(final, points, views),
            "compact_colors": lambda: fusion.compact_points(final, points, views, images),
            "run_scene": lambda: run(None),
            "run_scene_images": lambda: run(images)}
    want = index_loop()
    kept = sum(p.shape[0] for p in want)
    for name, fn in arms.items():                 # untimed pass per arm; every arm's points bit-identical to index_loop's
        r = fn()
        if name.startswith("compact"):
            pts, _, offs = r
            assert all(same_bits(pts[offs[b]:offs[b + 1]], want[b]) for b in views), name
        elif name.startswith("run_scene"):
            assert all(same_bits(r[0][i][0], want[i]) for i in views), name
        del r
    rows = {name: [] for name in arms}
    for k in range(rounds):
        for name in (list(arms) if k % 2 == 0 else list(arms)[::-1]):
            r, dev_ms, host_ms = timed(arms[name])
            row = {"ms": dev_ms, "wall_ms": host_ms}
            if name.startswith("run_scene"):
                row["fusion_ms"] = r[1]
            rows[name].append(row)
            del r
    pixels = N * H * W
    bytes_ = {"compact": 2 * pixels + 24 * kept, "compact_colors": 2 * pixels + 39 * kept}
    bytes_["index_loop"] = bytes_["compact"]
    out = {}
    for name, rs in rows.items():
        out[name] = {key: statistics.median(x[key] for x in rs) for key in rs[0]}
        out[name]["ms_min"], out[name]["ms_max"] = min(x["ms"] for x in rs), max(x["ms"] for x in rs)
        if name in bytes_:
            out[name]["algorithmic_GB"] = bytes_[name] / 1e9
            out[name]["GB_per_s"] = bytes_[name] / (out[name]["ms"] * 1e-3) / 1e9
    return {"filter": kind, "pixels": pixels, "kept_points": kept, "bit_identical": True, "arms": out}


def main(argv=None):
    a = parse(argv)
    assert torch.cuda.is_available(), "scene_points_bench.py measures on a CUDA device; there is no CPU path"
    from scene_batch_bench import card
    from scene_fusion_bench import build_scene
    dev = torch.device("cuda", 0)
    torch.cuda.set_device(dev)
    cfg = synthetic.SHAPES[a.shape]
    W, H, N = cfg["width"], cfg["height"], a.views
    depths, confs, cams, pairs = build_scene(N, a.sources, W, H, dev)
    u8 = torch.randint(0, 256, (N, 3, H, W), generator=torch.Generator().manual_seed(2), dtype=torch.uint8).to(dev)
    images = u8.float() / 255
    del u8
    kinds = ["dtu", "dynamic"] if a.filter == "both" else [a.filter]
    results = [bench_filter(k, depths, confs, cams, pairs, images, a.rounds) for k in kinds]
    line = {"tool": "scene_points_bench", "card": card(), "views": N, "shape": [W, H], "sources": a.sources, "rounds": a.rounds,
            "results": results,
            "note": "medians over rounds, arms alternated in one process after one untimed pass each; ms from CUDA events "
                    "around each arm including its host synchronisations; run_scene arms include the filter"}
    print(json.dumps(line), flush=True)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            json.dump(line, f, indent=1)


if __name__ == "__main__":
    main()
