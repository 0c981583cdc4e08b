"""Times the fused warp+correlation kernels at the DTU (or T&T) stage shapes in both feature layouts and
checks them against each other (the planar kernel is the one the parity tests pin to the oracle).

    python tools/warp_bench.py [dtu|tanks] [reps]
"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

import effimvs_b200  # noqa: E402,F401
from effimvs_b200 import capi, hotpath, ops, synthetic  # noqa: E402


def timed(fn, flush, reps):
    for _ in range(2):
        out = fn()
    ts = []
    for _ in range(reps):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = fn()
        e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ts.sort()
    return ts[len(ts) // 2], out


def main():
    shape = sys.argv[1] if len(sys.argv) > 1 else "dtu"
    reps = int(sys.argv[2]) if len(sys.argv) > 2 else 7
    only = [int(t) for t in sys.argv[3].split(",")] if len(sys.argv) > 3 else [1, 2, 3]
    dev = "cuda"
    torch.manual_seed(0)
    hp = hotpath.CudaHotPath("f32", native_projection=True)
    s = synthetic.make_sample(shape, seed=0, device=dev)
    V = s["imgs"].shape[1]
    Hf, Wf = s["imgs"].shape[-2:]
    D1 = 96 if shape == "tanks" else 48
    shapes = [(32, D1, Hf // 8, Wf // 8), (16, 8, Hf // 4, Wf // 4), (8, 8, Hf // 2, Wf // 2)]
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    rows = []
    for i, (C, D, H, W) in enumerate(shapes):
        if i + 1 not in only:
            continue
        feats = [torch.randn(1, C, H, W, device=dev) for _ in range(V)]
        feats_cl = [f.contiguous(memory_format=torch.channels_last) for f in feats]
        proj = hp.relative_projection(s["proj_matrices"]["stage{}".format(i + 1)])
        wts = torch.rand(1, V - 1, H, W, device=dev)
        if i == 0:
            planes = (1.0 / torch.linspace(1 / 935.0, 1 / 425.0, D, device=dev)).reshape(1, D)
            fn = lambda f: ops.warp_corr_views(f[0], f[1:], proj, planes, capi.HYP_PLANES, D)[0]   # noqa: E731
            by = 4.0 * (V * C * H * W + D + (V - 1) * D * H * W + (V - 1) * H * W)
        else:
            cur = 680.0 + 40 * torch.rand(1, 1, H, W, device=dev)
            iv = torch.full((1,), (1 / 425.0 - 1 / 935.0) / 384 * (2 if i == 1 else 1), device=dev)
            fn = lambda f: ops.warp_corr_agg(f[0], f[1:], proj, cur, capi.HYP_LOCAL, iv, wts, D, 1, True)[0]   # noqa: E731
            by = 4.0 * (V * C * H * W + H * W + (V - 1) * H * W + 2 * D * H * W)
        ms_p, out_p = timed(lambda: fn(feats), flush, reps)
        row = {"stage": i + 1, "C": C, "D": D, "H": H, "W": W, "planar_ms": ms_p, "planar_GBs": by / ms_p / 1e6}
        # channels-last maps: the staged tile kernel
        ms_c, out_c = timed(lambda: fn(feats_cl), flush, reps)
        row.update({"tile_ms": ms_c, "tile_GBs": by / ms_c / 1e6,
                    "tile_vs_planar_rel_diff": float((out_p - out_c).abs().max() / out_p.abs().max())})
        if i > 0:      # the same on a smooth surface (what a converged scene looks like)
            Es, Ks = synthetic.camera_ring(V, W, H)
            cur = synthetic.render_plane_scene(Es[:1], Ks, W, H, noise=0.0)[0].to(dev).reshape(1, 1, H, W)
            ms_s, _ = timed(lambda: fn(feats_cl), flush, reps)
            row.update({"tile_smooth_ms": ms_s, "tile_smooth_GBs": by / ms_s / 1e6})
        rows.append(row)
        print(json.dumps(row), flush=True)


if __name__ == "__main__":
    main()
