"""Timing of the update block's fp32-grade (bf16x3) tensor-core convolutions on a B200 (csrc/conv2d_tc.cu).

Per layer: the block's six 3x3 convolutions (cd2, dprime, zr, q, head1 -- one GRU iteration -- and mask[0]) at the DTU
stage-3 (800x592, hidden 16) and stage-2 (400x296, hidden 32) shapes, in four variants: the fp16 kernel, the bf16x3 kernel,
cuDNN fp32 (TF32 off) and cuDNN TF32.  The cuDNN variants time the convolution with its bias only (the block runs the gate
arithmetic after it in separate kernels); the own kernels include their fused epilogue.  CUDA events around each of 11
launches with three L2 flushes queued ahead of the bracket (as bench.py's kernel legs), median after a dropped cold launch.
Printed: ms, GB/s of 4 HW (cin + cout) bytes and TFLOP/s of 18 HW cin cout.

Whole forward: 1600x1184x5 with TF32 off, graph-replayed, net.EffiMVSPlus (channels-last conv weights, as in bench.py) with
CudaHotPath("bf16x3", native_projection=True)
without (the update block on cuDNN fp32) and with conv2d_precision="bf16x3", arms alternated in one process; the default
TF32 configuration (the fp16 kernel) beside them.

    python tools/conv2d_bf16x3_bench.py --out DIR [--rounds 5 --steps 20]
"""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

import effimvs_b200  # noqa: E402,F401
from effimvs_b200 import capi, hotpath, ops, synthetic  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return {"torch_name": torch.cuda.get_device_name(), "nvidia_smi": q.stdout.strip()}


def timer(reps=11):
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")

    def timed(fn):
        ts = []
        for _ in range(reps + 1):
            flush.zero_()
            flush.zero_()
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        ts = sorted(ts[1:])
        return ts[len(ts) // 2]
    return timed


def layers(h):
    """(name, cin, cout, mode, two input segments) of the block's six 3x3 convolutions at hidden size h"""
    return [("cd2", 2 * h, 2 * h, capi.CONV2D_BIAS_RELU, False), ("dprime", 2 * h, h, capi.CONV2D_ADD_RELU, False),
            ("zr", 2 * h, 2 * h, capi.CONV2D_GRU_GATES, False), ("q", 2 * h, h, capi.CONV2D_GRU_UPDATE, True),
            ("head1", h, h, capi.CONV2D_BIAS_RELU, False), ("mask0", h, 2 * h, capi.CONV2D_BIAS_RELU, False)]


def per_layer(timed):
    res = []
    for tag, h, H, W in (("stage3", 16, 592, 800), ("stage2", 32, 296, 400)):
        mk = lambda c: torch.randn(1, c, H, W, device="cuda").contiguous(memory_format=torch.channels_last)   # noqa: E731
        for name, cin, cout, mode, two in layers(h):
            x = mk(cin)
            w, b = 0.1 * torch.randn(cout, cin, 3, 3, device="cuda"), torch.randn(cout, device="cuda")
            hh = cout // 2 if mode == capi.CONV2D_GRU_GATES else cout
            out, aux0, aux1 = mk(hh), mk(hh), mk(hh)
            if mode == capi.CONV2D_GRU_UPDATE:
                aux0 = torch.rand_like(aux0)
            in0, in1 = (x[:, :cin // 2], x[:, cin // 2:]) if two else (x, None)
            row = {"stage": tag, "layer": name, "cin": cin, "cout": cout, "H": H, "W": W}
            for prec in ("f16", "bf16x3"):
                pk = ops.conv2d_tc_pack(w, prec)
                a0 = aux0 if mode >= capi.CONV2D_ADD_RELU else None
                a1 = aux1 if mode == capi.CONV2D_GRU_GATES else None
                bias = None if mode == capi.CONV2D_ADD_RELU else b
                row[prec] = timed(lambda: ops.conv2d_tc(in0, in1, pk, bias, cout, mode, out, a0, a1, prec))
            wcl = w.contiguous(memory_format=torch.channels_last)       # as the model holds its conv weights
            for key, tf32 in (("cudnn_fp32", False), ("cudnn_tf32", True)):
                torch.backends.cudnn.allow_tf32 = tf32
                F.conv2d(x, wcl, b, padding=1)
                row[key] = timed(lambda: F.conv2d(x, wcl, b, padding=1))
            torch.backends.cudnn.allow_tf32 = False
            by, fl = 4.0 * H * W * (cin + cout), 18.0 * H * W * cin * cout
            for k in ("f16", "bf16x3", "cudnn_fp32", "cudnn_tf32"):
                row[k] = {"ms": row[k], "gbs": by / row[k] / 1e6, "tflops": fl / row[k] / 1e9}
            res.append(row)
            print("{:6s} {:6s} {:3d}->{:3d}  ".format(tag, name, cin, cout) + "  ".join(
                "{} {:.4f} ms {:6.0f} GB/s {:5.1f} TF/s".format(k, row[k]["ms"], row[k]["gbs"], row[k]["tflops"])
                for k in ("f16", "bf16x3", "cudnn_fp32", "cudnn_tf32")), flush=True)
    return res


def whole_forward(rounds, steps):
    from util import dtu_model
    s = synthetic.make_sample("dtu", seed=0, device="cuda")
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    arms = {"fp32_update_cudnn": (False, {}), "fp32_update_bf16x3": (False, {"conv2d_precision": "bf16x3"}),
            "tf32_default": (True, {})}
    graphs = {}
    for name, (tf32, kw) in arms.items():
        torch.backends.cudnn.allow_tf32 = tf32
        model = dtu_model(hotpath.CudaHotPath("bf16x3", native_projection=True, **kw), "cuda", "48,8,8")
        for m in model.modules():       # 4-D conv weights channels-last, as bench.py sets the model up
            if isinstance(m, torch.nn.Conv2d):
                m.weight.data = m.weight.data.contiguous(memory_format=torch.channels_last)
        fwd = lambda m=model: m(s["imgs"], s["proj_matrices"], s["depth_values"])   # noqa: E731
        for _ in range(2):
            fwd()
        side = torch.cuda.Stream()
        side.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(side):
            fwd()
        torch.cuda.current_stream().wait_stream(side)
        g = torch.cuda.CUDAGraph()
        with torch.cuda.graph(g):
            out = fwd()
        graphs[name] = (g, model, out)
    torch.backends.cudnn.allow_tf32 = False
    times = {k: [] for k in arms}
    for _ in range(rounds):
        for name, (g, _, _) in graphs.items():           # arms alternate round by round
            for _ in range(3):
                g.replay()
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                flush.zero_()
                g.replay()
            e1.record()
            torch.cuda.synchronize()
            times[name].append(e0.elapsed_time(e1) / steps)
    a, b = graphs["fp32_update_cudnn"][2]["depth"], graphs["fp32_update_bf16x3"][2]["depth"]
    agree = min(float(((x - y).abs() <= 0.51).float().mean()) for x, y in zip(a, b))
    res = {k: {"ms_per_depth_map_median": sorted(v)[len(v) // 2], "rounds": v} for k, v in times.items()}
    res["fraction_within_0.51mm_bf16x3_vs_cudnn_fp32_worst_output"] = agree
    for k, v in times.items():
        print("whole forward 1600x1184x5 {:20s}: {:.3f} ms per depth map (median of {} rounds of {} graph replays, "
              "256 MiB L2 flush before each)".format(k, sorted(v)[len(v) // 2], rounds, steps), flush=True)
    print("bf16x3 vs cuDNN fp32 update block: worst fraction of pixels within 0.51 mm {:.5f}".format(agree))
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", required=True, help="directory for conv2d_bf16x3_bench.json")
    ap.add_argument("--rounds", type=int, default=5)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--skip-forward", action="store_true")
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("conv2d_bf16x3_bench needs a CUDA device")
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.set_grad_enabled(False)
    info = card()
    print("GPU: {} | nvidia-smi name, power limit, max SM clock: {}".format(info["torch_name"], info["nvidia_smi"]), flush=True)
    res = {"card": info, "per_layer": per_layer(timer())}
    if not a.skip_forward:
        res["whole_forward"] = whole_forward(a.rounds, a.steps)
    os.makedirs(a.out, exist_ok=True)
    with open(os.path.join(a.out, "conv2d_bf16x3_bench.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
