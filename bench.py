#!/usr/bin/env python
"""bench.py -- depth maps/s of the Effi-MVS+ cascade at the DTU evaluation shape
(1600x1184, 1 reference + 4 source views, ndepths 48,8,8, 3 GRU iterations per stage) with the
cost-volume hot path on hand-written sm_100a kernels.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--precision f32|bf16] [--dump-outputs DIR]

One JSON line on stdout (rank 0).  A "step" is one depth map (one pass of the whole cascade over
one 5-view batch of synthetic images).  `value` = depth maps/s with the inputs resident in HBM;
`e2e` = the same through the public API with pinned-host inputs copied in and the depth map read
back every step; `roofline` = the fused warp+correlation kernel (stage 3, the largest launch)
against the measured HBM copy peak; `cpu_baseline` / `--impl reference` = the oracle port of the
upstream path on the host cores (upstream itself is Python and does not travel to the GPU box).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time
import types

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

METRIC = "depth_maps_per_sec_1600x1184_5view"
UNIT = "depth maps/s"
WORKLOAD = "configs[2]: DTU eval shape 1600x1184, 5 views, full cross-scale cascade with dynamic cost volume (ndepths 48,8,8; GRU 3,3,3)"
# non-default --shape runs are labelled as what they are (the driver's contract run uses the default DTU shape)
LABELS = {"dtu": (METRIC, WORKLOAD),
          "tanks": ("depth_maps_per_sec_1920x1056_7view",
                    "configs[3]: Tanks & Temples shape 1920x1056, 7 views, full cross-scale cascade (ndepths 96,8,8; GRU 3,3,3)"),
          "plumbing": ("depth_maps_per_sec_640x512_5view",
                       "configs[0]: plumbing shape 640x512, 5 views, full cross-scale cascade (ndepths 48,8,8; GRU 3,3,3)")}


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10,
                    help="timed steps; impl reference runs at most this many, stopping at --cpu-budget-s (the line reports the number run)")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--precision", default=os.environ.get("EFFIMVS_PRECISION", "bf16x3"), choices=["f32", "bf16", "bf16x3"])
    ap.add_argument("--shape", default="dtu", choices=["dtu", "tanks", "plumbing"])
    ap.add_argument("--no-graph", action="store_true", help="do not capture the forward in a CUDA graph")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-scene", action="store_true", help="skip the 49-view scene leg (configs[4])")
    ap.add_argument("--scene-views", type=int, default=49)
    ap.add_argument("--profile-one", action="store_true",
                    help="3 warm eager forwards, then ONE forward between cudaProfilerStart/Stop and exit (for ncu --profile-from-start off)")
    ap.add_argument("--cpu-budget-s", type=float, default=240.0)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last timed step returned (rank 0) as DIR/<name>.npy: "
                         "depth00 .. depth12 and photometric_confidence, float32, every pixel (about 20 MB at the DTU shape)")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    return a


def output_arrays(out):
    """name -> copy of each output of one forward, taken where the tensors live (on the device: no host copy yet)"""
    arrays = {"depth{:02d}".format(i): d.detach().clone() for i, d in enumerate(out["depth"])}
    arrays["photometric_confidence"] = out["photometric_confidence"].detach().clone()
    return arrays


def dump_outputs(out_dir, arrays):
    """output_arrays() as DIR/<name>.npy; the inputs are seeded, so two builds can be compared file by file"""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        t = t.cpu()
        np.save(os.path.join(out_dir, name + ".npy"), t.numpy() if t.dtype == torch.float64 else t.float().numpy())


def build_model(hotpath, device, ndepths):
    import effimvs_b200  # noqa: F401
    from effimvs_b200 import net
    args = types.SimpleNamespace(ndepths=ndepths, GRUiters="3,3,3", CostNum=3)
    torch.manual_seed(0)
    model = net.EffiMVSPlus(args, hotpath=hotpath)
    wfile = os.path.join(ROOT, "tests", "golden", "dtu_weights.pt")
    data = "synthetic images/cameras (seeded); random-init weights (seed 0)"
    if os.path.exists(wfile):
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        from util import load_dtu_weights
        load_dtu_weights(model)
        data = "synthetic images/cameras (seeded); weights = upstream model_dtu.ckpt values (tests/golden/dtu_weights.pt)"
    model = model.to(device).eval()
    if torch.device(device).type == "cuda":
        for m in model.modules():                               # 4-D conv weights NHWC: cuDNN tensor-core kernels without layout round trips
            if isinstance(m, torch.nn.Conv2d):
                m.weight.data = m.weight.data.contiguous(memory_format=torch.channels_last)
    return model, data


def reference_model(device, ndepths):
    """The reference arm's model: UNMODIFIED upstream (oracle/_ref byte copy, kind "reference") when it is staged,
    else the oracle port inside this repo's host cascade (kind "port").  -> (model, kind, description)"""
    from oracle import upstream
    wfile = os.path.join(ROOT, "tests", "golden", "dtu_weights.pt")
    if upstream.available():
        sd = torch.load(wfile, map_location="cpu") if os.path.exists(wfile) else None
        torch.manual_seed(0)
        with _silenced():
            model = upstream.build_model(sd, ndepths, device)
        return model, "reference", "unmodified upstream Effi_MVS_plus.forward (oracle/_ref byte copy), eager PyTorch"
    from oracle import hotpath as ohp
    model, _ = build_model(ohp.OracleHotPath(), device, ndepths)
    return model, "port", "oracle port of the hot path inside this repo's host cascade, eager PyTorch"


class _silenced:
    """upstream's constructor prints its configuration; keep it off the bench's stdout / stderr"""

    def __enter__(self):
        import contextlib
        import io
        self.cm = contextlib.redirect_stdout(io.StringIO())
        return self.cm.__enter__()

    def __exit__(self, *a):
        return self.cm.__exit__(*a)


def config_keys(a, views, ndepths):
    """the `config` object BOTH arms print, value for value (the driver compares them to tell that the two arms ran
    the same workload); what differs between the arms is stated per arm inside it, run facts go to `run`"""
    _, workload = LABELS[a.shape]
    return {"workload": workload, "shape": a.shape, "views": views, "ndepths": ndepths,
            "l2": "impl ours: 256 MiB memset between steps, inside the timed region; impl reference: CPU arm, inputs in host memory",
            "sharding": "impl ours: one reference view per rank per step, no collective; impl reference: ONE CPU process on the "
                        "box's host cores whatever --gpus says",
            "stock_pytorch": "FPN, ConvGRU convolutions: cuDNN, TF32 allowed (torch default, as upstream) in impl ours; "
                             "impl reference: unmodified upstream, eager PyTorch fp32 on the CPU"}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms during the timed region."""
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=lambda: self.lines.extend(self.proc.stdout), daemon=True)
            self.th.start()
        except OSError:
            self.proc = None
        return self

    def __exit__(self, *a):
        if self.proc:
            time.sleep(0.25)
            self.proc.terminate()
            self.th.join(timeout=2)

    def summary(self):
        sm, mx, reasons = [], 0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx = max(mx, float(f[1]))
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": sorted(reasons), "samples": len(sm)}


def peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return p["hbm_gbs"], p["bf16_tflops"], "measured (MEASURED_PEAKS.json)"
    except (OSError, KeyError, ValueError):
        return 6650.0, 1590.0, "fallback (B200_PROFILING.md)"


# ------------------------------------------------------------------------------------------------
def run_reference(a, rank, world):
    """The reference's own implementation of the path on the box's host cores: unmodified upstream from oracle/_ref
    (kind 'reference'; the oracle port, kind 'port', only if the byte copy is not staged); rank 0 only -- at N > 1
    this is still ONE CPU box, not N of them."""
    if rank != 0:
        return
    import effimvs_b200  # noqa: F401
    from effimvs_b200 import synthetic
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    ndepths = synthetic.SHAPES[a.shape]["ndepths"]
    model, kind, what = reference_model("cpu", ndepths)
    s = synthetic.make_sample(a.shape, seed=0)
    times = []
    t_begin = time.perf_counter()
    done_w = 0
    last = 0.0
    result = [None]

    def one():
        t0 = time.perf_counter()
        result[0] = model(s["imgs"], s["proj_matrices"], s["depth_values"])
        return time.perf_counter() - t0

    with torch.no_grad():
        for i in range(max(a.warmup, 1)):
            if i >= 1 and (time.perf_counter() - t_begin) + last > 0.3 * a.cpu_budget_s:
                break
            last = one()
            done_w += 1
        for i in range(a.steps):
            if i >= 1 and (time.perf_counter() - t_begin) + last > a.cpu_budget_s:
                break
            last = one()
            times.append(last)
    if a.dump_outputs:
        dump_outputs(a.dump_outputs, output_arrays(result[0]))
    done_k = len(times)
    total = sum(times)
    value = done_k / total
    sample = "{} of {} requested steps, each one full {} depth map on {} host threads ({} warm-up; {:.0f} s cap); {}".format(
        done_k, a.steps, a.shape, cores, done_w, a.cpu_budget_s, what)
    metric, _ = LABELS[a.shape]
    data = "synthetic images/cameras (seeded); weights = upstream model_dtu.ckpt values (tests/golden/dtu_weights.pt)"
    cfg = config_keys(a, int(s["imgs"].shape[1]), ndepths)
    line = {"impl": "reference", "metric": metric, "value": value, "unit": UNIT, "n_gpus": a.gpus, "steps": done_k,
            "warmup": done_w, "ms_per_step": 1e3 * total / done_k, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32", "data": data, "config": cfg,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0,
            "run": {"device": "cpu", "cores": cores, "processes": 1}}
    OUT.emit(json.dumps(line))


# ------------------------------------------------------------------------------------------------
class TimedHotPath:
    """Wraps a hot-path table and brackets every call with CUDA events on the current stream."""

    def __init__(self, inner):
        self.inner, self.records = inner, []

    def _wrap(self, name):
        fn = getattr(self.inner, name)

        def call(*args, **kw):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = fn(*args, **kw)
            e1.record()
            self.records.append((name, args, e0, e1))
            return out
        return call

    def __getattr__(self, name):
        if name in ("stage1", "local_volume", "volume_lookup", "cross_scale", "dynamic_cost"):
            return self._wrap(name)
        return getattr(self.inner, name)


def ncu_traffic(tag):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the kernel whose label contains `tag`,
    from the committed `ncu --set full` summaries (profiles/r1b_forward_kernels_ncu_full.json, else
    profiles/r1_warp_tile_ncu.json); None if absent."""
    try:    # latest capture first: the kernel inside the bench forward (profiles/r1b_forward_kernels_ncu_full.json)
        with open(os.path.join(ROOT, "profiles", "r1b_forward_kernels_ncu_full.json")) as f:
            want = {"stage3": "warp_corr_tile_kernel<8", "stage2": "warp_corr_tile_kernel<16"}.get(tag)
            for k in json.load(f)["launches"]:
                if want and want in k["kernel"]:
                    return (k["dram_read_MB"] + k["dram_write_MB"]) * 1e6
    except (OSError, KeyError, ValueError, TypeError):
        pass
    try:
        with open(os.path.join(ROOT, "profiles", "r1_warp_tile_ncu.json")) as f:
            for k in json.load(f):
                if tag in k["label"] and "warp_corr" in k["label"]:
                    def mb(v):
                        num, unit = v.split()[:2]
                        return float(num) * {"Mbyte": 1e6, "Gbyte": 1e9, "Kbyte": 1e3, "byte": 1.0}[unit]
                    return mb(k["dram__bytes_read.sum"]) + mb(k["dram__bytes_write.sum"])
    except (OSError, KeyError, ValueError):
        pass
    return None


def kernel_rooflines(hp, model, sample, hbm_peak, tf_peak, peak_src, reps=11):
    """Per-kernel device time of the hot-path launches at the bench shape, timed in isolation with
    CUDA events on the launching stream, an L2 flush (256 MiB memset) before every launch."""
    from effimvs_b200 import capi, ops
    dev = sample["imgs"].device
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    feats = model.encode(sample["imgs"])
    out = {}

    # stage-2 / stage-3 inputs (current depth, view weights) exactly as they occur in the bench forward
    class Recorder:
        def __init__(self, inner):
            self.inner, self.calls = inner, []

        def __getattr__(self, name):
            fn = getattr(self.inner, name)
            if name != "local_volume":
                return fn

            def call(cur_depth, features, cams, interval, view_weights, ndepth, G):
                self.calls.append((cur_depth.clone(), view_weights.clone()))
                return fn(cur_depth, features, cams, interval, view_weights, ndepth, G)
            return call

    rec = Recorder(hp)
    model.set_hotpath(rec)
    try:
        model(sample["imgs"], sample["proj_matrices"], sample["depth_values"])
    finally:
        model.set_hotpath(hp)

    def timed(fn):
        # the events bracket the launch on an otherwise idle stream, so the host must have the kernel enqueued before the device
        # reaches the first event: three L2 flushes (~0.25 ms of device work) are queued ahead of it -- with one, a slow host
        # (Python op dispatch longer than the flush) left an idle gap inside the bracket and one box reported every isolated kernel
        # ~20 % slower than the others.  Median of `reps` launches after a dropped cold one.
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

    B, V = sample["imgs"].shape[:2]
    # stage 1: per-view similarity + entropy kernel
    f = feats[0]
    C, H, W = f[0].shape[1:]
    D = model.ndepths[0]
    cams = sample["proj_matrices"]["stage1"]
    proj = hp.relative_projection(cams)
    planes = (1.0 / torch.linspace(1 / 935.0, 1 / 425.0, D, device=dev)).reshape(1, D).repeat(B, 1)
    ms = timed(lambda: ops.warp_corr_views(f[0], f[1:], proj, planes, capi.HYP_PLANES, D))
    by = 4.0 * (V * C * H * W + D + (V - 1) * D * H * W + (V - 1) * H * W)
    out["warp_corr_views_stage1"] = {"ms": ms, "bytes": by, "gbs": by / ms / 1e6,
                                     "feature_layout": "NHWC" if not f[0].is_contiguous() else "NCHW"}
    fp = [t.contiguous() for t in f]
    ms = timed(lambda: ops.warp_corr_views(fp[0], fp[1:], proj, planes, capi.HYP_PLANES, D))
    out["warp_corr_views_stage1_nchw"] = {"ms": ms, "bytes": by, "gbs": by / ms / 1e6, "feature_layout": "NCHW"}
    # stages 2, 3: fused warp + correlation + aggregation with in-kernel hypotheses
    for s in (1, 2):
        f = feats[s]
        C, H, W = f[0].shape[1:]
        D = model.ndepths[s]
        cams = sample["proj_matrices"]["stage{}".format(s + 1)]
        proj = hp.relative_projection(cams)
        cur, wts = rec.calls[s - 1]
        iv = torch.full((B,), (1 / 425.0 - 1 / 935.0) / 384 * model.RATIOS[s], device=dev)
        ms = timed(lambda: ops.warp_corr_agg(f[0], f[1:], proj, cur, capi.HYP_LOCAL, iv, wts, D, 1, True))
        by = 4.0 * (V * C * H * W + H * W + (V - 1) * H * W + D * H * W + D * H * W)
        out["warp_corr_agg_stage{}".format(s + 1)] = {"ms": ms, "bytes": by, "gbs": by / ms / 1e6,
                                                      "feature_layout": "NHWC" if not f[0].is_contiguous() else "NCHW",
                                                      "inputs": "current depth and view weights recorded from the bench forward"}
        # the same launch on the depth of a smooth rendered surface (what a converged scene looks like: neighbouring
        # lanes sample neighbouring source pixels, no shared-memory bank-conflict replays)
        from effimvs_b200 import synthetic as _syn
        Es, Ks = _syn.camera_ring(V, W, H)
        smooth = _syn.render_plane_scene(Es[:1], Ks, W, H, noise=0.0)[0].to(dev).reshape(1, 1, H, W).repeat(B, 1, 1, 1)
        ms = timed(lambda: ops.warp_corr_agg(f[0], f[1:], proj, smooth, capi.HYP_LOCAL, iv, wts, D, 1, True))
        out["warp_corr_agg_stage{}_smooth_depth".format(s + 1)] = {"ms": ms, "bytes": by, "gbs": by / ms / 1e6,
                                                                   "inputs": "current depth = rendered smooth surface (synthetic.render_plane_scene)"}
        noise = torch.full((B, 1, H, W), 680.0, device=dev) + 40 * torch.rand(B, 1, H, W, device=dev)
        ms = timed(lambda: ops.warp_corr_agg(f[0], f[1:], proj, noise, capi.HYP_LOCAL, iv, wts, D, 1, True))
        out["warp_corr_agg_stage{}_noise_depth".format(s + 1)] = {"ms": ms, "bytes": by, "gbs": by / ms / 1e6,
                                                                  "inputs": "current depth = 680 + 40 * U(0,1) white noise (worst case for the gather)"}
        fp = [t.contiguous() for t in f]
        ms = timed(lambda: ops.warp_corr_agg(fp[0], fp[1:], proj, cur, capi.HYP_LOCAL, iv, wts, D, 1, True))
        out["warp_corr_agg_stage{}_nchw".format(s + 1)] = {"ms": ms, "bytes": by, "gbs": by / ms / 1e6, "feature_layout": "NCHW"}
    # regularization nets
    Hs, Ws = feats[0][0].shape[2:]
    x = torch.randn(B, 1, model.ndepths[0], Hs, Ws, device=dev)
    ms = timed(lambda: hp.cost_regularization(model.cost_regularization, x))
    vox = model.ndepths[0] * Hs * Ws
    fl = 2.0 * 27 * vox * (1 * 8 + 8 * 8 + 8 * 16 / 8 + 16 * 16 / 8 + 16 * 32 / 64 + 32 * 32 / 64 + 32 * 16 / 64 + 16 * 8 / 8 + 8)
    out["costreg_fpn3d"] = {"ms": ms, "flops": fl, "tflops": fl / ms / 1e9}
    for s in (1, 2):
        Hs, Ws = feats[s][0].shape[2:]
        D = model.ndepths[s]
        x = torch.randn(B, 1, D, Hs, Ws, device=dev)
        prev = torch.randn(B, 1, D, Hs // 2, Ws // 2, device=dev)
        ms = timed(lambda: hp.cross_scale(model.CSP_R[s - 1], x, prev))
        vq = D * (Hs // 2) * (Ws // 2)
        fl = 2.0 * 27 * vq * (8 + 8 + 16 * 8 + 8)
        out["cost_up_small_stage{}".format(s + 1)] = {"ms": ms, "flops": fl, "tflops": fl / ms / 1e9}
    # the update block's 3x3 convolutions on the tensor cores (csrc/conv2d_tc.cu) at the stage-3 / stage-2 shapes of this cascade:
    # algorithmic bytes = the fp32 input and output maps once each (+ the aux maps of the fused epilogues)
    for s, tag in ((2, "stage3"), (1, "stage2")):
        Hs, Ws = feats[s][0].shape[2:]
        h = model.HIDDEN[s]
        mk = lambda c: torch.randn(B, c, Hs, Ws, device=dev).contiguous(memory_format=torch.channels_last)   # noqa: E731
        hx, z, rh, cd = mk(2 * h), mk(h), mk(h), mk(2 * h)
        w_full, w_half = 0.1 * torch.randn(2 * h, 2 * h, 3, 3, device=dev), 0.1 * torch.randn(h, 2 * h, 3, 3, device=dev)
        bias2, bias1 = torch.randn(2 * h, device=dev), torch.randn(h, device=dev)
        if not (ops.conv2d_tc_supported(2 * h, 2 * h) and ops.conv2d_tc_supported(2 * h, h)):
            continue
        pk_full, pk_half = ops.conv2d_tc_pack(w_full), ops.conv2d_tc_pack(w_half)
        px = 4.0 * B * Hs * Ws
        ms = timed(lambda: ops.conv2d_tc(hx, None, pk_full, bias2, 2 * h, capi.CONV2D_BIAS_RELU, cd, None, None))
        out["conv2d_tc_{}_relu_{}to{}".format(tag, 2 * h, 2 * h)] = {"ms": ms, "bytes": px * 4 * h, "gbs": px * 4 * h / ms / 1e6,
                                                                     "flops": 18.0 * B * Hs * Ws * 4 * h * h, "tflops": 18.0 * B * Hs * Ws * 4 * h * h / ms / 1e9}
        ms = timed(lambda: ops.conv2d_tc(hx, None, pk_full, bias2, 2 * h, capi.CONV2D_GRU_GATES, rh, hx[:, :h], z))
        out["conv2d_tc_{}_gru_gates_{}to{}".format(tag, 2 * h, 2 * h)] = {"ms": ms, "bytes": px * 5 * h, "gbs": px * 5 * h / ms / 1e6}
        ms = timed(lambda: ops.conv2d_tc(rh, hx[:, h:], pk_half, bias1, h, capi.CONV2D_GRU_UPDATE, hx[:, :h], z, None))
        out["conv2d_tc_{}_gru_update_{}to{}".format(tag, 2 * h, h)] = {"ms": ms, "bytes": px * 5 * h, "gbs": px * 5 * h / ms / 1e6}
    dom = out["warp_corr_agg_stage3"]
    roof = {"kernel": "warp_corr_tile_kernel<8,1> (stage 3, 800x592, D=8, 4 source views)", "bound": "hbm",
            "achieved": dom["gbs"], "peak": hbm_peak, "unit": "GB/s", "frac": dom["gbs"] / hbm_peak, "traffic": ncu_traffic("stage3"),
            "peak_source": peak_src, "algorithmic_bytes": dom["bytes"], "ms": dom["ms"]}
    reg_ms = out["costreg_fpn3d"]["ms"] + 2 * out["cost_up_small_stage2"]["ms"] + 2 * out["cost_up_small_stage3"]["ms"]
    reg_fl = out["costreg_fpn3d"]["flops"] + 2 * out["cost_up_small_stage2"]["flops"] + 2 * out["cost_up_small_stage3"]["flops"]
    roof_reg = {"kernel": "3-D regularization (costreg_fpn3d + 4x cost_up_small)", "bound": "tensor", "achieved": reg_fl / reg_ms / 1e9,
                "peak": tf_peak, "unit": "TFLOP/s", "frac": reg_fl / reg_ms / 1e9 / tf_peak, "flops": reg_fl, "ms": reg_ms}
    c2 = out.get("conv2d_tc_stage3_relu_32to32")
    if c2:
        out["roofline_update_block"] = {"kernel": "conv2d_tc_kernel (stage 3, 800x592, 32 -> 32 + bias + relu)", "bound": "hbm", "achieved": c2["gbs"],
                                        "peak": hbm_peak, "unit": "GB/s", "frac": c2["gbs"] / hbm_peak, "algorithmic_bytes": c2["bytes"],
                                        "ms": c2["ms"], "tflops": c2["tflops"], "peak_source": peak_src}
    return roof, roof_reg, out


def scene_leg(a, model, rank, world, dev):
    """BASELINE.json configs[4]: depth maps for every view of a synthetic `--scene-views`-view scene at the DTU shape (4
    source views each), reference views sharded in balanced blocks over the ranks (every image encoded at most once per
    rank, encode / cascade replayed as CUDA graphs), ONE all-gather of the final depth maps (NCCL over NVLink at N > 1),
    then the geometric-consistency filter (10 source views) of the views each rank owns.  Returns the `scene49` object."""
    from effimvs_b200 import scene, synthetic
    N = a.scene_views
    cfg = synthetic.SHAPES["dtu"]
    W, H = cfg["width"], cfg["height"]
    g = torch.Generator().manual_seed(0)
    imgs = torch.rand(N, 3, H, W, generator=g).to(dev)
    E, K = synthetic.camera_arc(N, W, H)
    cams = {k: v[0].to(dev) for k, v in synthetic.stage_cameras(E, K, 1).items()}
    dv = torch.linspace(1 / 935.0, 1 / 425.0, 384, device=dev)
    nb = lambda i, n: [j for d in range(1, n // 2 + 1) for j in ((i - d) % N, (i + d) % N)]      # noqa: E731
    pairs, fpairs = [nb(i, 4) for i in range(N)], [nb(i, min(10, (N - 1) // 2 * 2)) for i in range(N)]
    infer, fuse = scene.cuda_scene_callables(model, imgs, cams, dv, 2.0, 6.0, 2, 0.3, feature_cache=True, graphed_src_views=4)
    for timed_pass in (False, True):        # one untimed pass over the scene (allocator pools, NCCL channels), then the timed one
        infer.clear_cache()                 # every pass encodes its images again
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        tm = {}
        t0 = time.perf_counter()
        out = scene.run_scene(infer, fuse, N, pairs, rank, world, dev, fuse_pairs=fpairs, timings=tm, sharding="block")
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
    stats = torch.tensor([time.perf_counter() - t0, tm.get("all_gather_ms", 0.0), tm.get("fusion_ms", 0.0), tm.get("depth_maps_ms", 0.0)],
                         device=dev)
    pts = torch.tensor([float(sum(v[0].shape[0] for v in out.values()))], device=dev)
    if world > 1:
        dist.all_reduce(stats, op=dist.ReduceOp.MAX)
        dist.all_reduce(pts)
    secs, ag_ms, fu_ms, dm_ms = (float(x) for x in stats)
    slots = scene.slots_per_rank(N, world)
    pure_ms = None
    if world > 1:       # the same collective once more with all ranks aligned: NVLink time without the wait for the slowest rank
        mine = torch.zeros(slots, H, W, device=dev)
        flat = torch.empty(world * slots, H, W, device=dev)
        dist.all_gather_into_tensor(flat, mine)
        torch.cuda.synchronize()
        dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        dist.all_gather_into_tensor(flat, mine)
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1)], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        pure_ms = float(t)
    recv = (world - 1) * slots * H * W * 4                      # bytes every rank receives from its peers
    return {"views": N, "shape": [W, H], "n_gpus": world, "seconds": secs, "depth_maps_per_sec_incl_fusion": N / secs,
            "all_gather_ms": ag_ms if world > 1 else None, "all_gather_bytes_received_per_rank": recv if world > 1 else 0,
            "all_gather_GBs_per_rank": (recv / ag_ms / 1e6) if world > 1 and ag_ms > 0 else None,
            "all_gather_aligned_ms": pure_ms, "all_gather_aligned_GBs_per_rank": (recv / pure_ms / 1e6) if pure_ms else None,
            "depth_maps_ms_max_rank": dm_ms, "fusion_ms_max_rank": fu_ms, "fused_points": int(pts), "sharding": "block (balanced): views per rank " +
            ",".join(str(len(scene.shard_views(N, r, world, "block"))) for r in range(world)),
            "note": "4 source views for depth, 10 for fusion; feature cache + CUDA graphs; wall clock around run_scene, max over ranks; "
                    "all_gather_ms: CUDA events around the collective inside the run, max over ranks, i.e. including the wait for the slowest rank; "
                    "all_gather_aligned_ms: the same collective repeated after a barrier"}


def run_ours(a, rank, world, local_rank):
    import effimvs_b200  # noqa: F401
    from effimvs_b200 import hotpath, ops, synthetic
    assert torch.cuda.is_available(), "bench.py (impl ours) needs a CUDA device; there is no CPU fallback"
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    torch.backends.cudnn.benchmark = True      # as upstream's test script (test_dtu_dypcd.py:41)
    hp = hotpath.CudaHotPath(a.precision, native_projection=True)
    ndepths = synthetic.SHAPES[a.shape]["ndepths"]
    model, data = build_model(hp, dev, ndepths)
    s_host = synthetic.make_sample(a.shape, seed=rank)
    # 8-bit images, as image files hold them; the fp32 images every leg computes on are u8 / 255 exactly as upstream's
    # loaders form them (np.float32 / 255., datasets/general_eval.py:83-87)
    import numpy as np
    u8 = (s_host["imgs"] * 255.0).round().clamp(0, 255).to(torch.uint8)
    f32 = torch.from_numpy(u8.numpy().astype(np.float32) / np.float32(255.0))
    rest = {"depth_values": s_host["depth_values"].pin_memory(),
            "proj_matrices": {k: v.pin_memory() for k, v in s_host["proj_matrices"].items() if k != "stage4"}}
    pin = dict(rest, imgs=f32.pin_memory())           # fp32 host images (what upstream's loaders hand over)
    pin_u8 = dict(rest, imgs=u8.pin_memory())         # 8-bit host images, normalised on the device
    stat = {"imgs": pin["imgs"].to(dev), "depth_values": pin["depth_values"].to(dev),
            "proj_matrices": {k: v.to(dev) for k, v in pin["proj_matrices"].items()}}
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def forward():
        return model(stat["imgs"], stat["proj_matrices"], stat["depth_values"])

    if a.profile_one:
        with torch.no_grad():
            for _ in range(3):
                forward()
            torch.cuda.synchronize()
            torch.cuda.profiler.start()
            forward()
            torch.cuda.synchronize()
            torch.cuda.profiler.stop()
        return

    graph = None
    with torch.no_grad():
        for _ in range(2):       # the first forward also prepares the persistent regularization workspaces
            out = forward()
        ops.LAUNCHES = 0
        out = forward()
        launches_per_step = ops.LAUNCHES
        torch.cuda.synchronize()
        if not a.no_graph:
            try:
                g = torch.cuda.CUDAGraph()
                side = torch.cuda.Stream()
                side.wait_stream(torch.cuda.current_stream())
                with torch.cuda.stream(side):
                    forward()
                torch.cuda.current_stream().wait_stream(side)
                with torch.cuda.graph(g):
                    out = forward()
                graph = g
            except Exception as e:  # noqa: BLE001  (capture is an optimisation; eager stays correct)
                sys.stderr.write("CUDA graph capture failed, running eagerly: {}\n".format(e))
                graph = None
                torch.cuda.synchronize()

        last = [out]      # what the latest step returned: the graph's output tensors, or a new eager result per step

        def step():
            flush.zero_()
            if graph is not None:
                graph.replay()
                return out
            last[0] = forward()
            return last[0]

        def barrier():
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()

        def timed(fn, K, W):
            for _ in range(W):
                fn()
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(K):
                fn()
            e1.record()
            barrier()
            ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
            if world > 1:
                dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            return float(ms)

        with ClockSampler(local_rank) as clk:
            ms_dev = timed(step, a.steps, max(a.warmup, 3))
            # a device-side copy: the host copy and the file writes wait until the clocks are no longer sampled
            dumped = output_arrays(last[0]) if a.dump_outputs and rank == 0 else None

            # end to end through the public API (effimvs_b200.pipeline.DepthMapPipeline): every step copies the
            # sample from pinned host memory to the device and reads depth + confidence back to the host; the
            # copy of sample k+1 overlaps the forward of sample k (two slots, one CUDA graph each)
            from effimvs_b200 import pipeline
            pipe = pipeline.DepthMapPipeline(model, pin, slots=2, use_graph=graph is not None, before_replay=flush.zero_)

            def e2e_timed(sample):
                def run(n):
                    prev = None
                    for _ in range(n):
                        t = pipe.submit(sample)
                        if prev is not None:
                            pipe.result(prev)
                        prev = t
                    return pipe.result(prev)

                run(max(a.warmup, 3))
                barrier()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record(pipe.copy)                      # the first timed operation is the H2D copy of step 0
                hd, hc = run(a.steps)
                e1.record(pipe.compute)                   # after the last D2H read
                barrier()
                ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
                if world > 1:
                    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
                return float(ms), hd.numel() * 4 + hc.numel() * 4

            ms_e2e, d2h = e2e_timed(pin_u8)               # headline: 8-bit images over PCIe
            ms_e2e_f32, _ = e2e_timed(pin)                # the same with fp32 host images (4x the image bytes)
        h2d, h2d_f32 = pipe.h2d_bytes(pin_u8), pipe.h2d_bytes(pin)
        if dumped is not None:
            dump_outputs(a.dump_outputs, dumped)
            del dumped

        # The same forward with fp32 products in every 2-D convolution (torch.backends.cudnn.allow_tf32 = False: cuDNN's fp32
        # kernels for the FPN and the update block, whose tensor-core kernel follows the same switch) -- the setting of the
        # parity tests.  The headline above keeps PyTorch's default, as upstream's scripts do.
        strict = None
        if rank == 0 and world == 1 and graph is not None and os.environ.get("EFFIMVS_BENCH_STRICT", "1") != "0":
            saved_tf32 = torch.backends.cudnn.allow_tf32
            torch.backends.cudnn.allow_tf32 = False
            try:
                forward()
                g32 = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g32):
                    forward()

                def step32():
                    flush.zero_()
                    g32.replay()
                ms32 = timed(step32, a.steps, max(a.warmup, 3))
                strict = {"ms_per_step": ms32 / a.steps, "value": a.steps / (ms32 / 1e3), "unit": UNIT,
                          "what": "torch.backends.cudnn.allow_tf32 = False: fp32 products in all 2-D convolutions (FPN, update block on cuDNN)"}
                del g32
            except Exception as e:  # noqa: BLE001  (an extra leg must not cost the headline line)
                strict = {"error": "{}: {}".format(type(e).__name__, e)}
            finally:
                torch.backends.cudnn.allow_tf32 = saved_tf32

        hbm_peak, tf_peak, peak_src = peaks()
        roof = roof_reg = kern = None
        if rank == 0:
            roof, roof_reg, kern = kernel_rooflines(hp, model, stat, hbm_peak, tf_peak, peak_src)

    scene49 = None
    if not a.no_scene and a.shape == "dtu":
        del pipe
        try:
            scene49 = scene_leg(a, model, rank, world, dev)
        except Exception as e:  # noqa: BLE001  (an extra leg must not cost the headline line)
            scene49 = {"error": "{}: {}".format(type(e).__name__, e)}
            if world > 1:
                raise
    cpu = eager = None
    if rank == 0 and world == 1 and not a.no_cpu_baseline:
        eager = gpu_eager_baseline(a, ndepths, stat, dev)
        cpu = cpu_baseline(a, ndepths)
    if rank != 0:
        return
    value = world * a.steps / (ms_dev / 1e3)
    e2e = world * a.steps / (ms_e2e / 1e3)
    metric, _ = LABELS[a.shape]
    line = {"metric": metric, "value": value, "unit": UNIT, "n_gpus": world, "steps": a.steps, "warmup": max(a.warmup, 3),
            "ms_per_step": ms_dev / a.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": {"f32": "f32", "bf16": "bf16 MMA, f32 accumulate (3-D regularization) / f32 (warp, lookup, regression)",
                      "bf16x3": "hi+lo bf16 MMA x3, f32 accumulate (3-D regularization, fp32-grade) / f32 (warp, lookup, regression)"}[a.precision],
            "data": data,
            "config": config_keys(a, int(stat["imgs"].shape[1]), ndepths),
            "run": {"device": "cuda", "cuda_graph": graph is not None, "processes": world},
            "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e / a.steps,
                    "api": "effimvs_b200.pipeline.DepthMapPipeline.submit/result with 8-bit host images (divided by 255 on the device, "
                           "upstream's loader arithmetic): pinned host -> device copy of step k+1 overlapped with the forward of step k"},
            "e2e_fp32_images": {"value": world * a.steps / (ms_e2e_f32 / 1e3), "unit": UNIT, "h2d_bytes_per_step": h2d_f32,
                                "d2h_bytes_per_step": d2h, "ms_per_step": ms_e2e_f32 / a.steps},
            "gpu_launches": launches_per_step * a.steps, "gpu_launches_per_step": launches_per_step,
            "conv2d": {"cudnn_allow_tf32": bool(torch.backends.cudnn.allow_tf32),
                       "update_block_3x3": "libeffimvs conv2d_tc (tcgen05, fp16 operands = TF32's 11 significant bits, fp32 accumulate, GRU gates as "
                                           "epilogues) on the 1/4- and 1/2-resolution stages, cuDNN (TF32) on the 1/8 stage and for the FPN"
                       if os.environ.get("EFFIMVS_CONV2D", "auto") != "0" else "cuDNN (TF32)"},
            "strict_fp32": strict,
            "clocks": clk.summary(), "roofline": roof, "roofline_regularization": roof_reg, "kernels": kern}
    if scene49:
        line["scene49"] = scene49
    if cpu:
        line["cpu_baseline"] = cpu
    if eager:
        line["gpu_eager_baseline"] = eager
    OUT.emit(json.dumps(line))


def cpu_baseline(a, ndepths):
    """The reference arm's model on this box's host cores, bounded to a few forwards."""
    from effimvs_b200 import synthetic
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    model, kind, what = reference_model("cpu", ndepths)
    s = synthetic.make_sample(a.shape, seed=0)
    ts = []
    with torch.no_grad():
        for i in range(3):
            t0 = time.perf_counter()
            model(s["imgs"], s["proj_matrices"], s["depth_values"])
            ts.append(time.perf_counter() - t0)
            if sum(ts) > 45:
                break
    timed = ts[1:] if len(ts) > 1 else ts
    v = len(timed) / sum(timed)
    return {"value": v, "unit": UNIT, "cores": cores, "kind": kind,
            "sample": "{} full {} depth map(s) after {} warm-up on {} threads; {}".format(
                len(timed), a.shape, len(ts) - len(timed), cores, what)}


def gpu_eager_baseline(a, ndepths, sample, dev, reps=3):
    """The reference's eager PyTorch forward on the SAME B200 (SURVEY section 8(d)): unmodified upstream, device-resident
    inputs, CUDA events around `reps` forwards after one warm-up, with TF32 off (the parity setting) and with torch's
    defaults for cuDNN (TF32 allowed for convolutions, as upstream's own test scripts run)."""
    model, kind, what = reference_model(dev, ndepths)
    out = {"kind": kind, "what": what, "unit": UNIT, "steps": reps}
    saved = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark)
    try:
        with torch.no_grad():
            for tag, tf32 in (("tf32_off", False), ("tf32_on", True)):
                torch.backends.cudnn.allow_tf32 = tf32
                torch.backends.cuda.matmul.allow_tf32 = False
                torch.backends.cudnn.benchmark = True          # as test_dtu_dypcd.py:41
                for _ in range(2):
                    model(sample["imgs"], sample["proj_matrices"], sample["depth_values"])
                torch.cuda.synchronize()
                e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                e0.record()
                for _ in range(reps):
                    model(sample["imgs"], sample["proj_matrices"], sample["depth_values"])
                e1.record()
                torch.cuda.synchronize()
                ms = e0.elapsed_time(e1) / reps
                out[tag] = {"ms_per_step": ms, "value": 1e3 / ms}
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark = saved
    del model
    torch.cuda.empty_cache()
    return out


class _QuietStdout:
    """Everything written to fd 1 by libraries (NCCL prints its version banner there) goes to stderr
    while the benchmark runs; `emit` restores stdout for the ONE JSON line."""

    def __init__(self):
        sys.stdout.flush()
        self.saved = os.dup(1)
        os.dup2(2, 1)

    def emit(self, line):
        sys.stdout.flush()
        os.dup2(self.saved, 1)
        print(line, flush=True)
        os.dup2(2, 1)


OUT = None


def main():
    global OUT
    OUT = _QuietStdout()
    a = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if a.impl == "reference":
        run_reference(a, rank, world)
        return
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    try:
        run_ours(a, rank, world, local_rank)
    finally:
        if world > 1:
            dist.destroy_process_group()


if __name__ == "__main__":
    main()
