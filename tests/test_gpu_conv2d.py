"""The update block's 3x3 convolutions on the tensor cores (csrc/conv2d_tc.cu, SURVEY section 8(f) row 3), ``-m gpu``.

Upstream: models/update.py:10-27 (DepthHead.conv1), :33-49 (ConvGRU), :69-99 (ProjectionInput), :106-110 (mask[0]).

Three bars, all through the C-ABI:
  (1) the kernel against its exact arithmetic -- operands rounded to IEEE half (11 significant bits, the precision class of
      TF32), products exact, accumulated here in fp64 -- 5e-6 of max|ref| for every epilogue mode, pixel strides, channel
      segments, and the stage shapes of the DTU cascade;
  (2) the kernel against the fp32 convolution: its error is that of its operand rounding, i.e. no larger than the error of the
      cuDNN TF32 kernel PyTorch would run for the same layer (measured and printed, bar: 1.5 x cuDNN-TF32's own error);
  (3) the update block and the whole cascade with these convolutions against upstream's fp32 eager forward, next to what
      upstream itself loses when PyTorch's default torch.backends.cudnn.allow_tf32 = True is left on.
"""
import os

import pytest
import torch
import torch.nn.functional as F

from util import GOLDEN, golden, rel_max

pytestmark = pytest.mark.gpu
DEV = "cuda"


@pytest.fixture(scope="module", autouse=True)
def _strict_fp32():
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.set_grad_enabled(False)
    yield
    torch.backends.cudnn.allow_tf32 = False


def f16(x):
    return x.half().float()


def _maps(B, H, W, c0, c1, cout, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    big0 = torch.randn(B, H, W, c0 + 16, device=DEV, generator=g)            # in0 is a channel slice of a wider map
    x0 = big0[..., 8:8 + c0].permute(0, 3, 1, 2)
    x1 = torch.randn(B, H, W, c1, device=DEV, generator=g).permute(0, 3, 1, 2) if c1 else None
    w = torch.randn(cout, c0 + c1, 3, 3, device=DEV, generator=g) * 0.1
    bias = torch.randn(cout, device=DEV, generator=g)
    return g, x0, x1, w, bias


def _cl(B, C, H, W, fill=None, g=None):
    t = torch.empty(B, C, H, W, device=DEV, memory_format=torch.channels_last)
    if g is not None:
        t.copy_(torch.randn(B, C, H, W, device=DEV, generator=g))
    elif fill is not None:
        t.fill_(fill)
    return t


CASES = [
    # B, H, W, c0, c1, cout, mode
    (1, 8, 40, 16, 0, 16, "bias"),             # one partial strip
    (1, 37, 200, 16, 0, 16, "relu"),           # two strips
    (2, 19, 130, 32, 0, 32, "relu"),           # batch 2, a strip of two pixels
    (1, 64, 128, 16, 16, 32, "gates"),         # two segments inside one K phase
    (1, 64, 300, 32, 32, 64, "gates"),         # one K phase of 64 channels over two segments
    (1, 33, 257, 16, 16, 16, "update"),
    (1, 50, 100, 32, 0, 16, "add"),
    (1, 50, 100, 64, 0, 32, "add"),
    (1, 30, 70, 48, 0, 48, "relu"),            # three K phases of 16
    (1, 30, 70, 16, 0, 12, "bias"),            # cout not a multiple of 16
    (1, 2, 5, 16, 0, 16, "bias"),              # tiny
    (1, 148, 200, 48, 48, 96, "gates"),        # DTU stage 1 (hidden 48): 96 -> 96, three K phases of 32
    (1, 148, 200, 96, 0, 48, "add"),
    (1, 296, 400, 64, 0, 64, "relu"),          # DTU stage 2 (hidden 32)
    (1, 296, 400, 32, 32, 32, "update"),
    (1, 592, 800, 32, 0, 32, "relu"),          # DTU stage 3 (hidden 16)
    (1, 592, 800, 16, 16, 32, "gates"),
    (1, 592, 800, 16, 16, 16, "update"),
    (1, 528, 960, 16, 0, 32, "relu"),          # Tanks & Temples stage 3, mask head
]


@pytest.mark.parametrize("B,H,W,c0,c1,cout,mode", CASES)
def test_conv2d_tc_vs_exact_arithmetic(B, H, W, c0, c1, cout, mode):
    from effimvs_b200 import capi, ops
    g, x0, x1, w, bias = _maps(B, H, W, c0, c1, cout, seed=H + W + cout)
    xin = x0 if x1 is None else torch.cat([x0, x1], dim=1)
    acc = F.conv2d(f16(xin).double(), f16(w).double(), padding=1)
    pk = ops.conv2d_tc_pack(w)
    bar = 5e-6
    if mode in ("bias", "relu"):
        outbig = torch.full((B, H, W, cout + 4), 7.0, device=DEV)
        out = outbig[..., 4:].permute(0, 3, 1, 2)                            # written into a channel slice
        ops.conv2d_tc(x0, x1, pk, bias, cout, capi.CONV2D_BIAS_RELU if mode == "relu" else capi.CONV2D_BIAS, out, None, None)
        want = acc + bias.double().reshape(1, -1, 1, 1)
        want = want.relu() if mode == "relu" else want
        assert bool((outbig[..., :4] == 7.0).all())
        errs = [float((out.double() - want).abs().max() / want.abs().max())]
    elif mode == "add":
        add = _cl(B, cout, H, W, g=g)
        out = _cl(B, cout, H, W)
        ops.conv2d_tc(x0, x1, pk, None, cout, capi.CONV2D_ADD_RELU, out, add, None)
        want = (acc + add.double()).relu()
        errs = [float((out.double() - want).abs().max() / want.abs().max())]
    elif mode == "gates":
        h = cout // 2
        hprev, z, out = _cl(B, h, H, W, g=g), _cl(B, h, H, W), _cl(B, h, H, W)
        ops.conv2d_tc(x0, x1, pk, bias, cout, capi.CONV2D_GRU_GATES, out, hprev, z)
        pre = acc + bias.double().reshape(1, -1, 1, 1)
        wz, wr = torch.sigmoid(pre[:, :h]), torch.sigmoid(pre[:, h:]) * hprev.double()
        errs = [float((z.double() - wz).abs().max()), float((out.double() - wr).abs().max() / wr.abs().max())]
    else:
        zz = torch.rand(B, cout, H, W, device=DEV, generator=g).contiguous(memory_format=torch.channels_last)
        netm = _cl(B, cout, H, W, g=g)
        want = (1 - zz.double()) * netm.double() + zz.double() * torch.tanh(acc + bias.double().reshape(1, -1, 1, 1))
        ops.conv2d_tc(x0, x1, pk, bias, cout, capi.CONV2D_GRU_UPDATE, netm, zz, None)
        errs = [float((netm.double() - want).abs().max() / want.abs().max())]
    print("conv2d_tc {}x{}x{} {}+{}->{} {}: {}".format(B, H, W, c0, c1, cout, mode, ["%.1e" % e for e in errs]))
    assert max(errs) < bar, errs


@pytest.mark.parametrize("H,W,cin,cout", [(592, 800, 32, 32), (296, 400, 64, 64), (148, 200, 96, 96)])
def test_conv2d_tc_error_class_is_tf32(H, W, cin, cout):
    """against the fp32 convolution (fp64 here): no worse than cuDNN's TF32 kernel for the same layer"""
    from effimvs_b200 import capi, ops
    g = torch.Generator(device=DEV).manual_seed(cin)
    x = torch.tanh(torch.randn(1, cin, H, W, device=DEV, generator=g)).contiguous(memory_format=torch.channels_last)
    w = (torch.randn(cout, cin, 3, 3, device=DEV, generator=g) * 0.1).contiguous(memory_format=torch.channels_last)
    bias = torch.randn(cout, device=DEV, generator=g)
    exact = F.conv2d(x.double(), w.double(), bias.double(), padding=1)
    out = _cl(1, cout, H, W)
    ops.conv2d_tc(x, None, ops.conv2d_tc_pack(w), bias, cout, capi.CONV2D_BIAS, out, None, None)
    torch.backends.cudnn.allow_tf32 = True
    try:
        tf = F.conv2d(x, w, bias, padding=1)
    finally:
        torch.backends.cudnn.allow_tf32 = False
    fp = F.conv2d(x, w, bias, padding=1)
    e_own, e_tf, e_fp = (float((t.double() - exact).abs().max() / exact.abs().max()) for t in (out, tf, fp))
    print("conv {}->{} at {}x{}: error vs fp64 -- own {:.2e}, cuDNN TF32 {:.2e}, cuDNN fp32 {:.2e}".format(cin, cout, H, W, e_own, e_tf, e_fp))
    assert e_own <= 1.5 * e_tf and e_own < 2e-3


def test_conv2d_tc_rejects_bad_arguments():
    from effimvs_b200 import capi, ops
    x = _cl(1, 16, 8, 8, fill=0.0)
    w = torch.zeros(16, 16, 3, 3, device=DEV)
    pk = ops.conv2d_tc_pack(w)
    out = _cl(1, 16, 8, 8)
    with pytest.raises(Exception):                       # planar (NCHW-contiguous) input
        ops.conv2d_tc(torch.zeros(1, 16, 8, 8, device=DEV), None, pk, None, 16, capi.CONV2D_BIAS, out, None, None)
    with pytest.raises(Exception):                       # ADD_RELU without the addend
        ops.conv2d_tc(x, None, pk, None, 16, capi.CONV2D_ADD_RELU, out, None, None)
    with pytest.raises(Exception):                       # packed weights of another shape
        ops.conv2d_tc(x, None, ops.conv2d_tc_pack(torch.zeros(32, 16, 3, 3, device=DEV)), None, 16, capi.CONV2D_BIAS, out, None, None)
    assert not ops.conv2d_tc_supported(12, 16) and not ops.conv2d_tc_supported(256, 256) and ops.conv2d_tc_supported(96, 96)
    with pytest.raises(Exception):
        ops.conv2d_tc_pack(torch.zeros(16, 12, 3, 3, device=DEV))


@pytest.mark.parametrize("h,cx,H,W", [(16, 4, 592, 800), (32, 8, 296, 400), (48, 12, 148, 200)])
def test_update_block_tc_vs_fp32(h, cx, H, W, monkeypatch):
    """BasicUpdateBlock (models/update.py:114-141) + upsample_depth at the three DTU stage shapes: the fused block with the
    tensor-core convolutions against the same block in fp32 (cuDNN, TF32 off), next to the fused block on cuDNN's TF32 kernels."""
    from test_net_host import _update_cost_fn
    from effimvs_b200 import hotpath, net
    hp = hotpath.CudaHotPath("f32")
    torch.manual_seed(h)
    blk = net.UpdateBlock(h, 6, 2, cx).to(DEV).eval()
    B = 1
    n0, ctx = torch.tanh(torch.randn(B, h, H, W, device=DEV)), torch.relu(torch.randn(B, cx, H, W, device=DEV))
    inv0 = torch.rand(B, 1, H, W, device=DEV)
    lo, hi = torch.tensor([1 / 935.0], device=DEV), torch.tensor([1 / 425.0], device=DEV)

    def run(conv2d, tf32):
        monkeypatch.setenv("EFFIMVS_CONV2D", conv2d)
        torch.backends.cudnn.allow_tf32 = tf32
        try:
            n, invs, deps, up, dup, _ = blk.forward_fused(hp, n0, _update_cost_fn, inv0, ctx, 3, lo, hi)
        finally:
            torch.backends.cudnn.allow_tf32 = False
        return n.clone(), invs[-1].clone(), up.clone(), dup.clone()

    want = run("0", False)
    tf = run("0", True)
    own = run("1", False)
    names = ("net", "inv", "up", "depth_up")
    e_tf = [float((a - b).abs().max()) for a, b in zip(tf, want)]
    e_own = [float((a - b).abs().max()) for a, b in zip(own, want)]
    print("update block h={} {}x{}: max|d| vs fp32 -- own {} | cuDNN TF32 {}".format(
        h, H, W, dict(zip(names, ["%.2e" % e for e in e_own])), dict(zip(names, ["%.2e" % e for e in e_tf]))))
    for a, b in zip(e_own, e_tf):
        assert a <= 2.0 * b + 1e-6, (e_own, e_tf)
    assert e_own[1] < 5e-3                       # normalised inverse depth in [0, 1]


def test_update_block_tc_golden(monkeypatch):
    """against upstream's own BasicUpdateBlock outputs (tests/golden/update_block.npz), TF32-class tolerance"""
    from test_net_host import load_update_block, _update_cost_fn
    from effimvs_b200 import hotpath
    monkeypatch.setenv("EFFIMVS_CONV2D", "1")
    hp = hotpath.CudaHotPath("f32")
    g = golden("update_block", DEV)
    blk = load_update_block(g, DEV)
    B = g["inv0"].shape[0]
    lo, hi = (1.0 / g["dmax"]).reshape(B), (1.0 / g["dmin"]).reshape(B)
    n, invs, deps, up, dup, _ = blk.forward_fused(hp, g["net0"], _update_cost_fn, g["inv0"], g["context"], 3, lo, hi)
    errs = [rel_max(n, g["net"])] + [float((invs[i] - g["inv{}".format(i + 1)]).abs().max()) for i in range(3)] + \
           [float((up - g["up"]).abs().max()), rel_max(dup, g["depth_up"])]
    print("update block (tensor-core convolutions) vs upstream golden:", ["%.2e" % e for e in errs])
    assert max(errs) < 3e-3


def test_cascade_tc_vs_upstream_full_shape(monkeypatch):
    """The configuration bench.py times (cuDNN TF32 allowed, as PyTorch ships; update-block convolutions on conv2d_tc) against
    upstream's fp32 eager forward at 1600x1184x5 -- and upstream itself with TF32 allowed against the same: the fraction of
    pixels within 0.51 mm must not be lower than upstream's own TF32 fraction (minus 0.2 %).  Where upstream's byte copy is
    not staged, the oracle port of its forward (net.EffiMVSPlus + OracleHotPath) stands in for it, in fp32 and with TF32."""
    from oracle import hotpath as ohp
    from oracle import upstream
    from effimvs_b200 import hotpath, synthetic
    from util import dtu_model
    s = synthetic.make_sample("dtu", seed=11, device=DEV)
    if upstream.available():
        ref_model = upstream.build_model(torch.load(os.path.join(GOLDEN, "dtu_weights.pt"), map_location="cpu"), "48,8,8", DEV)
    else:
        ref_model = dtu_model(ohp.OracleHotPath(), DEV, "48,8,8")
    want = [d.clone() for d in ref_model(s["imgs"], s["proj_matrices"], s["depth_values"])["depth"]]
    torch.backends.cudnn.allow_tf32 = True
    try:
        up_tf = [d.clone() for d in ref_model(s["imgs"], s["proj_matrices"], s["depth_values"])["depth"]]
        del ref_model
        torch.cuda.empty_cache()
        model = dtu_model(hotpath.CudaHotPath("bf16x3", native_projection=True), DEV, "48,8,8")
        monkeypatch.setenv("EFFIMVS_CONV2D", "auto")
        own = [d.clone() for d in model(s["imgs"], s["proj_matrices"], s["depth_values"])["depth"]]
        monkeypatch.setenv("EFFIMVS_CONV2D", "0")
        cud = [d.clone() for d in model(s["imgs"], s["proj_matrices"], s["depth_values"])["depth"]]
    finally:
        torch.backends.cudnn.allow_tf32 = False
    tol = 1e-3 * (935.0 - 425.0)
    frac = lambda got: [float(((a - b).abs() <= tol).float().mean()) for a, b in zip(got, want)]   # noqa: E731
    f_up, f_own, f_cud = frac(up_tf), frac(own), frac(cud)
    ref = "upstream" if upstream.available() else "the oracle port"
    print("fraction of pixels within 0.51 mm of {} fp32, worst of 13 outputs: {} with TF32 {:.5f}, cascade with cuDNN TF32 "
          "convolutions {:.5f}, cascade with conv2d_tc {:.5f}".format(ref, ref, min(f_up), min(f_cud), min(f_own)))
    assert min(f_own) >= min(f_up) - 0.002
    assert min(f_own) >= min(f_cud) - 0.002


def test_cascade_tc_graph_replay_equals_eager(monkeypatch):
    """the cascade with the tensor-core convolutions is deterministic and CUDA-graph capturable: a replay reproduces the eager
    forward bit for bit (all three stages forced onto conv2d_tc, 640x512x5)"""
    from effimvs_b200 import hotpath, synthetic
    from util import dtu_model
    monkeypatch.setenv("EFFIMVS_CONV2D", "1")
    s = synthetic.make_sample("plumbing", seed=5, device=DEV)
    model = dtu_model(hotpath.CudaHotPath("bf16x3", native_projection=True), DEV, "48,8,8")
    fwd = lambda: model(s["imgs"], s["proj_matrices"], s["depth_values"])   # noqa: E731
    fwd()
    eager = [d.clone() for d in fwd()["depth"]]
    side = torch.cuda.Stream()
    side.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(side):
        fwd()
    torch.cuda.current_stream().wait_stream(side)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out = fwd()
    for _ in range(2):
        g.replay()
        torch.cuda.synchronize()
        assert all(torch.equal(a, b) for a, b in zip(out["depth"], eager))
    assert all(bool(torch.isfinite(d).all()) for d in eager)


_PDL_SCRIPT = r"""
import os, sys
sys.path.insert(0, {root!r}); sys.path.insert(0, os.path.join({root!r}, "tests"))
import torch
import effimvs_b200  # noqa: F401
from effimvs_b200 import hotpath, synthetic
from util import dtu_model
torch.backends.cudnn.allow_tf32 = True                 # the update block on conv2d_tc (EFFIMVS_CONV2D_MIN_PIXELS lowered by the test)
dev = torch.device("cuda:0")
s = synthetic.make_sample("plumbing", seed=3, device=dev, width=640, height=512)
model = dtu_model(hotpath.CudaHotPath("bf16x3"), dev)
with torch.no_grad():
    out = model(s["imgs"], s["proj_matrices"], s["depth_values"])
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        out2 = model(s["imgs"], s["proj_matrices"], s["depth_values"])
    g.replay()
torch.cuda.synchronize()
torch.save({{"eager": [d.cpu() for d in out["depth"]], "graph": [d.cpu() for d in out2["depth"]]}}, sys.argv[1])
"""


@pytest.mark.gpu
def test_programmatic_dependent_launch_switch_gives_the_same_depth_maps(tmp_path):
    """EFFIMVS_PDL=1 (every hot-path kernel launched with the programmatic-stream-serialization attribute, griddepcontrol.wait
    before its first dependent access; csrc/common.cuh) against the classic launches: the whole cascade at 640x512x5, eager and
    as a CUDA graph (programmatic edges), in two fresh processes -- the switch is read once per process.  A kernel that touched a
    predecessor's output before its wait would show up as stale data in some of the 13 depth maps."""
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    script = tmp_path / "pdl_run.py"
    script.write_text(_PDL_SCRIPT.format(root=root))
    res = {}
    for flag in ("0", "1"):
        out = tmp_path / "pdl{}.pt".format(flag)
        env = dict(os.environ, EFFIMVS_PDL=flag, EFFIMVS_CONV2D_MIN_PIXELS="20000")     # tensor-core update block on stages 2 and 3
        subprocess.run([sys.executable, str(script), str(out)], check=True, env=env, timeout=600)
        res[flag] = torch.load(out)
    for kind in ("eager", "graph"):
        for a, b in zip(res["0"][kind], res["1"][kind]):
            # cuDNN picks its algorithms per process, so the two runs agree to convolution rounding, not bit for bit
            assert float(((a - b).abs() <= 0.05).float().mean()) >= 0.999
    for a, b in zip(res["1"]["eager"], res["1"]["graph"]):
        assert float(((a - b).abs() <= 0.05).float().mean()) >= 0.999
