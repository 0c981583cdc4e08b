"""The update block's 3x3 convolutions with fp32-grade operands (bf16x3: hi + lo bf16 pairs, three products, fp32 accumulation;
csrc/conv2d_tc.cu, CudaHotPath(conv2d_precision="bf16x3")), ``-m gpu``.

  (1) the kernel against its own arithmetic restated in fp64 (the hi / lo split by torch's round-to-nearest bf16 conversion,
      the three products summed exactly): 5e-6 of max|ref|, the case list of test_gpu_conv2d.py minus the 1/8-stage widths;
  (2) against the fp64 convolution of the unrounded operands: 2e-5 of max|y| and a tenth of cuDNN-TF32's error;
  (3) inputs of 1e5 - 1e6, beyond fp16's range: finite, within bar (2);
  (4) the fused update block against the same block on cuDNN fp32, and against upstream's BasicUpdateBlock golden;
  (5) the whole cascade with TF32 off against upstream's fp32 forward (or the oracle port), at the bars of check_outputs;
  (6) CUDA-graph replay, and one model run alternately under the fp16 and the bf16x3 kernels (packed images per precision).
"""
import copy

import pytest
import torch
import torch.nn.functional as F

from test_gpu_conv2d import CASES, _cl, _maps
from util import golden, rel_max

pytestmark = pytest.mark.gpu
DEV = "cuda"


@pytest.fixture(scope="module", autouse=True)
def _strict_fp32():
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    torch.set_grad_enabled(False)
    yield
    torch.backends.cudnn.allow_tf32 = False


def _split(x):
    """(hi, lo) as the kernel forms them: hi = bf16_rn(x), lo = bf16_rn(x - hi), in fp64"""
    hi = x.bfloat16().float()
    return hi.double(), (x - hi).bfloat16().double()


def _conv3(x, w):
    """hi.hi + hi.lo + lo.hi in fp64"""
    (xh, xl), (wh, wl) = _split(x), _split(w)
    return F.conv2d(xh, wh, padding=1) + F.conv2d(xh, wl, padding=1) + F.conv2d(xl, wh, padding=1)


@pytest.mark.parametrize("B,H,W,c0,c1,cout,mode", CASES)
def test_conv2d_bf16x3_vs_own_arithmetic(B, H, W, c0, c1, cout, mode):
    from effimvs_b200 import capi, ops
    P = "bf16x3"
    if not ops.conv2d_tc_supported(c0 + c1, cout, P):
        assert c0 + c1 == 96, "only the 1/8-stage widths may be unsupported"
        pytest.skip("{} -> {}: weights do not fit shared memory twice".format(c0 + c1, cout))
    g, x0, x1, w, bias = _maps(B, H, W, c0, c1, cout, seed=H + W + cout)
    xin = x0 if x1 is None else torch.cat([x0, x1], dim=1)
    acc = _conv3(xin, w)
    pk = ops.conv2d_tc_pack(w, P)
    bar = 5e-6
    if mode in ("bias", "relu"):
        outbig = torch.full((B, H, W, cout + 4), 7.0, device=DEV)
        out = outbig[..., 4:].permute(0, 3, 1, 2)
        ops.conv2d_tc(x0, x1, pk, bias, cout, capi.CONV2D_BIAS_RELU if mode == "relu" else capi.CONV2D_BIAS, out, None, None, P)
        want = acc + bias.double().reshape(1, -1, 1, 1)
        want = want.relu() if mode == "relu" else want
        assert bool((outbig[..., :4] == 7.0).all())
        errs = [float((out.double() - want).abs().max() / want.abs().max())]
    elif mode == "add":
        add = _cl(B, cout, H, W, g=g)
        out = _cl(B, cout, H, W)
        ops.conv2d_tc(x0, x1, pk, None, cout, capi.CONV2D_ADD_RELU, out, add, None, P)
        want = (acc + add.double()).relu()
        errs = [float((out.double() - want).abs().max() / want.abs().max())]
    elif mode == "gates":
        h = cout // 2
        hprev, z, out = _cl(B, h, H, W, g=g), _cl(B, h, H, W), _cl(B, h, H, W)
        ops.conv2d_tc(x0, x1, pk, bias, cout, capi.CONV2D_GRU_GATES, out, hprev, z, P)
        pre = acc + bias.double().reshape(1, -1, 1, 1)
        wz, wr = torch.sigmoid(pre[:, :h]), torch.sigmoid(pre[:, h:]) * hprev.double()
        errs = [float((z.double() - wz).abs().max()), float((out.double() - wr).abs().max() / wr.abs().max())]
    else:
        zz = torch.rand(B, cout, H, W, device=DEV, generator=g).contiguous(memory_format=torch.channels_last)
        netm = _cl(B, cout, H, W, g=g)
        want = (1 - zz.double()) * netm.double() + zz.double() * torch.tanh(acc + bias.double().reshape(1, -1, 1, 1))
        ops.conv2d_tc(x0, x1, pk, bias, cout, capi.CONV2D_GRU_UPDATE, netm, zz, None, P)
        errs = [float((netm.double() - want).abs().max() / want.abs().max())]
    print("conv2d bf16x3 {}x{}x{} {}+{}->{} {}: {}".format(B, H, W, c0, c1, cout, mode, ["%.1e" % e for e in errs]))
    assert max(errs) < bar, errs


def _error_vs_fp64(H, W, cin, cout, scale):
    from effimvs_b200 import capi, ops
    g = torch.Generator(device=DEV).manual_seed(cin + int(scale))
    x = torch.tanh(torch.randn(1, cin, H, W, device=DEV, generator=g))
    if scale > 1:      # magnitudes 1e5 .. 1e6 with random signs
        x = torch.sign(x) * (1e5 + (scale - 1e5) * torch.rand(1, cin, H, W, device=DEV, generator=g))
    x = x.contiguous(memory_format=torch.channels_last)
    w = (torch.randn(cout, cin, 3, 3, device=DEV, generator=g) * 0.1).contiguous(memory_format=torch.channels_last)
    bias = torch.randn(cout, device=DEV, generator=g)
    exact = F.conv2d(x.double(), w.double(), bias.double(), padding=1)
    out = _cl(1, cout, H, W)
    ops.conv2d_tc(x, None, ops.conv2d_tc_pack(w, "bf16x3"), bias, cout, capi.CONV2D_BIAS, out, None, None, "bf16x3")
    own16 = _cl(1, cout, H, W)
    ops.conv2d_tc(x, None, ops.conv2d_tc_pack(w), bias, cout, capi.CONV2D_BIAS, own16, None, None)
    torch.backends.cudnn.allow_tf32 = True
    try:
        tf = F.conv2d(x, w, bias, padding=1)
    finally:
        torch.backends.cudnn.allow_tf32 = False
    fp = F.conv2d(x, w, bias, padding=1)
    errs = [float((t.double() - exact).abs().max() / exact.abs().max()) for t in (out, tf, fp, own16)]
    print("conv {}->{} at {}x{}, |x| <= {:g}: error vs fp64 / max|y| -- bf16x3 {:.2e}, cuDNN TF32 {:.2e}, cuDNN fp32 {:.2e}, "
          "fp16 kernel {:.2e}".format(cin, cout, H, W, scale, *errs))
    return out, errs


@pytest.mark.parametrize("H,W,cin,cout", [(592, 800, 32, 32), (296, 400, 64, 64)])
def test_conv2d_bf16x3_error_class_is_fp32(H, W, cin, cout):
    _, (e_own, e_tf, _, _) = _error_vs_fp64(H, W, cin, cout, 1.0)
    assert e_own <= 2e-5 and e_own <= 0.1 * e_tf


@pytest.mark.parametrize("H,W,cin,cout", [(296, 400, 32, 32), (296, 400, 64, 64)])
def test_conv2d_bf16x3_range_beyond_fp16(H, W, cin, cout):
    out, (e_own, _, _, e16) = _error_vs_fp64(H, W, cin, cout, 1e6)
    assert bool(torch.isfinite(out).all())
    assert e_own <= 2e-5
    assert e16 > 1e-2          # the fp16 kernel saturates its operands at 65504 here


def _block_inputs(h, cx, H, W):
    from effimvs_b200 import net
    torch.manual_seed(h)
    blk = net.UpdateBlock(h, 6, 2, cx).to(DEV).eval()
    n0, ctx = torch.tanh(torch.randn(1, h, H, W, device=DEV)), torch.relu(torch.randn(1, cx, H, W, device=DEV))
    inv0 = torch.rand(1, 1, H, W, device=DEV)
    lo, hi = torch.tensor([1 / 935.0], device=DEV), torch.tensor([1 / 425.0], device=DEV)
    return blk, (n0, inv0, ctx, lo, hi)


def _run_block(blk, hp, args, tf32=False):
    from test_net_host import _update_cost_fn
    n0, inv0, ctx, lo, hi = args
    torch.backends.cudnn.allow_tf32 = tf32
    try:
        n, invs, deps, up, dup, _ = blk.forward_fused(hp, n0, _update_cost_fn, inv0, ctx, 3, lo, hi)
    finally:
        torch.backends.cudnn.allow_tf32 = False
    return n.clone(), invs[-1].clone(), up.clone(), dup.clone()


@pytest.mark.parametrize("h,cx,H,W", [(16, 4, 592, 800), (32, 8, 296, 400)])
def test_update_block_bf16x3_vs_fp32(h, cx, H, W, monkeypatch):
    """the fused block at the stage-3 / stage-2 shapes: bf16x3 convolutions (TF32 off) against the same block on cuDNN fp32,
    next to the fp16 kernel's distance from it"""
    from effimvs_b200 import hotpath
    blk, args = _block_inputs(h, cx, H, W)
    monkeypatch.setenv("EFFIMVS_CONV2D", "0")
    want = _run_block(blk, hotpath.CudaHotPath("f32"), args)
    monkeypatch.setenv("EFFIMVS_CONV2D", "1")
    f16 = _run_block(blk, hotpath.CudaHotPath("f32"), args)
    monkeypatch.setenv("EFFIMVS_CONV2D", "auto")
    own = _run_block(blk, hotpath.CudaHotPath("f32", conv2d_precision="bf16x3"), args)
    names = ("net", "inv", "up", "depth_up")
    e16 = [float((a - b).abs().max()) for a, b in zip(f16, want)]
    e3 = [float((a - b).abs().max()) for a, b in zip(own, want)]
    print("update block h={} {}x{}: max|d| vs cuDNN fp32 -- bf16x3 {} | fp16 kernel {}".format(
        h, H, W, dict(zip(names, ["%.2e" % e for e in e3])), dict(zip(names, ["%.2e" % e for e in e16]))))
    for a, b in zip(e3, e16):
        assert a <= 0.1 * b, (e3, e16)
    assert e3[1] < 5e-4


def test_update_block_bf16x3_golden(monkeypatch):
    """against upstream's own BasicUpdateBlock outputs (tests/golden/update_block.npz): bar 3e-4 (the fp16 kernel's is 3e-3)"""
    from test_net_host import load_update_block, _update_cost_fn
    from effimvs_b200 import hotpath
    monkeypatch.setenv("EFFIMVS_CONV2D", "1")        # the golden's maps are below the minimum pixel count
    hp = hotpath.CudaHotPath("f32", conv2d_precision="bf16x3")
    g = golden("update_block", DEV)
    blk = load_update_block(g, DEV)
    B = g["inv0"].shape[0]
    lo, hi = (1.0 / g["dmax"]).reshape(B), (1.0 / g["dmin"]).reshape(B)
    n, invs, deps, up, dup, _ = blk.forward_fused(hp, g["net0"], _update_cost_fn, g["inv0"], g["context"], 3, lo, hi)
    errs = [rel_max(n, g["net"])] + [float((invs[i] - g["inv{}".format(i + 1)]).abs().max()) for i in range(3)] + \
           [float((up - g["up"]).abs().max()), rel_max(dup, g["depth_up"])]
    print("update block (bf16x3 convolutions) vs upstream golden:", ["%.2e" % e for e in errs])
    assert max(errs) < 3e-4


@pytest.mark.parametrize("shape", ["dtu", "tanks"])
def test_cascade_bf16x3_parity_configuration(shape):
    """TF32 off, net.EffiMVSPlus + CudaHotPath("bf16x3", native_projection=True, conv2d_precision="bf16x3") against upstream's
    unpatched fp32 forward (the oracle port where upstream's copy is not staged), at the bars of check_outputs; the same
    cascade with the update block on cuDNN fp32 printed beside it."""
    from test_gpu_upstream import SHAPES, check_outputs, frac_within, sample_and_upstream_eager
    from effimvs_b200 import hotpath
    from util import dtu_model
    s, want = sample_and_upstream_eager(shape)
    model = dtu_model(hotpath.CudaHotPath("bf16x3", native_projection=True), DEV, SHAPES[shape])
    base = model(s["imgs"], s["proj_matrices"], s["depth_values"])
    fb = min(frac_within(a, b, 1e-3 * (935.0 - 425.0)) for a, b in zip(base["depth"], want["depth"]))
    print("update block on cuDNN fp32 [{}]: worst fraction within 0.51 mm {:.5f}".format(shape, fb))
    del base, model
    torch.cuda.empty_cache()
    model = dtu_model(hotpath.CudaHotPath("bf16x3", native_projection=True, conv2d_precision="bf16x3"), DEV, SHAPES[shape])
    got = model(s["imgs"], s["proj_matrices"], s["depth_values"])
    check_outputs(got, want, "net.EffiMVSPlus[{} bf16x3, conv2d bf16x3]".format(shape))


@pytest.mark.parametrize("shape", ["dtu", "tanks"])
def test_dropin_patch_bf16x3_parity_configuration(shape):
    """the same through dropin.patch on upstream's own model (needs upstream's copy staged)"""
    from oracle import upstream
    from test_gpu_upstream import SHAPES, _weights, check_outputs, sample_and_upstream_eager
    from effimvs_b200 import dropin, hotpath
    if not upstream.available():
        pytest.skip("patches upstream's own model: needs oracle/_ref (upstream byte copy) staged")
    s, want = sample_and_upstream_eager(shape)
    model = upstream.build_model(_weights(), SHAPES[shape], DEV)
    restore = dropin.patch(model, hotpath.CudaHotPath("bf16x3", conv2d_precision="bf16x3"))
    got = model(s["imgs"], s["proj_matrices"], s["depth_values"])
    check_outputs(got, want, "dropin.patch[{} bf16x3, conv2d bf16x3]".format(shape))
    restore()


def test_cascade_bf16x3_graph_replay_equals_eager(monkeypatch):
    """TF32 off, stages 2 and 3 forced onto the bf16x3 kernel (640x512x5): a CUDA-graph replay reproduces the eager forward bit for bit"""
    from effimvs_b200 import hotpath, synthetic
    from util import dtu_model
    monkeypatch.setenv("EFFIMVS_CONV2D", "1")            # below the minimum pixel count too; the 1/8 stage (96 -> 96) stays on cuDNN
    s = synthetic.make_sample("plumbing", seed=5, device=DEV)
    model = dtu_model(hotpath.CudaHotPath("bf16x3", native_projection=True, conv2d_precision="bf16x3"), DEV, "48,8,8")
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


def test_one_block_alternating_precisions_equals_fresh_blocks(monkeypatch):
    """one block run alternately under the fp16 kernel (CudaHotPath(), TF32 on) and the bf16x3 kernel (TF32 off) gives, each
    time, bit for bit what a fresh block gives under that hot path: its packed weight images are kept per precision"""
    from effimvs_b200 import hotpath
    monkeypatch.setenv("EFFIMVS_CONV2D", "auto")
    blk, args = _block_inputs(16, 4, 592, 800)
    fresh = copy.deepcopy(blk)
    hp16, hp3 = hotpath.CudaHotPath(), hotpath.CudaHotPath(conv2d_precision="bf16x3")
    want16 = _run_block(copy.deepcopy(fresh), hp16, args, tf32=True)
    want3 = _run_block(copy.deepcopy(fresh), hp3, args)
    assert not all(torch.equal(a, b) for a, b in zip(want16, want3))
    for _ in range(2):
        assert all(torch.equal(a, b) for a, b in zip(_run_block(blk, hp16, args, tf32=True), want16))
        assert all(torch.equal(a, b) for a, b in zip(_run_block(blk, hp3, args), want3))
