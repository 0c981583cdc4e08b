"""Host-side (stock PyTorch) network pieces: algebraic rewrites must equal the plain upstream form."""
import pytest
import torch

import effimvs_b200  # noqa: F401
from effimvs_b200 import net


def _randomise_bn(mod):
    for m in mod.modules():
        if isinstance(m, torch.nn.BatchNorm2d):
            m.running_mean.normal_()
            m.running_var.uniform_(0.5, 2.0)
            m.weight.data.normal_()
            m.bias.data.normal_()


@pytest.mark.parametrize("chans,heads", [((8, 16, 32, 64), (32, 16, 8)), ((4, 8, 16, 32), (60, 40, 20))])
@pytest.mark.parametrize("fmt", [torch.contiguous_format, torch.channels_last])
def test_fused_topdown_equals_upstream_form(chans, heads, fmt):
    """FeaturePyramid's fused top-down path (sub-pixel head, composed lateral conv, bias map, addmm
    lateral) against the literal upstream sequence (models/module.py:395-410), incl. odd borders."""
    torch.manual_seed(0)
    f = net.FeaturePyramid(chans, heads).eval()
    _randomise_bn(f)
    x = torch.randn(2, 3, 64, 96).contiguous(memory_format=fmt)
    with torch.no_grad():
        f.fused_topdown = False
        want = f(x)
        f.fused_topdown = True
        got = f(x)
    for w, g in zip(want, got):
        assert w.shape == g.shape
        assert float((w - g).abs().max()) <= 2e-5 * float(w.abs().max())


def test_fused_topdown_cache_follows_weight_updates():
    torch.manual_seed(1)
    f = net.FeaturePyramid((4, 8, 16, 32), (12, 8, 4)).eval()
    x = torch.randn(1, 3, 32, 32)
    with torch.no_grad():
        f.fused_topdown = True
        a = f(x)[2].clone()
        f.out3.weight.mul_(2.0)
        f.inner2.bias.add_(1.0)
        b = f(x)[2]
        f.fused_topdown = False
        want = f(x)[2]
    assert float((b - want).abs().max()) <= 2e-5 * float(want.abs().max())
    assert float((a - want).abs().max()) > 1e-3


def _update_cost_fn(depth, _iteration=0):
    """the analytic cost function tests/golden/make_golden_update.py used in place of the volume lookup"""
    k = torch.arange(1, 7, dtype=depth.dtype, device=depth.device).reshape(1, 6, 1, 1)
    return torch.sin(depth * (k * 0.01)) * 0.5


def load_update_block(g, device="cpu"):
    blk = net.UpdateBlock(16, 6, 2, 4).eval()
    blk.load_state_dict({k[3:].replace("__", "."): v for k, v in g.items() if k.startswith("w__")}, strict=True)
    return blk.to(device)


def test_update_block_matches_upstream_golden():
    """net.UpdateBlock / convex_upsample / to_depth (the stock-PyTorch host side) replay upstream's
    BasicUpdateBlock, upsample_depth and disp_to_depth bit for bit on CPU."""
    from util import golden
    g = golden("update_block")
    blk = load_update_block(g)
    lo, hi = 1.0 / g["dmax"], 1.0 / g["dmin"]
    to_depth = lambda inv: 1.0 / (lo + (hi - lo) * inv).clamp(min=1e-4)   # noqa: E731
    # the last bits of ATen's CPU convolution and softmax depend on how the intra-op thread count splits the work; the
    # golden was written with a few threads (with torch 2.11: 2 to 5, 7 and 8 reproduce it, with AVX2 and AVX-512 kernels
    # alike; 1 or 16 do not -- a torch that splits the work differently may need another count)
    threads = torch.get_num_threads()
    torch.set_num_threads(4)
    try:
        with torch.no_grad():
            n, mask, invs = blk(g["net0"], _update_cost_fn, g["inv0"], g["context"], 3, to_depth)
            up = net.convex_upsample(invs[-1], mask, 2)
    finally:
        torch.set_num_threads(threads)
    assert torch.equal(n, g["net"]) and torch.equal(mask, g["mask"]) and torch.equal(up, g["up"])
    for i in range(3):
        assert torch.equal(invs[i], g["inv{}".format(i + 1)])
        assert torch.equal(to_depth(invs[i]), g["depth{}".format(i + 1)])
    assert torch.equal(to_depth(up.unsqueeze(1)).squeeze(1), g["depth_up"])


@pytest.mark.parametrize("use_ctx_map", [False, True])
@pytest.mark.parametrize("want_mask", [False, True])
def test_fused_update_wiring_equals_plain_block(use_ctx_map, want_mask, monkeypatch):
    """net.update_block_forward_fused (merged gate convolution, block-diagonal encoder layer, context term inside the
    tail kernel, delta head, optional mask fold) wired to a plain-torch glue table equals UpdateBlock.forward +
    convex_upsample + disp_to_depth -- every host-side code path, on CPU."""
    from util import TorchGlue, golden
    g = golden("update_block")
    blk = load_update_block(g)
    torch.manual_seed(5)
    B, _, H, W = g["inv0"].shape
    ctx_map = torch.randn(B, 20, H, W)
    net0, context = torch.tanh(ctx_map[:, :16]), torch.relu(ctx_map[:, 16:])
    lo, hi = (1.0 / g["dmax"]).reshape(B), (1.0 / g["dmin"]).reshape(B)
    to_depth = lambda inv: 1.0 / (lo.reshape(B, 1, 1, 1) + (hi - lo).reshape(B, 1, 1, 1) * inv).clamp(min=1e-4)   # noqa: E731
    monkeypatch.setenv("EFFIMVS_UPSAMPLE_CONV", "1")       # exercise the folded mask head when no mask is wanted
    with torch.no_grad():
        n_w, mask_w, invs_w = blk(net0, _update_cost_fn, g["inv0"], context, 3, to_depth)
        up_w = net.convex_upsample(invs_w[-1], mask_w, 2)
        args = (None, _update_cost_fn, g["inv0"], None, 3, lo, hi, ctx_map) if use_ctx_map else \
               (net0, _update_cost_fn, g["inv0"], context, 3, lo, hi, None)
        n, invs, deps, up, dup, mask_pre = blk.forward_fused(TorchGlue, *args, want_mask=want_mask)
    close = lambda a, b: float((a - b).abs().max()) <= 1e-5 * max(1.0, float(b.abs().max()))   # noqa: E731
    assert close(n, n_w) and close(up, up_w) and close(dup, to_depth(up_w.unsqueeze(1)).squeeze(1))
    for i in range(3):
        assert close(invs[i], invs_w[i]) and close(deps[i], to_depth(invs_w[i]))
    if want_mask:
        assert close(0.25 * (mask_pre + blk.mask[2].bias.detach().reshape(1, -1, 1, 1)), mask_w)
    else:
        assert mask_pre is None


def test_feature_cache_equals_reencoding():
    """forward_from_features on per-image encodings (SURVEY section 8(f) row 1) equals forward() on the stacked views"""
    import types
    from effimvs_b200 import synthetic
    from oracle import hotpath as ohp
    from util import load_dtu_weights
    m = net.EffiMVSPlus(types.SimpleNamespace(ndepths="8,4,4", GRUiters="1,1,1", CostNum=3), hotpath=ohp.OracleHotPath())
    load_dtu_weights(m)
    m.eval()
    s = synthetic.make_sample("plumbing", seed=3, width=96, height=64, views=3)
    with torch.no_grad():
        want = m(s["imgs"], s["proj_matrices"], s["depth_values"])
        per_view = [[st[0] for st in m.encode(s["imgs"][:, v:v + 1])] for v in range(3)]
        feats = [[pv[k] for pv in per_view] for k in range(3)]
        got = m.forward_from_features(feats, s["imgs"][:, 0], s["proj_matrices"], s["depth_values"])
    for a, b in zip(want["depth"], got["depth"]):
        assert float((a - b).abs().max()) <= 1e-2      # mm at ~600 mm: batch-1 vs batch-3 convolution rounding
    assert float((want["photometric_confidence"] - got["photometric_confidence"]).abs().max()) <= 1e-5


def test_workspace_cache_keeps_one_buffer_per_key_and_evicts_least_recently_used():
    """hotpath._WorkspaceCache: the persistent regularization workspaces (one per network, shape, precision, device)"""
    from effimvs_b200 import hotpath
    c = hotpath._WorkspaceCache(cap=3)
    a = c.get(("costreg", 1), 1000, "cpu")
    assert a["ws"].numel() >= 1000 and a["ws"].dtype == torch.uint8 and a["stamp"] is None
    a["stamp"] = "prepared"
    assert c.get(("costreg", 1), 1000, "cpu") is a                   # same key: same buffer, stamp kept
    assert c.get(("costreg", 1), 5000, "cpu") is not a               # a larger request replaces it (unprepared)
    assert c.get(("costreg", 1), 5000, "cpu")["stamp"] is None
    for k in (2, 3):
        c.get(("cost_up", k), 10, "cpu")
    c.get(("costreg", 1), 10, "cpu")                                 # touch -> most recently used
    c.get(("cost_up", 4), 10, "cpu")                                 # evicts ("cost_up", 2)
    assert set(c._store) == {("costreg", 1), ("cost_up", 3), ("cost_up", 4)}


def test_encoder_head_host_table_cache(monkeypatch):
    """ops._encoder_head_table: the host-side weight tables of the constant-bank encoder head are cached by the identity and
    version of the four weight tensors, rebuilt after an in-place update, and never built while a stream is capturing (a miss
    there returns None = the kernel that reads the weights from device memory)."""
    from effimvs_b200 import ops
    capturing = [False]
    monkeypatch.setattr(torch.cuda, "is_current_stream_capturing", lambda: capturing[0])
    monkeypatch.setattr(ops, "_EH_TABLES", {})
    h, CD = 16, 6
    gen = torch.Generator().manual_seed(2)
    ws = (torch.randn(h, CD, 1, 1, generator=gen), torch.randn(h, generator=gen), torch.randn(h, 1, 7, 7, generator=gen),
          torch.randn(h, generator=gen))
    t0 = ops._encoder_head_table(ws, CD, h)
    assert t0.shape == (944,) and torch.equal(t0[:784].reshape(49, 16), ws[2][:, 0].reshape(16, 49).t())
    assert ops._encoder_head_table(ws, CD, h) is t0                       # same tensors, same versions: the cached table
    capturing[0] = True
    assert ops._encoder_head_table(ws, CD, h) is t0                       # a hit needs no copy, so it is fine under capture
    ws[2].mul_(2.0)                                                       # in-place update bumps the version
    assert ops._encoder_head_table(ws, CD, h) is None                     # miss under capture: no device -> host copy there
    capturing[0] = False
    t1 = ops._encoder_head_table(ws, CD, h)
    assert t1 is not t0 and torch.equal(t1[:784].reshape(49, 16), ws[2][:, 0].reshape(16, 49).t())
    fresh = tuple(w.clone() for w in ws)                                  # other tensor objects with the same values: their own entry
    t2 = ops._encoder_head_table(fresh, CD, h)
    assert t2 is not t1 and torch.equal(t2, t1)
    assert ops._encoder_head_table(ws, CD, h) is t1
