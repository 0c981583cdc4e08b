"""Shared helpers for the tests: golden-fixture loading and module reconstruction."""
import os
import types

import numpy as np
import torch
import torch.nn.functional as F

import effimvs_b200  # noqa: F401
from effimvs_b200 import net

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def golden(name, device="cpu"):
    z = np.load(os.path.join(GOLDEN, name + ".npz"))
    return {k: torch.from_numpy(z[k]).to(device) if z[k].ndim else z[k].item() for k in z.files}


def load_module(mod, arrays, prefix, device="cpu"):
    sd = {k[len(prefix):].replace("__", "."): v for k, v in arrays.items() if k.startswith(prefix)}
    missing = mod.load_state_dict(sd, strict=False)
    assert not [k for k in missing.missing_keys if "num_batches" not in k], missing
    assert not missing.unexpected_keys, missing
    return mod.to(device).eval()


def regnet(arrays, device="cpu"):
    return load_module(net.RegNet3D(1, 8), arrays, "reg__", device)


def cspnet(arrays, device="cpu"):
    return load_module(net.CrossScaleNet3D(1, 8), arrays, "csp__", device)


def pixelwise(arrays, device="cpu"):
    m = torch.nn.Sequential(net.ConvBNReLU2d(1, 16, 3, 1, 1), net.ConvBNReLU2d(16, 16, 3, 1, 1),
                            net.ConvBNReLU2d(16, 8, 3, 1, 1), torch.nn.Conv2d(8, 1, 1), torch.nn.Sigmoid())
    return load_module(m, arrays, "pwn__", device)


def dtu_model(hotpath, device="cpu", ndepths="48,8,8"):
    args = types.SimpleNamespace(ndepths=ndepths, GRUiters="3,3,3", CostNum=3)
    m = net.EffiMVSPlus(args, hotpath=hotpath)
    load_dtu_weights(m)
    return m.to(device).eval()


def load_dtu_weights(m):
    sd = torch.load(os.path.join(GOLDEN, "dtu_weights.pt"), map_location="cpu")
    full = dict(sd)
    for k, v in sd.items():          # re-create upstream's duplicate registrations
        for a, b in (("update_block_depth1.", "update_block.0."), ("update_block_depth2.", "update_block.1."),
                     ("update_block_depth3.", "update_block.2."), ("CSP_R1.", "CSP_R.0."), ("CSP_R2.", "CSP_R.1."),
                     ("CSP_C1.", "CSP_C.0."), ("CSP_C2.", "CSP_C.1.")):
            if k.startswith(a):
                full[b + k[len(a):]] = v
    res = m.load_state_dict(full, strict=False)
    assert not res.unexpected_keys and all("num_batches" in k for k in res.missing_keys), res


def headline_sample(depths, conf, k=1024):
    """A fixed sample of k pixels of each of the 13 depth maps and of the confidence map (flat indices i * 2654435761 mod n,
    distinct for k <= n since the multiplier is prime) -> 14 float32 arrays; what tests/golden/headline_port.npz stores."""
    out = []
    for t in list(depths) + [conf]:
        flat = t.detach().reshape(-1).float().cpu().numpy()
        out.append(flat[(np.arange(k, dtype=np.int64) * 2654435761) % flat.size])
    return out


def rel_max(a, b):
    """max|a-b| / max|b|  -- the north_star's cost-volume metric (SURVEY.md section 7 'hard parts')."""
    return float((a - b).abs().max() / b.abs().max().clamp(min=1e-30))


class TorchGlue:
    """Plain-torch stand-in for the update-block glue entries of the hot-path table (CudaHotPath.gru_init ...
    convex_upsample_conv): test infrastructure for the host-side wiring of net.update_block_forward_fused on CPU."""

    @staticmethod
    def _to_depth(inv, lo, hi):
        lo, hi = lo.reshape(-1, 1, 1, 1), hi.reshape(-1, 1, 1, 1)
        return 1.0 / (lo + (hi - lo) * inv).clamp(min=1e-4)

    @staticmethod
    def gru_init(ctx_map, h):
        B, _, H, W = ctx_map.shape
        hx = torch.full((B, 2 * h, H, W), float("nan"))
        hx[:, :h] = torch.tanh(ctx_map[:, :h])
        return hx

    @staticmethod
    def inv_init(cur_depth, lo, hi):
        l, hh = lo.reshape(-1, 1, 1, 1), hi.reshape(-1, 1, 1, 1)
        inv = (cur_depth.reciprocal() - l) / ((hh - l) + 1e-10)
        return inv, TorchGlue._to_depth(inv, lo, hi)

    @staticmethod
    def gru_init_ctx(ctx_map, h, w_ctx, bias):
        w4 = w_ctx.reshape(w_ctx.shape[0], -1, 1, 1)
        return TorchGlue.gru_init(ctx_map, h), F.conv2d(torch.relu(ctx_map[:, h:]), w4, bias)

    @staticmethod
    def encoder_head(cost, inv, wc1, bc1, wd1, bd1):
        return torch.cat([torch.relu(F.conv2d(cost, wc1, bc1)), torch.relu(F.conv2d(inv, wd1, bd1, padding=3))], dim=1)

    @staticmethod
    def encoder_tail(m, w, ctx_term, hx):
        h = ctx_term.shape[1]
        hx[:, h:] = torch.relu(F.conv2d(m, w) + ctx_term)

    @staticmethod
    def encoder_tail_ctx(m, w_m, ctx, ctx_offset, cx, ctx_relu, w_ctx, bias, hx):
        h = w_m.shape[0]
        c = ctx[:, ctx_offset:ctx_offset + cx]
        c = torch.relu(c) if ctx_relu else c
        hx[:, h:] = torch.relu(F.conv2d(m, w_m) + F.conv2d(c, w_ctx, bias))

    @staticmethod
    def gru_reset(zr_pre, bias_r, hx):
        h = zr_pre.shape[1] // 2
        out = hx.clone()
        out[:, :h] = torch.sigmoid(zr_pre[:, h:] + bias_r.reshape(1, -1, 1, 1)) * hx[:, :h]
        return out

    @staticmethod
    def gru_update(zr_pre, bias_z, q_pre, bias_q, hx):
        h = q_pre.shape[1]
        z = torch.sigmoid(zr_pre[:, :h] + bias_z.reshape(1, -1, 1, 1))
        net_new = (1 - z) * hx[:, :h] + z * torch.tanh(q_pre + bias_q.reshape(1, -1, 1, 1))
        hx[:, :h] = net_new
        return net_new.clone()

    @classmethod
    def gru_delta(cls, pre, bias, inv, lo, hi):
        new = inv.clone() if pre is None else inv + torch.tanh(pre + bias.reshape(1, -1, 1, 1))
        return new, cls._to_depth(new, lo, hi)

    @classmethod
    def delta_head(cls, t, weight, bias, inv, lo, hi):
        new = inv + torch.tanh(F.conv2d(t, weight, bias, padding=1))
        return new, cls._to_depth(new, lo, hi)

    @classmethod
    def convex_upsample(cls, mask_pre, mask_bias, scale, inv, lo, hi, ratio):
        mask = mask_pre if mask_bias is None else mask_pre + mask_bias.reshape(1, -1, 1, 1)
        up = net.convex_upsample(inv, scale * mask, ratio)
        return up, cls._to_depth(up.unsqueeze(1), lo, hi).squeeze(1)

    @classmethod
    def convex_upsample_conv(cls, t, mask_w, mask_bias, scale, inv, lo, hi, ratio):
        return cls.convex_upsample(F.conv2d(t, mask_w), mask_bias, scale, inv, lo, hi, ratio)
