"""Shared helpers for the GPU parity tests."""
import torch

from conftest import cfg1_shapes, golden_state_dict, load_golden  # noqa: F401
from oracle import hypernerf_oracle as orc
from oracle import ref_loader

EXTRA = dict(nerf_alpha=None, warp_alpha=None, hyper_alpha=None, hyper_sheet_alpha=None)
EMB = {'warp': list(range(100)), 'camera': [0], 'appearance': list(range(100)), 'time': list(range(100))}

# saved-activation slab map (hn_mlp_program.h make_slabs, cfg-1 shape), in 8-column chunks
TILE_ROWS = 256   # stash granularity: CTA tiles of 256 rows
X_IN_WS, X_HWS, X_IN_T, X_T, X_BOTT, X_IN_V, X_R, X_TOTAL = 0, 10, 154, 166, 454, 470, 476, 540


def make_model(n_fine=64, noise_std=1.0, sd=None, device="cuda"):
    from hypernerf_torch_b200.models import NerfModel
    kw = ref_loader.cfg1_kwargs(n_fine=n_fine, noise_std=noise_std)
    m = NerfModel(EMB, **kw)
    if sd is not None:
        m.load_state_dict(sd)
    return m.to(device)


def to_dev(sd, device="cuda"):
    return {k: v.to(device) for k, v in sd.items()}


def decode_slab(saved, n_rows, chunk0, ncols, total_chunks=X_TOTAL):
    """uint8 stash -> (n_rows, ncols) fp32 of the slab starting at chunk0 (layout: [half tile][chunk][64 rows][8])."""
    halves = (n_rows + TILE_ROWS - 1) // TILE_ROWS * (TILE_ROWS // 64)   # whole CTA tiles; the gate words follow the X slabs
    v = saved[:halves * total_chunks * 1024].view(torch.bfloat16).view(halves, total_chunks, 64, 8)
    x = v[:, chunk0:chunk0 + ncols // 8]                      # (halves, c, 64, 8)
    x = x.permute(0, 2, 1, 3).reshape(halves * 64, ncols)
    return x[:n_rows].float()


def oracle_layers(sd, level, points, viewdirs, ids):
    """Per-layer fp32 activations of the reference arithmetic (for localising a wrong layer)."""
    import torch.nn.functional as F
    B, S, _ = points.shape
    taps = {}
    embed = sd["warp_embed.embed.weight"][ids.reshape(-1)][:, None, :].expand(B, S, 8)
    in_w = torch.cat([orc.posenc_orig(points, 10), embed], -1)
    in_s = torch.cat([orc.posenc_orig(points, 7), embed], -1)
    taps['in_w'] = in_w

    def run(prefix, x, depth, tag):
        inputs = x
        for i in range(depth):
            x = F.relu(F.linear(x, sd[f"{prefix}.linears.{i}.weight"], sd[f"{prefix}.linears.{i}.bias"]))
            taps[f"{tag}{i}"] = x
            if i == 4:
                x = torch.cat([x, inputs], -1)
        return F.linear(x, sd[f"{prefix}.logit_layer.weight"], sd[f"{prefix}.logit_layer.bias"])

    dw = run("warp_field.mlp", in_w, 6, "warp")
    hy = run("hyper_sheet_mlp.mlp", in_s, 6, "sheet")
    wp = torch.cat([points + dw, hy], -1)
    taps['warped'] = wp
    feat = torch.cat([orc.posenc_orig(wp[..., :3], 10), orc.posenc_orig(wp[..., 3:], 6)], -1)
    taps['in_t'] = feat
    pre = "nerf_mlps_fine" if level == 1 else "nerf_mlps_coarse"
    t = F.relu(run(f"{pre}.trunk_mlp", feat, 8, "t"))
    taps['t8'] = t
    bott = F.linear(t, sd[f"{pre}.bottleneck_mlp.weight"], sd[f"{pre}.bottleneck_mlp.bias"])
    taps['bott'] = bott
    cond = orc.posenc_orig(viewdirs, 6)[:, None, :].expand(B, S, 39)
    taps['in_v'] = cond
    x = torch.cat([bott, cond], -1)
    for i in range(4):
        x = F.relu(F.linear(x, sd[f"{pre}.rgb_mlp.linears.{i}.weight"], sd[f"{pre}.rgb_mlp.linears.{i}.bias"]))
        taps[f"r{i}"] = x
    return taps


def rel_err(a, b):
    return ((a - b).norm() / (b.norm() + 1e-20)).item()


def gates_from_stash(saved, B, S):
    """ReLU gates (activation > 0) of every hidden layer, decoded from the kernels' own activation stash, so the
    oracle can differentiate through exactly the gates hn_mlp_bwd uses."""
    n = B * S

    def gate(chunk, ncols, lo=0, hi=None):
        x = decode_slab(saved, n, chunk, ncols)[:, lo:hi]
        return (x > 0).reshape(B, S, -1)

    return {
        'warp': [gate(X_HWS + 24 * l, 192, 0, 128) for l in range(6)],
        'sheet': [gate(X_HWS + 24 * l, 192, 128, 192) for l in range(6)],
        'trunk': [gate(X_T + 32 * l, 256) for l in range(9)],
        'rgb': [gate(X_R + 16 * l, 128) for l in range(4)],
    }
