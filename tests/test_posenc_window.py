"""Annealed positional encodings: the `extra_params` alphas (warp_alpha, hyper_sheet_alpha, nerf_alpha, hyper_alpha)
window the encoding bands of the warp field, the hyper sheet and both levels' trunks, as in Nerfies / HyperNeRF:
w_k(alpha) = 0.5 (1 - cos(pi clamp(alpha - k, 0, 1))) on band k's sin / cos columns.

The reference passes the alphas through its API and ignores them (its posenc window is commented out), so there is no
reference output to pin this to.  The windowed restatement here is the oracle run on a state dict whose encoded weight
columns are scaled by w: W (w . pe) = (W diag(w)) pe, which is also how the kernels apply the window.  The CPU tests
check that identity and the column-to-band mapping against the oracle's own encoders."""
import ctypes as C
import math

import pytest
import torch

from oracle import hypernerf_oracle as orc
from oracle import ref_loader
from hypernerf_torch_b200 import _lib, _packing

INF = float('inf')
DEV = "cuda"


def window(alpha, n_freqs, channels, identity, dtype=torch.float64):
    """Per-column window of posenc_orig (identity=True: [x, sin(2^0 x), cos(2^0 x), ...]) or of the SE3 field's
    posenc(points, 0, F) (identity=False: per scale [sin(s x), sin(s x + pi / 2)]): bands of 2 * channels columns."""
    k = torch.arange(n_freqs, dtype=dtype)
    wk = 0.5 * (1.0 - torch.cos(math.pi * torch.clamp(alpha - k, 0.0, 1.0)))
    cols = wk.repeat_interleave(2 * channels)
    return torch.cat([torch.ones(channels, dtype=dtype), cols]) if identity else cols


def window_specs(cfg, hyper_dim):
    """(weight name, first source column, alpha key, F, channels, identity) of every windowed column range of a
    configuration (oracle cfg dict), in the reference's state-dict names."""
    specs = []
    if cfg.get('use_warp', True):
        if cfg.get('warp_field', 'translation') == 'se3':
            for l, c in ((0, 0), (5, 128)):
                specs.append((f"warp_field.trunk.linears.{l}.weight", c, 'warp_alpha', 8, 3, False))
        else:
            for l, c in ((0, 0), (5, 128)):
                specs.append((f"warp_field.mlp.linears.{l}.weight", c, 'warp_alpha', 10, 3, True))
        if cfg.get('slice', 'bendy_sheet') == 'bendy_sheet':
            for l, c in ((0, 0), (5, 64)):
                specs.append((f"hyper_sheet_mlp.mlp.linears.{l}.weight", c, 'hyper_sheet_alpha', 7, 3, True))
    pe_x = 3 * (1 + 2 * cfg['xyz_freq'])
    for lvl in ("coarse", "fine"):
        for l, c in ((0, 0), (5, 256)):
            name = f"nerf_mlps_{lvl}.trunk_mlp.linears.{l}.weight"
            specs.append((name, c, 'nerf_alpha', cfg['xyz_freq'], 3, True))
            if cfg.get('use_warp', True):
                specs.append((name, c + pe_x, 'hyper_alpha', cfg['hyper_freq'], hyper_dim, True))
    return specs


def windowed_sd(sd, cfg, hyper_dim, extra_params):
    """The state dict with every encoded weight column scaled by its window (differentiable: autograd through it gives
    dW = (dY^T pe) . w).  Unset alphas leave their columns alone."""
    out = dict(sd)
    for name, c, key, F, ch, ident in window_specs(cfg, hyper_dim):
        a = (extra_params or {}).get(key)
        if a is None or name not in out:
            continue
        W = out[name]
        w = window(float(a), F, ch, ident, dtype=W.dtype).to(W.device)
        scale = torch.ones(W.shape[1], dtype=W.dtype, device=W.device)
        scale[c:c + w.numel()] = w
        out[name] = W * scale
    return out


# ---------------------------------------------------------------------------------------------------------- CPU
def test_window_values():
    for F in (6, 7, 8, 10):
        assert torch.equal(window(0.0, F, 1, False), torch.zeros(2 * F, dtype=torch.float64))
        assert torch.equal(window(-3.0, F, 1, False), torch.zeros(2 * F, dtype=torch.float64))
        assert torch.equal(window(float(F), F, 1, False), torch.ones(2 * F, dtype=torch.float64))
        assert torch.equal(window(INF, F, 1, False), torch.ones(2 * F, dtype=torch.float64))
        for k in range(F):
            w = window(k + 0.5, F, 1, False).view(F, 2)[:, 0]
            assert torch.allclose(w[k], torch.tensor(0.5, dtype=torch.float64), atol=1e-15)
            assert torch.equal(w[:k], torch.ones(k, dtype=torch.float64))
            assert torch.equal(w[k + 1:], torch.zeros(F - k - 1, dtype=torch.float64))
    # float32, as the kernels evaluate it: cos(pi) rounds to -1, so alpha >= F is exactly the unwindowed encoding
    assert torch.equal(window(10.0, 10, 3, True, dtype=torch.float32), torch.ones(63))


def test_column_bands_follow_the_encoders():
    """window() maps columns to bands the way the oracle's posenc_orig / posenc_scaled lay them out: windowing each band
    of the encoder output is the same as multiplying the encoding by the column window."""
    x = torch.randn(7, 3, dtype=torch.float64)
    a = 3.3
    for F in (7, 10):
        k = torch.arange(F, dtype=torch.float64)
        wk = 0.5 * (1.0 - torch.cos(math.pi * torch.clamp(a - k, 0.0, 1.0)))
        banded = torch.cat([x] + [t for i in range(F) for t in (wk[i] * torch.sin(2. ** i * x),
                                                                  wk[i] * torch.cos(2. ** i * x))], -1)
        assert torch.allclose(orc.posenc_orig(x, F) * window(a, F, 3, True), banded, atol=1e-14)
    h = torch.randn(7, 8, dtype=torch.float64)        # the hyper point: H channels per band half
    w = window(a, 6, 8, True)
    assert torch.allclose((orc.posenc_orig(h, 6) * w)[:, 8 + 2 * 8 * 3:8 + 2 * 8 * 4], 0.5 * (1 - math.cos(math.pi * 0.3)) *
                          orc.posenc_orig(h, 6)[:, 8 + 2 * 8 * 3:8 + 2 * 8 * 4], atol=1e-14)
    assert torch.all(w[8 + 2 * 8 * 4:] == 0) and torch.all(w[:8 + 2 * 8 * 3] == 1)
    pe = orc.posenc_scaled(x.float(), 0, 8).double()
    scales = 2. ** torch.linspace(0, 8, steps=8, dtype=torch.float64)
    ws = window(a, 8, 3, False)
    for i in range(8):                                  # scale i = band i: 6 columns, [sin(s x) | sin(s x + pi / 2)]
        assert torch.all(ws[6 * i:6 * i + 6] == ws[6 * i])
        assert torch.allclose(pe[:, 6 * i:6 * i + 3], torch.sin(scales[i] * x), atol=1e-4)


@pytest.mark.parametrize("kind", ["bendy_h2", "axis_h8", "se3"])
def test_windowed_features_equal_scaled_weight_columns(kind):
    """The identity the kernels rest on, in fp64 on every windowed layer of a configuration: a linear layer on
    windowed encodings equals the layer with its encoded columns scaled, and autograd's dW is dW' . w with
    dW' = dY^T (unwindowed input)."""
    H = {'bendy_h2': 2, 'axis_h8': 8, 'se3': 8}[kind]
    cfg = orc.default_cfg(slice='bendy_sheet' if kind == 'bendy_h2' else 'axis_aligned_plane',
                          warp_field='se3' if kind == 'se3' else 'translation')
    ep = {'warp_alpha': 2.7, 'hyper_sheet_alpha': 1.4, 'nerf_alpha': 5.5, 'hyper_alpha': 0.6}
    g = torch.Generator().manual_seed(0)
    by_name = {}
    for name, c, key, F, ch, ident in window_specs(cfg, H):
        by_name.setdefault(name, []).append((c, window(ep[key], F, ch, ident)))
    assert by_name
    for name, parts in by_name.items():
        width = max(c + w.numel() for c, w in parts) + 8          # + GLO / padding columns that are never windowed
        col = torch.ones(width, dtype=torch.float64)
        for c, w in parts:
            col[c:c + w.numel()] = w
        W = torch.randn(32, width, dtype=torch.float64, generator=g, requires_grad=True)
        x = torch.randn(50, width, dtype=torch.float64, generator=g)
        dy = torch.randn(50, 32, dtype=torch.float64, generator=g)
        y_feat = (x * col) @ W.t()
        (gW,) = torch.autograd.grad((y_feat * dy).sum(), W)
        sd = windowed_sd({name: W}, cfg, H, ep)
        y_w = x @ sd[name].t()
        assert torch.allclose(y_feat, y_w, rtol=1e-12, atol=1e-12), name
        (gW2,) = torch.autograd.grad((y_w * dy).sum(), W)
        assert torch.allclose(gW, (dy.t() @ x) * col, rtol=1e-12, atol=1e-12), name
        assert torch.allclose(gW2, gW, rtol=1e-12, atol=1e-12), name


def test_oracle_without_alphas_is_unchanged():
    from hypernerf_torch_b200 import synthetic
    sd = synthetic.make_state_dict(synthetic.cfg1_state_dict_shapes(), seed=2, boosted=False)
    cfg = orc.default_cfg()
    B, S = 3, 16
    g = torch.Generator().manual_seed(1)
    pts = torch.randn(B, S, 3, generator=g) * 0.3
    d = torch.nn.functional.normalize(torch.randn(B, 3, generator=g), dim=-1)
    ids = torch.tensor([1, 5, 9])
    base = orc.query_fields(sd, 'fine', pts, d, ids, cfg)
    for extra in (None, dict(nerf_alpha=None, warp_alpha=None, hyper_alpha=None, hyper_sheet_alpha=None)):
        got = orc.query_fields(windowed_sd(sd, cfg, 2, extra), 'fine', pts, d, ids, cfg)
        assert all(torch.equal(a, b) for a, b in zip(got, base))
    got = orc.query_fields(windowed_sd(sd, cfg, 2, {'nerf_alpha': 2.0}), 'fine', pts, d, ids, cfg)
    assert not torch.equal(got[0], base[0])


def test_pe_alphas_parsing():
    assert _packing.pe_alphas(None) is None
    assert _packing.pe_alphas({}) is None
    assert _packing.pe_alphas(dict(nerf_alpha=None, warp_alpha=None, hyper_alpha=None, hyper_sheet_alpha=None)) is None
    assert _packing.pe_alphas({'nerf_alpha': 3}) == (INF, INF, 3.0, INF)
    assert _packing.pe_alphas({'warp_alpha': 1.5, 'hyper_sheet_alpha': torch.tensor(2.0), 'hyper_alpha': 0}) == \
        (1.5, 2.0, INF, 0.0)
    for key in _packing.PE_ALPHA_KEYS:
        with pytest.raises(ValueError, match=key):
            _packing.pe_alphas({key: float('nan')})


def test_nan_alpha_raises_before_any_launch():
    from hypernerf_torch_b200 import model_utils, synthetic
    from hypernerf_torch_b200.models import NerfModel
    model = NerfModel(ref_loader.EMBEDDINGS, **ref_loader.cfg1_kwargs())     # CPU parameters: nothing can launch
    rays, _ = synthetic.train_rays(4, seed=0)
    with pytest.raises(ValueError, match="hyper_alpha"):
        model(model_utils.prepare_ray_dict(rays), {'hyper_alpha': float('nan')})


def _desc(**over):
    kw = dict(glo_dim=8, hyper_dim=2, xyz_freqs=10, hyper_freqs=6, view_freqs=6, warp_freqs=10, sheet_freqs=7,
              num_embeddings=100, flags=3)
    kw.update(over)
    return _lib.ModelDesc(*[kw[k] for k in ("glo_dim", "hyper_dim", "xyz_freqs", "hyper_freqs", "view_freqs",
                                            "warp_freqs", "sheet_freqs", "num_embeddings", "flags")])


def test_windowed_entry_points_check_their_arguments():
    L = _lib.lib()
    for name in ("hn_pack_weights_windowed", "hn_mlp_bwd_weights_windowed", "hn_mlp_bwd_trunk_weights_windowed"):
        assert name in _lib.EXPORTS
    offs = (C.c_int64 * _lib.HN_NUM_PARAM_TENSORS)(*([0] * _lib.HN_NUM_PARAM_TENSORS))
    buf = C.c_void_p(16)          # never dereferenced: every case below fails before a launch
    assert L.hn_pack_weights_windowed(C.byref(_desc()), buf, offs, 0, buf, None, None) < 0
    assert b"pe_alpha" in L.hn_last_error()
    assert L.hn_mlp_bwd_weights_windowed(C.byref(_desc()), buf, 4, 64, 0, offs, buf, buf, None, None) < 0
    assert b"pe_alpha" in L.hn_last_error()
    assert L.hn_mlp_bwd_trunk_weights_windowed(C.byref(_desc()), buf, 4, 64, 0, offs, buf, buf, None, None) < 0
    assert b"pe_alpha" in L.hn_last_error()
    assert L.hn_pack_weights_windowed(C.byref(_desc()), buf, offs, 2, buf, buf, None) < 0          # bad level
    assert b"level" in L.hn_last_error()
    assert L.hn_pack_weights_windowed(C.byref(_desc(hyper_dim=3)), buf, offs, 0, buf, buf, None) < 0   # bad shape
    assert b"instantiated" in L.hn_last_error()
    assert L.hn_mlp_bwd_weights_windowed(C.byref(_desc()), buf, -1, 64, 0, offs, buf, buf, buf, None) < 0   # bad B
    assert L.hn_mlp_bwd_weights_windowed(C.byref(_desc()), buf, 4, 64, 0, offs, buf, None, buf, None) < 0   # no workspace
    static = _desc(flags=_lib.HN_FLAG_STATIC_NERF, view_freqs=4)
    assert L.hn_pack_weights_windowed(C.byref(static), buf, offs, 0, buf, buf, None) == -13
    assert b"static" in L.hn_last_error()


# ---------------------------------------------------------------------------------------------------------- GPU
CONFIGS = {
    'bendy_h2': dict(hyper_slice_method='bendy_sheet', hyper_slice_out_dim=2),
    'bendy_h4': dict(hyper_slice_method='bendy_sheet', hyper_slice_out_dim=4),     # trunk input in ACT (FE_SKIPFEED)
    'axis_h8': dict(hyper_slice_method='axis_aligned_plane', hyper_slice_out_dim=8),
    'nowarp': dict(use_warp=False),
    'se3_axis': dict(hyper_slice_method='axis_aligned_plane', hyper_slice_out_dim=8, warp_field_type='se3'),
}
ALPHAS = {
    'zero': dict(warp_alpha=0.0, hyper_sheet_alpha=0.0, nerf_alpha=0.0, hyper_alpha=0.0),
    'fractional': dict(warp_alpha=3.5, hyper_sheet_alpha=2.25, nerf_alpha=6.5, hyper_alpha=1.5),
    'full': dict(warp_alpha=10.0, hyper_sheet_alpha=7.0, nerf_alpha=10.0, hyper_alpha=6.0),
}


def _model(conf, n_fine=64, stratified=True, seed=0):
    from hypernerf_torch_b200 import synthetic
    from hypernerf_torch_b200.models import NerfModel
    kw = ref_loader.cfg1_kwargs(n_fine=n_fine, noise_std=None)
    kw.update(CONFIGS[conf])
    model = NerfModel(ref_loader.EMBEDDINGS, **kw)
    model.load_state_dict(synthetic.make_state_dict(model, seed=seed, boosted=False))
    model = model.to(DEV)
    model.use_stratified_sampling = stratified
    return model, kw


def _forward(model, rays, draws, extra):
    from hypernerf_torch_b200 import model_utils
    with ref_loader._DrawTape(draws):
        return model(model_utils.prepare_ray_dict(rays), extra)


@pytest.mark.gpu
@pytest.mark.parametrize("alphas", list(ALPHAS))
@pytest.mark.parametrize("conf", list(CONFIGS))
def test_windowed_forward_matches_oracle(conf, alphas):
    from hypernerf_torch_b200 import synthetic
    model, kw = _model(conf)
    B = 48
    rays, _ = synthetic.train_rays(B, seed=4, device=DEV)
    g = torch.Generator(device=DEV).manual_seed(3)
    u_c, u_f = torch.rand(B, 64, device=DEV, generator=g), torch.rand(B, 64, device=DEV, generator=g)
    extra = ALPHAS[alphas]
    cfg = orc.cfg_from_kwargs(kw)
    sd = {k: v.detach() for k, v in model.state_dict().items()}
    with torch.no_grad():
        out = _forward(model, rays, [u_c, u_f], dict(extra))
        ref = orc.forward(windowed_sd(sd, cfg, kw['hyper_slice_out_dim'], extra), rays[:, :3], rays[:, 3:6],
                          rays[:, 8].long(), {'u_coarse': u_c, 'u_fine': u_f}, cfg)
    for lvl in ("coarse", "fine"):
        for k in ("rgb", "depth", "acc", "weights"):
            err = (out[lvl][k] - ref[lvl][k]).abs().max().item()
            print(f"{conf} {alphas} {lvl} {k} max_abs_err {err:.3e}")
            assert err < 2e-3, (lvl, k, err)


def _flat_grad(model, rays, rgbs, draws, extra):
    from hypernerf_torch_b200 import losses
    from hypernerf_torch_b200 import train as hn_train
    fg = hn_train.FlatGrads(model.parameters())
    model.attach_flat_grads(fg)
    fg.zero()
    out = _forward(model, rays, draws, extra)
    loss, _ = losses.mse_coarse_fine(out, rgbs, global_count=3.0 * rays.shape[0])
    loss.backward()
    model.attach_flat_grads(None)
    return out, fg


@pytest.mark.gpu
@pytest.mark.parametrize("conf", ["bendy_h2", "se3_axis"])
def test_no_alphas_and_infinite_alphas_run_the_unwindowed_numbers(conf):
    """All alphas None, no extra_params at all, and the windowed entry points at +inf: the same outputs bit for bit
    (w = 1 exactly packs the same bf16 images) and the same flat gradient; the weight-gradient kernel reduces with fp32
    atomics in an unspecified order, so the gradients are compared to that order's noise."""
    from hypernerf_torch_b200 import synthetic
    model, _ = _model(conf)
    B = 64
    rays, rgbs = synthetic.train_rays(B, seed=6, device=DEV)
    g = torch.Generator(device=DEV).manual_seed(8)
    draws = [torch.rand(B, 64, device=DEV, generator=g), torch.rand(B, 64, device=DEV, generator=g)]
    runs = []
    for extra in (dict(nerf_alpha=None, warp_alpha=None, hyper_alpha=None, hyper_sheet_alpha=None), {}, None,
                  dict(nerf_alpha=INF, warp_alpha=INF, hyper_alpha=INF, hyper_sheet_alpha=INF)):
        out, fg = _flat_grad(model, rays, rgbs, draws, extra)
        runs.append((out, fg.flat.clone()))
    for out, flat in runs[1:]:
        for lvl in ("coarse", "fine"):
            for k in ("rgb", "depth", "acc", "weights", "warped_points"):
                assert torch.equal(out[lvl][k], runs[0][0][lvl][k]), (lvl, k)
        rel = ((flat - runs[0][1]).norm() / runs[0][1].norm()).item()
        assert rel < 1e-5, rel


@pytest.mark.gpu
@pytest.mark.parametrize("level", [0, 1])
def test_windowed_parameter_gradients(level):
    """Per-tensor gradients of the fused network with windows against autograd of the bf16-emulated oracle on the
    windowed state dict, through the kernels' own ReLU gates (as tests/test_mlp.py does without windows); the
    weight-gradient columns of bands whose window is 0 are exactly zero."""
    import helpers as H
    from hypernerf_torch_b200 import synthetic
    from hypernerf_torch_b200.models import _FusedMlp
    B, S = 6, 64
    sd = synthetic.make_state_dict(H.cfg1_shapes(), seed=5, boosted=True)
    model = H.make_model(sd=sd)
    sd = H.to_dev(sd)
    rays, _ = synthetic.train_rays(B, seed=6)
    rays = rays.to(DEV)
    o, d, ids = rays[:, :3].contiguous(), rays[:, 3:6].contiguous(), rays[:, 8].long()
    g = torch.Generator(device=DEV).manual_seed(5)
    z, _ = torch.sort(torch.rand(B, S, device=DEV, generator=g), -1)
    pts = (o[:, None, :] + z[..., None] * d[:, None, :]).contiguous()
    extra = ALPHAS['fractional']
    params = model._canonical_params()
    names = [k for k, _ in model.named_parameters()]
    gs = torch.randn(B, S, device=DEV, generator=g)
    gr = torch.randn(B, S, 3, device=DEV, generator=g)
    gw = torch.randn(B, S, 5, device=DEV, generator=g) * 0.1
    sigma, rgb, warped = _FusedMlp.apply(model, (level, _packing.pe_alphas(extra)), pts, d, ids, None, 0.0, *params)
    gates = H.gates_from_stash(sigma.grad_fn.saved_tensors[4].clone(), B, S)
    ((sigma * gs).sum() + (rgb * gr).sum() + (warped * gw).sum()).backward()
    cfg = orc.default_cfg(emulate_bf16=True)
    sd_r = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    rgb_r, sigma_r, wp_r, _ = orc.query_fields(windowed_sd(sd_r, cfg, 2, extra), 'fine' if level else 'coarse', pts, d,
                                               ids, cfg, gates=gates)
    print("fwd vs windowed oracle: sigma", H.rel_err(sigma, sigma_r), "rgb", (rgb - rgb_r).abs().max().item(),
          "warped", (warped - wp_r).abs().max().item())
    assert (rgb - rgb_r).abs().max() < 5e-3 and H.rel_err(sigma, sigma_r) < 5e-3
    assert (warped - wp_r).abs().max() < 1e-3
    ((sigma_r * gs).sum() + (rgb_r * gr).sum() + (wp_r * gw).sum()).backward()
    other = "nerf_mlps_coarse" if level else "nerf_mlps_fine"
    bad = []
    for name, p in zip(names, params):
        if name.startswith(other):
            continue
        e = H.rel_err(p.grad, sd_r[name].grad)
        print(f"grad {name:55s} same_gates {e:.3e}")
        if e > (2e-2 if name.startswith(("warp_", "hyper_sheet")) else 1e-2):
            bad.append((name, e))
    assert not bad, bad
    # bands switched off: exactly zero weight-gradient columns (warp 3.5 -> bands 4..9, sheet 2.25 -> 3..6, nerf 6.5 ->
    # 7..9, hyper 1.5 -> 2..5)
    lvl = "fine" if level else "coarse"
    grads = dict(zip(names, [p.grad for p in params]))
    zero_cols = {"warp_field.mlp.linears.0.weight": range(3 + 6 * 4, 63),
                 "warp_field.mlp.linears.5.weight": range(128 + 3 + 6 * 4, 128 + 63),
                 "hyper_sheet_mlp.mlp.linears.0.weight": range(3 + 6 * 3, 45),
                 "hyper_sheet_mlp.mlp.linears.5.weight": range(64 + 3 + 6 * 3, 64 + 45),
                 f"nerf_mlps_{lvl}.trunk_mlp.linears.0.weight": list(range(3 + 6 * 7, 63)) + list(range(63 + 2 + 4 * 2, 89)),
                 f"nerf_mlps_{lvl}.trunk_mlp.linears.5.weight": [256 + c for c in list(range(3 + 6 * 7, 63)) +
                                                                  list(range(63 + 2 + 4 * 2, 89))]}
    for name, cols in zero_cols.items():
        gcols = grads[name][:, list(cols)]
        assert torch.count_nonzero(gcols) == 0, name
        assert torch.count_nonzero(grads[name]) > 0, name


@pytest.mark.gpu
def test_reused_coarse_warp_with_windows():
    """reuse_coarse_warp on and off with windows: the same outputs bit for bit; the flat gradient within 5e-3 and every
    tensor within 2e-2 (relative L2), the bounds of the unwindowed check in tests/test_full_size.py: the two paths
    round the summed warp / sheet upstream gradient to bf16 at different points."""
    from hypernerf_torch_b200 import synthetic
    model, _ = _model('bendy_h2', n_fine=64)
    B = 3000
    rays, rgbs = synthetic.train_rays(B, seed=12, device=DEV)
    g = torch.Generator(device=DEV).manual_seed(13)
    draws = [torch.rand(B, 64, device=DEV, generator=g), torch.rand(B, 64, device=DEV, generator=g)]
    res = {}
    for reuse in (True, False):
        model.reuse_coarse_warp = reuse
        res[reuse] = _flat_grad(model, rays, rgbs, draws, dict(ALPHAS['fractional']))
    for lvl in ("coarse", "fine"):
        for k in ("rgb", "depth", "acc", "weights", "warped_points"):
            assert torch.equal(res[True][0][lvl][k], res[False][0][lvl][k]), (lvl, k)
    a, b = res[True][1], res[False][1]
    rel = ((a.flat - b.flat).norm() / b.flat.norm()).item()
    assert rel < 5e-3, rel
    for p, off in zip(a.params, a.offsets):
        ga, gb = a.flat[off:off + p.numel()], b.flat[off:off + p.numel()]
        assert (ga - gb).norm() <= 2e-2 * gb.norm() + 1e-9, ((ga - gb).norm() / gb.norm()).item()


@pytest.mark.gpu
def test_graphed_train_step_replays_new_alphas():
    """GraphedTrainStep(windowed=True): one capture, three alpha sets written into its device buffer before each
    replay; each step's loss and flat gradient match an eager train_step with the same alphas (no random draws:
    linspace depths, no noise)."""
    from hypernerf_torch_b200 import synthetic
    from hypernerf_torch_b200 import train as hn_train
    model, _ = _model('bendy_h2', stratified=False)
    fg = hn_train.FlatGrads(model.parameters())
    model.attach_flat_grads(fg)
    rays, rgbs = synthetic.train_rays(2048, seed=3, device=DEV)
    step = hn_train.GraphedTrainStep(model, fg, 2048, chunk=1024, windowed=True)
    graph = None
    for extra in (ALPHAS['fractional'], ALPHAS['zero'], dict(nerf_alpha=4.0, warp_alpha=8.25)):
        loss_g = float(step(rays, rgbs, None, extra))
        flat_g = fg.flat.clone()
        graph = step.graph if graph is None else graph
        assert step.graph is graph                      # no new capture
        loss_e = float(hn_train.train_step(model, rays, rgbs, fg, chunk=1024, extra_params=extra))
        rel = ((flat_g - fg.flat).norm() / fg.flat.norm()).item()
        print(f"{extra}: loss graph {loss_g:.6f} eager {loss_e:.6f} grad rel {rel:.2e}")
        assert abs(loss_g - loss_e) <= 1e-4 * abs(loss_e) and rel < 1e-4, (extra, loss_g, loss_e, rel)
    unwindowed = hn_train.GraphedTrainStep(model, fg, 2048, chunk=1024)
    with pytest.raises(ValueError):
        unwindowed(rays, rgbs, None, {'nerf_alpha': 1.0})
    model.attach_flat_grads(None)


@pytest.mark.gpu
def test_frozen_block_rejects_other_alphas():
    from hypernerf_torch_b200 import model_utils, synthetic
    model, _ = _model('bendy_h2')
    rays, _ = synthetic.train_rays(8, seed=1, device=DEV)
    with torch.no_grad(), model.packed_frozen({'nerf_alpha': 2.0}):
        model(model_utils.prepare_ray_dict(rays), {'nerf_alpha': 2.0})
        with pytest.raises(ValueError, match="frozen"):
            model(model_utils.prepare_ray_dict(rays), {'nerf_alpha': 3.0})
        with pytest.raises(ValueError, match="frozen"):
            model(model_utils.prepare_ray_dict(rays), {})


@pytest.mark.gpu
@pytest.mark.parametrize("cuda_graph", [False, True])
def test_fit_schedule_holding_the_warp_window_closed(cuda_graph):
    """fit with a schedule that keeps warp_alpha = 0 (and anneals the others): every warp weight column the window
    covers, except the identity columns, is bit-unchanged after training."""
    from hypernerf_torch_b200 import synthetic
    from hypernerf_torch_b200 import train as hn_train
    model, _ = _model('bendy_h2')
    W0 = model.warp_field.mlp.linears[0].weight.detach().clone()
    W5 = model.warp_field.mlp.linears[5].weight.detach().clone()
    rays, rgbs = synthetic.train_rays(1024, seed=2, device=DEV)
    seen = []

    def schedule(step):
        seen.append(step)
        return {'warp_alpha': 0.0, 'nerf_alpha': 2.0 + step, 'hyper_alpha': 1.0 + 0.5 * step, 'hyper_sheet_alpha': step}

    log = hn_train.fit(model, rays, rgbs, num_epochs=1, batch_size=256, chunk=256, extra_params=schedule,
                       cuda_graph=cuda_graph)
    assert len(log) == 4 and seen == [0, 1, 2, 3]
    W0n, W5n = model.warp_field.mlp.linears[0].weight.detach(), model.warp_field.mlp.linears[5].weight.detach()
    assert torch.equal(W0n[:, 3:63], W0[:, 3:63]) and torch.equal(W5n[:, 128 + 3:128 + 63], W5[:, 128 + 3:128 + 63])
    assert not torch.equal(W0n[:, :3], W0[:, :3])       # identity columns still train
    assert all(math.isfinite(float(e['train/loss'])) for e in log)
