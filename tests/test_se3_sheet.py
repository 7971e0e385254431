"""SE3Field warp with bendy-sheet slicing (HyperNeRF's "DS" model: SE3 deformation + a learned ambient sheet), H = 2.

PARITY UNPINNED BY THE REFERENCE, as for config 5 (tests/test_se3.py): the reference never instantiates SE3Field, so the
kernels are compared with oracle.hypernerf_oracle.query_fields, which runs se3_field and then the hyper sheet on the
unwarped points.  The fused network merges the SE3 trunk and the sheet into one 192-wide warp stage whose input vector
[posenc(p, 0, 8) | posenc_orig(p, 7) | GLO] lives in the activation buffer (DESIGN.md §2d).

CPU: the descriptor's accepted and rejected shapes, hn_sizes against the slab map and the module, the oracle's
composition.  GPU: forward against the oracle, the warp-only and inherited-depth paths bit for bit against the full
network, every parameter gradient, windows, the background loss, train_step / GraphedTrainStep, ragged and 1 M-sample
launches."""
import ctypes as C
import math

import pytest
import torch

import helpers as H
from oracle import hypernerf_oracle as orc
from oracle import ref_loader
from hypernerf_torch_b200 import _lib, synthetic
from hypernerf_torch_b200 import model_utils as mu

DEV = "cuda"
SE3_SHEET = dict(hyper_slice_method='bendy_sheet', hyper_slice_out_dim=2, warp_field_type='se3')
TOL = 2e-3              # north star: rgb / depth / acc / weights within 2e-3 max-abs (DESIGN.md §2a)
BOOSTED_TOL = 3 * TOL   # the boosted stress weights, as tests/test_se3.py
WARPED_TOL = {False: 2e-3, True: 1e-2}
COARSE_BIN = 1.0 / 64   # the fine depths stay within one coarse bin of the oracle's (near 0, far 1, 64 coarse samples)

# saved-activation slab map of this shape (hn_mlp_program.h make_slabs), in 8-column chunks: the 112-column warp-stage
# vector, six 192-wide warp-stage layers (SE3 trunk 128 | sheet 64), the SE3 logit layer, the w / v hidden layer, then
# the template as in cfg 1
X_IN_WS, X_HWS, X_LOGIT, X_WV, X_IN_T, X_T, X_R, X_TOTAL = 0, 14, 158, 174, 206, 218, 528, 592
G_TOTAL, D_TOTAL = 132, 568
X_WARP, G_WARP, D_WARP = 206, 44, 196   # warp-only stash: the prefixes up to the trunk input


def _desc(**over):
    kw = dict(glo_dim=8, hyper_dim=2, xyz_freqs=10, hyper_freqs=6, view_freqs=6, warp_freqs=8, sheet_freqs=7,
              num_embeddings=100, flags=_lib.HN_FLAG_WARP_SE3 | _lib.HN_FLAG_SLICE_BENDY)
    kw.update(over)
    return _lib.ModelDesc(*[kw[k] for k in ("glo_dim", "hyper_dim", "xyz_freqs", "hyper_freqs", "view_freqs",
                                            "warp_freqs", "sheet_freqs", "num_embeddings", "flags")])


def _kwargs(**over):
    kw = ref_loader.cfg1_kwargs(n_fine=64, noise_std=1.0)
    kw.update(SE3_SHEET)
    kw.update(over)
    return kw


def _cpu_model(seed=0, boosted=False, **over):
    from hypernerf_torch_b200.models import NerfModel
    kw = _kwargs(**over)
    model = NerfModel(H.EMB, **kw)
    sd = synthetic.make_state_dict(model, seed=seed, boosted=boosted)
    model.load_state_dict(sd)
    return model, sd, kw


def _model(seed=0, boosted=False, **over):
    model, sd, kw = _cpu_model(seed, boosted, **over)
    return model.to(DEV), {k: v.to(DEV) for k, v in sd.items()}, kw


# ---------------------------------------------------------------------------------------------------------- CPU
def test_descriptor_accepts_h2_and_rejects_other_sheet_widths():
    L = _lib.lib()
    s = _lib.Sizes()
    assert L.hn_query(C.byref(_desc()), 0, C.byref(s)) == 0
    for h in (4, 8):
        assert L.hn_query(C.byref(_desc(hyper_dim=h)), 0, C.byref(s)) != 0
        assert b"bendy_sheet slicing is instantiated for G = 8, hyper_dim 2" in L.hn_last_error()
    for over in (dict(glo_dim=16), dict(sheet_freqs=6), dict(warp_freqs=10)):
        assert L.hn_query(C.byref(_desc(**over)), 0, C.byref(s)) != 0, over
    # the model surfaces the rejection at construction, as for every shape that is not instantiated
    model, _, _ = _cpu_model()
    assert model._forward_error is None
    for h in (4, 8):
        with pytest.raises(_lib.NativeLibraryError, match="hyper_dim 2"):
            _cpu_model(hyper_slice_out_dim=h)


def test_sizes_match_the_slab_map_and_the_module():
    L = _lib.lib()
    n = 1024 * 64
    halves = n // 64
    s = _lib.Sizes()
    assert L.hn_query(C.byref(_desc()), n, C.byref(s)) == 0
    assert s.saved_bytes == halves * X_TOTAL * 1024 + halves * G_TOTAL * 64 * 4
    assert s.workspace_bytes == halves * D_TOTAL * 1024
    assert s.warp_saved_bytes == halves * X_WARP * 1024 + halves * G_WARP * 64 * 4
    assert s.warp_workspace_bytes == halves * D_WARP * 1024
    model, _, _ = _cpu_model()
    kernel_visible = sum(p.numel() for p in model._slot_params() if p is not None)
    assert s.flat_param_floats == kernel_visible
    # every parameter of the module is one the kernels read
    assert kernel_visible == sum(p.numel() for p in model.parameters())


def test_oracle_composition_gives_every_warp_stage_tensor_a_gradient():
    model, sd, kw = _cpu_model(seed=2, boosted=True)
    cfg = orc.cfg_from_kwargs(kw)
    assert cfg['warp_field'] == 'se3' and cfg['slice'] == 'bendy_sheet'
    B, S = 4, 16
    rays, _ = synthetic.train_rays(B, seed=3)
    z = torch.rand(B, S)
    pts = rays[:, None, :3] + z[..., None] * rays[:, None, 3:6]
    sd_r = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    rgb, sigma, wp, _ = orc.query_fields(sd_r, 'coarse', pts, rays[:, 3:6], rays[:, 8].long(), cfg)
    assert wp.shape == (B, S, 5)
    (rgb.sum() + sigma.sum() + wp.sum()).backward()
    for k, v in sd_r.items():
        if k.startswith(("warp_field.", "hyper_sheet_mlp.", "warp_embed.", "nerf_mlps_coarse.")):
            assert v.grad is not None and v.grad.abs().max() > 0, k
    # the sheet reads the unwarped points: its output does not depend on the SE3 field
    w_only = orc.query_fields({**sd, "warp_field.w_net.logit_layer.bias": sd["warp_field.w_net.logit_layer.bias"] + 0.3},
                              'coarse', pts, rays[:, 3:6], rays[:, 8].long(), cfg)[2]
    assert torch.equal(w_only[..., 3:], wp.detach()[..., 3:])
    assert not torch.equal(w_only[..., :3], wp.detach()[..., :3])


# ---------------------------------------------------------------------------------------------------------- GPU
def _draws(B, n_fine, seed):
    g = torch.Generator().manual_seed(seed)
    return [torch.rand(B, 64, generator=g), torch.randn(B, 64, 1, generator=g), torch.rand(B, n_fine, generator=g),
            torch.randn(B, 64 + n_fine, 1, generator=g)]


def _points(n, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return (torch.rand(n, 3, device=DEV, generator=g) * 2 - 1).contiguous()


@pytest.mark.gpu
@pytest.mark.parametrize("boosted", [False, True])
def test_forward_matches_the_oracle(boosted):
    B = 96
    model, sd, kw = _model(3, boosted)
    rays, _ = synthetic.train_rays(B, seed=6, device=DEV)
    draws = [t.to(DEV) for t in _draws(B, 64, 1)]
    with torch.no_grad(), ref_loader._DrawTape(draws):
        out = model(mu.prepare_ray_dict(rays), dict(H.EXTRA))
    o, d = rays[:, :3], rays[:, 3:6]
    free = orc.forward(sd, o, d, rays[:, 8].long(), ref_loader.draws_to_dict(draws), orc.cfg_from_kwargs(kw))
    # the resampled depths inherit the coarse level's bf16 error through the inverse CDF
    def depth(points):
        return ((points - o[:, None, :]) * d[:, None, :]).sum(-1) / (d * d).sum(-1, keepdim=True)
    z_f = depth(out['fine']['points'])
    zerr = (z_f - depth(free['fine']['points'])).abs().max().item()
    print(f"se3+sheet boosted={boosted} fine depths max_abs_err {zerr:.3e} (coarse bin {COARSE_BIN:.3e})")
    assert zerr <= COARSE_BIN
    # the fine level of the oracle at the product's own depths (stage isolation, as tests/test_se3.py)
    ref = orc.forward(sd, o, d, rays[:, 8].long(), ref_loader.draws_to_dict(draws), orc.cfg_from_kwargs(kw), fine_z=z_f)
    tol = BOOSTED_TOL if boosted else TOL
    for lvl in ("coarse", "fine"):
        for k in ("rgb", "depth", "acc", "weights"):
            assert out[lvl][k].shape == ref[lvl][k].shape
            err = (out[lvl][k] - ref[lvl][k]).abs().max().item()
            print(f"se3+sheet boosted={boosted} {lvl} {k} max_abs_err {err:.3e}")
            assert err < tol, (lvl, k, err)
    assert torch.equal(out['coarse']['points'], ref['coarse']['points'])
    assert out['coarse']['warped_points'].shape[-1] == 5
    for cols, name in ((slice(0, 3), "xyz"), (slice(3, 5), "hyper")):
        werr = (out['coarse']['warped_points'][..., cols] - ref['coarse']['warped_points'][..., cols]).abs().max().item()
        print(f"se3+sheet boosted={boosted} coarse warped_points[{name}] max_abs_err {werr:.3e}")
        assert werr < WARPED_TOL[boosted], name


@pytest.mark.gpu
def test_inference_and_training_forward_agree():
    """The inference kernels (no stash, biases inside the UMMAs as bf16 pairs) and the training kernels (stash, fp32 bias
    adds) carry the biases differently, so they agree to the bias rounding, not bit for bit (as tests/test_se3.py); on the
    boosted weights the exp map amplifies that rounding in `warped_points` to the boosted bound against the oracle."""
    B = 40
    model, _, _ = _model(4, True)
    rays, _ = synthetic.train_rays(B, seed=7, device=DEV)
    draws = [t.to(DEV) for t in _draws(B, 64, 2)]
    with torch.no_grad(), ref_loader._DrawTape(draws):
        a = model(mu.prepare_ray_dict(rays), dict(H.EXTRA))
    with ref_loader._DrawTape(draws):
        b = model(mu.prepare_ray_dict(rays), dict(H.EXTRA))
    for lvl, keys in (("coarse", ("rgb", "depth", "acc", "weights", "warped_points")), ("fine", ("rgb", "depth", "acc"))):
        for k in keys:
            err = (a[lvl][k] - b[lvl][k].detach()).abs().max().item()
            assert err < (WARPED_TOL[True] if k == "warped_points" else TOL), (lvl, k, err)


@pytest.mark.gpu
@pytest.mark.parametrize("windowed", [False, True])
def test_warp_only_forward_is_bit_identical(windowed):
    """hn_mlp_fwd_warp (apply_warp, map_*) against the full network's `warped` and `aux`, inference and training, on small
    sizes and one launch of 1 000 003 samples (ragged last tile, several tiles per SM)."""
    from test_background_loss import _full_and_warp, WINDOW
    model, _, _ = _model(5, True)
    extra = dict(WINDOW) if windowed else dict(H.EXTRA)
    for B, S in ((3, 37), (1, 1), (11, 256), (1000003, 1)):
        pts = _points(B * S, B).view(B, S, 3)
        ids = torch.randint(0, 100, (B,), device=DEV)
        for train in (False, True):
            w_full, w_warp, aux = _full_and_warp(model, pts, ids, extra, train)
            assert w_full.shape == (B, S, 5)
            assert torch.equal(w_full, w_warp), (B, S, train)
            if aux is not None:
                assert torch.equal(aux[0], aux[1]), (B, S)
            del w_full, w_warp, aux
    torch.cuda.empty_cache()


@pytest.mark.gpu
def test_map_methods_and_sub_modules_equal_the_full_network():
    """apply_warp / map_points / map_spatial_points / map_hyper_points, warp_field(...) and hyper_sheet_mlp(...) on
    embedding vectors are the warp-stage columns of the full network's `warped`, bit for bit."""
    from hypernerf_torch_b200.models import _FusedMlp
    model, _, _ = _model(6, True)
    B, S = 16, 64
    pts = _points(B * S, 4).view(B, S, 3)
    ids = torch.randint(0, 100, (B,), device=DEV)
    e = model.warp_embed.embed.weight[ids].detach()[:, None, :].expand(B, S, 8)
    with torch.no_grad():
        _, _, full = _FusedMlp.apply(model, (0, None), pts, torch.zeros(B, 3, device=DEV), ids, None, 0.0,
                                     *[q.detach() for q in model._canonical_params()])
        mp, _ = model.map_points(pts, e, e, dict(H.EXTRA))
        sp, _ = model.map_spatial_points(pts, e, dict(H.EXTRA))
        hp = model.map_hyper_points(pts, e, dict(H.EXTRA))
        aw = model.apply_warp(pts, ids, dict(H.EXTRA))['warped_points']
    assert torch.equal(mp, full) and torch.equal(sp, full[..., :3]) and torch.equal(hp, full[..., 3:])
    assert torch.equal(aw, full[..., :3])


@pytest.mark.gpu
def test_reusing_the_coarse_warp_changes_nothing():
    """reuse_coarse_warp: the fine level's inherited depths run the template alone on the coarse pass's warped points;
    every output is bit-identical to the full evaluation, the gradient agrees to the bf16 rounding of the summed upstream
    gradient (tests/test_full_size.py)."""
    from hypernerf_torch_b200 import train as hn_train
    B = 1000
    rays, rgbs = synthetic.train_rays(B, seed=13, device=DEV)
    draws = [t.to(DEV) for t in _draws(B, 64, 23)]
    res = []
    for reuse in (False, True):
        model, _, _ = _model(7, False)
        model.reuse_coarse_warp = reuse
        fg = hn_train.FlatGrads(model.parameters())
        model.attach_flat_grads(fg)
        fg.zero()
        with ref_loader._DrawTape(draws):
            out = model(mu.prepare_ray_dict(rays), dict(H.EXTRA))
        loss = torch.nn.functional.mse_loss(out['coarse']['rgb'], rgbs) + torch.nn.functional.mse_loss(out['fine']['rgb'], rgbs) \
            + 0.1 * out['fine']['warped_points'].square().mean()
        loss.backward()
        with torch.no_grad(), ref_loader._DrawTape(draws):
            inf = model(mu.prepare_ray_dict(rays), dict(H.EXTRA))
        res.append((out, fg.flat.clone(), inf))
    (a, ga, ia), (b, gb, ib) = res
    for lvl in ('coarse', 'fine'):
        for k in a[lvl]:
            assert torch.equal(a[lvl][k], b[lvl][k]), (lvl, k)
            assert torch.equal(ia[lvl][k], ib[lvl][k]), ('inference', lvl, k)
    rel = ((ga - gb).norm() / ga.norm()).item()
    assert rel < 5e-3, rel


def _gates(saved, B, S):
    """ReLU gates of every hidden layer decoded from the kernels' activation stash."""
    def gate(chunk, ncols, lo=0, hi=None):
        x = H.decode_slab(saved, B * S, chunk, ncols, total_chunks=X_TOTAL)[:, lo:hi]
        return (x > 0).reshape(B, S, -1)
    return {'warp': [gate(X_HWS + 24 * l, 192, 0, 128) for l in range(6)],
            'sheet': [gate(X_HWS + 24 * l, 192, 128, 192) for l in range(6)],
            'w_net': [gate(X_WV, 256, 0, 128)], 'v_net': [gate(X_WV, 256, 128, 256)],
            'trunk': [gate(X_T + 32 * l, 256) for l in range(9)], 'rgb': [gate(X_R + 16 * l, 128) for l in range(4)]}


def _gate_parity(B, S, level, boosted, extra=None):
    """hn_mlp_bwd against autograd of the bf16-emulated oracle (on the window-scaled state dict with `extra`) through the
    kernels' own ReLU gates: per-tensor relative L2 errors of every parameter gradient of this level."""
    from hypernerf_torch_b200 import _packing
    from hypernerf_torch_b200.models import _FusedMlp
    from test_posenc_window import windowed_sd
    model, sd, kw = _model(5, boosted)
    rays, _ = synthetic.train_rays(B, seed=6, device=DEV)
    o, d, ids = rays[:, :3].contiguous(), rays[:, 3:6].contiguous(), rays[:, 8].long()
    g = torch.Generator(device=DEV).manual_seed(9)
    z, _ = torch.sort(torch.rand(B, S, device=DEV, generator=g), -1)
    pts = (o[:, None, :] + z[..., None] * d[:, None, :]).contiguous()
    gs = torch.randn(B, S, device=DEV, generator=g)
    gr = torch.randn(B, S, 3, device=DEV, generator=g)
    gw = torch.randn(B, S, 5, device=DEV, generator=g) * 0.1
    params = model._canonical_params()
    window = _packing.pe_alphas(extra) if extra is not None else None
    sigma, rgb, warped = _FusedMlp.apply(model, (level, window), pts, d, ids, None, 0.0, *params)
    gates = _gates(sigma.grad_fn.saved_tensors[4].clone(), B, S)
    ((sigma * gs).sum() + (rgb * gr).sum() + (warped * gw).sum()).backward()
    cfg = orc.cfg_from_kwargs(kw, emulate_bf16=True)
    sd_r = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    sd_w = windowed_sd(sd_r, cfg, 2, extra) if extra is not None else sd_r
    rgb_r, sigma_r, wp_r, _ = orc.query_fields(sd_w, 'fine' if level else 'coarse', pts, d, ids, cfg, gates=gates)
    print("fwd vs oracle[gates]: sigma", H.rel_err(sigma, sigma_r), "rgb", (rgb - rgb_r).abs().max().item(),
          "warped", (warped - wp_r).abs().max().item())
    tol = BOOSTED_TOL if boosted else TOL
    assert (rgb - rgb_r).abs().max() < tol and H.rel_err(sigma, sigma_r) < tol
    assert (warped - wp_r).abs().max() < WARPED_TOL[boosted]
    ((sigma_r * gs).sum() + (rgb_r * gr).sum() + (wp_r * gw).sum()).backward()
    other = "nerf_mlps_coarse" if level else "nerf_mlps_fine"
    errs = {}
    for name, p in model.named_parameters():
        r = sd_r[name].grad
        if name.startswith(other):
            assert p.grad is None or p.grad.abs().max() == 0, name
            continue
        assert r is not None and r.abs().max() > 0, name
        errs[name] = H.rel_err(p.grad, r)
        print(f"grad {name:55s} same_gates {errs[name]:.3e} |ref| {r.norm().item():.3e}")
    return errs


@pytest.mark.gpu
@pytest.mark.parametrize("B,S,level,boosted", [(6, 64, 0, True), (3, 128, 1, True), (5, 64, 1, False), (2, 100, 0, False)])
def test_backward_parameter_gradients(B, S, level, boosted):
    """Every gradient of the level, the sheet tensors and the GLO rows included, within the bounds and reasons of
    tests/test_se3.py::test_se3_backward_parameter_gradients.  On the boosted weights the template's tensors get 1.5e-2
    instead of 1e-2: config 5's hyper point is an exact GLO row, here it is the sheet's output, whose tensor-core
    summation order moves it by up to ~2e-3 against the emulation, and posenc_orig(hyper, 6) amplifies that up to 2^5-fold
    in the trunk input (measured: bottleneck / alpha head 1.1e-2 at 3 x 128 samples)."""
    errs = _gate_parity(B, S, level, boosted)
    assert "warp_embed.embed.weight" in errs and "hyper_sheet_mlp.mlp.logit_layer.weight" in errs
    bad = [(n, e) for n, e in errs.items()
           if e > ((4e-2 if boosted else 2e-2) if n.startswith(("warp_", "hyper_")) else (1.5e-2 if boosted else 1e-2))]
    assert not bad, bad


@pytest.mark.gpu
def test_windowed_forward_and_gradients():
    """warp_alpha windows the SE3 field's posenc(p, 0, 8) (band = c // 6), hyper_sheet_alpha the sheet's
    posenc_orig(p, 7): forward and gradients against the oracle on the window-scaled state dict."""
    from test_posenc_window import ALPHAS
    errs = _gate_parity(6, 64, 0, False, dict(ALPHAS['fractional']))
    bad = [(n, e) for n, e in errs.items() if e > (2e-2 if n.startswith(("warp_", "hyper_")) else 1e-2)]
    assert not bad, bad


@pytest.mark.gpu
def test_windowed_model_forward_matches_oracle_and_infinite_alphas_equal_none():
    from hypernerf_torch_b200 import losses
    from hypernerf_torch_b200 import train as hn_train
    from test_posenc_window import ALPHAS, windowed_sd
    model, sd, kw = _model(0, False, noise_std=None)
    B = 48
    rays, rgbs = synthetic.train_rays(B, seed=4, device=DEV)
    g = torch.Generator(device=DEV).manual_seed(3)
    u_c, u_f = torch.rand(B, 64, device=DEV, generator=g), torch.rand(B, 64, device=DEV, generator=g)
    cfg = orc.cfg_from_kwargs(kw)
    for name in ('fractional', 'zero'):
        extra = ALPHAS[name]
        with torch.no_grad(), ref_loader._DrawTape([u_c, u_f]):
            out = model(mu.prepare_ray_dict(rays), dict(extra))
        ref = orc.forward(windowed_sd(sd, cfg, 2, extra), rays[:, :3], rays[:, 3:6], rays[:, 8].long(),
                          {'u_coarse': u_c, 'u_fine': u_f}, cfg)
        for lvl in ("coarse", "fine"):
            for k in ("rgb", "depth", "acc", "weights"):
                err = (out[lvl][k] - ref[lvl][k]).abs().max().item()
                assert err < TOL, (name, lvl, k, err)
    runs = []
    for extra in (dict(H.EXTRA), {k: math.inf for k in H.EXTRA}):
        fg = hn_train.FlatGrads(model.parameters())
        model.attach_flat_grads(fg)
        fg.zero()
        with ref_loader._DrawTape([u_c, u_f]):
            out = model(mu.prepare_ray_dict(rays), extra)
        loss, _ = losses.mse_coarse_fine(out, rgbs, global_count=3.0 * B)
        loss.backward()
        model.attach_flat_grads(None)
        runs.append((out, fg.flat.clone()))
    (a, ga), (b, gb) = runs
    for lvl in ('coarse', 'fine'):
        for k in a[lvl]:
            assert torch.equal(a[lvl][k].detach(), b[lvl][k].detach()), (lvl, k)
    # the weight gradient reduces with float atomics: equal up to their order
    assert ((ga - gb).norm() / ga.norm()).item() < 1e-5


# Gradients against fp32 autograd of the oracle at reference-init weights, 512 rays: size, direction and the whole-gradient
# distance only, for the reasons of tests/test_se3.py::test_se3_gradients_match_restated_oracle.
GRAD_REL = {"warp_field": 0.4, "hyper_sheet_mlp": 0.4, "nerf_mlps": 0.2, "warp_embed": 0.4}
GRAD_COS = 0.95
WHOLE_GRAD_REL = 8e-2


@pytest.mark.gpu
def test_whole_gradient_matches_the_fp32_oracle():
    B = 512
    model, sd, kw = _model(5, False)
    rays, rgbs = synthetic.train_rays(B, seed=8, device=DEV)
    draws = [t.to(DEV) for t in _draws(B, 64, 3)]
    with ref_loader._DrawTape(draws):
        out = model(mu.prepare_ray_dict(rays), dict(H.EXTRA))
    loss = torch.nn.functional.mse_loss(out['coarse']['rgb'], rgbs) + torch.nn.functional.mse_loss(out['fine']['rgb'], rgbs)
    loss.backward()
    sdg = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    ref = orc.forward(sdg, rays[:, :3], rays[:, 3:6], rays[:, 8].long(), ref_loader.draws_to_dict(draws), orc.cfg_from_kwargs(kw))
    ref_loss = orc.mse_loss(ref, rgbs)
    ref_loss.backward()
    assert abs(loss.item() - ref_loss.item()) < 2e-3
    bad, num, den = [], 0.0, 0.0
    for k, p in model.named_parameters():
        r = sdg[k].grad
        assert r is not None and p.grad is not None, k
        num += float((p.grad - r).double().pow(2).sum())
        den += float(r.double().pow(2).sum())
        rel = ((p.grad - r).norm() / (r.norm() + 1e-20)).item()
        cos = torch.nn.functional.cosine_similarity(p.grad.flatten(), r.flatten(), dim=0).item()
        print(f"se3+sheet {k:52s} |g| {r.norm().item():.3e} rel {rel:.3e} cos {cos:.5f}")
        lim = next(v for pre, v in GRAD_REL.items() if k.startswith(pre))
        if r.norm().item() > 1e-7 and (rel > lim or (cos < GRAD_COS and r.numel() > 1)):
            bad.append((k, rel, cos))
    whole = (num / den) ** 0.5
    print(f"se3+sheet whole flat gradient, relative L2 vs the fp32 oracle: {whole:.3e}")
    assert not bad, bad
    assert whole < WHOLE_GRAD_REL


@pytest.mark.gpu
def test_background_loss_and_its_gradients():
    """The background loss reads the spatial columns only, so the sheet and the GLO table take exactly 0; the SE3 tensors'
    gradients against autograd of tests/background_oracle.py (bf16-emulated, the kernels' gates)."""
    import background_oracle as bgo
    from hypernerf_torch_b200 import losses
    from test_background_loss import _draws as bg_draws, LOSS_REL_BF16, LOSS_REL_FP32, WARP_GRAD_REL
    model, sd, kw = _model(3, False)
    P = 4096
    pts = _points(P, 8)
    cfg = orc.cfg_from_kwargs(kw)
    torch.manual_seed(12)
    loss = losses.background_loss(model, pts, dict(H.EXTRA), weight=0.5)
    node = loss.grad_fn.next_functions[0][0]
    while type(node).__name__ != "_FusedWarpBackward":
        node = node.next_functions[0][0]
    saved = node.saved_tensors[1].clone()

    def gate(chunk, ncols, lo, hi):
        return (H.decode_slab(saved, P, chunk, ncols, total_chunks=X_WARP)[:, lo:hi] > 0).reshape(P, 1, -1)
    gates = {'warp': [gate(X_HWS + 24 * l, 192, 0, 128) for l in range(6)], 'w_net': [gate(X_WV, 256, 0, 128)],
             'v_net': [gate(X_WV, 256, 128, 256)]}
    loss.backward()
    ids, noise = bg_draws(model, P, 12)
    ref16 = bgo.background_loss(sd, pts, ids, noise, {**cfg, 'emulate_bf16': True}, weight=0.5)
    ref32 = bgo.background_loss(sd, pts, ids, noise, cfg, weight=0.5)
    assert abs(float(loss) - float(ref16)) <= LOSS_REL_BF16 * abs(float(ref16))
    assert abs(float(loss) - float(ref32)) <= LOSS_REL_FP32 * abs(float(ref32))
    sd_r = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    bgo.background_loss(sd_r, pts, ids, noise, {**cfg, 'emulate_bf16': True}, weight=0.5, gates=gates).backward()
    bad = []
    for name, p in model.named_parameters():
        if name.startswith(("nerf_mlps_", "hyper_sheet_mlp", "warp_embed")):
            assert p.grad is None or p.grad.abs().max() == 0, name
            continue
        r = sd_r[name].grad
        e = ((p.grad - r).norm() / (r.norm() + 1e-30)).item()
        print(f"grad {name:45s} rel {e:.3e}")
        if e > WARP_GRAD_REL:
            bad.append((name, e))
    assert not bad, bad


@pytest.mark.gpu
def test_train_step_and_graphed_train_step_run():
    from hypernerf_torch_b200 import train as hn_train
    model, _, _ = _model(1, False, noise_std=None)
    model.use_stratified_sampling = False
    fg = hn_train.FlatGrads(model.parameters())
    model.attach_flat_grads(fg)
    rays, rgbs = synthetic.train_rays(2048, seed=3, device=DEV)
    bg = _points(4096, 10)
    stats = hn_train.train_step(model, rays, rgbs, fg, chunk=1024, return_stats=True, background_points=bg)
    assert math.isfinite(float(stats['train/background']))
    assert torch.isfinite(fg.flat).all() and fg.flat.norm() > 0
    loss_e = float(hn_train.train_step(model, rays, rgbs, fg, chunk=1024))
    flat_e = fg.flat.clone()
    for windowed in (False, True):
        step = hn_train.GraphedTrainStep(model, fg, 2048, chunk=1024, windowed=windowed)
        loss_g = float(step(rays, rgbs, None, dict(H.EXTRA) if windowed else None))
        assert math.isfinite(loss_g) and torch.isfinite(fg.flat).all()
        # deterministic depths, no noise: the replay computes the eager step's numbers up to the atomics' order
        assert abs(loss_g - loss_e) <= 1e-5 * abs(loss_e)
        assert ((fg.flat - flat_e).norm() / flat_e.norm()).item() < 1e-4


@pytest.mark.gpu
@pytest.mark.parametrize("B,S", [(1, 7), (3, 33), (2, 257), (5, 128)])
def test_forward_ragged_shapes(B, S):
    """One level through hn_mlp_fwd at sample counts that do not fill a 256-row CTA tile, inference and training kernels,
    against the oracle in bf16-emulation mode (boosted weights: the boosted bounds)."""
    from hypernerf_torch_b200.models import _FusedMlp
    model, sd, kw = _model(7, True)
    rays, _ = synthetic.train_rays(B, seed=9, device=DEV)
    o, d, ids = rays[:, :3].contiguous(), rays[:, 3:6].contiguous(), rays[:, 8].long()
    g = torch.Generator(device=DEV).manual_seed(1)
    z, _ = torch.sort(torch.rand(B, S, device=DEV, generator=g), -1)
    pts = (o[:, None, :] + z[..., None] * d[:, None, :]).contiguous()
    rgb_r, sigma_r, wp_r, _ = orc.query_fields(sd, 'coarse', pts, d, ids, orc.cfg_from_kwargs(kw, emulate_bf16=True))
    params = model._canonical_params()
    for train in (False, True):
        ps = params if train else [q.detach() for q in params]
        sigma, rgb, warped = _FusedMlp.apply(model, 0, pts, d, ids, None, 0.0, *ps)
        assert sigma.shape == (B, S) and rgb.shape == (B, S, 3) and warped.shape == (B, S, 5)
        assert (rgb.detach() - rgb_r).abs().max().item() < BOOSTED_TOL
        assert (warped.detach() - wp_r).abs().max().item() < WARPED_TOL[True]
        assert H.rel_err(sigma.detach(), sigma_r) < 1e-2
