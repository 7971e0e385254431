"""Background regularisation: the warp-stage-only fused network (hn_mlp_fwd_warp / hn_mlp_bwd_warp_*) and HyperNeRF's
robust background loss (hn_background_loss, losses.background_loss, train.train_step(background_points=...)).

CPU: the oracle's robust loss in fp64, the new ABI symbols, the warp-only stash sizes and the argument checks.
GPU: the warp-only forward is bit-identical to the full network's `warped` / `aux`; the loss and its parameter gradients
against the oracle on the same draws; windows; train_step linearity; map_points' gradient against the full-network route."""
import ctypes as C
import math

import pytest
import torch

from oracle import hypernerf_oracle as orc
from oracle import ref_loader
import background_oracle as bgo
from hypernerf_torch_b200 import _lib

DEV = "cuda"
EMB = {'warp': list(range(100)), 'camera': [0], 'appearance': list(range(100)), 'time': list(range(100))}
EXTRA = dict(nerf_alpha=None, warp_alpha=None, hyper_alpha=None, hyper_sheet_alpha=None)
WINDOW = dict(warp_alpha=3.5, hyper_sheet_alpha=2.25, nerf_alpha=6.5, hyper_alpha=1.5)

# Configurations of the warp stage (NerfModel kwargs on top of cfg-1): bendy sheet H = 2 / 4 / 8, axis-aligned slicing
# with the translation field, and the SE3 field (axis-aligned).
CONFIGS = {
    'bendy_h2': dict(hyper_slice_method='bendy_sheet', hyper_slice_out_dim=2),
    'bendy_h4': dict(hyper_slice_method='bendy_sheet', hyper_slice_out_dim=4),
    'bendy_h8': dict(hyper_slice_method='bendy_sheet', hyper_slice_out_dim=8),
    'axis': dict(hyper_slice_method='axis_aligned_plane', hyper_slice_out_dim=8),
    'se3': dict(hyper_slice_method='axis_aligned_plane', hyper_slice_out_dim=8, warp_field_type='se3'),
}
COND = {False: dict(use_nerf_embed=False, use_alpha_cond=False, use_rgb_cond=False),
        True: dict(use_nerf_embed=True, use_alpha_cond=True, use_rgb_cond=True)}

# Relative L2 bound of every warp-stage parameter gradient against autograd of the bf16-emulated oracle through the
# kernels' own ReLU gates: the band of the warp tensors in tests/test_se3.py and tests/test_grad_parity.py.  The kernels
# round the same operands to bf16 but sum in tensor-core order, and the deepest tensors (the first layers, reached through
# six transposed bf16 products) collect the most of that rounding.
WARP_GRAD_REL = 2e-2
# The loss against the oracle on the same draws: bf16-emulated (the kernels' numerics) and plain fp32.
LOSS_REL_BF16, LOSS_REL_FP32 = 1e-3, 1e-2


def _desc(**over):
    kw = dict(glo_dim=8, hyper_dim=2, xyz_freqs=10, hyper_freqs=6, view_freqs=6, warp_freqs=10, sheet_freqs=7,
              num_embeddings=100, flags=3)
    kw.update(over)
    return _lib.ModelDesc(*[kw[k] for k in ("glo_dim", "hyper_dim", "xyz_freqs", "hyper_freqs", "view_freqs",
                                            "warp_freqs", "sheet_freqs", "num_embeddings", "flags")])


SE3_DESC = dict(hyper_dim=8, warp_freqs=8, flags=_lib.HN_FLAG_WARP_SE3 | _lib.HN_FLAG_SLICE_AXIS)
AXIS_DESC = dict(hyper_dim=8, flags=_lib.HN_FLAG_WARP_TRANSLATION | _lib.HN_FLAG_SLICE_AXIS)
STATIC_DESC = dict(glo_dim=0, hyper_dim=0, view_freqs=4, flags=_lib.HN_FLAG_STATIC_NERF)
NOWARP_DESC = dict(hyper_dim=0, flags=0)


# ---------------------------------------------------------------------------------------------------------- CPU
def test_robust_loss_special_cases_and_derivative():
    s = 1e-3
    sq = (torch.logspace(-10, -2, 41, dtype=torch.float64)).requires_grad_(True)
    x = sq / (4 * s * s)
    # (rtol: the general form cancels in (x + 1)^(a/2) - 1 at small x)
    assert torch.allclose(bgo.robust_loss(sq, -2.0, s), 2 * x / (x + 1), rtol=1e-9, atol=0)    # Geman-McClure
    assert torch.allclose(bgo.robust_loss(sq, 2.0, s), sq / (2 * s * s), rtol=1e-6, atol=0)    # L2 (b = eps)
    eps = torch.finfo(torch.float32).eps
    for alpha in (-2.0, -0.5, 1.0):
        # Barron's general form |a - 2| / a ((x / |a - 2| + 1)^(a / 2) - 1), x = sq / s^2
        b = abs(alpha - 2)
        ref = b / alpha * ((sq / s ** 2 / b + 1) ** (alpha / 2) - 1)
        rho = bgo.robust_loss(sq, alpha, s)
        assert torch.allclose(rho, ref, rtol=1e-12, atol=0), alpha
        g, = torch.autograd.grad(rho.sum(), sq)
        a = (1.0 if alpha >= 0 else -1.0) * max(eps, abs(alpha))
        drho = (sq / s ** 2 / max(eps, b) + 1) ** (a / 2 - 1) / (2 * s * s)
        assert torch.allclose(g, drho.detach(), rtol=1e-10, atol=0), alpha


def test_new_symbols_and_warp_stash_sizes():
    L = _lib.lib()
    for n in ("hn_mlp_fwd_warp", "hn_mlp_bwd_warp_data", "hn_mlp_bwd_warp_weights", "hn_background_loss"):
        assert n in _lib.EXPORTS and hasattr(L, n), n
    assert C.sizeof(_lib.Sizes) == 64 and L.hn_abi_version() == 4
    n = 1024 * 64
    halves = n // 64
    # slab-map prefixes (hn_mlp_program.h make_slabs): X chunks up to the trunk input, gate words of the warp-stage ReLUs,
    # dY chunks up to and including the head's
    for over, x_pre, g_pre, d_pre in ((dict(), 10 + 6 * 24, 6 * 6, 6 * 24 + 2), (AXIS_DESC, 10 + 6 * 24, 6 * 6, 6 * 24 + 2),
                                      (dict(hyper_dim=4), 10 + 6 * 24, 6 * 6, 6 * 24 + 2),
                                      (SE3_DESC, 6 + 6 * 16 + 16 + 32, 6 * 4 + 8, 6 * 16 + 16 + 32 + 2)):
        s = _lib.Sizes()
        assert L.hn_query(C.byref(_desc(**over)), n, C.byref(s)) == 0
        assert s.warp_saved_bytes == halves * x_pre * 1024 + halves * g_pre * 64 * 4, over
        assert s.warp_workspace_bytes == halves * d_pre * 1024, over
        assert 2400 <= s.warp_saved_bytes / n <= 2650, over          # about 2.4-2.6 KB per sample instead of 9.1 KB
    s = _lib.Sizes()
    assert L.hn_query(C.byref(_desc()), n, C.byref(s)) == 0
    assert s.saved_bytes == halves * 540 * 1024 + halves * 124 * 64 * 4 and s.workspace_bytes == halves * 518 * 1024
    for over in (NOWARP_DESC, STATIC_DESC):
        assert L.hn_query(C.byref(_desc(**over)), n, C.byref(s)) == 0
        assert s.warp_saved_bytes == 0 and s.warp_workspace_bytes == 0


def test_warp_entry_points_check_their_arguments():
    """Null pointers, n <= 0, a static and a no-warp descriptor: a negative code and a message, before any launch (the
    non-null pointers below are never dereferenced)."""
    L = _lib.lib()
    p = C.c_void_p(4096)
    offs = (C.c_int64 * _lib.HN_NUM_PARAM_TENSORS)()

    def fwd(d, B=4, S=8, pts=p):
        return L.hn_mlp_fwd_warp(C.byref(d), p, pts, p, B, S, p, None, None, None)

    def data(d, B=4, S=8, g=p):
        return L.hn_mlp_bwd_warp_data(C.byref(d), p, p, p, g, B, S, offs, p, p, p, p, None)

    def weights(d, B=4, S=8, saved=p):
        return L.hn_mlp_bwd_warp_weights(C.byref(d), saved, B, S, offs, p, p, None, None)

    def expect(rc, word):
        assert rc < 0, rc
        assert word in L.hn_last_error(), L.hn_last_error()

    for fn, null_kw in ((fwd, dict(pts=None)), (data, dict(g=None)), (weights, dict(saved=None))):
        expect(fn(_desc(), **null_kw), b"null")
        expect(fn(_desc(), B=0), b"positive")
        expect(fn(_desc(), S=0), b"positive")
        expect(fn(_desc(**STATIC_DESC)), b"static")
        expect(fn(_desc(**NOWARP_DESC)), b"no warp")
    expect(L.hn_mlp_fwd_warp(None, p, p, p, 4, 8, p, None, None, None), b"null")
    expect(L.hn_mlp_fwd_warp(C.byref(_desc(**SE3_DESC)), p, p, p, 4, 8, p, p, None, None), b"aux")
    expect(L.hn_mlp_bwd_warp_data(C.byref(_desc(**SE3_DESC)), p, p, p, p, 4, 8, offs, p, p, None, None, None), b"SE3")
    expect(L.hn_background_loss(None, p, 4, 5, -2.0, 1e-3, 1.0, p, None, None), b"null")
    expect(L.hn_background_loss(p, p, 4, 5, -2.0, 1e-3, 1.0, None, None, None), b"null")
    expect(L.hn_background_loss(p, p, 0, 5, -2.0, 1e-3, 1.0, p, None, None), b"positive")
    expect(L.hn_background_loss(p, p, -3, 5, -2.0, 1e-3, 1.0, p, None, None), b"positive")
    expect(L.hn_background_loss(p, p, 4, 2, -2.0, 1e-3, 1.0, p, None, None), b"warped_cols")
    expect(L.hn_background_loss(p, p, 4, 5, -2.0, 0.0, 1.0, p, None, None), b"scale")


def test_background_loss_rejects_models_without_warp():
    from hypernerf_torch_b200 import losses
    from hypernerf_torch_b200.models import NerfModel
    from hypernerf_torch_b200.nerf import NeRF
    kw = ref_loader.cfg1_kwargs(n_fine=64, noise_std=None)
    pts = torch.zeros(16, 3)
    with pytest.raises(ValueError, match="warp"):
        losses.background_loss(NerfModel(EMB, **{**kw, 'use_warp': False, 'hyper_slice_method': None}), pts)
    with pytest.raises(ValueError, match="warp"):
        losses.background_loss(NeRF(), pts)
    model = NerfModel(EMB, **kw)
    for bad in (torch.zeros(16, 4), torch.zeros(2, 8, 3), torch.zeros(0, 3)):
        with pytest.raises(ValueError, match=r"\(P, 3\)"):
            losses.background_loss(model, bad)


# ---------------------------------------------------------------------------------------------------------- GPU
def _model(conf, cond=False, boosted=False, seed=3):
    from hypernerf_torch_b200 import synthetic
    from hypernerf_torch_b200.models import NerfModel
    kw = ref_loader.cfg1_kwargs(n_fine=64, noise_std=None)
    kw.update(CONFIGS[conf])
    kw.update(COND[cond])
    model = NerfModel(EMB, **kw)
    sd = synthetic.make_state_dict(model, seed=seed, boosted=boosted)
    model.load_state_dict(sd)
    return model.to(DEV), {k: v.to(DEV) for k, v in sd.items()}, kw


def _points(n, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return (torch.rand(n, 3, device=DEV, generator=g) * 2 - 1).contiguous()


def _full_and_warp(model, pts, ids, extra, train):
    """warped (and, SE3 training, aux) of the full level-0 network and of the warp stage alone, same blob and mode."""
    from hypernerf_torch_b200.models import _FusedMlp, _FusedWarp
    from hypernerf_torch_b200._packing import pe_alphas
    window = pe_alphas(extra)
    dirs = torch.zeros(pts.shape[0], 3, device=DEV)
    with model.packed_frozen(extra), torch.set_grad_enabled(train):
        params = model._canonical_params()
        wparams = model._warp_params()
        if not train:
            params = [q.detach() for q in params]
        _, _, w_full = _FusedMlp.apply(model, (0, window), pts, dirs, ids, None, 0.0, *params)
        w_warp = _FusedWarp.apply(model, window, pts, ids, *wparams)
        aux = None
        if train and model._se3:
            aux = (w_full.grad_fn.saved_tensors[7], w_warp.grad_fn.saved_tensors[4])
    return w_full.detach(), w_warp.detach(), aux


@pytest.mark.gpu
@pytest.mark.parametrize("windowed", [False, True])
@pytest.mark.parametrize("cond", [False, True])
@pytest.mark.parametrize("conf", list(CONFIGS))
def test_warp_only_forward_is_bit_identical(conf, cond, windowed):
    model, _, _ = _model(conf, cond, boosted=True)
    extra = dict(WINDOW) if windowed else dict(EXTRA)
    for B, S in ((3, 37), (1, 1), (11, 256)):
        pts = _points(B * S, B).view(B, S, 3)
        ids = torch.randint(0, 100, (B,), device=DEV)
        for train in (False, True):
            w_full, w_warp, aux = _full_and_warp(model, pts, ids, extra, train)
            assert torch.equal(w_full, w_warp), (B, S, train)
            if aux is not None:
                assert torch.equal(aux[0], aux[1]), (B, S)


@pytest.mark.gpu
@pytest.mark.parametrize("conf", ['bendy_h2', 'axis', 'se3'])
def test_warp_only_forward_is_bit_identical_at_scale(conf):
    """1 000 003 points: the last CTA tile is ragged and every SM runs several tiles."""
    model, _, _ = _model(conf, True, boosted=True)
    B, S = 1000003, 1
    pts = _points(B, 5).view(B, S, 3)
    ids = torch.randint(0, 100, (B,), device=DEV)
    for train in (False, True):
        w_full, w_warp, aux = _full_and_warp(model, pts, ids, dict(WINDOW), train)
        assert torch.equal(w_full, w_warp), train
        if aux is not None:
            assert torch.equal(aux[0], aux[1])
        del w_full, w_warp, aux
        torch.cuda.empty_cache()


def _tune_warp(model, sd, conf, target=4e-3):
    """Scales the warp field's output layer(s) so that the median warp displacement is ~`target` (r / s ~ 4 at
    s = 1e-3, where the robust loss is non-linear).  The translation offset is linear in the logit layer; the SE3 map is
    nearly linear for small screws."""
    names = (["warp_field.w_net.logit_layer", "warp_field.v_net.logit_layer"] if conf == 'se3'
             else ["warp_field.mlp.logit_layer"])
    pts = _points(4096, 17)
    ids = torch.randint(0, 100, (4096,), device=DEV)
    cfg = {'warp_field': 'se3' if conf == 'se3' else 'translation'}
    with torch.no_grad():
        d0 = _displacement(sd, pts, ids, cfg).median()
        f = target / float(d0)
        for n in names:
            for k in (n + ".weight", n + ".bias"):
                sd[k] = sd[k] * f
    model.load_state_dict({k: v.cpu() for k, v in sd.items()})
    return sd


def _displacement(sd, pts, ids, cfg):
    pb = pts[:, None, :]
    if cfg['warp_field'] == 'se3':
        w, _, _ = orc.se3_field(sd, pb)
    else:
        e = sd["warp_embed.embed.weight"][ids][:, None, :]
        w = pb + orc.mlp(sd, "warp_field.mlp", torch.cat([orc.posenc_orig(pb, 10), e], -1), 6)
    return (w[:, 0] - pts).norm(dim=-1)


def _draws(model, P, seed, noise_std=1e-3):
    """Replays losses.background_loss's draws (its docstring's order)."""
    torch.manual_seed(seed)
    ids = model.warp_embeds.to(DEV)[torch.randint(len(model.warp_embeds), (P,), device=DEV)]
    noise = torch.randn(P, 3, device=DEV) * noise_std
    return ids, noise


@pytest.mark.gpu
@pytest.mark.parametrize("weights", ["refinit", "boosted", "tuned"])
@pytest.mark.parametrize("conf", ['bendy_h2', 'se3'])
def test_background_loss_matches_oracle(conf, weights):
    from hypernerf_torch_b200 import losses
    model, sd, kw = _model(conf, boosted=(weights == "boosted"))
    if weights == "tuned":
        sd = _tune_warp(model, sd, conf)
        model.to(DEV)
    P = 16384
    pts = _points(P, 7)
    torch.manual_seed(11)
    with torch.no_grad():
        loss = losses.background_loss(model, pts, dict(EXTRA), weight=0.5)
    ids, noise = _draws(model, P, 11)
    cfg = orc.cfg_from_kwargs(kw)
    ref32 = bgo.background_loss(sd, pts, ids, noise, cfg, weight=0.5)
    ref16 = bgo.background_loss(sd, pts, ids, noise, {**cfg, 'emulate_bf16': True}, weight=0.5)
    r = float((_displacement(sd, pts + noise, ids, cfg) / 1e-3).median())
    print(f"{conf} {weights}: loss {float(loss):.6e} oracle bf16 {float(ref16):.6e} fp32 {float(ref32):.6e} median r/s {r:.3g}")
    if weights == "tuned":
        assert 1.0 <= r <= 10.0, r
    assert abs(float(loss) - float(ref16)) <= LOSS_REL_BF16 * abs(float(ref16))
    assert abs(float(loss) - float(ref32)) <= LOSS_REL_FP32 * abs(float(ref32))


def _warp_gates(saved, P, conf):
    """ReLU gates of the warp stage decoded from the warp-only stash (the X slabs of the prefix, stride = prefix length)."""
    from helpers import decode_slab
    total, hws, width = (150, 6, 128) if conf == 'se3' else (154, 10, 192)

    def gate(chunk, ncols, lo=0, hi=None):
        return (decode_slab(saved, P, chunk, ncols, total_chunks=total)[:, lo:hi] > 0).reshape(P, 1, -1)
    if conf == 'se3':
        wv = hws + 6 * 16 + 16
        return {'warp': [gate(hws + 16 * l, 128) for l in range(6)], 'w_net': [gate(wv, 256, 0, 128)],
                'v_net': [gate(wv, 256, 128, 256)]}
    return {'warp': [gate(hws + 24 * l, width, 0, 128) for l in range(6)]}


@pytest.mark.gpu
@pytest.mark.parametrize("conf", ['bendy_h2', 'se3'])
def test_background_loss_gradients(conf):
    from hypernerf_torch_b200 import losses
    model, sd, kw = _model(conf)
    sd = _tune_warp(model, sd, conf)
    model.to(DEV)
    P = 4096
    pts = _points(P, 8)
    torch.manual_seed(12)
    loss = losses.background_loss(model, pts, dict(EXTRA))
    warp_node = loss.grad_fn.next_functions[0][0]
    while type(warp_node).__name__ != "_FusedWarpBackward":
        warp_node = warp_node.next_functions[0][0]
    gates = _warp_gates(warp_node.saved_tensors[1].clone(), P, conf)
    loss.backward()
    ids, noise = _draws(model, P, 12)
    sd_r = {k: v.clone().requires_grad_(True) for k, v in sd.items()}
    cfg = {**orc.cfg_from_kwargs(kw), 'emulate_bf16': True}
    bgo.background_loss(sd_r, pts, ids, noise, cfg, gates=gates).backward()
    bad = []
    for name, p in model.named_parameters():
        if name.startswith(("nerf_mlps_", "hyper_sheet_mlp")):
            assert p.grad is None or p.grad.abs().max() == 0, name
            continue
        r = sd_r[name].grad if name in sd_r else None
        if name == "warp_embed.embed.weight" and conf == 'se3':
            # the SE3 field reads no GLO vector; the hyper columns take no gradient
            assert p.grad.abs().max() == 0
            continue
        if r is None:             # tables the kernels do not read (hyper_embed of axis-aligned slicing)
            assert p.grad is None or p.grad.abs().max() == 0, name
            continue
        e = ((p.grad - r).norm() / (r.norm() + 1e-30)).item()
        print(f"grad {name:45s} rel {e:.3e} |ref| {r.norm().item():.3e}")
        if e > WARP_GRAD_REL:
            bad.append((name, e))
    assert not bad, bad
    if conf != 'se3':
        # a batch too small to draw every warp id: the drawn GLO rows receive gradient, the others exactly 0
        model.warp_embed.embed.weight.grad = None
        torch.manual_seed(15)
        losses.background_loss(model, pts[:32], dict(EXTRA)).backward()
        ids, _ = _draws(model, 32, 15)
        drawn = torch.zeros(100, dtype=torch.bool, device=DEV)
        drawn[ids] = True
        g = model.warp_embed.embed.weight.grad
        assert (~drawn).any() and g[~drawn].abs().sum() == 0
        assert (g[drawn].abs().sum(-1) > 0).all()


@pytest.mark.gpu
@pytest.mark.parametrize("conf", ['bendy_h2', 'se3'])
def test_background_loss_windows(conf):
    """warp_alpha = 0 closes the warp field's encoding bands: the result is the oracle's on the window-scaled state dict;
    no alphas and +inf alphas run the same numbers."""
    from hypernerf_torch_b200 import losses
    from test_posenc_window import windowed_sd
    model, sd, kw = _model(conf, boosted=True)
    P = 8192
    pts = _points(P, 9)
    cfg = orc.cfg_from_kwargs(kw)
    closed = dict(EXTRA, warp_alpha=0.0)
    torch.manual_seed(13)
    with torch.no_grad():
        loss = losses.background_loss(model, pts, closed)
    ids, noise = _draws(model, P, 13)
    ref = bgo.background_loss(windowed_sd(sd, cfg, 8 if conf == 'se3' else 2, closed), pts, ids, noise,
                              {**cfg, 'emulate_bf16': True})
    assert abs(float(loss) - float(ref)) <= LOSS_REL_BF16 * abs(float(ref)), (float(loss), float(ref))

    def run(extra):
        for p in model.parameters():
            p.grad = None
        torch.manual_seed(14)
        val = losses.background_loss(model, pts, extra)
        val.backward()
        return val.detach(), {n: p.grad.clone() for n, p in model.named_parameters() if p.grad is not None}
    l0, g0 = run(dict(EXTRA))
    l1, g1 = run({k: math.inf for k in EXTRA})
    assert torch.allclose(l0, l1, rtol=1e-6, atol=0)   # the loss sums per-warp partials with float atomics
    assert g0.keys() == g1.keys()
    for n in g0:   # the weight gradient reduces with float atomics: equal up to their ordering
        rel = ((g0[n] - g1[n]).norm() / (g0[n].norm() + 1e-30)).item()
        assert rel <= 1e-5, (n, rel)


@pytest.mark.gpu
def test_train_step_adds_the_background_gradient():
    """train_step(background_points=...) == the MSE-only step + background_loss(...).backward() on the same draws."""
    from hypernerf_torch_b200 import losses, synthetic
    from hypernerf_torch_b200 import train as hn_train
    model, _, _ = _model('bendy_h2', boosted=True)
    fg = hn_train.FlatGrads(model.parameters())
    model.attach_flat_grads(fg)
    rays, rgbs = synthetic.train_rays(512, seed=1, device=DEV)
    bg = _points(4096, 10)
    torch.manual_seed(21)
    stats = hn_train.train_step(model, rays, rgbs, fg, chunk=256, return_stats=True, background_points=bg,
                                background_weight=0.3)
    with_bg = fg.flat.clone()
    torch.manual_seed(21)
    hn_train.train_step(model, rays, rgbs, fg, chunk=256)
    mse_only = fg.flat.clone()
    with model.packed_frozen(dict(hn_train.EXTRA_PARAMS)):
        extra = losses.background_loss(model, bg, dict(hn_train.EXTRA_PARAMS), weight=0.3)
        extra.backward()
    assert torch.allclose(stats['train/background'], extra.detach(), rtol=1e-6, atol=0)
    assert (mse_only - with_bg).norm() > 0
    rel = ((fg.flat - with_bg).norm() / with_bg.norm()).item()
    assert rel <= 1e-6, rel


@pytest.mark.gpu
@pytest.mark.parametrize("conf", ['bendy_h2', 'axis', 'se3'])
def test_map_points_gradient_matches_the_full_network_route(conf):
    """map_points now runs the warp stage alone; its gradient with respect to the parameters and the embedding equals
    the earlier route through the whole level-0 network with zero view directions (to the existing 5e-3)."""
    from hypernerf_torch_b200.models import _FusedMlp
    model, _, _ = _model(conf, boosted=True)
    B, S = 16, 64
    pts = _points(B * S, 4).view(B, S, 3)
    g = torch.Generator(device=DEV).manual_seed(5)
    embed = (torch.randn(B, 8, device=DEV, generator=g) * 0.5).requires_grad_(True)
    gw = torch.randn(B, S, 11 if conf != 'bendy_h2' else 5, device=DEV, generator=g)

    def grads(route):
        for p in model.parameters():
            p.grad = None
        embed.grad = None
        e = embed[:, None, :].expand(B, S, 8)
        if route == "warp":
            warped, _ = model.map_points(pts, e, e, dict(EXTRA))
        else:
            view = model._embed_view(e)
            ids = torch.arange(B, device=DEV)
            _, _, warped = _FusedMlp.apply(view, (0, None), pts, torch.zeros(B, 3, device=DEV), ids, None, 0.0,
                                           *view._canonical_params())
        (warped * gw).sum().backward()
        out = {n: p.grad.clone() for n, p in model.named_parameters()
               if p.grad is not None and not n.startswith("nerf_mlps_")}
        out['embed'] = embed.grad.clone()
        return out
    a, b = grads("warp"), grads("full")
    for n in b:
        if b[n].norm() == 0:
            assert a.get(n) is None or a[n].norm() == 0, n
            continue
        rel = ((a[n] - b[n]).norm() / b[n].norm()).item()
        assert rel <= 5e-3, (n, rel)
