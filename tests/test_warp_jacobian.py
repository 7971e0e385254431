"""Warp Jacobians and Nerfies' elastic loss for the translation warp: hn_mlp_fwd_warp_tangent (the gated tangent passes of
the warp stage), hn_elastic_loss, models._FusedWarpJacobian, return_warp_jacobian / return_jacobian of the reference API,
losses.elastic_loss and train.train_step(elastic_weight=...).

CPU: the kernel's closed form of the loss and its gradient against fp64 autograd of svdvals, the oracle's Jacobian against
torch.func.jacfwd, the new symbols and the argument checks.
GPU: `warped` of the Jacobian path is bit-identical to the warp-only path; J - I against the fp64 product of the bf16
weights through the kernel's own gates; the fused loss against svdvals autograd; per-tensor gradients against double
backward of the oracle; exact zeros where J takes no gradient; the forward's new key; ragged sizes; train_step."""
import ctypes as C

import pytest
import torch

from oracle import hypernerf_oracle as orc
from oracle import ref_loader
import elastic_oracle as eo
from hypernerf_torch_b200 import _lib
from test_background_loss import CONFIGS, EMB, EXTRA, WINDOW, _desc, _model, _points, _warp_gates
from test_posenc_window import windowed_sd

DEV = "cuda"
TRANSLATION = ['bendy_h2', 'bendy_h4', 'bendy_h8', 'axis']
# J - I against the fp64 product of the bf16-rounded packed weights masked by the kernel's own gates: the kernel rounds
# every tangent activation to bf16 (8 significant bits) between the layers, nothing else differs.
JAC_REL = 1e-2
# hn_elastic_loss (fp32 Jacobi eigen-decomposition) against fp64 svdvals autograd on the same J
LOSS_REL, SEED_REL = 1e-4, 1e-3
# per-tensor warp-field gradients against double backward of the bf16-emulated oracle: the warp-stage bound of
# tests/test_background_loss.py
WARP_GRAD_REL = 2e-2


def _rel(a, b):
    return float((a.double() - b.double()).norm() / b.double().norm().clamp_min(1e-30))


# ---------------------------------------------------------------------------------------------------------- CPU
def _cases(gen):
    n = 512
    rnd = torch.randn(n, 3, 3, dtype=torch.float64, generator=gen)
    near = torch.eye(3, dtype=torch.float64) + 1e-4 * torch.randn(n, 3, 3, dtype=torch.float64, generator=gen)
    Q, _ = torch.linalg.qr(torch.randn(n, 3, 3, dtype=torch.float64, generator=gen))
    R, _ = torch.linalg.qr(torch.randn(n, 3, 3, dtype=torch.float64, generator=gen))
    rep = Q @ torch.diag_embed(torch.tensor([1.3, 1.3, 0.7], dtype=torch.float64).expand(n, 3)) @ R   # repeated sigma
    small = Q @ torch.diag_embed(torch.tensor([1.1, 0.9, 2e-3], dtype=torch.float64).expand(n, 3)) @ R   # near zero
    clamp = Q @ torch.diag_embed(torch.tensor([1.2, 0.8, 1e-9], dtype=torch.float64).expand(n, 3)) @ R   # below eps
    return {'random': rnd, 'near_identity': near, 'repeated': rep, 'near_zero': small, 'eps_clamp': clamp}


def test_closed_form_matches_svdvals_autograd():
    """The kernel's arithmetic (eigenpairs of D + D^T + D^T D, spectral gradient) in fp64 against autograd of svdvals."""
    gen = torch.Generator().manual_seed(0)
    for name, J in _cases(gen).items():
        for alpha, scale in ((-2.0, 0.03), (1.0, 0.1)):
            Jr = J.clone().requires_grad_(True)
            rho = eo.elastic_rho(Jr, alpha, scale)
            g, = torch.autograd.grad(rho.sum(), Jr)
            rho_c, g_c = eo.elastic_closed_form(J, alpha, scale)
            assert torch.allclose(rho_c, rho.detach(), rtol=1e-9, atol=1e-15), (name, alpha)
            assert _rel(g_c, g) < 1e-7, (name, alpha, _rel(g_c, g))
    # the clamp: a singular value below eps contributes log(eps)^2 and no gradient through it
    J = torch.diag(torch.tensor([1.0, 1.0, 1e-9], dtype=torch.float64))[None]
    rho_c, g_c = eo.elastic_closed_form(J, -2.0, 0.03)
    assert torch.allclose(rho_c, eo.elastic_rho(J), rtol=1e-12) and g_c[0, 2, 2] == 0


def test_oracle_jacobian_matches_jacfwd():
    from hypernerf_torch_b200 import synthetic
    from hypernerf_torch_b200.models import NerfModel
    kw = ref_loader.cfg1_kwargs(n_fine=64, noise_std=None)
    sd = {k: v.double() for k, v in synthetic.make_state_dict(NerfModel(EMB, **kw), seed=1, boosted=True).items()}
    pts = torch.rand(8, 5, 3, dtype=torch.float64, generator=torch.Generator().manual_seed(2)) * 2 - 1
    ids = torch.arange(8) * 7
    J = eo.warp_jacobian(sd, pts, ids)
    ref = torch.func.jacfwd(lambda p: eo.translation_warp(sd, p[None, None], ids[i:i + 1])[0, 0])
    for i in range(8):
        for s in range(5):
            assert torch.allclose(J[i, s], ref(pts[i, s]), rtol=1e-10, atol=1e-12), (i, s)


def test_new_symbols_and_argument_checks():
    L = _lib.lib()
    for n in ("hn_mlp_fwd_warp_tangent", "hn_elastic_loss"):
        assert n in _lib.EXPORTS and hasattr(L, n), n
    assert L.hn_abi_version() == 4
    p = C.c_void_p(4096)

    def tangent(d, B=4, S=8, pts=p, primal=p, jac=p):
        return L.hn_mlp_fwd_warp_tangent(C.byref(d), p, pts, primal, B, S, jac, None, None)

    def expect(rc, word):
        assert rc < 0, rc
        assert word in L.hn_last_error(), L.hn_last_error()

    for kw in (dict(pts=None), dict(primal=None), dict(jac=None)):
        expect(tangent(_desc(), **kw), b"null")
    expect(L.hn_mlp_fwd_warp_tangent(None, p, p, p, 4, 8, p, None, None), b"null")
    expect(tangent(_desc(), B=0), b"positive")
    expect(tangent(_desc(), S=-1), b"positive")
    expect(tangent(_desc(glo_dim=0, hyper_dim=0, view_freqs=4, flags=_lib.HN_FLAG_STATIC_NERF)), b"static")
    expect(tangent(_desc(hyper_dim=0, flags=0)), b"no warp")
    expect(tangent(_desc(hyper_dim=8, warp_freqs=8, flags=_lib.HN_FLAG_WARP_SE3 | _lib.HN_FLAG_SLICE_AXIS)), b"SE3")
    expect(L.hn_elastic_loss(None, p, 4, -2.0, 0.03, 1e-6, 1.0, p, None, 0, None), b"null")
    expect(L.hn_elastic_loss(p, None, 4, -2.0, 0.03, 1e-6, 1.0, p, None, 0, None), b"null")
    expect(L.hn_elastic_loss(p, p, 4, -2.0, 0.03, 1e-6, 1.0, None, None, 0, None), b"null")
    expect(L.hn_elastic_loss(p, p, 0, -2.0, 0.03, 1e-6, 1.0, p, None, 0, None), b"positive")
    expect(L.hn_elastic_loss(p, p, 4, -2.0, 0.0, 1e-6, 1.0, p, None, 0, None), b"scale")
    expect(L.hn_elastic_loss(p, p, 4, -2.0, 0.03, 0.0, 1.0, p, None, 0, None), b"eps")
    expect(L.hn_elastic_loss(p, p, 4, -2.0, 0.03, 1e-6, 1.0, p, p, -1, None), b"hyper_cols")


def test_se3_and_no_warp_models():
    """SE3 raises with a message before any launch; a model without warp returns no Jacobian and raises nothing."""
    from hypernerf_torch_b200.models import NerfModel
    kw = ref_loader.cfg1_kwargs(n_fine=64, noise_std=None)
    se3 = NerfModel(EMB, **{**kw, **CONFIGS['se3']})
    pts = torch.zeros(2, 4, 3)
    emb = torch.zeros(2, 4, 8)
    with pytest.raises(NotImplementedError, match="exp map"):
        se3.map_points(pts, emb, None, dict(EXTRA), return_warp_jacobian=True)
    with pytest.raises(NotImplementedError, match="exp map"):
        se3.warp_field(pts, emb, dict(EXTRA), return_jacobian=True)
    nowarp = NerfModel(EMB, **{**kw, 'use_warp': False, 'hyper_slice_method': None})
    assert nowarp.map_spatial_points(pts, emb, dict(EXTRA), return_warp_jacobian=True) == (pts, None)


# ---------------------------------------------------------------------------------------------------------- GPU
def _jacobian(model, pts, ids, extra, grad=True):
    from hypernerf_torch_b200.models import _FusedWarpJacobian
    from hypernerf_torch_b200._packing import pe_alphas
    with torch.set_grad_enabled(grad):
        warped, jac = _FusedWarpJacobian.apply(model, pe_alphas(extra), pts, ids, *model._warp_params())
    return warped, jac


def _oracle_sd(sd, kw, extra, dtype=torch.float64):
    sd = {k: v.to(dtype) for k, v in sd.items()}
    return windowed_sd(sd, orc.cfg_from_kwargs(kw), kw['hyper_slice_out_dim'], extra)


@pytest.mark.gpu
@pytest.mark.parametrize("windowed", [False, True])
@pytest.mark.parametrize("weights", ["refinit", "boosted"])
@pytest.mark.parametrize("conf", TRANSLATION)
def test_jacobian_matches_gated_oracle(conf, weights, windowed):
    from hypernerf_torch_b200.models import _FusedWarp
    from hypernerf_torch_b200._packing import pe_alphas
    model, sd, kw = _model(conf, boosted=(weights == "boosted"))
    extra = dict(WINDOW) if windowed else dict(EXTRA)
    B, S = 64, 48
    P = B * S
    pts = _points(P, 21).view(B, S, 3)
    ids = torch.randint(0, 100, (B,), device=DEV)
    warped, jac = _jacobian(model, pts, ids, extra)
    # the primal of the Jacobian path is the training launch (it needs the gates): the same mode of the warp-only path
    ref_warped = _FusedWarp.apply(model, pe_alphas(extra), pts, ids, *model._warp_params())
    assert torch.equal(warped.detach(), ref_warped.detach())
    gates = _warp_gates(jac.grad_fn.saved_tensors[1], P, conf)['warp']
    gates = [g.view(B, S, -1) for g in gates]
    eye = torch.eye(3, device=DEV)
    ref64 = eo.warp_jacobian(_oracle_sd(sd, kw, extra), pts.double(), ids, q=orc.bf16_ste, gates=gates)
    ref32 = eo.warp_jacobian(_oracle_sd(sd, kw, extra, torch.float32), pts, ids, gates=gates)
    d = jac.detach() - eye
    e64, e32 = _rel(d, ref64 - eye.double()), _rel(d, ref32 - eye)
    print(f"{conf} {weights} windowed={windowed}: |J - I| {float(d.norm() / P ** 0.5):.3e}, rel L2 vs bf16-weight fp64 "
          f"{e64:.2e}, vs fp32 jacfwd {e32:.2e}")
    assert e64 <= JAC_REL, e64


@pytest.mark.gpu
def test_elastic_loss_kernel_matches_svdvals():
    from hypernerf_torch_b200 import losses
    gen = torch.Generator().manual_seed(3)
    cases = _cases(gen)
    # fp32 Jacobians: the random case with singular values in [0.1, 10] (a Gaussian 3 x 3 matrix can be arbitrarily close
    # to singular, and fp32 holds such a J itself only to a relative accuracy of ~1e-7 / sigma_min)
    n = cases['random'].shape[0]
    Q, _ = torch.linalg.qr(torch.randn(n, 3, 3, dtype=torch.float64, generator=gen))
    R, _ = torch.linalg.qr(torch.randn(n, 3, 3, dtype=torch.float64, generator=gen))
    cases['random'] = Q @ torch.diag_embed(10.0 ** (2 * torch.rand(n, 3, dtype=torch.float64, generator=gen) - 1)) @ R
    model, _, _ = _model('bendy_h2', boosted=True)
    B, S = 32, 64
    _, kj = _jacobian(model, _points(B * S, 4).view(B, S, 3), torch.randint(0, 100, (B,), device=DEV), dict(EXTRA), False)
    cases['kernel'] = kj.reshape(-1, 3, 3).double().cpu()
    for name, J in cases.items():
        J32 = J.float().to(DEV)
        w = torch.rand(J.shape[0], generator=gen).to(DEV)
        for alpha, scale in ((-2.0, 0.03), (1.0, 0.1)):
            Jk = J32.clone().requires_grad_(True)
            loss = losses.elastic_loss(Jk[:, None], w[:, None], alpha=alpha, scale=scale, weight=0.7)
            loss.backward()
            Jr = J32.double().clone().requires_grad_(True)
            ref = eo.elastic_loss(Jr, w.double(), alpha, scale, weight=0.7)
            ref.backward()
            el, eg = abs(float(loss) - float(ref)) / abs(float(ref)), _rel(Jk.grad, Jr.grad)
            print(f"{name} alpha={alpha}: loss rel {el:.2e}, dL/dJ rel L2 {eg:.2e}")
            assert el <= LOSS_REL, (name, alpha, el)
            assert eg <= SEED_REL, (name, alpha, eg)


def _tune_jacobian(model, sd, pts, ids, target):
    """Scales the warp field's output layer so that the median |J - I|_F is `target`: J - I is linear in it.  The boosted
    weights give Jacobians with singular values near 0, where d log sigma / dJ ~ 1 / sigma amplifies the bf16 rounding of
    the tangents without bound; a training warp stays near the identity."""
    with torch.no_grad():
        J = eo.warp_jacobian(sd, pts, ids)
        f = target / float((J - torch.eye(3, device=DEV)).flatten(-2).norm(dim=-1).median())
        for k in ("warp_field.mlp.logit_layer.weight", "warp_field.mlp.logit_layer.bias"):
            sd[k] = sd[k] * f
    model.load_state_dict({k: v.cpu() for k, v in sd.items()})
    model.to(DEV)
    return sd


@pytest.mark.gpu
@pytest.mark.parametrize("windowed", [False, True])
@pytest.mark.parametrize("conf", ['bendy_h2', 'bendy_h8', 'axis'])
def test_elastic_gradients_match_double_backward(conf, windowed):
    """At reference-init weights with the warp's output scaled to |J - I| ~ 0.05 (log sigma ~ the loss scale 0.03)."""
    from hypernerf_torch_b200 import losses
    model, sd, kw = _model(conf)
    extra = dict(WINDOW) if windowed else dict(EXTRA)
    B, S = 32, 64
    P = B * S
    pts = _points(P, 9).view(B, S, 3)
    ids = torch.randint(0, 100, (B,), device=DEV)
    sd = _tune_jacobian(model, sd, pts, ids, 0.05)
    w = torch.rand(B, S, device=DEV)
    _, jac = _jacobian(model, pts, ids, extra)
    gates = [g.view(B, S, -1) for g in _warp_gates(jac.grad_fn.saved_tensors[1], P, conf)['warp']]
    loss = losses.elastic_loss(jac, w, weight=3.0)
    loss.backward()
    sd_r = {k: v.double().clone().requires_grad_(True) for k, v in sd.items()}
    sd_w = windowed_sd(sd_r, orc.cfg_from_kwargs(kw), kw['hyper_slice_out_dim'], extra)
    J = eo.warp_jacobian(sd_w, pts.double(), ids, q=orc.bf16_ste, gates=gates, create_graph=True)
    ref = eo.elastic_loss(J, w.double(), weight=3.0)
    ref.backward()
    print(f"{conf} windowed={windowed}: loss {float(loss):.6e} oracle {float(ref):.6e}")
    assert abs(float(loss) - float(ref)) <= 1e-2 * abs(float(ref))
    checked = 0
    for name, p in model.named_parameters():
        g = p.grad
        if name.startswith("warp_field.") and name.endswith(".weight"):
            e = _rel(g, sd_r[name].grad)
            print(f"  {name}: rel L2 {e:.2e}")
            assert e <= WARP_GRAD_REL, (name, e)
            checked += 1
        else:   # biases, the GLO table, the hyper sheet and the template: J does not depend on them
            assert g is None or torch.count_nonzero(g) == 0, name
    assert checked == 7


def _rays(n, seed):
    from hypernerf_torch_b200 import model_utils, synthetic
    rays, _ = synthetic.train_rays(n, seed=seed, device=DEV)
    return model_utils.prepare_ray_dict(rays)


@pytest.mark.gpu
@pytest.mark.parametrize("windowed", [False, True])
def test_forward_return_warp_jacobian(windowed):
    model, _, _ = _model('bendy_h2', boosted=True)
    extra = dict(WINDOW) if windowed else dict(EXTRA)
    rd = _rays(256, 5)
    for grad in (True, False):
        with torch.set_grad_enabled(grad):
            torch.manual_seed(7)
            a = model(rd, dict(extra))
            torch.manual_seed(7)
            b = model(rd, dict(extra), return_warp_jacobian=True)
        for level in ('coarse', 'fine'):
            assert set(b[level]) == set(a[level]) | {'warp_jacobian'}
            for k, v in a[level].items():
                assert torch.equal(v, b[level][k]), (level, k)
            pts = b[level]['points']
            embed = model.warp_embed(rd['metadata']['warp'])
            with torch.no_grad():
                r = model.warp_field(pts, embed, dict(extra), return_jacobian=True)
            assert set(r) == {'warped_points', 'jacobian'}
            assert torch.equal(b[level]['warp_jacobian'].detach(), r['jacobian'])
            assert b[level]['warp_jacobian'].shape == pts.shape + (3,)


@pytest.mark.gpu
def test_ragged_sizes_match_split_calls():
    model, _, _ = _model('bendy_h2', boosted=True)
    n = 1000003
    pts = _points(n, 6).view(n, 1, 3)
    ids = torch.randint(0, 100, (n,), device=DEV)
    warped, jac = _jacobian(model, pts, ids, dict(WINDOW), False)
    for lo, hi in ((0, 1), (1, 300), (300, 4097), (4097, 500000), (500000, n)):
        w_s, j_s = _jacobian(model, pts[lo:hi], ids[lo:hi], dict(WINDOW), False)
        assert torch.equal(w_s, warped[lo:hi]) and torch.equal(j_s, jac[lo:hi]), (lo, hi)
    assert torch.isfinite(jac).all()


@pytest.mark.gpu
@pytest.mark.parametrize("windowed", [False, True])
def test_train_step_elastic(windowed):
    from hypernerf_torch_b200 import losses, model_utils, synthetic
    from hypernerf_torch_b200 import train as hn_train
    model, _, _ = _model('bendy_h2', boosted=True)
    fg = hn_train.FlatGrads(model.parameters())
    model.attach_flat_grads(fg)
    rays, rgbs = synthetic.train_rays(512, seed=3, device=DEV)
    extra = dict(WINDOW) if windowed else None
    res = {}
    for ew in (0.0, 0.05, 0.1):
        torch.manual_seed(8)
        st = hn_train.train_step(model, rays, rgbs, fg, chunk=256, return_stats=True, extra_params=extra, elastic_weight=ew)
        res[ew] = (st, fg.flat.clone())
        assert torch.isfinite(fg.flat).all() and torch.isfinite(st['train/loss'])
    mse = float(res[0.0][0]['train/loss'])
    for ew in (0.05, 0.1):
        st = res[ew][0]
        e = float(st['train/elastic'])
        assert e > 0 and abs(float(st['train/loss']) - (mse + e)) <= 1e-5 * (mse + e), ew
    assert abs(float(res[0.1][0]['train/elastic']) - 2 * float(res[0.05][0]['train/elastic'])) <= 1e-5 * float(res[0.1][0]['train/elastic'])
    g0, g1, g2 = res[0.0][1], res[0.05][1], res[0.1][1]
    assert _rel(g2 - g0, 2 * (g1 - g0)) <= 1e-3
    assert float((g1 - g0).norm()) > 0
    # the elastic term of the step is the loss of the same draws' forward
    model.attach_flat_grads(None)
    torch.manual_seed(8)
    with model.packed_frozen(hn_train._extra(extra)), torch.no_grad():
        e = 0.0
        for i in range(0, 512, 256):
            out = model(model_utils.prepare_ray_dict(rays[i:i + 256]), hn_train._extra(extra), return_warp_jacobian=True)
            e += sum(float(losses.elastic_loss(lv['warp_jacobian'], lv['weights'], weight=0.05, global_count=512))
                     for lv in out.values())
    assert abs(e - float(res[0.05][0]['train/elastic'])) <= 1e-4 * e
