"""losses.py of the reference (MSELoss, loss_dict) on the B200 path: one fused kernel (hn_mse_loss) computes
MSE(coarse.rgb) + MSE(fine.rgb), the gradient seed of both levels and the fine-level MSE that metrics.psnr needs.
`background_loss` adds HyperNeRF's robust background regularisation, which the torch port dropped."""
import torch
from torch import nn

from . import _lib
from ._lib import check, lib, ptr, stream
from ._packing import pe_alphas
from .models import NerfModel, _FusedWarp


class _FusedMSE(torch.autograd.Function):
    @staticmethod
    @torch.amp.custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, coarse, fine, targets, inv_count):
        c = coarse.contiguous()
        f = None if fine is None else fine.contiguous()
        t = targets.to(torch.float32).contiguous()
        B = c.shape[0]
        sums = torch.zeros(2, device=c.device, dtype=torch.float32)
        need = ctx.needs_input_grad[0] or ctx.needs_input_grad[1]
        gc = torch.empty_like(c) if need else None
        gf = torch.empty_like(f) if (need and f is not None) else None
        check(lib().hn_mse_loss(ptr(c), ptr(f), ptr(t), B, float(inv_count), ptr(sums), ptr(gc), ptr(gf), stream()),
              "hn_mse_loss")
        _lib.count(1)
        ctx.save_for_backward(gc, gf)
        ctx.mark_non_differentiable(sums)
        return (sums[0] + sums[1]) * inv_count, sums

    @staticmethod
    @torch.amp.custom_bwd(device_type="cuda")
    def backward(ctx, g_loss, _g_sums):
        gc, gf = ctx.saved_tensors
        return (None if gc is None else gc * g_loss, None if gf is None else gf * g_loss, None, None)


def mse_coarse_fine(inputs, targets, global_count=None):
    """Returns (loss, sums): loss = (sum_sq(coarse) + sum_sq(fine)) / global_count with global_count = 3 * B by default
    (losses.py:9-14), sums = per-level sums of squared errors (device tensor, no gradient)."""
    coarse = inputs['coarse']['rgb']
    fine = inputs['fine']['rgb'] if 'fine' in inputs else None
    n = targets.numel() if global_count is None else global_count
    return _FusedMSE.apply(coarse, fine, targets, 1.0 / float(n))


class _FusedBackground(torch.autograd.Function):
    @staticmethod
    @torch.amp.custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, warped, points, alpha, scale, grad_scale):
        y = warped.contiguous()
        p = points.contiguous()
        sums = torch.zeros(1, device=y.device, dtype=torch.float32)
        g = torch.empty_like(y) if ctx.needs_input_grad[0] else None
        check(lib().hn_background_loss(ptr(y), ptr(p), p.shape[0], y.shape[-1], float(alpha), float(scale),
                                       float(grad_scale), ptr(sums), ptr(g), stream()), "hn_background_loss")
        _lib.count(1)
        ctx.save_for_backward(g)
        return sums[0] * grad_scale

    @staticmethod
    @torch.amp.custom_bwd(device_type="cuda")
    def backward(ctx, g_loss):
        g, = ctx.saved_tensors
        return (None if g is None else g * g_loss), None, None, None, None


def background_loss(model, points, extra_params=None, *, noise_std=1e-3, alpha=-2.0, scale=1e-3, weight=1.0,
                    global_count=None):
    """HyperNeRF's background regularisation (compute_background_loss of the JAX original, hypernerf/training.py; the
    torch port has none): known-static points (P, 3), e.g. the scene's SfM points, are jittered with Gaussian noise, warped
    with a random warp id each, and their squared displacement r^2 = |warped - jittered|^2 is penalised with Barron's robust
    loss rho(r^2, alpha, scale) (general_loss_with_squared_residual; alpha = -2 is Geman-McClure).  Returns
    weight * sum(rho) / (global_count or P); autograd reaches the warp field, the hyper sheet's GLO rows and the GLO table.
    The warp stage runs alone (hn_mlp_fwd_warp) on the level-0 blob, with the encoding window of `extra_params`.

    Random draws, in this order, on the points' device with the default generator (a test replays them):
      1. ids = model.warp_embeds.to(dev)[torch.randint(len(model.warp_embeds), (P,), device=dev)]
      2. noise = torch.randn(P, 3, device=dev) * noise_std
    Raises ValueError for a model without warp (and for the static NeRF) and for points that are not (P, 3), P > 0."""
    if not isinstance(model, NerfModel):
        raise ValueError(f"background_loss needs a NerfModel with a warp field, got {type(model).__name__}")
    if not model.use_warp:
        raise ValueError("background_loss needs a model with a warp field (use_warp=True)")
    if model._forward_error is not None:
        raise RuntimeError(model._forward_error)
    if points.dim() != 2 or points.shape[1] != 3 or points.shape[0] == 0:
        raise ValueError(f"background points must be (P, 3) with P > 0, got {tuple(points.shape)}")
    dev, P = points.device, points.shape[0]
    ids = model.warp_embeds.to(dev)[torch.randint(len(model.warp_embeds), (P,), device=dev)]
    noise = torch.randn(P, 3, device=dev) * noise_std
    jittered = (points.detach().to(torch.float32) + noise).contiguous()
    warped = _FusedWarp.apply(model, pe_alphas(extra_params), jittered[:, None, :], ids, *model._warp_params())
    count = P if global_count is None else global_count
    return _FusedBackground.apply(warped[:, 0, :], jittered, alpha, scale, float(weight) / float(count))


class _FusedElastic(torch.autograd.Function):
    @staticmethod
    @torch.amp.custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, jac, weights, alpha, scale, eps, grad_scale):
        J = jac.contiguous()
        w = weights.detach().contiguous()
        n = w.numel()
        sums = torch.zeros(1, device=J.device, dtype=torch.float32)
        g = torch.empty(3, n, 3, device=J.device, dtype=torch.float32) if ctx.needs_input_grad[0] else None
        check(lib().hn_elastic_loss(ptr(J), ptr(w), n, float(alpha), float(scale), float(eps), float(grad_scale), ptr(sums),
                                    ptr(g), 0, stream()), "hn_elastic_loss")
        _lib.count(1)
        ctx.save_for_backward(g)
        ctx.shape = J.shape
        return sums[0] * grad_scale

    @staticmethod
    @torch.amp.custom_bwd(device_type="cuda")
    def backward(ctx, g_loss):
        g, = ctx.saved_tensors
        # plane c of the seed holds column c of dL/dJ
        g_jac = None if g is None else g.permute(1, 2, 0).reshape(ctx.shape) * g_loss
        return g_jac, None, None, None, None, None


def elastic_loss(jacobian, weights, *, alpha=-2.0, scale=0.03, eps=1e-6, weight=1.0, global_count=None):
    """Nerfies' elastic regularisation (compute_elastic_loss with loss_type 'log_svals' and elastic_reduce_method
    'weight'; the torch port has none): r^2 = sum_i log^2 max(sigma_i(J), eps) of the warp's Jacobians `jacobian`
    (B, S, 3, 3) (NerfModel.forward(..., return_warp_jacobian=True)['coarse' / 'fine']['warp_jacobian']) is penalised with
    Barron's robust loss rho(r^2, alpha, scale), weighted by the rendering weights (B, S), which take no gradient.  Returns
    weight * sum_{b,s} w_bs rho_bs / (global_count or B) — the reference's (weights * loss).sum(-1).mean().  One fused
    kernel computes the loss and its gradient seed; autograd takes the seed through the warp field."""
    if jacobian.shape[-2:] != (3, 3) or jacobian.shape[:-2] != weights.shape or weights.numel() == 0:
        raise ValueError(f"elastic_loss needs Jacobians (..., 3, 3) and weights of the leading shape, got "
                         f"{tuple(jacobian.shape)} and {tuple(weights.shape)}")
    count = weights.shape[0] if global_count is None else global_count
    return _FusedElastic.apply(jacobian, weights, alpha, scale, eps, float(weight) / float(count))


class MSELoss(nn.Module):
    """losses.py:4-14: MSE(inputs['coarse']['rgb'], targets) [+ MSE(inputs['fine']['rgb'], targets)], mean reduction."""

    def __init__(self):
        super().__init__()

    def forward(self, inputs, targets):
        return mse_coarse_fine(inputs, targets)[0]


loss_dict = {'mse': MSELoss}
