"""TEST INFRASTRUCTURE — not product code.  Nerfies' elastic loss and the translation warp's Jacobian restated in plain
torch (CPU or GPU tensors) on top of the oracle's primitives (oracle/hypernerf_oracle.py).  The JAX Nerfies has the loss
(nerfies/training.py: compute_elastic_loss, loss_type 'log_svals'; utils.general_loss_with_squared_residual); the torch
port raises for warp Jacobians, so this is a restatement whose parity the reference cannot pin (DESIGN.md §2e).
"""
import torch

from oracle import hypernerf_oracle as orc
import background_oracle as bgo


def elastic_rho(jac, alpha=-2.0, scale=0.03, eps=1e-6):
    """Per-sample rho(sum_i log^2 max(sigma_i(J), eps)) of Jacobians (..., 3, 3): svdvals, the eps clamp as
    jnp.maximum(svals, eps), Barron's loss of the squared residual."""
    log_s = torch.log(torch.clamp_min(torch.linalg.svdvals(jac), eps))
    return bgo.robust_loss((log_s ** 2).sum(-1), alpha, scale)


def elastic_loss(jac, weights, alpha=-2.0, scale=0.03, eps=1e-6, weight=1.0, count=None):
    """elastic_reduce_method 'weight': weight * sum(w rho) / count (count defaults to the leading dimension B)."""
    n = jac.shape[0] if count is None else count
    return weight * (weights.detach() * elastic_rho(jac, alpha, scale, eps)).sum() / n


def elastic_closed_form(jac, alpha=-2.0, scale=0.03, eps=1e-6):
    """The arithmetic of hn_elastic_loss (hypernerf_torch_b200/csrc/hn_render.cu) in the dtype of `jac`: the eigenpairs
    (mu, V) of J^T J - I = D + D^T + D^T D (D = J - I), log sigma_i = log1p(mu_i) / 2, or log |J v_i| for mu_i <= -1/2
    (eps-clamped), and
    d r^2 / dJ = J V diag(2 l_i / (1 + mu_i) [sigma_i >= eps]) V^T.  Returns (rho, d rho / dJ) per sample."""
    eye = torch.eye(3, dtype=jac.dtype, device=jac.device)
    D = jac - eye
    M = D + D.transpose(-1, -2) + D.transpose(-1, -2) @ D
    mu, V = torch.linalg.eigh(M)
    # 1 + mu near sigma = 1, |J v|^2 for the small singular values (relative accuracy at both ends)
    small = mu <= -0.5
    lam = torch.where(small, ((jac @ V) ** 2).sum(-2), 1.0 + mu)
    open_ = lam >= eps * eps
    safe = torch.where(open_, lam, torch.ones_like(lam))
    lg = torch.where(small, 0.5 * torch.log(safe), 0.5 * torch.log1p(torch.where(open_ & ~small, mu, torch.zeros_like(mu))))
    l = torch.where(open_, lg, torch.full_like(mu, float(torch.log(torch.tensor(eps, dtype=torch.float64)))))
    f = torch.where(open_, 2 * l / lam, torch.zeros_like(mu))
    r2 = (l ** 2).sum(-1)
    r2v = r2.detach().clone().requires_grad_(True)
    rho = bgo.robust_loss(r2v, alpha, scale)
    drho, = torch.autograd.grad(rho.sum(), r2v)
    S = V @ torch.diag_embed(f) @ V.transpose(-1, -2)
    return rho.detach(), drho[..., None, None] * (jac @ S)


def translation_warp(sd, points, ids, q=orc._ident, gates=None):
    """TranslationField (warping.py:98-125): points (P, S, 3) + mlp([posenc_orig(points, 10) | GLO]) -> (P, S, 3)."""
    embed = sd["warp_embed.embed.weight"][ids.reshape(-1)][:, None, :].expand(-1, points.shape[1], -1)
    warp_in = q(torch.cat([orc.posenc_orig(points, 10), embed], -1))
    return points + orc.mlp(sd, "warp_field.mlp", warp_in, 6, q=q, gates=gates)


def warp_jacobian(sd, points, ids, q=orc._ident, gates=None, create_graph=False):
    """J[p, s, r, c] = d warped_r / d points_c of translation_warp, by reverse mode (one pass per output row; the
    samples are independent).  create_graph=True keeps J differentiable in sd (double backward)."""
    x = points.detach().clone().requires_grad_(True)
    with torch.enable_grad():
        w = translation_warp(sd, x, ids, q=q, gates=gates)
        rows = [torch.autograd.grad(w[..., r].sum(), x, create_graph=create_graph, retain_graph=True)[0] for r in range(3)]
    return torch.stack(rows, -2)
