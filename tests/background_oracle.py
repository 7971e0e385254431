"""TEST INFRASTRUCTURE — not product code.  HyperNeRF's background loss restated in plain torch (CPU or GPU tensors) on
top of the oracle's primitives (oracle/hypernerf_oracle.py), with every random draw passed in explicitly.  The JAX
original has it (hypernerf/training.py: compute_background_loss; hypernerf/utils.py: general_loss_with_squared_residual);
the torch port does not, so this is a restatement whose parity the reference cannot pin (DESIGN.md §2c).
"""
import torch

from oracle import hypernerf_oracle as orc


def robust_loss(sq, alpha, scale):
    """utils.general_loss_with_squared_residual of the JAX HyperNeRF (Barron's general robust loss on a squared residual):
    b = max(eps, |alpha - 2|), a = sign(alpha) max(eps, |alpha|) (sign(0) = +1), eps = fp32 machine epsilon,
    rho = (b / a) ((sq / scale^2 / b + 1)^(a / 2) - 1).  alpha = -2: Geman-McClure 2 (sq / 4 s^2) / (sq / 4 s^2 + 1);
    alpha = 2: sq / (2 s^2)."""
    eps = torch.finfo(torch.float32).eps
    b = max(eps, abs(alpha - 2.0))
    a = (1.0 if alpha >= 0 else -1.0) * max(eps, abs(alpha))
    return (b / a) * ((sq / scale ** 2 / b + 1.0) ** (0.5 * a) - 1.0)


def background_loss(sd, points, ids, noise, cfg, alpha=-2.0, scale=1e-3, weight=1.0, count=None, gates=None):
    """compute_background_loss of the JAX HyperNeRF (hypernerf/training.py): the known-static points (P, 3) jittered by
    `noise` (P, 3, already scaled), warped with warp ids `ids` (P,) through the TranslationField (or the SE3Field of
    cfg['warp_field'] == 'se3'), rho of the squared displacement of the spatial columns, summed and divided by `count`
    (default P), times `weight`.  cfg['emulate_bf16'] rounds where the kernels hold bf16 operands (as query_fields);
    gates: optional ReLU gates {'warp': [6 x (P, 1, 128)]} or the SE3 ones (se3_field)."""
    q = orc.bf16_ste if cfg.get('emulate_bf16') else orc._ident
    g = gates or {}
    pts = points + noise
    pb = pts[:, None, :]
    if cfg.get('warp_field', 'translation') == 'se3':
        warped, _, _ = orc.se3_field(sd, pb, q=q, gates=g)
    else:
        embed = sd["warp_embed.embed.weight"][ids.reshape(-1)][:, None, :]
        warp_in = q(torch.cat([orc.posenc_orig(pb, 10), embed], -1))
        warped = pb + orc.mlp(sd, "warp_field.mlp", warp_in, 6, q=q, gates=g.get('warp'))
    sq = ((warped[:, 0, :3] - pts) ** 2).sum(-1)
    n = pts.shape[0] if count is None else count
    return weight * robust_loss(sq, alpha, scale).sum() / n
