"""Parameter containers with the reference's module tree, so `state_dict()` keys and shapes are identical to
songrise/HyperNeRF-torch (hypernerf/modules.py:46-337, hypernerf/warping.py:28-125; SURVEY.md App. A.6) and
reference checkpoints load unchanged.

These modules own parameters only.  The arithmetic of the hot path runs in the fused CUDA kernels reached from
`NerfModel.forward`; calling a sub-module on its own is not part of the hot path and is not implemented.
"""
import functools
import weakref

import torch
import torch.nn as nn


def posenc_channels(in_ch: int, n_freqs: int) -> int:
    """Width of posenc_orig's output (model_utils.py:234-252): identity + sin/cos per frequency."""
    return in_ch * (1 + 2 * n_freqs)


class _FusedOnly(nn.Module):
    def forward(self, *args, **kwargs):  # pragma: no cover - guard
        raise NotImplementedError(
            f"{type(self).__name__} holds parameters for the fused B200 kernels; evaluate it through "
            "NerfModel.forward (hn_mlp_fwd).  There is no stand-alone / CPU path.")

    # The warp field and the hyper sheet of a NerfModel can be called on their own like in the reference: the call is
    # served by the model's fused network (NerfModel.map_spatial_points / map_hyper_points).  The back reference is weak
    # and bypasses nn.Module's attribute registration (a registered parent would make the module tree cyclic).
    def _bind(self, model):
        object.__setattr__(self, "_owner_ref", weakref.ref(model))

    def __getstate__(self):            # deepcopy / pickle: the back reference is re-made by NerfModel.__setstate__
        state = self.__dict__.copy()
        state.pop("_owner_ref", None)
        return state

    def _owner(self):
        ref = getattr(self, "_owner_ref", None)
        model = ref() if ref is not None else None
        if model is None:
            raise NotImplementedError(
                f"a {type(self).__name__} outside a NerfModel cannot be evaluated: the fused B200 kernels run the whole "
                "per-sample network and need the model it belongs to.  There is no stand-alone / CPU path.")
        return model


class MLP(_FusedOnly):
    """Parameters of modules.MLP (modules.py:46-127): linears[0]: in->W, linears[i+1]: (W+in if i in skips else W)->W,
    logit_layer: W->out."""

    def __init__(self, in_ch, out_ch, depth=8, width=256, hidden_init=None, output_init=None, skips=None):
        super().__init__()
        self.in_ch, self.out_ch, self.depth, self.width = in_ch, out_ch, depth, width
        self.skips = [4] if skips is None else skips
        hidden_init = nn.init.xavier_uniform_ if hidden_init is None else hidden_init
        output_init = nn.init.xavier_uniform_ if output_init is None else output_init
        self.linears = nn.ModuleList(
            [nn.Linear(in_ch, width)] +
            [nn.Linear(width + in_ch if i in self.skips else width, width) for i in range(depth - 1)])
        self.logit_layer = nn.Linear(width, out_ch)
        for lin in self.linears:
            hidden_init(lin.weight)
        output_init(self.logit_layer.weight)


class GLOEmbed(nn.Module):
    """modules.py:131-167.  Inside NerfModel.forward the lookup happens in the fused kernels (ids in, table in the packed
    blob); the module's own forward — a row gather, used by the reference's encode_*_embed helpers (models.py:352-402) —
    is the plain table lookup."""

    def __init__(self, num_embeddings, embedding_dim):
        super().__init__()
        self.num_embeddings, self.embedding_dim = num_embeddings, embedding_dim
        self.embed = nn.Embedding(num_embeddings, embedding_dim)
        nn.init.normal_(self.embed.weight, std=0.1 / embedding_dim)

    def forward(self, inputs):
        if inputs.shape[-1] == 1:     # modules.py:164-165
            inputs = torch.squeeze(inputs, dim=-1)
        return self.embed(inputs)


class NerfMLP(_FusedOnly):
    """modules.py:172-298: trunk 8x256 (+256->256 ReLU logit layer), bottleneck 256->128, alpha Linear, rgb MLP."""

    def __init__(self, in_ch, trunk_depth=8, trunk_width=256, rgb_branch_depth=4, rgb_branch_width=128,
                 rgb_channels=3, alpha_channels=1, skips=None, alpha_condition_dim=0, rgb_condition_dim=39):
        super().__init__()
        skips = [4] if skips is None else skips
        self.trunk_mlp = MLP(in_ch, trunk_width, depth=trunk_depth, width=trunk_width, skips=skips)
        self.bottleneck_mlp = nn.Linear(trunk_width, trunk_width // 2)
        self.rgb_mlp = MLP(rgb_branch_width + rgb_condition_dim, rgb_channels, depth=rgb_branch_depth,
                           width=rgb_branch_width, skips=skips)
        self.alpha_mlp = nn.Linear(128 + alpha_condition_dim, alpha_channels)
        nn.init.xavier_uniform_(self.alpha_mlp.weight)


class HyperSheetMLP(_FusedOnly):
    """modules.py:302-337: input [posenc_orig(points, 7) | embed], 6x64, skip@4, output normal(std=1e-5)."""

    n_freq = 7

    def __init__(self, in_ch=3, in_ch_embed=8, out_ch=3, depth=6, width=64, skips=None):
        super().__init__()
        self.in_ch = posenc_channels(in_ch, self.n_freq) + in_ch_embed
        self.mlp = MLP(self.in_ch, out_ch, depth=depth, width=width, skips=[4] if skips is None else skips,
                       output_init=functools.partial(nn.init.normal_, std=1e-5))

    def forward(self, pts, embed, alpha=None):
        """modules.py:331-337: hyper coordinates (B, S, out_ch) for points (B, S, 3) and embedding vectors (B, S, G)."""
        return self._owner().map_hyper_points(pts, embed, {'hyper_sheet_alpha': alpha})


class TranslationField(_FusedOnly):
    """warping.py:28-125: input [posenc_orig(points, 10) | embed], 6x128, skip@4, output uniform(0, 1e-4)."""

    n_freq = 10

    def __init__(self, in_ch=3, in_ch_embed=8, depth=6, hidden_channels=128, skips=None):
        super().__init__()
        self.in_ch = posenc_channels(in_ch, self.n_freq) + in_ch_embed
        self.mlp = MLP(self.in_ch, 3, depth=depth, width=hidden_channels, skips=[4] if skips is None else skips,
                       hidden_init=nn.init.xavier_normal_, output_init=functools.partial(nn.init.uniform_, b=1e-4))

    def forward(self, points, metadata, extra_params, return_jacobian=False):
        """warping.py:98-125: `metadata` = embedding vectors (B, S, G); returns {'warped_points': (B, S, 3)}, plus
        'jacobian' (B, S, 3, 3) = d warped / d points with return_jacobian."""
        warped, jac = self._owner().map_spatial_points(points, metadata, extra_params, return_warp_jacobian=return_jacobian)
        if return_jacobian:
            return {'warped_points': warped, 'jacobian': jac}
        return {'warped_points': warped}


class SE3Field(_FusedOnly):
    """warping.py:128-209: trunk MLP 6x128 (skip@4, 128 outputs, no output activation) on posenc(points, 0, 8) — 48 channels,
    the metadata embedding is not an input (warping.py:223-224) —, then w_net / v_net: depth 0 in the reference's MLP still
    builds ONE hidden 128 layer (modules.py:95-98) + 3 outputs initialised uniform(0, 1e-4)."""

    min_deg, max_deg = 0, 8

    def __init__(self, in_ch=3, out_ch=1):
        super().__init__()
        self.out_ch = out_ch   # unused, as in the reference
        self.in_ch = 2 * in_ch * (self.max_deg - self.min_deg)
        self.trunk = MLP(self.in_ch, 128, depth=6, width=128, skips=(4,), hidden_init=nn.init.xavier_normal_)
        head_init = functools.partial(nn.init.uniform_, b=1e-4)
        self.w_net = MLP(128, 3, depth=0, width=128, hidden_init=nn.init.xavier_normal_, output_init=head_init)
        self.v_net = MLP(128, 3, depth=0, width=128, hidden_init=nn.init.xavier_normal_, output_init=head_init)

    def forward(self, points, metadata, extra_params, return_jacobian=False):
        """warping.py:242-272 (the metadata is not an input of this field, :223-224, but selects the hyper point that the
        fused network evaluates alongside)."""
        if return_jacobian:   # warping.py:266-271
            raise NotImplementedError(
                "the SE3 warp's Jacobian is not built: its backward needs the second derivatives of the exp map")
        return {'warped_points': self._owner().map_spatial_points(points, metadata, extra_params)[0]}
