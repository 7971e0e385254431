"""Drop-in `NerfModel` for songrise/HyperNeRF-torch (hypernerf/models.py:67-780) whose per-ray hot path runs in
the sm_100a kernels of libhypernerf_b200.so.

Boundary B1 of SURVEY.md §8(b): same constructor, same `forward` signature, same nested output dictionary and
the same `state_dict()` names / shapes as the reference, so `train.py:48-67,96-114` and `eval.py:77-135` can swap
the import.  What runs where:

    sample_along_rays        -> hn_sample_coarse           (model_utils.py:6-41)
    render_samples           -> hn_mlp_fwd (+ hn_mlp_bwd)  (models.py:587-650, 447-493; modules.py; warping.py)
                                hn_composite_fwd/bwd       (model_utils.py:43-107, 319-362)
    sample_pdf               -> hn_sample_pdf              (model_utils.py:160-232)

Random draws use the same torch generator calls, in the same order and shapes as the reference
(SURVEY.md App. A.5), and are handed to the kernels as tensors.
"""
import ctypes as C
import os
from typing import Any, Dict, Optional

import torch
import torch.nn as nn

from . import _lib, model_utils, modules
from ._packing import PackedWeights, pe_alphas
from ._lib import check, lib, ptr, stream


class _FilterSigma(torch.autograd.Function):
    """hn_filter_sigma with the mask re-applied to the upstream gradient."""

    @staticmethod
    @torch.amp.custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, points, sigma, dust, use_dust, bbox):
        pts = points.detach().to(torch.float32).contiguous()
        sig = sigma.detach().contiguous()
        out = torch.empty_like(sig)
        box = None if bbox is None else (C.c_float * 6)(*[float(v) for v in bbox])
        check(lib().hn_filter_sigma(ptr(pts), ptr(sig), ptr(sig), sig.numel(), float(dust), int(use_dust), box, ptr(out),
                                    stream()), "hn_filter_sigma")
        _lib.count(1)
        ctx.save_for_backward(pts, sig)
        ctx.cfg = (float(dust), int(use_dust), box)
        return out

    @staticmethod
    @torch.amp.custom_bwd(device_type="cuda")
    def backward(ctx, g):
        pts, sig = ctx.saved_tensors
        dust, use_dust, box = ctx.cfg
        g = g.to(torch.float32).contiguous()
        out = torch.empty_like(g)
        check(lib().hn_filter_sigma(ptr(pts), ptr(sig), ptr(g), g.numel(), dust, use_dust, box, ptr(out), stream()),
              "hn_filter_sigma")
        _lib.count(1)
        return None, out, None, None, None


def filter_sigma(points, sigma, render_opts):
    """models.py:35-63 (dust threshold / bounding box); a no-op unless render_opts is given."""
    if render_opts is None:
        return sigma
    use_dust = 'dust_threshold' in render_opts
    bbox = render_opts.get('bounding_box') if 'bounding_box' in render_opts else None
    if not use_dust and bbox is None:
        return sigma
    return _FilterSigma.apply(points, sigma, render_opts.get('dust_threshold', 0.0) if use_dust else 0.0, use_dust, bbox)


def _param_grads(ctx, model, level, flat_grad, offs, first):
    """Gradients of the autograd inputs `*params` (the model's slot parameters, model._slot_params()) as views of the
    flat buffer; the other level's tensors and anything that needs no gradient get None."""
    other = range(*model._level_param_range(1 - level))
    grads = []
    for i, (slot, shape, n) in enumerate(ctx.param_meta):
        if slot in other or not ctx.needs_input_grad[first + i]:
            grads.append(None)
        else:
            grads.append(flat_grad[offs[slot]:offs[slot] + n].view(shape))
    return grads


def _level_window(level):
    """The `level` argument of the fused autograd functions: the level (0 coarse, 1 fine), or (level, encoding window of
    _packing.pe_alphas) to run on a blob packed with that window."""
    return (level, None) if isinstance(level, int) else level


def _bwd_weights(model, trunk, saved, B, S, level, offs, flat_grad, work, pe_alpha):
    """hn_mlp_bwd[_trunk]_weights, or their windowed forms for a blob packed with an encoding window."""
    d, L = C.byref(model._desc), lib()
    if pe_alpha is None:
        fn, name, extra = (L.hn_mlp_bwd_trunk_weights, "hn_mlp_bwd_trunk_weights", ()) if trunk else \
            (L.hn_mlp_bwd_weights, "hn_mlp_bwd_weights", ())
    else:
        fn, name, extra = (L.hn_mlp_bwd_trunk_weights_windowed, "hn_mlp_bwd_trunk_weights_windowed", (ptr(pe_alpha),)) \
            if trunk else (L.hn_mlp_bwd_weights_windowed, "hn_mlp_bwd_weights_windowed", (ptr(pe_alpha),))
    check(fn(d, ptr(saved), B, S, level, offs, ptr(flat_grad), ptr(work), *extra, stream()), name)


class _FusedMlp(torch.autograd.Function):
    """hn_mlp_fwd / hn_mlp_bwd as one autograd node per level.  Inputs after the fixed arguments are the parameter
    tensors of the canonical slots this configuration has (include/hypernerf_b200.h); gradients come back as views of
    one flat fp32 buffer."""

    @staticmethod
    @torch.amp.custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, model, level, points, viewdirs, ids, noise, noise_std, *params):
        B, S = points.shape[0], points.shape[1]
        dev = points.device
        desc = model._desc
        level, window = _level_window(level)
        packed, pe_alpha = model._packed_window(level, window)
        pts = points.detach().to(torch.float32).contiguous()
        vd = viewdirs.detach().to(torch.float32).contiguous()
        ids = ids.reshape(-1).to(torch.int64).contiguous()
        if ids.numel() != B:
            raise ValueError(f"metadata ids must have one entry per ray, got {tuple(ids.shape)} for {B} rays")
        sigma = torch.empty(B, S, device=dev, dtype=torch.float32)
        rgb = torch.empty(B, S, 3, device=dev, dtype=torch.float32)
        warped = torch.empty(B, S, 3 + desc.hyper_dim, device=dev, dtype=torch.float32)
        need_grad = any(ctx.needs_input_grad[7:])  # grad mode is off inside forward(); autograd tells us here
        saved = aux = None
        if need_grad:
            sizes = model._sizes(B * S)
            saved = torch.empty(sizes.saved_bytes, device=dev, dtype=torch.uint8)
            if model._se3:   # the screw parameters (w, v) of every sample, for the exp map's chain rule
                aux = torch.empty(B, S, 6, device=dev, dtype=torch.float32)
        with _lib.timed("mlp_fwd", B * S):
            check(lib().hn_mlp_fwd(C.byref(desc), ptr(packed), ptr(pts), ptr(vd), ptr(ids), ptr(noise),
                                   float(noise_std), B, S, None, 0, ptr(sigma), ptr(rgb), ptr(warped), ptr(saved), ptr(aux),
                                   stream()), "hn_mlp_fwd")
        _lib.count(1)
        ctx.model, ctx.level, ctx.shape = model, level, (B, S)
        ctx.param_meta = [(slot, p.shape, p.numel()) for slot, p in zip(model._slots_present(), params)]
        ctx.save_for_backward(ids, sigma, rgb, warped, saved, packed, pts if aux is not None else None, aux, pe_alpha)
        ctx.set_materialize_grads(False)
        return sigma, rgb, warped

    @staticmethod
    @torch.amp.custom_bwd(device_type="cuda")
    def backward(ctx, g_sigma, g_rgb, g_warped):
        ids, sigma, rgb, warped, saved, packed, pts, aux, pe_alpha = ctx.saved_tensors
        model, level = ctx.model, ctx.level
        B, S = ctx.shape
        if saved is None:
            raise RuntimeError("hn_mlp_bwd needs the activation stash; forward ran without grad enabled")
        dev = sigma.device
        g_sigma = torch.zeros_like(sigma) if g_sigma is None else g_sigma.to(torch.float32).contiguous()
        g_rgb = torch.zeros_like(rgb) if g_rgb is None else g_rgb.to(torch.float32).contiguous()
        g_warped = None if g_warped is None else g_warped.to(torch.float32).contiguous()
        direct = model._flat_grads is not None and model._flat_grads.flat.device == dev
        if direct:
            # accumulate straight into the bound flat gradient buffer (train.FlatGrads): no per-tensor adds
            offs, flat_grad = model._flat_offsets(), model._flat_grads.flat
        else:
            offs, total = model._grad_offsets()
            flat_grad = torch.zeros(total, device=dev, dtype=torch.float32)
        sizes = model._sizes(B * S)
        work = torch.empty(sizes.workspace_bytes, device=dev, dtype=torch.uint8)
        with _lib.timed("mlp_dgrad", B * S):
            check(lib().hn_mlp_bwd_data(C.byref(model._desc), ptr(packed), ptr(ids), ptr(sigma), ptr(rgb), ptr(warped),
                                        ptr(saved), ptr(g_sigma), ptr(g_rgb), ptr(g_warped), B, S, None, 0, level, offs,
                                        ptr(flat_grad), ptr(work), ptr(pts), ptr(aux), stream()), "hn_mlp_bwd_data")
        with _lib.timed("mlp_wgrad", B * S):
            _bwd_weights(model, False, saved, B, S, level, offs, flat_grad, work, pe_alpha)
        _lib.count(2)
        if direct:
            return (None,) * (7 + len(ctx.param_meta))
        return (None,) * 7 + tuple(_param_grads(ctx, model, level, flat_grad, offs, 7))


class _FusedWarp(torch.autograd.Function):
    """hn_mlp_fwd_warp / hn_mlp_bwd_warp_*: the warp stage alone (TranslationField + HyperSheetMLP, or the SE3Field) on
    the level-0 blob, -> warped (B, S, 3 + H), bit-identical to _FusedMlp's `warped`.  Inputs after the fixed arguments are
    the parameter tensors of the warp-stage slots (NerfModel._warp_slots); gradients come back as views of one flat fp32
    buffer, or go straight into the attached train.FlatGrads.  The sample points take no gradient."""

    @staticmethod
    @torch.amp.custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, model, window, points, ids, *params):
        B, S = points.shape[0], points.shape[1]
        dev = points.device
        desc = model._desc
        packed, pe_alpha = model._packed_window(0, window)
        pts = points.detach().to(torch.float32).contiguous()
        ids = ids.reshape(-1).to(torch.int64).contiguous()
        if ids.numel() != B:
            raise ValueError(f"metadata ids must have one entry per ray, got {tuple(ids.shape)} for {B} rays")
        warped = torch.empty(B, S, 3 + desc.hyper_dim, device=dev, dtype=torch.float32)
        need_grad = any(ctx.needs_input_grad[4:])
        saved = aux = None
        if need_grad:
            saved = torch.empty(model._sizes(B * S).warp_saved_bytes, device=dev, dtype=torch.uint8)
            if model._se3:   # the screw parameters (w, v) of every sample, for the exp map's chain rule
                aux = torch.empty(B, S, 6, device=dev, dtype=torch.float32)
        with _lib.timed("mlp_fwd_warp", B * S):
            check(lib().hn_mlp_fwd_warp(C.byref(desc), ptr(packed), ptr(pts), ptr(ids), B, S, ptr(warped), ptr(saved),
                                        ptr(aux), stream()), "hn_mlp_fwd_warp")
        _lib.count(1)
        ctx.model, ctx.shape = model, (B, S)
        ctx.param_meta = [(slot, p.shape, p.numel()) for slot, p in zip(model._warp_slots(), params)]
        ctx.save_for_backward(ids, saved, packed, pts if aux is not None else None, aux, pe_alpha)
        ctx.set_materialize_grads(False)
        return warped

    @staticmethod
    @torch.amp.custom_bwd(device_type="cuda")
    def backward(ctx, g_warped):
        ids, saved, packed, pts, aux, pe_alpha = ctx.saved_tensors
        model = ctx.model
        B, S = ctx.shape
        if g_warped is None:
            return (None,) * (4 + len(ctx.param_meta))
        if saved is None:
            raise RuntimeError("hn_mlp_bwd_warp needs the activation stash; forward ran without grad enabled")
        dev = g_warped.device
        g_warped = g_warped.to(torch.float32).contiguous()
        direct = model._flat_grads is not None and model._flat_grads.flat.device == dev
        if direct:
            offs, flat_grad = model._flat_offsets(), model._flat_grads.flat
        else:
            offs, total = model._grad_offsets()
            flat_grad = torch.zeros(total, device=dev, dtype=torch.float32)
        work = torch.empty(model._sizes(B * S).warp_workspace_bytes, device=dev, dtype=torch.uint8)
        d = C.byref(model._desc)
        with _lib.timed("mlp_dgrad_warp", B * S):
            check(lib().hn_mlp_bwd_warp_data(d, ptr(packed), ptr(ids), ptr(saved), ptr(g_warped), B, S, offs, ptr(flat_grad),
                                             ptr(work), ptr(pts), ptr(aux), stream()), "hn_mlp_bwd_warp_data")
        with _lib.timed("mlp_wgrad_warp", B * S):
            check(lib().hn_mlp_bwd_warp_weights(d, ptr(saved), B, S, offs, ptr(flat_grad), ptr(work), ptr(pe_alpha),
                                                stream()), "hn_mlp_bwd_warp_weights")
        _lib.count(2)
        if direct:
            return (None,) * (4 + len(ctx.param_meta))
        return (None,) * 4 + tuple(flat_grad[offs[slot]:offs[slot] + n].view(shape) if ctx.needs_input_grad[4 + i] else None
                                   for i, (slot, shape, n) in enumerate(ctx.param_meta))


_SE3_JACOBIAN = ("the SE3 warp's Jacobian is not built: its backward needs the second derivatives of the exp map; the "
                 "fused Jacobian covers the translation warp")


class _FusedWarpJacobian(torch.autograd.Function):
    """The translation warp and its Jacobian, (warped (B, S, 3 + H), jac (B, S, 3, 3)) with jac[b, s, r, c] =
    d warped_r / d points_c (JAX jacfwd's convention), on the level-0 blob.  The forward runs the warp-only primal with a
    stash (its ReLU gates are needed even under no_grad), then hn_mlp_fwd_warp_tangent: the bias-free pass of the warp
    stage along each input direction, gated by the primal's gates (DESIGN.md §2e).  The backward runs the primal's backward
    for g_warped and, for g_jac, per direction c the warp stage's data gradient on the primal's gates with
    g_warped = (g_jac[..., c], 0) and its weight gradient on tangent plane c; biases, the GLO table and the hyper sheet take
    no gradient from J.  Gradients go into one flat fp32 buffer, or straight into the attached train.FlatGrads."""

    @staticmethod
    @torch.amp.custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, model, window, points, ids, *params):
        if model._se3:
            raise NotImplementedError(_SE3_JACOBIAN)
        B, S = points.shape[0], points.shape[1]
        dev = points.device
        desc = model._desc
        packed, pe_alpha = model._packed_window(0, window)
        pts = points.detach().to(torch.float32).contiguous()
        ids = ids.reshape(-1).to(torch.int64).contiguous()
        if ids.numel() != B:
            raise ValueError(f"metadata ids must have one entry per ray, got {tuple(ids.shape)} for {B} rays")
        sizes = model._sizes(B * S)
        warped = torch.empty(B, S, 3 + desc.hyper_dim, device=dev, dtype=torch.float32)
        jac = torch.empty(B, S, 3, 3, device=dev, dtype=torch.float32)
        saved = torch.empty(sizes.warp_saved_bytes, device=dev, dtype=torch.uint8)
        need_grad = any(ctx.needs_input_grad[4:])
        tangent = torch.empty(3 * sizes.warp_saved_bytes, device=dev, dtype=torch.uint8) if need_grad else None
        with _lib.timed("mlp_fwd_warp", B * S):
            check(lib().hn_mlp_fwd_warp(C.byref(desc), ptr(packed), ptr(pts), ptr(ids), B, S, ptr(warped), ptr(saved),
                                        None, stream()), "hn_mlp_fwd_warp")
        with _lib.timed("mlp_fwd_warp_tangent", B * S):
            check(lib().hn_mlp_fwd_warp_tangent(C.byref(desc), ptr(packed), ptr(pts), ptr(saved), B, S, ptr(jac),
                                                ptr(tangent), stream()), "hn_mlp_fwd_warp_tangent")
        _lib.count(2)
        ctx.model, ctx.shape = model, (B, S)
        ctx.param_meta = [(slot, p.shape, p.numel()) for slot, p in zip(model._warp_slots(), params)]
        ctx.save_for_backward(ids, saved if need_grad else None, tangent, packed, pe_alpha)
        ctx.set_materialize_grads(False)
        return warped, jac

    @staticmethod
    @torch.amp.custom_bwd(device_type="cuda")
    def backward(ctx, g_warped, g_jac):
        ids, saved, tangent, packed, pe_alpha = ctx.saved_tensors
        model = ctx.model
        B, S = ctx.shape
        n = B * S
        if g_warped is None and g_jac is None:
            return (None,) * (4 + len(ctx.param_meta))
        if saved is None:
            raise RuntimeError("the warp Jacobian's backward needs the activation stashes; forward ran without grad enabled")
        dev = saved.device
        direct = model._flat_grads is not None and model._flat_grads.flat.device == dev
        if direct:
            offs, flat_grad = model._flat_offsets(), model._flat_grads.flat
        else:
            offs, total = model._grad_offsets()
            flat_grad = torch.zeros(total, device=dev, dtype=torch.float32)
        sizes = model._sizes(n)
        work = torch.empty(sizes.warp_workspace_bytes, device=dev, dtype=torch.uint8)
        d, L = C.byref(model._desc), lib()
        if g_warped is not None:
            g_warped = g_warped.to(torch.float32).contiguous()
            with _lib.timed("mlp_dgrad_warp", n):
                check(L.hn_mlp_bwd_warp_data(d, ptr(packed), ptr(ids), ptr(saved), ptr(g_warped), B, S, offs,
                                             ptr(flat_grad), ptr(work), None, None, stream()), "hn_mlp_bwd_warp_data")
            with _lib.timed("mlp_wgrad_warp", n):
                check(L.hn_mlp_bwd_warp_weights(d, ptr(saved), B, S, offs, ptr(flat_grad), ptr(work), ptr(pe_alpha),
                                                stream()), "hn_mlp_bwd_warp_weights")
            _lib.count(2)
        if g_jac is not None:
            H = model._desc.hyper_dim
            planes = torch.zeros(3, n, 3 + H, device=dev, dtype=torch.float32)
            planes[:, :, :3] = g_jac.to(torch.float32).reshape(n, 3, 3).permute(2, 0, 1)
            warp_jacobian_backward(model, packed, ids, saved, tangent, planes, B, S, offs, flat_grad, work, pe_alpha)
        if direct:
            return (None,) * (4 + len(ctx.param_meta))
        return (None,) * 4 + tuple(flat_grad[offs[slot]:offs[slot] + n_].view(shape) if ctx.needs_input_grad[4 + i] else None
                                   for i, (slot, shape, n_) in enumerate(ctx.param_meta))


# canonical slots that take no gradient from the Jacobian (include/hypernerf_b200.h): the GLO table, every sheet and warp bias
_JACOBIAN_NO_GRAD_SLOTS = (0,) + tuple(range(2, 29, 2))


def warp_jacobian_backward(model, packed, ids, saved, tangent, g_planes, B, S, offs, flat_grad, work, pe_alpha):
    """dL/dJ (given as the three g_warped planes (3, B*S, 3 + H) of hn_elastic_loss) -> the warp-field weight gradients in
    flat_grad (offsets `offs` by slot): per input direction c, the warp stage's data gradient on the primal stash `saved`
    with g_warped = plane c, and the weight gradient on tangent plane c of `tangent`.  The data gradient's GLO-table output
    (products with the zero tangent of the GLO columns) goes to a scratch table."""
    d, L = C.byref(model._desc), lib()
    n = B * S
    plane_bytes = model._sizes(n).warp_saved_bytes
    scratch_offs = (C.c_int64 * _lib.HN_NUM_PARAM_TENSORS)(*([0] + [-1] * (_lib.HN_NUM_PARAM_TENSORS - 1)))
    scratch = torch.empty(model._desc.num_embeddings * model._desc.glo_dim, device=flat_grad.device, dtype=torch.float32)
    w_offs = (C.c_int64 * _lib.HN_NUM_PARAM_TENSORS)(*offs)
    for slot in _JACOBIAN_NO_GRAD_SLOTS:
        w_offs[slot] = -1
    for c in range(3):
        with _lib.timed("mlp_dgrad_warp_tangent", n):
            check(L.hn_mlp_bwd_warp_data(d, ptr(packed), ptr(ids), ptr(saved), ptr(g_planes[c]), B, S, scratch_offs,
                                         ptr(scratch), ptr(work), None, None, stream()), "hn_mlp_bwd_warp_data")
        with _lib.timed("mlp_wgrad_warp_tangent", n):
            check(L.hn_mlp_bwd_warp_weights(d, tangent.data_ptr() + c * plane_bytes, B, S, w_offs, ptr(flat_grad),
                                            ptr(work), ptr(pe_alpha), stream()), "hn_mlp_bwd_warp_weights")
    _lib.count(6)


class _FusedTrunk(torch.autograd.Function):
    """hn_mlp_fwd_trunk / hn_mlp_bwd_trunk: the template NeRF of one level on rows whose warped point / hyper coordinates
    are given (differentiable input).  Used for the coarse depths the fine level inherits: the warp / sheet nets are
    shared between the levels, so their outputs at those depths are the coarse pass's."""

    @staticmethod
    @torch.amp.custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, model, level, warped_in, viewdirs, ids, noise, noise_std, *params):
        B, S = warped_in.shape[0], warped_in.shape[1]
        dev = warped_in.device
        desc = model._desc
        level, window = _level_window(level)
        packed, pe_alpha = model._packed_window(level, window)
        wi = warped_in.detach().to(torch.float32).contiguous()
        vd = viewdirs.detach().to(torch.float32).contiguous()
        sigma = torch.empty(B, S, device=dev, dtype=torch.float32)
        rgb = torch.empty(B, S, 3, device=dev, dtype=torch.float32)
        if ids is not None:
            ids = ids.reshape(-1).to(torch.int64).contiguous()
            if ids.numel() != B:
                raise ValueError(f"metadata ids must have one entry per ray, got {tuple(ids.shape)} for {B} rays")
        need_grad = ctx.needs_input_grad[2] or any(ctx.needs_input_grad[7:])
        saved = None
        if need_grad:
            saved = torch.empty(model._sizes(B * S).saved_bytes, device=dev, dtype=torch.uint8)
        with _lib.timed("mlp_fwd_trunk", B * S):
            check(lib().hn_mlp_fwd_trunk(C.byref(desc), ptr(packed), ptr(wi), ptr(vd), ptr(ids), ptr(noise), float(noise_std),
                                         B, S, None, 0, ptr(sigma), ptr(rgb), None, ptr(saved), stream()), "hn_mlp_fwd_trunk")
        _lib.count(1)
        ctx.model, ctx.level, ctx.shape = model, level, (B, S)
        ctx.param_meta = [(slot, p.shape, p.numel()) for slot, p in zip(model._slots_present(), params)]
        ctx.save_for_backward(sigma, rgb, wi, saved, packed, ids, pe_alpha)
        ctx.set_materialize_grads(False)
        return sigma, rgb

    @staticmethod
    @torch.amp.custom_bwd(device_type="cuda")
    def backward(ctx, g_sigma, g_rgb):
        sigma, rgb, wi, saved, packed, ids, pe_alpha = ctx.saved_tensors
        model, level = ctx.model, ctx.level
        B, S = ctx.shape
        if saved is None:
            raise RuntimeError("hn_mlp_bwd_trunk needs the activation stash; forward ran without grad enabled")
        dev = sigma.device
        g_sigma = torch.zeros_like(sigma) if g_sigma is None else g_sigma.to(torch.float32).contiguous()
        g_rgb = torch.zeros_like(rgb) if g_rgb is None else g_rgb.to(torch.float32).contiguous()
        direct = model._flat_grads is not None and model._flat_grads.flat.device == dev
        if direct:
            offs, flat_grad = model._flat_offsets(), model._flat_grads.flat
        else:
            offs, total = model._grad_offsets()
            flat_grad = torch.zeros(total, device=dev, dtype=torch.float32)
        work = torch.empty(model._sizes(B * S).workspace_bytes, device=dev, dtype=torch.uint8)
        # a model without warp feeds the raw sample points: nothing upstream wants their gradient
        g_wi = torch.empty_like(wi) if (ctx.needs_input_grad[2] or model.use_warp) else None
        with _lib.timed("mlp_dgrad_trunk", B * S):
            check(lib().hn_mlp_bwd_trunk_data(C.byref(model._desc), ptr(packed), ptr(ids), ptr(sigma), ptr(rgb), ptr(wi),
                                              ptr(saved), ptr(g_sigma), ptr(g_rgb), None, B, S, None, 0, level, offs,
                                              ptr(flat_grad), ptr(g_wi), ptr(work), stream()), "hn_mlp_bwd_trunk_data")
        with _lib.timed("mlp_wgrad_trunk", B * S):
            _bwd_weights(model, True, saved, B, S, level, offs, flat_grad, work, pe_alpha)
        _lib.count(2)
        head = (None, None, g_wi if ctx.needs_input_grad[2] else None, None, None, None, None)
        if direct:
            return head + (None,) * len(ctx.param_meta)
        return head + tuple(_param_grads(ctx, model, level, flat_grad, offs, 7))


class _FusedFineLevel(torch.autograd.Function):
    """One autograd node for the fine level when it reuses the coarse pass's warp / sheet outputs (`reuse_coarse_warp`):
    the full network (hn_mlp_fwd) on the depths sample_pdf added and the template alone (hn_mlp_fwd_trunk) on the inherited
    ones, both launches writing straight into the sorted (B, S) rows through their position tables (hn_sample_pdf_ranks),
    and the backward launches reading the upstream gradients through the same tables — no gather / scatter / cat passes."""

    @staticmethod
    @torch.amp.custom_fwd(device_type="cuda", cast_inputs=torch.float32)
    def forward(ctx, model, level, points, viewdirs, ids, noise, noise_std, known_warped, pos_known, pos_new, *params):
        B, S = points.shape[0], points.shape[1]
        Sk, Sn = pos_known.shape[1], pos_new.shape[1]
        dev = points.device
        desc = model._desc
        level, window = _level_window(level)
        packed, pe_alpha = model._packed_window(level, window)
        pts = points.detach().to(torch.float32).contiguous()
        vd = viewdirs.detach().to(torch.float32).contiguous()
        kw = known_warped.detach().to(torch.float32).contiguous()
        ids = ids.reshape(-1).to(torch.int64).contiguous()
        if ids.numel() != B:
            raise ValueError(f"metadata ids must have one entry per ray, got {tuple(ids.shape)} for {B} rays")
        if noise is not None:
            noise = noise.detach().to(torch.float32).contiguous()
        sigma = torch.empty(B, S, device=dev, dtype=torch.float32)
        rgb = torch.empty(B, S, 3, device=dev, dtype=torch.float32)
        warped = torch.empty(B, S, 3 + desc.hyper_dim, device=dev, dtype=torch.float32)
        need_grad = ctx.needs_input_grad[7] or any(ctx.needs_input_grad[10:])
        saved_n = saved_k = aux = None
        if need_grad:
            saved_n = torch.empty(model._sizes(B * Sn).saved_bytes, device=dev, dtype=torch.uint8)
            saved_k = torch.empty(model._sizes(B * Sk).saved_bytes, device=dev, dtype=torch.uint8)
            if model._se3:
                aux = torch.empty(B, Sn, 6, device=dev, dtype=torch.float32)
        with _lib.timed("mlp_fwd", B * Sn):
            check(lib().hn_mlp_fwd(C.byref(desc), ptr(packed), ptr(pts), ptr(vd), ptr(ids), ptr(noise), float(noise_std), B, Sn,
                                   ptr(pos_new), S, ptr(sigma), ptr(rgb), ptr(warped), ptr(saved_n), ptr(aux), stream()),
                  "hn_mlp_fwd")
        with _lib.timed("mlp_fwd_trunk", B * Sk):
            check(lib().hn_mlp_fwd_trunk(C.byref(desc), ptr(packed), ptr(kw), ptr(vd), ptr(ids), ptr(noise), float(noise_std),
                                         B, Sk, ptr(pos_known), S, ptr(sigma), ptr(rgb), ptr(warped), ptr(saved_k), stream()),
                  "hn_mlp_fwd_trunk")
        _lib.count(2)
        ctx.model, ctx.level, ctx.shape = model, level, (B, S, Sk, Sn)
        ctx.param_meta = [(slot, p.shape, p.numel()) for slot, p in zip(model._slots_present(), params)]
        ctx.save_for_backward(ids, sigma, rgb, warped, kw, saved_n, saved_k, packed, pos_known, pos_new,
                              pts if aux is not None else None, aux, pe_alpha)
        ctx.set_materialize_grads(False)
        return sigma, rgb, warped

    @staticmethod
    @torch.amp.custom_bwd(device_type="cuda")
    def backward(ctx, g_sigma, g_rgb, g_warped):
        ids, sigma, rgb, warped, kw, saved_n, saved_k, packed, pos_known, pos_new, pts, aux, pe_alpha = ctx.saved_tensors
        model, level = ctx.model, ctx.level
        B, S, Sk, Sn = ctx.shape
        if saved_n is None:
            raise RuntimeError("hn_mlp_bwd needs the activation stash; forward ran without grad enabled")
        dev = sigma.device
        g_sigma = torch.zeros_like(sigma) if g_sigma is None else g_sigma.to(torch.float32).contiguous()
        g_rgb = torch.zeros_like(rgb) if g_rgb is None else g_rgb.to(torch.float32).contiguous()
        g_warped = None if g_warped is None else g_warped.to(torch.float32).contiguous()
        direct = model._flat_grads is not None and model._flat_grads.flat.device == dev
        if direct:
            offs, flat_grad = model._flat_offsets(), model._flat_grads.flat
        else:
            offs, total = model._grad_offsets()
            flat_grad = torch.zeros(total, device=dev, dtype=torch.float32)
        d = C.byref(model._desc)
        work = torch.empty(model._sizes(B * max(Sk, Sn)).workspace_bytes, device=dev, dtype=torch.uint8)
        g_kw = torch.empty_like(kw)
        with _lib.timed("mlp_dgrad", B * Sn):
            check(lib().hn_mlp_bwd_data(d, ptr(packed), ptr(ids), ptr(sigma), ptr(rgb), ptr(warped), ptr(saved_n), ptr(g_sigma),
                                        ptr(g_rgb), ptr(g_warped), B, Sn, ptr(pos_new), S, level, offs, ptr(flat_grad),
                                        ptr(work), ptr(pts), ptr(aux), stream()), "hn_mlp_bwd_data")
        with _lib.timed("mlp_wgrad", B * Sn):
            _bwd_weights(model, False, saved_n, B, Sn, level, offs, flat_grad, work, pe_alpha)
        with _lib.timed("mlp_dgrad_trunk", B * Sk):
            check(lib().hn_mlp_bwd_trunk_data(d, ptr(packed), ptr(ids), ptr(sigma), ptr(rgb), ptr(kw), ptr(saved_k), ptr(g_sigma),
                                              ptr(g_rgb), ptr(g_warped), B, Sk, ptr(pos_known), S, level, offs, ptr(flat_grad),
                                              ptr(g_kw), ptr(work), stream()), "hn_mlp_bwd_trunk_data")
        with _lib.timed("mlp_wgrad_trunk", B * Sk):
            _bwd_weights(model, True, saved_k, B, Sk, level, offs, flat_grad, work, pe_alpha)
        _lib.count(4)
        head = (None,) * 7 + (g_kw if ctx.needs_input_grad[7] else None, None, None)
        if direct:
            return head + (None,) * len(ctx.param_meta)
        return head + tuple(_param_grads(ctx, model, level, flat_grad, offs, 10))


class NerfModel(PackedWeights, nn.Module):
    """Nerf NN Model with both coarse and fine MLPs (reference: hypernerf/models.py:67-780).

    Configurations (the combinations that run in the reference, SURVEY.md App. B.2):
      use_warp + hyper_slice_method='bendy_sheet'          TranslationField + HyperSheetMLP, hyper_slice_out_dim in {2, 4, 8}
      use_warp + 'axis_aligned_plane'                      hyper point = the GLO vector, hyper_slice_out_dim == GLO_dim == 8
      use_warp=False (any slicing argument)                the template NeRF on the raw points (models.py:568-569)
      use_warp + 'axis_aligned_plane' + warp_field_type='se3'   SE3Field warp (restated; the reference never instantiates it)
      use_warp + 'bendy_sheet' + warp_field_type='se3'          SE3Field + HyperSheetMLP (HyperNeRF's "DS" model), hyper_slice_out_dim 2
    each with or without template GLO conditioning (use_nerf_embed + use_alpha_cond [+ use_rgb_cond], models.py:404-445),
    view_fourier_dim <= 6, xyz / hyper fourier dims 10 / 6, GLO_dim 8.  Combinations that fail inside the reference's
    forward (use_warp with slicing 'none'; use_nerf_embed without use_alpha_cond; use_rgb_cond without use_nerf_embed:
    matmul shape errors) construct, like there, and raise RuntimeError when called."""

    # The fine level's sorted depths contain the coarse depths (models.py:752-755), and the warp field / hyper sheet are
    # shared between the levels (models.py:143-182), so the reference evaluates them twice at those points.  With this on,
    # the fine level runs the full network only on its new depths and the template NeRF alone (hn_mlp_fwd_trunk) on the
    # inherited ones, fed with the coarse pass's warped points; outputs are bit-identical, the warp / sheet parameters
    # receive the sum of both levels' gradients through one backward pass.
    reuse_coarse_warp = os.environ.get("HN_REUSE_COARSE_WARP", "1") != "0"

    def __init__(self, embeddings_dict,
                 near: float = 0.0, far: float = 1.0,
                 n_samples_coarse: int = 64,
                 n_samples_fine: int = 128,
                 noise_std: float = None,
                 use_warp: bool = True,
                 use_nerf_embed: bool = True,
                 use_alpha_cond: bool = True,
                 use_rgb_cond: bool = False,
                 hyper_slice_method: str = None,
                 hyper_slice_out_dim: int = 4,
                 GLO_dim: int = 8,
                 share_GLO: bool = True,
                 xyz_fourier_dim: int = 10,
                 hyper_fourier_dim: int = 6,
                 view_fourier_dim: int = 4,
                 warp_field_type: str = 'translation'):
        """`warp_field_type` is the one argument the reference's constructor does not have: there the warp field class is
        the attribute `warp_field_cls` (models.py:195, "SE3 untested") and the instantiation is hard-coded to
        TranslationField (models.py:234).  'se3' builds warping.SE3Field (warping.py:128-272) in its place — BASELINE.json
        config 5 —, evaluated batched as DESIGN.md §"SE3 warp" restates it (the reference's own exp map only takes one point)."""
        super().__init__()
        self.embeddings_dict = embeddings_dict
        self.near, self.far = near, far
        self.use_viewdirs = True
        self.noise_std = noise_std
        self.nerf_trunk_depth, self.nerf_trunk_width = 8, 256
        self.nerf_rgb_branch_depth, self.nerf_rgb_branch_width = 4, 128
        self.nerf_skips = [4]
        self.num_coarse_samples, self.num_fine_samples = n_samples_coarse, n_samples_fine
        self.use_stratified_sampling = True
        self.use_white_background = False
        self.use_linear_disparity = False
        self.use_sample_at_infinity = True
        self.alpha_channels, self.rgb_channels = 1, 3
        if not share_GLO:
            # the reference leaves nerf_use_warp_embed unbound in this case (models.py:167-174)
            raise UnboundLocalError("share_GLO=False is not usable in the reference (models.py:167-174)")
        self.nerf_use_warp_embed = self.hyper_use_warp_embed = use_warp
        self.use_nerf_embed = use_nerf_embed
        self.nerf_embed_key = 'warp'
        self.use_alpha_condition, self.use_rgb_condition = use_alpha_cond, use_rgb_cond
        self.hyper_slice_method = 'none' if hyper_slice_method is None else hyper_slice_method
        self.hyper_embed_key = 'time'
        self.hyper_sheet_out_dim = hyper_slice_out_dim
        self.use_warp = use_warp
        self.warp_embed_key = 'time'
        self.use_original_embed = True
        self.xyz_freq, self.dir_freq, self.hyper_freq = xyz_fourier_dim, view_fourier_dim, hyper_fourier_dim
        self.GLO_dim = GLO_dim

        if self.use_nerf_embed and not (self.use_rgb_condition or self.use_alpha_condition):
            raise ValueError('Template metadata is enabled but none of the condition'
                             'branches are.')

        # ---- module tree in the reference's registration order (models.py:215-309): state_dict names / order ---------
        def n_embed(key):
            return max(self.embeddings_dict[key]) + 1

        if self.use_nerf_embed:
            self.nerf_embed = modules.GLOEmbed(num_embeddings=n_embed(self.nerf_embed_key), embedding_dim=GLO_dim)
        if self.use_warp:
            self.warp_embed = modules.GLOEmbed(num_embeddings=n_embed(self.warp_embed_key), embedding_dim=GLO_dim)
        if self.hyper_slice_method == 'axis_aligned_plane':
            self.hyper_embed = modules.GLOEmbed(num_embeddings=n_embed(self.hyper_embed_key), embedding_dim=GLO_dim)
        elif self.hyper_slice_method == 'bendy_sheet':
            if not self.hyper_use_warp_embed:
                self.hyper_embed = modules.GLOEmbed(num_embeddings=n_embed(self.hyper_embed_key), embedding_dim=GLO_dim)
            self.hyper_sheet_mlp = modules.HyperSheetMLP(out_ch=self.hyper_sheet_out_dim, in_ch_embed=GLO_dim)
        if warp_field_type not in ('translation', 'se3'):
            raise ValueError(f"Unknown warp field type {warp_field_type}.")
        self._se3 = self.use_warp and warp_field_type == 'se3'
        self.warp_field_cls = modules.SE3Field if warp_field_type == 'se3' else modules.TranslationField
        if self.use_warp:
            self.warp_field = modules.SE3Field(in_ch=3) if self._se3 else modules.TranslationField(in_ch=3, in_ch_embed=GLO_dim)
        self._bind_sub_modules()
        self.alpha_default = 0.0
        self.nerf_in_ch_pos = modules.posenc_channels(3, self.xyz_freq)
        self.nerf_cond_ch_rgb = modules.posenc_channels(3, self.dir_freq)
        self.hyper_feat_ch = modules.posenc_channels(self.hyper_sheet_out_dim, self.hyper_freq)
        if self.use_warp:
            self.nerf_in_ch_pos += self.hyper_feat_ch
        if self.use_rgb_condition:
            self.nerf_cond_ch_rgb += GLO_dim

        def make_nerf_mlp():
            return modules.NerfMLP(in_ch=self.nerf_in_ch_pos, trunk_depth=self.nerf_trunk_depth,
                                   trunk_width=self.nerf_trunk_width, rgb_branch_depth=self.nerf_rgb_branch_depth,
                                   rgb_branch_width=self.nerf_rgb_branch_width, skips=self.nerf_skips,
                                   alpha_channels=self.alpha_channels, rgb_channels=self.rgb_channels,
                                   alpha_condition_dim=GLO_dim if self.use_nerf_embed else 0,
                                   rgb_condition_dim=self.nerf_cond_ch_rgb)

        self.nerf_mlps_coarse = make_nerf_mlp()
        if self.num_fine_samples > 0:
            self.nerf_mlps_fine = make_nerf_mlp()
        else:
            raise NotImplementedError("n_samples_fine == 0: the reference itself fails here (models.py:292-309)")

        # ---- what the reference's own forward cannot run: same exception type, raised at call time -------------------
        self._forward_error = None
        if self.use_warp and self.hyper_slice_method == 'none':
            self._forward_error = ("use_warp with hyper_slice_method 'none': the trunk is built for posenc(xyz) + posenc(hyper) "
                                   "channels but map_points yields no hyper point (models.py:269-270, 575-579)")
        elif self.use_warp and self.hyper_slice_method == 'axis_aligned_plane' and hyper_slice_out_dim != GLO_dim:
            self._forward_error = ("axis_aligned_plane: the hyper point is the GLO vector (models.py:533-534), so "
                                   "hyper_slice_out_dim must equal GLO_dim")
        elif self.use_nerf_embed and not self.use_alpha_condition:
            self._forward_error = "use_nerf_embed without use_alpha_cond: alpha_mlp expects 128 + GLO_dim inputs (modules.py:283)"
        elif self.use_rgb_condition and not self.use_nerf_embed:
            self._forward_error = "use_rgb_cond without use_nerf_embed: rgb_mlp expects the GLO columns (models.py:269-272)"
        elif self.hyper_slice_method not in ('none', 'bendy_sheet', 'axis_aligned_plane'):
            self._forward_error = f'Unknown hyper slice method {self.hyper_slice_method}.'   # models.py:394-396

        # ---- the kernels' view of the model ---------------------------------------------------------------------------
        cond_a = self.use_nerf_embed and self.use_alpha_condition
        cond_r = self.use_nerf_embed and self.use_rgb_condition
        flags = (_lib.HN_FLAG_ALPHA_COND if cond_a else 0) | (_lib.HN_FLAG_RGB_COND if cond_r else 0)
        self._ids_key, n_rows = None, 0
        if self.use_warp:
            flags |= _lib.HN_FLAG_WARP_SE3 if self._se3 else _lib.HN_FLAG_WARP_TRANSLATION
            flags |= _lib.HN_FLAG_SLICE_AXIS if self.hyper_slice_method == 'axis_aligned_plane' else _lib.HN_FLAG_SLICE_BENDY
            self._ids_key, n_rows = self.warp_embed_key, n_embed(self.warp_embed_key)
        elif cond_a or cond_r:
            # without warp the condition comes from nerf_embed[metadata['warp']] (models.py:425-430)
            self._ids_key, n_rows = self.nerf_embed_key, n_embed(self.nerf_embed_key)
        self._desc = _lib.ModelDesc(GLO_dim, hyper_slice_out_dim if self.use_warp else 0, xyz_fourier_dim, hyper_fourier_dim,
                                    view_fourier_dim, modules.SE3Field.max_deg if self._se3 else modules.TranslationField.n_freq,
                                    modules.HyperSheetMLP.n_freq, n_rows, flags)
        self._slot_cache = None
        self._pack_levels = 2
        self._init_packing()
        self._flat_grads = None
        self._flat_off_cache = None
        self._grad_off_cache = None
        self._size_cache = {}
        if self._forward_error is None:
            sizes = _lib.Sizes()
            check(lib().hn_query(C.byref(self._desc), 0, C.byref(sizes)), "hn_query")   # rejects shapes that are not built
            self._packed_bytes = sizes.packed_bytes
            n_params = sum(p.numel() for p in self._slot_params() if p is not None)
            if n_params != sizes.flat_param_floats:
                raise _lib.NativeLibraryError(f"parameter layout mismatch: module has {n_params} kernel-visible parameters, "
                                              f"library expects {sizes.flat_param_floats}")

    def _bind_sub_modules(self):
        """Lets `self.warp_field(...)` / `self.hyper_sheet_mlp(...)` be called on their own (modules._FusedOnly._bind)."""
        if self.use_warp:
            self.warp_field._bind(self)
        if 'hyper_sheet_mlp' in self._modules:
            self.hyper_sheet_mlp._bind(self)

    def __setstate__(self, state):       # copy.deepcopy / pickle
        super().__setstate__(state)
        self._bind_sub_modules()

    # ------------------------------------------------------------------------------------------------------
    # native plumbing
    # ------------------------------------------------------------------------------------------------------
    def _slot_params(self):
        """The parameter tensors by canonical slot (include/hypernerf_b200.h, HN_NUM_PARAM_TENSORS entries); None for a
        slot this configuration does not have."""
        if self._slot_cache is not None:
            return self._slot_cache
        out = [None] * _lib.HN_NUM_PARAM_TENSORS

        def put(first, lins):
            for i, lin in enumerate(lins):
                out[first + 2 * i], out[first + 2 * i + 1] = lin.weight, lin.bias

        bendy = self.hyper_slice_method == 'bendy_sheet'
        if self.use_warp:
            out[0] = self.warp_embed.embed.weight
            if bendy:
                put(1, list(self.hyper_sheet_mlp.mlp.linears) + [self.hyper_sheet_mlp.mlp.logit_layer])
            if self._se3:
                wf = self.warp_field
                put(15, list(wf.trunk.linears) + [wf.trunk.logit_layer])
                put(94, [wf.w_net.linears[0], wf.w_net.logit_layer, wf.v_net.linears[0], wf.v_net.logit_layer])
            else:
                put(15, list(self.warp_field.mlp.linears) + [self.warp_field.mlp.logit_layer])
        elif self.use_nerf_embed:
            out[93] = self.nerf_embed.embed.weight
        for level, nm in enumerate((self.nerf_mlps_coarse, self.nerf_mlps_fine)):
            put(29 + 32 * level, list(nm.trunk_mlp.linears) + [nm.trunk_mlp.logit_layer, nm.bottleneck_mlp] +
                list(nm.rgb_mlp.linears) + [nm.rgb_mlp.logit_layer, nm.alpha_mlp])
        self._slot_cache = out
        return out

    def _slots_present(self):
        return [i for i, p in enumerate(self._slot_params()) if p is not None]

    def _canonical_params(self):
        """The kernel-visible parameter tensors in slot order (the `*params` of the autograd functions)."""
        return [p for p in self._slot_params() if p is not None]

    def _warp_slots(self):
        """The slots of the warp stage (GLO table, warp field, hyper sheet): everything but the two template levels."""
        lo, hi = self._level_param_range(0)[0], self._level_param_range(1)[1]
        return [i for i in self._slots_present() if not lo <= i < hi]

    def _warp_params(self):
        """The `*params` of _FusedWarp, detached when grad mode is off (the inference kernel then writes no stash)."""
        slots = self._slot_params()
        params = [slots[i] for i in self._warp_slots()]
        return params if torch.is_grad_enabled() else [q.detach() for q in params]

    @staticmethod
    def _level_param_range(level):
        return 29 + 32 * level, 29 + 32 * (level + 1)

    def _c_offsets(self, offset_of):
        return (C.c_int64 * _lib.HN_NUM_PARAM_TENSORS)(*[-1 if p is None else offset_of(p) for p in self._slot_params()])

    def _param_offsets(self, base):
        """Element offsets of the slot parameters relative to `base` (hn_pack_weights); -1 for absent slots."""
        return self._c_offsets(lambda p: (p.data_ptr() - base) // 4)

    def _grad_offsets(self):
        """Private flat gradient layout (autograd path without train.FlatGrads): (offsets by slot, total floats)."""
        if self._grad_off_cache is None:
            offs, total = {}, 0
            for p in self._canonical_params():
                offs[id(p)] = total
                total += (p.numel() + 3) // 4 * 4  # 16-byte aligned slices
            self._grad_off_cache = (self._c_offsets(lambda p: offs[id(p)]), total)
        return self._grad_off_cache

    def _flat_offsets(self):
        """Offsets by slot into the attached train.FlatGrads buffer."""
        if self._flat_off_cache is None:
            self._flat_off_cache = self._c_offsets(self._flat_grads.offset_of)
        return self._flat_off_cache

    def attach_flat_grads(self, flat_grads):
        """Opt-in: hn_mlp_bwd accumulates directly into `flat_grads.flat` (train.FlatGrads built over
        `self.parameters()`), bypassing autograd's per-tensor accumulation.  Pass None to detach."""
        if flat_grads is not None:
            for q in self._canonical_params():
                flat_grads.offset_of(q)    # raises if a kernel-visible parameter is not part of the buffer
        self._flat_grads = flat_grads
        self._flat_off_cache = None

    def _sizes(self, n_samples):
        s = self._size_cache.get(n_samples)
        if s is None:
            s = _lib.Sizes()
            check(lib().hn_query(C.byref(self._desc), n_samples, C.byref(s)), "hn_query")
            self._size_cache[n_samples] = s
        return s

    # ------------------------------------------------------------------------------------------------------
    # reference API
    # ------------------------------------------------------------------------------------------------------
    @property
    def num_nerf_embeds(self):
        return max(self.embeddings_dict[self.nerf_embed_key]) + 1

    @property
    def num_warp_embeds(self):
        return max(self.embeddings_dict[self.warp_embed_key]) + 1

    @property
    def num_hyper_embeds(self):
        return max(self.embeddings_dict[self.hyper_embed_key]) + 1

    @property
    def nerf_embeds(self):
        return torch.tensor(self.embeddings_dict[self.nerf_embed_key])

    @property
    def warp_embeds(self):
        return torch.tensor(self.embeddings_dict[self.warp_embed_key])

    @property
    def hyper_embeds(self):
        return torch.tensor(self.embeddings_dict[self.hyper_embed_key])

    @staticmethod
    def _encode_embed(embed, embed_fn):
        """models.py:352-374: a (*, 1) id, or (*, 3) = (left id, right id, progression) blended linearly."""
        if embed.shape[-1] == 3:
            left, right, progression = torch.split(embed, 1, dim=-1)   # (the reference's split size 3 returns one chunk
            left = embed_fn(left.type(torch.int32))                    #  and cannot unpack: :368; one column each is meant)
            right = embed_fn(right.type(torch.int32))
            return (1.0 - progression) * left + progression * right
        return embed_fn(embed)

    def encode_hyper_embed(self, metadata):
        """models.py:376-396."""
        if self.hyper_slice_method in ('axis_aligned_plane', 'bendy_sheet'):
            if self.hyper_use_warp_embed:
                return self._encode_embed(metadata[self.warp_embed_key], self.warp_embed)
            return self._encode_embed(metadata[self.hyper_embed_key], self.hyper_embed)
        raise RuntimeError(f'Unknown hyper slice method {self.hyper_slice_method}.')

    def encode_nerf_embed(self, metadata):
        return self._encode_embed(metadata[self.nerf_embed_key], self.nerf_embed)

    def encode_warp_embed(self, metadata):
        return self._encode_embed(metadata[self.warp_embed_key], self.warp_embed)

    @property
    def has_hyper(self):
        return self.hyper_slice_method != 'none'

    @property
    def has_hyper_embed(self):
        return self.has_hyper

    @property
    def has_embeds(self):
        return self.has_hyper_embed or self.use_warp or self.use_nerf_embed

    # ------------------------------------------------------------------------------------------------------
    # pre-encoded embeddings and the pieces of render_samples (models.py:447-585)
    # ------------------------------------------------------------------------------------------------------
    def _embed_view(self, embed):
        """This model with its GLO table replaced by per-ray embedding vectors: `embed` (B, G), (B, 1, G) or the broadcast
        (B, S, G) of models.py:627-632 (row 0 of the sample axis is taken: embeddings are per ray).  A shallow copy that
        shares every parameter; its table slot is `embed` itself, so the kernels read ray b's vector at id b, weights are
        packed per view, and the gradient of the table slot is the gradient with respect to `embed`."""
        if self._ids_key is None:
            raise RuntimeError("this configuration takes no metadata embedding")
        e = embed[:, 0, :] if embed.dim() == 3 else embed
        if e.dim() != 2 or e.shape[1] != self.GLO_dim:
            raise ValueError(f"embedding must be (B, {self.GLO_dim}) or (B, S, {self.GLO_dim}), got {tuple(embed.shape)}")
        e = e.to(torch.float32).contiguous()
        view = object.__new__(type(self))           # shallow: shares _parameters / _modules (and the sub-modules'
        view.__dict__.update(self.__dict__)         # back references, which keep pointing at self)
        d = self._desc
        view._desc = _lib.ModelDesc(d.glo_dim, d.hyper_dim, d.xyz_freqs, d.hyper_freqs, d.view_freqs, d.warp_freqs,
                                    d.sheet_freqs, e.shape[0], d.flags)
        slots = list(self._slot_params())
        slots[0 if self.use_warp else 93] = e
        view._slot_cache = slots
        view._init_packing()
        view._flat_grads, view._flat_off_cache, view._grad_off_cache, view._size_cache = None, None, None, {}
        sizes = _lib.Sizes()
        check(lib().hn_query(C.byref(view._desc), 0, C.byref(sizes)), "hn_query")
        view._packed_bytes = sizes.packed_bytes
        return view

    def _encoded_view(self, metadata):
        """metadata_encoded=True (models.py:605-625, 420-421): 'encoded_warp' / 'encoded_hyper' / 'encoded_nerf' hold the
        embedding vectors themselves.  The kernels take ONE vector per ray for the warp field, the hyper sheet / hyper point
        and the template condition (the reference shares them too: models.py:167-182, 421-423), so the entries this
        configuration reads must be the same tensor."""
        keys = []
        if self.use_warp:
            keys.append('encoded_warp')
            if self.has_hyper_embed:
                keys.append('encoded_hyper')
        if self.use_nerf_embed:
            keys.append('encoded_nerf')
        tensors = [metadata[k] for k in keys]
        first = tensors[0]
        for k, t in zip(keys[1:], tensors[1:]):
            if t is not first and not (t.shape == first.shape and t.data_ptr() == first.data_ptr()):
                raise NotImplementedError(f"metadata_encoded with '{k}' different from '{keys[0]}' is not built: the fused "
                                          "kernels share one embedding per ray between warp, slicing and conditioning")
        return self._embed_view(first)

    def apply_warp(self, points, warp_embed, extra_params):
        """models.py:583-585: `warp_embed` holds metadata IDS here (the method embeds them itself); returns
        {'warped_points': (B, S, 3)}.  Runs the warp stage alone (hn_mlp_fwd_warp) on the level-0 blob."""
        if not self.use_warp:
            raise AttributeError("'NerfModel' object has no attribute 'warp_field'")   # as in the reference
        warped = _FusedWarp.apply(self, pe_alphas(extra_params), points, warp_embed, *self._warp_params())
        return {'warped_points': warped[..., :3]}

    def map_points(self, points, warp_embed, hyper_embed, extra_params, use_warp=True, return_warp_jacobian=False,
                   hyper_point_override=None):
        """models.py:545-581: embedding VECTORS in ((B, S, G) broadcasts of per-ray rows), (warped points (B, S, 3 + H),
        None) out.  One launch of the warp stage (hn_mlp_fwd_warp) on a view whose table is the given vectors."""
        if not (self.use_warp and use_warp):
            return points, None
        if return_warp_jacobian and self._se3:
            raise NotImplementedError(_SE3_JACOBIAN)
        if hyper_point_override is not None:
            raise NotImplementedError('hyper_point_override is not implemented.')
        if self._forward_error is not None:
            raise RuntimeError(self._forward_error)
        if hyper_embed is not None and hyper_embed is not warp_embed and hyper_embed.data_ptr() != warp_embed.data_ptr():
            raise NotImplementedError("distinct warp / hyper embeddings are not built (one embedding per ray)")
        view = self._embed_view(warp_embed)
        ids = torch.arange(points.shape[0], device=points.device, dtype=torch.int64)
        if return_warp_jacobian:   # (warped, jac (B, S, 3, 3)): warping.py:115-122
            return _FusedWarpJacobian.apply(view, pe_alphas(extra_params), points, ids, *view._warp_params())
        return _FusedWarp.apply(view, pe_alphas(extra_params), points, ids, *view._warp_params()), None

    def map_spatial_points(self, points, warp_embed, extra_params, use_warp=True, return_warp_jacobian=False):
        """models.py:495-512."""
        if not (self.use_warp and use_warp):
            return points, None
        warped, jac = self.map_points(points, warp_embed, None, extra_params, use_warp, return_warp_jacobian)
        return warped[..., :3], jac

    def map_hyper_points(self, points, hyper_embed, extra_params, hyper_point_override=None):
        """models.py:514-543: the hyper coordinates (B, S, H); None without slicing."""
        if hyper_point_override is not None:
            raise NotImplementedError('hyper_point_override is not implemented.')
        if self.hyper_slice_method not in ('axis_aligned_plane', 'bendy_sheet') or not self.use_warp:
            return None
        warped, _ = self.map_points(points, hyper_embed, hyper_embed, extra_params)
        return warped[..., 3:]

    def query_template(self, level, points, viewdirs, metadata, extra_params, metadata_encoded=False):
        """models.py:447-493: the template NeRF of one level on (warped) points (B, S, 3 [+ H]) -> (rgb (B, S, 3),
        sigma (B, S)), with the density noise of model_utils.py:300-317 when the model has one."""
        if self._forward_error is not None:
            raise RuntimeError(self._forward_error)
        B, S = points.shape[0], points.shape[1]
        owner, ids = self, None
        if self._ids_key is not None and metadata_encoded:
            owner = self._encoded_view(metadata)
            ids = torch.arange(B, device=points.device, dtype=torch.int64)
        elif self._ids_key is not None:
            ids = metadata[self._ids_key]
        noise, noise_std = None, 0.0
        if (self.noise_std is not None) and self.noise_std > 0.0 and self.use_stratified_sampling:
            noise = torch.randn((B, S, 1), device=points.device, dtype=torch.float32)
            noise_std = float(self.noise_std)
        params = owner._canonical_params() if torch.is_grad_enabled() else [q.detach() for q in owner._canonical_params()]
        with owner.packed_frozen(extra_params):
            sigma, rgb = _FusedTrunk.apply(owner, (1 if level == 'fine' else 0, pe_alphas(extra_params)), points, viewdirs,
                                           ids, noise, noise_std, *params)
        return rgb, sigma

    def render_samples(self, level, points, z_vals, directions, viewdirs, metadata, extra_params, use_warp=True,
                       metadata_encoded=False, return_warp_jacobian=False, use_sample_at_infinity=False,
                       render_opts=None, _inherited=None, _view=None):
        """models.py:587-671.  _inherited = (warped points of the inherited depths (B,Ni,3+H), their positions (B,Ni) and
        the positions (B,S-Ni) of the remaining depths in the sorted row): see `reuse_coarse_warp`."""
        if self._forward_error is not None:
            raise RuntimeError(self._forward_error)
        if return_warp_jacobian and self.use_warp and self._se3:
            raise NotImplementedError(_SE3_JACOBIAN)
        if self.use_warp and not use_warp:
            # the reference hands the raw 3-channel points to a trunk built for posenc(xyz) + posenc(hyper) channels
            raise RuntimeError("use_warp=False at call time on a model built with use_warp=True: the template expects the "
                               "hyper channels (models.py:568-569, 269-270)")
        if metadata.get('hyper_point') is not None:
            raise NotImplementedError('hyper_point_override is not implemented.')  # models.py:528-529
        out = {'points': points}
        B, S = points.shape[0], points.shape[1]
        owner, ids = self, None
        if self._ids_key is not None and metadata_encoded:
            # pre-encoded metadata (models.py:605-625, 420-421): the kernels read ray b's embedding from row b of a table
            owner = _view if _view is not None else self._encoded_view(metadata)
            ids = torch.arange(B, device=points.device, dtype=torch.int64)
        elif self._ids_key is not None:
            ids = metadata[self._ids_key]
        noise, noise_std = None, 0.0
        if (self.noise_std is not None) and self.noise_std > 0.0 and self.use_stratified_sampling:
            # noise_regularize (model_utils.py:300-317): same draw, same shape, applied inside the kernel
            noise = torch.randn((B, S, 1), device=points.device, dtype=torch.float32)
            noise_std = float(self.noise_std)
        params = owner._canonical_params()
        if not torch.is_grad_enabled():
            # autograd.Function reports needs_input_grad for parameters even under no_grad; detached parameters make
            # the eval path (eval.py:77 @torch.no_grad) take the inference kernel, which writes no activation stash
            params = [q.detach() for q in params]
        lvl = (1 if level == 'fine' else 0, pe_alphas(extra_params))
        if not self.use_warp:
            # map_points returns the raw points (models.py:568-569): the template alone
            sigma, rgb = _FusedTrunk.apply(owner, lvl, points, viewdirs, ids, noise, noise_std, *params)
            warped_points = points
        elif _inherited is None:
            sigma, rgb, warped_points = _FusedMlp.apply(owner, lvl, points, viewdirs, ids, noise, noise_std, *params)
        else:
            known_warped, pos_known, pos_new = _inherited
            sigma, rgb, warped_points = _FusedFineLevel.apply(owner, lvl, points, viewdirs, ids, noise, noise_std, known_warped,
                                                              pos_known, pos_new, *params)
        if return_warp_jacobian and self.use_warp:
            # models.py:650-652: the warp field's Jacobian at this level's points (for the elastic loss)
            _, out['warp_jacobian'] = _FusedWarpJacobian.apply(owner, lvl[1], points, ids, *owner._warp_params())
        sigma = filter_sigma(points, sigma, render_opts)
        out['warped_points'] = warped_points
        comp = model_utils.volumetric_rendering(rgb, sigma, z_vals, directions,
                                                use_white_background=self.use_white_background,
                                                sample_at_infinity=use_sample_at_infinity, _return_index=True)
        depth_indices = comp.pop('_med_idx')
        out.update(comp)
        # models.py:664-669: gather with a (B,1,1) index -> channel 0 of the warped point at the median sample
        out['med_points'] = torch.gather(warped_points, dim=-2, index=depth_indices[..., None, None])
        return out

    def forward(self, rays_dict: Dict[str, Any], extra_params: Dict[str, Any], metadata_encoded=False, use_warp=True,
                return_points=False, return_weights=False, return_warp_jacobian=False, near=None, far=None,
                use_sample_at_infinity=None, render_opts=None, deterministic=False):
        """models.py:673-780.  Returns {'coarse': {...}, 'fine': {...}} with the reference's keys."""
        if self._forward_error is not None:
            raise RuntimeError(self._forward_error)
        if rays_dict['origins'].shape[0] == 0:
            raise ValueError("NerfModel.forward: empty ray batch (the reference fails on it too: model_utils.py:389, models.py:668)")
        # re-packs the bf16 weight blobs (with the encoding window of extra_params) unless an enclosing block froze them
        with self.packed_frozen(extra_params):
            return self._forward(rays_dict, extra_params, metadata_encoded, use_warp, return_points, return_weights,
                                 return_warp_jacobian, near, far, use_sample_at_infinity, render_opts, deterministic)

    def _forward(self, rays_dict, extra_params, metadata_encoded, use_warp, return_points, return_weights,
                 return_warp_jacobian, near, far, use_sample_at_infinity, render_opts, deterministic):
        use_warp = self.use_warp and use_warp
        # column slices of the (B,9) ray rows are strided views: one contiguous copy each, reused by every stage below
        origins = rays_dict['origins'].contiguous()
        directions = rays_dict['directions'].contiguous()
        metadata = rays_dict['metadata']
        if 'viewdirs' in rays_dict and rays_dict['viewdirs'] is not None:
            viewdirs = rays_dict['viewdirs']
        else:
            viewdirs = directions
        near = self.near if near is None else near
        far = self.far if far is None else far
        if use_sample_at_infinity is None:
            use_sample_at_infinity = self.use_sample_at_infinity

        view = self._encoded_view(metadata) if (metadata_encoded and self._ids_key is not None) else None
        z_vals, points = model_utils.sample_along_rays(origins, directions, self.num_coarse_samples, near, far,
                                                       self.use_stratified_sampling, self.use_linear_disparity)
        coarse_ret = self.render_samples('coarse', points, z_vals, directions, viewdirs, metadata, extra_params,
                                         use_warp=use_warp, metadata_encoded=metadata_encoded,
                                         return_warp_jacobian=return_warp_jacobian,
                                         use_sample_at_infinity=self.use_sample_at_infinity, _view=view)
        out = {'coarse': coarse_ret}
        if self.num_fine_samples > 0:
            inherited = None
            if self.use_stratified_sampling and self.reuse_coarse_warp and self.use_warp:
                z_vals, points, (pos_c, pos_n) = model_utils.sample_pdf_fused(
                    z_vals, coarse_ret['weights'], origins, directions, self.num_fine_samples, want_ranks=True)
                inherited = (coarse_ret['warped_points'], pos_c, pos_n)
            elif self.use_stratified_sampling:
                z_vals, points = model_utils.sample_pdf_fused(z_vals, coarse_ret['weights'], origins, directions,
                                                              self.num_fine_samples)
            else:
                z_mid = .5 * (z_vals[..., 1:] + z_vals[..., :-1])
                z_vals, points = model_utils.sample_pdf(z_mid, coarse_ret['weights'][..., 1:-1], origins, directions,
                                                        z_vals, self.num_fine_samples, False)
            out['fine'] = self.render_samples('fine', points, z_vals, directions, viewdirs, metadata, extra_params,
                                              use_warp=use_warp, metadata_encoded=metadata_encoded,
                                              return_warp_jacobian=return_warp_jacobian,
                                              use_sample_at_infinity=use_sample_at_infinity, render_opts=render_opts,
                                              _inherited=inherited, _view=view)
        return out
