"""Life cycle of the packed bf16 weight blobs (hn_pack_weights) behind NerfModel / NeRF.

The kernels read kernel-layout bf16 copies of the fp32 master parameters.  No host-side key can tell reliably that a
parameter changed: optimizers that update through `p.data` (the reference's RAdam / Ranger, utils/optimizers.py:88,163,
242,396), EMA swaps and manual re-initialisation do not bump `Tensor._version`.  So the policy is not a cache key:

  * every top-level call (NerfModel.forward, NeRF.query) re-packs — one small launch per level, always correct;
  * callers that KNOW the weights cannot change between calls (the chunk loops of train.train_step and
    train.render_rays) wrap them in `with model.packed_frozen():` — packed once at entry, reused inside;
  * direct calls of the autograd functions outside any of those (tests, profiling scripts) fall back to a
    (`_version`, `data_ptr`) key, and `invalidate_packed()` drops the blobs explicitly.

Annealed positional encodings (`extra_params` alphas, include/hypernerf_b200.h: hn_pack_weights_windowed) are packed
into the blobs: a blob carries the window it was packed with, next to a 4-float device snapshot of its alphas that the
forward saves for the weight gradient.  A frozen block is packed with the alphas given at its entry; a forward inside it
that asks for other alphas raises instead of running on the stale blob.  Without alphas the unwindowed entry points run.
"""
import contextlib
import ctypes as C

import torch

from . import _lib
from ._lib import check, lib, ptr, stream


# extra_params keys of the encoding windows, in the order of the kernels' pe_alpha array
PE_ALPHA_KEYS = ('warp_alpha', 'hyper_sheet_alpha', 'nerf_alpha', 'hyper_alpha')


def pe_alphas(extra_params):
    """The encoding window of `extra_params`: None when no alpha is set (the unwindowed path), else a tuple of the four
    alphas in PE_ALPHA_KEYS order with +inf (no window) for the unset ones.  A NaN alpha raises ValueError."""
    if not extra_params:
        return None
    vals = [extra_params.get(k) for k in PE_ALPHA_KEYS]
    if all(v is None for v in vals):
        return None
    out = tuple(float('inf') if v is None else float(v) for v in vals)
    for k, v in zip(PE_ALPHA_KEYS, out):
        if v != v:
            raise ValueError(f"extra_params['{k}'] is NaN")
    return out


class _DeviceWindow:
    """Window read from a caller-owned device buffer (train.GraphedTrainStep(windowed=True)): its values change between
    graph replays without a re-pack, so the host cannot compare them."""

    def __init__(self, buf):
        self.buf = buf


class PackedWeights:
    """Mixin: needs `_canonical_params()`, `_desc`, `_packed_bytes` and `_pack_levels` (1 or 2)."""

    def _init_packing(self):
        self._pack_cache = {}
        self._pack_depth = 0
        self._frozen_window = None

    def invalidate_packed(self):
        """Drop the packed blobs: the next call re-packs from the fp32 parameters."""
        self._pack_cache = {}

    def _pack_key(self, params):
        return (tuple(p._version for p in params), tuple(p.data_ptr() for p in params))

    def refresh_packed(self, window=None):
        """Pack every level now (hn_pack_weights), unconditionally.  window: None, a pe_alphas() tuple, or a
        _DeviceWindow (hn_pack_weights_windowed)."""
        params = self._canonical_params()
        dev = params[0].device
        if dev.type != 'cuda':
            raise _lib.NativeLibraryError("parameters must live on a CUDA device (no CPU path)")
        for p in params:
            if p.dtype != torch.float32 or not p.is_contiguous():
                raise _lib.NativeLibraryError("parameters must be contiguous fp32 tensors")
        base = min(p.data_ptr() for p in params)
        if hasattr(self, "_param_offsets"):      # slot table with gaps (NerfModel): -1 for absent slots
            offs = self._param_offsets(base)
        else:
            offs = (C.c_int64 * len(params))(*[(p.data_ptr() - base) // 4 for p in params])
        key = self._pack_key(params)
        alpha = None
        if isinstance(window, _DeviceWindow):
            alpha = window.buf
        elif window is not None:
            alpha = torch.tensor(window, device=dev, dtype=torch.float32)   # this blob's snapshot of its alphas
        for level in range(self._pack_levels):
            hit = self._pack_cache.get(level)
            # the blob is reused as storage when nothing that was handed out can still be referenced by a pending
            # backward: a new tensor per re-pack keeps saved-for-backward blobs of earlier forwards intact
            packed = torch.empty(self._packed_bytes, device=dev, dtype=torch.uint8)
            if alpha is None:
                check(lib().hn_pack_weights(C.byref(self._desc), C.c_void_p(base), offs, level, ptr(packed), stream()),
                      "hn_pack_weights")
            else:
                check(lib().hn_pack_weights_windowed(C.byref(self._desc), C.c_void_p(base), offs, level, ptr(packed),
                                                     ptr(alpha), stream()), "hn_pack_weights_windowed")
            _lib.count(1)
            self._pack_cache[level] = (key, packed, window, alpha)
            del hit

    @contextlib.contextmanager
    def packed_frozen(self, extra_params=None, _window=None):
        """Pack once at entry of the outermost block, with the encoding window of `extra_params`; every forward inside
        reuses the blobs (and must ask for the same alphas)."""
        window = pe_alphas(extra_params) if _window is None else _window
        if self._pack_depth == 0:
            self.refresh_packed(window)
            self._frozen_window = window
        elif _window is not None or not isinstance(self._frozen_window, _DeviceWindow):
            self._check_window(window)
        self._pack_depth += 1
        try:
            yield self
        finally:
            self._pack_depth -= 1
            if self._pack_depth == 0:
                self._frozen_window = None

    def _check_window(self, window):
        if window != self._frozen_window:
            raise ValueError(f"the weights are frozen with the encoding window {self._frozen_window} (packed_frozen), "
                             f"but a forward inside the block asks for {window}: pass the same extra_params alphas")

    def _packed_window(self, level, window):
        """(blob, its device alphas or None) of `level` for the encoding window `window` (pe_alphas())."""
        hit = self._pack_cache.get(level)
        if self._pack_depth > 0 and hit is not None:
            if not isinstance(self._frozen_window, _DeviceWindow):   # a device window is what the caller installed
                self._check_window(window)
            return hit[1], hit[3]
        if hit is None or hit[0] != self._pack_key(self._canonical_params()) or hit[2] != window:
            self.refresh_packed(window)
        hit = self._pack_cache[level]
        return hit[1], hit[3]

    def _packed_weights(self, level=0):
        return self._packed_window(level, None)[0]
