"""ctypes binding of libhypernerf_b200.so (include/hypernerf_b200.h).

The library is the product: there is no CPU or torch fallback behind these calls.  If the shared object is
missing, or a call returns non-zero, this module raises.
"""
import ctypes as C
import os
import subprocess

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("HN_LIB") or os.path.join(_HERE, "libhypernerf_b200.so")  # HN_LIB: profiling build
HN_NUM_PARAM_TENSORS = 102
HN_FLAG_WARP_TRANSLATION = 1
HN_FLAG_SLICE_BENDY = 2
HN_FLAG_STATIC_NERF = 4
HN_FLAG_SLICE_AXIS = 8
HN_FLAG_ALPHA_COND = 16
HN_FLAG_RGB_COND = 32
HN_FLAG_WARP_SE3 = 64
HN_NUM_STATIC_PARAM_TENSORS = 24
HN_COMP_WHITE_BKGD = 1
HN_COMP_ACC_ALL = 2

EXPORTS = [
    "hn_abi_version", "hn_last_error", "hn_query", "hn_pack_weights", "hn_sample_coarse", "hn_sample_pdf", "hn_sample_pdf_ranks",
    "hn_composite_fwd", "hn_composite_bwd", "hn_filter_sigma", "hn_mse_loss", "hn_make_ndc_rays", "hn_adam_step", "hn_mlp_fwd", "hn_mlp_bwd", "hn_mlp_bwd_data", "hn_mlp_bwd_weights", "hn_mlp_fwd_trunk", "hn_mlp_bwd_trunk", "hn_mlp_bwd_trunk_data", "hn_mlp_bwd_trunk_weights",
    "hn_pack_weights_windowed", "hn_mlp_bwd_weights_windowed", "hn_mlp_bwd_trunk_weights_windowed",
    "hn_mlp_fwd_warp", "hn_mlp_bwd_warp_data", "hn_mlp_bwd_warp_weights", "hn_background_loss",
    "hn_mlp_fwd_warp_tangent", "hn_elastic_loss",
]
# microbenchmarks / descriptor probes: their own library and header (include/hypernerf_b200_probe.h), not the product ABI
PROBE_LIB_PATH = os.path.join(_HERE, "libhypernerf_b200_probe.so")
PROBE_EXPORTS = ["hn_umma_probe", "hn_umma_probe2", "hn_umma_rate", "hn_umma_rate2", "hn_umma_rate3", "hn_umma_rate4",
                 "hn_epi_rate", "hn_tmem_rate", "hn_overlap_rate"]


class ModelDesc(C.Structure):
    _fields_ = [(n, C.c_int32) for n in
                ("glo_dim", "hyper_dim", "xyz_freqs", "hyper_freqs", "view_freqs", "warp_freqs", "sheet_freqs",
                 "num_embeddings", "flags")] + [("reserved", C.c_int32 * 7)]


class Sizes(C.Structure):
    _fields_ = [("packed_bytes", C.c_int64), ("saved_bytes", C.c_int64), ("workspace_bytes", C.c_int64),
                ("flat_param_floats", C.c_int64), ("warp_saved_bytes", C.c_int64), ("warp_workspace_bytes", C.c_int64),
                ("reserved", C.c_int64 * 2)]


class NativeLibraryError(RuntimeError):
    pass


def build(verbose: bool = False) -> str:
    """Compile csrc/ for sm_100a into libhypernerf_b200.so (nvcc cross-compiles without a GPU)."""
    cmd = ["make", "-C", os.path.join(_HERE, "csrc"), "-j8"]
    res = subprocess.run(cmd, capture_output=True, text=True)
    if verbose or res.returncode != 0:
        print(res.stdout)
        print(res.stderr)
    if res.returncode != 0:
        raise NativeLibraryError("building libhypernerf_b200.so failed")
    return LIB_PATH


_lib = None


def lib():
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise NativeLibraryError(
            f"{LIB_PATH} not found: build it with `python -c 'import __graft_entry__ as g; g.build()'` "
            "(there is no fallback path)")
    L = C.CDLL(LIB_PATH)
    vp, i64, i32, f32 = C.c_void_p, C.c_int64, C.c_int, C.c_float
    L.hn_abi_version.restype = C.c_int
    L.hn_last_error.restype = C.c_char_p
    L.hn_query.argtypes = [C.POINTER(ModelDesc), i64, C.POINTER(Sizes)]
    L.hn_pack_weights.argtypes = [C.POINTER(ModelDesc), vp, C.POINTER(C.c_int64), i32, vp, vp]
    L.hn_sample_coarse.argtypes = [vp, vp, vp, vp, vp, i64, i32, vp, vp, vp]
    L.hn_sample_pdf.argtypes = [vp, vp, vp, i64, vp, vp, vp, i64, i32, i32, i32, vp, vp, vp, vp]
    L.hn_sample_pdf_ranks.argtypes = [vp, vp, vp, i64, vp, vp, vp, i64, i32, i32, i32, vp, vp, vp, vp, vp, vp]
    L.hn_composite_fwd.argtypes = [vp, vp, vp, vp, i64, i32, i32, f32, f32, vp, vp, vp, vp, vp, vp, vp]
    L.hn_composite_bwd.argtypes = [vp, vp, vp, vp, i64, i32, i32, f32, f32, vp, vp, vp, vp, vp, vp, vp]
    L.hn_filter_sigma.argtypes = [vp, vp, vp, i64, f32, i32, C.POINTER(C.c_float), vp, vp]
    L.hn_mse_loss.argtypes = [vp, vp, vp, i64, f32, vp, vp, vp, vp]
    L.hn_make_ndc_rays.argtypes = [i32, i32, f32, C.POINTER(C.c_float), f32, f32, i32, vp, vp]
    L.hn_adam_step.argtypes = [vp, vp, vp, vp, i64, f32, f32, f32, f32, f32, i64, f32, vp]
    L.hn_mlp_fwd.argtypes = [C.POINTER(ModelDesc), vp, vp, vp, vp, vp, f32, i64, i32, vp, i32, vp, vp, vp, vp, vp, vp]
    L.hn_mlp_bwd.argtypes = [C.POINTER(ModelDesc), vp, vp, vp, vp, vp, vp, vp, vp, vp, i64, i32, vp, i32, i32,
                             C.POINTER(C.c_int64), vp, vp, vp, vp, vp]
    L.hn_mlp_bwd_data.argtypes = L.hn_mlp_bwd.argtypes
    L.hn_mlp_bwd_weights.argtypes = [C.POINTER(ModelDesc), vp, i64, i32, i32, C.POINTER(C.c_int64), vp, vp, vp]
    L.hn_mlp_fwd_trunk.argtypes = [C.POINTER(ModelDesc), vp, vp, vp, vp, vp, f32, i64, i32, vp, i32, vp, vp, vp, vp, vp]
    L.hn_mlp_bwd_trunk.argtypes = [C.POINTER(ModelDesc), vp, vp, vp, vp, vp, vp, vp, vp, vp, i64, i32, vp, i32, i32,
                                   C.POINTER(C.c_int64), vp, vp, vp, vp]
    L.hn_mlp_bwd_trunk_data.argtypes = L.hn_mlp_bwd_trunk.argtypes
    L.hn_mlp_bwd_trunk_weights.argtypes = L.hn_mlp_bwd_weights.argtypes
    L.hn_pack_weights_windowed.argtypes = [C.POINTER(ModelDesc), vp, C.POINTER(C.c_int64), i32, vp, vp, vp]
    L.hn_mlp_bwd_weights_windowed.argtypes = [C.POINTER(ModelDesc), vp, i64, i32, i32, C.POINTER(C.c_int64), vp, vp, vp, vp]
    L.hn_mlp_bwd_trunk_weights_windowed.argtypes = L.hn_mlp_bwd_weights_windowed.argtypes
    L.hn_mlp_fwd_warp.argtypes = [C.POINTER(ModelDesc), vp, vp, vp, i64, i32, vp, vp, vp, vp]
    L.hn_mlp_bwd_warp_data.argtypes = [C.POINTER(ModelDesc), vp, vp, vp, vp, i64, i32, C.POINTER(C.c_int64), vp, vp, vp, vp,
                                       vp]
    L.hn_mlp_bwd_warp_weights.argtypes = [C.POINTER(ModelDesc), vp, i64, i32, C.POINTER(C.c_int64), vp, vp, vp, vp]
    L.hn_background_loss.argtypes = [vp, vp, i64, i32, f32, f32, f32, vp, vp, vp]
    L.hn_mlp_fwd_warp_tangent.argtypes = [C.POINTER(ModelDesc), vp, vp, vp, i64, i32, vp, vp, vp]
    L.hn_elastic_loss.argtypes = [vp, vp, i64, f32, f32, f32, f32, vp, vp, i32, vp]
    if hasattr(L, "hn_debug_set_timing_buffer"):   # role-timing builds only (make timing; HN_LIB selects them)
        L.hn_debug_set_timing_buffer.argtypes = [vp]
        L.hn_debug_set_timing_buffer.restype = C.c_int
    for name in EXPORTS:
        fn = getattr(L, name)
        if name not in ("hn_last_error",):
            fn.restype = C.c_int
    _lib = L
    return L


_probe = None


def probe_lib():
    """libhypernerf_b200_probe.so (include/hypernerf_b200_probe.h): test / measurement hooks, not the product ABI."""
    global _probe
    if _probe is not None:
        return _probe
    if not os.path.exists(PROBE_LIB_PATH):
        raise NativeLibraryError(f"{PROBE_LIB_PATH} not found: build it with __graft_entry__.build()")
    L = C.CDLL(PROBE_LIB_PATH)
    vp, i32 = C.c_void_p, C.c_int
    L.hn_last_error.restype = C.c_char_p
    L.hn_tmem_rate.argtypes = [i32, i32, i32, i32, vp, vp]
    L.hn_umma_rate.argtypes = [i32, i32, i32, i32, i32, i32, i32, vp, vp]
    L.hn_umma_rate2.argtypes = [i32] * 9 + [vp, vp]
    L.hn_umma_rate3.argtypes = [i32] * 5 + [vp, vp]
    L.hn_epi_rate.argtypes = [i32, i32, i32, vp, vp, vp]
    L.hn_umma_probe2.argtypes = [vp, vp, vp, i32, i32, vp]
    L.hn_umma_rate4.argtypes = [i32] * 5 + [vp, vp]
    L.hn_umma_probe.argtypes = [vp, vp, vp, i32, i32, i32, i32, vp]
    L.hn_overlap_rate.argtypes = [i32, i32, i32, i32, i32, i32, vp, vp, vp, vp]
    for name in PROBE_EXPORTS:
        getattr(L, name).restype = C.c_int
    _probe = L
    return L


# number of kernels of this library launched so far (bench.py reports the count inside its timed region)
launches = 0
# when a list, every MLP kernel call appends (name, n_samples, start_event, end_event) (bench.py roofline leg)
profile = None


def count(n: int):
    global launches
    launches += n


class timed:
    """Context manager: CUDA events around one kernel call on the current stream when profiling is on."""

    def __init__(self, name, n_samples):
        self.name, self.n = name, n_samples

    def __enter__(self):
        if profile is not None:
            self.e0 = torch.cuda.Event(enable_timing=True)
            self.e1 = torch.cuda.Event(enable_timing=True)
            self.e0.record()
        return self

    def __exit__(self, *exc):
        if profile is not None:
            self.e1.record()
            profile.append((self.name, self.n, self.e0, self.e1))


def check(rc: int, what: str, library=None):
    if rc != 0:
        msg = (library or lib()).hn_last_error().decode("utf-8", "replace")
        raise NativeLibraryError(f"{what} failed (rc={rc}): {msg}")


def ptr(t):
    """Device pointer of a contiguous CUDA tensor (None -> NULL)."""
    if t is None:
        return None
    if not t.is_cuda:
        raise NativeLibraryError("hypernerf_b200 kernels take CUDA tensors only (no CPU path)")
    if not t.is_contiguous():
        raise NativeLibraryError("hypernerf_b200 kernels take contiguous tensors")
    if t.device.index != torch.cuda.current_device():
        # the C entry points launch on the CURRENT device and stream(): a tensor of another GPU would be dereferenced by
        # the wrong device.  Callers on multi-GPU hosts wrap their calls in torch.cuda.device(t.device).
        raise NativeLibraryError(f"tensor lives on cuda:{t.device.index} but the current device is "
                                 f"cuda:{torch.cuda.current_device()}; use torch.cuda.set_device / torch.cuda.device()")
    return C.c_void_p(t.data_ptr())


def stream():
    return C.c_void_p(torch.cuda.current_stream().cuda_stream)


MIN_TORCH = (2, 4)   # torch.autograd.graph.increment_version(iterable), torch.amp.custom_fwd(device_type=...)
if tuple(int(x) for x in torch.__version__.split("+")[0].split(".")[:2]) < MIN_TORCH:
    raise ImportError(f"hypernerf_torch_b200 needs torch >= {MIN_TORCH[0]}.{MIN_TORCH[1]}, found {torch.__version__}")
