"""ctypes binding of libflowcon_b200.so (see include/flowcon_b200.h).

Plain pointers and sizes only: tensors are passed as `data_ptr()`, the stream as the raw cudaStream_t of
torch's current stream.  There is NO fallback: if the library has not been built, or a tensor is not a
CUDA fp32 tensor, the call raises.
"""
import ctypes
import os

import torch

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("FC_LIB") or os.path.join(_HERE, "lib", "libflowcon_b200.so")  # FC_LIB: A/B experiments only

FC_OK = 0
ERRORS = {-1: "invalid argument", -2: "unsupported configuration", -3: "CUDA launch error"}
STATUS_INPUT_OUTSIDE_DOMAIN = 1
STATUS_NEGATIVE_DISCRIMINANT = 2
TAILS_NONE, TAILS_LINEAR = 0, 1
AFFINE_BLOCKED, AFFINE_INTERLEAVED = 0, 1
BATCHNORM_TRAIN, BATCHNORM_EVAL_FORWARD, BATCHNORM_EVAL_INVERSE = 0, 1, 2
SCALE_SIGMOID2, SCALE_SOFTPLUS_CLAMP3, SCALE_SOFTPLUS_EPS = 0, 1, 2
LINEAR_A_T128, LINEAR_OUT_T128, LINEAR_RESIDUAL_GATES = 1, 2, 4
POINTWISE_SIGMOID, POINTWISE_TANH, POINTWISE_LEAKY_RELU, POINTWISE_EXP, POINTWISE_CAUCHY_CDF = 0, 1, 2, 3, 4

EXPORTS = ["fc_rqs_apply", "fc_rqs_backward", "fc_rqs_bins", "fc_linspline_apply", "fc_linspline_backward",
           "fc_quadspline_apply", "fc_quadspline_backward", "fc_cubicspline_apply", "fc_cubicspline_backward", "fc_affine_apply", "fc_affine_backward", "fc_sos_apply",
           "fc_sos_backward", "fc_sos_inverse_backward", "fc_stdnormal_log_prob", "fc_linear_pack", "fc_linear_apply", "fc_linear_rqs_apply",
           "fc_linear_affine_apply", "fc_linear_splitk_t_apply", "fc_linear_pack_transposed",
           "fc_linear_debug_profile",
           "fc_elementwise_last_path", "fc_conditioner_layer_bytes", "fc_conditioner_pack_layer", "fc_conditioner_rqs_apply", "fc_conditioner_sos_apply", "fc_conditioner_affine_apply", "fc_conditioner_store_apply", "fc_context_terms", "fc_conditioner_error", "fc_conditioner_profile",
           "fc_actnorm_apply", "fc_actnorm_workspace_floats", "fc_actnorm_backward",
           "fc_lulinear_apply", "fc_lulinear_workspace_floats", "fc_lulinear_backward",
           "fc_batchnorm_workspace_floats", "fc_batchnorm_stats", "fc_batchnorm_apply", "fc_batchnorm_backward",
           "fc_diagnormal_log_prob", "fc_diagnormal_log_prob_backward", "fc_diagnormal_sample",
           "fc_diagnormal_sample_backward", "fc_diagnormal_workspace_floats",
           "fc_pointwise_apply", "fc_pointwise_workspace_floats", "fc_pointwise_backward",
           "fc_made_inverse_smem_bytes", "fc_made_inverse_profile", "fc_made_inverse_rqs", "fc_made_inverse_affine",
           "fc_made_inverse_sos", "fc_made_inverse_linspline", "fc_made_inverse_quadspline", "fc_made_inverse_cubicspline",
           "fc_version", "fc_built_for_sm"]
COND_MAX_LAYERS = 10
COND_INITIAL, COND_BLOCK_FIRST, COND_BLOCK_SECOND, COND_FINAL = 0, 1, 2, 3
COND_TERM_NONE, COND_TERM_ADD, COND_TERM_ADD_RELU, COND_TERM_GATE = 0, 1, 2, 3


class RqsConfig(ctypes.Structure):
    """struct fc_rqs_config"""
    _fields_ = [("num_bins", ctypes.c_int32), ("tails", ctypes.c_int32), ("identity_init", ctypes.c_int32),
                ("inverse", ctypes.c_int32), ("left", ctypes.c_float), ("right", ctypes.c_float),
                ("bottom", ctypes.c_float), ("top", ctypes.c_float), ("min_bin_width", ctypes.c_float),
                ("min_bin_height", ctypes.c_float), ("min_derivative", ctypes.c_float), ("wh_scale", ctypes.c_float)]


class QuadSplineConfig(ctypes.Structure):
    """struct fc_quadspline_config"""
    _fields_ = [("num_bins", ctypes.c_int32), ("tails", ctypes.c_int32), ("inverse", ctypes.c_int32),
                ("left", ctypes.c_float), ("right", ctypes.c_float), ("bottom", ctypes.c_float), ("top", ctypes.c_float),
                ("min_bin_width", ctypes.c_float), ("min_bin_height", ctypes.c_float), ("wh_scale", ctypes.c_float)]


class PointwiseConfig(ctypes.Structure):
    """struct fc_pointwise_config"""
    _fields_ = [("op", ctypes.c_int32), ("inverse", ctypes.c_int32), ("slope", ctypes.c_float), ("eps", ctypes.c_float),
                ("temperature", ctypes.c_void_p)]


class Cols(ctypes.Structure):
    """struct fc_cols"""
    _fields_ = [("idx", ctypes.c_void_p), ("n", ctypes.c_int32)]


class LinearWeights(ctypes.Structure):
    """struct fc_linear_weights"""
    _fields_ = [("w", ctypes.c_void_p), ("bias", ctypes.c_void_p), ("n_pad", ctypes.c_int32),
                ("k_pad", ctypes.c_int32)]


class ConditionerLayer(ctypes.Structure):
    """struct fc_conditioner_layer"""
    _fields_ = [("kind", ctypes.c_int32), ("n_tiles", ctypes.c_int32), ("relu_next", ctypes.c_int32),
                ("term_mode", ctypes.c_int32), ("w_offset", ctypes.c_int64), ("bias", ctypes.c_void_p),
                ("winv", ctypes.c_void_p), ("terms", ctypes.c_void_p), ("term_width", ctypes.c_int64)]


class Conditioner(ctypes.Structure):
    """struct fc_conditioner"""
    _fields_ = [("weights", ctypes.c_void_p), ("n_layers", ctypes.c_int32), ("hidden", ctypes.c_int32),
                ("k_in", ctypes.c_int32), ("hidden_k", ctypes.c_int32), ("layers", ConditionerLayer * COND_MAX_LAYERS)]


MADE_MAX_TERM_ARRAYS = 8


class MadeTermArray(ctypes.Structure):
    """struct fc_made_term_array"""
    _fields_ = [("array", ctypes.c_int32), ("column", ctypes.c_int32), ("b_off", ctypes.c_int32), ("relu", ctypes.c_int32)]


class MadeProgramStruct(ctypes.Structure):
    """struct fc_made_program"""
    _fields_ = [("phases", ctypes.c_void_p), ("weights", ctypes.c_void_p), ("bias", ctypes.c_void_p),
                ("n_phases", ctypes.c_int32), ("features", ctypes.c_int32), ("params_per_feature", ctypes.c_int32),
                ("n_arrays", ctypes.c_int32), ("hidden", ctypes.c_int32), ("n_bias", ctypes.c_int32),
                ("terms", ctypes.c_void_p), ("term_width", ctypes.c_int32), ("n_term_arrays", ctypes.c_int32),
                ("term_arrays", MadeTermArray * MADE_MAX_TERM_ARRAYS)]


class LibraryMissing(RuntimeError):
    pass


_lib = None


def lib():
    """Load the library once; raise loudly when it is missing (no CPU / eager fallback exists)."""
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise LibraryMissing(
                "libflowcon_b200.so not found at {}. Build it with `python -m flowconductor_b200.build` "
                "(needs nvcc; targets sm_100a). flowconductor_b200 has no CPU or eager fallback.".format(LIB_PATH))
        L = ctypes.CDLL(LIB_PATH)
        vp, i64, i32, f32 = ctypes.c_void_p, ctypes.c_int64, ctypes.c_int32, ctypes.c_float
        L.fc_rqs_apply.argtypes = [vp, i64, vp, i64, vp, i64, vp, i32, i64, i32, Cols, Cols,
                                   ctypes.POINTER(RqsConfig), vp, vp]
        L.fc_rqs_backward.argtypes = [vp, i64, vp, i64, vp, i64, vp, vp, i64, vp, i64, i64, i32, Cols, Cols,
                                      ctypes.POINTER(RqsConfig), vp]
        L.fc_rqs_bins.argtypes = [vp, i64, vp, i64, i64, i32, Cols, ctypes.POINTER(RqsConfig), vp, vp, vp]
        L.fc_linspline_apply.argtypes = [vp, i64, vp, i64, vp, i64, vp, i32, i64, i32, Cols, Cols, i32, i32, f32, f32,
                                         f32, f32, i32, vp, vp]
        L.fc_linspline_backward.argtypes = [vp, i64, vp, i64, vp, i64, vp, vp, i64, vp, i64, i64, i32, Cols, Cols, i32,
                                            i32, f32, f32, f32, f32, i32, vp]
        L.fc_quadspline_apply.argtypes = [vp, i64, vp, i64, vp, i64, vp, i32, i64, i32, Cols, Cols,
                                          ctypes.POINTER(QuadSplineConfig), vp, vp]
        L.fc_quadspline_backward.argtypes = [vp, i64, vp, i64, vp, i64, vp, vp, i64, vp, i64, i64, i32, Cols, Cols,
                                             ctypes.POINTER(QuadSplineConfig), vp]
        L.fc_cubicspline_apply.argtypes = L.fc_quadspline_apply.argtypes
        L.fc_cubicspline_backward.argtypes = L.fc_quadspline_backward.argtypes
        L.fc_affine_apply.argtypes = [vp, i64, vp, i64, vp, i64, vp, i32, i64, i32, Cols, Cols, i32, i32, i32, vp]
        L.fc_affine_backward.argtypes = [vp, i64, vp, i64, vp, i64, vp, vp, i64, vp, i64, i64, i32, Cols, Cols, i32,
                                         i32, i32, vp]
        L.fc_sos_apply.argtypes = [vp, i64, vp, i64, vp, i64, vp, i32, i64, i32, i32, f32, i32, i32, f32, vp]
        L.fc_sos_backward.argtypes = [vp, i64, vp, i64, vp, i64, vp, vp, i64, vp, i64, i64, i32, i32, vp]
        L.fc_sos_inverse_backward.argtypes = L.fc_sos_backward.argtypes
        L.fc_stdnormal_log_prob.argtypes = [vp, i64, vp, vp, i64, i32, vp]
        L.fc_linear_pack.argtypes = [vp, i64, vp, i64, vp, i32, i32, vp, vp, i32, i32, vp, vp, vp]
        L.fc_linear_apply.argtypes = [vp, i64, i64, i32, ctypes.POINTER(LinearWeights), i32, vp, i64, i32, i32, vp,
                                      i64, i32, vp]
        L.fc_linear_rqs_apply.argtypes = [vp, i64, i64, i32, ctypes.POINTER(LinearWeights), i32, vp, i64, vp, i64, vp,
                                          i32, i32, Cols, Cols, ctypes.POINTER(RqsConfig), vp, i32, vp]
        L.fc_linear_affine_apply.argtypes = [vp, i64, i64, i32, ctypes.POINTER(LinearWeights), i32, vp, i64, vp, i64,
                                             vp, i32, i32, Cols, Cols, i32, i32, i32, vp]
        L.fc_linear_splitk_t_apply.argtypes = [vp, i64, i64, i64, ctypes.POINTER(LinearWeights), i32, vp, i64, i64, i32, vp, vp]
        L.fc_linear_pack_transposed.argtypes = [vp, i64, i64, i32, i32, i32, i32, vp, vp, vp]
        L.fc_conditioner_layer_bytes.argtypes = [i32, i32, i32]
        L.fc_conditioner_pack_layer.argtypes = [vp, i64, vp, i64, vp, i32, i32, vp, vp, i32, i32, i32, vp, vp, vp, vp]
        L.fc_conditioner_rqs_apply.argtypes = [ctypes.POINTER(Conditioner), vp, i64, i64, vp, i64, vp, i64, vp, i32, i32,
                                               Cols, Cols, ctypes.POINTER(RqsConfig), vp, vp]
        L.fc_conditioner_sos_apply.argtypes = [ctypes.POINTER(Conditioner), vp, i64, i64, vp, i64, vp, i64, vp, i32, i32,
                                               Cols, Cols, i32, f32, vp]
        L.fc_conditioner_affine_apply.argtypes = [ctypes.POINTER(Conditioner), vp, i64, i64, vp, i64, vp, i64, vp, i32,
                                                  i32, Cols, Cols, i32, i32, vp]
        L.fc_conditioner_store_apply.argtypes = [ctypes.POINTER(Conditioner), vp, i64, i64, vp, i64, i32, vp]
        L.fc_context_terms.argtypes = [vp, i64, i64, i32, vp, vp, i32, vp, vp]
        L.fc_conditioner_error.argtypes = [ctypes.POINTER(ctypes.c_int32)]
        L.fc_conditioner_profile.argtypes = [ctypes.POINTER(ctypes.c_uint64)]
        L.fc_actnorm_apply.argtypes = [vp, i64, vp, vp, vp, i64, vp, i32, i64, i32, i32, vp]
        L.fc_actnorm_workspace_floats.argtypes = [i64, i32]
        L.fc_actnorm_backward.argtypes = [vp, i64, vp, vp, vp, i64, vp, vp, i64, vp, vp, vp, i64, i32, i32, vp]
        L.fc_lulinear_apply.argtypes = [vp, i64, vp, vp, vp, vp, i64, vp, i32, i64, i32, vp]
        L.fc_lulinear_workspace_floats.argtypes = [i64, i32]
        L.fc_lulinear_backward.argtypes = [vp, i64, vp, vp, i64, vp, i64, vp, vp, vp, i64, i32, vp]
        L.fc_batchnorm_workspace_floats.argtypes = [i64, i32]
        L.fc_batchnorm_stats.argtypes = [vp, i64, vp, vp, vp, i64, i32, vp]
        L.fc_batchnorm_apply.argtypes = [vp, i64, vp, vp, vp, vp, f32, vp, i64, vp, i64, i32, i32, vp]
        L.fc_batchnorm_backward.argtypes = [vp, i64, vp, vp, vp, vp, f32, vp, i64, vp, vp, i64, vp, vp, vp, i64, i32,
                                            i32, vp]
        L.fc_diagnormal_log_prob.argtypes = [vp, i64, vp, i64, vp, vp, i64, i32, i64, vp]
        L.fc_diagnormal_log_prob_backward.argtypes = [vp, i64, vp, i64, vp, vp, i64, vp, vp, i64, i32, i64, vp]
        L.fc_diagnormal_sample.argtypes = [vp, i64, vp, i64, vp, i64, i64, i32, i64, vp]
        L.fc_diagnormal_sample_backward.argtypes = [vp, i64, vp, i64, vp, i64, vp, vp, i64, i32, i64, vp]
        L.fc_diagnormal_workspace_floats.argtypes = [i64, i32, i64]
        L.fc_pointwise_apply.argtypes = [vp, i64, vp, i64, vp, i32, i64, i64, ctypes.POINTER(PointwiseConfig), vp, vp]
        L.fc_pointwise_workspace_floats.argtypes = [i64, i64]
        L.fc_pointwise_backward.argtypes = [vp, i64, vp, i64, vp, vp, i64, vp, vp, i64, i64,
                                            ctypes.POINTER(PointwiseConfig), vp]
        L.fc_made_inverse_smem_bytes.argtypes = [i32, i32, i32, i32, i32]
        L.fc_made_inverse_profile.argtypes = [ctypes.POINTER(ctypes.c_uint64)]
        L.fc_made_inverse_rqs.argtypes = [ctypes.POINTER(MadeProgramStruct), vp, i64, vp, i64, vp, i32, i64,
                                          ctypes.POINTER(RqsConfig), vp, vp]
        L.fc_made_inverse_affine.argtypes = [ctypes.POINTER(MadeProgramStruct), vp, i64, vp, i64, vp, i32, i64, i32, vp]
        L.fc_made_inverse_sos.argtypes = [ctypes.POINTER(MadeProgramStruct), vp, i64, vp, i64, vp, i32, i64, i32, f32, i32,
                                          f32, vp]
        L.fc_made_inverse_linspline.argtypes = [ctypes.POINTER(MadeProgramStruct), vp, i64, vp, i64, vp, i32, i64, i32, i32,
                                                f32, f32, f32, f32, vp, vp]
        L.fc_made_inverse_quadspline.argtypes = [ctypes.POINTER(MadeProgramStruct), vp, i64, vp, i64, vp, i32, i64,
                                                 ctypes.POINTER(QuadSplineConfig), vp, vp]
        L.fc_made_inverse_cubicspline.argtypes = L.fc_made_inverse_quadspline.argtypes
        L.fc_version.restype = ctypes.c_char_p
        for name in EXPORTS:
            if name not in ("fc_version",):
                getattr(L, name).restype = ctypes.c_int
        L.fc_conditioner_layer_bytes.restype = ctypes.c_int64
        L.fc_made_inverse_smem_bytes.restype = ctypes.c_int64
        L.fc_actnorm_workspace_floats.restype = ctypes.c_int64
        L.fc_lulinear_workspace_floats.restype = ctypes.c_int64
        L.fc_batchnorm_workspace_floats.restype = ctypes.c_int64
        L.fc_diagnormal_workspace_floats.restype = ctypes.c_int64
        L.fc_pointwise_workspace_floats.restype = ctypes.c_int64
        _lib = L
    return _lib


def check(rc, what):
    if rc != FC_OK:
        raise RuntimeError("{} failed: {} ({})".format(what, ERRORS.get(rc, "unknown error"), rc))


def require_cuda_f32(t, name):
    if not t.is_cuda:
        raise RuntimeError(
            "{} must be a CUDA tensor: flowconductor_b200 runs only on the GPU (no CPU fallback)".format(name))
    if t.dtype != torch.float32:
        raise RuntimeError("{} must be float32 (got {})".format(name, t.dtype))
    return t


def rows(t, broadcast_ok=False):
    """(pointer, row stride in elements) of a 2-D tensor whose last dim is dense.  broadcast_ok: a row shared by the whole
    batch (an `expand`ed [1, n] tensor: row stride 0) is passed as it is — the kernels read `base + row * stride` — instead
    of being materialised B times (the unconditional CDF layers' learnable parameters: ADVICE r1)."""
    if t.dim() != 2:
        raise ValueError("expected a 2-D tensor")
    if t.shape[1] > 1 and t.stride(1) != 1:
        t = t.contiguous()
    if broadcast_ok and t.shape[0] > 1 and t.stride(0) == 0:
        return t, t.data_ptr(), 0
    if t.shape[0] > 1 and t.stride(0) < t.shape[1]:
        t = t.contiguous()
    return t, t.data_ptr(), (t.stride(0) if t.shape[0] > 1 else t.shape[1])


def cols(t):
    if t is None or t.numel() == 0:
        return Cols(None, 0)
    assert t.dtype == torch.int32 and t.is_cuda and t.is_contiguous()
    return Cols(t.data_ptr(), t.numel())


def stream_ptr(device):
    return ctypes.c_void_p(torch.cuda.current_stream(device).cuda_stream)


# ------------------------------------------------------------------------------------------------
# launch accounting: every C-ABI kernel launch goes through `launch(...)`
# ------------------------------------------------------------------------------------------------
class LaunchStats:
    """Counts kernel launches and, when `timing` is on, brackets each one with CUDA events recorded on the
    launching stream (bench.py uses this for `gpu_launches` and the per-kernel roofline)."""

    def __init__(self):
        self.counts = {}
        self.timing = False
        self.events = {}

    def reset(self):
        self.counts = {}
        self.events = {}

    def total(self):
        return sum(self.counts.values())

    def elapsed_ms(self, name):
        """(number of timed launches, their summed device time in ms); call after a synchronize."""
        pairs = self.events.get(name, [])
        return len(pairs), sum(a.elapsed_time(b) for a, b in pairs)


STATS = LaunchStats()

# NVTX ranges (SURVEY.md 5: the reference has no tracing): with FC_NVTX=1 in the environment, or `_cabi.NVTX = True`, every
# C-ABI launch is bracketed by an NVTX range named after its entry point, and CompositeTransform brackets every layer
# ("layer 3: PiecewiseRationalQuadraticCouplingTransform.forward"), so an nsys / ncu --nvtx timeline reads in the reference's
# own vocabulary.  Off by default: two host calls per launch.
NVTX = os.environ.get("FC_NVTX", "0") == "1"


class nvtx_range:
    """Context manager: an NVTX range when NVTX is on, nothing otherwise."""
    __slots__ = ("name", "on")

    def __init__(self, name):
        self.name = name
        self.on = NVTX

    def __enter__(self):
        if self.on:
            torch.cuda.nvtx.range_push(self.name)
        return self

    def __exit__(self, *exc):
        if self.on:
            torch.cuda.nvtx.range_pop()
        return False


class launch:
    __slots__ = ("name", "device", "start")

    def __init__(self, name, device):
        self.name = name
        self.device = device

    def __enter__(self):
        STATS.counts[self.name] = STATS.counts.get(self.name, 0) + 1
        if NVTX:
            torch.cuda.nvtx.range_push(self.name)
        self.start = None
        if STATS.timing:
            self.start = torch.cuda.Event(enable_timing=True)
            self.start.record(torch.cuda.current_stream(self.device))
        return self

    def __exit__(self, *exc):
        if self.start is not None:
            end = torch.cuda.Event(enable_timing=True)
            end.record(torch.cuda.current_stream(self.device))
            STATS.events.setdefault(self.name, []).append((self.start, end))
        if NVTX:
            torch.cuda.nvtx.range_pop()
        return False
