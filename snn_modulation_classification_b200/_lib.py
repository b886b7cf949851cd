"""ctypes binding of libdcll_b200.so (include/dcll_b200.h).

There is no CPU fallback: if the library is missing this module raises at import
time with the build command, and every entry point raises on a non-zero status.
"""
import ctypes as C
import os

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "libdcll_b200.so")
ABI_VERSION = 12

OK, EINVAL, ECUDA, EUNSUPPORTED = 0, -1, -2, -3
COEF_SCALAR, COEF_CHANNEL, COEF_ELEMENT = 0, 1, 2
X_DENSE, X_CELLS = 0, 1
LOSS_SMOOTHL1, LOSS_MSE, LOSS_L1, LOSS_EXTERNAL = 0, 1, 2, 3
LOSS_CROSS_ENTROPY, LOSS_BCE_LOGITS, LOSS_SOFT_MARGIN, LOSS_KL_DIV, LOSS_POISSON_NLL, LOSS_HINGE = 4, 5, 6, 7, 8, 9
PREC_FP32, PREC_BF16X3, PREC_F16X2 = 0, 1, 2
OPT_ADAM, OPT_ADAMW, OPT_ADAMAX, OPT_NADAM, OPT_RADAM = 0, 1, 2, 3, 4

_fp = C.c_void_p  # device pointers travel as integers


class Adam(C.Structure):
    _fields_ = [("lr", C.c_double), ("beta1", C.c_double), ("beta2", C.c_double), ("eps", C.c_double),
                ("weight_decay", C.c_double), ("step", C.c_int64),
                ("m_w", _fp), ("v_w", _fp), ("m_b", _fp), ("v_b", _fp)]


class Optim(C.Structure):
    _fields_ = [("kind", C.c_int32), ("decoupled_wd", C.c_int32), ("momentum_decay", C.c_double), ("mu_product", C.c_float)]


class ConvLayer(C.Structure):
    _fields_ = [("B", C.c_int32), ("Cin", C.c_int32), ("H", C.c_int32), ("W", C.c_int32),
                ("Cout", C.c_int32), ("KH", C.c_int32), ("KW", C.c_int32), ("padH", C.c_int32), ("padW", C.c_int32),
                ("poolH", C.c_int32), ("poolW", C.c_int32), ("K", C.c_int32), ("output_layer", C.c_int32),
                ("coef_mode", C.c_int32), ("x_mode", C.c_int32), ("precision", C.c_int32), ("cur", C.c_int32),
                ("write_pvmem", C.c_int32), ("quantized", C.c_int32), ("alpharp", C.c_float), ("wrp", C.c_float),
                ("alpha", _fp), ("alphas", _fp), ("tau_m", _fp), ("tau_s", _fp),
                ("weight", _fp), ("weight_t", _fp), ("weight_mma", _fp), ("bias", _fp), ("wo", _fp), ("bo", _fp),
                ("wout", _fp), ("bout", _fp),
                ("eps0", _fp * 2), ("eps1", _fp * 2), ("eps1_mma", _fp), ("arp", _fp),
                ("spikes", _fp), ("pv", _fp), ("pvmem", _fp), ("pool_idx", _fp), ("pvoutput", _fp),
                ("output", _fp), ("g_u", _fp), ("workspace", _fp), ("workspace_bytes", C.c_size_t),
                ("a_exp", C.c_int32), ("g_exp", C.c_int32), ("w_exp", _fp)]


class TrainArgs(C.Structure):
    _fields_ = [("target", _fp), ("g_o_ext", _fp), ("g_o2_ext", _fp), ("loss_kind", C.c_int32),
                ("apply_update", C.c_int32), ("adam_i2h", Adam), ("adam_out", Adam),
                ("grad_w", _fp), ("grad_b", _fp), ("grad_wout", _fp), ("grad_bout", _fp), ("loss_out", _fp)]


class DenseLayer(C.Structure):
    _fields_ = [("B", C.c_int32), ("In", C.c_int32), ("Out", C.c_int32), ("K", C.c_int32), ("coef_mode", C.c_int32),
                ("alpharp", C.c_float), ("wrp", C.c_float),
                ("alpha", _fp), ("alphas", _fp), ("tau_m", _fp), ("tau_s", _fp), ("weight", _fp), ("bias", _fp),
                ("wo", _fp), ("bo", _fp), ("eps0", _fp), ("eps1", _fp), ("arp", _fp), ("spikes", _fp), ("pv", _fp),
                ("vmem", _fp), ("pvoutput", _fp), ("g_o", _fp), ("g_u", _fp), ("grad_w", _fp), ("grad_b", _fp)]


class DcllError(RuntimeError):
    pass


def _load():
    if not os.path.exists(LIB_PATH):
        raise ImportError(
            "libdcll_b200.so is not built (%s). Build it with `python -m snn_modulation_classification_b200.build` "
            "(needs nvcc; sm_100a only). There is no CPU fallback." % LIB_PATH)
    lib = C.CDLL(LIB_PATH)
    lib.dcll_abi_version.restype = C.c_int
    lib.dcll_last_error.restype = C.c_char_p
    lib.dcll_sizeof_conv_layer.restype = C.c_size_t
    lib.dcll_sizeof_train_args.restype = C.c_size_t
    if lib.dcll_abi_version() != ABI_VERSION:
        raise ImportError("libdcll_b200.so has ABI %d, binding expects %d: rebuild" % (lib.dcll_abi_version(), ABI_VERSION))
    lib.dcll_sizeof_dense_layer.restype = C.c_size_t
    if lib.dcll_sizeof_conv_layer() != C.sizeof(ConvLayer) or lib.dcll_sizeof_train_args() != C.sizeof(TrainArgs) \
            or lib.dcll_sizeof_dense_layer() != C.sizeof(DenseLayer):
        raise ImportError("struct layout mismatch between include/dcll_b200.h and _lib.py")
    P = C.POINTER
    sig = {
        "dcll_iq_encode": [_fp, C.c_int, C.c_int, C.c_double, C.c_double, C.c_double, C.c_double, C.c_int, C.c_int,
                           C.c_int, C.c_int, C.c_int, _fp, _fp],
        "dcll_cells_to_frames": [_fp, C.c_int, C.c_int, C.c_int, C.c_int, _fp, _fp],
        "dcll_image_encode": [_fp, _fp, _fp, C.c_int, C.c_int, C.c_int, C.c_double, C.c_uint64, _fp, _fp],
        "dcll_conv_sync_weights": [P(ConvLayer), _fp],
        "dcll_conv_step_fwd": [P(ConvLayer), _fp, _fp, _fp],
        "dcll_conv_step_fwd_chain": [P(ConvLayer), P(ConvLayer), C.c_int, _fp, _fp, _fp],
        "dcll_conv_chain_fusable": [P(ConvLayer), P(ConvLayer)],
        "dcll_conv_core_fwd": [P(ConvLayer), _fp, _fp],
        "dcll_conv_step_bwd_update": [P(ConvLayer), P(TrainArgs), _fp],
        "dcll_conv_apply_update": [P(ConvLayer), P(TrainArgs), _fp],
        "dcll_net_window": [P(ConvLayer), P(TrainArgs), C.c_int, _fp, _fp, C.c_int64, C.c_int, C.c_int, C.c_int,
                            P(C.c_int32), _fp, _fp],
        "dcll_dense_step_fwd": [P(DenseLayer), _fp, _fp, _fp],
        "dcll_dense_step_bwd_update": [P(DenseLayer), P(TrainArgs), _fp],
        "dcll_net_window_stats": [P(ConvLayer), P(TrainArgs), C.c_int, _fp, _fp, C.c_int64, C.c_int, C.c_int, C.c_int,
                                  P(C.c_int32), _fp, _fp, C.c_int, C.c_int, _fp],
        "dcll_infer_stack16": [P(ConvLayer), C.c_int, _fp, C.c_int, P(_fp), _fp],
        "dcll_conv_readout_rows": [P(ConvLayer), _fp, _fp],
        "dcll_vote": [_fp, C.c_int, C.c_int, C.c_int, C.c_int, _fp, _fp],
        "dcll_dp_unique_id": [C.c_char_p, _fp],
        "dcll_dp_create": [C.c_char_p, _fp, C.c_int, C.c_int, C.c_int, P(_fp)],
        "dcll_dp_destroy": [_fp],
        "dcll_net_window_dp": [_fp, P(ConvLayer), P(TrainArgs), C.c_int, _fp, _fp, C.c_int64, C.c_int, C.c_int, P(C.c_int32), _fp,
                               P(_fp), P(C.c_size_t), _fp],
        "dcll_conv_step_bwd_update_opt": [P(ConvLayer), P(TrainArgs), P(Optim), _fp],
        "dcll_conv_apply_update_opt": [P(ConvLayer), P(TrainArgs), P(Optim), _fp],
        "dcll_dense_step_bwd_update_opt": [P(DenseLayer), P(TrainArgs), P(Optim), _fp],
        "dcll_net_window_stats_opt": [P(ConvLayer), P(TrainArgs), P(Optim), C.c_int, _fp, _fp, C.c_int64, C.c_int, C.c_int,
                                      C.c_int, P(C.c_int32), _fp, _fp, C.c_int, C.c_int, _fp],
        "dcll_net_window_dp_opt": [_fp, P(ConvLayer), P(TrainArgs), P(Optim), C.c_int, _fp, _fp, C.c_int64, C.c_int, C.c_int,
                                   P(C.c_int32), _fp, P(_fp), P(C.c_size_t), _fp],
        "dcll_quantize": [_fp, C.c_int, C.c_int, _fp, _fp, _fp],
        "dcll_dequantize": [_fp, _fp, C.c_int, C.c_int, _fp, _fp],
    }
    for name, argtypes in sig.items():
        fn = getattr(lib, name)
        fn.argtypes = argtypes
        fn.restype = C.c_int
    lib.dcll_launch_count.argtypes = [C.c_int]
    lib.dcll_launch_count.restype = C.c_int64
    lib.dcll_profile_enable.argtypes = [C.c_int]
    lib.dcll_profile_enable.restype = C.c_int
    lib.dcll_profile_read.argtypes = [P(C.c_double), P(C.c_int64)]
    lib.dcll_profile_read.restype = C.c_int
    lib.dcll_debug_timeline.argtypes = [P(C.c_uint64), C.c_int]
    lib.dcll_debug_timeline.restype = C.c_int
    lib.dcll_conv_workspace_bytes.argtypes = [P(ConvLayer)]
    lib.dcll_conv_workspace_bytes.restype = C.c_size_t
    return lib


lib = _load()
KERNEL_CLASSES = ["encode", "conv_fwd", "readout_fwd", "readout_bwd", "wgrad", "adam", "misc", "trace"]


def profile_read():
    """{(kernel_class, layer): (total_ms, samples)} of the brackets sampled since the last read."""
    ms = (C.c_double * (len(KERNEL_CLASSES) * 8))()
    n = (C.c_int64 * (len(KERNEL_CLASSES) * 8))()
    check(lib.dcll_profile_read(ms, n))
    out = {}
    for c, name in enumerate(KERNEL_CLASSES):
        for l in range(8):
            if n[c * 8 + l]:
                out[(name, l)] = (ms[c * 8 + l], n[c * 8 + l])
    return out


EXPORTS = ["dcll_launch_count", "dcll_profile_enable", "dcll_profile_read", "dcll_abi_version", "dcll_last_error", "dcll_sizeof_conv_layer", "dcll_sizeof_train_args", "dcll_iq_encode",
           "dcll_cells_to_frames", "dcll_conv_workspace_bytes", "dcll_conv_sync_weights", "dcll_conv_step_fwd",
           "dcll_conv_core_fwd", "dcll_conv_step_bwd_update", "dcll_conv_apply_update", "dcll_net_window", "dcll_vote",
           "dcll_quantize", "dcll_dequantize", "dcll_sizeof_dense_layer", "dcll_dense_step_fwd",
           "dcll_dense_step_bwd_update", "dcll_net_window_stats", "dcll_infer_stack16", "dcll_conv_readout_rows", "dcll_conv_step_fwd_chain",
           "dcll_conv_chain_fusable", "dcll_dp_unique_id", "dcll_dp_create", "dcll_dp_destroy", "dcll_net_window_dp", "dcll_image_encode", "dcll_debug_timeline",
           "dcll_conv_step_bwd_update_opt", "dcll_conv_apply_update_opt", "dcll_dense_step_bwd_update_opt",
           "dcll_net_window_stats_opt", "dcll_net_window_dp_opt"]


def check(rc):
    """Raise on a non-zero status: ValueError for bad arguments (the reference raises ValueError /
    Exception from its constructors), NotImplementedError for shapes without an sm_100a instantiation,
    RuntimeError for CUDA failures."""
    if rc == OK:
        return
    msg = lib.dcll_last_error().decode("utf-8", "replace")
    if rc == EINVAL:
        raise ValueError(msg)
    if rc == EUNSUPPORTED:
        raise NotImplementedError(msg)
    raise DcllError(msg)


def ptr(t):
    """Device pointer of a torch tensor (None -> NULL). The tensor must be contiguous."""
    if t is None:
        return None
    if not t.is_contiguous():
        raise ValueError("tensor passed to libdcll_b200 must be contiguous")
    return t.data_ptr()


def current_stream():
    import torch

    return torch.cuda.current_stream().cuda_stream


def nccl_library_path():
    """The libnccl.so.2 this process has loaded (torch's bundled copy once torch.distributed's NCCL backend is up), else the
    one shipped in the nvidia.nccl wheel, else None (default search path).  dcll_dp_* dlopen it by this path."""
    try:
        for line in open("/proc/self/maps"):
            if "libnccl.so" in line:
                return line.split()[-1]
    except OSError:
        pass
    try:
        import importlib.util
        spec = importlib.util.find_spec("nvidia.nccl")
        for loc in (spec.submodule_search_locations or []) if spec else []:
            p = os.path.join(loc, "lib", "libnccl.so.2")
            if os.path.isfile(p):
                return p
    except Exception:
        pass
    return None
