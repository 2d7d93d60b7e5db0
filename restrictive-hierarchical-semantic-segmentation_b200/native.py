"""ctypes binding of librhseg_b200.so (include/rhseg_b200.h).

There is no fallback: if the shared library is missing the first call raises with the
build command, and every kernel entry point requires CUDA tensors."""
import ctypes
import os
import threading

import torch

PKG_DIR = os.path.dirname(os.path.abspath(__file__))
# RHSEG_LIB: development only -- A/B of two builds inside one GPU call (tools/ab.sh); the product is the in-tree library
LIB_PATH = os.environ.get("RHSEG_LIB") or os.path.join(PKG_DIR, "librhseg_b200.so")

MAX_K = 16
KERNEL_MAX_K = 8
TABLE_INTS = 4 + 5 * MAX_K
NSTAT = 5
XCHG_HANDLE_BYTES = 64
DZ_PREZEROED = 1
FEATS_BF16 = 0x10  # RHSEG_FEATS_BF16: the feature (and dfeats) tensors of the call are bf16
FEATS_NHWC = 0x20  # RHSEG_FEATS_NHWC: the feature (and dfeats) tensors of the call are channels-last [B,H,W,C]
ACT_SIGMOID, ACT_GROUPED, ACT_ZEROS = 0, 1, 2

_c = ctypes
_P, _I, _L, _D, _U = _c.c_void_p, _c.c_int, _c.c_long, _c.c_double, _c.c_uint32

# name -> argtypes, exactly the prototypes of include/rhseg_b200.h
SIGNATURES = {
    "rhseg_abi_version": [],
    "rhseg_status_string": [_I],
    "rhseg_device_info": [_P, _P, _P],
    "rhseg_tree_compile_level": [_P, _I, _I, _P],
    "rhseg_film_fold": [_P, _P, _P, _P, _P, _D, _I, _I, _I, _I, _P, _P, _P, _P],
    "rhseg_head_level_fwd": [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P, _P, _P, _P, _I, _P],
    "rhseg_head_level_fwd_eval": [_P, _P, _P, _P, _P, _I, _I, _I, _I, _I, _I, _I, _I, _I, _P, _P, _P, _P,
                                  _P, _L, _L, _P, _L, _L, _P, _P, _P, _I, _P],
    "rhseg_head_act_bwd": [_P, _P, _P, _P, _P, _D, _P, _U, _I, _I, _I, _I, _I, _I, _P, _P, _P],
    "rhseg_upsample_adjoint": [_P, _I, _I, _I, _I, _I, _I, _P, _P, _I, _P],
    "rhseg_head_dz_lowres_fused": [_P, _P, _L, _L, _P, _P, _P, _P, _P, _P, _D, _P, _U, _I, _I, _I, _I, _I, _I, _I, _I, _P, _P, _P, _I, _P],
    "rhseg_pack_f64": [_P, _P, _I, _P, _P],
    "rhseg_unpack_f32": [_P, _D, _P, _P, _I, _P],
    "rhseg_xchg_create": [_L, _I, _P, _P],
    "rhseg_xchg_connect": [_P, _I, _P],
    "rhseg_xchg_all_reduce": [_P, _P, _L, _P, _P, _I, _P, _P],
    "rhseg_xchg_status": [_P, _P],
    "rhseg_xchg_set_timeout_ms": [_P, _L],
    "rhseg_xchg_destroy": [_P],
    "rhseg_head_conv_bwd": [_P, _P, _P, _I, _I, _I, _I, _P, _P, _P, _I, _P],
    "rhseg_head_conv_bwd_params": [_P, _P, _P, _I, _I, _I, _I, _P, _P, _P, _I, _P, _P, _P, _P, _D, _I, _P, _P, _P, _P, _P, _P, _P],
    "rhseg_head_param_grads": [_P, _P, _P, _P, _P, _P, _D, _I, _I, _I, _I, _P, _P, _P, _P, _P, _I, _P],
    "rhseg_loss_stats": [_P, _P, _L, _L, _I, _I, _I, _I, _P, _P],
    "rhseg_loss_finalize": [_P, _P, _I, _I, _D, _P, _P, _P],
    "rhseg_loss_bwd": [_P, _P, _L, _L, _P, _P, _P, _I, _I, _I, _I, _P, _P],
    "rhseg_consistency_sums": [_P, _P, _P, _I, _I, _I, _I, _P, _P],
    "rhseg_confusion_matrix": [_P, _L, _L, _P, _L, _L, _I, _I, _I, _I, _P, _P],
    "rhseg_metric_ratios": [_P, _I, _P, _P],
    "rhseg_predict_onehot": [_P, _P, _L, _L, _I, _I, _I, _P, _P, _P, _P],
    "rhseg_head_dz_fullres_fused": [_P, _P, _L, _L, _P, _P, _P, _P, _P, _P, _D, _P, _U, _I, _I, _I, _I, _I, _P, _P, _P],
    "rhseg_step_finalize": [_P, _P, _I, _I, _P, _P, _D, _L, _U, _P, _P, _P, _P],
    "rhseg_dp_grad_scales": [_P, _P, _I, _I, _P, _P, _P],
    "rhseg_level_eval": [_P, _P, _L, _L, _P, _L, _L, _P, _P, _I, _I, _I, _I, _P, _P, _I, _P],
    "rhseg_targets_i8_to_f32": [_P, _L, _P, _P],
    "rhseg_concat_image_logits": [_P, _I, _P, _I, _I, _I, _P, _P],
    "rhseg_stitch_levels": [_P, _I, _I, _I, _P, _I, _P, _P],
    "rhseg_confusion_from_logits": [_P, _P, _L, _L, _I, _I, _I, _I, _P, _P],
}

_lib = None
_lock = threading.Lock()
launch_count = 0  # kernels-launching C-ABI calls issued (bench.py reports it)


class NativeError(RuntimeError):
    pass


def lib():
    """The loaded library; raises NativeError when it has not been built."""
    global _lib
    if _lib is None:
        with _lock:
            if _lib is None:
                if not os.path.exists(LIB_PATH):
                    raise NativeError(
                        "librhseg_b200.so is missing (%s). Build it with "
                        "`python -c 'import __graft_entry__ as g; g.build()'` or "
                        "`python restrictive-hierarchical-semantic-segmentation_b200/build.py`. "
                        "There is no CPU / PyTorch fallback for this path." % LIB_PATH)
                handle = ctypes.CDLL(LIB_PATH)
                for name, argtypes in SIGNATURES.items():
                    fn = getattr(handle, name)  # AttributeError = symbol missing = broken build
                    fn.argtypes = argtypes
                    fn.restype = _c.c_char_p if name == "rhseg_status_string" else _I
                if handle.rhseg_abi_version() != 1:
                    raise NativeError("librhseg_b200.so ABI version mismatch; rebuild")
                _lib = handle
    return _lib


def check(rc, what):
    if rc != 0:
        msg = lib().rhseg_status_string(rc)
        raise NativeError("%s failed: %s (status %d)" % (what, msg.decode() if msg else "?", rc))


def status_string(rc) -> str:
    msg = lib().rhseg_status_string(int(rc))
    return msg.decode() if msg else "?"


def ptr(t):
    """Device pointer of a tensor (None -> NULL)."""
    return None if t is None else t.data_ptr()


_raw_stream = getattr(torch._C, "_cuda_getCurrentRawStream", None)


def stream_of(t):
    """Raw cudaStream_t of the current stream on the tensor's device (the raw accessor avoids building a Stream object:
    ~9 us -> < 1 us per call on the eager drop-in route, which is bound by host time)."""
    if _raw_stream is not None and t.device.index is not None:
        return _raw_stream(t.device.index)
    return torch.cuda.current_stream(t.device).cuda_stream


_current_device = getattr(torch._C, "_cuda_getDevice", None) or torch.cuda.current_device  # the raw accessor: no lazy-init checks


class _NoGuard:
    def __enter__(self):
        return None

    def __exit__(self, *a):
        return False


_NO_GUARD = _NoGuard()


def device_guard(t):
    """Context manager that makes the tensor's device current while kernels are launched for it (they launch on the
    device's current stream and size their grids for the current device).  Free when it already is."""
    idx = t.device.index
    if idx is None or idx == _current_device():
        return _NO_GUARD
    return torch.cuda.device(idx)


def require_cuda(*tensors):
    for t in tensors:
        if t is not None and not t.is_cuda:
            raise NativeError("rhseg_b200 kernels need CUDA tensors (got a %s tensor); there is no CPU fallback"
                              % t.device.type)


def call(name, *args):
    """Invoke one kernel-launching entry point and check its status."""
    global launch_count
    launch_count += 1
    check(getattr(lib(), name)(*args), name)


def compile_level_table(parent_ch, k_prev):
    """Host-side: parent channel list of one level -> int32 table (list of TABLE_INTS ints)."""
    K = len(parent_ch)
    src = (_c.c_int32 * K)(*parent_ch)
    dst = (_c.c_int32 * TABLE_INTS)()
    check(lib().rhseg_tree_compile_level(src, K, int(k_prev), dst), "rhseg_tree_compile_level")
    return list(dst)
