"""ctypes binding of libmsda_b200.so (include/msda_b200.h) and of its companions: the mixed-precision
libmsda_b200_amp.so (include/msda_b200_amp.h), the training library libmsda_b200_train.so
(include/msda_b200_train.h), the bf16-autocast training library libmsda_b200_amp_train.so
(include/msda_b200_amp_train.h) and the float16-storage attention library libmsda_b200_f16.so
(include/msda_b200_f16.h).

This is the ONLY way the package reaches compute: there is no CPU fallback and no alternate
backend.  If a library is missing, its callers fail loudly.
"""
import ctypes
import os

from .build import AMP_LIB_PATH, AMP_TRAIN_LIB_PATH, F16_LIB_PATH, LIB_PATH, TRAIN_LIB_PATH

MSDA_ABI_VERSION = 4
MSDA_AMP_ABI_VERSION = 1
MSDA_TRAIN_ABI_VERSION = 1
MSDA_AMP_TRAIN_ABI_VERSION = 1
MSDA_F16_ABI_VERSION = 1

MSDA_OK = 0
MSDA_ERR_INVALID_ARGUMENT = 1
MSDA_ERR_IM2COL_STEP = 2
MSDA_ERR_UNSUPPORTED_DTYPE = 3
MSDA_ERR_WORKSPACE = 4
MSDA_ERR_TOO_LARGE = 5
MSDA_ERR_CUDA = 6

MSDA_DTYPE_F32 = 0
MSDA_DTYPE_F64 = 1
MSDA_DTYPE_BF16 = 2

MSDA_FLAG_DETERMINISTIC = 1
MSDA_FLAG_ACCUMULATE_VALUE = 2
MSDA_FLAG_PRESUMMED = 4
MSDA_FLAG_PLANAR = 8

# every symbol include/msda_b200.h declares
EXPORTS = (
    "msda_abi_version", "msda_error_string", "msda_last_cuda_error", "msda_forward",
    "msda_backward", "msda_backward_workspace_bytes", "msda_masked_zero", "msda_snippet_forward",
    "msda_snippet_backward", "msda_snippet_backward_workspace_bytes", "msda_snippet_num_slots", "msda_snippet_prefers_presum", "msda_frame_sum",
    "msda_frame_unsum", "msda_layer_tail", "msda_planar_slot_bytes", "msda_frame_sum_planar", "msda_frame_unsum_planar",
)
# every symbol include/msda_b200_amp.h declares
AMP_EXPORTS = ("msda_amp_abi_version", "msda_amp_last_cuda_error", "msda_amp_layer_tail")
# every symbol include/msda_b200_train.h declares
TRAIN_EXPORTS = ("msda_train_abi_version", "msda_train_last_cuda_error", "msda_train_layer_tail_forward",
                 "msda_train_layer_tail_workspace_bytes", "msda_train_layer_tail_backward")
# every symbol include/msda_b200_amp_train.h declares
AMP_TRAIN_EXPORTS = ("msda_amp_train_abi_version", "msda_amp_train_last_cuda_error",
                     "msda_amp_train_layer_tail_forward", "msda_amp_train_layer_tail_workspace_bytes",
                     "msda_amp_train_layer_tail_backward")
# every symbol include/msda_b200_f16.h declares
F16_EXPORTS = ("msda_f16_abi_version", "msda_f16_last_cuda_error", "msda_f16_forward", "msda_f16_backward",
               "msda_f16_snippet_forward", "msda_f16_snippet_backward", "msda_f16_frame_sum", "msda_f16_frame_unsum")

_lib = None
_amp_lib = None
_train_lib = None
_amp_train_lib = None
_f16_lib = None


class MsdaError(RuntimeError):
    def __init__(self, status, message):
        super().__init__(message)
        self.status = status


def lib():
    """Load (once) and return the ctypes handle; raise if the library was not built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "libmsda_b200.so is not built (%s). Build it with "
            "`python -c 'import __graft_entry__ as g; g.build()'` or `python -m snipper_b200.build`. "
            "There is no CPU / PyTorch fallback for this op." % LIB_PATH)
    L = ctypes.CDLL(LIB_PATH)
    vp, i32, i64, u32, sz = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_uint, ctypes.c_size_t
    L.msda_abi_version.restype = i32
    L.msda_abi_version.argtypes = []
    L.msda_error_string.restype = ctypes.c_char_p
    L.msda_error_string.argtypes = [i32]
    L.msda_last_cuda_error.restype = i32
    L.msda_last_cuda_error.argtypes = []
    L.msda_forward.restype = i32
    L.msda_forward.argtypes = [vp] * 6 + [i32] * 7 + [i64, i32, i32, vp]
    L.msda_backward.restype = i32
    L.msda_backward.argtypes = [vp] * 9 + [i32] * 7 + [i64, i32, i32, u32, vp, sz, vp]
    L.msda_backward_workspace_bytes.restype = sz
    L.msda_backward_workspace_bytes.argtypes = [i32] * 8 + [u32]
    L.msda_masked_zero.restype = i32
    L.msda_masked_zero.argtypes = [vp, vp, i64, i32, vp]
    L.msda_snippet_forward.restype = i32
    L.msda_snippet_forward.argtypes = [vp] * 7 + [i32] * 10 + [i64] * 6 + [vp, vp, vp, vp, i64, i32, i32, u32, vp]
    L.msda_snippet_backward.restype = i32
    L.msda_snippet_backward.argtypes = [vp] * 10 + [i32] * 10 + [i64] * 6 + [vp, vp, vp, vp, i64, i32, i32, u32, vp, sz, vp]
    L.msda_snippet_backward_workspace_bytes.restype = sz
    L.msda_snippet_backward_workspace_bytes.argtypes = [i32] * 10 + [u32]
    L.msda_snippet_num_slots.restype = i32
    L.msda_snippet_num_slots.argtypes = [i32, i32]
    L.msda_snippet_prefers_presum.restype = i32
    L.msda_snippet_prefers_presum.argtypes = [i32] * 7
    L.msda_frame_sum.restype = i32
    L.msda_frame_sum.argtypes = [vp, vp, vp] + [i32] * 6 + [i64, i64, i64, i32, i32, vp]
    L.msda_frame_unsum.restype = i32
    L.msda_frame_unsum.argtypes = [vp, vp, vp] + [i32] * 6 + [i64, i32, i32, vp]
    L.msda_planar_slot_bytes.restype = sz
    L.msda_planar_slot_bytes.argtypes = [i32] * 4
    L.msda_frame_sum_planar.restype = i32
    L.msda_frame_sum_planar.argtypes = [vp, vp, vp] + [i32] * 7 + [i64, i64, i64, i32, i32, vp]
    L.msda_frame_unsum_planar.restype = i32
    L.msda_frame_unsum_planar.argtypes = [vp, vp, vp] + [i32] * 7 + [i64, i32, i32, vp]
    L.msda_layer_tail.restype = i32
    L.msda_layer_tail.argtypes = [vp] * 8 + [i64, i32, ctypes.c_float, i32, vp]
    if L.msda_abi_version() != MSDA_ABI_VERSION:
        raise RuntimeError("libmsda_b200.so ABI %d != binding ABI %d; rebuild" %
                           (L.msda_abi_version(), MSDA_ABI_VERSION))
    _lib = L
    return L


def amp_lib():
    """Load (once) and return the ctypes handle of libmsda_b200_amp.so; raise if it was not built."""
    global _amp_lib
    if _amp_lib is not None:
        return _amp_lib
    if not os.path.exists(AMP_LIB_PATH):
        raise RuntimeError(
            "libmsda_b200_amp.so is not built (%s). Build it with "
            "`python -c 'import __graft_entry__ as g; g.build()'` or `python -m snipper_b200.build`. "
            "There is no CPU / PyTorch fallback for this op." % AMP_LIB_PATH)
    L = ctypes.CDLL(AMP_LIB_PATH)
    vp, i32, i64 = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64
    L.msda_amp_abi_version.restype = i32
    L.msda_amp_abi_version.argtypes = []
    L.msda_amp_last_cuda_error.restype = i32
    L.msda_amp_last_cuda_error.argtypes = []
    L.msda_amp_layer_tail.restype = i32
    L.msda_amp_layer_tail.argtypes = [vp, vp, vp, i32] + [vp] * 6 + [i64, i32, ctypes.c_float, vp]
    if L.msda_amp_abi_version() != MSDA_AMP_ABI_VERSION:
        raise RuntimeError("libmsda_b200_amp.so ABI %d != binding ABI %d; rebuild" %
                           (L.msda_amp_abi_version(), MSDA_AMP_ABI_VERSION))
    _amp_lib = L
    return L


def train_lib():
    """Load (once) and return the ctypes handle of libmsda_b200_train.so; raise if it was not built."""
    global _train_lib
    if _train_lib is not None:
        return _train_lib
    if not os.path.exists(TRAIN_LIB_PATH):
        raise RuntimeError(
            "libmsda_b200_train.so is not built (%s). Build it with "
            "`python -c 'import __graft_entry__ as g; g.build()'` or `python -m snipper_b200.build`. "
            "There is no CPU / PyTorch fallback for this op." % TRAIN_LIB_PATH)
    L = ctypes.CDLL(TRAIN_LIB_PATH)
    vp, i32, i64, f32 = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_float
    L.msda_train_abi_version.restype = i32
    L.msda_train_abi_version.argtypes = []
    L.msda_train_last_cuda_error.restype = i32
    L.msda_train_last_cuda_error.argtypes = []
    L.msda_train_layer_tail_forward.restype = i32
    L.msda_train_layer_tail_forward.argtypes = [vp] * 4 + [f32] + [vp] * 7 + [i64, i32, f32, vp]
    L.msda_train_layer_tail_workspace_bytes.restype = ctypes.c_size_t
    L.msda_train_layer_tail_workspace_bytes.argtypes = [i64, i32]
    L.msda_train_layer_tail_backward.restype = i32
    L.msda_train_layer_tail_backward.argtypes = [vp] * 5 + [f32] + [vp] * 5 + [i64, i32, vp]
    if L.msda_train_abi_version() != MSDA_TRAIN_ABI_VERSION:
        raise RuntimeError("libmsda_b200_train.so ABI %d != binding ABI %d; rebuild" %
                           (L.msda_train_abi_version(), MSDA_TRAIN_ABI_VERSION))
    _train_lib = L
    return L


def amp_train_lib():
    """Load (once) and return the ctypes handle of libmsda_b200_amp_train.so; raise if it was not built."""
    global _amp_train_lib
    if _amp_train_lib is not None:
        return _amp_train_lib
    if not os.path.exists(AMP_TRAIN_LIB_PATH):
        raise RuntimeError(
            "libmsda_b200_amp_train.so is not built (%s). Build it with "
            "`python -c 'import __graft_entry__ as g; g.build()'` or `python -m snipper_b200.build`. "
            "There is no CPU / PyTorch fallback for this op." % AMP_TRAIN_LIB_PATH)
    L = ctypes.CDLL(AMP_TRAIN_LIB_PATH)
    vp, i32, i64, f32 = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_float
    L.msda_amp_train_abi_version.restype = i32
    L.msda_amp_train_abi_version.argtypes = []
    L.msda_amp_train_last_cuda_error.restype = i32
    L.msda_amp_train_last_cuda_error.argtypes = []
    L.msda_amp_train_layer_tail_forward.restype = i32
    L.msda_amp_train_layer_tail_forward.argtypes = [vp] * 3 + [i32, vp, f32] + [vp] * 8 + [i64, i32, f32, vp]
    L.msda_amp_train_layer_tail_workspace_bytes.restype = ctypes.c_size_t
    L.msda_amp_train_layer_tail_workspace_bytes.argtypes = [i64, i32]
    L.msda_amp_train_layer_tail_backward.restype = i32
    L.msda_amp_train_layer_tail_backward.argtypes = [vp] * 6 + [f32] + [vp] * 2 + [i32] + [vp] * 3 + [i64, i32, vp]
    if L.msda_amp_train_abi_version() != MSDA_AMP_TRAIN_ABI_VERSION:
        raise RuntimeError("libmsda_b200_amp_train.so ABI %d != binding ABI %d; rebuild" %
                           (L.msda_amp_train_abi_version(), MSDA_AMP_TRAIN_ABI_VERSION))
    _amp_train_lib = L
    return L


def f16_lib():
    """Load (once) and return the ctypes handle of libmsda_b200_f16.so; raise if it was not built."""
    global _f16_lib
    if _f16_lib is not None:
        return _f16_lib
    if not os.path.exists(F16_LIB_PATH):
        raise RuntimeError(
            "libmsda_b200_f16.so is not built (%s). Build it with "
            "`python -c 'import __graft_entry__ as g; g.build()'` or `python -m snipper_b200.build`. "
            "There is no CPU / PyTorch fallback for this op." % F16_LIB_PATH)
    L = ctypes.CDLL(F16_LIB_PATH)
    vp, i32, i64, u32 = ctypes.c_void_p, ctypes.c_int, ctypes.c_int64, ctypes.c_uint
    L.msda_f16_abi_version.restype = i32
    L.msda_f16_abi_version.argtypes = []
    L.msda_f16_last_cuda_error.restype = i32
    L.msda_f16_last_cuda_error.argtypes = []
    # the argument lists of the msda_* twins without dtype (and without the deterministic workspace)
    L.msda_f16_forward.restype = i32
    L.msda_f16_forward.argtypes = [vp] * 6 + [i32] * 7 + [i64, i32, vp]
    L.msda_f16_backward.restype = i32
    L.msda_f16_backward.argtypes = [vp] * 9 + [i32] * 7 + [i64, i32, u32, vp]
    L.msda_f16_snippet_forward.restype = i32
    L.msda_f16_snippet_forward.argtypes = [vp] * 7 + [i32] * 10 + [i64] * 6 + [vp, vp, vp, vp, i64, i32, u32, vp]
    L.msda_f16_snippet_backward.restype = i32
    L.msda_f16_snippet_backward.argtypes = [vp] * 10 + [i32] * 10 + [i64] * 6 + [vp, vp, vp, vp, i64, i32, u32, vp]
    L.msda_f16_frame_sum.restype = i32
    L.msda_f16_frame_sum.argtypes = [vp, vp, vp] + [i32] * 6 + [i64, i64, i64, i32, vp]
    L.msda_f16_frame_unsum.restype = i32
    L.msda_f16_frame_unsum.argtypes = [vp, vp, vp] + [i32] * 6 + [i64, i32, vp]
    if L.msda_f16_abi_version() != MSDA_F16_ABI_VERSION:
        raise RuntimeError("libmsda_b200_f16.so ABI %d != binding ABI %d; rebuild" %
                           (L.msda_f16_abi_version(), MSDA_F16_ABI_VERSION))
    _f16_lib = L
    return L


def check(status, what, batch=None, im2col_step=None, last_cuda_error=None):
    """Turn a status code into the exception the reference would have raised.  ``last_cuda_error``: the
    ``*_last_cuda_error`` function of the library that returned ``status`` (default: libmsda_b200.so's)."""
    if status == MSDA_OK:
        return
    L = lib()
    msg = L.msda_error_string(status).decode()
    if status == MSDA_ERR_IM2COL_STEP and batch is not None:
        # reference message: ms_deform_attn_cuda.cu:52
        msg = "batch(%d) must divide im2col_step(%d)" % (batch, min(batch, im2col_step) if im2col_step > 0 else im2col_step)
    if status == MSDA_ERR_CUDA:
        msg += " [cudaError %d]" % (last_cuda_error or L.msda_last_cuda_error)()
    raise MsdaError(status, "%s: %s" % (what, msg))
