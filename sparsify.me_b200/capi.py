"""ctypes binding of libsparsifyme_b200.so -- one Python callable per C-ABI entry point
declared in include/spfy_b200.h (same names, same argument order).

Every wrapper raises SpfyError (carrying spfy_last_error_string()) on a non-zero status.
The library is loaded from sparsify.me_b200/lib/ (built in-tree by build.py); a missing
library is an ImportError -- there is no Python or CPU fallback for any entry point.
"""
import ctypes
import os
from ctypes import (c_char_p, c_float, c_int, c_int32, c_int64, c_size_t, c_uint64, c_void_p,
                    POINTER)

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("SPFY_LIB") or os.path.join(HERE, "lib", "libsparsifyme_b200.so")  # SPFY_LIB: A/B builds

# enums of include/spfy_b200.h
F16, BF16, F32, F64 = 0, 1, 2, 3
PRUNE_STRIP_MAG, PRUNE_TILE_MAG, PRUNE_TILE_TRANSPOSABLE = 0, 1, 2
LAYOUT_CANONICAL, LAYOUT_SM100 = 0, 1
OP_N, OP_T = 0, 1
OUT_T = 0x10  # flag OR-ed into opB: D is written transposed, [n][m]
SPMM_ALG_DEFAULT, SPMM_ALG_CUDA_CORE, SPMM_ALG_TENSOR, SPMM_ALG_TENSOR_FAST = 0, 1, 2, 3
GEMM_PRECISE, GEMM_FAST = 0, 1
ACT_NONE, ACT_RELU, ACT_GELU_TANH = 0, 1, 2
OPTIM_SGD, OPTIM_ADAMW = 0, 1
OK, E_INVALID, E_UNSUPPORTED, E_CUDA, E_WORKSPACE, E_NCCL = 0, -1, -2, -3, -4, -5


class SpfyError(RuntimeError):
    def __init__(self, code, where, msg):
        super().__init__(f"{where} failed with status {code}: {msg}")
        self.code = code


if not os.path.exists(LIB_PATH):
    raise ImportError(
        f"{LIB_PATH} is missing: build it with `python sparsify.me_b200/build.py` "
        "(sparsify.me_b200 has no fallback path)")
_lib = ctypes.CDLL(LIB_PATH)

_P = c_void_p
_SZ = c_size_t
# name -> (restype, argtypes); status-returning functions have restype c_int
SIGNATURES = {
    "spfy_version": (c_int, []),
    "spfy_init": (c_int, []),
    "spfy_last_error_string": (c_char_p, []),
    "spfy_launch_count": (c_uint64, []),
    "spfy_convert": (c_int, [c_int, c_int, _P, _P, _SZ, _P]),
    "spfy_prune_blocks_ref": (c_int, [c_int, _P, _P, _SZ, _SZ, _SZ, _SZ, c_float, _P]),
    "spfy_compressed_bytes": (c_int, [c_int, _SZ, _SZ, c_int, POINTER(_SZ), POINTER(_SZ)]),
    "spfy_prune24": (c_int, [c_int, c_int, c_int, _P, _SZ, _P, _SZ, _P, _P, _P, _SZ, _SZ, _P]),
    "spfy_prune24_check": (c_int, [c_int, _P, _SZ, _SZ, _SZ, _P, _P]),
    "spfy_prune24_batched": (c_int, [c_int, c_int, c_int, _P, _SZ, _P]),
    "spfy_transpose24": (c_int, [c_int, _P, _P, _SZ, _SZ, _SZ, _P, _P, _P, _P]),
    "spfy_recompress24": (c_int, [c_int, _P, _SZ, c_int, _SZ, _SZ, _P, _P, _P, _SZ, _P]),
    "spfy_optim24_step": (c_int, [c_int, _P, _SZ, _P, _SZ, _P, _P, _P]),
    "spfy_transpose24_conv_bytes": (c_int, [c_int, _SZ, _SZ, _SZ, _SZ, _SZ, _SZ, POINTER(_SZ), POINTER(_SZ)]),
    "spfy_transpose24_conv": (c_int, [c_int, _P, _P, _SZ, _SZ, _SZ, _SZ, _SZ, _SZ, _P, _P, _P, _P]),
    "spfy_spmma_workspace_bytes": (c_int, [c_int, _SZ, _SZ, _SZ, POINTER(_SZ)]),
    "spfy_spmma": (c_int, [c_int, c_int, _SZ, _SZ, _SZ, c_float, _P, _P, _P, _SZ, c_float, _P, _SZ,
                           _P, _SZ, _P, _SZ, _P]),
    "spfy_spmma_conv": (c_int, [c_int, _P, _SZ, c_float, _P, _P, _P, c_float, _P, _SZ, _P, _SZ, _P]),
    "spfy_spmma_conv_nhwc": (c_int, [c_int, _P, _SZ, c_float, _P, _P, _P, _P, _SZ, _P]),
    "spfy_spmma_ex": (c_int, [c_int, c_int, _SZ, _SZ, _SZ, c_float, _P, _P, _P, _SZ, c_float, _P, _SZ,
                              _P, _SZ, _P, _SZ, _P, _P]),
    "spfy_spmma_conv_ex": (c_int, [c_int, _P, _SZ, c_float, _P, _P, _P, c_float, _P, _SZ, _P, _SZ, c_int, _P, _P]),
    "spfy_spmma_conv_dgrad": (c_int, [c_int, _P, _SZ, c_float, _P, _P, _P, c_float, _P, _P]),
    "spfy_conv_wgrad24_workspace_bytes": (c_int, [c_int, _P, _SZ, POINTER(_SZ)]),
    "spfy_conv_wgrad24": (c_int, [c_int, _P, _SZ, c_float, _P, _P, _P, c_float, _P, _P, _SZ, _P]),
    "spfy_permute_conv_weights": (c_int, [_P, _P, _SZ, _SZ, _SZ, _SZ, _P]),
    "spfy_spmma_plan_create": (c_int, [c_int, _P, _SZ, POINTER(c_void_p)]),
    "spfy_spmma_plan_create_replicated": (c_int, [c_int, _P, _SZ, _SZ, _P, POINTER(c_void_p)]),
    "spfy_spmma_plan_create_conv": (c_int, [c_int, _P, _P, _SZ, POINTER(c_void_p)]),
    "spfy_spmma_plan_create_ex": (c_int, [c_int, _P, _P, _P, _SZ, POINTER(c_void_p)]),
    "spfy_spmma_plan_run": (c_int, [_P, _P]),
    "spfy_spmma_plan_launches": (c_int, [_P]),
    "spfy_spmma_plan_run_launch": (c_int, [_P, c_int, _P]),
    "spfy_spmma_plan_launch_info": (c_int, [_P, c_int, POINTER(c_int), POINTER(c_int), POINTER(c_int), POINTER(c_int)]),
    "spfy_spmma_plan_destroy": (c_int, [_P]),
    "spfy_packed_bytes": (c_int, [c_int, _SZ, _SZ, c_int, POINTER(_SZ)]),
    "spfy_packed_write": (c_int, [c_int, c_int, _SZ, _SZ, _P, _P, _P, _SZ]),
    "spfy_packed_read": (c_int, [_P, _SZ, POINTER(c_int), POINTER(c_int), POINTER(_SZ), POINTER(_SZ), POINTER(_SZ),
                                 POINTER(_SZ), POINTER(_SZ), POINTER(_SZ)]),
    "spfy_threshold_workspace_bytes": (c_int, [_SZ, _SZ, POINTER(_SZ)]),
    "spfy_threshold_to_coo": (c_int, [c_int, _P, _SZ, _SZ, _SZ, c_float, _P, _P, _P, _SZ, _P, _P,
                                      _P, _SZ, _P]),
    "spfy_coo_to_csr": (c_int, [_P, _SZ, _SZ, _P, _P]),
    "spfy_spmm_workspace_bytes": (c_int, [c_int, _SZ, _SZ, _SZ, _SZ, _SZ, POINTER(_SZ)]),
    "spfy_spmm_coo_strided_batched": (c_int, [c_int, _SZ, _SZ, _SZ, _SZ, _SZ, _P, _P, _P, _P, _SZ, _SZ, _P,
                                              _SZ, _SZ, c_float, c_float, _P, _SZ, _P]),
    "spfy_spmm_csr_strided_batched": (c_int, [c_int, _SZ, _SZ, _SZ, _SZ, _P, _P, _P, _P, _SZ, _SZ, _P, _SZ,
                                              _SZ, c_float, c_float, _P, _SZ, _P]),
    "spfy_spmm_bell_workspace_bytes": (c_int, [c_int, c_int, _SZ, _SZ, _SZ, _SZ, POINTER(_SZ)]),
    "spfy_spmm_bell_batched": (c_int, [c_int, c_int, _SZ, _SZ, _SZ, _SZ, _SZ, _SZ, _P, _P, _P, _SZ, _P, _SZ,
                                       c_float, c_float, _P, _SZ, _P]),
    "spfy_peer_alloc": (c_int, [_SZ, POINTER(c_void_p), _P]),
    "spfy_peer_free": (c_int, [_P]),
    "spfy_peer_open": (c_int, [_P, POINTER(c_void_p)]),
    "spfy_peer_close": (c_int, [_P]),
    "spfy_mg_unique_id": (c_int, [_P]),
    "spfy_mg_create": (c_int, [c_int, c_int, _P, POINTER(c_void_p)]),
    "spfy_mg_destroy": (c_int, [_P]),
    "spfy_mg_rank": (c_int, [_P]),
    "spfy_mg_world": (c_int, [_P]),
    "spfy_mg_allgather": (c_int, [_P, _P, _P, _SZ, _P]),
    "spfy_mg_broadcast_many": (c_int, [_P, _P, _P, _P, _SZ, _P]),
    "spfy_gemm_workspace_bytes": (c_int, [c_int, c_int, c_int, _SZ, _SZ, _SZ, _SZ, _SZ, _SZ, POINTER(_SZ)]),
    "spfy_gemm_strided_batched": (c_int, [c_int, c_int, c_int, c_int, _SZ, _SZ, _SZ, c_float, _P, _SZ, _SZ, _P, _SZ,
                                          _SZ, c_float, _P, _SZ, _SZ, _SZ, _P, _SZ, _P]),
    "spfy_gemm_batched": (c_int, [c_int, c_int, c_int, c_int, _SZ, _SZ, _SZ, c_float, _P, _SZ, _P, _SZ, c_float, _P,
                                  _SZ, _SZ, _P, _SZ, _P]),
}

_NO_STATUS = {"spfy_version", "spfy_last_error_string", "spfy_launch_count", "spfy_spmma_plan_launches", "spfy_mg_rank",
              "spfy_mg_world"}


class SpmmaProblem(ctypes.Structure):
    """struct spfy_spmma_problem"""
    _fields_ = [("opB", c_int), ("m", c_size_t), ("n", c_size_t), ("k", c_size_t), ("comp_vals", c_void_p),
                ("meta", c_void_p), ("B", c_void_p), ("ldb", c_size_t), ("C", c_void_p), ("ldc", c_size_t),
                ("D", c_void_p), ("ldd", c_size_t), ("alpha", c_float), ("beta", c_float)]


class ConvDesc(ctypes.Structure):
    """struct spfy_conv_desc"""
    _fields_ = [("batch", c_size_t), ("h", c_size_t), ("w", c_size_t), ("c", c_size_t), ("kh", c_size_t), ("kw", c_size_t),
                ("stride", c_size_t), ("pad", c_size_t)]


class Epilogue(ctypes.Structure):
    """struct spfy_epilogue"""
    _fields_ = [("scale", c_void_p), ("bias", c_void_p), ("act", c_int)]


class Prune24Item(ctypes.Structure):
    """struct spfy_prune24_item"""
    _fields_ = [("in_", c_void_p), ("ld_in", c_size_t), ("out_dense", c_void_p), ("ld_out", c_size_t),
                ("comp_vals", c_void_p), ("meta", c_void_p), ("rows", c_size_t), ("cols", c_size_t)]


class Optim24Item(ctypes.Structure):
    """struct spfy_optim24_item"""
    _fields_ = [("param", c_void_p), ("grad", c_void_p), ("state1", c_void_p), ("state2", c_void_p), ("step", c_void_p),
                ("first", c_void_p), ("rows", c_size_t), ("cols", c_size_t), ("ld", c_size_t), ("group", c_size_t),
                ("dtype", c_int), ("meta", c_void_p), ("vals", c_void_p), ("vals_t", c_void_p), ("kh", c_size_t),
                ("kw", c_size_t), ("stride", c_size_t), ("pad", c_size_t)]


class Optim24Hparams(ctypes.Structure):
    """struct spfy_optim24_hparams"""
    _fields_ = [("lr", ctypes.c_double), ("momentum", ctypes.c_double), ("dampening", ctypes.c_double),
                ("weight_decay", ctypes.c_double), ("beta1", ctypes.c_double), ("beta2", ctypes.c_double),
                ("eps", ctypes.c_double), ("nesterov", c_int)]


def last_error():
    s = _lib.spfy_last_error_string()
    return s.decode("utf-8", "replace") if s else ""


def _bind(name, restype, argtypes):
    fn = getattr(_lib, name)  # AttributeError if the library does not export it
    fn.restype = restype
    fn.argtypes = argtypes
    if name in _NO_STATUS:
        return fn

    def checked(*args):
        rc = fn(*args)
        if rc != 0:
            raise SpfyError(rc, name, last_error())
        return rc

    checked.__name__ = name
    checked.raw = fn
    return checked


def _missing(name):
    def stub(*_args):
        raise SpfyError(E_UNSUPPORTED, name, "not exported by the library selected with SPFY_LIB")
    stub.__name__ = name
    return stub


for _name, (_res, _args) in SIGNATURES.items():
    try:
        globals()[_name] = _bind(_name, _res, _args)
    except AttributeError:
        if not os.environ.get("SPFY_LIB"):  # the shipped library must export everything the header declares
            raise
        globals()[_name] = _missing(_name)  # A/B runs against an older build


def version():
    return _lib.spfy_version()


def launch_count():
    """Number of kernels this library has launched in this process (bench: gpu_launches)."""
    return int(_lib.spfy_launch_count())


def exported_symbols():
    """Names the loaded library actually exports from the declared set (used by the tests)."""
    return [n for n in SIGNATURES if hasattr(_lib, n)]
