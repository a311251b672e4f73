"""sparsify.me_b200 -- host-side Python mirror of the `include/sparsify.me` operator API.

The product is libsparsifyme_b200.so (hand-written sm_100a CUDA behind the C ABI of
include/spfy_b200.h).  This module is the thin host layer the Python tests, the bench and
the multi-GPU driver use: it mirrors the reference's operator names and argument meaning

    sparsifyme::sparsify<BLK_M,BLK_N>      include/sparsify.me/sparsify.hxx:24-82   -> sparsify()
    sparsifyme::spmma                      include/sparsify.me/spmma.hxx:21-118     -> spmma()
    sparsifyme::batched::spmm              include/sparsify.me/spmm.hxx:30-138      -> batched.spmm()
    sparsifyme::batched::strided_coo       include/sparsify.me/spmm.hxx:140-193     -> batched.strided_coo()

and exposes the C ABI one-to-one under `capi`.  torch is used for device memory and streams
only.  There is NO CPU fallback: if the shared library is missing the import fails, and
every compute entry point fails without a CUDA device.

The directory name contains a dot (it is the reference's name), so it is loaded with
`__graft_entry__.load_package()` rather than a plain `import`.
"""
import ctypes
import os

from . import capi  # noqa: F401  (fails loudly if the .so is missing)
from .capi import (F16, BF16, F32, F64, PRUNE_STRIP_MAG, PRUNE_TILE_MAG, PRUNE_TILE_TRANSPOSABLE,  # noqa: F401
                   LAYOUT_CANONICAL, LAYOUT_SM100, OP_N, OP_T, OUT_T, SPMM_ALG_DEFAULT, SPMM_ALG_CUDA_CORE, SPMM_ALG_TENSOR,
                   SPMM_ALG_TENSOR_FAST, ACT_NONE, ACT_RELU, ACT_GELU_TANH, GEMM_PRECISE, GEMM_FAST, OPTIM_SGD, OPTIM_ADAMW, SpfyError, launch_count, last_error, version)
from .ops import (sparsify, prune24, prune24_check, compressed_bytes, spmma_compressed, spmma,  # noqa: F401
                  threshold_to_coo, coo_to_csr, batched, Compressed24, SpmmaPlan, prune24_batched,
                  alloc_compressed, pack_compressed, unpack_compressed, spmma_conv, spmma_conv_nhwc, permute_conv_weights,
                  Epilogue, fold_batchnorm, transpose24, recompress24, Linear24,
                  Transpose24Conv, transpose24_conv, spmma_conv_dgrad_nhwc, conv_wgrad24_nhwc, Conv2d24,
                  SGD24, AdamW24)
from . import shapes  # noqa: F401
from . import multigpu  # noqa: F401

__all__ = [
    "capi", "sparsify", "prune24", "prune24_check", "compressed_bytes", "spmma_compressed", "spmma",
    "threshold_to_coo", "coo_to_csr", "batched", "Compressed24", "SpmmaPlan", "prune24_batched", "alloc_compressed", "Epilogue", "fold_batchnorm", "transpose24", "recompress24", "Linear24", "Transpose24Conv", "transpose24_conv", "spmma_conv_dgrad_nhwc", "conv_wgrad24_nhwc", "Conv2d24", "SGD24", "AdamW24", "pack_compressed", "unpack_compressed", "shapes", "multigpu", "SpfyError",
    "launch_count", "last_error", "version",
]
