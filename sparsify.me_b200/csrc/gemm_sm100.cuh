// gemm_sm100.cuh -- internal interface of the dense tcgen05 GEMM (gemm_sm100.cu), shared with the
// unstructured-SpMM entry points of spmm.cu, which densify their sparse operand and contract on tensor cores.
#pragma once
#include "common.cuh"

namespace spfy {

// One column-major (BLAS convention) batched problem:
//   C_b[m x n, ldc] = alpha * op(A_b)[m x k] * op(B_b)[k x n] + beta * C_b,   b in [0, nb)
// A_b = A + b*strideA elements (strideA == 0: one A shared by all batches), same for B.  C_b = c_ptrs[b] when
// c_ptrs (a DEVICE array of nb pointers) is given, else C + b*strideC.  opX = SPFY_OP_N: the operand is stored as
// its op() shape in column-major order; SPFY_OP_T: as the transposed shape.
struct TcGemmProblem {
  int opA = 0, opB = 0;
  size_t m = 0, n = 0, k = 0, nb = 1;
  const void* A = nullptr;
  size_t lda = 0, strideA = 0;
  const void* B = nullptr;
  size_t ldb = 0, strideB = 0;
  void* C = nullptr;
  const void* const* c_ptrs = nullptr;
  size_t ldc = 0, strideC = 0;
  float alpha = 1.f, beta = 0.f;
};

enum { TC_GEMM_PRECISE = 0, TC_GEMM_FAST = 1 };  // fp32 inputs: 3xTF32 (fp32-level accuracy) / one TF32 product

// TMA contract for an operand: 16-byte aligned base, leading dimension and batch stride multiples of 16 bytes.
// tc_gemm_run copies an operand that misses it into the workspace with padded rows first (one extra pass over that
// operand); callers for which that pass is not worth it ask tc_gemm_supported(..., allow_repack = false) and take
// their CUDA-core path on SPFY_E_UNSUPPORTED.  `ws` must hold tc_gemm_workspace_bytes(...) bytes: the device
// copy of the problem table when count > 1 plus the padded copies.
int tc_gemm_supported(int dtype, const TcGemmProblem& p, bool allow_repack);
size_t tc_gemm_workspace_bytes(int dtype, const TcGemmProblem* problems, size_t count);
// `gate` (optional device word): the launch does its work only if (*gate != 0) == gate_run_if -- for callers that
// let the device choose between this kernel and a CUDA-core one and launch both.
int tc_gemm_run(int dtype, int precision, const TcGemmProblem* problems, size_t count, void* ws, size_t ws_bytes,
                cudaStream_t stream, const int* gate = nullptr, int gate_run_if = 1);
void warm_gemm_kernels();

}  // namespace spfy
