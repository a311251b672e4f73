// spmm.cu -- unstructured path: threshold prune -> COO/CSR, and SpMM with a CSR, COO or blocked-ELL operand
//
//   spfy_threshold_to_coo / spfy_coo_to_csr   magnitude-threshold compaction
//   spfy_spmm_csr_strided_batched             C_b = alpha*A*B_b + beta*C_b  (A shared)
//   spfy_spmm_coo_strided_batched             same, A in row-sorted COO
//                                             (reference: include/sparsify.me/spmm.hxx:140-193)
//   spfy_spmm_bell_batched                    blocked-ELL A_b per batch, B shared
//                                             (reference: include/sparsify.me/spmm.hxx:30-138)
//
// All dense operands are column-major like the reference's cuSPARSE descriptors (spmm.hxx:63,67,170,173).
// The file holds, in this order (each section's comment has the details):
//   - the threshold compaction (one chained-scan pass to sorted COO, and the CSR row pointers);
//   - the row-split kernel: the stand-in for 16-bit blocked-ELL operands that have no tensor-core route
//     (operands outside the TMA contract, repeated block ids);
//   - the CUDA-core kernels for fp32 CSR / blocked-ELL: one per non-zero, and the dense walk for dense operands;
//   - the tensor-core route: the sparse operand scattered / expanded into a dense matrix and contracted by the
//     tcgen05 GEMM of gemm_sm100.cu.
#include "common.cuh"
#include "gemm_sm100.cuh"

#include <cstdlib>
#include <type_traits>

namespace spfy {
namespace {

// ------------------------------------------------------------------------
// threshold -> COO/CSR in one pass (chained scan over 4096-element chunks, see threshold_compact_kernel);
// entries come out sorted by (row, col).
// ------------------------------------------------------------------------
// One pass, chained scan.  The matrix is walked in row-major element order in chunks of 4096 elements
// (256 threads x 4 groups of 4), one per CTA.  A CTA counts the kept elements of its chunk, publishes the count,
// looks back over its predecessors' (aggregate | inclusive prefix) words, 32 per step, until it meets an inclusive prefix,
// publishes its own, and writes its entries at prefix + rank: the input is read from DRAM once and the COO
// comes out sorted by (row, column).  The kept elements wait in shared memory at their rank inside the chunk,
// so the look-back overlaps that staging and the entries leave as full, coalesced lines.  A warp request covers 128 consecutive elements (32 lanes x 4): with
// 16-byte aligned rows one 128-bit (fp32) or 64-bit (fp16 / bf16) load per lane.  The counts of a thread's four
// groups travel as four bytes of one word, so one shuffle scan per warp serves all four.  row_ptr[r] is the
// position of the first element of row r, written by whoever holds that element.
constexpr int TC_THREADS = 256;
constexpr int TC_GROUPS = 4;                          // groups of 4 elements per thread
constexpr int TC_CHUNK = TC_THREADS * TC_GROUPS * 4;  // elements per chunk
constexpr unsigned long long TC_AGGREGATE = 1ull << 62, TC_PREFIX = 2ull << 62, TC_VALUE = (1ull << 62) - 1;

template <typename T>
__device__ __forceinline__ void load_group(const T* p, bool vec, uint32_t n, float (&x)[4]);
template <>
__device__ __forceinline__ void load_group<float>(const float* p, bool vec, uint32_t n, float (&x)[4]) {
  if (vec) {
    const float4 v = __ldg(reinterpret_cast<const float4*>(p));
    x[0] = v.x; x[1] = v.y; x[2] = v.z; x[3] = v.w;
  } else {
#pragma unroll
    for (int i = 0; i < 4; ++i) x[i] = (uint32_t)i < n ? __ldg(p + i) : 0.f;
  }
}
template <>
__device__ __forceinline__ void load_group<__half>(const __half* p, bool vec, uint32_t n, float (&x)[4]) {
  if (vec) {
    const uint2 v = __ldg(reinterpret_cast<const uint2*>(p));
    const __half2 lo = *reinterpret_cast<const __half2*>(&v.x), hi = *reinterpret_cast<const __half2*>(&v.y);
    x[0] = __low2float(lo); x[1] = __high2float(lo); x[2] = __low2float(hi); x[3] = __high2float(hi);
  } else {
#pragma unroll
    for (int i = 0; i < 4; ++i) x[i] = (uint32_t)i < n ? __half2float(p[i]) : 0.f;
  }
}
template <>
__device__ __forceinline__ void load_group<__nv_bfloat16>(const __nv_bfloat16* p, bool vec, uint32_t n, float (&x)[4]) {
  if (vec) {
    const uint2 v = __ldg(reinterpret_cast<const uint2*>(p));
    x[0] = __uint_as_float(v.x << 16); x[1] = __uint_as_float(v.x & 0xffff0000u);
    x[2] = __uint_as_float(v.y << 16); x[3] = __uint_as_float(v.y & 0xffff0000u);
  } else {
#pragma unroll
    for (int i = 0; i < 4; ++i) x[i] = (uint32_t)i < n ? __bfloat162float(p[i]) : 0.f;
  }
}

// n / cols for n < 2^31 with the host-made multiplier floor(2^(31+l) / cols) + 1, l = ceil(log2 cols)
__device__ __forceinline__ uint32_t tc_div(uint32_t n, uint32_t cols, uint32_t mul, uint32_t shift) {
  return cols == 1u ? n : __umulhi(n, mul) >> shift;
}

// the 16 elements of one thread for one chunk: values, and row / column of the first element of every group
template <typename T, bool FAST>
__device__ __forceinline__ void tc_load(const T* __restrict__ in, size_t ld, uint32_t cols, uint32_t div_mul,
                                        uint32_t div_shift, int vec, uint32_t total, uint32_t e_chunk, uint32_t warp,
                                        uint32_t lane, float (&x)[TC_GROUPS][4], uint32_t (&gr)[TC_GROUPS],
                                        uint32_t (&gc)[TC_GROUPS]) {
#pragma unroll
  for (int g = 0; g < TC_GROUPS; ++g) {
    // group g of this lane: elements e0 .. e0+3, 128 consecutive elements per warp and g
    const uint32_t e0 = e_chunk + (warp * TC_GROUPS + g) * 128u + lane * 4u;
    const uint32_t n = FAST ? 4u : (e0 < total ? min(4u, total - e0) : 0u);
    uint32_t r = 0, c = 0;
    if (n) {
      r = tc_div(e0, cols, div_mul, div_shift);
      c = e0 - r * cols;
    }
    gr[g] = r;
    gc[g] = c;
    if (FAST || (n && vec)) {
      load_group<T>(in + (size_t)r * ld + c, true, 4, x[g]);
    } else {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        x[g][i] = 0.f;
        if ((uint32_t)i < n) {
          const uint32_t cc = c + i;  // may run past the row end when a group straddles rows
          const uint32_t dr = tc_div(cc, cols, div_mul, div_shift);
          float one[4];
          load_group<T>(in + (size_t)(r + dr) * ld + (cc - dr * cols), false, 1, one);
          x[g][i] = one[0];
        }
      }
    }
  }
}

// vec: cols % 4 == 0, ld % 4 == 0 and the base is aligned to four elements, so a group never straddles a row.
// One chunk per CTA, chunk = block index: blocks are dispatched in index order, so every predecessor of a
// running chunk is running or done (the assumption CUB's decoupled look-back scans make).  Measured
// alternatives that lost: a ticket counter in front of the loads (+1 L2 round trip per CTA), and a persistent
// grid with ticketed chunks and prefetched loads, and four consecutive chunks per CTA (in both, a CTA's later
// chunk gates some other CTA's current one: the chain turns serial, 379 us and 48 ms).  What is left is the rate
// at which CTAs start: ~100 chunks per microsecond whatever a chunk holds (fp32, fp16 and 147-column inputs alike).
// FAST: the chunk is complete and the vector path applies -- no per-element bounds tests (the kernel is bound
// by instruction issue, and almost every chunk is such a chunk)
template <typename T, bool FAST>
__device__ __forceinline__ void tc_chunk(const T* __restrict__ in, size_t ld, uint32_t rows, uint32_t cols, uint32_t div_mul,
                                         uint32_t div_shift, float thr, int vec, uint32_t nchunks,
                                         int32_t* __restrict__ row_idx, int32_t* __restrict__ col_idx,
                                         float* __restrict__ vals, size_t capacity, int32_t* __restrict__ row_ptr,
                                         int64_t* __restrict__ nnz_out, unsigned long long* __restrict__ status,
                                         uint32_t* s_warp_total, float* s_val, uint16_t* s_elem) {
  const uint32_t lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const uint32_t total = rows * cols;  // < 2^31 (checked by the host)

  const uint32_t chunk = blockIdx.x;
  float x[TC_GROUPS][4];
  uint32_t gr[TC_GROUPS], gc[TC_GROUPS];
  tc_load<T, FAST>(in, ld, cols, div_mul, div_shift, vec, total, chunk * (uint32_t)TC_CHUNK, warp, lane, x, gr, gc);

  {
    const uint32_t e_chunk = chunk * (uint32_t)TC_CHUNK;
    unsigned keep = 0;    // 4 bits per group
    uint32_t packed = 0;  // kept count of group g in byte g
#pragma unroll
    for (int g = 0; g < TC_GROUPS; ++g) {
      const uint32_t e0 = e_chunk + (warp * TC_GROUPS + g) * 128u + lane * 4u;
      const uint32_t n = FAST ? 4u : (e0 < total ? min(4u, total - e0) : 0u);
      unsigned k4 = 0;
#pragma unroll
      for (int i = 0; i < 4; ++i) k4 |= ((uint32_t)i < n && fabsf(x[g][i]) > thr) ? 1u << i : 0u;
      keep |= k4 << (4 * g);
      packed |= (uint32_t)__popc(k4) << (8 * g);
    }
    // inclusive scan over the lanes, all four byte lanes at once (a byte holds at most 32 * 4 = 128)
    uint32_t incl = packed;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const uint32_t y = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= (uint32_t)o) incl += y;
    }
    const uint32_t tot = __shfl_sync(0xffffffffu, incl, 31);  // per-group totals of this warp
    const uint32_t excl = incl - packed;
    // group g of the warp precedes group g+1: bases of the four groups inside the warp
    const uint32_t t0 = tot & 0xffu, t1 = (tot >> 8) & 0xffu, t2 = (tot >> 16) & 0xffu, t3 = tot >> 24;
    if (lane == 0) s_warp_total[warp] = t0 + t1 + t2 + t3;
    __syncthreads();
    uint32_t warp_base = 0, cta_total = 0;
#pragma unroll
    for (int w = 0; w < TC_THREADS / 32; ++w) {
      const uint32_t v = s_warp_total[w];
      if ((uint32_t)w < warp) warp_base += v;
      cta_total += v;
    }
    // the count goes out first: successors can already add it while this chunk is still looking back
    if (threadIdx.x == 0 && chunk > 0) atomicExch(&status[chunk], TC_AGGREGATE | (unsigned long long)cta_total);

    // ---- kept elements to shared memory at their rank inside the chunk ----
    const uint32_t gbase[TC_GROUPS] = {0u, t0, t0 + t1, t0 + t1 + t2};
    uint32_t first_rank[TC_GROUPS];  // chunk-local rank of the first element of every group (kept or not)
#pragma unroll
    for (int g = 0; g < TC_GROUPS; ++g) {
      uint32_t rank = warp_base + gbase[g] + ((excl >> (8 * g)) & 0xffu);
      first_rank[g] = rank;
      const unsigned k4 = (keep >> (4 * g)) & 0xfu;
      const uint32_t local = (warp * TC_GROUPS + g) * 128u + lane * 4u;
      // ranks written out instead of a running counter: four independent predicated store pairs, no branches
      const uint32_t r1 = rank + (k4 & 1u), r2 = r1 + (k4 >> 1 & 1u), r3 = r2 + (k4 >> 2 & 1u);
      if (k4 & 1u) { s_val[rank] = x[g][0]; s_elem[rank] = (uint16_t)local; }
      if (k4 & 2u) { s_val[r1] = x[g][1]; s_elem[r1] = (uint16_t)(local + 1u); }
      if (k4 & 4u) { s_val[r2] = x[g][2]; s_elem[r2] = (uint16_t)(local + 2u); }
      if (k4 & 8u) { s_val[r3] = x[g][3]; s_elem[r3] = (uint16_t)(local + 3u); }
    }

    // ---- chained scan across chunks.  The whole CTA looks back, 256 predecessors per step (thread i reads
    // the word of chunk - 1 - i) ----
    uint32_t before = 0;  // kept elements in all earlier chunks (the same value in every thread)
    for (int64_t j0 = (int64_t)chunk - 1; chunk > 0; j0 -= TC_THREADS) {
      const int64_t j = j0 - (int64_t)threadIdx.x;
      unsigned long long w = TC_PREFIX;  // before the first chunk: an inclusive prefix of 0
      if (j >= 0) {
        do {
          w = *reinterpret_cast<volatile unsigned long long*>(&status[j]);
        } while ((w >> 62) == 0);
      }
      const unsigned has_prefix = __ballot_sync(0xffffffffu, (w >> 62) == 2);
      const uint32_t upto = has_prefix ? (uint32_t)__ffs(has_prefix) - 1u : 31u;  // nearest inclusive prefix
      uint32_t v = lane <= upto ? (uint32_t)(w & TC_VALUE) : 0u;
#pragma unroll
      for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
      __syncthreads();  // s_warp_total is free (everyone has read it / the previous step's result)
      if (lane == 0) s_warp_total[warp] = v | (has_prefix ? 0x80000000u : 0u);  // counts are < 2^31
      __syncthreads();
      bool done = false;
#pragma unroll
      for (int w8 = 0; w8 < TC_THREADS / 32; ++w8) {
        const uint32_t t = s_warp_total[w8];
        if (!done) before += t & 0x7fffffffu;
        done = done || (t >> 31);
      }
      if (done) break;
    }
    if (threadIdx.x == 0) {
      atomicExch(&status[chunk], TC_PREFIX | (unsigned long long)(before + cta_total));
      if (chunk + 1 == nchunks) {
        if (nnz_out) *nnz_out = (int64_t)(before + cta_total);
        if (row_ptr) row_ptr[rows] = (int32_t)(before + cta_total);
      }
    }
    __syncthreads();  // the staged entries of all warps are in place
    const uint32_t base = before;

    // ---- entries out, coalesced; (row, column) are recomputed from the element index ----
    // positions are < 2^31: 32-bit compares, and entries beyond `capacity` are dropped by shortening the loop
    const uint32_t cap32 = capacity > 0x7fffffffull ? 0x7fffffffu : (uint32_t)capacity;
    const uint32_t n_out = base >= cap32 ? 0u : min(cta_total, cap32 - base);
    int32_t* const ro = row_idx + base;
    int32_t* const co = col_idx + base;
    float* const vo = vals + base;
    for (uint32_t i = threadIdx.x; i < n_out; i += TC_THREADS) {
      const uint32_t e = e_chunk + s_elem[i];
      const uint32_t r = tc_div(e, cols, div_mul, div_shift);
      ro[i] = (int32_t)r;
      co[i] = (int32_t)(e - r * cols);
      vo[i] = s_val[i];
    }
    // ---- row_ptr[r] = position of the first element of row r ----
    if (row_ptr) {
#pragma unroll
      for (int g = 0; g < TC_GROUPS; ++g) {
        const uint32_t e0 = e_chunk + (warp * TC_GROUPS + g) * 128u + lane * 4u;
        const unsigned k4 = (keep >> (4 * g)) & 0xfu;
        uint32_t r = gr[g], c = gc[g], rank = first_rank[g];
        if (c != 0 && c + 4u <= cols) continue;  // no row starts inside this group
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          if (FAST || e0 + i < total) {
            if (c == 0) row_ptr[r] = (int32_t)(base + rank);
            rank += k4 >> i & 1u;
            if (++c == cols) {
              c = 0;
              ++r;
            }
          }
        }
      }
    }
  }
}

// vec: cols % 4 == 0, ld % 4 == 0 and the base is aligned to four elements, so a group never straddles a row
template <typename T>
__global__ void __launch_bounds__(TC_THREADS, 6)
threshold_compact_kernel(const T* __restrict__ in, size_t ld, uint32_t rows, uint32_t cols, uint32_t div_mul,
                         uint32_t div_shift, float thr, int vec, uint32_t nchunks,
                         int32_t* __restrict__ row_idx, int32_t* __restrict__ col_idx, float* __restrict__ vals,
                         size_t capacity, int32_t* __restrict__ row_ptr, int64_t* __restrict__ nnz_out,
                         unsigned long long* __restrict__ status) {
  __shared__ uint32_t s_warp_total[TC_THREADS / 32];
  __shared__ float s_val[TC_CHUNK];      // the chunk's kept values in output order ...
  __shared__ uint16_t s_elem[TC_CHUNK];  // ... and where in the chunk each one came from
  if (vec && ((size_t)blockIdx.x + 1) * TC_CHUNK <= (size_t)rows * cols)
    tc_chunk<T, true>(in, ld, rows, cols, div_mul, div_shift, thr, vec, nchunks, row_idx, col_idx, vals, capacity, row_ptr,
                      nnz_out, status, s_warp_total, s_val, s_elem);
  else
    tc_chunk<T, false>(in, ld, rows, cols, div_mul, div_shift, thr, vec, nchunks, row_idx, col_idx, vals, capacity, row_ptr,
                       nnz_out, status, s_warp_total, s_val, s_elem);
}

__global__ void __launch_bounds__(256)
coo_to_csr_kernel(const int32_t* __restrict__ row_idx, size_t nnz, uint32_t rows,
                  int32_t* __restrict__ row_ptr) {
  const size_t nthreads = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i <= nnz; i += nthreads) {
    const int64_t prev = i == 0 ? -1 : (int64_t)row_idx[i - 1];
    const int64_t cur = i == nnz ? (int64_t)rows : (int64_t)row_idx[i];
    for (int64_t r = prev + 1; r <= cur && r <= (int64_t)rows; ++r) row_ptr[r] = (int32_t)i;
  }
}

// ------------------------------------------------------------------------
// Row-split SpMM: a CTA owns a tile of TM rows x 32 columns.  The dense operand tile B[k-chunk x 32] is staged
// TRANSPOSED in shared memory so that for one non-zero (i, c) the 32 lanes of a warp read 32 consecutive words
// (one per output column).  A warp owns RPW rows; it loads 32 non-zeros with one coalesced request and broadcasts
// them with shuffles.  Accumulators live in registers; the C tile goes back through shared memory so the
// column-major stores are coalesced along rows.
// ------------------------------------------------------------------------
constexpr int SP_WARPS = 16;           // warps per CTA
constexpr int SP_RPW = 8;              // rows per warp
constexpr int SP_TM = SP_WARPS * SP_RPW;  // 128 rows per CTA
constexpr int SP_TN = 32;              // columns per CTA (one per lane)
constexpr int SP_PAD = SP_TN + 1;      // padded row of the transposed B tile

template <typename T>
struct BellRows {  // blocked-ELL, one matrix per batch (reference: containers/ell.hxx:24-33)
  const int64_t* const* col_idx;  // [batch] -> [(rows/block) x (ell_cols/block)]
  const T* const* values;         // [batch] -> [rows x ell_cols]
  uint32_t block, ell_cols, bcols;
  __device__ __forceinline__ void range(uint32_t, uint32_t, uint32_t& b, uint32_t& e) const {
    b = 0;
    e = ell_cols;
  }
  __device__ __forceinline__ void fetch(uint32_t batch, uint32_t row, uint32_t idx, int32_t& c, float& v) const {
    const int64_t bc = col_idx[batch][(size_t)(row / block) * bcols + idx / block];
    c = bc < 0 ? -1 : (int32_t)(bc * block + idx % block);
    v = to_f32(values[batch][(size_t)row * ell_cols + idx]);
  }
};

struct SpmmDense {
  const void* B;
  void* C;                 // single slab (strided batches) ...
  void* const* Cs;         // ... or per-batch pointers (BELL); one of the two is null
  size_t ldb, strideB, ldc, strideC;
  uint32_t m, k, n, num_batches;
  uint32_t kc;             // rows of B staged per chunk
  float alpha, beta;
  const int* gate;         // device flag (null = run): work only if (*gate != 0) == gate_run_if
  uint32_t gate_run_if;
};

template <typename T, typename Rows>
__global__ void __launch_bounds__(SP_WARPS * 32, 1)
spmm_rowsplit_kernel(const Rows A, const SpmmDense D) {
  extern __shared__ float sB[];  // [kc][SP_PAD]; reused as [SP_TN][SP_TM+1] for the C tile
  if (D.gate && (*D.gate != 0) != (D.gate_run_if != 0)) return;  // another kernel handles this batch (device-side choice)
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const uint32_t row_tiles = (D.m + SP_TM - 1) / SP_TM;
  const uint32_t col_tiles = (D.n + SP_TN - 1) / SP_TN;
  const uint32_t rt = blockIdx.x % row_tiles;         // row tile fastest: CTAs that share a
  const uint32_t ct_all = blockIdx.x / row_tiles;     // B tile are co-resident (L2 reuse)
  const uint32_t batch = ct_all / col_tiles, ct = ct_all % col_tiles;
  const uint32_t j0 = ct * SP_TN, i0 = rt * SP_TM;
  const T* Bb = reinterpret_cast<const T*>(D.B) + (size_t)batch * D.strideB;
  T* Cb = D.Cs ? reinterpret_cast<T*>(D.Cs[batch]) : reinterpret_cast<T*>(D.C) + (size_t)batch * D.strideC;

  float acc[SP_RPW];
#pragma unroll
  for (int r = 0; r < SP_RPW; ++r) acc[r] = 0.f;

  for (uint32_t k0 = 0; k0 < D.k; k0 += D.kc) {
    const uint32_t kn = min(D.kc, D.k - k0);
    __syncthreads();
    // stage B[k0:k0+kn, j0:j0+32] transposed: coalesced along k in global memory
    for (uint32_t j = warp; j < SP_TN; j += SP_WARPS) {
      const bool col_ok = j0 + j < D.n;
      const T* src = Bb + (size_t)(j0 + j) * D.ldb + k0;
      for (uint32_t kk = lane; kk < kn; kk += 32)
        sB[kk * SP_PAD + j] = col_ok ? to_f32(src[kk]) : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int r = 0; r < SP_RPW; ++r) {
      const uint32_t row = i0 + warp * SP_RPW + r;
      if (row >= D.m) break;
      uint32_t eb, ee;
      A.range(batch, row, eb, ee);
      for (uint32_t e0 = eb; e0 < ee; e0 += 32) {
        int32_t c = -1;
        float v = 0.f;
        if (e0 + lane < ee) A.fetch(batch, row, e0 + lane, c, v);
        const int32_t rel = c - (int32_t)k0;
        const bool in_chunk = c >= 0 && rel >= 0 && rel < (int32_t)kn;
        unsigned live = __ballot_sync(0xffffffffu, in_chunk);
        while (live) {
          const int src_lane = __ffs(live) - 1;
          live &= live - 1;
          const int32_t rc = __shfl_sync(0xffffffffu, rel, src_lane);
          const float rv = __shfl_sync(0xffffffffu, v, src_lane);
          acc[r] = fmaf(rv, sB[rc * SP_PAD + lane], acc[r]);
        }
      }
    }
  }

  // C tile through shared memory: sC[j][i] so that global stores run along rows
  __syncthreads();
  float* sC = sB;
#pragma unroll
  for (int r = 0; r < SP_RPW; ++r) sC[lane * (SP_TM + 1) + warp * SP_RPW + r] = acc[r];
  __syncthreads();
  for (uint32_t idx = threadIdx.x; idx < SP_TN * SP_TM; idx += SP_WARPS * 32) {
    const uint32_t j = idx / SP_TM, i = idx % SP_TM;
    if (j0 + j < D.n && i0 + i < D.m) {
      T* dst = Cb + (size_t)(j0 + j) * D.ldc + i0 + i;
      float out = D.alpha * sC[j * (SP_TM + 1) + i];
      if (D.beta != 0.f) out += D.beta * to_f32(*dst);
      *dst = from_f32<T>(out);
    }
  }
}

template <typename T, typename Rows>
int launch_spmm(const Rows& A, SpmmDense D, cudaStream_t s) {
  DeviceInfo di;
  int rc = device_info(&di);
  if (rc) return rc;
  // chunk of k staged per pass: as much as fits next to the C tile
  const size_t c_tile = (size_t)SP_TN * (SP_TM + 1) * 4;
  size_t budget = (size_t)di.max_smem_optin - 1024;
  size_t kc = budget / (SP_PAD * 4);
  if (kc > D.k) kc = D.k;
  if (kc == 0) kc = 1;
  size_t smem = kc * SP_PAD * 4;
  if (smem < c_tile) smem = c_tile;
  D.kc = (uint32_t)kc;
  rc = allow_dynamic_smem<spmm_rowsplit_kernel<T, Rows>>(budget);
  if (rc) return rc;
  const size_t row_tiles = ceil_div(D.m, SP_TM), col_tiles = ceil_div(D.n, SP_TN);
  const size_t ctas = row_tiles * col_tiles * D.num_batches;
  if (ctas == 0) return SPFY_OK;
  if (ctas >= (1ull << 31)) return fail(SPFY_E_UNSUPPORTED, "spmm: grid too large");
  spmm_rowsplit_kernel<T, Rows><<<(unsigned)ctas, SP_WARPS * 32, smem, s>>>(A, D);
  SPFY_LAUNCH_OK("spmm_rowsplit_kernel");
  return SPFY_OK;
}

// ------------------------------------------------------------------------
// CSR / COO SpMM, fp32 (the operand types of spmm.hxx:165-180): C_b = alpha * A * B_b + beta * C_b,
// one sparse A shared by all batch elements, B_b / C_b column-major.
//
// Every FMA needs one dynamically addressed B element, which can only come from shared memory, so
// the kernel is bound by shared-memory wavefronts (128 B/clk/SM), not by the FMA pipe: a lane owns
// CSR_TJ = 4 columns, one non-zero costs one broadcast LDS.64 (value + column) plus four LDS.32 for
// four FMAs.  CTA tile = (16 warps x RPW rows) x 128 columns, one CTA per SM; K is walked in chunks
// of 192 rows of B staged as sB[column][k] (odd row pitch: conflict-free both for the fill along k
// and for the per-non-zero reads across columns).  The fill is software-pipelined through
// registers: the 48 floats a thread contributes to chunk c+1 are requested before chunk c is
// multiplied and stored after it, so a whole chunk (96 KiB per SM) is in flight under the math.
// A warp reads the non-zeros of a row 32 at a time with one coalesced request, compacts the ones
// that fall into the staged chunk into a per-warp scratch line and replays them.  With ascending
// columns inside a row (what spfy_threshold_to_coo emits; `*sorted` says so) a per-row cursor makes
// this one visit per non-zero; otherwise every chunk rescans the row.  The C tile goes back through
// shared memory so the column-major stores run along rows.
// ------------------------------------------------------------------------
constexpr int CSR_WARPS = 16;
constexpr int CSR_THREADS = CSR_WARPS * 32;
constexpr int CSR_TN = 128;
constexpr int CSR_TJ = CSR_TN / 32;
constexpr int CSR_KC = 192;
constexpr int CSR_PITCH = CSR_KC + 1;
constexpr int CSR_PF = CSR_TN * CSR_KC / CSR_THREADS;  // 48 floats per thread and chunk

struct CsrSpmmParams {
  const int32_t* row_ptr;
  const int32_t* col_idx;
  const float* vals;
  const float* B;
  float* C;
  const int* sorted;        // device flag: columns ascend inside every row
  const int* gate;          // device flag (null = run): the kernel works only if (*gate != 0) == gate_run_if, so a
  uint32_t gate_run_if;     // caller that leaves the kernel choice to the device launches every candidate
  size_t ldb, strideB, ldc, strideC;
  uint32_t m, k, n, num_batches;
  uint32_t row_tiles, col_tiles;  // col tiles over the num_batches * n columns
  uint32_t vec;                    // B columns are 16-byte aligned: 128-bit fill
  float alpha, beta;
  // blocked-ELL source (spmm.hxx:30-138): one A per batch element, B shared, one C pointer per batch
  const int64_t* const* bell_cols;  // [batch] -> [(m / block) x bcols] block-column ids, < 0 = padding
  const float* const* bell_vals;    // [batch] -> [m x ell_cols]
  float* const* Cs;                 // [batch] -> m x n column-major
  uint32_t block, ell_cols, bcols;
};

// blocked-ELL rows are "sorted" when block-column ids ascend and padding only trails
__global__ void __launch_bounds__(256)
bell_check_sorted_kernel(const int64_t* const* __restrict__ cols, uint32_t block_rows, uint32_t bcols,
                         uint32_t num_batches, int* __restrict__ sorted) {
  const size_t total = (size_t)num_batches * block_rows * bcols;
  const size_t nthreads = (size_t)gridDim.x * blockDim.x;
  bool bad = false;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += nthreads) {
    const uint32_t j = (uint32_t)(i % bcols);
    if (j == 0) continue;
    const size_t br = i / bcols;
    const int64_t* c = cols[br / block_rows] + (br % block_rows) * (size_t)bcols;
    const int64_t a = c[j - 1], b = c[j];
    bad |= a < 0 ? b >= 0 : (b >= 0 && b < a);
  }
  if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) atomicExch(sorted, 0);
}

__global__ void __launch_bounds__(256)
csr_check_sorted_kernel(const int32_t* __restrict__ row_ptr, const int32_t* __restrict__ col_idx, uint32_t m,
                        int* __restrict__ sorted, int* __restrict__ walk, uint32_t walk_nnz) {
  const uint32_t lane = threadIdx.x & 31;
  if (walk && blockIdx.x == 0 && threadIdx.x == 0) *walk = (uint32_t)row_ptr[m] >= walk_nnz;
  const uint32_t warps = (gridDim.x * blockDim.x) >> 5;
  bool bad = false;
  for (uint32_t r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < m; r += warps) {
    const int32_t b = row_ptr[r], e = row_ptr[r + 1];
    for (int32_t i = b + 1 + (int32_t)lane; i < e; i += 32) bad |= col_idx[i] < col_idx[i - 1];
  }
  if (__any_sync(0xffffffffu, bad) && lane == 0) atomicExch(sorted, 0);
}

// the 48 floats of one thread for the chunk starting at k0.  `wide`: a quarter warp per column and
// request (8 lanes x 16 bytes = one line; the four columns of a request fall into four different
// bank groups, so the scalar stores are conflict-free); otherwise a warp per column, lanes along k.
__device__ __forceinline__ void csr_chunk_load(float (&pf)[CSR_PF], const CsrSpmmParams& P, const size_t* colB,
                                               uint32_t k0, uint32_t kn, bool wide, uint32_t warp, uint32_t lane) {
  if (wide) {
    const uint32_t l8 = lane & 7u;
#pragma unroll
    for (int s = 0; s < 2; ++s) {
      const uint32_t jj = s * 64 + warp * 4 + (lane >> 3);
      const size_t off = colB[jj];
      const float4* src = reinterpret_cast<const float4*>(P.B + (off == ~(size_t)0 ? 0 : off) + k0);
#pragma unroll
      for (int q = 0; q < 6; ++q) {
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (off != ~(size_t)0) v = __ldg(src + q * 8 + l8);
        pf[(s * 6 + q) * 4 + 0] = v.x;
        pf[(s * 6 + q) * 4 + 1] = v.y;
        pf[(s * 6 + q) * 4 + 2] = v.z;
        pf[(s * 6 + q) * 4 + 3] = v.w;
      }
    }
  } else {
#pragma unroll
    for (int s = 0; s < 8; ++s) {
      const uint32_t jj = s * 16 + warp;
      const size_t off = colB[jj];
      const float* src = P.B + (off == ~(size_t)0 ? 0 : off) + k0;
#pragma unroll
      for (int u = 0; u < 6; ++u) {
        const uint32_t kk = u * 32 + lane;
        pf[s * 6 + u] = (off != ~(size_t)0 && kk < kn) ? __ldg(src + kk) : 0.f;
      }
    }
  }
}

template <int PITCH>
__device__ __forceinline__ void csr_chunk_store(const float (&pf)[CSR_PF], float* sB, bool wide, uint32_t warp,
                                                uint32_t lane) {
  if (wide) {
    const uint32_t l8 = lane & 7u;
#pragma unroll
    for (int s = 0; s < 2; ++s) {
      float* dst = sB + (s * 64 + warp * 4 + (lane >> 3)) * PITCH + l8 * 4;
#pragma unroll
      for (int q = 0; q < 6; ++q)
#pragma unroll
        for (int i = 0; i < 4; ++i) dst[q * 32 + i] = pf[(s * 6 + q) * 4 + i];
    }
  } else {
#pragma unroll
    for (int s = 0; s < 8; ++s) {
      float* dst = sB + (s * 16 + warp) * PITCH + lane;
#pragma unroll
      for (int u = 0; u < 6; ++u) dst[u * 32] = pf[s * 6 + u];
    }
  }
}

// one request of a row: lane `lane` reads entry `idx` (CSR: position in col_idx / vals; blocked-ELL: slot
// of the row); returns the column (0x7fffffff = nothing) and the value
template <bool BELL>
__device__ __forceinline__ void csr_fetch(const CsrSpmmParams& P, uint32_t batch, uint32_t row, uint32_t idx,
                                          bool ok, int32_t& c, float& v) {
  c = 0x7fffffff;
  v = 0.f;
  if (!ok) return;
  if (BELL) {
    const int64_t bc = P.bell_cols[batch][(size_t)(row / P.block) * P.bcols + idx / P.block];
    if (bc >= 0) c = (int32_t)(bc * P.block + idx % P.block);
    v = P.bell_vals[batch][(size_t)row * P.ell_cols + idx];
  } else {
    c = P.col_idx[idx];
    v = P.vals[idx];
  }
}

// element offsets of a tile's 128 columns inside B and C (~0: past the last column); CSR / COO: the batch
// elements' columns form one long column axis, blocked-ELL: tiles are per batch element
template <bool BELL>
__device__ __forceinline__ void spmm_tile_columns(const CsrSpmmParams& P, uint64_t j0, uint64_t ncols, size_t* colB,
                                                  size_t* colC) {
  if (threadIdx.x < CSR_TN) {
    const uint64_t J = j0 + threadIdx.x;
    size_t ob = ~(size_t)0, oc = ~(size_t)0;
    if (J < ncols) {
      const uint32_t bt = BELL ? 0u : (ncols <= 0xffffffffull ? (uint32_t)J / P.n : (uint32_t)(J / P.n));
      const size_t jc = (size_t)(J - (uint64_t)bt * P.n);
      ob = (size_t)bt * P.strideB + jc * P.ldb;
      oc = (size_t)bt * P.strideC + jc * P.ldc;
    }
    colB[threadIdx.x] = ob;
    colC[threadIdx.x] = oc;
  }
}

// the C tile staged as sC[column][TM + 1] goes out along rows (column-major C): alpha * acc + beta * C
template <int TM, int THREADS>
__device__ __forceinline__ void spmm_store_c_tile(const CsrSpmmParams& P, float* Cbase, const float* sC,
                                                  const size_t* colC, uint32_t rbase) {
#pragma unroll 4
  for (uint32_t idx = threadIdx.x; idx < (uint32_t)(CSR_TN * TM); idx += THREADS) {
    const uint32_t jj = idx / TM, i = idx % TM;
    const size_t oc = colC[jj];
    if (oc != ~(size_t)0 && rbase + i < P.m) {
      float* dst = Cbase + oc + rbase + i;
      float out = P.alpha * sC[jj * (TM + 1) + i];
      if (P.beta != 0.f) out += P.beta * *dst;
      *dst = out;
    }
  }
}

// MODE 0: CSR rows.  MODE 1: blocked-ELL rows, every slot an independent non-zero (any block size).
// MODE 2: blocked-ELL with an even block size, walked as (row pair) x (column pair): the two rows of a pair
// share their block-column ids, so one 64-bit read of B[c], B[c+1] per output column feeds four FMAs -- half
// the shared-memory wavefronts per FMA of MODE 1 (even row pitch: the 64-bit reads are aligned and
// conflict-free per half warp).
enum { SPMM_CSR = 0, SPMM_BELL = 1, SPMM_BELL_PAIRS = 2 };
constexpr int CSR_PITCH_PAIRS = CSR_KC + 2;
constexpr int CSR_SCRATCH_FLOATS = CSR_WARPS * 32 * 5;  // per warp: 32 x (column + up to four values)

template <int RPW, int MODE>
__global__ void __launch_bounds__(CSR_THREADS, 1)
spmm_csr_kernel(const __grid_constant__ CsrSpmmParams P) {
  constexpr bool BELL = MODE != SPMM_CSR;
  constexpr int PITCH = MODE == SPMM_BELL_PAIRS ? CSR_PITCH_PAIRS : CSR_PITCH;
  constexpr int TM = CSR_WARPS * RPW;
  extern __shared__ float smem_f[];
  float* sB = smem_f;                                                         // [CSR_TN][PITCH]
  float* scratch_f = smem_f + CSR_TN * CSR_PITCH_PAIRS + (threadIdx.x >> 5) * (32 * 5);
  uint2* scratch = reinterpret_cast<uint2*>(scratch_f);                       // MODE 0/1: 32 x (column, value)
  size_t* colB = reinterpret_cast<size_t*>(smem_f + CSR_TN * CSR_PITCH_PAIRS + CSR_SCRATCH_FLOATS);  // [CSR_TN]
  size_t* colC = colB + CSR_TN;                                                              // [CSR_TN]
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (P.gate && (*P.gate != 0) != (P.gate_run_if != 0)) return;  // another kernel handles this A (device-side choice)
  const bool sorted = *P.sorted != 0;
  const uint32_t nnz_total = BELL ? P.ell_cols : (uint32_t)P.row_ptr[P.m];
  // CSR: the batch elements' columns form one long column axis; blocked-ELL: tiles are per batch element
  const uint64_t ncols = BELL ? (uint64_t)P.n : (uint64_t)P.n * P.num_batches;
  const uint32_t tiles = P.row_tiles * P.col_tiles * (BELL ? P.num_batches : 1u);
  const uint32_t nchunks = (P.k + CSR_KC - 1) / CSR_KC;

  for (uint32_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const uint32_t rt = tile % P.row_tiles, ct_all = tile / P.row_tiles;  // row tile fastest: CTAs that
    const uint32_t i0 = rt * TM + warp * RPW;                              // share B columns run together
    const uint32_t batch = BELL ? ct_all / P.col_tiles : 0u;
    const uint32_t ct = BELL ? ct_all - batch * P.col_tiles : ct_all;
    const uint64_t j0 = (uint64_t)ct * CSR_TN;
    float* const Cbase = BELL ? P.Cs[batch] : P.C;

    __syncthreads();  // the previous tile's C stores have left shared memory
    spmm_tile_columns<BELL>(P, j0, ncols, colB, colC);
    __syncthreads();

    uint32_t cur[RPW];  // scan position of every row (row ends are re-read per chunk: registers are scarce)
    float acc[RPW][CSR_TJ];
#pragma unroll
    for (int r = 0; r < RPW; ++r) {
      const uint32_t row = i0 + r;
      cur[r] = (!BELL && row < P.m) ? (uint32_t)P.row_ptr[row] : 0u;
#pragma unroll
      for (int j = 0; j < CSR_TJ; ++j) acc[r][j] = 0.f;
    }

    float pf[CSR_PF];
    csr_chunk_load(pf, P, colB, 0, min((uint32_t)CSR_KC, P.k), P.vec && P.k >= (uint32_t)CSR_KC, warp, lane);

    for (uint32_t ch = 0; ch < nchunks; ++ch) {
      const uint32_t k0 = ch * CSR_KC;
      const uint32_t kn = min((uint32_t)CSR_KC, P.k - k0);
      if (ch) __syncthreads();  // everyone is done with the previous chunk
      csr_chunk_store<PITCH>(pf, sB, P.vec && kn == (uint32_t)CSR_KC, warp, lane);
      __syncthreads();
      if (ch + 1 < nchunks) {
        const uint32_t k1 = k0 + CSR_KC, kn1 = min((uint32_t)CSR_KC, P.k - k1);
        csr_chunk_load(pf, P, colB, k1, kn1, P.vec && kn1 == (uint32_t)CSR_KC, warp, lane);
      }

      // ---- multiply: every warp walks its RPW rows ----
      const uint32_t k_end = k0 + kn;
      const float* sBl = sB + lane * PITCH;
      if (MODE == SPMM_BELL_PAIRS) {
        // ---- blocked-ELL, (row pair) x (column pair); cur[2*rp] is the pair cursor of row pair rp ----
        uint32_t* sc = reinterpret_cast<uint32_t*>(scratch_f);       // [32] column (relative to k0)
        float4* sv = reinterpret_cast<float4*>(scratch_f + 32);      // [32] a(r0,c) a(r0,c+1) a(r0+1,c) a(r0+1,c+1)
        const uint32_t npairs = P.ell_cols / 2;
#pragma unroll
        for (int rp = 0; rp < RPW / 2; ++rp) {
          const uint32_t r0 = i0 + 2 * rp;
          if (r0 >= P.m) break;
          const bool r1_ok = r0 + 1 < P.m;
          const int64_t* bcol = P.bell_cols[batch] + (size_t)(r0 / P.block) * P.bcols;
          const float* v0p = P.bell_vals[batch] + (size_t)r0 * P.ell_cols;
          const float* v1p = v0p + P.ell_cols;
          uint32_t pos = sorted ? cur[2 * rp] : 0u;
          while (pos < npairs) {
            const uint32_t p = pos + lane;
            int32_t c = 0x7fffffff;
            float4 a = make_float4(0.f, 0.f, 0.f, 0.f);
            if (p < npairs) {
              const int64_t bc = bcol[(2 * p) / P.block];
              if (bc >= 0) c = (int32_t)(bc * P.block + (2 * p) % P.block);
              a.x = v0p[2 * p];
              a.y = v0p[2 * p + 1];
              if (r1_ok) {
                a.z = v1p[2 * p];
                a.w = v1p[2 * p + 1];
              }
            }
            unsigned cnt, adv;
            if (sorted) {
              cnt = adv = __popc(__ballot_sync(0xffffffffu, c < (int32_t)k_end));
              if (lane < cnt) {
                sc[lane] = (uint32_t)(c - (int32_t)k0);
                sv[lane] = a;
              }
            } else {
              const bool in = c >= (int32_t)k0 && c < (int32_t)k_end;
              const unsigned in_mask = __ballot_sync(0xffffffffu, in);
              cnt = __popc(in_mask);
              adv = 32u;
              if (in) {
                const unsigned at = __popc(in_mask & ((1u << lane) - 1u));
                sc[at] = (uint32_t)(c - (int32_t)k0);
                sv[at] = a;
              }
            }
            __syncwarp();
#pragma unroll 2
            for (unsigned t = 0; t < cnt; ++t) {
              const float4 av = sv[t];
              const float* bp = sBl + sc[t];
#pragma unroll
              for (int j = 0; j < CSR_TJ; ++j) {
                const float2 b = *reinterpret_cast<const float2*>(bp + j * 32 * PITCH);
                acc[2 * rp][j] = fmaf(av.y, b.y, fmaf(av.x, b.x, acc[2 * rp][j]));
                acc[2 * rp + 1][j] = fmaf(av.w, b.y, fmaf(av.z, b.x, acc[2 * rp + 1][j]));
              }
            }
            __syncwarp();
            pos += adv;
            if (sorted && adv < 32u) break;  // the rest of the row pair lies beyond this chunk
          }
          if (sorted) cur[2 * rp] = pos;
        }
      } else
      // rows are handled four at a time: the first request of each of the four goes out before any is
      // processed (cur[] doubles as the scan position; unsorted rows restart from the row start)
#pragma unroll
      for (int r0 = 0; r0 < RPW; r0 += 4) {
        int32_t c_[4];
        float v_[4];
        uint32_t end[4];
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int r = r0 + q;
          const bool row_ok = i0 + r < P.m;
          if (!sorted) cur[r] = (!BELL && row_ok) ? (uint32_t)P.row_ptr[i0 + r] : 0u;
          end[q] = row_ok ? (BELL ? P.ell_cols : (uint32_t)P.row_ptr[i0 + r + 1]) : 0u;
          // the request does not wait for the row end: any index below nnz is readable
          const uint32_t idx = cur[r] + lane;
          csr_fetch<BELL>(P, batch, i0 + r, idx, idx < nnz_total && (!BELL || row_ok), c_[q], v_[q]);
        }
#pragma unroll
        for (int q = 0; q < 4; ++q)
          if (cur[r0 + q] + lane >= end[q]) c_[q] = 0x7fffffff;
#pragma unroll
        for (int q = 0; q < 4; ++q) {
          const int r = r0 + q;
          while (true) {
            const int32_t c = c_[q];
            unsigned cnt, adv;
            if (sorted) {
              // everything at or after the cursor is >= k0, and what is below k_end is a prefix of the request
              cnt = adv = __popc(__ballot_sync(0xffffffffu, c < (int32_t)k_end));
              if (lane < cnt) scratch[lane] = make_uint2((uint32_t)(c - (int32_t)k0), __float_as_uint(v_[q]));
            } else {
              const bool in = c >= (int32_t)k0 && c < (int32_t)k_end;
              const unsigned in_mask = __ballot_sync(0xffffffffu, in);
              cnt = __popc(in_mask);
              adv = 32u;
              if (in)
                scratch[__popc(in_mask & ((1u << lane) - 1u))] =
                    make_uint2((uint32_t)(c - (int32_t)k0), __float_as_uint(v_[q]));
            }
            __syncwarp();
#pragma unroll 4
            for (unsigned t = 0; t < cnt; ++t) {
              const uint2 e = scratch[t];
              const float a = __uint_as_float(e.y);
              const float* bp = sBl + e.x;
#pragma unroll
              for (int j = 0; j < CSR_TJ; ++j) acc[r][j] = fmaf(a, bp[j * 32 * PITCH], acc[r][j]);
            }
            __syncwarp();
            bool more;
            if (sorted) {
              cur[r] += adv;
              more = adv == 32u;       // the whole request was below k_end: the row may continue in this chunk
            } else {
              cur[r] += 32u;
              more = cur[r] < end[q];  // unsorted: scan the whole row for every chunk
            }
            if (!more) break;
            const uint32_t idx = cur[r] + lane;
            csr_fetch<BELL>(P, batch, i0 + r, idx, idx < end[q], c_[q], v_[q]);
          }
        }
      }
    }

    // ---- C tile through shared memory: sC[column][row], stores run along rows ----
    __syncthreads();
    float* sC = smem_f;  // [CSR_TN][TM + 1]
#pragma unroll
    for (int r = 0; r < RPW; ++r)
#pragma unroll
      for (int j = 0; j < CSR_TJ; ++j) sC[(lane + 32 * j) * (TM + 1) + warp * RPW + r] = acc[r][j];
    __syncthreads();
    spmm_store_c_tile<TM, CSR_THREADS>(P, Cbase, sC, colC, rt * TM);
  }
}

// ------------------------------------------------------------------------
// Dense walk: the same product for an A that is not sparse enough for the kernel above.  There every
// FMA costs a shared-memory wavefront of its own (one B word per lane and FMA), which caps it at a
// quarter of the FP32 pipe; at 50 % sparsity (BASELINE configs[2], and the reference driver's
// blocked-ELL construction, examples/spmm.cu:47-48) it is cheaper to multiply by the zeros:
// per k-chunk a warp scatters its RPW rows of A into a zero-filled dense strip sA[row][k] and then
// walks k four at a time -- RPW broadcast LDS.128 of A and four LDS.128 of B feed 16 * RPW FMAs, so
// the FP32 pipe is the limit.  A broadcast LDS.128 costs two wavefronts and a per-lane one four (ncu), i.e.
// 16 + 2 * RPW wavefronts per 16 * RPW FMA instructions and warp: with RPW = 8 the shared-memory pipe is as
// busy as the FP32 pipe (measured: both 44 %), so a warp owns RPW = 16 rows (64 accumulators per lane, hence
// 8 warps per CTA).  Tile (8 warps x RPW rows) x 128 columns, same B/C conventions and sortedness handling
// as above; B chunks of 96 k
// are double-buffered with 16-byte cp.async (row pitch 100 floats: 16-byte aligned, and the eight
// lanes of a quarter warp land in eight different bank groups), so the next chunk streams in under
// the multiply.  Duplicate (row, column) entries add up (shared-memory atomics).
// Chosen for CSR / COO operands when nnz >= SPFY_SPMM_WALK_DENSITY (default 0.35) * m * k: by the host when it
// knows nnz (COO entry), else by a device flag that lets exactly one of the two kernels run.  Blocked-ELL
// operands stay on the per-non-zero kernel (measured: see spfy_spmm_bell_batched).
// ------------------------------------------------------------------------
constexpr int DW_KC = 96;
constexpr int DW_PITCH = 100;
constexpr int DW_Q = DW_PITCH / 4;
constexpr int DW_WARPS = 8;  // 256 threads: a warp needs 16 rows x 4 columns of accumulators per lane (see above)
constexpr int DW_THREADS = DW_WARPS * 32;

__device__ __forceinline__ void cp_async_16(float* dst_smem, const float* src, bool valid) {
  const uint32_t d = (uint32_t)__cvta_generic_to_shared(dst_smem);
  const uint32_t n = valid ? 16u : 0u;  // 0: the 16 bytes are zero-filled, src is not read
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(d), "l"(src), "r"(n) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;" ::: "memory"); }

// stage B[k0 .. k0+kn) x (the tile's 128 columns) as buf[column][k]; k in [kn, 96) is zero-filled
__device__ __forceinline__ void dw_fill(float* buf, const CsrSpmmParams& P, const size_t* colB, uint32_t k0,
                                        uint32_t kn, bool vec) {
  if (vec && kn == (uint32_t)DW_KC) {
#pragma unroll
    for (int i = 0; i < CSR_TN * (DW_KC / 4) / DW_THREADS; ++i) {
      const uint32_t p = threadIdx.x + i * DW_THREADS;
      const uint32_t col = p / (DW_KC / 4), q = p % (DW_KC / 4);
      const size_t off = colB[col];
      const bool ok = off != ~(size_t)0;
      cp_async_16(buf + col * DW_PITCH + q * 4, P.B + (ok ? off + k0 + q * 4 : 0), ok);
    }
  } else {
    for (uint32_t idx = threadIdx.x; idx < (uint32_t)(CSR_TN * DW_KC); idx += DW_THREADS) {
      const uint32_t col = idx / DW_KC, kk = idx % DW_KC;
      const size_t off = colB[col];
      buf[col * DW_PITCH + kk] = (off != ~(size_t)0 && kk < kn) ? __ldg(P.B + off + k0 + kk) : 0.f;
    }
  }
}

// packed fp32 pairs (sm_100 FFMA2): a three-register FFMA issues every other cycle per scheduler, so the FP32
// peak is only reachable two FMAs per instruction
__device__ __forceinline__ unsigned long long pack2(float lo, float hi) {
  unsigned long long r;
  asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(lo), "f"(hi));
  return r;
}
__device__ __forceinline__ void unpack2(unsigned long long v, float& lo, float& hi) {
  asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ void fma2(unsigned long long& d, unsigned long long a, unsigned long long b) {
  asm("fma.rn.f32x2 %0, %1, %2, %0;" : "+l"(d) : "l"(a), "l"(b));
}

// A strip of a warp: sA[k][RPW rows], the 4-row chunks of a k rotated by k / 2 so that the entries of one row
// (what a scatter request holds) spread over eight banks instead of two; the multiply undoes the rotation
// statically (two q per trip)
template <int RPW>
__device__ __forceinline__ uint32_t dw_a_slot(uint32_t kk, int r) {
  constexpr uint32_t NCH = RPW / 4;
  return kk * RPW + ((((uint32_t)r >> 2) + (kk >> 1)) & (NCH - 1)) * 4 + ((uint32_t)r & 3u);
}

template <int RPW, bool BELL>
__global__ void __launch_bounds__(DW_THREADS, 1)
spmm_dense_walk_kernel(const __grid_constant__ CsrSpmmParams P) {
  constexpr int TM = DW_WARPS * RPW;
  extern __shared__ __align__(16) float smem_f[];
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (P.gate && (*P.gate != 0) != (P.gate_run_if != 0)) return;  // another kernel handles this A (device-side choice)
  float* const sB0 = smem_f;                                        // [2][CSR_TN][DW_PITCH]
  float* const sA = smem_f + 2 * CSR_TN * DW_PITCH + warp * RPW * DW_PITCH;  // this warp's strip [DW_KC][RPW]
  size_t* colB = reinterpret_cast<size_t*>(smem_f + 2 * CSR_TN * DW_PITCH + DW_WARPS * 16 * DW_PITCH);  // [CSR_TN]
  size_t* colC = colB + CSR_TN;
  const bool sorted = *P.sorted != 0;
  const uint64_t ncols = BELL ? (uint64_t)P.n : (uint64_t)P.n * P.num_batches;
  const uint32_t tiles = P.row_tiles * P.col_tiles * (BELL ? P.num_batches : 1u);
  const uint32_t nchunks = (P.k + DW_KC - 1) / DW_KC;

  for (uint32_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    const uint32_t rt = tile % P.row_tiles, ct_all = tile / P.row_tiles;
    const uint32_t i0 = rt * TM + warp * RPW;
    const uint32_t batch = BELL ? ct_all / P.col_tiles : 0u;
    const uint32_t ct = BELL ? ct_all - batch * P.col_tiles : ct_all;
    const uint64_t j0 = (uint64_t)ct * CSR_TN;
    float* const Cbase = BELL ? P.Cs[batch] : P.C;

    __syncthreads();  // the previous tile's C stores have left shared memory
    spmm_tile_columns<BELL>(P, j0, ncols, colB, colC);
    __syncthreads();

    uint32_t cur[RPW], end[RPW];
    int32_t pc[RPW];  // first request of every row for the coming chunk (cursor mode)
    float pv[RPW];
    unsigned long long acc2[RPW / 2][CSR_TJ];  // rows (2p, 2p + 1) of column j as one packed pair
#pragma unroll
    for (int r = 0; r < RPW; ++r) {
      const uint32_t row = i0 + r;
      const bool row_ok = row < P.m;
      cur[r] = (!BELL && row_ok) ? (uint32_t)P.row_ptr[row] : 0u;
      end[r] = row_ok ? (BELL ? P.ell_cols : (uint32_t)P.row_ptr[row + 1]) : 0u;
    }
#pragma unroll
    for (int p2 = 0; p2 < RPW / 2; ++p2)
#pragma unroll
      for (int j = 0; j < CSR_TJ; ++j) acc2[p2][j] = 0ull;
#pragma unroll
    for (int r = 0; r < RPW; ++r)
      csr_fetch<BELL>(P, batch, i0 + r, cur[r] + lane, sorted && cur[r] + lane < end[r], pc[r], pv[r]);

    dw_fill(sB0, P, colB, 0, min((uint32_t)DW_KC, P.k), P.vec != 0);
    cp_async_commit();

    for (uint32_t ch = 0; ch < nchunks; ++ch) {
      const uint32_t k0 = ch * DW_KC;
      const uint32_t kn = min((uint32_t)DW_KC, P.k - k0);
      const uint32_t k_end = k0 + kn;
      float* const sB = sB0 + (ch & 1u) * (CSR_TN * DW_PITCH);
      cp_async_wait_all();
      __syncthreads();  // chunk ch has landed for everyone; everyone is done with chunk ch - 1
      if (ch + 1 < nchunks) {
        const uint32_t k1 = k0 + DW_KC;
        dw_fill(sB0 + ((ch + 1) & 1u) * (CSR_TN * DW_PITCH), P, colB, k1, min((uint32_t)DW_KC, P.k - k1), P.vec != 0);
      }
      cp_async_commit();

      // ---- densify this warp's rows of A for k in [k0, k_end) ----
      for (uint32_t i = lane; i < (uint32_t)(RPW * DW_KC / 4); i += 32)
        reinterpret_cast<float4*>(sA)[i] = make_float4(0.f, 0.f, 0.f, 0.f);
      __syncwarp();
      if (sorted) {
        // cursor mode.  The first request of every row was issued before the previous chunk's multiply
        // (pc / pv); further requests of all rows that need one go out together, so a chunk exposes the
        // global-load latency once per round, not once per row.
        unsigned more = 0;
#pragma unroll
        for (int r = 0; r < RPW; ++r) {
          const int32_t c = pc[r];
          if (c < (int32_t)k_end) atomicAdd(sA + dw_a_slot<RPW>((uint32_t)(c - (int32_t)k0), r), pv[r]);  // c >= k0: at/after the cursor
          const unsigned cnt = __popc(__ballot_sync(0xffffffffu, c < (int32_t)k_end));
          cur[r] += cnt;
          if (cnt == 32u) more |= 1u << r;
        }
        while (more) {
          __syncwarp();
#pragma unroll
          for (int r = 0; r < RPW; ++r)
            if (more >> r & 1u) csr_fetch<BELL>(P, batch, i0 + r, cur[r] + lane, cur[r] + lane < end[r], pc[r], pv[r]);
          unsigned again = 0;
#pragma unroll
          for (int r = 0; r < RPW; ++r)
            if (more >> r & 1u) {
              const int32_t c = pc[r];
              if (c < (int32_t)k_end) atomicAdd(sA + dw_a_slot<RPW>((uint32_t)(c - (int32_t)k0), r), pv[r]);
              const unsigned cnt = __popc(__ballot_sync(0xffffffffu, c < (int32_t)k_end));
              cur[r] += cnt;
              if (cnt == 32u) again |= 1u << r;
            }
          more = again;
        }
        if (ch + 1 < nchunks) {
#pragma unroll
          for (int r = 0; r < RPW; ++r)
            csr_fetch<BELL>(P, batch, i0 + r, cur[r] + lane, cur[r] + lane < end[r], pc[r], pv[r]);
        }
      } else {
        // columns in no particular order: every chunk rescans the whole row
#pragma unroll
        for (int r = 0; r < RPW; ++r) {
          const uint32_t beg = (!BELL && i0 + r < P.m) ? (uint32_t)P.row_ptr[i0 + r] : 0u;
          for (uint32_t pos = beg; pos < end[r]; pos += 32u) {
            int32_t c;
            float v;
            csr_fetch<BELL>(P, batch, i0 + r, pos + lane, pos + lane < end[r], c, v);
            if (c >= (int32_t)k0 && c < (int32_t)k_end) atomicAdd(sA + dw_a_slot<RPW>((uint32_t)(c - (int32_t)k0), r), v);
          }
        }
      }
      __syncwarp();

      // ---- multiply.  One k is a rank-1 update of the warp's RPW x 128 block: RPW / 4 broadcast LDS.128 of A
      // (four rows each) against the lane's four columns -- 2 * RPW packed FMAs (row pairs) none of which depends
      // on another;
      // B arrives four k at a time (one LDS.128 per column).  k in [kn, 96) is zero on both sides. ----
      constexpr int NCH = RPW / 4;
      const float4* a4 = reinterpret_cast<const float4*>(sA);
      const float4* b4 = reinterpret_cast<const float4*>(sB) + lane * DW_Q;
      const uint32_t nq = ((kn + 3u) / 4u + 1u) & ~1u;
      for (uint32_t q2 = 0; q2 < nq; q2 += 2) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          const uint32_t q = q2 + h;
          float b[CSR_TJ][4];
#pragma unroll
          for (int j = 0; j < CSR_TJ; ++j) {
            const float4 t = b4[j * 32 * DW_Q + q];
            b[j][0] = t.x; b[j][1] = t.y; b[j][2] = t.z; b[j][3] = t.w;
          }
#pragma unroll
          for (int c = 0; c < 4; ++c) {
            const int rot = (2 * h + (c >> 1)) & (NCH - 1);  // = ((4q + c) / 2) mod NCH, q2 being even
            unsigned long long ap[RPW / 2], bb[CSR_TJ];
#pragma unroll
            for (int g = 0; g < NCH; ++g) {
              const float4 t = a4[(q * 4 + c) * NCH + ((g + rot) & (NCH - 1))];
              ap[2 * g] = pack2(t.x, t.y);
              ap[2 * g + 1] = pack2(t.z, t.w);
            }
#pragma unroll
            for (int j = 0; j < CSR_TJ; ++j) bb[j] = pack2(b[j][c], b[j][c]);
#pragma unroll
            for (int p2 = 0; p2 < RPW / 2; ++p2)
#pragma unroll
              for (int j = 0; j < CSR_TJ; ++j) fma2(acc2[p2][j], ap[p2], bb[j]);
          }
        }
      }
    }

    // ---- C tile through shared memory: sC[column][row], stores run along rows ----
    __syncthreads();
    float* sC = smem_f;  // [CSR_TN][TM + 1] <= the two B buffers
#pragma unroll
    for (int p2 = 0; p2 < RPW / 2; ++p2)
#pragma unroll
      for (int j = 0; j < CSR_TJ; ++j) {
        float lo, hi;
        unpack2(acc2[p2][j], lo, hi);
        sC[(lane + 32 * j) * (TM + 1) + warp * RPW + 2 * p2] = lo;
        sC[(lane + 32 * j) * (TM + 1) + warp * RPW + 2 * p2 + 1] = hi;
      }
    __syncthreads();
    spmm_store_c_tile<TM, DW_THREADS>(P, Cbase, sC, colC, rt * TM);
  }
}

template <int RPW, bool BELL>
int launch_spmm_dense_walk(const CsrSpmmParams& P, int sm_count, cudaStream_t s) {
  const size_t smem = ((size_t)2 * CSR_TN * DW_PITCH + (size_t)DW_WARPS * 16 * DW_PITCH) * 4 + 2 * CSR_TN * sizeof(size_t);
  int rc = allow_dynamic_smem<spmm_dense_walk_kernel<RPW, BELL>>(smem);
  if (rc) return rc;
  const uint32_t tiles = P.row_tiles * P.col_tiles * (BELL ? P.num_batches : 1u);
  const uint32_t grid = tiles < (uint32_t)sm_count ? tiles : (uint32_t)sm_count;
  spmm_dense_walk_kernel<RPW, BELL><<<grid, DW_THREADS, smem, s>>>(P);
  SPFY_LAUNCH_OK("spmm_dense_walk_kernel");
  return SPFY_OK;
}

// fraction of non-zeros from which the dense walk is used (SPFY_SPMM_WALK_DENSITY; > 1 disables it)
double walk_density() {
  static const double d = [] {
    const char* e = dev_switch("SPFY_SPMM_WALK_DENSITY");
    return e ? atof(e) : 0.35;  // measured crossover: M=256 K=2304 at 30 % non-zeros, M=64 K=576 at 40 % (profiles/r01_summary.md)
  }();
  return d;
}

template <int RPW, int MODE>
int launch_spmm_csr(const CsrSpmmParams& P, int sm_count, cudaStream_t s) {
  constexpr bool BELL = MODE != SPMM_CSR;
  size_t smem = ((size_t)CSR_TN * CSR_PITCH_PAIRS) * 4;  // >= the C tile [CSR_TN][TM + 1] for TM <= 128
  smem += (size_t)CSR_SCRATCH_FLOATS * 4 + 2 * CSR_TN * sizeof(size_t);  // scratch lines + column offsets
  int rc = allow_dynamic_smem<spmm_csr_kernel<RPW, MODE>>(smem);
  if (rc) return rc;
  const uint32_t tiles = P.row_tiles * P.col_tiles * (BELL ? P.num_batches : 1u);
  const uint32_t grid = tiles < (uint32_t)sm_count ? tiles : (uint32_t)sm_count;
  spmm_csr_kernel<RPW, MODE><<<grid, CSR_THREADS, smem, s>>>(P);
  SPFY_LAUNCH_OK("spmm_csr_kernel");
  return SPFY_OK;
}

// ------------------------------------------------------------------------
// Tensor-core route of the unstructured SpMMs.  A ResNet weight matrix with 5-50 % non-zeros is far too dense to
// beat a dense contraction by skipping zeros on CUDA cores: one shared-memory wavefront per FMA (the per-non-zero
// kernel) or the fp32 pipe (the dense walk) cap at 7-13 TFLOP/s, whereas the dense 3xTF32 GEMM of gemm_sm100.cu
// runs the whole M x K at fp32-level accuracy at a few hundred.  So the sparse operand is scattered into a dense
// K-major matrix in the workspace (zero-filled; duplicates add, like cuSPARSE) and contracted on tcgen05.
// ------------------------------------------------------------------------
__global__ void __launch_bounds__(256)
coo_scatter_kernel(const int32_t* __restrict__ rows, const int32_t* __restrict__ cols, const float* __restrict__ vals,
                   size_t nnz, uint32_t m, uint32_t k, float* __restrict__ D, size_t ld) {
  const size_t nthreads = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < nnz; i += nthreads) {
    const uint32_t r = (uint32_t)rows[i], c = (uint32_t)cols[i];
    if (r < m && c < k) atomicAdd(D + (size_t)r * ld + c, vals[i]);
  }
}

__global__ void __launch_bounds__(256)
csr_scatter_kernel(const int32_t* __restrict__ row_ptr, const int32_t* __restrict__ cols, const float* __restrict__ vals,
                   uint32_t m, uint32_t k, float* __restrict__ D, size_t ld) {
  const uint32_t lane = threadIdx.x & 31, warps = (gridDim.x * blockDim.x) >> 5;
  for (uint32_t r = (blockIdx.x * blockDim.x + threadIdx.x) >> 5; r < m; r += warps) {
    const int32_t b = row_ptr[r], e = row_ptr[r + 1];
    for (int32_t i = b + (int32_t)lane; i < e; i += 32) {
      const uint32_t c = (uint32_t)cols[i];
      if (c < k) atomicAdd(D + (size_t)r * ld + c, vals[i]);
    }
  }
}

// blocked-ELL -> dense for `nbatch` matrices starting at batch `b0`, gather form: a warp owns one block-row.  It
// first inverts the block-row's id list into shared memory (inv[block column] = position in the list, -1 = absent),
// then writes all `block` dense rows left to right -- every dense element is written exactly once (zeros included),
// so the target needs no memset and no atomics, and both the value reads (ids usually ascend) and the writes are
// coalesced.  ids < 0 are padding, ids beyond the matrix are ignored.  A repeated id in one block-row (cuSPARSE
// leaves that undefined; our CUDA-core kernel and the oracle add the blocks) cannot be expressed this way: it
// raises *dup, and the caller's gated launches then let the CUDA-core kernel do the work instead.
template <typename T>
__global__ void __launch_bounds__(256)
bell_expand_kernel(const int64_t* const* __restrict__ col_ptrs, const void* const* __restrict__ val_ptrs, uint32_t b0,
                   uint32_t nbatch, uint32_t rows, uint32_t cols, uint32_t ell_cols, uint32_t block, uint32_t bcols,
                   uint32_t block_rows, uint32_t nbc, T* __restrict__ D, size_t ld, size_t stride, int* __restrict__ dup) {
  extern __shared__ int32_t bell_inv[];
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  int32_t* inv = bell_inv + (size_t)warp * nbc;
  const size_t items = (size_t)nbatch * block_rows;
  const size_t nwarps = (size_t)gridDim.x * (blockDim.x >> 5);
  bool saw_dup = false;
  // pairs of elements per lane when a pair can never straddle a block or an alignment boundary
  const bool pairs = sizeof(T) <= 4 && block % 2 == 0 && ell_cols % 2 == 0 && ld % 2 == 0;
  for (size_t item = (size_t)blockIdx.x * (blockDim.x >> 5) + warp; item < items; item += nwarps) {
    const uint32_t b = (uint32_t)(item / block_rows), br = (uint32_t)(item - (size_t)b * block_rows);
    for (uint32_t c = lane; c < nbc; c += 32) inv[c] = -1;
    __syncwarp();
    const int64_t* ids = col_ptrs[b0 + b] + (size_t)br * bcols;
    for (uint32_t j = lane; j < bcols; j += 32) {
      const int64_t id = ids[j];
      if (id >= 0 && id < (int64_t)nbc) saw_dup |= atomicExch(&inv[id], (int32_t)j) != -1;
    }
    __syncwarp();
    const T* vals = reinterpret_cast<const T*>(val_ptrs[b0 + b]);
    T* out = D + (size_t)b * stride;
    for (uint32_t r = 0; r < block; ++r) {
      const uint32_t row = br * block + r;
      if (row >= rows) break;
      const T* src = vals + (size_t)row * ell_cols;
      T* dst = out + (size_t)row * ld;
      uint32_t done = 0;
      if (pairs) {
        using P2 = typename std::conditional<sizeof(T) == 4, float2, uint32_t>::type;
        const uint32_t npairs = cols / 2;
        for (uint32_t i = lane; i < npairs; i += 32) {
          const uint32_t c = 2 * i;
          const int32_t j = inv[c / block];
          P2 v;
          memset(&v, 0, sizeof(v));
          if (j >= 0) v = *reinterpret_cast<const P2*>(src + (size_t)j * block + c % block);
          *reinterpret_cast<P2*>(dst + c) = v;
        }
        done = npairs * 2;
      }
      for (uint32_t c = done + lane; c < cols; c += 32) {
        const int32_t j = inv[c / block];
        T v;
        memset(&v, 0, sizeof(v));
        if (j >= 0) v = src[(size_t)j * block + c % block];
        dst[c] = v;
      }
    }
    __syncwarp();
  }
  if (__any_sync(0xffffffffu, saw_dup) && lane == 0) atomicExch(dup, 1);
}

// (one signature for every T, so that the caller can pick the instance by dtype)
template <typename T>
int launch_bell_expand(int grid, size_t inv_bytes, cudaStream_t s, const int64_t* const* col_ptrs, const void* const* val_ptrs,
                       uint32_t b0, uint32_t nbatch, uint32_t rows, uint32_t cols, uint32_t ell_cols, uint32_t block,
                       uint32_t bcols, uint32_t block_rows, uint32_t nbc, void* D, size_t ld, size_t stride, int* dup) {
  if (inv_bytes > 48 * 1024) {
    int rc = allow_dynamic_smem<bell_expand_kernel<T>>(200 * 1024);
    if (rc) return rc;
  }
  bell_expand_kernel<T><<<grid, 256, inv_bytes, s>>>(col_ptrs, val_ptrs, b0, nbatch, rows, cols, ell_cols, block, bcols,
                                                    block_rows, nbc, (T*)D, ld, stride, dup);
  SPFY_LAUNCH_OK("bell_expand_kernel");
  return SPFY_OK;
}

// density of non-zeros from which the tensor-core route is taken when the caller leaves the choice to the library:
// dense 3xTF32 issues 3 x 2MKN tensor FLOPs at several hundred TFLOP/s, the per-non-zero kernel 2*nnz*N at ~7
double tensor_density() {
  static const double d = [] {
    const char* e = dev_switch("SPFY_SPMM_TENSOR_DENSITY");
    return e ? atof(e) : 0.02;
  }();
  return d;
}

size_t dense_ld(size_t k, size_t elem) { return round_up(k, 16 / elem); }  // TMA: row pitch multiple of 16 bytes

constexpr size_t SPMM_FLAG_BYTES = 256;  // device words: [0] columns sorted, [1] dense-walk / tensor route, [2] dup ids

size_t spmm_base_ws(size_t m) { return round_up((m + 1) * 4, 256) + SPMM_FLAG_BYTES; }

// C_b[m x n] = alpha * A[m x k] * B_b[k x n] + beta * C_b with A given densely (row-major, pitch ld): the batches
// are folded into the column dimension when the slabs are contiguous, so that a 196-column image does not leave a
// quarter of every 128-row tile empty.
TcGemmProblem coo_dense_problem(const float* dense, size_t ld, size_t m, size_t k, size_t n, size_t nb,
                                const float* B, size_t ldb, size_t strideB, float* C, size_t ldc, size_t strideC,
                                float alpha, float beta) {
  TcGemmProblem p;
  p.opA = SPFY_OP_T;  // the row-major m x k dense matrix is a column-major k x m one
  p.opB = SPFY_OP_N;
  p.m = m; p.k = k;
  p.A = dense; p.lda = ld; p.strideA = 0;
  p.B = B; p.ldb = ldb;
  p.C = C; p.ldc = ldc;
  p.alpha = alpha; p.beta = beta;
  if (nb > 1 && strideB == ldb * n && strideC == ldc * n) {
    p.n = n * nb; p.nb = 1;
  } else {
    p.n = n; p.nb = nb; p.strideB = strideB; p.strideC = strideC;
  }
  return p;
}

template <typename T>
int threshold_impl(const void* in, size_t ld, size_t rows, size_t cols, float thr, int32_t* row_idx,
                   int32_t* col_idx, float* vals, size_t capacity, int64_t* d_nnz,
                   int32_t* row_ptr, unsigned long long* status, size_t status_bytes, cudaStream_t s) {
  const size_t chunks = ceil_div(rows * cols, (size_t)TC_CHUNK);
  SPFY_CUDA_OK(cudaMemsetAsync(status, 0, status_bytes, s));
  const int vec = cols % 4 == 0 && ld % 4 == 0 && (uintptr_t)in % (4 * sizeof(T)) == 0;
  uint32_t div_mul = 0, div_shift = 0;
  if (cols > 1) {
    uint32_t l = 0;
    while ((1ull << l) < cols) ++l;  // ceil(log2 cols) >= 1
    div_mul = (uint32_t)((1ull << (31 + l)) / cols + 1);
    div_shift = l - 1;
  }
  threshold_compact_kernel<T><<<(unsigned)chunks, TC_THREADS, 0, s>>>((const T*)in, ld, (uint32_t)rows, (uint32_t)cols,
                                                                     div_mul, div_shift, thr, vec, (uint32_t)chunks, row_idx,
                                                                     col_idx, vals, capacity, row_ptr, d_nnz, status);
  SPFY_LAUNCH_OK("threshold_compact_kernel");
  return SPFY_OK;
}

}  // namespace
}  // namespace spfy

void spfy::warm_spmm_kernels() {
  touch_kernel(threshold_compact_kernel<float>);
  touch_kernel(threshold_compact_kernel<__half>);
  touch_kernel(threshold_compact_kernel<__nv_bfloat16>);
  touch_kernel(coo_to_csr_kernel);
  touch_kernel(csr_check_sorted_kernel);
  touch_kernel(bell_check_sorted_kernel);
  touch_kernel(spmm_csr_kernel<4, SPMM_CSR>);
  touch_kernel(spmm_csr_kernel<8, SPMM_CSR>);
  touch_kernel(spmm_csr_kernel<4, SPMM_BELL>);
  touch_kernel(spmm_csr_kernel<8, SPMM_BELL>);
  touch_kernel(spmm_csr_kernel<4, SPMM_BELL_PAIRS>);
  touch_kernel(spmm_csr_kernel<8, SPMM_BELL_PAIRS>);
  touch_kernel(spmm_dense_walk_kernel<8, false>);
  touch_kernel(spmm_dense_walk_kernel<16, false>);
  touch_kernel(coo_scatter_kernel);
  touch_kernel(csr_scatter_kernel);
  touch_kernel(bell_expand_kernel<float>);
  touch_kernel(bell_expand_kernel<__half>);
  touch_kernel(bell_expand_kernel<__nv_bfloat16>);
}

using namespace spfy;

extern "C" {

int spfy_threshold_workspace_bytes(size_t rows, size_t cols, size_t* bytes) {
  // one 64-bit scan word per 4096-element chunk
  if (bytes) *bytes = round_up(ceil_div(rows * cols, (size_t)TC_CHUNK) * 8 + 8, 256);
  return SPFY_OK;
}

int spfy_threshold_to_coo(int dtype, const void* in, size_t ld_in, size_t rows, size_t cols,
                          float threshold, int32_t* row_idx, int32_t* col_idx, float* vals,
                          size_t capacity, int64_t* d_nnz, int32_t* d_row_ptr_or_null,
                          void* workspace, size_t workspace_bytes, spfy_stream_t stream) {
  if (!in || !row_idx || !col_idx || !vals || !d_nnz)
    return fail(SPFY_E_INVALID, "threshold_to_coo: null pointer");
  if (ld_in < cols) return fail(SPFY_E_INVALID, "threshold_to_coo: ld < cols");
  if (rows >= (1ull << 31) || cols >= (1ull << 31) || rows * cols >= (1ull << 31))
    return fail(SPFY_E_UNSUPPORTED, "threshold_to_coo: matrix too large for int32 offsets");
  size_t need = 0;
  spfy_threshold_workspace_bytes(rows, cols, &need);
  if (!workspace || workspace_bytes < need)
    return fail(SPFY_E_WORKSPACE, "threshold_to_coo: workspace %zu < %zu bytes", workspace_bytes, need);
  cudaStream_t s = (cudaStream_t)stream;
  unsigned long long* status = (unsigned long long*)workspace;
  int32_t* row_ptr = d_row_ptr_or_null;
  if ((uintptr_t)workspace % 8) return fail(SPFY_E_INVALID, "threshold_to_coo: workspace must be 8-byte aligned");
  if (rows == 0 || cols == 0) {
    SPFY_CUDA_OK(cudaMemsetAsync(d_nnz, 0, sizeof(int64_t), s));
    if (d_row_ptr_or_null) SPFY_CUDA_OK(cudaMemsetAsync(d_row_ptr_or_null, 0, (rows + 1) * 4, s));
    return SPFY_OK;
  }
  switch (dtype) {
    case SPFY_F32: return threshold_impl<float>(in, ld_in, rows, cols, threshold, row_idx, col_idx, vals, capacity, d_nnz, row_ptr, status, need, s);
    case SPFY_F16: return threshold_impl<__half>(in, ld_in, rows, cols, threshold, row_idx, col_idx, vals, capacity, d_nnz, row_ptr, status, need, s);
    case SPFY_BF16: return threshold_impl<__nv_bfloat16>(in, ld_in, rows, cols, threshold, row_idx, col_idx, vals, capacity, d_nnz, row_ptr, status, need, s);
    default: return fail(SPFY_E_UNSUPPORTED, "threshold_to_coo: dtype %d", dtype);
  }
}

int spfy_coo_to_csr(const int32_t* row_idx, size_t nnz, size_t rows, int32_t* row_ptr,
                    spfy_stream_t stream) {
  if ((!row_idx && nnz) || !row_ptr) return fail(SPFY_E_INVALID, "coo_to_csr: null pointer");
  if (nnz >= (1ull << 31) || rows >= (1ull << 31)) return fail(SPFY_E_UNSUPPORTED, "coo_to_csr: too large");
  int grid = 1;
  int rc = capped_grid(ceil_div(nnz + 1, 256), 8, &grid);
  if (rc) return rc;
  coo_to_csr_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(row_idx, nnz, (uint32_t)rows, row_ptr);
  SPFY_LAUNCH_OK("coo_to_csr_kernel");
  return SPFY_OK;
}

static bool alg_ok(int alg) { return alg >= SPFY_SPMM_ALG_DEFAULT && alg <= SPFY_SPMM_ALG_TENSOR_FAST; }
static bool alg_may_use_tensor(int alg) { return alg != SPFY_SPMM_ALG_CUDA_CORE; }

// padded copy of all B_b when their leading dimension is not a multiple of 16 bytes (k = 147: the first conv layer)
static size_t spmm_repack_ws(size_t k, size_t n, size_t num_batches) {
  return k % 4 ? 512 + round_up(num_batches * n * dense_ld(k, 4) * sizeof(float), 256) : 0;
}

int spfy_spmm_workspace_bytes(int alg, size_t m, size_t k, size_t n, size_t num_batches, size_t nnz, size_t* bytes) {
  (void)nnz;
  if (!alg_ok(alg)) return fail(SPFY_E_INVALID, "spmm_workspace_bytes: bad algorithm %d", alg);
  // row_ptr (COO entry) + the device flag words (+ the dense fp32 image of A for the tensor-core route, + the padded
  // copy of B when ldb = k is not TMA-addressable)
  size_t need = spmm_base_ws(m);
  if (alg_may_use_tensor(alg)) need += round_up(m * dense_ld(k, 4) * sizeof(float), 256) + spmm_repack_ws(k, n, num_batches);
  if (bytes) *bytes = need;
  return SPFY_OK;
}

// nnz_host < 0: the host does not know nnz (CSR entry) -- every candidate kernel is launched and device flags let one run
static int spmm_csr_impl(int alg, size_t m, size_t k, size_t n, size_t num_batches,
                         const int32_t* row_ptr, const int32_t* col_idx, const float* vals,
                         const float* B, size_t ldb, size_t strideB, float* C, size_t ldc,
                         size_t strideC, float alpha, float beta, void* workspace,
                         size_t workspace_bytes, spfy_stream_t stream, long long nnz_host,
                         const int32_t* coo_rows) {
  if (!alg_ok(alg)) return fail(SPFY_E_INVALID, "spmm_csr: bad algorithm %d", alg);
  if (m == 0 || n == 0 || num_batches == 0) return SPFY_OK;
  if (!row_ptr || !B || !C) return fail(SPFY_E_INVALID, "spmm_csr: null pointer");
  const size_t base = spmm_base_ws(m);
  if (!workspace || workspace_bytes < base)
    return fail(SPFY_E_WORKSPACE, "spmm_csr: workspace %zu < %zu bytes", workspace_bytes, base);
  if (ldb < k || ldc < m) return fail(SPFY_E_INVALID, "spmm_csr: leading dimension too small");
  if (m >= (1ull << 31) || n >= (1ull << 31) || k >= (1ull << 31))
    return fail(SPFY_E_UNSUPPORTED, "spmm_csr: dimension too large");
  if (m * 1ull >= (1ull << 31) || (unsigned long long)n * num_batches >= (1ull << 40))
    return fail(SPFY_E_UNSUPPORTED, "spmm_csr: problem too large");
  DeviceInfo di;
  int rc = device_info(&di);
  if (rc) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  int* d_sorted = (int*)((uint8_t*)workspace + base - SPMM_FLAG_BYTES);
  int* d_dense = d_sorted + 1;  // 1 -> the dense route (tensor cores, else the CUDA-core dense walk) handles this A

  // ---- tensor-core route: scatter A into a dense fp32 matrix and contract with 3xTF32 (or one TF32 product) ----
  const size_t ld = dense_ld(k, 4);
  const size_t dense_bytes = round_up(m * ld * sizeof(float), 256);
  float* dense = reinterpret_cast<float*>((uint8_t*)workspace + base);
  TcGemmProblem gp = coo_dense_problem(dense, ld, m, k, n, num_batches, B, ldb, strideB, C, ldc, strideC, alpha, beta);
  bool tensor = false, repack = false;
  size_t gemm_ws_bytes = 0;
  if (alg_may_use_tensor(alg)) {
    const bool forced = alg != SPFY_SPMM_ALG_DEFAULT;
    int trc = workspace_bytes >= base + dense_bytes ? tc_gemm_supported(SPFY_F32, gp, false)
                                                    : fail(SPFY_E_WORKSPACE, "spmm_csr: workspace %zu < %zu bytes for the "
                                                           "tensor-core route", workspace_bytes, base + dense_bytes);
    if (trc == SPFY_E_UNSUPPORTED && tc_gemm_supported(SPFY_F32, gp, true) == SPFY_OK) {
      // B_b is not TMA-addressable as given (ldb = k = 147 floats): the GEMM can run on a padded copy, one extra pass
      // over all of B -- taken when the caller sized the workspace for it (and, if the choice is ours, only for an A
      // dense enough that the CUDA-core kernels lose by more than that pass: 20 % non-zeros)
      gemm_ws_bytes = tc_gemm_workspace_bytes(SPFY_F32, &gp, 1);
      if (workspace_bytes >= base + dense_bytes + gemm_ws_bytes + 256) {
        trc = SPFY_OK;
        repack = true;
      } else {
        trc = fail(SPFY_E_WORKSPACE, "spmm_csr: workspace %zu < %zu bytes for the tensor-core route with a padded copy of B",
                   workspace_bytes, base + dense_bytes + gemm_ws_bytes + 256);
      }
    }
    if (trc != SPFY_OK && forced) return trc;
    tensor = trc == SPFY_OK;
  }
  const double dense_from = tensor ? (alg == SPFY_SPMM_ALG_DEFAULT ? (repack ? 0.2 : tensor_density()) : 0.0) : walk_density();
  const double dense_nnz_f = dense_from * (double)m * (double)k;
  const uint32_t dense_nnz = dense_nnz_f >= 4294967295.0 ? 0xffffffffu : (uint32_t)dense_nnz_f;
  // host-side choice when nnz is known, device-side (flag) otherwise
  const bool host_knows = nnz_host >= 0;
  const bool run_dense = host_knows ? (unsigned long long)nnz_host >= dense_nnz && dense_nnz != 0xffffffffu
                                    : dense_nnz != 0xffffffffu;
  const bool run_sparse = host_knows ? !run_dense : dense_nnz != 0;
  const bool gated = !host_knows && run_dense && run_sparse;

  SPFY_CUDA_OK(cudaMemsetAsync(d_sorted, 0xff, sizeof(int), s));
  if (run_sparse || (run_dense && !tensor)) {
    int grid = 1;
    rc = capped_grid(ceil_div(m * 32, 256), 8, &grid);
    if (rc) return rc;
    csr_check_sorted_kernel<<<grid, 256, 0, s>>>(row_ptr, col_idx, (uint32_t)m, d_sorted, gated ? d_dense : nullptr,
                                                 dense_nnz);
    SPFY_LAUNCH_OK("csr_check_sorted_kernel");
  }
  CsrSpmmParams P;
  memset(&P, 0, sizeof(P));
  P.row_ptr = row_ptr; P.col_idx = col_idx; P.vals = vals;
  P.B = B; P.C = C; P.sorted = d_sorted;
  P.ldb = ldb; P.strideB = strideB; P.ldc = ldc; P.strideC = strideC;
  P.m = (uint32_t)m; P.k = (uint32_t)k; P.n = (uint32_t)n; P.num_batches = (uint32_t)num_batches;
  P.alpha = alpha; P.beta = beta;
  P.vec = ((uintptr_t)B % 16 == 0) && ldb % 4 == 0 && strideB % 4 == 0;
  const size_t total_cols = n * num_batches;
  const size_t col_tiles = ceil_div(total_cols, CSR_TN);
  // 128-row tiles halve the re-staging of B when A has more than 64 rows
  const bool tall = m > 64;
  P.row_tiles = (uint32_t)ceil_div(m, tall ? 128 : 64);
  if (col_tiles * P.row_tiles >= (1ull << 32)) return fail(SPFY_E_UNSUPPORTED, "spmm_csr: too many tiles");
  P.col_tiles = (uint32_t)col_tiles;
  if (run_sparse) {
    P.gate = gated ? d_dense : nullptr;
    P.gate_run_if = 0;
    rc = tall ? launch_spmm_csr<8, SPMM_CSR>(P, di.sm_count, s) : launch_spmm_csr<4, SPMM_CSR>(P, di.sm_count, s);
    if (rc) return rc;
  }
  if (!run_dense) return SPFY_OK;
  if (!tensor) {
    P.gate = gated ? d_dense : nullptr;
    P.gate_run_if = 1;
    return tall ? launch_spmm_dense_walk<16, false>(P, di.sm_count, s) : launch_spmm_dense_walk<8, false>(P, di.sm_count, s);
  }
  // (the memset and the scatter are not gated: a few MB at most, and a sparse A scatters next to nothing)
  SPFY_CUDA_OK(cudaMemsetAsync(dense, 0, m * ld * sizeof(float), s));
  {
    int grid = 1;
    if (coo_rows) {
      rc = capped_grid(ceil_div((size_t)nnz_host, 256), 8, &grid);
      if (rc) return rc;
      if (nnz_host > 0) {
        coo_scatter_kernel<<<grid, 256, 0, s>>>(coo_rows, col_idx, vals, (size_t)nnz_host, (uint32_t)m, (uint32_t)k, dense, ld);
        SPFY_LAUNCH_OK("coo_scatter_kernel");
      }
    } else {
      rc = capped_grid(ceil_div(m * 32, 256), 8, &grid);
      if (rc) return rc;
      csr_scatter_kernel<<<grid, 256, 0, s>>>(row_ptr, col_idx, vals, (uint32_t)m, (uint32_t)k, dense, ld);
      SPFY_LAUNCH_OK("csr_scatter_kernel");
    }
  }
  return tc_gemm_run(SPFY_F32, alg == SPFY_SPMM_ALG_TENSOR_FAST ? TC_GEMM_FAST : TC_GEMM_PRECISE, &gp, 1,
                     repack ? (uint8_t*)workspace + base + dense_bytes : nullptr, repack ? gemm_ws_bytes + 256 : 0, s,
                     gated ? d_dense : nullptr, 1);
}

int spfy_spmm_csr_strided_batched(int alg, size_t m, size_t k, size_t n, size_t num_batches,
                                  const int32_t* row_ptr, const int32_t* col_idx, const float* vals,
                                  const float* B, size_t ldb, size_t strideB, float* C, size_t ldc,
                                  size_t strideC, float alpha, float beta, void* workspace,
                                  size_t workspace_bytes, spfy_stream_t stream) {
  return spmm_csr_impl(alg, m, k, n, num_batches, row_ptr, col_idx, vals, B, ldb, strideB, C, ldc, strideC, alpha, beta,
                       workspace, workspace_bytes, stream, -1, nullptr);
}

int spfy_spmm_coo_strided_batched(int alg, size_t m, size_t k, size_t nnz, size_t n, size_t num_batches,
                                  const int32_t* row_idx, const int32_t* col_idx, const float* vals,
                                  const float* B, size_t ldb, size_t strideB, float* C, size_t ldc,
                                  size_t strideC, float alpha, float beta, void* workspace,
                                  size_t workspace_bytes, spfy_stream_t stream) {
  if (!workspace || workspace_bytes < spmm_base_ws(m))
    return fail(SPFY_E_WORKSPACE, "spmm_coo: workspace %zu < %zu bytes", workspace_bytes, spmm_base_ws(m));
  int rc = spfy_coo_to_csr(row_idx, nnz, m, (int32_t*)workspace, stream);
  if (rc) return rc;
  return spmm_csr_impl(alg, m, k, n, num_batches, (const int32_t*)workspace, col_idx, vals, B, ldb, strideB, C, ldc,
                       strideC, alpha, beta, workspace, workspace_bytes, stream, (long long)nnz, row_idx);
}

// dense images of at most this many bytes are expanded at a time (the batch is processed in chunks)
static const size_t BELL_DENSE_CHUNK_BYTES = (size_t)1 << 30;

// room for the padded copy of the shared B when TMA cannot address it as given (ldb = k = 147), see gemm_sm100.cuh
static size_t bell_gemm_ws(size_t cols, size_t n, size_t es) { return 512 + round_up(n * dense_ld(cols, es) * es, 256); }

int spfy_spmm_bell_workspace_bytes(int alg, int dtype, size_t rows, size_t cols, size_t n, size_t num_batches,
                                   size_t* bytes) {
  if (!alg_ok(alg)) return fail(SPFY_E_INVALID, "spmm_bell_workspace_bytes: bad algorithm %d", alg);
  const size_t es = dtype_bytes(dtype);
  if (es != 2 && es != 4) return fail(SPFY_E_UNSUPPORTED, "spmm_bell_workspace_bytes: dtype %d", dtype);
  size_t need = spmm_base_ws(rows);
  if (alg_may_use_tensor(alg) && rows && cols && num_batches) {
    need += bell_gemm_ws(cols, n, es);
    const size_t mat = round_up(rows * dense_ld(cols, es) * es, 256);
    size_t chunk = BELL_DENSE_CHUNK_BYTES / mat;
    if (chunk < 1) chunk = 1;
    if (chunk > num_batches) chunk = num_batches;
    need += chunk * mat;
  }
  if (bytes) *bytes = need;
  return SPFY_OK;
}

int spfy_spmm_bell_batched(int alg, int dtype, size_t rows, size_t cols, size_t n, size_t block,
                           size_t ell_cols, size_t num_batches, const int64_t* const* col_idx,
                           const void* const* values, const void* B, size_t ldb, void* const* Cs,
                           size_t ldc, float alpha, float beta, void* workspace, size_t workspace_bytes,
                           spfy_stream_t stream) {
  if (!alg_ok(alg)) return fail(SPFY_E_INVALID, "spmm_bell: bad algorithm %d", alg);
  if (rows == 0 || n == 0 || num_batches == 0) return SPFY_OK;
  if (!col_idx || !values || !B || !Cs) return fail(SPFY_E_INVALID, "spmm_bell: null pointer");
  if (block == 0 || ell_cols % block) return fail(SPFY_E_INVALID, "spmm_bell: ell_cols must be a multiple of block");
  if (ldb < cols || ldc < rows) return fail(SPFY_E_INVALID, "spmm_bell: leading dimension too small");
  const size_t es = dtype_bytes(dtype);
  if (es != 2 && es != 4) return fail(SPFY_E_UNSUPPORTED, "spmm_bell: dtype %d", dtype);
  if (rows >= (1ull << 31) || n >= (1ull << 31) || cols >= (1ull << 31) || ell_cols >= (1ull << 31) ||
      num_batches >= (1ull << 31) || ceil_div(rows, 64) * ceil_div(n, CSR_TN) * num_batches >= (1ull << 32))
    return fail(SPFY_E_UNSUPPORTED, "spmm_bell: problem too large");
  const size_t base = spmm_base_ws(rows);
  if (!workspace || workspace_bytes < base)
    return fail(SPFY_E_WORKSPACE, "spmm_bell: workspace %zu < %zu bytes", workspace_bytes, base);
  DeviceInfo di;
  int rc = device_info(&di);
  if (rc) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  int* d_sorted = (int*)((uint8_t*)workspace + base - SPMM_FLAG_BYTES);
  int* d_dup = d_sorted + 2;
  const size_t block_rows = ceil_div(rows, block), bcols = ell_cols / block, nbc = ceil_div(cols, block);

  // ---- tensor-core route: expand a chunk of the batch into dense matrices, contract, next chunk ----
  const size_t ld = dense_ld(cols, es);
  const size_t mat = round_up(rows * ld * es, 256);
  size_t chunk = 0;
  bool tensor = false;
  const size_t inv_bytes = 8 * nbc * sizeof(int32_t);  // 8 warps per CTA, one inverse map each
  const size_t gws = bell_gemm_ws(cols, n, es);
  if (alg_may_use_tensor(alg)) {
    const bool forced = alg != SPFY_SPMM_ALG_DEFAULT;
    chunk = workspace_bytes > base + gws ? (workspace_bytes - base - gws) / mat : 0;
    if (chunk > num_batches) chunk = num_batches;
    TcGemmProblem probe;
    probe.opA = SPFY_OP_T; probe.opB = SPFY_OP_N;
    probe.m = rows; probe.n = n; probe.k = cols; probe.nb = chunk ? chunk : 1;
    probe.A = (uint8_t*)workspace + base + gws; probe.lda = ld; probe.strideA = mat / es;
    probe.B = B; probe.ldb = ldb;
    probe.c_ptrs = Cs; probe.ldc = ldc;
    int trc = chunk ? tc_gemm_supported(dtype, probe, true)
                    : fail(SPFY_E_WORKSPACE, "spmm_bell: workspace %zu < %zu bytes for the tensor-core route",
                           workspace_bytes, base + gws + mat);
    if (trc == SPFY_OK && inv_bytes > 200 * 1024)
      trc = fail(SPFY_E_UNSUPPORTED, "spmm_bell: %zu block columns do not fit the expansion kernel", nbc);
    if (trc != SPFY_OK && forced) return trc;
    tensor = trc == SPFY_OK;
  }

  // CUDA-core launch over batches [b0, b0 + nbatch): the only route (gate == null) or the stand-in for block-rows
  // with repeated ids (gated on *d_dup)
  auto cuda_core = [&](size_t b0, size_t nbatch, const int* gate) -> int {
    if (dtype == SPFY_F32) {
      CsrSpmmParams P;
      memset(&P, 0, sizeof(P));
      P.B = (const float*)B; P.sorted = d_sorted;
      P.ldb = ldb; P.ldc = ldc;
      P.m = (uint32_t)rows; P.k = (uint32_t)cols; P.n = (uint32_t)n; P.num_batches = (uint32_t)nbatch;
      P.alpha = alpha; P.beta = beta;
      P.vec = ((uintptr_t)B % 16 == 0) && ldb % 4 == 0;
      P.bell_cols = col_idx + b0; P.bell_vals = (const float* const*)values + b0; P.Cs = (float* const*)Cs + b0;
      P.block = (uint32_t)block; P.ell_cols = (uint32_t)ell_cols; P.bcols = (uint32_t)bcols;
      P.gate = gate; P.gate_run_if = 1;
      const bool tall = rows > 64;
      P.row_tiles = (uint32_t)ceil_div(rows, tall ? 128 : 64);
      P.col_tiles = (uint32_t)ceil_div(n, CSR_TN);
      if (block % 2 == 0 && ell_cols % 2 == 0 && cols % 2 == 0)
        return tall ? launch_spmm_csr<8, SPMM_BELL_PAIRS>(P, di.sm_count, s)
                    : launch_spmm_csr<4, SPMM_BELL_PAIRS>(P, di.sm_count, s);
      return tall ? launch_spmm_csr<8, SPMM_BELL>(P, di.sm_count, s) : launch_spmm_csr<4, SPMM_BELL>(P, di.sm_count, s);
    }
    // 16-bit values without a tensor-core route (operands that miss the TMA contract, repeated ids): row-split kernel
    SpmmDense D;
    memset(&D, 0, sizeof(D));
    D.B = B; D.C = nullptr; D.Cs = Cs + b0;
    D.ldb = ldb; D.strideB = 0; D.ldc = ldc; D.strideC = 0;
    D.m = (uint32_t)rows; D.k = (uint32_t)cols; D.n = (uint32_t)n; D.num_batches = (uint32_t)nbatch;
    D.alpha = alpha; D.beta = beta;
    D.gate = gate; D.gate_run_if = 1;
    if (dtype == SPFY_F16) {
      BellRows<__half> A{col_idx + b0, (const __half* const*)values + b0, (uint32_t)block, (uint32_t)ell_cols, (uint32_t)bcols};
      return launch_spmm<__half, BellRows<__half>>(A, D, s);
    }
    BellRows<__nv_bfloat16> A{col_idx + b0, (const __nv_bfloat16* const*)values + b0, (uint32_t)block, (uint32_t)ell_cols,
                              (uint32_t)bcols};
    return launch_spmm<__nv_bfloat16, BellRows<__nv_bfloat16>>(A, D, s);
  };

  SPFY_CUDA_OK(cudaMemsetAsync(d_sorted, 0xff, sizeof(int), s));
  SPFY_CUDA_OK(cudaMemsetAsync(d_dup, 0, sizeof(int), s));
  if (bcols > 1 && dtype == SPFY_F32) {
    // (the CUDA-core kernel's cursor mode needs to know whether the ids ascend; cheap next to the values)
    int grid = 1;
    rc = capped_grid(ceil_div(num_batches * block_rows * bcols, 256), 8, &grid);
    if (rc) return rc;
    if (!tensor) {
      bell_check_sorted_kernel<<<grid, 256, 0, s>>>(col_idx, (uint32_t)block_rows, (uint32_t)bcols,
                                                   (uint32_t)num_batches, d_sorted);
      SPFY_LAUNCH_OK("bell_check_sorted_kernel");
    } else {
      SPFY_CUDA_OK(cudaMemsetAsync(d_sorted, 0, sizeof(int), s));  // stand-in launches rescan (always correct)
    }
  }
  if (!tensor) return cuda_core(0, num_batches, nullptr);

  uint8_t* gemm_ws = (uint8_t*)workspace + base;
  uint8_t* dense = gemm_ws + gws;
  const int precision = alg == SPFY_SPMM_ALG_TENSOR_FAST ? TC_GEMM_FAST : TC_GEMM_PRECISE;
  for (size_t b0 = 0; b0 < num_batches; b0 += chunk) {
    const size_t nbatch = std::min(chunk, num_batches - b0);
    int grid = 1;
    rc = capped_grid(ceil_div(nbatch * block_rows, 8), 8, &grid);  // one warp per block row
    if (rc) return rc;
    const auto expand = dtype == SPFY_F32 ? launch_bell_expand<float>
                        : dtype == SPFY_F16 ? launch_bell_expand<__half> : launch_bell_expand<__nv_bfloat16>;
    rc = expand(grid, inv_bytes, s, col_idx, values, (uint32_t)b0, (uint32_t)nbatch, (uint32_t)rows, (uint32_t)cols,
                (uint32_t)ell_cols, (uint32_t)block, (uint32_t)bcols, (uint32_t)block_rows, (uint32_t)nbc, dense, ld, mat / es,
                d_dup);
    if (rc) return rc;
    TcGemmProblem p;
    p.opA = SPFY_OP_T; p.opB = SPFY_OP_N;  // row-major dense A_b = column-major k x m; B is k x n column-major
    p.m = rows; p.n = n; p.k = cols; p.nb = nbatch;
    p.A = dense; p.lda = ld; p.strideA = mat / es;
    p.B = B; p.ldb = ldb; p.strideB = 0;
    p.c_ptrs = Cs + b0; p.ldc = ldc;
    p.alpha = alpha; p.beta = beta;
    rc = tc_gemm_run(dtype, precision, &p, 1, gemm_ws, gws, s, d_dup, 0);
    if (rc) return rc;
    rc = cuda_core(b0, nbatch, d_dup);
    if (rc) return rc;
  }
  return SPFY_OK;
}

}  // extern "C"
