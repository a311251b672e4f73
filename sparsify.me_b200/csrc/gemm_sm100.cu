// gemm_sm100.cu -- dense batched GEMM on tcgen05 (sm_100a): kind::f16 for fp16 / bf16 operands, one kind::tf32
// product for fp32 operands with SPFY_GEMM_FAST, and 3xTF32 at fp32-level accuracy for fp32 operands by default.
//
// Replaces the library contractions of the reference that are dense (or dense enough to be run densely):
//     sparsifyme::batched::gemm          cublas{H,S}gemmBatched          include/sparsify.me/gemm.hxx:25-195
//     sparsifyme::batched::strided_coo   cusparseSpMM COO_ALG4           include/sparsify.me/spmm.hxx:140-193
//     sparsifyme::batched::spmm          cusparseSpMM blocked-ELL        include/sparsify.me/spmm.hxx:30-138
// (the two SpMM entries scatter / expand their sparse operand into a dense one first, spmm.cu), and, as a mode of
// tcgemm_kernel, the split-K weight gradient of a 2:4 convolution (spfy_conv_wgrad24, at the end of the file).
//
// The kernel works in "UMMA terms": D[Mu x Nu] = Au[Mu x K] * Bu[Nu x K]^T with fp32 accumulators in TMEM.  Each
// operand may be K-major (K contiguous) or MN-major (its Mu / Nu dimension contiguous); the result is written
// with either dimension contiguous.  The host maps a column-major BLAS problem onto this so that the long,
// streamed dimension becomes Mu (128-row tiles = TMEM lanes) and the short one becomes Nu (one UMMA of up to 256
// columns), e.g. a weight matrix with 64 rows costs N = 64 MMAs instead of a half-empty M = 128 tile.
//
// Two kernels, both persistent with 1 CTA/SM and work unit = (problem, batch, m-group, n-tile), n-tile fastest so
// that CTAs running side by side share the streamed Au tile through L2:
//
// tcgemm_kernel<KIND>: 16-bit operands, and fp32 operands with SPFY_GEMM_FAST.  192 threads:
//   warp 0      producer : TMA tensor loads of the Au / Bu tiles of one 128-byte K slab per ring stage
//   warp 1      MMA      : per stage 4 k-steps of 32 bytes, one kind::f16 or kind::tf32 MMA each
//   warps 2-5   epilogue : tcgen05.ld 16 columns at a time -> alpha / beta -> coalesced global stores
// TMEM: two accumulator slots of 256 columns, so the epilogue of one unit overlaps the MMAs of the next.
//
// tcgemm_ts_kernel: fp32 operands with SPFY_GEMM_PRECISE (3xTF32, hi*lo + lo*hi + hi*hi).  480 threads; the streamed
// Au tile is split in registers into hi and lo and stored to tensor memory, the MMAs read it from there, and the
// small Bu tile keeps its raw bytes as hi with lo written behind it in shared memory (layout above the kernel).
//
// Accuracy of the 3xTF32 path: Au's hi is x rounded to TF32 (|lo| <= 2^-11 |x|), Bu's hi is x truncated to TF32 by
// the tensor core (|lo| < 2^-10 |x|); the lo*lo term is dropped and each lo is read to TF32 precision, so every
// product is exact to ~2^-19 relative in the worst case, accumulation is fp32.  The parity tests bound the result
// against an fp64 oracle by 4e-6 * sum_k |a||b| (tests/test_gpu_tensor.py).
// Special values: rounding Au's hi carries into the Inf exponent for a finite |x| >= 0x7f7ff000 (the top 2^-11 of the
// fp32 range), so hi = ±Inf, lo = ∓Inf and every output such a value reaches is NaN; Bu's truncated hi stays finite.
// A guard that truncates there instead costs the Au splitters, which bound this kernel, extra instructions per value.
// Measured on a B200 (1000 W limit), old and new builds alternating, three runs each (spread <= 0.011 ms), bench.py
// --workload coo, 14.14 ms per step without a guard:
//   |x| < EDGE ? 0x1000 : 0 added to x (FSETP on |x| + a predicated move, 2 per value)   14.79 ms  (+4.6 %)
//   compare on x << 1 and select (3 per value)                                           15.13 ms  (+7 %)
//   max of |x| over the 16 values of a piece, guarded path only when it reaches EDGE      15.70 ms  (+11 %)
// and the fp32 GEMM sweep of profiling/gemm_timing 4-8 % slower.  So no guard is taken: spfy_b200.h states the range.
// An Inf or NaN operand has lo = NaN on either side: every output it reaches is NaN (tests/test_gpu_fp32_edges.py).
#include "gemm_sm100.cuh"
#include "tc_ptx.cuh"

#include <algorithm>
#include <cmath>
#include <vector>

namespace spfy {
namespace {
using namespace ptx;

constexpr int GM_BM = 128;        // rows of Au per tile (UMMA M)
constexpr int GM_MAX_BN = 256;    // columns of one UMMA / TMEM slot
constexpr int GM_ROW_BYTES = 128; // bytes of K per operand row and stage (one swizzle atom)
constexpr int GM_A_BYTES = GM_BM * GM_ROW_BYTES;
constexpr int GM_THREADS = 192;  // producer, MMA and 4 epilogue warps
constexpr int GM_EPI_WARPS = 4;
constexpr int GM_ACC_SLOTS = 2;
constexpr int GM_MAX_STAGES = 8;
constexpr int GM_SMEM_LIMIT = 232448;
constexpr uint32_t GM_BAR_BYTES = 512;

enum { KIND_F16 = 0, KIND_BF16 = 1, KIND_F32 = 2 };

struct alignas(64) GemmProblemDev {
  CUtensorMap tmap_a;      // Au: {inner, outer, batch}; K-major: inner = K, MN-major: inner = Mu
  CUtensorMap tmap_b;      // Bu likewise
  uint8_t* C;              // batch 0 of the result
  const uint64_t* c_ptrs;  // optional device array of per-batch result pointers
  uint64_t ldc, stride_c;  // elements
  uint32_t mu, nu, k, nb;
  uint32_t m_tiles, n_tiles, k_tiles;
  uint32_t g, m_groups;    // m-tiles per unit (1; 2 in the 3xTF32 kernel when there are two) and units along Mu
  uint32_t bn;             // columns of one n-tile: multiple of 16 (of the MN group when Bu is MN-major)
  uint32_t a_mn, b_mn;     // operand is MN-major
  uint32_t a_batched, b_batched;
  uint32_t out_mu_contig;  // result element (i, j) at i + j*ldc (1) or j + i*ldc (0)
  uint32_t unit_begin, units;
  float alpha, beta;
};

struct GemmLaunch {
  const GemmProblemDev* table;  // null -> the single problem passed by value
  uint32_t num_problems, total_units;
  uint32_t stages, stage_bytes, raw_bytes;  // stage = [Au 16 KiB][Bu bn_max*128]
                                            // (3xTF32 kernel: Bu stage = [raw tile][lo tile], raw_bytes each)
  uint32_t bar_off;
  uint32_t write_hi;  // 3xTF32 kernel (SPFY_GEMM_WRITE_HI, dev builds only): the Bu splitters also store hi = x rounded
                      // to TF32 over the raw tile, instead of leaving the tensor core to truncate it
  uint32_t idesc;     // instruction descriptor without N and the major bits
  uint32_t kelems;    // elements of K per stage (32 fp32 / 64 half)
  const int* gate;    // optional device word: the launch does its work only if (*gate != 0) == gate_run_if
  uint32_t gate_run_if;
  uint32_t dbg;       // development switches (SPFY_GEMM_DEBUG, dev builds only; timing experiments, results are garbage):
                      // 1 no MMAs, 2 no Bu split, 4 no tcgen05.st, 8 no hi/lo arithmetic
  uint32_t a_stages;  // 3xTF32 kernel: depth of the Au ring (raw tiles only; the Bu ring has `stages` slots)
  uint32_t acc_slots, d_cols;  // 3xTF32 kernel: accumulator slots (2 x TS_G x 64 columns, or 1 x TS_G x 128)
  uint32_t b_off;     // ... and where the Bu ring starts
  // weight-gradient mode of tcgemm_kernel (spfy_conv_wgrad24): the convolution behind the im2col map tmap_a
  struct {
    uint32_t c, kw, wo, ho, stride;
    int off_h, off_w;    // base pixel of output position (0, 0): -pad
    uint32_t dn, dh, dw; // one stage = 64 output positions = dn images + dh rows + dw columns
  } wg;
};

// Units are numbered (batch, m-group, n-tile) with the n-tile fastest.  The walker keeps that position incrementally --
// the stride is split once per problem into its (batch, m-group, n-tile) digits -- and reads the problem table only when
// a unit leaves the cached range: five roles decode every unit, and a 32-bit division is ~40 dependent instructions.
struct GemmWalker {
  const GemmProblemDev* single;
  const GemmProblemDev* table;
  uint32_t num_problems, total_units, u, p;
  uint32_t stride;
  uint32_t p_begin, p_end;          // unit range of problem p; p_end == 0: nothing cached yet
  uint32_t n_tiles, m_groups;       // of problem p
  uint32_t nt, md, bb;              // n-tile, m-group and batch of unit u
  uint32_t s_nt, s_md, s_bb;        // the stride in the same digits
  __device__ __forceinline__ GemmWalker(const GemmProblemDev* s, const GemmLaunch& L)
      : single(s), table(L.table), num_problems(L.num_problems), total_units(L.total_units), u(blockIdx.x), p(0),
        stride(gridDim.x), p_begin(0), p_end(0) {}
  __device__ __forceinline__ const GemmProblemDev* prob(uint32_t i) const { return table ? table + i : single; }
  __device__ __forceinline__ bool valid() const { return u < total_units; }
  __device__ __forceinline__ const GemmProblemDev* current() {
    if (u >= p_end) {  // (also the first call)
      while (p + 1 < num_problems && u >= prob(p)->unit_begin + prob(p)->units) ++p;
      p = uni(p);
      const GemmProblemDev* P = prob(p);
      p_begin = uni(P->unit_begin);
      p_end = p_begin + uni(P->units);
      n_tiles = uni(P->n_tiles);
      m_groups = uni(P->m_groups);
      const uint32_t local = u - p_begin, t1 = local / n_tiles, sq = stride / n_tiles;
      nt = local - t1 * n_tiles;
      bb = t1 / m_groups;
      md = t1 - bb * m_groups;
      s_nt = stride - sq * n_tiles;
      s_bb = sq / m_groups;
      s_md = sq - s_bb * m_groups;
    }
    return prob(p);
  }
  __device__ __forceinline__ void next() {
    u += stride;
    nt += s_nt;
    md += s_md;
    bb += s_bb;
    if (nt >= n_tiles) { nt -= n_tiles; ++md; }
    if (md >= m_groups) { md -= m_groups; ++bb; }
  }
};

template <int KIND>
struct OutT { using type = float; };
template <> struct OutT<KIND_F16> { using type = __half; };
template <> struct OutT<KIND_BF16> { using type = __nv_bfloat16; };


// Epilogue role (4 warps: TMEM lane quarter = warp & 3), shared by the two kernels: drains accumulator slot
// job % slots (slot_cols columns apart) of every unit the CTA walks.
// A unit holds g accumulators (m-tiles mg*g ...), tile_cols columns apart inside its slot.
template <int KIND>
__device__ __forceinline__ void gemm_epilogue(GemmWalker& W, uint32_t tmem_base, uint32_t bar_acc_full, uint32_t bar_acc_empty,
                                              uint32_t slots, uint32_t slot_cols, uint32_t tile_cols, uint32_t warp,
                                              uint32_t lane) {
  using out_t = typename OutT<KIND>::type;
  const uint32_t quarter = warp & 3u;  // TMEM lanes [32*quarter, 32*quarter + 32)
  uint32_t job = 0;
  const GemmProblemDev* last = nullptr;
  uint32_t m_tiles = 1, g = 1, bn = 0, mu = 0, nu = 0, mu_contig = 1;
  uint64_t ldc = 0, stride_c = 0;
  uint8_t* Cbase = nullptr;
  const uint64_t* c_ptrs = nullptr;
  float alpha = 1.f, beta = 0.f;
  for (; W.valid(); W.next(), ++job) {
    const GemmProblemDev* P = W.current();
    if (P != last) {
      last = P;
      m_tiles = P->m_tiles; g = P->g; bn = P->bn; mu = P->mu; nu = P->nu;
      mu_contig = P->out_mu_contig; ldc = P->ldc; stride_c = P->stride_c; Cbase = P->C; c_ptrs = P->c_ptrs;
      alpha = P->alpha; beta = P->beta;
    }
    const uint32_t nt = W.nt, mg = W.md, b = W.bb;
    const uint32_t g_count = min(g, m_tiles - mg * g);
    out_t* C = c_ptrs ? reinterpret_cast<out_t*>(c_ptrs[b]) : reinterpret_cast<out_t*>(Cbase) + (size_t)b * stride_c;
    const uint32_t slot = job % slots;
    mbar_wait(bar_acc_full + slot * 8, (job / slots) & 1u);
    tc_fence_after();
    for (uint32_t tile = 0; tile < g_count; ++tile) {
    const uint32_t mt = mg * g + tile;
    const uint32_t row = mt * GM_BM + quarter * 32u + lane;  // index along Mu
    const bool row_ok = row < mu;
    const bool warp_ok = mt * GM_BM + quarter * 32u < mu;
    const uint32_t tcol = tmem_base + slot * slot_cols + tile * tile_cols + ((quarter * 32u) << 16);
    const bool last_tile = tile + 1 == g_count;
    // 16 accumulator columns at a time (bn is a multiple of 16): keeps the role at ~50 registers
    const uint32_t chunks = bn / 16u;
    for (uint32_t c = 0; c < chunks; ++c) {
      const uint32_t col0 = nt * bn + c * 16u;  // index along Nu
      const uint32_t ncols = nu > col0 ? min(16u, nu - col0) : 0u;
      uint32_t acc[16];
      if (warp_ok && ncols) {
        tmem_ld_x16(tcol + c * 16u, acc);
        tmem_wait_ld();
      }
      if (c + 1 == chunks && last_tile) {
        // accumulator fully read by this warp: hand the slot back to the MMA warp
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_acc_empty + slot * 8);
      }
      if (!row_ok || !ncols) continue;
      if (mu_contig) {
        // element (row, col) at row + col*ldc: a warp's 32 rows are one 128-byte (fp32) line per column
        out_t* dst = C + row + (size_t)col0 * ldc;
#pragma unroll
        for (uint32_t j = 0; j < 16; ++j)
          if (j < ncols) {
            float v = alpha * __uint_as_float(acc[j]);
            if (beta != 0.f) v += beta * to_f32(dst[(size_t)j * ldc]);
            dst[(size_t)j * ldc] = from_f32<out_t>(v);
          }
      } else {
        // element (row, col) at col + row*ldc: the thread owns 16 consecutive elements
        out_t* dst = C + (size_t)row * ldc + col0;
        constexpr uint32_t VEC = 16 / sizeof(out_t);  // elements per 16-byte store
        if (ncols == 16u && ((uintptr_t)dst % 16 == 0)) {
#pragma unroll
          for (uint32_t q = 0; q < 16 / VEC; ++q) {
            float v[VEC];
#pragma unroll
            for (uint32_t x = 0; x < VEC; ++x) v[x] = alpha * __uint_as_float(acc[q * VEC + x]);
            if (beta != 0.f) {
              const uint4 old = *reinterpret_cast<const uint4*>(dst + q * VEC);
              const out_t* o = reinterpret_cast<const out_t*>(&old);
#pragma unroll
              for (uint32_t x = 0; x < VEC; ++x) v[x] += beta * to_f32(o[x]);
            }
            uint4 w;
            out_t* wo = reinterpret_cast<out_t*>(&w);
#pragma unroll
            for (uint32_t x = 0; x < VEC; ++x) wo[x] = from_f32<out_t>(v[x]);
            *reinterpret_cast<uint4*>(dst + q * VEC) = w;
          }
        } else {
#pragma unroll
          for (uint32_t j = 0; j < 16; ++j)
            if (j < ncols) {
              float v = alpha * __uint_as_float(acc[j]);
              if (beta != 0.f) v += beta * to_f32(dst[j]);
              dst[j] = from_f32<out_t>(v);
            }
        }
      }
    }
    }  // tile
  }
}

// Producer of tcgemm_kernel's weight-gradient mode (one problem; the unit's batch digit is its split of K)
__device__ __forceinline__ void wgrad_producer(GemmWalker& W, const GemmLaunch& L, uint32_t smem_base, uint32_t bar_full,
                                               uint32_t bar_empty) {
  const uint32_t NS = L.stages;
  const bool leader = elect_one();
  uint32_t stage = 0, phase = 0;
  const GemmProblemDev* P = W.current();  // (one problem)
  if (leader) { prefetch_tmap(&P->tmap_a); prefetch_tmap(&P->tmap_b); }
  const uint32_t mu = uni(P->mu), k_tiles = uni(P->k_tiles), bn = uni(P->bn);
  const uint32_t cc = L.wg.c, kw = L.wg.kw, wo = L.wg.wo, ho = L.wg.ho, str = L.wg.stride;
  const uint32_t dn = L.wg.dn, dh = L.wg.dh, dw = L.wg.dw;
  const int off_h = L.wg.off_h, off_w = L.wg.off_w;
  constexpr uint32_t GROUP_BYTES = 64u * GM_ROW_BYTES;  // one MN group: 64 k-rows (positions) x 64 elements
  for (; W.valid(); W.next()) {
    const uint32_t nt = W.nt, mt = W.md, s = W.bb;
    // the tile's 64-row groups of Mu (mu is a multiple of 64): filter tap and channel offset of each (per unit, so
    // the divisions stay out of the stage loop)
    const uint32_t r0 = mt * (uint32_t)GM_BM, groups = min(2u, (mu - r0) / 64u);
    const uint32_t tap0 = r0 / cc, c0 = r0 - tap0 * cc;
    const uint32_t tap1 = c0 + 64u == cc ? tap0 + 1u : tap0, c1 = c0 + 64u == cc ? 0u : c0 + 64u;
    const uint16_t th0 = (uint16_t)(tap0 / kw), tw0 = (uint16_t)(tap0 - th0 * kw);
    const uint16_t th1 = (uint16_t)(tap1 / kw), tw1 = (uint16_t)(tap1 - th1 * kw);
    // output position of the unit's first stage as (image, row, column), then stepped by 64 positions per stage
    const uint32_t p0 = s * k_tiles * 64u, row = p0 / wo;
    uint32_t w = p0 - row * wo, n = row / ho, h = row - n * ho;
    const uint32_t tx = groups * GROUP_BYTES + bn * (uint32_t)GM_ROW_BYTES;
    for (uint32_t kt = 0; kt < k_tiles; ++kt) {
      mbar_wait(bar_empty + stage * 8, phase ^ 1u);
      const uint32_t full = bar_full + stage * 8;
      const uint32_t sa = smem_base + stage * L.stage_bytes, sb = sa + GM_A_BYTES;
      if (leader) {
        mbar_expect_tx(full, tx);
        const int cw = (int)(w * str) + off_w, ch = (int)(h * str) + off_h;
        tma_load_im2col_4d(sa, &P->tmap_a, (int)c0, cw, ch, (int)n, tw0, th0, full, HINT_EVICT_NORMAL);
        if (groups > 1u)
          tma_load_im2col_4d(sa + GROUP_BYTES, &P->tmap_a, (int)c1, cw, ch, (int)n, tw1, th1, full, HINT_EVICT_NORMAL);
        for (uint32_t g = 0; g * 64u < bn; ++g)
          tma_load_3d(sb + g * GROUP_BYTES, &P->tmap_b, (int)(nt * bn + g * 64u), (int)(p0 + kt * 64u), 0, full,
                      HINT_EVICT_NORMAL);
      }
      w += dw;
      if (w >= wo) { w -= wo; ++h; }
      h += dh;
      if (h >= ho) { h -= ho; ++n; }
      n += dn;
      if (++stage == NS) { stage = 0; phase ^= 1u; }
    }
  }
}

// WGRAD: the weight gradient of a convolution (spfy_conv_wgrad24), a mode that differs from the GEMM in the producer and
// in what the epilogue writes.  Au = im2col(X) (Mu = kh*kw*c in (kh, kw, c) order, MN-major: each 64-row group of a
// tile is one im2col load of 64 output positions x 64 channels at one filter tap), Bu = dY as {m, positions}
// (MN-major), K = output positions.  The batch digit of a unit is its split s of K: k_tiles stages from position
// s * k_tiles * 64 on (the last split runs past the end into zero fill), and the epilogue writes the fp32 partial tile to
// slab s of the workspace (alpha 1, beta 0).  The MMA issuer is the GEMM's.
template <int KIND, bool WGRAD = false>
__global__ void __launch_bounds__(GM_THREADS, 1)
tcgemm_kernel(const __grid_constant__ GemmProblemDev single, const __grid_constant__ GemmLaunch L) {
  using out_t = typename OutT<KIND>::type;
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  // a caller that decides on the device which of two kernels handles a problem launches both (spmm.cu)
  if (L.gate && (*L.gate != 0) != (L.gate_run_if != 0)) return;

  const uint32_t NS = L.stages;
  const uint32_t bar_full = smem_base + L.bar_off;                   // [GM_MAX_STAGES] producer -> MMA
  const uint32_t bar_empty = bar_full + GM_MAX_STAGES * 8;           // [GM_MAX_STAGES] MMA -> producer
  const uint32_t bar_acc_full = bar_empty + GM_MAX_STAGES * 8;       // [GM_ACC_SLOTS]
  const uint32_t bar_acc_empty = bar_acc_full + GM_ACC_SLOTS * 8;    // [GM_ACC_SLOTS]
  const uint32_t tmem_ptr_off = L.bar_off + (2 * GM_MAX_STAGES + 2 * GM_ACC_SLOTS) * 8;
  volatile uint32_t* tmem_ptr_smem = reinterpret_cast<volatile uint32_t*>(smem_gen + tmem_ptr_off);

  if (warp == 1 && lane == 0) {
    for (uint32_t s = 0; s < (uint32_t)GM_MAX_STAGES; ++s) {
      mbar_init(bar_full + s * 8, 1);
      mbar_init(bar_empty + s * 8, 1);
    }
    for (int a = 0; a < GM_ACC_SLOTS; ++a) {
      mbar_init(bar_acc_full + a * 8, 1);
      mbar_init(bar_acc_empty + a * 8, GM_EPI_WARPS);
    }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc(smem_base + tmem_ptr_off, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  GemmWalker W(&single, L);

  if (warp == 0) {
    if constexpr (WGRAD) {
      wgrad_producer(W, L, smem_base, bar_full, bar_empty);
    } else {
      // ===================== producer =====================
      const bool leader = elect_one();
      uint32_t stage = 0, phase = 0;
      const GemmProblemDev* last = nullptr;
      const CUtensorMap *tmap_a = nullptr, *tmap_b = nullptr;
      uint32_t m_tiles = 1, n_tiles = 1, k_tiles = 0, bn = 0, a_mn = 0, b_mn = 0, a_bat = 0, b_bat = 0, unit_begin = 0;
      const uint32_t kel = L.kelems;                      // K elements per stage == k rows of an MN-major slab
      const uint32_t gsz = kel;                           // MN elements per 128-byte group (32 fp32 / 64 half)
      const uint32_t group_bytes = kel * GM_ROW_BYTES;    // one MN group: kel k-rows x 128 bytes
      for (; W.valid(); W.next()) {
        const GemmProblemDev* P = W.current();
        if (P != last) {
          last = P;
          tmap_a = &P->tmap_a; tmap_b = &P->tmap_b;
          if (leader) { prefetch_tmap(tmap_a); prefetch_tmap(tmap_b); }
          m_tiles = uni(P->m_tiles); n_tiles = uni(P->n_tiles); k_tiles = uni(P->k_tiles); bn = uni(P->bn);
          a_mn = uni(P->a_mn); b_mn = uni(P->b_mn); a_bat = uni(P->a_batched); b_bat = uni(P->b_batched);
          unit_begin = uni(P->unit_begin);
        }
        const uint32_t nt = W.nt, mt = W.md, b = W.bb;  // (one m-tile per unit in this kernel: m-group = m-tile)
        const int ba = a_bat ? (int)b : 0, bb = b_bat ? (int)b : 0;
        const uint32_t tx = (uint32_t)GM_A_BYTES + bn * (uint32_t)GM_ROW_BYTES;
        for (uint32_t kt = 0; kt < k_tiles; ++kt) {
          mbar_wait(bar_empty + stage * 8, phase ^ 1u);
          const uint32_t full = bar_full + stage * 8;
          const uint32_t sa = smem_base + stage * L.stage_bytes, sb = sa + GM_A_BYTES;
          if (leader) {
            mbar_expect_tx(full, tx);
            if (!a_mn) {
              tma_load_3d(sa, tmap_a, (int)(kt * kel), (int)(mt * GM_BM), ba, full, HINT_EVICT_NORMAL);
            } else {
              for (uint32_t g = 0; g * gsz < (uint32_t)GM_BM; ++g)
                tma_load_3d(sa + g * group_bytes, tmap_a, (int)(mt * GM_BM + g * gsz), (int)(kt * kel), ba, full,
                            HINT_EVICT_NORMAL);
            }
            if (!b_mn) {
              tma_load_3d(sb, tmap_b, (int)(kt * kel), (int)(nt * bn), bb, full, HINT_EVICT_NORMAL);
            } else {
              for (uint32_t g = 0; g * gsz < bn; ++g)
                tma_load_3d(sb + g * group_bytes, tmap_b, (int)(nt * bn + g * gsz), (int)(kt * kel), bb, full,
                            HINT_EVICT_NORMAL);
            }
          }
          if (++stage == NS) { stage = 0; phase ^= 1u; }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    const bool leader = elect_one();
    const uint32_t tmem_b = uni(tmem_base);
    uint32_t stage = 0, phase = 0, job = 0;
    const GemmProblemDev* last = nullptr;
    uint32_t k_tiles = 0, pk = 0, bn = 0, a_mn = 0, b_mn = 0;
    const uint32_t kel = L.kelems;
    const uint32_t umma_k = kel / 4u;               // K elements per MMA (32 bytes)
    const uint32_t group_bytes = kel * GM_ROW_BYTES;
    // K-major: rows of 128 bytes, 8-row atoms 1024 bytes apart, a k-step advances 32 bytes inside the swizzled row.
    // MN-major: 128-byte groups of MN, 8 k-rows per 1024-byte atom (SBO), groups `group_bytes` apart (LBO); a k-step
    // is umma_k k-rows = umma_k * 128 bytes.
    // 32-bit MN-major operands exist in one shared-memory layout only: 128-byte rows of MN, 4 k-rows per 512-byte atom,
    // 32-byte chunks XOR-ed with (k-row & 3) (TMA: SWIZZLE_128B_ATOM_32B)
    const uint64_t desc_k = make_smem_desc(0, 16, 1024, LAYOUT_SW128);
    const uint64_t desc_mn = KIND == KIND_F32 ? make_smem_desc(0, group_bytes, 512, LAYOUT_SW128_BASE32B)
                                              : make_smem_desc(0, group_bytes, 1024, LAYOUT_SW128);
    const uint32_t step_mn = (umma_k * GM_ROW_BYTES) >> 4;
    for (; W.valid(); W.next()) {
      const GemmProblemDev* P = W.current();
      if (P != last) {
        last = P;
        k_tiles = uni(P->k_tiles); pk = uni(P->k); bn = uni(P->bn); a_mn = uni(P->a_mn); b_mn = uni(P->b_mn);
      }
      const uint32_t slot = job % GM_ACC_SLOTS, use = job / GM_ACC_SLOTS;
      mbar_wait(bar_acc_empty + slot * 8, (use & 1u) ^ 1u);
      tc_fence_after();
      const uint32_t tmem_d = tmem_b + slot * (uint32_t)GM_MAX_BN;
      const uint32_t idesc = L.idesc | (a_mn << 15) | (b_mn << 16) | ((bn >> 3) << 17);
      const uint64_t da_hi = a_mn ? desc_mn : desc_k, db_hi = b_mn ? desc_mn : desc_k;
      const uint32_t a_step = a_mn ? step_mn : 2u, b_step = b_mn ? step_mn : 2u;
      uint32_t k_left = pk;
      for (uint32_t kt = 0; kt < k_tiles; ++kt, k_left -= kel) {
        mbar_wait(bar_full + stage * 8, phase);
        tc_fence_after();
        const uint32_t sa = smem_base + stage * L.stage_bytes;
        const uint32_t a0 = (sa >> 4) & 0x3fffu, b0 = ((sa + GM_A_BYTES) >> 4) & 0x3fffu;
        const uint32_t nk = k_left >= kel ? 4u : (k_left + umma_k - 1u) / umma_k;
        if (leader) {
#pragma unroll
          for (uint32_t j = 0; j < 4; ++j) {
            if (j < nk) {
              const uint64_t da = da_hi | (uint64_t)(a0 + a_step * j), db = db_hi | (uint64_t)(b0 + b_step * j);
              const uint32_t acc = (kt | j) ? 1u : 0u;
              if (KIND == KIND_F32) tc_mma_tf32(tmem_d, da, db, idesc, acc);
              else                  tc_mma_f16(tmem_d, da, db, idesc, acc);
            }
          }
          tc_commit(bar_empty + stage * 8);
        }
        if (++stage == NS) { stage = 0; phase ^= 1u; }
      }
      if (leader) tc_commit(bar_acc_full + slot * 8);
      ++job;
    }
  } else {
    gemm_epilogue<WGRAD ? KIND_F32 : KIND>(W, tmem_base, bar_acc_full, bar_acc_empty, GM_ACC_SLOTS, GM_MAX_BN, GM_MAX_BN, warp,
                                           lane);
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// ------------------------------------------------------------------------------------------------------------
// fp32 operands at fp32-level accuracy (3xTF32) with the streamed operand in TENSOR MEMORY.
//
// With both operands split in shared memory, 3xTF32 is bound by shared-memory bandwidth, not by the
// tensor pipe or HBM: per 32-wide K slab the (128 + N) x 128 bytes of operands are written by TMA, read and
// written twice over by the splitter (hi, lo) and read three times by the MMAs -- 7 passes at 128 B/clk
// (measured: 2000 cycles per slab at N = 64 against 720 for HBM).  Here the splitter warps take the raw Au tile
// out of shared memory ONCE, split it in registers and store hi and lo to tensor memory with tcgen05.st, and the
// MMAs read Au from there (`tcgen05.mma [d], [a_tmem], b_desc`): shared memory carries the raw Au tile once and
// the small Bu tile (weights: raw via TMA, lo written behind it, read by three MMAs per k-step).
//
// What is left is the traffic INTO the SM: a byte costs the same from L2 as from HBM on this part (DESIGN.md 4), and
// the weight tile is fetched again for every 128-row tile of Au.  So a unit covers up to TWO m-tiles (g = 2) that
// share every Bu stage: half the weight traffic and half the splitting work per byte of Au.
//
//   warps 0, 10 producers: two rings with a producer warp each, so that the Au ring (raw tiles of one 32-wide K slab for
//                          the unit's m-tiles, 32 KiB a stage) runs ahead of the 4-deep Bu ring the MMAs release
//   warps 2-5   Au splitters: thread = one row = one TMEM lane, per m-tile 32 values -> hi, lo -> tcgen05.st; the Au stage is
//                          handed back as soon as it has been read
//   warps 11-14 Bu splitters: lo = x - trunc(x) behind the raw tile (the tensor core ignores the low 13 mantissa bits itself)
//   warp 1      MMA      : per m-tile and k-step hi*lo, lo*hi, hi*hi; commits free the Bu stage and the TMEM operand slot
//   warps 6-9   epilogue : as in tcgemm_kernel, one accumulator per m-tile
// TMEM (512 columns): accumulators [0, 256) = slots x 2 m-tiles x (64 or 128) columns -- two slots when every tile of the
// launch has at most 64 columns, else one; Au operand ring [256, 512) = 2 slots x 2 m-tiles x (32 hi + 32 lo).
// An MN-major Au tile is fetched unswizzled (a thread reads its row as 32 conflict-free 4-byte loads); an
// MN-major Bu tile uses the 32B-base swizzle the tensor core requires of 32-bit MN-major operands.
// ------------------------------------------------------------------------------------------------------------
constexpr int TS_MAX_BN = 128;
constexpr int TS_G = 2;                             // m-tiles per unit that share a Bu stage
constexpr int TS_A_COL = 256;                       // first TMEM column of the Au operand ring
constexpr int TS_T_SLOTS = 2;                       // TMEM operand slots (each TS_G x 64 columns)
constexpr int TS_B_STAGES = 4;
constexpr int TS_MAX_A_STAGES = 8;
constexpr int TS_A_STAGE_BYTES = TS_G * GM_A_BYTES; // one K slab of the unit's m-tiles
constexpr int TS_ASPLIT_WARPS = 4;                  // warps 2-5
constexpr int TS_BSPLIT_WARPS = 4;                  // warps 11-14
constexpr int TS_THREADS = (2 + TS_ASPLIT_WARPS + GM_EPI_WARPS + 1 + TS_BSPLIT_WARPS) * 32;  // warps 0-14

// (15 warps: a scheduler holds four of them, so a thread gets at most 16384 / 4 / 32 = 128 registers)
__global__ void __launch_bounds__(TS_THREADS, 1)
tcgemm_ts_kernel(const __grid_constant__ GemmProblemDev single, const __grid_constant__ GemmLaunch L) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  if (L.gate && (*L.gate != 0) != (L.gate_run_if != 0)) return;

  const uint32_t NA = L.a_stages, NB = L.stages;
  const uint32_t bar_afull = smem_base + L.bar_off;                      // [TS_MAX_A_STAGES] producer -> Au splitters
  const uint32_t bar_aempty = bar_afull + TS_MAX_A_STAGES * 8;           // [TS_MAX_A_STAGES] Au splitters -> producer
  const uint32_t bar_bfull = bar_aempty + TS_MAX_A_STAGES * 8;           // [TS_B_STAGES] producer -> Bu splitters
  const uint32_t bar_ready = bar_bfull + TS_B_STAGES * 8;                // [TS_B_STAGES] all splitters -> MMA
  const uint32_t bar_bfree = bar_ready + TS_B_STAGES * 8;                // [TS_B_STAGES] MMA -> Bu producer
  const uint32_t bar_tfree = bar_bfree + TS_B_STAGES * 8;                // [TS_T_SLOTS] MMA -> Au splitters (TMEM operand slot)
  const uint32_t bar_acc_full = bar_tfree + TS_T_SLOTS * 8;              // [2]
  const uint32_t bar_acc_empty = bar_acc_full + 2 * 8;                   // [2]
  const uint32_t tmem_ptr_off = L.bar_off + (2 * TS_MAX_A_STAGES + 3 * TS_B_STAGES + TS_T_SLOTS + 4) * 8;
  volatile uint32_t* tmem_ptr_smem = reinterpret_cast<volatile uint32_t*>(smem_gen + tmem_ptr_off);

  if (warp == 1 && lane == 0) {
    for (uint32_t s = 0; s < (uint32_t)TS_MAX_A_STAGES; ++s) {
      mbar_init(bar_afull + s * 8, 1);
      mbar_init(bar_aempty + s * 8, TS_ASPLIT_WARPS);
    }
    for (uint32_t s = 0; s < (uint32_t)TS_B_STAGES; ++s) {
      mbar_init(bar_bfull + s * 8, 1);
      mbar_init(bar_ready + s * 8, TS_ASPLIT_WARPS + TS_BSPLIT_WARPS);
      mbar_init(bar_bfree + s * 8, 1);
    }
    for (uint32_t s = 0; s < (uint32_t)TS_T_SLOTS; ++s) mbar_init(bar_tfree + s * 8, 1);
    for (int a = 0; a < 2; ++a) {
      mbar_init(bar_acc_full + a * 8, 1);
      mbar_init(bar_acc_empty + a * 8, GM_EPI_WARPS);
    }
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc(smem_base + tmem_ptr_off, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  GemmWalker W(&single, L);
  constexpr uint32_t KEL = 32;                 // fp32 elements of K per slab (128 bytes): one stage of either ring
  constexpr uint32_t GROUP_BYTES = KEL * 128;  // one 32-wide MN group of an MN-major tile

  if (warp == 0) {
    // ===================== Au producer: one stage = one K slab of the unit's m-tiles =====================
    const bool leader = elect_one();
    uint32_t st = 0, ph = 0;
    const GemmProblemDev* last = nullptr;
    const CUtensorMap* tmap = nullptr;
    uint32_t m_tiles = 1, g = 1, k_tiles = 0, mn = 0, bat = 0;
    for (; W.valid(); W.next()) {
      const GemmProblemDev* P = W.current();
      if (P != last) {
        last = P;
        tmap = &P->tmap_a;
        if (leader) prefetch_tmap(tmap);
        m_tiles = uni(P->m_tiles); g = uni(P->g);
        k_tiles = uni(P->k_tiles); mn = uni(P->a_mn); bat = uni(P->a_batched);
      }
      const uint32_t mg = W.md, b = W.bb;
      const uint32_t mt0 = mg * g, g_count = min(g, m_tiles - mt0);
      const int bc = bat ? (int)b : 0;
      for (uint32_t kt = 0; kt < k_tiles; ++kt) {
        mbar_wait(bar_aempty + st * 8, ph ^ 1u);
        const uint32_t full = bar_afull + st * 8, dst = smem_base + st * (uint32_t)TS_A_STAGE_BYTES;
        if (leader) {
          mbar_expect_tx(full, g_count * (uint32_t)GM_A_BYTES);
          for (uint32_t t = 0; t < g_count; ++t) {
            const int row0 = (int)((mt0 + t) * GM_BM);
            const uint32_t d = dst + t * (uint32_t)GM_A_BYTES;
            if (!mn) {
              tma_load_3d(d, tmap, (int)(kt * KEL), row0, bc, full, HINT_EVICT_NORMAL);
            } else {
              // MN-major, unswizzled: four groups of 32 rows, each [32 k-rows][32 rows]; k rows beyond K are zero-filled
              for (uint32_t q = 0; q < 4; ++q)
                tma_load_3d(d + q * GROUP_BYTES, tmap, row0 + (int)(q * KEL), (int)(kt * KEL), bc, full, HINT_EVICT_NORMAL);
            }
          }
        }
        if (++st == NA) { st = 0; ph ^= 1u; }
      }
    }
  } else if (warp == 10) {
    // ===================== Bu producer =====================
    const bool leader = elect_one();
    uint32_t st = 0, ph = 0;
    const GemmProblemDev* last = nullptr;
    const CUtensorMap* tmap = nullptr;
    uint32_t k_tiles = 0, bn = 0, mn = 0, bat = 0;
    for (; W.valid(); W.next()) {
      const GemmProblemDev* P = W.current();
      if (P != last) {
        last = P;
        tmap = &P->tmap_b;
        if (leader) prefetch_tmap(tmap);
        k_tiles = uni(P->k_tiles); bn = uni(P->bn);
        mn = uni(P->b_mn); bat = uni(P->b_batched);
      }
      const uint32_t nt = W.nt, b = W.bb;
      const int bc = bat ? (int)b : 0, row0 = (int)(nt * bn);
      for (uint32_t kt = 0; kt < k_tiles; ++kt) {
        mbar_wait(bar_bfree + st * 8, ph ^ 1u);
        const uint32_t full = bar_bfull + st * 8, dst = smem_base + L.b_off + st * L.stage_bytes;
        if (leader) {
          mbar_expect_tx(full, bn * (uint32_t)GM_ROW_BYTES);
          if (!mn) {
            tma_load_3d(dst, tmap, (int)(kt * KEL), row0, bc, full, HINT_EVICT_LAST);  // re-read by every unit: keep in L2
          } else {
            for (uint32_t q = 0; q * KEL < bn; ++q)
              tma_load_3d(dst + q * GROUP_BYTES, tmap, row0 + (int)(q * KEL), (int)(kt * KEL), bc, full, HINT_EVICT_LAST);
          }
        }
        if (++st == NB) { st = 0; ph ^= 1u; }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    const bool leader = elect_one();
    const uint32_t tmem_b = uni(tmem_base);
    uint32_t sb = 0, phb = 0, slab = 0, job = 0;
    const GemmProblemDev* last = nullptr;
    uint32_t m_tiles = 1, g = 1, k_tiles = 0, pk = 0, bn = 0, b_mn = 0;
    const uint32_t lo_off = L.raw_bytes >> 4;  // Bu lo tile sits raw_bytes behind the raw one (16-byte units)
    const uint64_t desc_k = make_smem_desc(0, 16, 1024, LAYOUT_SW128);
    const uint64_t desc_mn = make_smem_desc(0, GROUP_BYTES, 512, LAYOUT_SW128_BASE32B);
    for (; W.valid(); W.next()) {
      const GemmProblemDev* P = W.current();
      if (P != last) {
        last = P;
        m_tiles = uni(P->m_tiles); g = uni(P->g);
        k_tiles = uni(P->k_tiles); pk = uni(P->k); bn = uni(P->bn); b_mn = uni(P->b_mn);
      }
      const uint32_t mg = W.md;
      const uint32_t g_count = min(g, m_tiles - mg * g);
      const uint32_t slot = job % L.acc_slots, use = job / L.acc_slots;
      mbar_wait(bar_acc_empty + slot * 8, (use & 1u) ^ 1u);
      tc_fence_after();
      const uint32_t tmem_d = tmem_b + slot * (uint32_t)TS_G * L.d_cols;  // m-tile t at + t * d_cols
      const uint32_t idesc = L.idesc | (b_mn << 16) | ((bn >> 3) << 17);  // the A operand in TMEM is K-major by construction
      const uint64_t db_hi = b_mn ? desc_mn : desc_k;
      const uint32_t b_step = b_mn ? (8u * GM_ROW_BYTES) >> 4 : 2u;       // 8 k-rows of 128 bytes / 32 bytes inside the row
      uint32_t k_left = pk;
      for (uint32_t kt = 0; kt < k_tiles; ++kt, k_left -= KEL, ++slab) {
        mbar_wait(bar_ready + sb * 8, phb);
        tc_fence_after();
        const uint32_t b0 = ((smem_base + L.b_off + sb * L.stage_bytes) >> 4) & 0x3fffu;
        const uint32_t ts = slab % TS_T_SLOTS;
        const uint32_t ta = tmem_b + (uint32_t)TS_A_COL + ts * (uint32_t)(TS_G * 64);
        const uint32_t nk = k_left >= KEL ? 4u : (k_left + 7u) / 8u;
        if (leader) {
#pragma unroll
          for (uint32_t t = 0; t < (uint32_t)TS_G; ++t) {
            if (t < g_count && !(L.dbg & 1u)) {
#pragma unroll
              for (uint32_t j = 0; j < 4; ++j) {
                if (j < nk) {
                  const uint64_t db = db_hi | (uint64_t)(b0 + b_step * j);
                  const uint32_t a_hi = ta + t * 64u + 8u * j, a_lo = a_hi + 32u, d = tmem_d + t * L.d_cols;
                  tc_mma_tf32_ts(d, a_hi, db + lo_off, idesc, (kt | j) ? 1u : 0u);  // hi * lo
                  tc_mma_tf32_ts(d, a_lo, db, idesc, 1u);                           // lo * hi
                  tc_mma_tf32_ts(d, a_hi, db, idesc, 1u);                           // hi * hi
                }
              }
            }
          }
          tc_commit(bar_bfree + sb * 8);
          tc_commit(bar_tfree + ts * 8);
        }
        if (++sb == NB) { sb = 0; phb ^= 1u; }
      }
      if (leader) tc_commit(bar_acc_full + slot * 8);
      ++job;
    }
  } else if (warp < 2 + TS_ASPLIT_WARPS) {
    // ===================== Au splitters: thread = one row of a tile = one TMEM lane =====================
    const uint32_t row = (warp & 3u) * 32u + lane;  // the TMEM lane quarter a warp may touch is warp % 4
    uint32_t sa = 0, pha = 0, sb = 0, phb = 0, slab = 0;
    const GemmProblemDev* last = nullptr;
    uint32_t m_tiles = 1, g = 1, k_tiles = 0, a_mn = 0;
    for (; W.valid(); W.next()) {
      const GemmProblemDev* P = W.current();
      if (P != last) {
        last = P;
        m_tiles = P->m_tiles; g = P->g; k_tiles = P->k_tiles; a_mn = P->a_mn;
      }
      const uint32_t mg = W.md;
      const uint32_t g_count = min(g, m_tiles - mg * g);
      for (uint32_t kt = 0; kt < k_tiles; ++kt, ++slab) {
        mbar_wait(bar_afull + sa * 8, pha);
        const uint32_t src = smem_base + sa * (uint32_t)TS_A_STAGE_BYTES;
        const uint32_t ts = slab % TS_T_SLOTS;
        const uint32_t ta = tmem_base + (uint32_t)TS_A_COL + ts * (uint32_t)(TS_G * 64) + (((warp & 3u) * 32u) << 16);
        for (uint32_t t = 0; t < g_count; ++t) {
          // the row in two pieces of 16 values (keeps the working set at 32 registers)
#pragma unroll
          for (uint32_t q = 0; q < 2; ++q) {
            uint32_t x[16], h[16];
            if (!a_mn) {
              // K-major, 128B-swizzled: chunk c of row r at (c ^ (r & 7)) * 16 -- 8 lanes cover all banks
              const uint32_t rbase = src + t * (uint32_t)GM_A_BYTES + row * 128u, sw = row & 7u;
#pragma unroll
              for (uint32_t c = 0; c < 4; ++c) {
                const uint4 v = ld_shared_v4(rbase + (((4u * q + c) ^ sw) << 4));
                x[4 * c] = v.x; x[4 * c + 1] = v.y; x[4 * c + 2] = v.z; x[4 * c + 3] = v.w;
              }
            } else {
              // MN-major, unswizzled groups of 32 rows x 32 k-rows: k-row kk at kk*128, my element at (row % 32) * 4
              const uint32_t rbase = src + t * (uint32_t)GM_A_BYTES + (row >> 5) * GROUP_BYTES + q * 16u * 128u + (row & 31u) * 4u;
#pragma unroll
              for (uint32_t kk = 0; kk < 16; ++kk) x[kk] = ld_shared_u32(rbase + kk * 128u);
            }
            if (q == 1 && t + 1 == g_count) {  // the stage has been read: hand it back before doing anything else
              __syncwarp();
              if (lane == 0) mbar_arrive(bar_aempty + sa * 8);
            }
            // hi = x rounded to the nearest TF32 (the tensor core reads it exactly), lo = x - hi (exact in fp32)
            if (!(L.dbg & 8u)) {
#pragma unroll
              for (int i = 0; i < 16; ++i) h[i] = (x[i] + 0x1000u) & 0xffffe000u;
#pragma unroll
              for (int i = 0; i < 16; ++i) x[i] = __float_as_uint(__uint_as_float(x[i]) - __uint_as_float(h[i]));
            } else {
#pragma unroll
              for (int i = 0; i < 16; ++i) h[i] = x[i];
            }
            if (q == 0 && t == 0) {
              // the TMEM operand slot is free once the MMAs of the slab that used it last have completed
              mbar_wait(bar_tfree + ts * 8, (((slab / TS_T_SLOTS) & 1u) ^ 1u));
              tc_fence_after();
            }
            if (!(L.dbg & 4u)) {
              tmem_st_x16(ta + t * 64u + q * 16u, h);
              tmem_st_x16(ta + t * 64u + 32u + q * 16u, x);
            }
          }
        }
        if (++sa == NA) { sa = 0; pha ^= 1u; }
        if (!(L.dbg & 4u)) tmem_wait_st();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_ready + sb * 8);
        if (++sb == NB) { sb = 0; phb ^= 1u; }
      }
    }
  } else if (warp >= 11) {
    // ===================== Bu splitters: element-wise over the stage (the layout does not matter) =====================
    const uint32_t t = threadIdx.x - 11u * 32u;
    const bool write_hi = L.write_hi != 0;
    uint32_t sb = 0, phb = 0;
    const GemmProblemDev* last = nullptr;
    uint32_t k_tiles = 0, bn = 0;
    const uint32_t raw = L.raw_bytes;
    for (; W.valid(); W.next()) {
      const GemmProblemDev* P = W.current();
      if (P != last) { last = P; k_tiles = P->k_tiles; bn = P->bn; }
      const uint32_t used = (L.dbg & 2u) ? 0u : bn * (uint32_t)GM_ROW_BYTES;
      for (uint32_t kt = 0; kt < k_tiles; ++kt) {
        mbar_wait(bar_bfull + sb * 8, phb);
        const uint32_t sbase = smem_base + L.b_off + sb * L.stage_bytes;
        // four 16-byte pieces per trip, loads first: the trip costs one shared-memory round trip, not four
        constexpr uint32_t STRIDE = TS_BSPLIT_WARPS * 32u * 16u;
        for (uint32_t off = t * 16u; off < used; off += 4u * STRIDE) {
          uint4 v[4];
#pragma unroll
          for (uint32_t u = 0; u < 4; ++u)
            if (off + u * STRIDE < used) v[u] = ld_shared_v4(sbase + off + u * STRIDE);
#pragma unroll
          for (uint32_t u = 0; u < 4; ++u) {
            if (off + u * STRIDE >= used) break;
            // write_hi: hi = x rounded to nearest TF32, stored over the raw tile.  Without it the raw tile stays and the
            // tensor core itself drops the low 13 mantissa bits, so hi = x truncated and lo = x - hi (one store less)
            const uint32_t rnd = write_hi ? 0x1000u : 0u;
            const uint32_t h0 = (v[u].x + rnd) & 0xffffe000u, h1 = (v[u].y + rnd) & 0xffffe000u;
            const uint32_t h2 = (v[u].z + rnd) & 0xffffe000u, h3 = (v[u].w + rnd) & 0xffffe000u;
            const float l0 = __uint_as_float(v[u].x) - __uint_as_float(h0), l1 = __uint_as_float(v[u].y) - __uint_as_float(h1);
            const float l2 = __uint_as_float(v[u].z) - __uint_as_float(h2), l3 = __uint_as_float(v[u].w) - __uint_as_float(h3);
            st_shared_v4(sbase + raw + off + u * STRIDE, __float_as_uint(l0), __float_as_uint(l1), __float_as_uint(l2),
                         __float_as_uint(l3));
            if (write_hi) st_shared_v4(sbase + off + u * STRIDE, h0, h1, h2, h3);
          }
        }
        fence_proxy_async_smem();  // generic-proxy writes of Bu -> visible to the tensor core's async-proxy reads
        __syncwarp();
        if (lane == 0) mbar_arrive(bar_ready + sb * 8);
        if (++sb == NB) { sb = 0; phb ^= 1u; }
      }
    }
  } else {  // warps 6-9
    gemm_epilogue<KIND_F32>(W, tmem_base, bar_acc_full, bar_acc_empty, L.acc_slots, (uint32_t)TS_G * L.d_cols, L.d_cols, warp, lane);
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

// An operand TMA cannot address (base not 16-byte aligned, or a leading dimension / batch stride that is not a
// multiple of 16 bytes -- e.g. ld = k = 147 floats for the first conv layer of every ResNet) is copied once into the
// workspace with its rows padded to 16 bytes.  One thread per element, coalesced along the contiguous dimension.
template <typename T>
__global__ void __launch_bounds__(256)
repack_kernel(const T* __restrict__ src, size_t ld, size_t stride, T* __restrict__ dst, size_t ldp, size_t stride_p,
              size_t inner, size_t outer, size_t batches) {
  const size_t per = inner * outer, total = per * batches;
  const size_t nthreads = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += nthreads) {
    const size_t b = i / per, r = (i - b * per) / inner, c = i - b * per - r * inner;
    dst[b * stride_p + r * ldp + c] = src[b * stride + r * ld + c];
  }
}

// dW = alpha * (sum of the S slabs in ascending s) + beta * dW where the metadata keeps the element, +0 where it prunes it
// (dW is not read when beta == 0).  One thread = one 2:4 group: 4 columns, one metadata nibble, one 16-byte store.
__global__ void __launch_bounds__(256)
wgrad24_reduce_kernel(const float4* __restrict__ part, uint32_t splits, size_t groups, uint32_t kq, const uint8_t* __restrict__ meta,
                      uint32_t meta_m_tiles, float alpha, float beta, float4* dw) {
  const size_t nthreads = (size_t)gridDim.x * blockDim.x;
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < groups; t += nthreads) {
    float4 v = part[t];
    for (uint32_t s = 1; s < splits; ++s) {
      const float4 p = part[(size_t)s * groups + t];
      v.x += p.x; v.y += p.y; v.z += p.z; v.w += p.w;
    }
    const size_t r = t / kq;
    const uint32_t row = (uint32_t)r, col = (uint32_t)(t - r * kq) * 4u;
    const size_t st = (size_t)(col >> 7) * meta_m_tiles + (row >> 7);  // storage index of the metadata tile
    const uint32_t word = *reinterpret_cast<const uint16_t*>(meta + st * 2048 + sm100_meta_word(row & 127u, (col & 127u) >> 4));
    const uint32_t nib = word >> (4u * ((col >> 2) & 3u));
    const uint32_t keep = (1u << (nib & 3u)) | (1u << ((nib >> 2) & 3u));
    float4 o = make_float4(alpha * v.x, alpha * v.y, alpha * v.z, alpha * v.w);
    if (beta != 0.f) {
      const float4 d = dw[t];
      o.x += beta * d.x; o.y += beta * d.y; o.z += beta * d.z; o.w += beta * d.w;
    }
    dw[t] = make_float4(keep & 1u ? o.x : 0.f, keep & 2u ? o.y : 0.f, keep & 4u ? o.z : 0.f, keep & 8u ? o.w : 0.f);
  }
}

// ------------------------------------------------------------------------------------------ host side
size_t elem_bytes(int dtype) { return dtype == SPFY_F32 ? 4 : 2; }

// One operand as the kernel sees it: extent `mn` x `k`, element (i, kk) at (mn_major ? i + kk*ld : kk + i*ld)
struct OperandView {
  const void* base;
  size_t mn, k, ld, stride;  // stride: elements between batches, 0 = shared
  bool mn_major;
};

bool operand_ok(int dtype, const OperandView& v, size_t nb) {
  const size_t es = elem_bytes(dtype);
  if ((uintptr_t)v.base % 16 || (v.ld * es) % 16) return false;
  if (nb > 1 && v.stride && (v.stride * es) % 16) return false;
  const size_t inner = v.mn_major ? v.mn : v.k;
  return v.ld >= inner;
}

size_t padded_ld(int dtype, const OperandView& v) {
  return round_up(v.mn_major ? v.mn : v.k, 16 / elem_bytes(dtype));
}
// bytes of workspace the padded copy of an operand takes (0: TMA can address it as it is)
size_t repack_bytes(int dtype, const OperandView& v, size_t nb) {
  if (operand_ok(dtype, v, nb)) return 0;
  const size_t outer = v.mn_major ? v.k : v.mn, batches = nb > 1 && v.stride ? nb : 1;
  return round_up(batches * outer * padded_ld(dtype, v) * elem_bytes(dtype), 256);
}

int make_operand_map(CUtensorMap* map, int dtype, const OperandView& v, size_t nb, uint32_t box_rows,
                     CUtensorMapSwizzle swizzle, uint32_t mn_box_k = 0) {
  const size_t es = elem_bytes(dtype);
  const uint32_t per_row = (uint32_t)(GM_ROW_BYTES / es);  // elements in 128 bytes
  const size_t inner = v.mn_major ? v.mn : v.k, outer = v.mn_major ? v.k : v.mn;
  const bool batched = nb > 1 && v.stride != 0;
  cuuint64_t dims[3] = {inner, outer, batched ? nb : 1};
  size_t bstride = batched ? v.stride * es : round_up(std::max<size_t>(outer, 1) * v.ld * es, 16);
  cuuint64_t strides[2] = {v.ld * es, bstride};
  // K-major: box = 128 bytes of K x box_rows rows; MN-major: 128 bytes of MN x `per_row` k-rows (one group)
  cuuint32_t box[3] = {per_row, v.mn_major ? (mn_box_k ? mn_box_k : per_row) : box_rows, 1};
  return encode_tiled(map, dtype, 3, v.base, dims, strides, box, swizzle, "tc_gemm");
}

// column split of the Nu dimension: one tile when it fits a UMMA, equal tiles otherwise
void split_nu(size_t nu, size_t gran, size_t max_bn, uint32_t* bn, uint32_t* n_tiles) {
  size_t tiles = ceil_div(nu, max_bn);
  size_t b = round_up(ceil_div(nu, tiles), gran);
  if (b > max_bn) { b = max_bn; }
  *bn = (uint32_t)b;
  *n_tiles = (uint32_t)ceil_div(nu, b);
}

struct Orientation {
  OperandView a, b;  // Au, Bu
  size_t mu, nu;
  bool mu_contig;
  uint32_t bn, n_tiles;
  size_t padded;     // MACs per unit of K actually issued
};

// views of op(A) (extent m) and op(B)^T (extent n) of the column-major problem
void blas_views(const TcGemmProblem& p, OperandView* va, OperandView* vb) {
  // op(A)(i, kk): opA = N -> A is m x k, element i + kk*lda (MN-major); opA = T -> A is k x m, kk + i*lda (K-major)
  *va = OperandView{p.A, p.m, p.k, p.lda, p.strideA, p.opA == SPFY_OP_N};
  // op(B)(kk, j): opB = N -> B is k x n, element kk + j*ldb (K-major); opB = T -> B is n x k, j + kk*ldb (MN-major)
  *vb = OperandView{p.B, p.n, p.k, p.ldb, p.strideB, p.opB != SPFY_OP_N};
}

Orientation orient(int dtype, const TcGemmProblem& p, size_t max_bn) {
  OperandView va, vb;
  blas_views(p, &va, &vb);
  const size_t group = GM_ROW_BYTES / elem_bytes(dtype);
  Orientation o[2];
  // 0: Mu = m (C's contiguous dimension runs along TMEM lanes); 1: Mu = n
  o[0].a = va; o[0].b = vb; o[0].mu = p.m; o[0].nu = p.n; o[0].mu_contig = true;
  o[1].a = vb; o[1].b = va; o[1].mu = p.n; o[1].nu = p.m; o[1].mu_contig = false;
  for (int i = 0; i < 2; ++i) {
    split_nu(o[i].nu, o[i].b.mn_major ? group : 16, max_bn, &o[i].bn, &o[i].n_tiles);
    o[i].padded = round_up(o[i].mu, GM_BM) * (size_t)o[i].bn * o[i].n_tiles;
  }
  if (o[0].padded != o[1].padded) return o[0].padded < o[1].padded ? o[0] : o[1];
  return o[0].mu >= o[1].mu ? o[0] : o[1];
}

int check_problem(int dtype, const TcGemmProblem& p, bool allow_repack) {
  if (dtype != SPFY_F16 && dtype != SPFY_BF16 && dtype != SPFY_F32)
    return fail(SPFY_E_UNSUPPORTED, "tc_gemm: dtype %d (need F16 / BF16 / F32)", dtype);
  if ((p.opA != SPFY_OP_N && p.opA != SPFY_OP_T) || (p.opB != SPFY_OP_N && p.opB != SPFY_OP_T))
    return fail(SPFY_E_INVALID, "tc_gemm: bad transpose flags %d %d", p.opA, p.opB);
  if (p.m == 0 || p.n == 0 || p.nb == 0) return SPFY_OK;
  if (p.k == 0) return fail(SPFY_E_UNSUPPORTED, "tc_gemm: k == 0");
  if (!p.A || !p.B || (!p.C && !p.c_ptrs)) return fail(SPFY_E_INVALID, "tc_gemm: null operand");
  if (p.m >= (1ull << 31) || p.n >= (1ull << 31) || p.k >= (1ull << 31) || p.nb >= (1ull << 31))
    return fail(SPFY_E_UNSUPPORTED, "tc_gemm: dimension too large");
  if (p.ldc < p.m) return fail(SPFY_E_INVALID, "tc_gemm: ldc < m");
  OperandView va, vb;
  blas_views(p, &va, &vb);
  if (va.ld < (va.mn_major ? va.mn : va.k) || vb.ld < (vb.mn_major ? vb.mn : vb.k))
    return fail(SPFY_E_INVALID, "tc_gemm: leading dimension too small (lda %zu ldb %zu)", p.lda, p.ldb);
  if (!allow_repack && (!operand_ok(dtype, va, p.nb) || !operand_ok(dtype, vb, p.nb)))
    return fail(SPFY_E_UNSUPPORTED,
                "tc_gemm: operands must be 16-byte aligned with leading dimensions / batch strides that are multiples "
                "of 16 bytes (lda %zu ldb %zu strideA %zu strideB %zu)", p.lda, p.ldb, p.strideA, p.strideB);
  return SPFY_OK;
}

// `ts`: the 3xTF32 kernel with Au in tensor memory (tiles of at most TS_MAX_BN columns, up to two m-tiles per unit)
// Tile width and m-tiles per unit of a problem that has a 3xTF32 launch to itself, chosen for the WAVE count: units are
// dealt to one CTA per SM, so 224 equal units on 148 SMs take as long as 296 (784 x 256 x 2304 at b = 32: seven tiles of
// 112 columns -> nine of 96 fills two waves with 14 % shorter units).  Cost of a unit per 32-wide K slab = the larger of
// its MMA time (3 MMAs per k-step and m-tile, ~0.66 cycles per column and k-step measured) and the time its operand bytes
// take to enter the SM (~28 B/clk), plus a per-unit constant for the epilogue.
void balance_tiles(const Orientation& o, size_t nb, size_t k_tiles, int sm_count, size_t gran, uint32_t* bn, uint32_t* n_tiles,
                   uint32_t* g) {
  const size_t m_tiles = ceil_div(o.mu, GM_BM);
  double best = 0;
  for (size_t b = gran; b <= (size_t)TS_MAX_BN; b += gran) {
    const size_t nt = ceil_div(o.nu, b);
    if (nt > 1 && (nt - 1) * b >= o.nu) continue;
    for (uint32_t gg = 1; gg <= (uint32_t)TS_G; ++gg) {
      if (gg > m_tiles) break;
      const double units = (double)ceil_div(m_tiles, gg) * (double)nt * (double)nb;
      const double rounds = std::ceil(units / (double)sm_count);
      const double mma = 4.0 * 3.0 * 0.66 * (double)b * gg;
      const double ingest = (double)(gg * GM_BM + b) * GM_ROW_BYTES / 28.0;
      const double cost = rounds * ((double)k_tiles * std::max(mma, ingest) + 3000.0 + 8.0 * (double)b * gg);
      if (best == 0 || cost < best * 0.999) { best = cost; *bn = (uint32_t)b; *n_tiles = (uint32_t)nt; *g = gg; }
    }
  }
}

// `launch_half_units`: units of the whole launch if every problem paired its m-tiles (the G = 2 rule looks at the launch,
// not at one problem: a pointer-array batch is a table of one-batch problems)
int fill_problem(GemmProblemDev* d, int dtype, const TcGemmProblem& p, bool ts, int sm_count, bool alone = false,
                 uint64_t launch_half_units = 0) {
  memset(d, 0, sizeof(*d));
  Orientation o = orient(dtype, p, ts ? TS_MAX_BN : GM_MAX_BN);
  uint32_t g_balanced = 0;
  if (ts && alone && !dev_switch("SPFY_GEMM_NO_BALANCE"))
    balance_tiles(o, p.nb, ceil_div(p.k, GM_ROW_BYTES / elem_bytes(dtype)), sm_count,
                  o.b.mn_major ? GM_ROW_BYTES / elem_bytes(dtype) : 16, &o.bn, &o.n_tiles, &g_balanced);
  // K-major tiles and 16-bit MN-major tiles: 128-byte swizzle.  32-bit MN-major tiles: the tensor core reads them in
  // the 32B-base swizzle only; the 3xTF32 kernel reads its Au tile with ordinary loads and wants it unswizzled.
  const bool f32 = dtype == SPFY_F32;
  const CUtensorMapSwizzle sw_a = !(f32 && o.a.mn_major) ? CU_TENSOR_MAP_SWIZZLE_128B
                                  : ts ? CU_TENSOR_MAP_SWIZZLE_NONE : CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B;
  const CUtensorMapSwizzle sw_b = f32 && o.b.mn_major ? CU_TENSOR_MAP_SWIZZLE_128B_ATOM_32B : CU_TENSOR_MAP_SWIZZLE_128B;
  int rc = make_operand_map(&d->tmap_a, dtype, o.a, p.nb, GM_BM, sw_a);
  if (rc) return rc;
  rc = make_operand_map(&d->tmap_b, dtype, o.b, p.nb, o.bn, sw_b);
  if (rc) return rc;
  const size_t kel = GM_ROW_BYTES / elem_bytes(dtype);
  d->C = (uint8_t*)p.C;
  d->c_ptrs = reinterpret_cast<const uint64_t*>(p.c_ptrs);
  d->ldc = p.ldc;
  d->stride_c = p.strideC;
  d->mu = (uint32_t)o.mu;
  d->nu = (uint32_t)o.nu;
  d->k = (uint32_t)p.k;
  d->nb = (uint32_t)p.nb;
  d->m_tiles = (uint32_t)ceil_div(o.mu, GM_BM);
  d->n_tiles = o.n_tiles;
  d->k_tiles = (uint32_t)ceil_div(p.k, kel);
  d->bn = o.bn;
  d->a_mn = o.a.mn_major;
  d->b_mn = o.b.mn_major;
  d->a_batched = p.nb > 1 && o.a.stride != 0;
  d->b_batched = p.nb > 1 && o.b.stride != 0;
  d->out_mu_contig = o.mu_contig;
  d->alpha = p.alpha;
  d->beta = p.beta;
  // two m-tiles share every Bu stage whenever that leaves at least half a wave of units (bytes entering the SMs, not
  // units, are what the kernel is short of: DESIGN.md 4)
  d->g = 1;
  const uint64_t half_units = std::max<uint64_t>(launch_half_units, (uint64_t)ceil_div(d->m_tiles, TS_G) * d->n_tiles * d->nb);
  if (ts && d->m_tiles >= 2 && 2 * half_units >= (uint64_t)sm_count && !dev_switch("SPFY_GEMM_G1"))
    d->g = TS_G;
  if (g_balanced) d->g = g_balanced;
  d->m_groups = (uint32_t)ceil_div(d->m_tiles, d->g);
  const uint64_t units = (uint64_t)d->m_groups * d->n_tiles * d->nb;
  if (units >= (1ull << 31)) return fail(SPFY_E_UNSUPPORTED, "tc_gemm: too many tiles");
  d->units = (uint32_t)units;
  return SPFY_OK;
}

template <int KIND>
int launch_kind(const GemmProblemDev& single, const GemmLaunch& L, uint32_t smem, int grid, cudaStream_t s) {
  int rc = allow_dynamic_smem<tcgemm_kernel<KIND>>(GM_SMEM_LIMIT);
  if (rc) return rc;
  tcgemm_kernel<KIND><<<grid, GM_THREADS, smem, s>>>(single, L);
  SPFY_LAUNCH_OK("tcgemm_kernel");
  return SPFY_OK;
}

int launch_ts(const GemmProblemDev& single, const GemmLaunch& L, uint32_t smem, int grid, cudaStream_t s) {
  int rc = allow_dynamic_smem<tcgemm_ts_kernel>(GM_SMEM_LIMIT);
  if (rc) return rc;
  tcgemm_ts_kernel<<<grid, TS_THREADS, smem, s>>>(single, L);
  SPFY_LAUNCH_OK("tcgemm_ts_kernel");
  return SPFY_OK;
}

}  // namespace

void warm_gemm_kernels() {
  touch_kernel(tcgemm_ts_kernel);
  touch_kernel(tcgemm_kernel<KIND_F16>);
  touch_kernel(tcgemm_kernel<KIND_BF16>);
  touch_kernel(tcgemm_kernel<KIND_F32>);
  touch_kernel(tcgemm_kernel<KIND_F16, true>);
  touch_kernel(tcgemm_kernel<KIND_BF16, true>);
  touch_kernel(wgrad24_reduce_kernel);
}

int tc_gemm_supported(int dtype, const TcGemmProblem& p, bool allow_repack) {
  DeviceInfo di;
  int rc = require_sm100("tc_gemm", &di);
  if (rc) return rc;
  return check_problem(dtype, p, allow_repack);
}

static size_t table_bytes(size_t count) { return count > 1 ? round_up(count * sizeof(GemmProblemDev) + 64, 256) : 0; }

size_t tc_gemm_workspace_bytes(int dtype, const TcGemmProblem* problems, size_t count) {
  size_t need = table_bytes(count);
  if (dtype != SPFY_F16 && dtype != SPFY_BF16 && dtype != SPFY_F32) return need;
  for (size_t i = 0; i < count; ++i) {
    OperandView va, vb;
    blas_views(problems[i], &va, &vb);
    need += repack_bytes(dtype, va, problems[i].nb) + repack_bytes(dtype, vb, problems[i].nb);
  }
  return need;
}

namespace {
// padded copies made during one tc_gemm_run call (an operand shared by several problems is copied once)
struct Repacked {
  const void* src;
  size_t inner, outer, ld, stride, batches;
  const void* dst;
};

int repack_operand(int dtype, OperandView* v, size_t nb, uint8_t* ws, size_t ws_bytes, size_t* used,
                   std::vector<Repacked>* done, cudaStream_t s) {
  if (operand_ok(dtype, *v, nb)) return SPFY_OK;
  const size_t es = elem_bytes(dtype), inner = v->mn_major ? v->mn : v->k, outer = v->mn_major ? v->k : v->mn;
  const size_t batches = nb > 1 && v->stride ? nb : 1, ldp = padded_ld(dtype, *v);
  for (const Repacked& r : *done)
    if (r.src == v->base && r.inner == inner && r.outer == outer && r.ld == v->ld && r.stride == v->stride &&
        r.batches == batches) {
      v->base = r.dst; v->ld = ldp; v->stride = batches > 1 ? outer * ldp : 0;
      return SPFY_OK;
    }
  const size_t bytes = repack_bytes(dtype, *v, nb);
  if (!ws || *used + bytes > ws_bytes)
    return fail(SPFY_E_WORKSPACE, "tc_gemm: workspace %zu < %zu bytes (padded copy of an operand TMA cannot address)",
                ws_bytes, *used + bytes);
  uint8_t* dst = ws + *used;
  *used += bytes;
  const size_t total = batches * outer * inner;
  int grid = 1;
  int rc = capped_grid(ceil_div(total, 256), 16, &grid);
  if (rc) return rc;
  if (es == 4)
    repack_kernel<uint32_t><<<grid, 256, 0, s>>>((const uint32_t*)v->base, v->ld, v->stride, (uint32_t*)dst, ldp, outer * ldp,
                                                inner, outer, batches);
  else
    repack_kernel<uint16_t><<<grid, 256, 0, s>>>((const uint16_t*)v->base, v->ld, v->stride, (uint16_t*)dst, ldp, outer * ldp,
                                                inner, outer, batches);
  SPFY_LAUNCH_OK("repack_kernel");
  done->push_back(Repacked{v->base, inner, outer, v->ld, v->stride, batches, dst});
  v->base = dst; v->ld = ldp; v->stride = batches > 1 ? outer * ldp : 0;
  return SPFY_OK;
}
}  // namespace

int tc_gemm_run(int dtype, int precision, const TcGemmProblem* problems, size_t count, void* ws, size_t ws_bytes,
                cudaStream_t stream, const int* gate, int gate_run_if) {
  if (precision != TC_GEMM_PRECISE && precision != TC_GEMM_FAST)
    return fail(SPFY_E_INVALID, "tc_gemm: precision %d (need SPFY_GEMM_PRECISE or SPFY_GEMM_FAST)", precision);
  if (count == 0) return SPFY_OK;
  if (!problems) return fail(SPFY_E_INVALID, "tc_gemm: null problem list");
  DeviceInfo di;
  int rc = require_sm100("tc_gemm", &di);
  if (rc) return rc;
  std::vector<GemmProblemDev> table;
  table.reserve(count);
  uint32_t units = 0, bn_max = 16;
  const bool ts = dtype == SPFY_F32 && precision == TC_GEMM_PRECISE;
  // workspace: [device copy of the problem table (count > 1)][padded copies of operands TMA cannot address]
  uint8_t* ws8 = (uint8_t*)ws;
  const size_t ws_pad = ws8 ? (256 - (uintptr_t)ws8 % 256) % 256 : 0;
  if (ws8 && ws_bytes >= ws_pad) { ws8 += ws_pad; ws_bytes -= ws_pad; } else { ws8 = nullptr; ws_bytes = 0; }
  size_t ws_used = table_bytes(count);
  std::vector<Repacked> repacked;
  uint64_t launch_half_units = 0;
  for (size_t i = 0; i < count && ts; ++i) {
    if (check_problem(dtype, problems[i], true) != SPFY_OK || problems[i].m == 0 || problems[i].n == 0 || problems[i].nb == 0)
      continue;
    const Orientation o = orient(dtype, problems[i], TS_MAX_BN);
    launch_half_units += (uint64_t)ceil_div(ceil_div(o.mu, GM_BM), TS_G) * o.n_tiles * problems[i].nb;
  }
  for (size_t i = 0; i < count; ++i) {
    rc = check_problem(dtype, problems[i], true);
    if (rc) return rc;
    if (problems[i].m == 0 || problems[i].n == 0 || problems[i].nb == 0) continue;
    TcGemmProblem q = problems[i];
    {
      OperandView va, vb;
      blas_views(q, &va, &vb);
      rc = repack_operand(dtype, &va, q.nb, ws8, ws_bytes, &ws_used, &repacked, stream);
      if (rc) return rc;
      rc = repack_operand(dtype, &vb, q.nb, ws8, ws_bytes, &ws_used, &repacked, stream);
      if (rc) return rc;
      q.A = va.base; q.lda = va.ld; q.strideA = va.stride;
      q.B = vb.base; q.ldb = vb.ld; q.strideB = vb.stride;
    }
    GemmProblemDev d;
    rc = fill_problem(&d, dtype, q, ts, di.sm_count, count == 1, launch_half_units);
    if (rc) return rc;
    d.unit_begin = units;
    if ((uint64_t)units + d.units >= (1ull << 31)) return fail(SPFY_E_UNSUPPORTED, "tc_gemm: too many tiles");
    units += d.units;
    bn_max = std::max(bn_max, d.bn);
    table.push_back(d);
  }
  if (table.empty()) return SPFY_OK;

  GemmLaunch L;
  memset(&L, 0, sizeof(L));
  const bool f32 = dtype == SPFY_F32;
  // The tensor core ignores the low 13 mantissa bits of a TF32 operand (measured: tools/gpu_wh.sh, same error with and
  // without the store), so the 3xTF32 kernel leaves the raw Bu tile in place as "hi" and only writes lo = x - trunc(x).
  if (const char* e = dev_switch("SPFY_GEMM_WRITE_HI")) L.write_hi = (uint32_t)atoi(e);
  L.kelems = (uint32_t)(GM_ROW_BYTES / elem_bytes(dtype));
  L.gate = gate;
  L.gate_run_if = gate_run_if ? 1u : 0u;
  if (const char* e = dev_switch("SPFY_GEMM_DEBUG")) L.dbg = (uint32_t)atoi(e);
  uint32_t smem = 0;
  if (ts) {
    // [Au ring: a_stages x 16 KiB][Bu ring: 4 x (hi | lo)][barriers]
    L.raw_bytes = bn_max * (uint32_t)GM_ROW_BYTES;
    L.stage_bytes = 2u * L.raw_bytes;
    L.stages = TS_B_STAGES;
    uint32_t a_stages = (GM_SMEM_LIMIT - 1024u - GM_BAR_BYTES - L.stages * L.stage_bytes) / (uint32_t)TS_A_STAGE_BYTES;
    if (a_stages > (uint32_t)TS_MAX_A_STAGES) a_stages = TS_MAX_A_STAGES;
    if (const char* e = dev_switch("SPFY_GEMM_STAGES")) {
      const uint32_t c = (uint32_t)atoi(e);
      if (c >= 1 && c < a_stages) a_stages = c;
    }
    L.a_stages = a_stages;
    if (a_stages < 2) return fail(SPFY_E_UNSUPPORTED, "tc_gemm: tile does not fit shared memory");
    L.d_cols = bn_max <= 64 ? 64u : 128u;   // accumulators [0, 256): slots x TS_G m-tiles x d_cols
    L.acc_slots = bn_max <= 64 ? 2u : 1u;
    L.b_off = a_stages * (uint32_t)TS_A_STAGE_BYTES;
    L.bar_off = L.b_off + L.stages * L.stage_bytes;
    smem = L.bar_off + GM_BAR_BYTES + 1024u;
  } else {
    L.stage_bytes = (uint32_t)GM_A_BYTES + bn_max * (uint32_t)GM_ROW_BYTES;
    uint32_t stages = (GM_SMEM_LIMIT - 1024u - GM_BAR_BYTES) / L.stage_bytes;
    if (stages > (uint32_t)GM_MAX_STAGES) stages = GM_MAX_STAGES;
    if (const char* e = dev_switch("SPFY_GEMM_STAGES")) {
      const uint32_t c = (uint32_t)atoi(e);
      if (c >= 1 && c < stages) stages = c;
    }
    if (stages < 2) return fail(SPFY_E_UNSUPPORTED, "tc_gemm: tile does not fit shared memory");
    L.stages = stages;
    L.bar_off = stages * L.stage_bytes;
    smem = L.bar_off + GM_BAR_BYTES + 1024u;
  }
  // instruction descriptor: D = F32; A / B format (F16 0, BF16 1, TF32 2); M = 128; N and majors per problem
  const uint32_t fmt = f32 ? 2u : (dtype == SPFY_BF16 ? 1u : 0u);
  L.idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(GM_BM >> 4) << 24);
  L.num_problems = (uint32_t)table.size();
  L.total_units = units;
  L.table = nullptr;
  if (table.size() > 1) {
    const size_t need = table.size() * sizeof(GemmProblemDev);
    if (!ws8 || ws_bytes < table_bytes(count))
      return fail(SPFY_E_WORKSPACE, "tc_gemm: workspace %zu < %zu bytes", ws_bytes, table_bytes(count));
    // pageable source: the runtime stages the bytes before the call returns, so `table` may go out of scope
    SPFY_CUDA_OK(cudaMemcpyAsync(ws8, table.data(), need, cudaMemcpyHostToDevice, stream));
    L.table = reinterpret_cast<const GemmProblemDev*>(ws8);
  }
  const int grid = (int)std::min<uint32_t>(units, (uint32_t)di.sm_count);
  if (ts) return launch_ts(table[0], L, smem, grid, stream);
  if (f32) return launch_kind<KIND_F32>(table[0], L, smem, grid, stream);
  if (dtype == SPFY_BF16) return launch_kind<KIND_BF16>(table[0], L, smem, grid, stream);
  return launch_kind<KIND_F16>(table[0], L, smem, grid, stream);
}

// ------------------------------------------------------------------------------------------------------------
// Weight gradient of a 2:4 convolution (spfy_conv_wgrad24): tcgemm_kernel<KIND, true> writes S fp32 partial sums of
// dW = dY^T im2col(X) to the workspace, one per split of the output positions, and wgrad24_reduce_kernel adds them up.
// ------------------------------------------------------------------------------------------------------------
namespace {

// The split count targets one wave of units on the 148 SMs of a B200 with at least WG_MIN_STAGES stages (64 output
// positions each) per unit.  It is a constant of the shape, not of the device, so that the workspace query needs no
// device and a shape always sums in the same order.
constexpr size_t WG_SMS = 148;
constexpr size_t WG_MIN_STAGES = 8;

struct WgradShape {
  size_t ho, wo, positions, kk;  // kk = kh * kw * c
  uint32_t m_tiles, n_tiles, bn, k_tiles, splits;  // m-tiles along kk, n-tiles along m, stages per split, S
};

int wgrad_shape(int dtype, const spfy_conv_desc* conv, size_t m, WgradShape* out) {
  const char* who = "conv_wgrad24";
  if (dtype != SPFY_F16 && dtype != SPFY_BF16) return fail(SPFY_E_UNSUPPORTED, "%s: dtype %d (need F16/BF16)", who, dtype);
  if (!conv) return fail(SPFY_E_INVALID, "%s: null descriptor", who);
  const spfy_conv_desc& c = *conv;
  if (!c.batch || !c.h || !c.w || !c.c || !c.kh || !c.kw || !c.stride || !m)
    return fail(SPFY_E_INVALID, "%s: empty dimension", who);
  if (c.c % 64) return fail(SPFY_E_UNSUPPORTED, "%s: channels must be a multiple of 64 (got %zu)", who, c.c);
  if (m % 8) return fail(SPFY_E_UNSUPPORTED, "%s: m (the channels of dY) must be a multiple of 8 (got %zu)", who, m);
  if (c.kh > 16 || c.kw > 16 || c.pad > 8 || c.stride > 8)
    return fail(SPFY_E_UNSUPPORTED, "%s: filter / padding / stride outside what the im2col tensor map encodes", who);
  if (c.h + 2 * c.pad < c.kh || c.w + 2 * c.pad < c.kw) return fail(SPFY_E_INVALID, "%s: filter larger than the padded image", who);
  WgradShape s;
  s.ho = (c.h + 2 * c.pad - c.kh) / c.stride + 1;
  s.wo = (c.w + 2 * c.pad - c.kw) / c.stride + 1;
  s.positions = c.batch * s.ho * s.wo;
  s.kk = c.kh * c.kw * c.c;
  if (s.positions >= (1ull << 31) || m >= (1ull << 20) || c.c >= (1ull << 20) || c.batch * c.h * c.w >= (1ull << 31) ||
      m * s.kk >= (1ull << 31))
    return fail(SPFY_E_UNSUPPORTED, "%s: dimension too large", who);
  split_nu(m, 64, GM_MAX_BN, &s.bn, &s.n_tiles);
  s.m_tiles = (uint32_t)ceil_div(s.kk, GM_BM);
  const size_t stages = ceil_div(s.positions, 64), tiles = (size_t)s.m_tiles * s.n_tiles;
  const size_t s0 = std::max<size_t>(1, std::min(WG_SMS / tiles, stages / WG_MIN_STAGES));
  s.k_tiles = (uint32_t)ceil_div(stages, s0);
  s.splits = (uint32_t)ceil_div(stages, s.k_tiles);
  *out = s;
  return SPFY_OK;
}

size_t wgrad_workspace(const WgradShape& s, size_t m) { return (size_t)s.splits * m * s.kk * sizeof(float); }

}  // namespace

int conv_wgrad24_run(int dtype, const spfy_conv_desc* conv, size_t m, float alpha, const void* X, const void* dY,
                     const void* meta, float beta, float* dW, void* ws, size_t ws_bytes, cudaStream_t stream) {
  const char* who = "conv_wgrad24";
  WgradShape s;
  int rc = wgrad_shape(dtype, conv, m, &s);
  if (rc) return rc;
  if (!X || !dY || !meta || !dW || !ws) return fail(SPFY_E_INVALID, "%s: null buffer", who);
  if ((uintptr_t)X % 16 || (uintptr_t)dY % 16 || (uintptr_t)meta % 16 || (uintptr_t)dW % 16 || (uintptr_t)ws % 16)
    return fail(SPFY_E_INVALID, "%s: buffers must be 16-byte aligned", who);
  const size_t need = wgrad_workspace(s, m);
  if (ws_bytes < need) return fail(SPFY_E_WORKSPACE, "%s: workspace %zu < %zu bytes", who, ws_bytes, need);
  DeviceInfo di;
  rc = require_sm100(who, &di);
  if (rc) return rc;
  const spfy_conv_desc& c = *conv;

  GemmProblemDev d;
  memset(&d, 0, sizeof(d));
  rc = make_tmap_im2col(&d.tmap_a, dtype, X, im2col_of(c), 64);
  if (rc) return rc;
  rc = make_operand_map(&d.tmap_b, dtype, OperandView{dY, m, s.positions, m, 0, true}, 1, s.bn, CU_TENSOR_MAP_SWIZZLE_128B);
  if (rc) return rc;
  d.C = (uint8_t*)ws;
  d.ldc = s.kk;
  d.stride_c = m * s.kk;
  d.mu = (uint32_t)s.kk;
  d.nu = (uint32_t)m;
  d.k = s.k_tiles * 64u;
  d.nb = s.splits;
  d.m_tiles = s.m_tiles;
  d.n_tiles = s.n_tiles;
  d.k_tiles = s.k_tiles;
  d.g = 1;
  d.m_groups = s.m_tiles;
  d.bn = s.bn;
  d.a_mn = d.b_mn = 1;
  d.out_mu_contig = 1;
  d.units = s.m_tiles * s.n_tiles * s.splits;
  d.alpha = 1.f;

  GemmLaunch L;
  memset(&L, 0, sizeof(L));
  L.kelems = 64;
  L.stage_bytes = (uint32_t)GM_A_BYTES + s.bn * (uint32_t)GM_ROW_BYTES;
  L.stages = std::min<uint32_t>((GM_SMEM_LIMIT - 1024u - GM_BAR_BYTES) / L.stage_bytes, GM_MAX_STAGES);
  L.bar_off = L.stages * L.stage_bytes;
  const uint32_t smem = L.bar_off + GM_BAR_BYTES + 1024u;
  const uint32_t fmt = dtype == SPFY_BF16 ? 1u : 0u;
  L.idesc = (1u << 4) | (fmt << 7) | (fmt << 10) | ((uint32_t)(GM_BM >> 4) << 24);
  L.num_problems = 1;
  L.total_units = d.units;
  L.wg.c = (uint32_t)c.c;
  L.wg.kw = (uint32_t)c.kw;
  L.wg.wo = (uint32_t)s.wo;
  L.wg.ho = (uint32_t)s.ho;
  L.wg.stride = (uint32_t)c.stride;
  L.wg.off_h = L.wg.off_w = -(int)c.pad;
  const size_t img = s.ho * s.wo;
  L.wg.dn = (uint32_t)(64 / img);
  L.wg.dh = (uint32_t)(64 % img / s.wo);
  L.wg.dw = (uint32_t)(64 % img % s.wo);

  const int grid = (int)std::min<uint32_t>(d.units, (uint32_t)di.sm_count);
  const size_t groups = m * s.kk / 4;
  int rgrid = 1;
  rc = capped_grid(ceil_div(groups, 256), 8, &rgrid);
  if (rc) return rc;
  if (dtype == SPFY_BF16) {
    rc = allow_dynamic_smem<tcgemm_kernel<KIND_BF16, true>>(GM_SMEM_LIMIT);
    if (rc) return rc;
    tcgemm_kernel<KIND_BF16, true><<<grid, GM_THREADS, smem, stream>>>(d, L);
  } else {
    rc = allow_dynamic_smem<tcgemm_kernel<KIND_F16, true>>(GM_SMEM_LIMIT);
    if (rc) return rc;
    tcgemm_kernel<KIND_F16, true><<<grid, GM_THREADS, smem, stream>>>(d, L);
  }
  SPFY_LAUNCH_OK("tcgemm_kernel (weight gradient)");
  wgrad24_reduce_kernel<<<rgrid, 256, 0, stream>>>((const float4*)ws, s.splits, groups, (uint32_t)(s.kk / 4), (const uint8_t*)meta,
                                                   (uint32_t)ceil_div(m, 128), alpha, beta, (float4*)dW);
  SPFY_LAUNCH_OK("wgrad24_reduce_kernel");
  return SPFY_OK;
}

}  // namespace spfy

using namespace spfy;

extern "C" {

static TcGemmProblem make_problem(int opA, int opB, size_t m, size_t n, size_t k, float alpha, const void* A, size_t lda,
                                  size_t strideA, const void* B, size_t ldb, size_t strideB, float beta, void* C,
                                  size_t ldc, size_t strideC, size_t nb) {
  TcGemmProblem p;
  p.opA = opA; p.opB = opB; p.m = m; p.n = n; p.k = k; p.nb = nb;
  p.A = A; p.lda = lda; p.strideA = strideA;
  p.B = B; p.ldb = ldb; p.strideB = strideB;
  p.C = C; p.ldc = ldc; p.strideC = strideC;
  p.alpha = alpha; p.beta = beta;
  return p;
}

int spfy_gemm_workspace_bytes(int dtype, int opA, int opB, size_t m, size_t n, size_t k, size_t lda, size_t ldb,
                              size_t num_batches, size_t* bytes) {
  // a table of num_batches problems (batched form) + a padded copy per batch element of every operand whose leading
  // dimension TMA cannot address.  Bases are taken to be 16-byte aligned (cudaMalloc gives 256); pass lda = 0 /
  // ldb = 0 to size for a misaligned base as well.
  const size_t es = elem_bytes(dtype);
  size_t need = 256 + (num_batches > 1 ? round_up(num_batches * sizeof(GemmProblemDev) + 64, 256) : 0);
  const size_t a_inner = opA == SPFY_OP_N ? m : k, a_outer = opA == SPFY_OP_N ? k : m;
  const size_t b_inner = opB == SPFY_OP_N ? k : n, b_outer = opB == SPFY_OP_N ? n : k;
  if (lda == 0 || (lda * es) % 16) need += num_batches * round_up(a_outer * round_up(a_inner, 16 / es) * es, 256);
  if (ldb == 0 || (ldb * es) % 16) need += num_batches * round_up(b_outer * round_up(b_inner, 16 / es) * es, 256);
  if (bytes) *bytes = need;
  return SPFY_OK;
}

int spfy_gemm_strided_batched(int dtype, int precision, int opA, int opB, size_t m, size_t n, size_t k, float alpha,
                              const void* A, size_t lda, size_t strideA, const void* B, size_t ldb, size_t strideB,
                              float beta, void* C, size_t ldc, size_t strideC, size_t num_batches, void* workspace,
                              size_t workspace_bytes, spfy_stream_t stream) {
  const TcGemmProblem p = make_problem(opA, opB, m, n, k, alpha, A, lda, strideA, B, ldb, strideB, beta, C, ldc, strideC,
                                       num_batches);
  return tc_gemm_run(dtype, precision, &p, 1, workspace, workspace_bytes, (cudaStream_t)stream);
}

int spfy_gemm_batched(int dtype, int precision, int opA, int opB, size_t m, size_t n, size_t k, float alpha,
                      const void* const* A_ptrs, size_t lda, const void* const* B_ptrs, size_t ldb, float beta,
                      void* const* C_ptrs, size_t ldc, size_t num_batches, void* workspace, size_t workspace_bytes,
                      spfy_stream_t stream) {
  if (num_batches == 0) return SPFY_OK;
  if (!A_ptrs || !B_ptrs || !C_ptrs) return fail(SPFY_E_INVALID, "gemm_batched: null pointer array");
  std::vector<TcGemmProblem> ps(num_batches);
  for (size_t b = 0; b < num_batches; ++b)
    ps[b] = make_problem(opA, opB, m, n, k, alpha, A_ptrs[b], lda, 0, B_ptrs[b], ldb, 0, beta, C_ptrs[b], ldc, 0, 1);
  return tc_gemm_run(dtype, precision, ps.data(), ps.size(), workspace, workspace_bytes, (cudaStream_t)stream);
}

int spfy_conv_wgrad24_workspace_bytes(int dtype, const spfy_conv_desc* conv, size_t m, size_t* bytes) {
  WgradShape s;
  const int rc = wgrad_shape(dtype, conv, m, &s);
  if (rc) return rc;
  if (bytes) *bytes = wgrad_workspace(s, m);
  return SPFY_OK;
}

int spfy_conv_wgrad24(int dtype, const spfy_conv_desc* conv, size_t m, float alpha, const void* X, const void* dY,
                      const void* meta, float beta, float* dW, void* workspace, size_t workspace_bytes, spfy_stream_t stream) {
  return conv_wgrad24_run(dtype, conv, m, alpha, X, dY, meta, beta, dW, workspace, workspace_bytes, (cudaStream_t)stream);
}

}  // extern "C"
