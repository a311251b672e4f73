// spmma_sm100.cu -- 2:4 structured-sparse GEMM on tcgen05.mma.sp (sm_100a)
//
// Replaces cusparseLtMatmul (reference: include/sparsify.me/spmma.hxx:106-114):
//     D[m x n] = alpha * A(2:4)[m x k] * op(B)[k x n] + beta * C[m x n]
// all row-major like the reference's descriptors (spmma.hxx:56-64), fp16 or bf16 in, fp32
// accumulation in TMEM, fp16/bf16 out.  Two entry points share one kernel:
//     spfy_spmma            one problem (what the header template calls); spfy_spmma_ex adds the epilogue
//                           (per-row scale / bias, ReLU / GELU, beta * C with the transposed output)
//     spfy_spmma_plan_*     a list of independent problems (the per-layer GEMMs of a
//                           datasets/*.csv table) executed by one persistent launch per launch class
//                           present (ring geometry; six classes), chained tail-to-head
//
// Every ResNet shape is HBM-bound for this operator.  Two measured facts shape the kernel
// (DESIGN.md section 4): the chip-wide L2->SM throughput is only ~1.9x the HBM bandwidth, so
// operand re-reads from L2 are nearly as expensive as DRAM traffic; and one trip of the
// single-thread producer/MMA handshake costs ~600 cycles whatever it carries, so a ring stage
// must carry tens of KiB.  Hence:
//   * work unit = (problem, n-tile of 128 columns, group of G <= 2 m-tiles): one 32 KiB B stage
//     in shared memory feeds the MMAs of both m-tiles of the group;
//   * "resident" problems (whole compressed A <= 96 KiB): A values + metadata are loaded into
//     shared memory once per CTA and problem, the ring then streams B only;
//   * a stage is 128 logical k and is filled by at most three bulk/TMA operations;
//   * units are dealt round-robin to the persistent CTAs, so neighbouring CTAs stream
//     neighbouring B columns at the same time (DRAM page locality, L2 hits for the other m-group).
//
// CTA = 320 threads, 1 CTA/SM:
//   warp 0      producer : cp.async.bulk (A value tiles / metadata tiles, pre-swizzled by
//                          spfy_prune24) + TMA tensor loads (B), one mbarrier per ring stage
//   warp 1      MMA      : one thread issues tcgen05.cp (metadata smem -> TMEM) and
//                          tcgen05.mma.sp.cta_group::1.kind::f16 (M128 x N128 x K32);
//                          tcgen05.commit frees ring stages / publishes accumulators
//   warps 2-9   epilogue : a warp owns 32 rows x 64 columns of an accumulator: tcgen05.ld ->
//                          alpha/beta (or the epilogue) -> fp16/bf16 -> its own swizzled 4 KiB staging buffer -> its own
//                          TMA store.  No CTA-wide barrier in steady state.  Streaming classes
//                          run 4 of the 8 warps (2 column halves each) to leave room for the ring.
// TMEM: three 128-column accumulator slots used as a ring over (unit, m-tile) jobs, so the epilogue
// of one job overlaps the MMAs of the next ones; metadata lives in 16 columns behind them.
//
// Operand format (spfy_prune24, layout SPFY_LAYOUT_SM100): tile (mt, kt) covers rows
// [128mt, 128mt+128) x logical columns [128kt, 128kt+128) and sits at index kt*m_tiles + mt
// (k-tile major, so the m-tiles of a group are adjacent).  A 16 KiB value tile is the exact
// 128B-swizzled K-major shared-memory image (row r at r*128, 16-byte chunk c at c ^ (r&7)); a 2 KiB
// metadata tile is the exact `tcgen05.cp.128x128b` source image of the kind::f16 sparse-metadata
// TMEM layout.
#include "tc_ptx.cuh"

#include <algorithm>
#include <cstdlib>
#include <memory>
#include <vector>

namespace spfy {
namespace {

constexpr int BM = 128;              // rows of A per m-tile (UMMA M)
constexpr int BN = 128;              // columns of B/D per unit (UMMA N)
constexpr int BK = 128;              // logical K per ring stage (4 MMAs of K=32)
constexpr int MAX_G = 2;             // m-tiles that share one B stage
constexpr int A_TILE_BYTES = 16384;  // 128 rows x 128 bytes
constexpr int E_TILE_BYTES = 2048;   // metadata of 128 rows x 128 logical k
constexpr int B_STAGE_BYTES = BK * BN * 2;
constexpr int NUM_EPI_WARPS = 8;
constexpr int NUM_THREADS = (2 + NUM_EPI_WARPS) * 32;
constexpr int C_BUF_BYTES = 32 * 128;  // one epilogue warp: 32 rows x 64 columns x 2 bytes
constexpr int ACC_SLOTS = 3;
constexpr int TMEM_COLS = 512;
constexpr int TMEM_E_COL = ACC_SLOTS * BN;  // 384: metadata columns
constexpr int MAX_STAGES = 8;
constexpr int SMEM_LIMIT = 232448;  // 227 KiB opt-in maximum per CTA

// one GEMM as the kernel sees it (lives in kernel-parameter space for spfy_spmma, in a device
// table for plans; the tensor maps must be 64-byte aligned)
struct alignas(64) ProblemDev {
  // B.  b3d: viewed as [groups of 64 inner elements][outer rows][64]: one box (64, 128, 2) fills a
  // whole stage; otherwise 2-D with two (64, 128) boxes per stage.
  CUtensorMap tmap_b;
  CUtensorMap tmap_d;  // D: [m][n] boxes (64 n, 32 m)
  const uint8_t* a_vals;
  const uint8_t* a_meta;
  const void* C;       // only read when beta != 0
  uint64_t ldc;
  uint32_t m, n, k;
  uint32_t m_tiles, k_tiles, n_tiles, m_groups;
  uint32_t G;          // m-tiles per unit
  uint32_t resident;   // 1: whole A lives in shared memory; 2: the unit's m-group slice of A does (reloaded when the
                       // CTA's next unit belongs to another m-group, which never happens when gridDim % m_groups == 0)
  uint32_t b3d;
  uint32_t unit_begin, units;  // this problem's range in the launch-wide unit order
  // Tail splitting (single calls): units [0, split_units) pair the m-tiles (G) of n-tiles [0, split_nt); the n-tiles
  // from split_nt on -- the last, partial wave -- are dealt one m-tile per unit, so that the tail costs about half a unit
  // on twice as many SMs instead of a whole unit on a few.  No split: split_units = units, split_nt = n_tiles.
  uint32_t split_units, split_nt;
  float alpha, beta;
  uint64_t hint_b;
  // replicated outputs (fused output gather, spfy_spmma_plan_create_replicated): every D tile is also stored through
  // these maps -- the same matrix at other base addresses, e.g. this rank's slab of the gather arena in every peer
  // GPU's memory (peer mappings over NVLink)
  const CUtensorMap* tmap_rep;
  uint32_t n_rep;
  uint32_t out_t;              // D (and its replicas) are [n][m]: tmap_d boxes are (32 m, 64 n), unswizzled
  // implicit GEMM (spfy_spmma_conv): B is never materialised -- tmap_b is an im2col map over the NHWC activations and a
  // B stage (128 positions x 128 k) is gathered as two (128 positions x 64 channels) pieces, one filter tap each
  uint32_t conv;               // 0: B is a matrix
  uint32_t conv_c, conv_kw;    // channels (multiple of 64), filter width
  uint32_t conv_wo, conv_ho;   // output width / height
  uint32_t conv_stride;
  int32_t conv_off_h, conv_off_w;  // base pixel of output position (0, 0): -pad, or a data-gradient phase's dy offset
  // epilogue of the _ex entry points: v = (alpha * scale[row]) * acc + beta * C + bias[row], D = act(v).  epi != 0 selects
  // the epilogue code that applies it (also taken for beta != 0 with the transposed output, whose C is [n][m] like D);
  // epi == 0 runs the alpha / beta code of the plain entry points, unchanged.
  const float* scale;  // [m] or null
  const float* bias;   // [m] or null
  uint32_t act;        // SPFY_ACT_*
  uint32_t epi;
  // scattered NHWC output (spfy_spmma_conv_dgrad, kernels instantiated with SCATTER): position (image, i, j) of the
  // [batch][conv_ho][conv_wo] grid is the row ((image * sc_h + sc_s * i + sc_a) * sc_w + sc_s * j + sc_b) of D [.][ldd],
  // which is written with 16-byte stores instead of through tmap_d (and C, when beta != 0, read at the same row)
  void* D;
  uint64_t ldd;
  uint32_t sc_h, sc_w, sc_s, sc_a, sc_b;
};

struct LaunchParams {
  const ProblemDev* table;  // null -> the single problem passed by value
  uint32_t num_problems;
  uint32_t total_units;
  uint32_t idesc;
  // shared-memory geometry of this launch
  uint32_t stages, stage_bytes, a_off, e_off;  // ring stage: [B 32 KiB][A tile x G][E tile x G]
  uint32_t res_off, res_e_off;                 // resident A values / metadata
  uint32_t c_off, bar_off;
  uint32_t epi_warps;  // 8: one column half per warp; 4: warps 2-5 do both halves
  uint32_t bk;         // logical k per ring stage: 128, or 64 for the k <= 64 class (half-size stages)
  uint32_t dbg;        // development switches (SPFY_SPMMA_DEBUG): 2 no epilogue work, 4 no B loads, 8 no MMAs,
                       // 16 no streamed A loads, 32 no TMA stores (timing experiments only: results are garbage)
#ifdef SPFY_DEV_SWITCHES
  long long* trace;    // SPFY_SPMMA_TRACE: CTA 0 logs clock64() at the hand-over points of its first TRACE_UNITS units
#endif
};

#ifdef SPFY_DEV_SWITCHES
constexpr uint32_t TRACE_UNITS = 24, TRACE_SLOTS = 8;  // [role 0 producer / 1 MMA / 2 epilogue warp 2][unit][slot]
#define SPFY_TRACE(role, unit, slot)                                                                     \
  do {                                                                                                   \
    if (L.trace && blockIdx.x == 0 && (unit) < TRACE_UNITS && (threadIdx.x & 31u) == 0u)                 \
      L.trace[((role) * TRACE_UNITS + (unit)) * TRACE_SLOTS + (slot)] = clock64();                       \
  } while (0)
#else
#define SPFY_TRACE(role, unit, slot) do { } while (0)
#endif

using namespace ptx;

__device__ __forceinline__ uint32_t rows_valid_of(uint32_t m, uint32_t mt) {
  const uint32_t left = m - mt * BM;
  return left >= (uint32_t)BM ? (uint32_t)BM : ((left + 15u) & ~15u);
}


// GELU, tanh form (torch's gelu(approximate="tanh")): one tanh.approx per value on the MUFU pipe
__device__ __forceinline__ float gelu_tanh(float x) {
  float t;
  asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(0.7978845608028654f * fmaf(0.044715f * x, x * x, x)));
  return 0.5f * x * (1.f + t);
}

// scattered output: the D (or C) row of position n of the problem's [batch][conv_ho][conv_wo] grid
__device__ __forceinline__ size_t scatter_row(const ProblemDev* P, uint32_t n) {
  const uint32_t t = n / P->conv_wo, j = n - t * P->conv_wo, img = t / P->conv_ho, i = t - img * P->conv_ho;
  return ((size_t)img * P->sc_h + P->sc_s * i + P->sc_a) * P->sc_w + P->sc_s * j + P->sc_b;
}

// All three roles walk the same sequence of units: u = blockIdx.x, blockIdx.x + gridDim.x, ...
// The walker keeps the unit's position inside its problem -- (n-tile, m-group) -> first m-tile and m-tiles of the unit --
// INCREMENTALLY: the stride gridDim is split once per problem into a quotient and a remainder by m_groups, so a step
// costs two additions and a wrap instead of a division, and the problem table is only read when a unit leaves the
// cached range of the current problem.  (Measured with SPFY_SPMMA_TRACE on the k <= 64 class: the issuing warps spent
// ~800 of ~1900 cycles per unit between units.)
struct UnitWalker {
  const ProblemDev* single;
  const ProblemDev* table;
  uint32_t num_problems, total_units;
  uint32_t u, p;
  uint32_t p_begin, p_end;                 // unit range of problem p
  uint32_t m_groups, G, m_tiles, split_units, split_nt, step_q, step_r;
  uint32_t nt, mg, mt0, g_count;           // decoded position of unit u
  bool changed;                            // the problem changed since the caller last looked
  __device__ __forceinline__ UnitWalker(const ProblemDev* s, const LaunchParams& L)
      : single(s), table(L.table), num_problems(L.num_problems), total_units(L.total_units),
        u(blockIdx.x), p(0), p_begin(0), p_end(0), changed(false) {
    if (valid()) enter();
  }
  __device__ __forceinline__ const ProblemDev* prob(uint32_t i) const { return table ? table + i : single; }
  __device__ __forceinline__ bool valid() const { return u < total_units; }
  __device__ __forceinline__ const ProblemDev* current() const { return prob(p); }
  // by division: on entering a problem, and in the split tail of a single call (the last, partial wave dealt one
  // m-tile per unit, see split_tail)
  __device__ __forceinline__ void decode(uint32_t local) {
    if (local < split_units) {
      nt = local / m_groups;
      mg = local - nt * m_groups;
      mt0 = mg * G;
      g_count = min(G, m_tiles - mt0);
    } else {
      const uint32_t l2 = local - split_units, q = l2 / m_tiles;
      nt = split_nt + q;
      mt0 = l2 - q * m_tiles;
      mg = mt0 / G;
      g_count = 1u;
    }
  }
  // units are visited in increasing order, so p only advances
  __device__ __forceinline__ void enter() {
    while (p + 1 < num_problems && u >= prob(p)->unit_begin + prob(p)->units) ++p;
    p = uni(p);  // the table reads above hide from the compiler that every lane took the same path
    const ProblemDev* P = prob(p);
    p_begin = uni(P->unit_begin);
    p_end = p_begin + uni(P->units);
    m_groups = uni(P->m_groups); G = uni(P->G); m_tiles = uni(P->m_tiles);
    split_units = uni(P->split_units); split_nt = uni(P->split_nt);
    step_q = gridDim.x / m_groups;
    step_r = gridDim.x - step_q * m_groups;
    decode(u - p_begin);
    changed = true;
  }
  __device__ __forceinline__ void next() {
    u += gridDim.x;
    if (u >= total_units) return;
    if (u >= p_end) {
      enter();
      return;
    }
    const uint32_t local = u - p_begin;
    if (local < split_units) {
      nt += step_q;
      mg += step_r;
      if (mg >= m_groups) {
        mg -= m_groups;
        ++nt;
      }
      mt0 = mg * G;
      g_count = min(G, m_tiles - mt0);
    } else {
      decode(local);
    }
  }
};

// ------------------------------------------------------------------- kernel
// EPI: some problem of the launch has an epilogue (ProblemDev::epi).  A launch without one compiles to the code the kernel
// had before epilogues existed (152 registers instead of 168, measured 0.3-1 % faster on the ResNet-50 plans).
// SCATTER: the transposed output goes to scattered rows (ProblemDev::D, spfy_spmma_conv_dgrad); only with OPB_T and EPI.
template <bool BF16, bool OPB_T, bool EPI, bool SCATTER>
__global__ void __launch_bounds__(NUM_THREADS, 1)
spmma_kernel(const __grid_constant__ ProblemDev single, const __grid_constant__ LaunchParams L) {
  extern __shared__ uint8_t smem_raw[];
  const uint32_t smem_base = (smem_u32(smem_raw) + 1023u) & ~1023u;
  uint8_t* smem_gen = smem_raw + (smem_base - smem_u32(smem_raw));
  const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

  const uint32_t NS = L.stages;
  const uint32_t bar_full = smem_base + L.bar_off;              // [MAX_STAGES]
  const uint32_t bar_empty = bar_full + MAX_STAGES * 8;         // [MAX_STAGES]
  const uint32_t bar_acc_full = bar_empty + MAX_STAGES * 8;     // [ACC_SLOTS]
  const uint32_t bar_acc_empty = bar_acc_full + ACC_SLOTS * 8;  // [ACC_SLOTS]
  const uint32_t bar_res_full = bar_acc_empty + ACC_SLOTS * 8;
  const uint32_t bar_res_empty = bar_res_full + 8;
  const uint32_t tmem_ptr_off = L.bar_off + (2 * MAX_STAGES + 2 * ACC_SLOTS + 2) * 8;
  volatile uint32_t* tmem_ptr_smem = reinterpret_cast<volatile uint32_t*>(smem_gen + tmem_ptr_off);

  // The launches of a plan are independent problems issued back to back with programmatic stream
  // serialization: letting the next launch's CTAs in as soon as ours retire overlaps its ramp-up with
  // our tail (there is no data dependence between them; griddepcontrol.wait is only issued at the very end,
  // to keep completion transitive).
  if (threadIdx.x == 0) asm volatile("griddepcontrol.launch_dependents;" ::: "memory");
  if (warp == 1 && lane == 0) {
    for (uint32_t s = 0; s < (uint32_t)MAX_STAGES; ++s) {
      mbar_init(bar_full + s * 8, 1);
      mbar_init(bar_empty + s * 8, 1);
    }
    for (int a = 0; a < ACC_SLOTS; ++a) {
      mbar_init(bar_acc_full + a * 8, 1);
      mbar_init(bar_acc_empty + a * 8, L.epi_warps);  // every active epilogue warp reads a part of every job
    }
    mbar_init(bar_res_full, 1);
    mbar_init(bar_res_empty, 1);
    fence_barrier_init();
  }
  if (warp == 2) tmem_alloc(smem_base + tmem_ptr_off, TMEM_COLS);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_ptr_smem;

  UnitWalker W(&single, L);
  // NOTE on the role loops: every PTX wrapper is an `asm volatile` with a "memory" clobber, so
  // anything read through a pointer inside a loop is re-loaded on every trip.  The single-thread
  // producer / MMA loops are latency-bound scalar code, so all per-problem and per-unit state is
  // copied into registers first and the ring position is advanced without divisions.

  if (warp == 0) {
    // ===================== producer (whole warp, one lane issues) =====================
    {
      const bool leader = elect_one();
      uint32_t stage = 0, phase = 0;  // ring position (continuous over units)
      uint32_t res_loads = 0;         // resident (re)loads issued so far
      const ProblemDev* res_owner = nullptr;
      uint32_t res_mg = 0;            // ... and the m-group they hold (sliced residency)
      const CUtensorMap* tmap_b = nullptr;
      const uint8_t *a_vals = nullptr, *a_meta = nullptr;
      uint32_t pm = 0, k_tiles = 0, m_tiles = 0, G = 1, resident = 0, b3d = 0;
      uint32_t conv = 0, conv_c = 64, conv_kw = 1, conv_wo = 1, conv_ho = 1, conv_stride = 1, pk = 0;
      int conv_off_h = 0, conv_off_w = 0;
      uint64_t hint_b = 0;
      const bool no_b = (L.dbg & 4u) != 0, no_a = (L.dbg & 16u) != 0;
      uint32_t tr_unit = 0;
      (void)tr_unit;
      for (; W.valid(); W.next()) {
        const ProblemDev* P = W.current();
        if (W.changed) {
          W.changed = false;
          tmap_b = &P->tmap_b;
          if (leader) prefetch_tmap(tmap_b);
          a_vals = uni(P->a_vals); a_meta = uni(P->a_meta);
          pm = uni(P->m); k_tiles = uni(P->k_tiles); m_tiles = W.m_tiles; b3d = uni(P->b3d);
          G = W.G; resident = uni(P->resident);
          hint_b = uni(P->hint_b);
          conv = uni(P->conv); pk = uni(P->k);
          if (conv) {
            conv_c = uni(P->conv_c); conv_kw = uni(P->conv_kw); conv_wo = uni(P->conv_wo); conv_ho = uni(P->conv_ho);
            conv_stride = uni(P->conv_stride); conv_off_h = (int)uni((uint32_t)P->conv_off_h);
            conv_off_w = (int)uni((uint32_t)P->conv_off_w);
          }
        }
        const uint32_t nt = W.nt, mt0 = W.mt0, g_count = W.g_count, mg = W.mg;
        // implicit GEMM: base pixel of the unit's first output position (input coordinates of filter tap (0, 0))
        int cw = 0, ch = 0, cn = 0;
        if (conv) {
          const uint32_t p0 = nt * (uint32_t)BN, row = p0 / conv_wo;
          cw = (int)((p0 - row * conv_wo) * conv_stride) + conv_off_w;
          cn = (int)(row / conv_ho);
          ch = (int)((row - (uint32_t)cn * conv_ho) * conv_stride) + conv_off_h;
        }
        // the G tiles of a k-tile are adjacent in the operand, so one copy per array fetches a group's share of it
        const uint32_t rv0 = rows_valid_of(pm, mt0);
        const uint32_t rv1 = g_count > 1 ? rows_valid_of(pm, mt0 + 1) : 0u;
        const uint32_t a_bytes = g_count > 1 ? (uint32_t)A_TILE_BYTES + rv1 * 128u : rv0 * 128u;
        const uint32_t e_bytes = g_count > 1 ? (uint32_t)E_TILE_BYTES + rv1 * 16u : rv0 * 16u;
        const uint32_t res_key = resident == 2u ? mg : 0u;
        if (resident && (res_owner != P || res_mg != res_key)) {
          // (re)load the compressed A of this problem (or of this m-group of it) into the resident region
          mbar_wait(bar_res_empty, (res_loads & 1u) ^ 1u);
          if (leader) {
            if (resident == 2u) {
              // m-group slice: k-tile kt of the group at kt * G tiles
              mbar_expect_tx(bar_res_full, k_tiles * (a_bytes + e_bytes));
              for (uint32_t kt = 0; kt < k_tiles; ++kt) {
                bulk_load_1d(smem_base + L.res_off + kt * G * (uint32_t)A_TILE_BYTES,
                             a_vals + ((size_t)kt * m_tiles + mt0) * A_TILE_BYTES, a_bytes, bar_res_full, HINT_EVICT_LAST);
                bulk_load_1d(smem_base + L.res_e_off + kt * G * (uint32_t)E_TILE_BYTES,
                             a_meta + ((size_t)kt * m_tiles + mt0) * E_TILE_BYTES, e_bytes, bar_res_full, HINT_EVICT_LAST);
              }
            } else if (m_tiles == 1) {
              // a single, possibly short, m-tile: compact rows, one copy per k-tile and array
              const uint32_t rv = rows_valid_of(pm, 0);
              mbar_expect_tx(bar_res_full, k_tiles * rv * 144u);
              for (uint32_t kt = 0; kt < k_tiles; ++kt) {
                bulk_load_1d(smem_base + L.res_off + kt * rv * 128u, a_vals + (size_t)kt * A_TILE_BYTES, rv * 128u,
                             bar_res_full, HINT_EVICT_LAST);
                bulk_load_1d(smem_base + L.res_e_off + kt * rv * 16u, a_meta + (size_t)kt * E_TILE_BYTES, rv * 16u,
                             bar_res_full, HINT_EVICT_LAST);
              }
            } else {
              // the arrays are contiguous (padding rows included): two copies fetch everything
              const uint32_t tiles = k_tiles * m_tiles;
              mbar_expect_tx(bar_res_full, tiles * (uint32_t)(A_TILE_BYTES + E_TILE_BYTES));
              bulk_load_1d(smem_base + L.res_off, a_vals, tiles * A_TILE_BYTES, bar_res_full, HINT_EVICT_LAST);
              bulk_load_1d(smem_base + L.res_e_off, a_meta, tiles * E_TILE_BYTES, bar_res_full, HINT_EVICT_LAST);
            }
          }
          res_owner = P;
          res_mg = res_key;
          ++res_loads;
        }
        const uint8_t* av = a_vals + (size_t)mt0 * A_TILE_BYTES;
        const uint8_t* am = a_meta + (size_t)mt0 * E_TILE_BYTES;
        const size_t av_step = (size_t)m_tiles * A_TILE_BYTES, am_step = (size_t)m_tiles * E_TILE_BYTES;
        const bool stream_a = !resident && !no_a;
        const uint32_t tx_a = stream_a ? a_bytes + e_bytes : 0u;
        const uint32_t tx_full = (no_b ? 0u : L.bk * (uint32_t)(BN * 2)) + tx_a;
        // implicit GEMM: (channel offset, filter column, filter row) of the next 64-channel piece, stepped without
        // divisions (the two per piece that stood here made the producer the slowest warp of every convolution layer:
        // ~1340 cycles per k-tile, ncu stall samples spread evenly over its scalar code)
        uint32_t pc0 = 0, pts = 0, ptr = 0;
        for (uint32_t kt = 0; kt < k_tiles; ++kt, av += av_step, am += am_step) {
          if (kt == 0) SPFY_TRACE(0, tr_unit, 0);
          mbar_wait(bar_empty + stage * 8, phase ^ 1u);
          if (kt == 0) SPFY_TRACE(0, tr_unit, 1);
          const uint32_t full = bar_full + stage * 8;
          const uint32_t sbase = smem_base + stage * L.stage_bytes;
          // implicit GEMM: 64-channel pieces of this k-tile that exist (K = taps * C is a multiple of 64, not of 128)
          const uint32_t pieces = conv ? min(L.bk / 64u, (pk - kt * L.bk + 63u) / 64u) : 0u;
          const uint32_t tx = conv && !no_b ? pieces * (uint32_t)(BN * 128) + tx_a : tx_full;
          if (leader) {
            if (tx) mbar_expect_tx(full, tx); else mbar_arrive(full);
            // B first: it comes from DRAM and is the long pole of the stage; A and its metadata are L2 hits
            if (no_b) {
            } else if (conv) {
              if (OPB_T) {
                // (the leader issues; every lane steps the position below.  At most two pieces per stage.)
                tma_load_im2col_4d(sbase, tmap_b, (int)pc0, cw, ch, cn, (uint16_t)pts, (uint16_t)ptr, full, hint_b);
                if (pieces > 1u) {
                  uint32_t c0 = pc0 + 64u, ts = pts, tr = ptr;
                  if (c0 == conv_c) {
                    c0 = 0;
                    if (++ts == conv_kw) { ts = 0; ++tr; }
                  }
                  tma_load_im2col_4d(sbase + (uint32_t)(BN * 128), tmap_b, (int)c0, cw, ch, cn, (uint16_t)ts, (uint16_t)tr,
                                     full, hint_b);
                }
              }
            } else if (b3d) {
              // one box fills the stage: [2 groups of 64][128 outer rows][64]
              if (!OPB_T) tma_load_3d(sbase, tmap_b, 0, (int)(kt * BK), (int)(nt * 2), full, hint_b);
              else        tma_load_3d(sbase, tmap_b, 0, (int)(nt * BN), (int)(kt * 2), full, hint_b);
            } else if (!OPB_T) {
              // B is k x n row-major: boxes of [128 rows of k][64 columns of n] -> MN-major SW128
              tma_load_2d(sbase, tmap_b, (int)(nt * BN), (int)(kt * BK), full, hint_b);
              tma_load_2d(sbase + L.bk * 128u, tmap_b, (int)(nt * BN + 64), (int)(kt * BK), full, hint_b);
            } else {
              // B is n x k row-major: boxes of [128 rows of n][64 columns of k] -> K-major SW128
              tma_load_2d(sbase, tmap_b, (int)(kt * BK), (int)(nt * BN), full, hint_b);
              if (L.bk == (uint32_t)BK) tma_load_2d(sbase + BN * 128, tmap_b, (int)(kt * BK + 64), (int)(nt * BN), full, hint_b);
            }
            if (stream_a) {
              bulk_load_1d(sbase + L.a_off, av, a_bytes, full, HINT_EVICT_LAST);
              bulk_load_1d(sbase + L.e_off, am, e_bytes, full, HINT_EVICT_LAST);
            }
          }
#pragma unroll
          for (uint32_t h = 0; h < 2u; ++h) {
            if (h < pieces) {
              pc0 += 64u;
              if (pc0 == conv_c) {
                pc0 = 0;
                if (++pts == conv_kw) { pts = 0; ++ptr; }
              }
            }
          }
          if (++stage == NS) { stage = 0; phase ^= 1u; }
        }
        SPFY_TRACE(0, tr_unit, 2);
        ++tr_unit;
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer (whole warp, one lane issues) =====================
    {
      const bool leader = elect_one();
      const uint32_t tmem_b = uni(tmem_base);
      uint32_t stage = 0, phase = 0, eblk = 0, res_loads = 0, res_mg = 0;
      uint32_t acc_slot = 0, acc_par = 0;  // accumulator slot of the next job and the parity of its use count
      const ProblemDev* res_owner = nullptr;
      uint32_t pm = 0, pk = 0, k_tiles = 0, m_tiles = 0, G = 1, resident = 0;
      const bool no_mma = (L.dbg & 8u) != 0;
      uint32_t tr_unit = 0;
      (void)tr_unit;
      // constant halves of the shared-memory descriptors (the start address is OR-ed in per MMA)
      const uint64_t desc_a_hi = make_smem_desc(0, 16, 1024, LAYOUT_SW128);
      const uint64_t desc_b_hi = OPB_T ? make_smem_desc(0, 16, 1024, LAYOUT_SW128)
                                       : make_smem_desc(0, L.bk * 128u, 1024, LAYOUT_SW128);
      const uint64_t desc_e_hi = make_smem_desc(0, 16, 128, LAYOUT_NONE);
      for (; W.valid(); W.next()) {
        const ProblemDev* P = W.current();
        if (W.changed) {
          W.changed = false;
          pm = uni(P->m); pk = uni(P->k); k_tiles = uni(P->k_tiles); m_tiles = W.m_tiles;
          G = W.G; resident = uni(P->resident);
        }
        const uint32_t mt0 = W.mt0, g_count = W.g_count, mg = W.mg;
        const uint32_t res_key = resident == 2u ? mg : 0u;
        if (resident && (res_owner != P || res_mg != res_key)) {
          mbar_wait(bar_res_full, res_loads & 1u);
          res_owner = P;
          res_mg = res_key;
          ++res_loads;
        }
        // accumulator slots of this unit's jobs (ring of ACC_SLOTS, advanced without divisions)
        const uint32_t slot0 = acc_slot, par0 = acc_par;
        if (++acc_slot == (uint32_t)ACC_SLOTS) { acc_slot = 0; acc_par ^= 1u; }
        const uint32_t slot1 = acc_slot, par1 = acc_par;
        if (g_count > 1) {
          if (++acc_slot == (uint32_t)ACC_SLOTS) { acc_slot = 0; acc_par ^= 1u; }
        }
        SPFY_TRACE(1, tr_unit, 0);
        mbar_wait(bar_acc_empty + slot0 * 8, par0 ^ 1u);
        if (g_count > 1) mbar_wait(bar_acc_empty + slot1 * 8, par1 ^ 1u);
        tc_fence_after();
        SPFY_TRACE(1, tr_unit, 1);
        const uint32_t tmem_d0 = tmem_b + slot0 * BN, tmem_d1 = tmem_b + slot1 * BN;
        // resident operands: tile (kt, mt) at (kt*m_tiles + mt) * stride
        const uint32_t rv_single = rows_valid_of(pm, 0);
        const uint32_t rsv = m_tiles == 1 ? rv_single * 128u : (uint32_t)A_TILE_BYTES;
        const uint32_t rse = m_tiles == 1 ? rv_single * 16u : (uint32_t)E_TILE_BYTES;
        // (a slice holds the G tiles of its m-group only)
        const uint32_t res_first = resident == 2u ? 0u : mt0, res_tiles = resident == 2u ? G : m_tiles;
        uint32_t ra = smem_base + L.res_off + res_first * rsv, re = smem_base + L.res_e_off + res_first * rse;
        uint32_t k_left = pk;
        for (uint32_t kt = 0; kt < k_tiles; ++kt, k_left -= BK, ra += res_tiles * rsv, re += res_tiles * rse) {
          mbar_wait(bar_full + stage * 8, phase);
          tc_fence_after();
          if (kt == 0) SPFY_TRACE(1, tr_unit, 2);
          const uint32_t sbase = smem_base + stage * L.stage_bytes;
          // metadata of these 128 logical k -> TMEM (4 columns per m-tile)
          const uint32_t ecol0 = tmem_b + TMEM_E_COL + (eblk & 1u) * (MAX_G * 4u), ecol1 = ecol0 + 4u;
          ++eblk;
          const uint32_t e0 = resident ? re : sbase + L.e_off;
          const uint32_t sa0 = resident ? ra : sbase + L.a_off;
          const uint32_t sa1 = sa0 + (resident ? rsv : (uint32_t)A_TILE_BYTES);
          const uint32_t e1 = e0 + (resident ? rse : (uint32_t)E_TILE_BYTES);
          const uint32_t nk = k_left >= (uint32_t)BK ? 4u : (k_left + 31u) / 32u;
          // Descriptor start addresses in 16-byte units (shared memory < 256 KiB: they fit the 14-bit field and
          // adding the per-MMA step cannot carry out of it), so every operand below is "base + constant":
          //   A: K-major SW128, 32 logical k = 16 stored halves = 32 bytes per MMA              -> +2 per j
          //   B: MN-major SW128 (8 k-rows per 1024 B atom): 32 k-rows = 4096 bytes per MMA      -> +256 per j
          //      K-major SW128 (opB = T): two 64-wide k halves BN*128 bytes apart, 64 B per MMA  -> (j>>1)*1024 + (j&1)*4
          //   metadata: TMEM columns ecol + (j & 2), instruction-descriptor selector bit j & 1 (ecol is even)
          const uint32_t a0 = (sa0 >> 4) & 0x3fffu, a1 = (sa1 >> 4) & 0x3fffu, b0 = (sbase >> 4) & 0x3fffu;
          const bool two = g_count > 1;
          if (leader) {
            tc_cp_128x128b(ecol0, desc_e_hi | (uint64_t)((e0 >> 4) & 0x3fffu));
            if (two) tc_cp_128x128b(ecol1, desc_e_hi | (uint64_t)((e1 >> 4) & 0x3fffu));
            if (!no_mma) {
#pragma unroll
              for (uint32_t j = 0; j < 4; ++j) {
                if (j < nk) {
                  const uint32_t bj = OPB_T ? b0 + (j >> 1) * (uint32_t)(BN * 128 / 16) + (j & 1u) * 4u : b0 + j * 256u;
                  const uint64_t db = desc_b_hi | (uint64_t)bj;
                  const uint32_t first = j ? 1u : kt;  // accumulate except for the very first MMA of the unit
                  tc_mma_sp_f16(tmem_d0, desc_a_hi | (uint64_t)(a0 + 2u * j), db, ecol0 + (j & 2u), L.idesc | (j & 1u), first);
                  if (two)
                    tc_mma_sp_f16(tmem_d1, desc_a_hi | (uint64_t)(a1 + 2u * j), db, ecol1 + (j & 2u), L.idesc | (j & 1u), first);
                }
              }
            }
            tc_commit(bar_empty + stage * 8);
          }
          if (++stage == NS) { stage = 0; phase ^= 1u; }
        }
        // last use of what the resident region holds: the CTA's next unit is another problem's, or another m-group's
        const uint32_t nu = W.u + gridDim.x;
        const bool last_of_problem = resident && (nu >= L.total_units || nu >= W.p_end || (resident == 2u && W.step_r != 0u));
        if (leader) {
          tc_commit(bar_acc_full + slot0 * 8);
          if (g_count > 1) tc_commit(bar_acc_full + slot1 * 8);
          if (last_of_problem) tc_commit(bar_res_empty);  // every MMA that reads the resident region has completed
        }
        SPFY_TRACE(1, tr_unit, 3);
        ++tr_unit;
        if (last_of_problem) res_owner = nullptr;
      }
    }
  } else if (warp - 2 < L.epi_warps) {
    // ===================== epilogue (warps 2..9, or 2..5 doing both column halves) =====================
    const uint32_t e = warp - 2;
    const uint32_t quarter = warp & 3u;  // TMEM lanes this warp may read: [32*quarter, 32*quarter+32)
    const uint32_t halves = L.epi_warps == (uint32_t)NUM_EPI_WARPS ? 1u : 2u;
    const uint32_t half0 = halves == 1u ? (e >> 2) : 0u;
    const uint32_t row_in_tile = quarter * 32 + lane;
    const uint32_t sc = smem_base + L.c_off + e * C_BUF_BYTES;
    const uint32_t st_base = sc + lane * 128;
    const uint32_t sw = lane & 7u;
    const bool no_epi = (L.dbg & 2u) != 0, no_store = (L.dbg & 32u) != 0;
    uint32_t job = 0, acc_slot = 0, acc_par = 0;
    (void)job;
    const CUtensorMap* tmap_d = nullptr;
    const CUtensorMap* tmap_rep = nullptr;
    uint32_t n_rep = 0, out_t = 0;
    const uint16_t* Cptr = nullptr;
    uint64_t ldc = 0;
    uint32_t pm = 0, pn = 0;
    float alpha = 1.f, beta = 0.f;
    float alpha_t = 1.f;  // the factor the transposed staging loop applies: 1 once the epilogue has applied alpha
    const float* scale = nullptr;
    const float* bias = nullptr;
    uint32_t act = 0, epi = 0;
    for (; W.valid(); W.next()) {
      const ProblemDev* P = W.current();
      if (W.changed) {
        W.changed = false;
        tmap_d = &P->tmap_d;
        tmap_rep = P->tmap_rep;
        n_rep = P->n_rep;
        out_t = P->out_t;
        Cptr = reinterpret_cast<const uint16_t*>(P->C);
        ldc = P->ldc;
        pm = P->m; pn = P->n;
        alpha = P->alpha; beta = P->beta;
        if (EPI) {
          scale = P->scale; bias = P->bias; act = P->act; epi = P->epi;
        }
        alpha_t = epi ? 1.f : alpha;
      }
      const uint32_t nt = W.nt, mt0 = W.mt0, g_count = W.g_count;
      for (uint32_t g = 0; g < g_count; ++g, ++job) {
        const uint32_t slot = acc_slot, par = acc_par;
        if (++acc_slot == (uint32_t)ACC_SLOTS) { acc_slot = 0; acc_par ^= 1u; }
        const uint32_t m0 = (mt0 + g) * BM;
        if (e == 0) SPFY_TRACE(2, job, 0);
        mbar_wait(bar_acc_full + slot * 8, par);
        tc_fence_after();
        if (e == 0) SPFY_TRACE(2, job, 1);
        for (uint32_t hh = 0; hh < halves; ++hh) {
          const uint32_t half = half0 + hh;
          const uint32_t n0 = nt * BN + half * 64;
          const bool warp_has_rows = m0 + quarter * 32 < pm && n0 < pn;
          uint32_t acc[64];
          if (warp_has_rows) {
            const uint32_t taddr = tmem_base + slot * BN + half * 64 + ((quarter * 32) << 16);
            tmem_ld_x32(taddr, acc);
            tmem_ld_x32(taddr + 32, acc + 32);
            tmem_wait_ld();
          }
          if (hh + 1 == halves) {
            // accumulator fully read by this warp: hand the slot back to the MMA warp
            tc_fence_before();
            __syncwarp();
            if (lane == 0) mbar_arrive(bar_acc_empty + slot * 8);
            if (e == 0) SPFY_TRACE(2, job, 2);
          }
          if (warp_has_rows && !no_epi) {
            if (lane == 0) bulk_wait_read_all();  // my previous store has finished reading the staging buffer
            __syncwarp();
            if (e == 0 && hh == 0) SPFY_TRACE(2, job, 3);
            const uint32_t grow = m0 + row_in_tile;
            if (epi) {
              // the epilogue, in place on the accumulators: v = (alpha * scale[row]) * acc + beta * C + bias[row], then
              // the activation; the staging below only converts.  A missing bias adds -0, which leaves every value as it is.
              const bool row_ok = grow < pm;
              const float as = scale && row_ok ? alpha * scale[grow] : alpha;
              const float bs = bias && row_ok ? bias[grow] : -0.f;
              if (beta != 0.f && out_t) {
                // C is [n][m] like D: the warp copies its (64 n x 32 m) box of C into its staging buffer -- the geometry
                // of the store box, 64 contiguous bytes per n -- with 16-byte asynchronous copies that bypass the
                // registers, and every lane then reads its own column of it, where the staging loop below writes the
                // result.  (Halfword loads of C into registers spill at the 168 registers this CTA shape allows.)
                const uint32_t mc = m0 + quarter * 32 + (lane & 3u) * 8;  // m % 8 == 0: these 8 m are all in or all out
                const uint32_t r0 = lane >> 2, n_in = mc < pm ? pn - n0 : 0u;   // rows r0, r0 + 8, ... of the box
                const uint16_t* src = Cptr + (size_t)(n0 + r0) * ldc + mc;
                const uint32_t dst = sc + r0 * 64u + (lane & 3u) * 16u;
                if (SCATTER) {
                  for (uint32_t i = 0; i < 8; ++i) {
                    const bool in = r0 + 8 * i < n_in;
                    cp_async_16(dst + i * 512u, in ? Cptr + scatter_row(P, n0 + r0 + 8 * i) * ldc + mc : Cptr, in);
                  }
                } else {
#pragma unroll
                  for (uint32_t i = 0; i < 8; ++i, src += 8 * ldc)
                    cp_async_16(dst + i * 512u, r0 + 8 * i < n_in ? src : Cptr, r0 + 8 * i < n_in);
                }
                cp_async_wait_all();
                __syncwarp();
#pragma unroll
                for (int j = 0; j < 64; ++j) {
                  const float c = unpack2<BF16>(ld_shared_u16(sc + (uint32_t)j * 64u + lane * 2u)).x;
                  acc[j] = __float_as_uint(__fadd_rn(__fmaf_rn(beta, c, __fmul_rn(as, __uint_as_float(acc[j]))), bs));
                }
              } else if (beta != 0.f && row_ok) {
                {
#pragma unroll
                  for (int q = 0; q < 8; ++q) {
                    float v[8];
#pragma unroll
                    for (int x = 0; x < 8; ++x) v[x] = __fmul_rn(as, __uint_as_float(acc[q * 8 + x]));
                    if (n0 + q * 8 < pn) {
                      const uint4 cw = *reinterpret_cast<const uint4*>(Cptr + (size_t)grow * ldc + n0 + q * 8);
                      const uint32_t cws[4] = {cw.x, cw.y, cw.z, cw.w};
#pragma unroll
                      for (int x = 0; x < 4; ++x) {
                        const float2 f = unpack2<BF16>(cws[x]);
                        v[2 * x] = __fmaf_rn(beta, f.x, v[2 * x]);
                        v[2 * x + 1] = __fmaf_rn(beta, f.y, v[2 * x + 1]);
                      }
                    }
#pragma unroll
                    for (int x = 0; x < 8; ++x) acc[q * 8 + x] = __float_as_uint(__fadd_rn(v[x], bs));
                  }
                }
              } else {
#pragma unroll
                for (int j = 0; j < 64; ++j) acc[j] = __float_as_uint(__fadd_rn(__fmul_rn(as, __uint_as_float(acc[j])), bs));
              }
              if (act == SPFY_ACT_RELU) {
#pragma unroll
                for (int j = 0; j < 64; ++j) acc[j] = __float_as_uint(fmaxf(__uint_as_float(acc[j]), 0.f));
              } else if (act == SPFY_ACT_GELU_TANH) {
#pragma unroll
                for (int j = 0; j < 64; ++j) acc[j] = __float_as_uint(gelu_tanh(__uint_as_float(acc[j])));
              }
            }
            if (out_t) {
              // transposed output [n][m]: the staging buffer holds 64 rows (n) of 32 halfwords (my quarter's m), so a
              // lane -- one m -- drops column j of its 64 into row j; C (beta != 0) only through the epilogue above
#pragma unroll
              for (int j = 0; j < 32; ++j) {
                const uint32_t w = pack2<BF16>(alpha_t * __uint_as_float(acc[2 * j]), alpha_t * __uint_as_float(acc[2 * j + 1]));
                st_shared_u16(sc + (uint32_t)(2 * j) * 64u + lane * 2u, w);
                st_shared_u16(sc + (uint32_t)(2 * j + 1) * 64u + lane * 2u, w >> 16);
              }
            } else if (epi || (alpha == 1.f && beta == 0.f)) {
              // the common case (the reference's defaults, spmma.hxx:32-33), or values the epilogue has finished:
              // convert and stage, nothing else.
              // Kept apart from the general path: predicated-off C loads / FMAs still cost issue slots, and
              // with two epilogue warps per scheduler the conversion loop is what bounds the small-K classes.
#pragma unroll
              for (int q = 0; q < 8; ++q)
                st_shared_v4(st_base + ((q ^ sw) << 4),
                             pack2<BF16>(__uint_as_float(acc[q * 8 + 0]), __uint_as_float(acc[q * 8 + 1])),
                             pack2<BF16>(__uint_as_float(acc[q * 8 + 2]), __uint_as_float(acc[q * 8 + 3])),
                             pack2<BF16>(__uint_as_float(acc[q * 8 + 4]), __uint_as_float(acc[q * 8 + 5])),
                             pack2<BF16>(__uint_as_float(acc[q * 8 + 6]), __uint_as_float(acc[q * 8 + 7])));
            } else {
              const bool use_c = beta != 0.f && grow < pm;
#pragma unroll
              for (int q = 0; q < 8; ++q) {
                float v[8];
#pragma unroll
                for (int x = 0; x < 8; ++x) v[x] = alpha * __uint_as_float(acc[q * 8 + x]);
                if (use_c && n0 + q * 8 < pn) {
                  const uint4 cw = *reinterpret_cast<const uint4*>(Cptr + (size_t)grow * ldc + n0 + q * 8);
                  const uint32_t cws[4] = {cw.x, cw.y, cw.z, cw.w};
#pragma unroll
                  for (int x = 0; x < 4; ++x) {
                    const float2 f = unpack2<BF16>(cws[x]);
                    v[2 * x] += beta * f.x;
                    v[2 * x + 1] += beta * f.y;
                  }
                }
                st_shared_v4(st_base + ((q ^ sw) << 4), pack2<BF16>(v[0], v[1]), pack2<BF16>(v[2], v[3]),
                             pack2<BF16>(v[4], v[5]), pack2<BF16>(v[6], v[7]));
              }
            }
            fence_proxy_async_smem();
            __syncwarp();
            if (SCATTER) {
              // a staging row (64 bytes: 32 channels of one position) lands at the position's scattered row of D; lane l
              // moves the 8 channels (l & 3) of rows l >> 2, + 8, ...  (m % 8 == 0: those 8 channels are all in or all out)
              const uint32_t mc = m0 + quarter * 32 + (lane & 3u) * 8, r0 = lane >> 2;
              uint16_t* D = reinterpret_cast<uint16_t*>(P->D);
              const uint64_t ldd = P->ldd;
              if (mc < pm && !no_store) {
                for (uint32_t i = 0; i < 8; ++i) {
                  const uint32_t r = r0 + 8 * i;
                  if (n0 + r < pn)
                    *reinterpret_cast<uint4*>(D + scatter_row(P, n0 + r) * ldd + mc) = ld_shared_v4(sc + r * 64u + (lane & 3u) * 16u);
                }
              }
            } else if (lane == 0 && !no_store) {
              // (coordinates are (inner, outer): (n, m) for the row-major output, (m, n) for the transposed one)
              const int c0 = out_t ? (int)(m0 + quarter * 32) : (int)n0, c1 = out_t ? (int)n0 : (int)(m0 + quarter * 32);
              tma_store_2d(tmap_d, sc, c0, c1);
              for (uint32_t r = 0; r < n_rep; ++r) tma_store_2d(tmap_rep + r, sc, c0, c1);
              bulk_commit();
            }
            if (e == 0 && hh == 0) SPFY_TRACE(2, job, 4);
          }
        }
      }
    }
    if (lane == 0) bulk_wait_all();
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 2) {
    tc_fence_after();
    tmem_dealloc(tmem_base, TMEM_COLS);
  }
  // Completion must be transitive along a plan's chain of programmatic launches: this grid may have started while
  // its predecessor's tail was still running, so one thread waits for the predecessor before the CTA retires (all
  // the work is done by now, the ramp-up overlap is kept; a no-op for launches without the attribute).  Whatever
  // is enqueued after spfy_spmma_plan_run therefore sees every launch of the plan finished.
  if (threadIdx.x == 0) asm volatile("griddepcontrol.wait;" ::: "memory");
}

// ------------------------------------------------------------- host side
// 2-D row-major tensor [outer x inner] of 16-bit elements, pitch ld elements
int make_tmap_2d(CUtensorMap* map, int dtype, const void* base, uint64_t inner, uint64_t outer,
                 uint64_t ld, uint32_t box_inner, uint32_t box_outer,
                 CUtensorMapSwizzle swizzle = CU_TENSOR_MAP_SWIZZLE_128B) {
  const cuuint64_t dims[2] = {inner, outer}, strides[1] = {ld * 2};
  const cuuint32_t box[2] = {box_inner, box_outer};
  return encode_tiled(map, dtype, 2, base, dims, strides, box, swizzle, "spmma");
}

// The same matrix (inner % 64 == 0) viewed as [inner/64 groups][outer][64]: a box of
// (64, box_outer, 2) lands in shared memory as two consecutive 128B-swizzled (box_outer x 64)
// blocks -- exactly the two halves of a B stage -- with ONE TMA instruction.
int make_tmap_grouped(CUtensorMap* map, int dtype, const void* base, uint64_t inner, uint64_t outer,
                      uint64_t ld, uint32_t box_outer, uint32_t box_groups) {
  const cuuint64_t dims[3] = {64, outer, inner / 64}, strides[2] = {ld * 2, 128};
  const cuuint32_t box[3] = {64, box_outer, box_groups};
  return encode_tiled(map, dtype, 3, base, dims, strides, box, CU_TENSOR_MAP_SWIZZLE_128B, "spmma (grouped view)");
}

struct HostProblem {
  int opB;
  size_t m, n, k;
  const void *comp_vals, *meta, *B, *C;
  void* D;
  size_t ldb, ldc, ldd;
  float alpha, beta;
  bool conv = false;                     // implicit GEMM: B is the NHWC activation tensor, never unfolded (view `im`)
  Im2col im{};
  bool out_t = false;                    // D is written transposed: [n][m] row-major, pitch ldd >= m (SPFY_OUT_T)
  spfy_epilogue epi{nullptr, nullptr, SPFY_ACT_NONE};
  bool ex = false;                       // called through an _ex entry: beta != 0 allowed with out_t (C is then [n][m])
  bool scatter = false;                  // out_t rows scattered to the phase (sc_a, sc_b) of an sc_h x sc_w image
  uint32_t sc_h = 0, sc_w = 0, sc_s = 1, sc_a = 0, sc_b = 0;
};

// the `opB` argument of the C ABI carries the output layout in bit 4 (SPFY_OUT_T)
inline int op_of(int opB) { return opB & ~SPFY_OUT_T; }
inline bool out_t_of(int opB) { return (opB & SPFY_OUT_T) != 0; }

// D of a problem, or a replica of D at `base`: boxes of 64 n x 32 m, or of 32 m x 64 n (unswizzled) when transposed
int make_tmap_d(CUtensorMap* map, int dtype, const HostProblem& h, void* base) {
  return h.out_t ? make_tmap_2d(map, dtype, base, h.m, h.n, h.ldd, 32, 64, CU_TENSOR_MAP_SWIZZLE_NONE)
                 : make_tmap_2d(map, dtype, base, h.n, h.m, h.ldd, 64, 32);
}


int validate(int dtype, const HostProblem& h, const char* who) {
  if (dtype != SPFY_F16 && dtype != SPFY_BF16)
    return fail(SPFY_E_UNSUPPORTED, "%s: dtype %d (need F16/BF16)", who, dtype);
  if (h.opB != SPFY_OP_N && h.opB != SPFY_OP_T) return fail(SPFY_E_INVALID, "%s: bad opB %d", who, h.opB);
  if (h.epi.act < SPFY_ACT_NONE || h.epi.act > SPFY_ACT_GELU_TANH)
    return fail(SPFY_E_INVALID, "%s: bad epilogue activation %d", who, h.epi.act);
  if ((uintptr_t)h.epi.scale % 4 || (uintptr_t)h.epi.bias % 4)
    return fail(SPFY_E_INVALID, "%s: epilogue scale / bias must be 4-byte aligned", who);
  if (h.m == 0 || h.n == 0) return SPFY_OK;
  if (!h.comp_vals || !h.meta || !h.B || !h.D) return fail(SPFY_E_INVALID, "%s: null operand", who);
  if (h.beta != 0.f && !h.C) return fail(SPFY_E_INVALID, "%s: beta != 0 needs C", who);
  if (h.k == 0) return fail(SPFY_E_UNSUPPORTED, "%s: k == 0", who);
  if (h.m >= (1u << 31) || h.n >= (1u << 31) || h.k >= (1u << 31))
    return fail(SPFY_E_UNSUPPORTED, "%s: dimension too large", who);
  const size_t b_inner = h.opB == SPFY_OP_N ? h.n : h.k;
  if (h.out_t && h.beta != 0.f && !h.ex)
    return fail(SPFY_E_UNSUPPORTED, "%s: a transposed output (SPFY_OUT_T) needs beta == 0", who);
  // (a TMA store moves whole 16-byte pieces of a row: the contiguous dimension of the output is a multiple of 8 elements)
  if (h.out_t && h.m % 8)
    return fail(SPFY_E_UNSUPPORTED, "%s: a transposed output (SPFY_OUT_T) needs m %% 8 == 0 (m=%zu)", who, h.m);
  if ((!h.conv && h.ldb < b_inner) || h.ldd < (h.out_t ? h.m : h.n) || (h.beta != 0.f && h.ldc < (h.out_t ? h.m : h.n)))
    return fail(SPFY_E_INVALID, "%s: leading dimension too small", who);
  // TMA contract == the reference's own fp16 contract (spmma.hxx:45-49): multiples of 8
  // (a scattered output is written position by position: n is free)
  if ((!h.conv && h.ldb % 8) || h.ldd % 8 || (h.beta != 0.f && h.ldc % 8) || (!h.scatter && h.n % 8) ||
      (h.opB == SPFY_OP_T && h.k % 8))
    return fail(SPFY_E_UNSUPPORTED,
                "%s: n, ldb, ldc, ldd (and k for opB=T) must be multiples of 8 elements "
                "(n=%zu k=%zu ldb=%zu ldc=%zu ldd=%zu)", who, h.n, h.k, h.ldb, h.ldc, h.ldd);
  if ((uintptr_t)h.B % 16 || (uintptr_t)h.D % 16 || (h.beta != 0.f && (uintptr_t)h.C % 16) ||
      (uintptr_t)h.comp_vals % 16 || (uintptr_t)h.meta % 16)
    return fail(SPFY_E_INVALID, "%s: operands must be 16-byte aligned", who);
  return SPFY_OK;
}

// launch classes: problems of one class share a shared-memory geometry and one launch
// resident classes differ in ring depth: the smaller the resident operand, the more B stages fit, and
// more B in flight is what the HBM-bound shapes need (measured: 1/2/3/4 stages -> 0.45/0.69/0.79/0.93 of
// the copy rate); k <= 64 gets half-size stages so that no stage is half empty.
// Streaming problems with few k-tiles per unit (K <= 512) write far more than they read: they trade ring
// depth (2 stages) for all eight epilogue warps.
enum { CLASS_RES_K64 = 0, CLASS_RES_SMALL = 1, CLASS_RES_LARGE = 2, CLASS_STREAM_G2_SHORT = 3, CLASS_STREAM_G1 = 4,
       CLASS_STREAM_G2 = 5, NUM_CLASSES = 6 };
constexpr size_t SHORT_K = 512;
inline bool is_resident_class(int cls) { return cls <= CLASS_RES_LARGE; }
constexpr uint32_t BAR_BYTES = 512;
constexpr uint32_t RES_MAX_BYTES = 96 * 1024;    // resident A (values + metadata)
constexpr uint32_t RES_SMALL_BYTES = 48 * 1024;  // ... small enough for a fourth 32 KiB stage

size_t resident_bytes(size_t m, size_t k) {
  const size_t m_tiles = ceil_div(m, BM), k_tiles = ceil_div(k, 128);
  const size_t rows = m_tiles == 1 ? round_up(m, 16) : 128;
  return m_tiles * k_tiles * rows * 144;  // 128 B of values + 16 B of metadata per row and k-tile
}

// Sliced residency: A as a whole is too large, but the two m-tiles of one m-group (all k-tiles) fit, and every CTA
// keeps meeting the same m-group (units are dealt nt-major with the m-group fastest and a stride of gridDim, so the
// group a CTA sees is constant when the grid is a multiple of m_groups).  The CTA then loads its slice once and streams
// B only, like the resident classes, instead of pulling the same 36 KiB per k-tile through the ring for every unit.
size_t slice_bytes(size_t k) { return 2 * ceil_div(k, 128) * (size_t)(A_TILE_BYTES + E_TILE_BYTES); }

bool sliced_residency(const HostProblem& h, int sm_count) {
  static const bool off = dev_switch("SPFY_SPMMA_NO_SLICES") != nullptr;
  const size_t m_tiles = ceil_div(h.m, BM), n_tiles = ceil_div(h.n, BN), m_groups = ceil_div(m_tiles, 2);
  return !off && m_tiles >= 2 && h.k > 64 && resident_bytes(h.m, h.k) > RES_MAX_BYTES && slice_bytes(h.k) <= RES_MAX_BYTES &&
         (size_t)sm_count % m_groups == 0 && m_groups * n_tiles >= 2 * (size_t)sm_count;
}

int classify(const HostProblem& h, bool grouped, int sm_count) {
  const size_t m_tiles = ceil_div(h.m, BM), n_tiles = ceil_div(h.n, BN);
  if (resident_bytes(h.m, h.k) <= RES_MAX_BYTES && n_tiles >= (size_t)sm_count) {
    if (h.k <= 64) return CLASS_RES_K64;
    return resident_bytes(h.m, h.k) <= RES_SMALL_BYTES ? CLASS_RES_SMALL : CLASS_RES_LARGE;
  }
  if (sliced_residency(h, sm_count)) return slice_bytes(h.k) <= RES_SMALL_BYTES ? CLASS_RES_SMALL : CLASS_RES_LARGE;
  static const double g2_min_waves = [] {
    const char* e = dev_switch("SPFY_SPMMA_G2_MIN_WAVES");
    return e ? atof(e) : 0.5;
  }();
  // Two m-tiles share every B stage whenever there are two: the L2 -> SM path is barely faster than HBM on this part,
  // so a second CTA re-reading the same B columns costs nearly as much as reading them from DRAM again.  Measured on
  // single calls (bench.py --per-layer): 256 x 2304 x 25088 41.0 -> 36.9 us, 512 x 4608 x 6272 41.0 -> 33.7 us with
  // G = 2 even though only 98-196 units are left for 148 SMs.  One m-tile per unit only below half a wave.
  if (m_tiles >= 2 && (grouped || (double)(ceil_div(m_tiles, 2) * n_tiles) >= g2_min_waves * (double)sm_count))
    return h.k <= SHORT_K ? CLASS_STREAM_G2_SHORT : CLASS_STREAM_G2;
  return CLASS_STREAM_G1;
}

// fill the device view of one problem (tensor maps included); unit_begin is set by the caller
int fill_problem(ProblemDev* d, int dtype, const HostProblem& h, int cls) {
  const uint32_t bk = cls == CLASS_RES_K64 ? 64u : (uint32_t)BK;
  memset(d, 0, sizeof(*d));
  int rc;
  // B: inner = contiguous dimension (n for opB = N, k for opB = T), outer = the other one
  const size_t b_inner = h.opB == SPFY_OP_N ? h.n : h.k, b_outer = h.opB == SPFY_OP_N ? h.k : h.n;
  d->b3d = b_inner % 64 == 0;
  rc = SPFY_OK;
  // one stage of B: opB = N -> bk rows of k x 128 columns (two 64-column groups);
  //                 opB = T -> 128 rows of n x bk columns of k (bk/64 groups)
  const uint32_t box_outer = h.opB == SPFY_OP_N ? bk : 128u, box_groups = h.opB == SPFY_OP_N ? 2u : bk / 64u;
  if (h.conv) {
    d->b3d = 0;
    rc = make_tmap_im2col(&d->tmap_b, dtype, h.B, h.im, BN);
    if (rc) return rc;
    d->conv = 1;
    d->conv_c = (uint32_t)h.im.c;
    d->conv_kw = (uint32_t)h.im.kw;
    d->conv_wo = (uint32_t)h.im.wo;
    d->conv_ho = (uint32_t)h.im.ho;
    d->conv_stride = (uint32_t)h.im.stride;
    d->conv_off_h = h.im.lo_h;
    d->conv_off_w = h.im.lo_w;
  } else {
    if (d->b3d && make_tmap_grouped(&d->tmap_b, dtype, h.B, b_inner, b_outer, h.ldb, box_outer, box_groups) != SPFY_OK)
      d->b3d = 0;  // the driver refused the grouped view: fall back to 2-D boxes (64 inner elements each)
    if (!d->b3d) rc = make_tmap_2d(&d->tmap_b, dtype, h.B, b_inner, b_outer, h.ldb, 64, box_outer);
    if (rc) return rc;
  }
  rc = make_tmap_d(&d->tmap_d, dtype, h, h.D);
  if (rc) return rc;
  d->out_t = h.out_t;
  d->a_vals = (const uint8_t*)h.comp_vals;
  d->a_meta = (const uint8_t*)h.meta;
  d->C = h.C;
  d->ldc = h.ldc;
  d->m = (uint32_t)h.m;
  d->n = (uint32_t)h.n;
  d->k = (uint32_t)h.k;
  d->m_tiles = (uint32_t)ceil_div(h.m, BM);
  d->k_tiles = (uint32_t)ceil_div(h.k, 128);
  d->n_tiles = (uint32_t)ceil_div(h.n, BN);
  d->resident = !is_resident_class(cls) ? 0u : (resident_bytes(h.m, h.k) <= RES_MAX_BYTES ? 1u : 2u);
  d->G = (cls == CLASS_STREAM_G1) ? 1u : (d->m_tiles >= 2 ? 2u : 1u);
  d->m_groups = (uint32_t)ceil_div(d->m_tiles, d->G);
  d->units = d->m_groups * d->n_tiles;
  d->split_units = d->units;
  d->split_nt = d->n_tiles;
  d->alpha = h.alpha;
  d->beta = h.beta;
  d->scale = h.epi.scale;
  d->bias = h.epi.bias;
  d->act = (uint32_t)h.epi.act;
  // an identity epilogue (no scale, no bias, no activation) runs the code of the plain entry points
  d->epi = h.epi.scale || h.epi.bias || h.epi.act != SPFY_ACT_NONE || (h.out_t && h.beta != 0.f);
  if (h.scatter) {
    d->D = h.D;
    d->ldd = h.ldd;
    d->sc_h = h.sc_h; d->sc_w = h.sc_w; d->sc_s = h.sc_s; d->sc_a = h.sc_a; d->sc_b = h.sc_b;
  }
  // B is streamed once when one unit covers all of M; otherwise the other m-groups of the same
  // columns will want it from L2 shortly after
  d->hint_b = d->m_groups == 1 ? HINT_EVICT_FIRST : HINT_EVICT_NORMAL;
  // implicit GEMM: every activation is read kh * kw times (by the other filter taps and the neighbouring tiles), so the
  // lines must not be marked for early eviction
  if (h.conv) {
    const char* e = dev_switch("SPFY_CONV_HINT");
    d->hint_b = e && atoi(e) == 1 ? HINT_EVICT_FIRST : e && atoi(e) == 2 ? HINT_EVICT_LAST : HINT_EVICT_NORMAL;
  }
  return SPFY_OK;
}

// shared-memory geometry of a class; `res_vals` / `res_meta` = bytes of the largest resident problem
void geometry(int cls, uint32_t res_vals, uint32_t res_meta, LaunchParams* L, uint32_t* smem_bytes) {
  uint32_t stage, res = 0;
  L->a_off = B_STAGE_BYTES;
  L->bk = cls == CLASS_RES_K64 ? 64u : (uint32_t)BK;
  if (is_resident_class(cls)) {
    stage = L->bk * (uint32_t)(BN * 2);
    L->e_off = stage;
    res = (uint32_t)round_up(res_vals, 1024) + (uint32_t)round_up(res_meta, 1024);
    L->epi_warps = NUM_EPI_WARPS;  // small K: the epilogue is the hot part
  } else {
    const uint32_t G = cls == CLASS_STREAM_G1 ? 1u : 2u;
    L->e_off = B_STAGE_BYTES + G * A_TILE_BYTES;
    stage = L->e_off + G * E_TILE_BYTES;
    // large K: shared memory goes to the ring instead of staging buffers for four more epilogue warps
    L->epi_warps = cls == CLASS_STREAM_G2_SHORT ? NUM_EPI_WARPS : NUM_EPI_WARPS / 2;
  }
  const uint32_t c_bytes = L->epi_warps * C_BUF_BYTES;
  const uint32_t fixed = 1024 /*alignment slack*/ + c_bytes + BAR_BYTES + res;
  uint32_t stages = (SMEM_LIMIT - fixed) / stage;
  if (stages > (uint32_t)MAX_STAGES) stages = MAX_STAGES;
  if (const char* cap = dev_switch("SPFY_SPMMA_STAGES")) {  // tuning experiment: fewer ring stages
    const uint32_t c = (uint32_t)atoi(cap);
    if (c >= 1 && c < stages) stages = c;
  }
  L->stages = stages;
  L->stage_bytes = stage;
  L->res_off = stages * stage;
  L->res_e_off = L->res_off + (uint32_t)round_up(res_vals, 1024);
  L->c_off = L->res_off + res;
  L->bar_off = L->c_off + c_bytes;
  *smem_bytes = L->bar_off + BAR_BYTES + 1024;
}

// A single streaming call whose last wave is partial: deal that wave's n-tiles one m-tile per unit when the G = 1 units
// still fit one wave (256 x 2304 x 25088: 196 units on 148 SMs = 148 + 48 -> 148 + 96 half units).
void split_tail(ProblemDev* d, int cls, int sm_count) {
  static const bool off = dev_switch("SPFY_SPMMA_NO_TAIL_SPLIT") != nullptr;
  if (off || is_resident_class(cls) || d->G != 2u || d->m_tiles < 2u) return;
  const uint32_t sm = (uint32_t)sm_count, full = d->units / sm, rem = d->units % sm;
  if (full == 0 || rem == 0 || rem % d->m_groups) return;
  const uint32_t tail_nt = rem / d->m_groups, tail_units = tail_nt * d->m_tiles;
  if (tail_units > sm) return;
  d->split_units = d->units - rem;
  d->split_nt = d->n_tiles - tail_nt;
  d->units = d->split_units + tail_units;
  d->hint_b = HINT_EVICT_NORMAL;  // the tail's B tiles are read by every m-tile's unit
}

uint32_t make_idesc(int dtype, int opB) {
  // instruction descriptor (kind::f16, sparse): c=F32, a/b format, b major, N>>3, M>>4
  const uint32_t fmt = dtype == SPFY_BF16 ? 1u : 0u;
  return (1u << 2) | (1u << 4) | (fmt << 7) | (fmt << 10) | ((opB == SPFY_OP_N ? 1u : 0u) << 16) |
         ((uint32_t)(BN >> 3) << 17) | ((uint32_t)(BM >> 4) << 24);
}

template <bool BF16, bool OPB_T, bool EPI, bool SCATTER = false>
int launch_t(const ProblemDev& single, const LaunchParams& L, uint32_t smem, int grid, cudaStream_t s,
             bool overlap_previous) {
  int rc = allow_dynamic_smem<spmma_kernel<BF16, OPB_T, EPI, SCATTER>>(SMEM_LIMIT);
  if (rc) return rc;
  cudaLaunchConfig_t cfg;
  memset(&cfg, 0, sizeof(cfg));
  cfg.gridDim = dim3((unsigned)grid);
  cfg.blockDim = dim3(NUM_THREADS);
  cfg.dynamicSmemBytes = smem;
  cfg.stream = s;
  cudaLaunchAttribute attr;
  memset(&attr, 0, sizeof(attr));
  attr.id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr.val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = &attr;
  cfg.numAttrs = overlap_previous ? 1 : 0;
  SPFY_CUDA_OK(cudaLaunchKernelEx(&cfg, spmma_kernel<BF16, OPB_T, EPI, SCATTER>, single, L));
  SPFY_LAUNCH_OK("spmma_kernel");
  return SPFY_OK;
}

template <bool EPI>
int launch_e(int dtype, int opB, const ProblemDev& single, const LaunchParams& L, uint32_t smem, int grid,
             cudaStream_t s, bool overlap_previous) {
  if (dtype == SPFY_BF16)
    return opB == SPFY_OP_N ? launch_t<true, false, EPI>(single, L, smem, grid, s, overlap_previous)
                            : launch_t<true, true, EPI>(single, L, smem, grid, s, overlap_previous);
  return opB == SPFY_OP_N ? launch_t<false, false, EPI>(single, L, smem, grid, s, overlap_previous)
                          : launch_t<false, true, EPI>(single, L, smem, grid, s, overlap_previous);
}

// overlap_previous: the kernel launched just before on this stream is another launch of the same plan (or another
// phase of the same data gradient); epi: some problem of the launch has an epilogue; a single problem with a scattered
// output (opB = T) takes the SCATTER kernels
int launch(int dtype, int opB, bool epi, const ProblemDev& single, const LaunchParams& L, uint32_t smem, int grid,
           cudaStream_t s, bool overlap_previous = false) {
  if (single.D)
    return dtype == SPFY_BF16 ? launch_t<true, true, true, true>(single, L, smem, grid, s, overlap_previous)
                              : launch_t<false, true, true, true>(single, L, smem, grid, s, overlap_previous);
  return epi ? launch_e<true>(dtype, opB, single, L, smem, grid, s, overlap_previous)
             : launch_e<false>(dtype, opB, single, L, smem, grid, s, overlap_previous);
}

#ifdef SPFY_DEV_SWITCHES
// SPFY_SPMMA_TRACE=path: CTA 0's hand-over timestamps of this launch, written to `path` (the call becomes synchronous)
int launch_traced(const char* path, int dtype, int opB, const ProblemDev& d, LaunchParams L, uint32_t smem, int grid, cudaStream_t s) {
  static long long* trace = nullptr;
  const size_t n = 3 * TRACE_UNITS * TRACE_SLOTS;
  if (!trace) SPFY_CUDA_OK(cudaMallocManaged((void**)&trace, n * sizeof(long long)));
  SPFY_CUDA_OK(cudaStreamSynchronize(s));
  memset(trace, 0, n * sizeof(long long));
  L.trace = trace;
  int rc = launch(dtype, opB, d.epi != 0, d, L, smem, grid, s);
  if (rc) return rc;
  SPFY_CUDA_OK(cudaStreamSynchronize(s));
  if (FILE* f = fopen(path, "w")) {
    fprintf(f, "# m=%u n=%u k=%u units=%u grid=%d stages=%u conv=%u\nrole,unit", d.m, d.n, d.k, d.units, grid, L.stages, d.conv);
    for (uint32_t sl = 0; sl < TRACE_SLOTS; ++sl) fprintf(f, ",t%u", sl);
    fprintf(f, "\n");
    long long t0 = 0;
    for (size_t i = 0; i < n; ++i) if (trace[i] && (!t0 || trace[i] < t0)) t0 = trace[i];
    for (uint32_t r = 0; r < 3; ++r)
      for (uint32_t u = 0; u < TRACE_UNITS; ++u) {
        fprintf(f, "%u,%u", r, u);
        for (uint32_t sl = 0; sl < TRACE_SLOTS; ++sl) {
          const long long v = trace[(r * TRACE_UNITS + u) * TRACE_SLOTS + sl];
          fprintf(f, ",%lld", v ? v - t0 : -1);
        }
        fprintf(f, "\n");
      }
    fclose(f);
  }
  return SPFY_OK;
}
#endif

uint32_t res_rows(const ProblemDev& d) { return d.m_tiles == 1 ? (uint32_t)round_up(d.m, 16) : 128u; }
uint32_t res_tiles(const ProblemDev& d) { return (d.resident == 2u ? d.G : d.m_tiles) * d.k_tiles; }
uint32_t res_values_bytes(const ProblemDev& d) { return res_tiles(d) * res_rows(d) * 128u; }
uint32_t res_meta_bytes(const ProblemDev& d) { return res_tiles(d) * res_rows(d) * 16u; }

// a convolution layer as a GEMM problem: n and k follow from the descriptor, B is the NHWC activation tensor (opB = T:
// a B stage is [128 positions][128 k], gathered by the im2col tensor map)
int conv_problem(int dtype, const spfy_conv_desc* conv, size_t m, float alpha, const void* comp_vals, const void* meta,
                 const void* X, float beta, const void* C, size_t ldc, void* D, size_t ldd, bool out_t,
                 const spfy_epilogue* epi, bool ex, const char* who, HostProblem* out) {
  if (!conv) return fail(SPFY_E_INVALID, "%s: null descriptor", who);
  const spfy_conv_desc& c = *conv;
  if (!c.batch || !c.h || !c.w || !c.c || !c.kh || !c.kw || !c.stride)
    return fail(SPFY_E_INVALID, "%s: empty dimension in the descriptor", who);
  if (c.c % 64) return fail(SPFY_E_UNSUPPORTED, "%s: channels must be a multiple of 64 (got %zu): unfold explicitly", who, c.c);
  if (c.h + 2 * c.pad < c.kh || c.w + 2 * c.pad < c.kw) return fail(SPFY_E_INVALID, "%s: filter larger than the padded image", who);
  if (c.kh > 16 || c.kw > 16 || c.pad > 8 || c.stride > 8)
    return fail(SPFY_E_UNSUPPORTED, "%s: filter / padding / stride outside what the im2col tensor map encodes", who);
  if ((uintptr_t)X % 16) return fail(SPFY_E_INVALID, "%s: activations must be 16-byte aligned", who);
  const size_t ho = (c.h + 2 * c.pad - c.kh) / c.stride + 1, wo = (c.w + 2 * c.pad - c.kw) / c.stride + 1;
  const size_t n = c.batch * ho * wo, k = c.kh * c.kw * c.c;
  HostProblem h{SPFY_OP_T, m, n, k, comp_vals, meta, X, C, D, /*ldb*/ k, ldc, ldd, alpha, beta};
  h.conv = true;
  h.im = im2col_of(c);
  h.out_t = out_t;
  if (epi) h.epi = *epi;
  h.ex = ex;
  *out = h;
  return validate(dtype, h, who);
}

// SPFY_SPMMA_DEBUG=mode: a dev-build ablation of the kernel (L.dbg)
uint32_t debug_mode() {
  const char* e = dev_switch("SPFY_SPMMA_DEBUG");
  return e ? (uint32_t)atoi(e) : 0u;
}

// one validated, non-empty problem in a launch of its own, built (tensor maps encoded) but not yet launched
struct SingleLaunch {
  ProblemDev d;
  LaunchParams L;
  uint32_t smem;
  int grid;
};
int prepare_single(int dtype, const HostProblem& h, const DeviceInfo& di, SingleLaunch* out) {
  const int cls = classify(h, false, di.sm_count);
  ProblemDev& d = out->d;
  int rc = fill_problem(&d, dtype, h, cls);
  if (rc) return rc;
  d.unit_begin = 0;
  split_tail(&d, cls, di.sm_count);
  LaunchParams& L = out->L;
  memset(&L, 0, sizeof(L));
  out->smem = 0;
  geometry(cls, res_values_bytes(d), res_meta_bytes(d), &L, &out->smem);
  L.table = nullptr;
  L.num_problems = 1;
  L.total_units = d.units;
  L.idesc = make_idesc(dtype, h.opB);
  L.dbg = debug_mode();
  out->grid = (int)(d.units < (uint32_t)di.sm_count ? d.units : (uint32_t)di.sm_count);
  return SPFY_OK;
}

// one validated problem (spfy_spmma*, spfy_spmma_conv*) in a launch of its own
int run_single(int dtype, const HostProblem& h, cudaStream_t s) {
  if (h.m == 0 || h.n == 0) return SPFY_OK;
  DeviceInfo di;
  int rc = require_sm100(h.conv ? "spmma_conv" : "spmma", &di);
  if (rc) return rc;
  SingleLaunch sl;
  rc = prepare_single(dtype, h, di, &sl);
  if (rc) return rc;
#ifdef SPFY_DEV_SWITCHES
  if (const char* path = dev_switch("SPFY_SPMMA_TRACE"))
    return launch_traced(path, dtype, h.opB, sl.d, sl.L, sl.smem, sl.grid, s);
#endif
  return launch(dtype, h.opB, sl.d.epi != 0, sl.d, sl.L, sl.smem, sl.grid, s);
}

// the dX pixels of a strided data gradient that no filter tap reaches (bit a * s + b of `empty`: phase (a, b) has no
// taps): +0 for beta == 0 (whatever dX held), else beta * dX.  16 bytes (8 channels) per thread and step.
template <typename T>
__global__ void __launch_bounds__(256)
dgrad_fill_kernel(T* dx, size_t chunks, uint32_t c8, uint32_t h, uint32_t w, uint32_t s, uint64_t empty, float beta) {
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < chunks; t += (size_t)gridDim.x * blockDim.x) {
    const size_t px = t / c8;
    const uint32_t x = (uint32_t)(px % w), y = (uint32_t)(px / w % h);
    if (!(empty >> ((y % s) * s + x % s) & 1u)) continue;
    uint4* p = reinterpret_cast<uint4*>(dx) + t;
    if (beta == 0.f) {
      *p = make_uint4(0u, 0u, 0u, 0u);
    } else {
      union {
        uint4 v;
        T e[8];
      } u;
      u.v = *p;
#pragma unroll
      for (int i = 0; i < 8; ++i) u.e[i] = from_f32<T>(beta * to_f32(u.e[i]));
      *p = u.v;
    }
  }
}

struct Plan {
  int dtype = 0;
  ProblemDev* d_table = nullptr;  // all launches back to back
  CUtensorMap* d_rep = nullptr;   // replica maps of all problems ([problem in table order][n_rep])
  struct Launch {
    int opB;
    uint32_t first, count;  // range in d_table
    LaunchParams L;
    uint32_t smem;
    int grid;
    bool epi;  // some problem of the launch has an epilogue
  };
  std::vector<Launch> launches;
};

}  // namespace
}  // namespace spfy

void spfy::warm_spmma_kernels() {
  touch_kernel(spmma_kernel<false, false, false, false>);
  touch_kernel(spmma_kernel<false, true, false, false>);
  touch_kernel(spmma_kernel<true, false, false, false>);
  touch_kernel(spmma_kernel<true, true, false, false>);
  touch_kernel(spmma_kernel<false, false, true, false>);
  touch_kernel(spmma_kernel<false, true, true, false>);
  touch_kernel(spmma_kernel<true, false, true, false>);
  touch_kernel(spmma_kernel<true, true, true, false>);
  touch_kernel(spmma_kernel<false, true, true, true>);
  touch_kernel(spmma_kernel<true, true, true, true>);
  touch_kernel(dgrad_fill_kernel<__half>);
  touch_kernel(dgrad_fill_kernel<__nv_bfloat16>);
  EncodeTiledFn enc;
  (void)get_encoder(&enc);
}

using namespace spfy;

extern "C" {

int spfy_spmma_workspace_bytes(int dtype, size_t m, size_t n, size_t k, size_t* bytes) {
  (void)dtype; (void)m; (void)n; (void)k;
  if (bytes) *bytes = 0;  // the kernel needs no global scratch
  return SPFY_OK;
}

static int spmma_impl(int dtype, int opB, size_t m, size_t n, size_t k, float alpha, const void* comp_vals,
                      const void* meta, const void* B, size_t ldb, float beta, const void* C, size_t ldc, void* D,
                      size_t ldd, const spfy_epilogue* epi, bool ex, spfy_stream_t stream) {
  HostProblem h{op_of(opB), m, n, k, comp_vals, meta, B, C, D, ldb, ldc, ldd, alpha, beta};
  h.out_t = out_t_of(opB);
  if (epi) h.epi = *epi;
  h.ex = ex;
  int rc = validate(dtype, h, "spmma");
  if (rc) return rc;
  return run_single(dtype, h, (cudaStream_t)stream);
}

int spfy_spmma(int dtype, int opB, size_t m, size_t n, size_t k, float alpha, const void* comp_vals,
               const void* meta, const void* B, size_t ldb, float beta, const void* C, size_t ldc,
               void* D, size_t ldd, void* workspace, size_t workspace_bytes, spfy_stream_t stream) {
  (void)workspace; (void)workspace_bytes;
  return spmma_impl(dtype, opB, m, n, k, alpha, comp_vals, meta, B, ldb, beta, C, ldc, D, ldd, nullptr, false, stream);
}

int spfy_spmma_ex(int dtype, int opB, size_t m, size_t n, size_t k, float alpha, const void* comp_vals,
                  const void* meta, const void* B, size_t ldb, float beta, const void* C, size_t ldc,
                  void* D, size_t ldd, void* workspace, size_t workspace_bytes, const spfy_epilogue* epi,
                  spfy_stream_t stream) {
  (void)workspace; (void)workspace_bytes;
  return spmma_impl(dtype, opB, m, n, k, alpha, comp_vals, meta, B, ldb, beta, C, ldc, D, ldd, epi, true, stream);
}

static int spmma_conv_impl(int dtype, const spfy_conv_desc* conv, size_t m, float alpha, const void* comp_vals,
                           const void* meta, const void* X, float beta, const void* C, size_t ldc, void* D, size_t ldd,
                           bool out_t, const spfy_epilogue* epi, bool ex, spfy_stream_t stream) {
  HostProblem h;
  int rc = conv_problem(dtype, conv, m, alpha, comp_vals, meta, X, beta, C, ldc, D, ldd, out_t, epi, ex, "spmma_conv", &h);
  if (rc) return rc;
  return run_single(dtype, h, (cudaStream_t)stream);
}

int spfy_spmma_conv(int dtype, const spfy_conv_desc* conv, size_t m, float alpha, const void* comp_vals,
                    const void* meta, const void* X, float beta, const void* C, size_t ldc, void* D, size_t ldd,
                    spfy_stream_t stream) {
  return spmma_conv_impl(dtype, conv, m, alpha, comp_vals, meta, X, beta, C, ldc, D, ldd, false, nullptr, false, stream);
}

int spfy_spmma_conv_nhwc(int dtype, const spfy_conv_desc* conv, size_t m, float alpha, const void* comp_vals,
                         const void* meta, const void* X, void* Y, size_t ldy, spfy_stream_t stream) {
  return spmma_conv_impl(dtype, conv, m, alpha, comp_vals, meta, X, 0.f, nullptr, 0, Y, ldy, true, nullptr, false, stream);
}

int spfy_spmma_conv_dgrad(int dtype, const spfy_conv_desc* conv, size_t m, float alpha, const void* vals_t,
                          const void* meta_t, const void* dY, float beta, void* dX, spfy_stream_t stream) {
  const char* who = "spmma_conv_dgrad";
  if (dtype != SPFY_F16 && dtype != SPFY_BF16) return fail(SPFY_E_UNSUPPORTED, "%s: dtype %d (need F16/BF16)", who, dtype);
  if (!conv) return fail(SPFY_E_INVALID, "%s: null descriptor", who);
  const spfy_conv_desc& c = *conv;
  if (!c.batch || !c.h || !c.w || !c.c || !c.kh || !c.kw || !c.stride || !m)
    return fail(SPFY_E_INVALID, "%s: empty dimension", who);
  if (m % 64)
    return fail(SPFY_E_UNSUPPORTED, "%s: m (the channels of dY) must be a multiple of 64 (got %zu)", who, m);
  if (c.c % 8) return fail(SPFY_E_UNSUPPORTED, "%s: c (the channels of dX) must be a multiple of 8 (got %zu)", who, c.c);
  if (c.kh > 16 || c.kw > 16 || c.pad > 8 || c.stride > 8)
    return fail(SPFY_E_UNSUPPORTED, "%s: filter / padding / stride outside what spfy_spmma_conv accepts", who);
  if (c.h + 2 * c.pad < c.kh || c.w + 2 * c.pad < c.kw) return fail(SPFY_E_INVALID, "%s: filter larger than the padded image", who);
  if (!vals_t || !meta_t || !dY || !dX) return fail(SPFY_E_INVALID, "%s: null operand", who);
  if ((uintptr_t)vals_t % 16 || (uintptr_t)meta_t % 16 || (uintptr_t)dY % 16 || (uintptr_t)dX % 16)
    return fail(SPFY_E_INVALID, "%s: operands must be 16-byte aligned", who);
  const size_t s = c.stride, ho = (c.h + 2 * c.pad - c.kh) / s + 1, wo = (c.w + 2 * c.pad - c.kw) / s + 1;
  // every phase, validated before any device work; the phase operands lie back to back in the order of
  // spfy_transpose24_conv, whether or not the phase has dX pixels
  HostProblem phases[64];
  int count = 0;
  uint64_t empty = 0;
  size_t tiles = 0;
  for (size_t a = 0; a < s; ++a)
    for (size_t b = 0; b < s; ++b) {
      const DgradPhase ph = dgrad_phase(c.kh, s, c.pad, a), pw = dgrad_phase(c.kw, s, c.pad, b);
      const size_t ha = dgrad_phase_extent(c.h, s, a), wb = dgrad_phase_extent(c.w, s, b);
      if (!ph.taps || !pw.taps) {
        if (ha && wb) empty |= 1ull << (a * s + b);
        continue;
      }
      const size_t k = (size_t)ph.taps * pw.taps * m;
      const size_t first = tiles;
      tiles += ceil_div(c.c, 128) * ceil_div(k, 128);
      if (!ha || !wb) continue;
      // a stride-1 correlation of dY: base pixels [d0, d0 + phase extent) per dimension
      Im2col im{c.batch, ho, wo, m, ph.taps, pw.taps, 1, ph.d0, pw.d0, ph.d0 + (int)ha - (int)ho, pw.d0 + (int)wb - (int)wo,
                ha, wb};
      if (std::min({im.lo_h, im.lo_w, im.up_h, im.up_w}) < -128 || std::max({im.lo_h, im.lo_w, im.up_h, im.up_w}) > 127)
        return fail(SPFY_E_UNSUPPORTED, "%s: phase (%zu, %zu) needs im2col corners outside [-128, 127]", who, a, b);
      HostProblem h{SPFY_OP_T, c.c, c.batch * ha * wb, k, (const uint8_t*)vals_t + first * A_TILE_BYTES,
                    (const uint8_t*)meta_t + first * E_TILE_BYTES, dY, dX, dX, /*ldb*/ k, c.c, c.c, alpha, beta};
      h.conv = true;
      h.im = im;
      h.out_t = true;
      h.ex = true;
      h.scatter = true;
      h.sc_h = (uint32_t)c.h; h.sc_w = (uint32_t)c.w; h.sc_s = (uint32_t)s; h.sc_a = (uint32_t)a; h.sc_b = (uint32_t)b;
      int rc = validate(dtype, h, who);
      if (rc) return rc;
      phases[count++] = h;
    }
  // every phase built (tensor maps encoded) before any device work, so that a failure leaves dX untouched
  DeviceInfo di;
  int rc = require_sm100(who, &di);
  if (rc) return rc;
  std::vector<SingleLaunch> launches((size_t)count);
  for (int i = 0; i < count; ++i) {
    rc = prepare_single(dtype, phases[i], di, &launches[(size_t)i]);
    if (rc) return rc;
  }
  cudaStream_t st = (cudaStream_t)stream;
  if (empty && beta != 1.f) {
    const size_t chunks = c.batch * c.h * c.w * (c.c / 8);
    int grid = 1;
    rc = capped_grid(ceil_div(chunks, 256), 8, &grid);
    if (rc) return rc;
    if (dtype == SPFY_BF16)
      dgrad_fill_kernel<__nv_bfloat16><<<grid, 256, 0, st>>>((__nv_bfloat16*)dX, chunks, (uint32_t)(c.c / 8), (uint32_t)c.h,
                                                             (uint32_t)c.w, (uint32_t)s, empty, beta);
    else
      dgrad_fill_kernel<__half><<<grid, 256, 0, st>>>((__half*)dX, chunks, (uint32_t)(c.c / 8), (uint32_t)c.h, (uint32_t)c.w,
                                                      (uint32_t)s, empty, beta);
    SPFY_LAUNCH_OK("dgrad_fill_kernel");
  }
  // The phases write disjoint pixels of dX, so each launch may start while the previous one still runs: a phase of a
  // small layer (26-52 units at 14 x 14, b = 32) leaves most SMs to the next one.  SPFY_SPMMA_NO_OVERLAP (dev builds,
  // read on every call) serialises them, for timing the two forms against each other.
  const bool serial = dev_switch("SPFY_SPMMA_NO_OVERLAP") != nullptr;
  for (int i = 0; i < count; ++i) {
    const SingleLaunch& sl = launches[(size_t)i];
    rc = launch(dtype, SPFY_OP_T, sl.d.epi != 0, sl.d, sl.L, sl.smem, sl.grid, st, i > 0 && !serial);
    if (rc) return rc;
  }
  return SPFY_OK;
}

int spfy_spmma_conv_ex(int dtype, const spfy_conv_desc* conv, size_t m, float alpha, const void* comp_vals,
                       const void* meta, const void* X, float beta, const void* C, size_t ldc, void* D, size_t ldd,
                       int layout, const spfy_epilogue* epi, spfy_stream_t stream) {
  if (layout != 0 && layout != SPFY_OUT_T) return fail(SPFY_E_INVALID, "spmma_conv_ex: bad output layout %d", layout);
  return spmma_conv_impl(dtype, conv, m, alpha, comp_vals, meta, X, beta, C, ldc, D, ldd, layout == SPFY_OUT_T, epi, true,
                         stream);
}

static void plan_free(Plan* plan) {
  if (plan->d_table) cudaFree(plan->d_table);
  if (plan->d_rep) cudaFree(plan->d_rep);
  delete plan;
}

// problem i of a plan as the host sees it (a convolution layer when convs[i] is given: B = X, n / k / ldb / opB from the
// descriptor, the SPFY_OUT_T bit of opB still selects the NHWC output)
static int plan_problem(int dtype, const spfy_spmma_problem& q, const spfy_conv_desc* conv, const spfy_epilogue* epi, bool ex,
                        HostProblem* h) {
  if (conv)
    return conv_problem(dtype, conv, q.m, q.alpha, q.comp_vals, q.meta, q.B, q.beta, q.C, q.ldc, q.D, q.ldd, out_t_of(q.opB),
                        epi, ex, "spmma_plan_create", h);
  *h = HostProblem{op_of(q.opB), q.m, q.n, q.k, q.comp_vals, q.meta, q.B, q.C, q.D, q.ldb, q.ldc, q.ldd, q.alpha, q.beta};
  h->out_t = out_t_of(q.opB);
  if (epi) h->epi = *epi;
  h->ex = ex;
  return validate(dtype, *h, "spmma_plan_create");
}

static int plan_create_impl(int dtype, const spfy_spmma_problem* problems, const spfy_conv_desc* const* convs,
                            const spfy_epilogue* const* epis, bool ex, size_t count, size_t n_rep, void* const* rep_d,
                            spfy_spmma_plan_t* out) {
  if (!out) return fail(SPFY_E_INVALID, "spmma_plan_create: null plan pointer");
  *out = nullptr;
  if (count && !problems) return fail(SPFY_E_INVALID, "spmma_plan_create: null problem list");
  DeviceInfo di;
  int rc = require_sm100("spmma_plan_create", &di);
  if (rc) return rc;
  // every non-empty problem, validated and classified once
  struct Member {
    size_t index;
    HostProblem h;
    int cls;
  };
  std::vector<Member> members;
  for (size_t i = 0; i < count; ++i) {
    HostProblem h;
    rc = plan_problem(dtype, problems[i], convs ? convs[i] : nullptr, epis ? epis[i] : nullptr, ex, &h);
    if (rc) return rc;
    if (h.m && h.n) members.push_back(Member{i, h, classify(h, true, di.sm_count)});
  }
  // members of a launch, longest units first: the CTAs walk the unit list with a fixed stride, so
  // whatever comes last sets the tail -- it should be the problems whose units are short
  std::stable_sort(members.begin(), members.end(),
                   [](const Member& a, const Member& b) { return ceil_div(a.h.k, 128) > ceil_div(b.h.k, 128); });
  std::unique_ptr<Plan, decltype(&plan_free)> plan(new Plan(), plan_free);
  plan->dtype = dtype;
  std::vector<ProblemDev> table;
  std::vector<CUtensorMap> reps;  // replica maps in table order
  if (n_rep && count) {
    const cudaError_t e = cudaMalloc((void**)&plan->d_rep, count * n_rep * sizeof(CUtensorMap));
    if (e != cudaSuccess) return fail(SPFY_E_CUDA, "spmma_plan_create: %s", cudaGetErrorString(e));
  }
  // launches overlap tail-to-head (programmatic stream serialization), so only the last launch's tail is
  // exposed: go from the class with the longest units (streaming, G = 2) to the one with the shortest (k <= 64)
  for (int cls = NUM_CLASSES - 1; cls >= 0; --cls) {
    for (int opB = 0; opB < 2; ++opB) {
      Plan::Launch ln;
      memset(&ln.L, 0, sizeof(ln.L));
      ln.opB = opB;
      ln.epi = false;
      ln.first = (uint32_t)table.size();
      ln.count = 0;
      uint32_t units = 0, res_vals = 0, res_meta = 0;
      for (const Member& mb : members) {
        if (mb.cls != cls || mb.h.opB != opB) continue;
        ProblemDev d;
        rc = fill_problem(&d, dtype, mb.h, cls);
        if (rc) return rc;
        d.unit_begin = units;
        if ((uint64_t)units + d.units >= (1ull << 32)) return fail(SPFY_E_UNSUPPORTED, "spmma_plan_create: too many tiles");
        units += d.units;
        if (n_rep) {
          d.tmap_rep = plan->d_rep + reps.size();
          d.n_rep = (uint32_t)n_rep;
          for (size_t r = 0; r < n_rep; ++r) {
            reps.emplace_back();
            rc = make_tmap_d(&reps.back(), dtype, mb.h, rep_d[mb.index * n_rep + r]);
            if (rc) return rc;
          }
        }
        if (d.resident && res_values_bytes(d) > res_vals) res_vals = res_values_bytes(d);
        if (d.resident && res_meta_bytes(d) > res_meta) res_meta = res_meta_bytes(d);
        ln.epi = ln.epi || d.epi;
        table.push_back(d);
        ++ln.count;
      }
      if (!ln.count) continue;
      geometry(cls, res_vals, res_meta, &ln.L, &ln.smem);
      ln.L.num_problems = ln.count;
      ln.L.total_units = units;
      ln.L.idesc = make_idesc(dtype, opB);
      ln.L.dbg = debug_mode();
      ln.grid = (int)(units < (uint32_t)di.sm_count ? units : (uint32_t)di.sm_count);
      plan->launches.push_back(ln);
    }
  }
  if (!table.empty()) {
    cudaError_t e = cudaMalloc((void**)&plan->d_table, table.size() * sizeof(ProblemDev));
    if (e == cudaSuccess)
      e = cudaMemcpy(plan->d_table, table.data(), table.size() * sizeof(ProblemDev), cudaMemcpyHostToDevice);
    if (e == cudaSuccess && !reps.empty())
      e = cudaMemcpy(plan->d_rep, reps.data(), reps.size() * sizeof(CUtensorMap), cudaMemcpyHostToDevice);
    if (e != cudaSuccess) return fail(SPFY_E_CUDA, "spmma_plan_create: %s", cudaGetErrorString(e));
    for (auto& ln : plan->launches) ln.L.table = plan->d_table + ln.first;
  }
  *out = (spfy_spmma_plan_t)plan.release();
  return SPFY_OK;
}

int spfy_spmma_plan_create(int dtype, const spfy_spmma_problem* problems, size_t count,
                           spfy_spmma_plan_t* out) {
  return plan_create_impl(dtype, problems, nullptr, nullptr, false, count, 0, nullptr, out);
}

int spfy_spmma_plan_create_conv(int dtype, const spfy_spmma_problem* problems, const spfy_conv_desc* const* convs,
                                size_t count, spfy_spmma_plan_t* out) {
  return plan_create_impl(dtype, problems, convs, nullptr, false, count, 0, nullptr, out);
}

int spfy_spmma_plan_create_ex(int dtype, const spfy_spmma_problem* problems, const spfy_conv_desc* const* convs,
                              const spfy_epilogue* const* epilogues, size_t count, spfy_spmma_plan_t* out) {
  return plan_create_impl(dtype, problems, convs, epilogues, true, count, 0, nullptr, out);
}

int spfy_spmma_plan_create_replicated(int dtype, const spfy_spmma_problem* problems, size_t count, size_t replicas,
                                      void* const* replica_d, spfy_spmma_plan_t* out) {
  if (replicas > 15) return fail(SPFY_E_UNSUPPORTED, "spmma_plan_create_replicated: %zu replicas (at most 15)", replicas);
  if (replicas && count && !replica_d) return fail(SPFY_E_INVALID, "spmma_plan_create_replicated: null replica list");
  for (size_t i = 0; i < count * replicas; ++i)
    if (problems && problems[i / replicas].m && problems[i / replicas].n && (!replica_d[i] || (uintptr_t)replica_d[i] % 16))
      return fail(SPFY_E_INVALID, "spmma_plan_create_replicated: replica %zu of problem %zu is null or not 16-byte aligned",
                  i % replicas, i / replicas);
  return plan_create_impl(dtype, problems, nullptr, nullptr, false, count, replicas, replica_d, out);
}

int spfy_spmma_plan_run(spfy_spmma_plan_t p, spfy_stream_t stream) {
  if (!p) return fail(SPFY_E_INVALID, "spmma_plan_run: null plan");
  Plan* plan = (Plan*)p;
  ProblemDev dummy;
  memset(&dummy, 0, sizeof(dummy));
  static const bool serial = dev_switch("SPFY_SPMMA_NO_OVERLAP") != nullptr;
  bool first = true;
  for (const auto& ln : plan->launches) {
    int rc = launch(plan->dtype, ln.opB, ln.epi, dummy, ln.L, ln.smem, ln.grid, (cudaStream_t)stream, !first && !serial);
    if (rc) return rc;
    first = false;
  }
  return SPFY_OK;
}

int spfy_spmma_plan_launches(spfy_spmma_plan_t p) { return p ? (int)((Plan*)p)->launches.size() : 0; }

int spfy_spmma_plan_run_launch(spfy_spmma_plan_t p, int index, spfy_stream_t stream) {
  if (!p) return fail(SPFY_E_INVALID, "spmma_plan_run_launch: null plan");
  Plan* plan = (Plan*)p;
  if (index < 0 || index >= (int)plan->launches.size())
    return fail(SPFY_E_INVALID, "spmma_plan_run_launch: launch %d of %zu", index, plan->launches.size());
  ProblemDev dummy;
  memset(&dummy, 0, sizeof(dummy));
  const auto& ln = plan->launches[index];
  return launch(plan->dtype, ln.opB, ln.epi, dummy, ln.L, ln.smem, ln.grid, (cudaStream_t)stream);
}

int spfy_spmma_plan_launch_info(spfy_spmma_plan_t p, int index, int* problems, int* units, int* stages,
                                int* smem_bytes) {
  if (!p) return fail(SPFY_E_INVALID, "spmma_plan_launch_info: null plan");
  Plan* plan = (Plan*)p;
  if (index < 0 || index >= (int)plan->launches.size())
    return fail(SPFY_E_INVALID, "spmma_plan_launch_info: launch %d of %zu", index, plan->launches.size());
  const auto& ln = plan->launches[index];
  if (problems) *problems = (int)ln.count;
  if (units) *units = (int)ln.L.total_units;
  if (stages) *stages = (int)ln.L.stages;
  if (smem_bytes) *smem_bytes = (int)ln.smem;
  return SPFY_OK;
}

int spfy_spmma_plan_destroy(spfy_spmma_plan_t p) {
  if (!p) return SPFY_OK;
  plan_free((Plan*)p);
  return SPFY_OK;
}

}  // extern "C"
