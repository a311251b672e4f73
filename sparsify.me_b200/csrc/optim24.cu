// optim24.cu -- one optimizer step (SGD or AdamW) over a whole model in one launch (sm_100a)
//
//   spfy_optim24_step : a table of items, each a dense fp32 parameter or the fp32 master of a 2:4 layer.  A 2:4 item is
//                       updated at its kept positions, re-masked (+0 in master and state) at the pruned ones, and its
//                       compressed values -- the forward operand's and, optionally, the transposed operand's -- are
//                       refilled in the same pass, byte for byte what spfy_recompress24 and spfy_transpose24(_conv)
//                       write.  The metadata never changes (the mask is fixed), so it is only read.
//
// HBM-bound like transpose24.cu: no shared memory, no workspace, every master element read and written once.
#include <vector>

#include "common.cuh"

namespace spfy {
namespace {

// ------------------------------------------------------------------------
// The launch: a grid-stride loop over CTA tiles; every tile belongs to one item (binary search on tile_prefix, as in
// prune24_batched_kernel), so the item and its rule are CTA-uniform.
//   2:4 item: one tile = one 128 x 128 tile of the transposed operand A' of one phase (transpose24_kernel's walk).  Each
//             phase owns a disjoint set of filter taps, so the tiles of all phases cover every element of A once.  An
//             item without vals_t walks A' = A^T (one phase, taps = 1), which covers A just the same.
//             Warp w takes the 16-column unit w of the A' tile, lane l its rows 4l .. 4l+3; for each of its four
//             4 x 4 blocks a lane reads four 16-byte rows of master, gradient and state(s) (the 32 lanes: 512
//             contiguous bytes of each A row), writes them back, writes the four 32-bit value pairs of `vals` (one
//             128-byte tile row per warp and row), and at the end writes four whole 16-byte chunks of vals_t.
//   dense item: one tile = 16384 consecutive elements, float4 per thread when every pointer is 16-byte aligned.
// Bytes per element (fp32 master p, gradient g, state): SGD with momentum reads p, g, buf and writes p, buf (20 B);
// AdamW reads p, g, m, v and writes p, m, v (28 B); a 2:4 item adds 1 B of vals and 1 B of vals_t per element (half
// the elements are kept, 2 B each) and 1/8 B of metadata read.
// ------------------------------------------------------------------------
constexpr int OPTIM_MAX_ITEMS = 192;   // ResNet-50's 161 parameters travel in one launch
constexpr int OPTIM_MAX_PHASES = 256;  // phase entries of all 2:4 items of one launch (one per item without vals_t)
constexpr int OPTIM_MAX_GROUPS = 16;   // hyperparameter groups per launch: a table with more takes more launches
constexpr uint32_t DENSE_TILE = 16384;

struct OptimPhase {
  uint32_t tile_begin, taps, nb, src0;  // as Transpose24Phase, tile_begin relative to the item
};
struct OptimItem {
  float* p;
  const float* g;
  float* s1;            // SGD: momentum buffer (null without momentum); AdamW: exp_avg
  float* s2;            // AdamW: exp_avg_sq
  const float* step;    // AdamW: the step count of this step
  const float* first;   // SGD (may be null): nonzero -> torch's first step, buf = g
  const uint8_t* meta;  // null: a dense item of `cols` elements
  uint8_t* vals;
  uint8_t* vals_t;      // null: not refilled
  uint32_t rows, cols, ld;   // A: rows x cols, leading dimension ld (elements)
  uint32_t C;                // A' rows: cols / taps (taps = kh * kw with vals_t, else 1)
  uint32_t m_tiles, m_tiles_t, step_h, step_w;
  uint16_t phase0, phases;   // entries of the phase pool
  uint8_t group, bf16, vec;  // group: index into this launch's group table
};
struct OptimGroup {
  double lr, beta1, beta2;  // AdamW: the bias corrections are formed in double, as torch forms them from a step count
  float wd, mom, omd, nlr;  // SGD: weight decay, momentum, 1 - dampening, -lr
  float wdmul, omb1, b2, omb2, eps;  // AdamW: 1 - lr * wd, 1 - beta1, beta2, 1 - beta2, eps
  int nesterov, has_wd;
};
struct OptimBatch {
  OptimItem item[OPTIM_MAX_ITEMS];
  OptimPhase phase[OPTIM_MAX_PHASES];
  OptimGroup group[OPTIM_MAX_GROUPS];
  uint32_t tile_prefix[OPTIM_MAX_ITEMS + 1];
  int count;
  const float* grad_scale;  // optional: divides the gradient
  const float* found_inf;   // optional: nonzero -> the launch writes nothing
};

static_assert(sizeof(OptimBatch) <= 32764, "the item table must fit the kernel parameter space");

// the per-tile constants of an item's rule
struct Rule {
  float gs;  // gradient scale (1 without one)
  float wd, mom, omd, nlr;
  float wdmul, omb1, b2, omb2, eps, nss, bc2s;  // AdamW: nss = -lr / (1 - beta1^t), bc2s = sqrt(1 - beta2^t)
  bool nesterov, has_wd, first;
};

template <int ALGO>
__device__ __forceinline__ Rule make_rule(const OptimBatch& B, const OptimItem& it) {
  const OptimGroup& G = B.group[it.group];
  Rule R;
  R.gs = B.grad_scale ? *B.grad_scale : 1.f;
  R.wd = G.wd; R.mom = G.mom; R.omd = G.omd; R.nlr = G.nlr;
  R.wdmul = G.wdmul; R.omb1 = G.omb1; R.b2 = G.b2; R.omb2 = G.omb2; R.eps = G.eps;
  R.nesterov = G.nesterov != 0; R.has_wd = G.has_wd != 0; R.first = it.first && *it.first != 0.f;
  R.nss = 0.f; R.bc2s = 1.f;
  if (ALGO == SPFY_OPTIM_ADAMW) {
    const double t = (double)*it.step;
    R.nss = (float)(-(G.lr / (1.0 - pow(G.beta1, t))));
    R.bc2s = (float)sqrt(1.0 - pow(G.beta2, t));
  }
  return R;
}

// One element, operation by operation as torch's _multi_tensor_sgd / _multi_tensor_adam (decoupled weight decay) in fp32
template <int ALGO>
__device__ __forceinline__ void update(const Rule& R, float& p, float g, float& s1, float& s2) {
  if (R.gs != 1.f) g = g / R.gs;
  if (ALGO == SPFY_OPTIM_SGD) {
    if (R.has_wd) g = fmaf(R.wd, p, g);                        // grad + wd * p
    if (R.mom != 0.f) {
      s1 = R.first ? g : fmaf(R.omd, g, s1 * R.mom);            // buf = grad | buf * mom + (1 - damp) * grad
      g = R.nesterov ? fmaf(R.mom, s1, g) : s1;
    }
    p = fmaf(R.nlr, g, p);                                      // p - lr * grad
  } else {
    if (R.has_wd) p = p * R.wdmul;                              // p * (1 - lr * wd)
    s1 = fmaf(R.omb1, g - s1, s1);                              // lerp(m, g, 1 - beta1)
    s2 = fmaf(R.omb2 * g, g, s2 * R.b2);                        // v * beta2 + (1 - beta2) * g * g
    const float denom = sqrtf(s2) / R.bc2s + R.eps;
    p = fmaf(R.nss, s1 / denom, p);                             // p - step_size * m / denom
  }
}

template <int ALGO>
__device__ __forceinline__ void dense_tile(const OptimItem& it, const Rule& R, uint32_t local) {
  const size_t n = it.cols, base = (size_t)local * DENSE_TILE;
  const bool st = ALGO == SPFY_OPTIM_ADAMW || R.mom != 0.f;
  if (it.vec) {
#pragma unroll 1
    for (uint32_t k = 0; k < DENSE_TILE / 1024u; ++k) {
      const size_t i = base + (size_t)(k * 256u + threadIdx.x) * 4u;
      if (i >= n) break;
      if (i + 4 <= n) {
        float4 p = *reinterpret_cast<const float4*>(it.p + i), g = *reinterpret_cast<const float4*>(it.g + i);
        float4 a = st ? *reinterpret_cast<const float4*>(it.s1 + i) : make_float4(0.f, 0.f, 0.f, 0.f);
        float4 b = ALGO == SPFY_OPTIM_ADAMW ? *reinterpret_cast<const float4*>(it.s2 + i) : make_float4(0.f, 0.f, 0.f, 0.f);
        update<ALGO>(R, p.x, g.x, a.x, b.x);
        update<ALGO>(R, p.y, g.y, a.y, b.y);
        update<ALGO>(R, p.z, g.z, a.z, b.z);
        update<ALGO>(R, p.w, g.w, a.w, b.w);
        *reinterpret_cast<float4*>(it.p + i) = p;
        if (st) *reinterpret_cast<float4*>(it.s1 + i) = a;
        if (ALGO == SPFY_OPTIM_ADAMW) *reinterpret_cast<float4*>(it.s2 + i) = b;
      } else {
        for (size_t e = i; e < n; ++e) {
          float p = it.p[e], a = st ? it.s1[e] : 0.f, b = ALGO == SPFY_OPTIM_ADAMW ? it.s2[e] : 0.f;
          update<ALGO>(R, p, it.g[e], a, b);
          it.p[e] = p;
          if (st) it.s1[e] = a;
          if (ALGO == SPFY_OPTIM_ADAMW) it.s2[e] = b;
        }
      }
    }
  } else {
#pragma unroll 1
    for (uint32_t k = 0; k < DENSE_TILE / 256u; ++k) {
      const size_t e = base + k * 256u + threadIdx.x;
      if (e >= n) break;
      float p = it.p[e], a = st ? it.s1[e] : 0.f, b = ALGO == SPFY_OPTIM_ADAMW ? it.s2[e] : 0.f;
      update<ALGO>(R, p, it.g[e], a, b);
      it.p[e] = p;
      if (st) it.s1[e] = a;
      if (ALGO == SPFY_OPTIM_ADAMW) it.s2[e] = b;
    }
  }
}

__device__ __forceinline__ uint32_t raw16(bool bf16, float f) {
  return bf16 ? (uint32_t)__bfloat16_as_ushort(__float2bfloat16_rn(f)) : (uint32_t)__half_as_ushort(__float2half_rn(f));
}

__device__ __forceinline__ float pick(float4 v, uint32_t i) { return i == 0 ? v.x : i == 1 ? v.y : i == 2 ? v.z : v.w; }

template <int ALGO>
__device__ __forceinline__ void sparse_tile(const OptimBatch& B, const OptimItem& it, const Rule& R, uint32_t local) {
  const uint32_t lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
  uint32_t p = it.phase0;
  const uint32_t pend = it.phase0 + it.phases;
  while (p + 1u < pend && local >= B.phase[p + 1u].tile_begin) ++p;
  const OptimPhase& ph = B.phase[p];
  local -= ph.tile_begin;
  const uint32_t cols_t = ph.taps * it.rows;
  const uint32_t kt = local / it.m_tiles_t, mt = local - kt * it.m_tiles_t;  // A' storage order: k-tile major
  const uint32_t ci0 = mt * 128u + lane * 4u, j0 = kt * 128u + w * 16u;
  if (ci0 >= it.C) return;  // the lane's four A' rows are padding (C % 8 == 0)
  const bool st = ALGO == SPFY_OPTIM_ADAMW || R.mom != 0.f;
  const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);
  uint32_t ov[4][4];  // [A' row j][group k]: the two kept values
#pragma unroll
  for (int k = 0; k < 4; ++k) {
    const uint32_t col = j0 + 4u * k;
#pragma unroll
    for (int j = 0; j < 4; ++j) ov[j][k] = 0u;
    if (col >= cols_t) continue;  // padding of A': +0
    const uint32_t tp = col / it.rows, r0 = col - tp * it.rows;
    const uint32_t th = tp / ph.nb;
    const uint32_t src = ph.src0 - th * it.step_h - (tp - th * ph.nb) * it.step_w;  // source tap of A' tap tp
    const uint32_t c = src * it.C + ci0;  // first column of the A block
    const uint32_t q = (c & 127u) >> 4, g = (c >> 2) & 3u;
    uint32_t v[4], n[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const uint32_t row = r0 + i, r = row & 127u;
      const size_t t = (size_t)(c >> 7) * it.m_tiles + (row >> 7);
      n[i] = (*reinterpret_cast<const uint16_t*>(it.meta + t * 2048 + sm100_meta_word(r, q)) >> (4u * g)) & 0xfu;
      const size_t e = (size_t)row * it.ld + c;
      float4 pv = *reinterpret_cast<const float4*>(it.p + e);
      const float4 gv = *reinterpret_cast<const float4*>(it.g + e);
      float4 a = st ? *reinterpret_cast<const float4*>(it.s1 + e) : zero4;
      float4 b = ALGO == SPFY_OPTIM_ADAMW ? *reinterpret_cast<const float4*>(it.s2 + e) : zero4;
      update<ALGO>(R, pv.x, gv.x, a.x, b.x);
      update<ALGO>(R, pv.y, gv.y, a.y, b.y);
      update<ALGO>(R, pv.z, gv.z, a.z, b.z);
      update<ALGO>(R, pv.w, gv.w, a.w, b.w);
      const uint32_t i0 = n[i] & 3u, i1 = n[i] >> 2;
      const uint32_t keep = (1u << i0) | (1u << i1);
      // re-mask: +0 at the pruned positions (whatever the gradient held there)
      pv = make_float4(keep & 1u ? pv.x : 0.f, keep & 2u ? pv.y : 0.f, keep & 4u ? pv.z : 0.f, keep & 8u ? pv.w : 0.f);
      *reinterpret_cast<float4*>(it.p + e) = pv;
      if (st) {
        a = make_float4(keep & 1u ? a.x : 0.f, keep & 2u ? a.y : 0.f, keep & 4u ? a.z : 0.f, keep & 8u ? a.w : 0.f);
        *reinterpret_cast<float4*>(it.s1 + e) = a;
      }
      if (ALGO == SPFY_OPTIM_ADAMW) {
        b = make_float4(keep & 1u ? b.x : 0.f, keep & 2u ? b.y : 0.f, keep & 4u ? b.z : 0.f, keep & 8u ? b.w : 0.f);
        *reinterpret_cast<float4*>(it.s2 + e) = b;
      }
      v[i] = raw16(it.bf16, pick(pv, i0)) | (raw16(it.bf16, pick(pv, i1)) << 16);
      *reinterpret_cast<uint32_t*>(it.vals + t * 16384 + sm100_val_chunk(r, q) + g * 4u) = v[i];
    }
    if (!it.vals_t) continue;
    // A' group (row ci0 + j, this block) keeps A[r0 + i][c + j] for every i whose nibble names column j
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      uint32_t cnt = 0, lo = 0, hi = 0;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const uint32_t a = n[i] & 3u, b = n[i] >> 2;
        if (a != (uint32_t)j && b != (uint32_t)j) continue;
        const uint32_t val = a == (uint32_t)j ? (v[i] & 0xffffu) : (v[i] >> 16);
        if (cnt == 0) lo = val; else hi = val;
        ++cnt;
      }
      ov[j][k] = lo | (hi << 16);
    }
  }
  if (!it.vals_t || j0 >= cols_t) return;
  uint8_t* vt = it.vals_t + ((size_t)ph.tile_begin + local) * 16384;
#pragma unroll
  for (int j = 0; j < 4; ++j)
    *reinterpret_cast<uint4*>(vt + sm100_val_chunk(lane * 4u + j, w)) = make_uint4(ov[j][0], ov[j][1], ov[j][2], ov[j][3]);
}

template <int ALGO>
__global__ void __launch_bounds__(256)
optim24_kernel(const __grid_constant__ OptimBatch B) {
  if (B.found_inf && *B.found_inf != 0.f) return;  // GradScaler found an inf / NaN: the step is skipped
  const uint32_t tiles = B.tile_prefix[B.count];
  for (uint32_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    int lo = 0, hi = B.count - 1;  // last item with tile_prefix <= tile
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (B.tile_prefix[mid] <= tile) lo = mid; else hi = mid - 1;
    }
    const OptimItem& it = B.item[lo];
    const Rule R = make_rule<ALGO>(B, it);
    if (it.meta) sparse_tile<ALGO>(B, it, R, tile - B.tile_prefix[lo]);
    else dense_tile<ALGO>(it, R, tile - B.tile_prefix[lo]);
  }
}

bool misaligned(const void* p, size_t a) { return (uintptr_t)p % a != 0; }

}  // namespace
}  // namespace spfy

void spfy::warm_optim24_kernels() {
  touch_kernel(optim24_kernel<SPFY_OPTIM_SGD>);
  touch_kernel(optim24_kernel<SPFY_OPTIM_ADAMW>);
}

using namespace spfy;

extern "C" {

int spfy_optim24_step(int algo, const spfy_optim24_item* items, size_t count, const spfy_optim24_hparams* groups,
                      size_t n_groups, const float* grad_scale, const float* found_inf, spfy_stream_t stream) {
  if (algo != SPFY_OPTIM_SGD && algo != SPFY_OPTIM_ADAMW) return fail(SPFY_E_INVALID, "optim24_step: bad algo %d", algo);
  if ((count && !items) || (n_groups && !groups)) return fail(SPFY_E_INVALID, "optim24_step: null table");
  if (misaligned(grad_scale, 4) || misaligned(found_inf, 4))
    return fail(SPFY_E_INVALID, "optim24_step: grad_scale / found_inf not aligned");
  static thread_local OptimBatch B;  // 28 KB: keep it off the stack
  B.grad_scale = grad_scale;
  B.found_inf = found_inf;
  std::vector<OptimGroup> all(n_groups);
  for (size_t gi = 0; gi < n_groups; ++gi) {
    const spfy_optim24_hparams& h = groups[gi];
    if (!(h.lr >= 0.0) || (algo == SPFY_OPTIM_ADAMW && !(h.eps >= 0.0)))
      return fail(SPFY_E_INVALID, "optim24_step: group %zu: negative lr or eps", gi);
    if (algo == SPFY_OPTIM_SGD && h.nesterov && (h.momentum <= 0.0 || h.dampening != 0.0))
      return fail(SPFY_E_INVALID, "optim24_step: group %zu: nesterov needs momentum > 0 and dampening = 0", gi);
    OptimGroup& G = all[gi];
    G.lr = h.lr;
    G.beta1 = h.beta1;
    G.beta2 = h.beta2;
    G.wd = (float)h.weight_decay;
    G.mom = (float)h.momentum;
    G.omd = (float)(1.0 - h.dampening);
    G.nlr = (float)(-h.lr);
    G.wdmul = (float)(1.0 - h.lr * h.weight_decay);
    G.omb1 = (float)(1.0 - h.beta1);
    G.b2 = (float)h.beta2;
    G.omb2 = (float)(1.0 - h.beta2);
    G.eps = (float)h.eps;
    G.nesterov = h.nesterov != 0;
    G.has_wd = h.weight_decay != 0.0;
  }
  // every refusal comes before the first launch
  for (size_t i = 0; i < count; ++i) {
    const spfy_optim24_item& it = items[i];
    if (it.rows == 0 || it.cols == 0) continue;  // an empty parameter: nothing to read, its pointers may be null
    if (it.group >= n_groups) return fail(SPFY_E_INVALID, "optim24_step: item %zu: group %zu out of range", i, it.group);
    const spfy_optim24_hparams& h = groups[it.group];
    if (!it.param || !it.grad) return fail(SPFY_E_INVALID, "optim24_step: item %zu: null param or grad", i);
    if (algo == SPFY_OPTIM_SGD && h.momentum != 0.0 && !it.state1)
      return fail(SPFY_E_INVALID, "optim24_step: item %zu: momentum without a momentum buffer", i);
    if (algo == SPFY_OPTIM_ADAMW && (!it.state1 || !it.state2 || !it.step))
      return fail(SPFY_E_INVALID, "optim24_step: item %zu: AdamW needs exp_avg, exp_avg_sq and step", i);
    const size_t a = it.meta ? 16 : 4;
    if (misaligned(it.param, a) || misaligned(it.grad, a) || misaligned(it.state1, a) || misaligned(it.state2, a) ||
        misaligned(it.step, 4) || misaligned(it.first, 4))
      return fail(SPFY_E_INVALID, "optim24_step: item %zu: fp32 buffers not %zu-byte aligned", i, a);
    if (!it.meta) {
      if (it.rows * it.cols >= (1ull << 31)) return fail(SPFY_E_UNSUPPORTED, "optim24_step: item %zu too large", i);
      continue;
    }
    if (it.dtype != SPFY_F16 && it.dtype != SPFY_BF16)
      return fail(SPFY_E_UNSUPPORTED, "optim24_step: item %zu: dtype %d (need F16/BF16)", i, it.dtype);
    if (!it.vals) return fail(SPFY_E_INVALID, "optim24_step: item %zu: null vals", i);
    if (misaligned(it.meta, 16) || misaligned(it.vals, 16) || misaligned(it.vals_t, 16))
      return fail(SPFY_E_INVALID, "optim24_step: item %zu: SM100 buffers must be 16-byte aligned", i);
    if (it.ld < it.cols || it.ld % 4) return fail(SPFY_E_INVALID, "optim24_step: item %zu: ld %zu", i, it.ld);
    if (it.rows % 8 || it.cols % 8)
      return fail(SPFY_E_UNSUPPORTED, "optim24_step: item %zu: rows (%zu) and cols (%zu) must be multiples of 8", i,
                  it.rows, it.cols);
    if (it.rows >= (1ull << 24) || it.cols >= (1ull << 24) || it.ld >= (1ull << 31) || it.rows * it.ld >= (1ull << 40))
      return fail(SPFY_E_UNSUPPORTED, "optim24_step: item %zu too large", i);
    if (it.vals_t) {
      const size_t taps = it.kh * it.kw;
      if (!taps || !it.stride || it.cols % taps || (it.cols / taps) % 8)
        return fail(SPFY_E_UNSUPPORTED, "optim24_step: item %zu: cols %zu is not kh*kw*c with c %% 8 == 0", i, it.cols);
      if (it.kh > 16 || it.kw > 16 || it.pad > 8 || it.stride > 8)
        return fail(SPFY_E_UNSUPPORTED, "optim24_step: item %zu: filter / padding / stride outside what the "
                    "convolutions accept", i);
    }
  }
  cudaStream_t s = (cudaStream_t)stream;
  auto launch = [&]() -> int {
    if (B.count == 0 || B.tile_prefix[B.count] == 0) return SPFY_OK;
    int grid = 1;
    int rc = capped_grid(B.tile_prefix[B.count], 8, &grid);
    if (rc) return rc;
    if (algo == SPFY_OPTIM_SGD) optim24_kernel<SPFY_OPTIM_SGD><<<grid, 256, 0, s>>>(B);
    else optim24_kernel<SPFY_OPTIM_ADAMW><<<grid, 256, 0, s>>>(B);
    SPFY_LAUNCH_OK("optim24_kernel");
    return SPFY_OK;
  };
  // a launch ends when its items, phases, groups or tiles would overflow; `local` maps a group to its slot in the
  // launch's group table (-1: not in it)
  std::vector<int> local(n_groups, -1);
  int ngl = 0;
  B.count = 0;
  B.tile_prefix[0] = 0;
  uint32_t nph = 0;
  for (size_t i = 0; i < count; ++i) {
    const spfy_optim24_item& it = items[i];
    if (it.rows == 0 || it.cols == 0) continue;
    // the item's phases: those of spfy_transpose24_conv with vals_t, else one phase of A^T
    OptimPhase ph[64];
    uint32_t phases = 1, tiles = 0, C = (uint32_t)it.cols, step_h = 1, step_w = 1;
    if (!it.meta) {
      tiles = (uint32_t)ceil_div(it.rows * it.cols, DENSE_TILE);
    } else if (!it.vals_t) {
      ph[0] = OptimPhase{0u, 1u, 1u, 0u};
      tiles = (uint32_t)(ceil_div(it.cols, 128) * ceil_div(it.rows, 128));
    } else {
      C = (uint32_t)(it.cols / (it.kh * it.kw));
      step_h = (uint32_t)(it.stride * it.kw);
      step_w = (uint32_t)it.stride;
      phases = 0;
      for (size_t a = 0; a < it.stride; ++a)
        for (size_t b = 0; b < it.stride; ++b) {
          const DgradPhase dh = dgrad_phase(it.kh, it.stride, it.pad, a), dw = dgrad_phase(it.kw, it.stride, it.pad, b);
          if (!dh.taps || !dw.taps) continue;
          OptimPhase& q = ph[phases++];
          q.tile_begin = tiles;
          q.taps = dh.taps * dw.taps;
          q.nb = dw.taps;
          q.src0 = dh.k0 * (uint32_t)it.kw + dw.k0;
          tiles += (uint32_t)(ceil_div(C, 128) * ceil_div((size_t)q.taps * it.rows, 128));
        }
    }
    if (B.count == OPTIM_MAX_ITEMS || nph + phases > (uint32_t)OPTIM_MAX_PHASES ||
        (local[it.group] < 0 && ngl == OPTIM_MAX_GROUPS) || (uint64_t)B.tile_prefix[B.count] + tiles >= (1ull << 32)) {
      int rc = launch();
      if (rc) return rc;
      B.count = 0;
      B.tile_prefix[0] = 0;
      nph = 0;
      std::fill(local.begin(), local.end(), -1);
      ngl = 0;
    }
    if (local[it.group] < 0) {
      local[it.group] = ngl;
      B.group[ngl++] = all[it.group];
    }
    OptimItem& d = B.item[B.count];
    d.p = it.param;
    d.g = it.grad;
    d.s1 = it.state1;
    d.s2 = it.state2;
    d.step = it.step;
    d.meta = (const uint8_t*)it.meta;
    d.vals = (uint8_t*)it.vals;
    d.vals_t = (uint8_t*)it.vals_t;
    d.first = it.first;
    d.group = (uint8_t)local[it.group];
    d.bf16 = it.dtype == SPFY_BF16;
    if (!it.meta) {
      d.rows = 1;
      d.cols = (uint32_t)(it.rows * it.cols);
      d.vec = !misaligned(it.param, 16) && !misaligned(it.grad, 16) && !misaligned(it.state1, 16) &&
              !misaligned(it.state2, 16);
      d.phases = 0;
    } else {
      d.rows = (uint32_t)it.rows;
      d.cols = (uint32_t)it.cols;
      d.ld = (uint32_t)it.ld;
      d.C = C;
      d.m_tiles = (uint32_t)ceil_div(it.rows, 128);
      d.m_tiles_t = (uint32_t)ceil_div(C, 128);
      d.step_h = step_h;
      d.step_w = step_w;
      d.phase0 = (uint16_t)nph;
      d.phases = (uint16_t)phases;
      for (uint32_t k = 0; k < phases; ++k) B.phase[nph++] = ph[k];
    }
    B.tile_prefix[B.count + 1] = B.tile_prefix[B.count] + tiles;
    ++B.count;
  }
  return launch();
}

}  // extern "C"
