// transpose24.cu -- 2:4 fine-tuning support on compressed operands (sm_100a)
//
//   spfy_transpose24  : SM100 compressed A -> SM100 compressed A' (A^T, or the flipped, channel-swapped filter of a
//                       convolution's data gradient).  Valid when A's mask keeps two of four along columns too (TILE).
//   spfy_transpose24_conv : the same for a strided convolution: one A' per output phase of its data gradient, each
//                       built from the phase's subset of filter taps, all in one launch.
//   spfy_recompress24 : new values under a fixed mask: dense (F32 / F16 / BF16) -> compressed values at the positions an
//                       existing operand's metadata keeps, and / or the dense input with the pruned positions zeroed.
//
// Both are HBM-bound byte movers like prune.cu: no shared memory, no workspace, one pass.
#include "common.cuh"

namespace spfy {
namespace {

// ------------------------------------------------------------------------
// transpose24
// A is rows x (taps * C), A' is C x (taps * rows):  A'[ci][t' * rows + r] = A[r][(taps - 1 - t') * C + ci].
// rows % 8 == 0 and C % 8 == 0, so a 4x4 block of A maps whole onto a 4x4 block of A', and the four 2:4 groups of an
// A' block are the four columns of the A block.
// One CTA writes one 128 x 128 tile of A': warp w the 16-column unit w of every row, lane l the rows 4l .. 4l + 3.
// Every lane of a warp reads the same A rows, 32 consecutive 4-column groups of them: 128 contiguous bytes of values.
// ------------------------------------------------------------------------
// PHASED (spfy_transpose24_conv): the output is several A', one per phase of a strided convolution's data gradient, back
// to back in tile order.  Phase ph owns the tiles [tile_begin, next tile_begin) and its column tap t' = th * nb + tw
// reads the source tap src0 - th * step_h - tw * step_w.  One phase with nb = 1, src0 = taps - 1 and step_h = 1 is the
// plain transpose.
constexpr int MAX_PHASES = 64;  // stride <= 8 in both dimensions
struct Transpose24Phase {
  uint32_t tile_begin, taps, nb, src0;
};
struct Transpose24Params {
  const uint8_t* vals;
  const uint8_t* meta;
  uint8_t* vals_t;
  uint8_t* meta_t;
  uint32_t rows, C, taps;  // A: rows x (taps * C)
  uint32_t m_tiles;        // A: 128-row tiles
  uint32_t m_tiles_t;      // A': 128-row tiles (of C rows)
  uint32_t tiles_t;        // A': tiles (of all phases)
  int* invalid;
};
// the phase table, a kernel parameter of its own: the plain transpose passes a one-entry table it never reads, so its
// launches do not carry the 1 KiB of a full one
template <int N>
struct Transpose24Phases {
  uint32_t phases, step_h, step_w;
  Transpose24Phase ph[N];
};

template <bool PHASED>
__global__ void __launch_bounds__(256)
transpose24_kernel(const __grid_constant__ Transpose24Params P,
                   const __grid_constant__ Transpose24Phases<PHASED ? MAX_PHASES : 1> T) {
  const uint32_t lane = threadIdx.x & 31u, w = threadIdx.x >> 5;
  uint32_t cols_t = P.taps * P.rows;
  bool bad = false;
  for (uint32_t tile = blockIdx.x; tile < P.tiles_t; tile += gridDim.x) {
    uint32_t local = tile, nb = 1u, src0 = P.taps - 1u;
    if (PHASED) {
      uint32_t p = 0;
      while (p + 1u < T.phases && tile >= T.ph[p + 1u].tile_begin) ++p;
      local = tile - T.ph[p].tile_begin;
      cols_t = T.ph[p].taps * P.rows;
      nb = T.ph[p].nb;
      src0 = T.ph[p].src0;
    }
    const uint32_t kt = local / P.m_tiles_t, mt = local - kt * P.m_tiles_t;  // storage order: k-tile major
    const uint32_t ci0 = mt * 128u + lane * 4u, j0 = kt * 128u + w * 16u;
    uint32_t ov[4][4];                  // [A' row j][group k]: the two kept values
    uint32_t on[4] = {0u, 0u, 0u, 0u};  // [A' row j]: the unit's four nibbles
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const uint32_t col = j0 + 4u * k;
      if (ci0 >= P.C || col >= cols_t) {  // padding of A': +0, neutral nibble
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          ov[j][k] = 0u;
          on[j] |= 0x4u << (4 * k);
        }
        continue;
      }
      const uint32_t tp = col / P.rows, r0 = col - tp * P.rows;
      uint32_t src = P.taps - 1u - tp;  // source tap of A' tap tp
      if (PHASED) {
        const uint32_t th = tp / nb;
        src = src0 - th * T.step_h - (tp - th * nb) * T.step_w;
      }
      const uint32_t c = src * P.C + ci0;  // first column of the A block
      const uint32_t q = (c & 127u) >> 4, g = (c >> 2) & 3u;
      uint32_t v[4], n[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const uint32_t row = r0 + i, r = row & 127u;
        const size_t t = (size_t)(c >> 7) * P.m_tiles + (row >> 7);
        v[i] = *reinterpret_cast<const uint32_t*>(P.vals + t * 16384 + sm100_val_chunk(r, q) + g * 4u);
        n[i] = (*reinterpret_cast<const uint16_t*>(P.meta + t * 2048 + sm100_meta_word(r, q)) >> (4u * g)) & 0xfu;
      }
      // A' group (row ci0 + j, this block) keeps A[r0 + i][c + j] for every i whose nibble names column j
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        uint32_t cnt = 0, lo = 0, hi = 0, i0 = 0, i1 = 0;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const uint32_t a = n[i] & 3u, b = n[i] >> 2;
          if (a != (uint32_t)j && b != (uint32_t)j) continue;
          const uint32_t val = a == (uint32_t)j ? (v[i] & 0xffffu) : (v[i] >> 16);
          if (cnt == 0) { lo = val; i0 = i; } else { hi = val; i1 = i; }
          ++cnt;
        }
        bad |= cnt != 2u;
        ov[j][k] = lo | (hi << 16);
        on[j] |= (i0 | (i1 << 2)) << (4 * k);
      }
    }
    uint8_t* vt = P.vals_t + (size_t)tile * 16384;
    uint8_t* et = P.meta_t + (size_t)tile * 2048;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const uint32_t r = lane * 4u + j;
      *reinterpret_cast<uint4*>(vt + sm100_val_chunk(r, w)) = make_uint4(ov[j][0], ov[j][1], ov[j][2], ov[j][3]);
      *reinterpret_cast<uint16_t*>(et + sm100_meta_word(r, w)) = (uint16_t)on[j];
    }
  }
  if (P.invalid && __any_sync(0xffffffffu, bad) && lane == 0) atomicExch(P.invalid, 1);
}

// ------------------------------------------------------------------------
// recompress24
// One thread = one 16-column unit of one row, walked in SM100 tile storage order like prune24_unit: 8 consecutive
// threads write the 128 value bytes of one tile row.  Padding rows and columns of the operand get +0; the metadata is
// only read.
// ------------------------------------------------------------------------
struct Recompress24Params {
  const void* in;
  size_t ld_in;
  const uint8_t* meta;
  uint8_t* comp_vals;
  void* out;  // may alias in: the same thread reads, then writes, the same elements
  size_t ld_out;
  uint32_t rows, cols, m_tiles, k_tiles;
  int vec_in, vec_out;  // 16-byte loads / stores of whole units
};

template <int IN_DT> struct RawOf { using T = uint16_t; };
template <> struct RawOf<SPFY_F32> { using T = uint32_t; };

template <int DT>
__device__ __forceinline__ float raw_to_f32(uint32_t b) {
  if (DT == SPFY_F32) return __uint_as_float(b);
  if (DT == SPFY_F16) return __half2float(__ushort_as_half((unsigned short)b));
  return __bfloat162float(__ushort_as_bfloat16((unsigned short)b));
}
template <int DT>
__device__ __forceinline__ uint32_t f32_to_raw16(float f) {
  if (DT == SPFY_F16) return __half_as_ushort(__float2half_rn(f));
  return __bfloat16_as_ushort(__float2bfloat16_rn(f));
}
// the compressed value of one input element: its bits when the types match, else rounded to nearest even
template <int IN_DT, int DT>
__device__ __forceinline__ uint32_t comp_bits(uint32_t raw) {
  if (IN_DT == DT) return raw;
  return f32_to_raw16<DT>(raw_to_f32<IN_DT>(raw));
}

template <int IN_DT, int DT>
__global__ void __launch_bounds__(256)
recompress24_kernel(const __grid_constant__ Recompress24Params P) {
  using Raw = typename RawOf<IN_DT>::T;
  constexpr int VECS = 16 * (int)sizeof(Raw) / 16;  // uint4 per unit
  const size_t total = (size_t)P.m_tiles * P.k_tiles * 1024;
  const size_t nthreads = (size_t)gridDim.x * blockDim.x;
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += nthreads) {
    const uint32_t tile = (uint32_t)(t >> 10);
    const uint32_t mt = tile / P.k_tiles, kt = tile - mt * P.k_tiles;
    const uint32_t r = ((uint32_t)t >> 3) & 127u, q = (uint32_t)t & 7u;
    const uint32_t row = mt * 128u + r, c0 = kt * 128u + q * 16u;
    const size_t st = (size_t)kt * P.m_tiles + mt;  // storage index
    uint8_t* cv_dst = P.comp_vals ? P.comp_vals + st * 16384 + sm100_val_chunk(r, q) : nullptr;
    if (row >= P.rows || c0 >= P.cols) {
      if (cv_dst) *reinterpret_cast<uint4*>(cv_dst) = make_uint4(0u, 0u, 0u, 0u);
      continue;
    }
    const uint32_t nibs = *reinterpret_cast<const uint16_t*>(P.meta + st * 2048 + sm100_meta_word(r, q));
    union {
      Raw e[16];
      uint4 v[VECS];
    } x;
    const Raw* src = reinterpret_cast<const Raw*>(P.in) + (size_t)row * P.ld_in + c0;
    const bool full = c0 + 16u <= P.cols;
    if (full && P.vec_in) {
#pragma unroll
      for (int i = 0; i < VECS; ++i) x.v[i] = reinterpret_cast<const uint4*>(src)[i];
    } else {
#pragma unroll
      for (int i = 0; i < 16; ++i) x.e[i] = c0 + i < P.cols ? src[i] : (Raw)0;
    }
    uint32_t keep = 0, cv[4];
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      const uint32_t i0 = (nibs >> (4 * g)) & 3u, i1 = (nibs >> (4 * g + 2)) & 3u;
      keep |= ((1u << i0) | (1u << i1)) << (4 * g);
      // (selects, not x.e[4 * g + i]: a run-time index would put x in local memory)
      const Raw e0 = x.e[4 * g], e1 = x.e[4 * g + 1], e2 = x.e[4 * g + 2], e3 = x.e[4 * g + 3];
      const Raw k0 = i0 == 0 ? e0 : i0 == 1 ? e1 : i0 == 2 ? e2 : e3, k1 = i1 == 0 ? e0 : i1 == 1 ? e1 : i1 == 2 ? e2 : e3;
      cv[g] = comp_bits<IN_DT, DT>(k0) | (comp_bits<IN_DT, DT>(k1) << 16);
    }
    if (cv_dst) *reinterpret_cast<uint4*>(cv_dst) = make_uint4(cv[0], cv[1], cv[2], cv[3]);
    if (P.out) {
#pragma unroll
      for (int i = 0; i < 16; ++i)
        if (!(keep >> i & 1u)) x.e[i] = (Raw)0;
      Raw* dst = reinterpret_cast<Raw*>(P.out) + (size_t)row * P.ld_out + c0;
      if (full && P.vec_out) {
#pragma unroll
        for (int i = 0; i < VECS; ++i) reinterpret_cast<uint4*>(dst)[i] = x.v[i];
      } else {
#pragma unroll
        for (int i = 0; i < 16; ++i)
          if (c0 + i < P.cols) dst[i] = x.e[i];
      }
    }
  }
}

template <int IN_DT>
void launch_recompress24(int dtype, int grid, const Recompress24Params& P, cudaStream_t s) {
  if (dtype == SPFY_BF16) recompress24_kernel<IN_DT, SPFY_BF16><<<grid, 256, 0, s>>>(P);
  else recompress24_kernel<IN_DT, SPFY_F16><<<grid, 256, 0, s>>>(P);
}

bool misaligned16(const void* p) { return (uintptr_t)p % 16 != 0; }

// the phase table of spfy_transpose24_conv: every phase (a, b) with taps in both dimensions, in (a, b) row-major order;
// `tiles` = the tiles of all of them
int conv_phase_table(const char* who, size_t m, size_t c, size_t kh, size_t kw, size_t stride, size_t pad,
                     Transpose24Phases<MAX_PHASES>* P, size_t* tiles) {
  if (!m || !c || !kh || !kw || !stride) return fail(SPFY_E_INVALID, "%s: empty dimension", who);
  if (m % 8 || c % 8) return fail(SPFY_E_UNSUPPORTED, "%s: m (%zu) and c (%zu) must be multiples of 8", who, m, c);
  if (kh > 16 || kw > 16 || pad > 8 || stride > 8)
    return fail(SPFY_E_UNSUPPORTED, "%s: filter / padding / stride outside what the convolutions accept", who);
  if (m >= (1ull << 24) || c >= (1ull << 24)) return fail(SPFY_E_UNSUPPORTED, "%s: dimension too large", who);
  P->phases = 0;
  P->step_h = (uint32_t)(stride * kw);
  P->step_w = (uint32_t)stride;
  size_t t = 0;
  for (size_t a = 0; a < stride; ++a)
    for (size_t b = 0; b < stride; ++b) {
      const DgradPhase ph = dgrad_phase(kh, stride, pad, a), pw = dgrad_phase(kw, stride, pad, b);
      if (!ph.taps || !pw.taps) continue;
      Transpose24Phase& q = P->ph[P->phases++];
      q.tile_begin = (uint32_t)t;
      q.taps = ph.taps * pw.taps;
      q.nb = pw.taps;
      q.src0 = ph.k0 * (uint32_t)kw + pw.k0;
      t += ceil_div(c, 128) * ceil_div(q.taps * m, 128);
    }
  if (t >= (1ull << 22)) return fail(SPFY_E_UNSUPPORTED, "%s: more than 2^22 SM100 tiles", who);
  *tiles = t;
  return SPFY_OK;
}

}  // namespace
}  // namespace spfy

void spfy::warm_transpose24_kernels() {
  touch_kernel(transpose24_kernel<false>);
  touch_kernel(transpose24_kernel<true>);
  touch_kernel(recompress24_kernel<SPFY_F32, SPFY_F16>);
  touch_kernel(recompress24_kernel<SPFY_F32, SPFY_BF16>);
  touch_kernel(recompress24_kernel<SPFY_F16, SPFY_F16>);
  touch_kernel(recompress24_kernel<SPFY_F16, SPFY_BF16>);
  touch_kernel(recompress24_kernel<SPFY_BF16, SPFY_F16>);
  touch_kernel(recompress24_kernel<SPFY_BF16, SPFY_BF16>);
}

using namespace spfy;

extern "C" {

int spfy_transpose24(int dtype, const void* vals, const void* meta, size_t rows, size_t cols, size_t taps,
                     void* vals_t, void* meta_t, int* d_invalid, spfy_stream_t stream) {
  if (dtype != SPFY_F16 && dtype != SPFY_BF16)
    return fail(SPFY_E_UNSUPPORTED, "transpose24: dtype %d (need F16/BF16)", dtype);
  if (taps == 0) return fail(SPFY_E_INVALID, "transpose24: taps == 0");
  if (!vals || !meta || !vals_t || !meta_t) return fail(SPFY_E_INVALID, "transpose24: null pointer");
  if (cols % taps) return fail(SPFY_E_INVALID, "transpose24: cols %zu is not a multiple of taps %zu", cols, taps);
  const size_t C = cols / taps;
  if (rows % 8 || C % 8)
    return fail(SPFY_E_UNSUPPORTED, "transpose24: rows (%zu) and cols / taps (%zu) must be multiples of 8", rows, C);
  if (rows >= (1ull << 31) || cols >= (1ull << 31))
    return fail(SPFY_E_UNSUPPORTED, "transpose24: dimension too large");
  if (ceil_div(rows, 128) * ceil_div(cols, 128) >= (1ull << 22) || ceil_div(C, 128) * ceil_div(taps * rows, 128) >= (1ull << 22))
    return fail(SPFY_E_UNSUPPORTED, "transpose24: more than 2^22 SM100 tiles");
  if (misaligned16(vals) || misaligned16(meta) || misaligned16(vals_t) || misaligned16(meta_t))
    return fail(SPFY_E_INVALID, "transpose24: SM100 buffers must be 16-byte aligned");
  cudaStream_t s = (cudaStream_t)stream;
  if (d_invalid) SPFY_CUDA_OK(cudaMemsetAsync(d_invalid, 0, sizeof(int), s));
  if (rows == 0 || cols == 0) return SPFY_OK;
  Transpose24Params P;
  P.vals = (const uint8_t*)vals;
  P.meta = (const uint8_t*)meta;
  P.vals_t = (uint8_t*)vals_t;
  P.meta_t = (uint8_t*)meta_t;
  P.rows = (uint32_t)rows;
  P.C = (uint32_t)C;
  P.taps = (uint32_t)taps;
  P.m_tiles = (uint32_t)ceil_div(rows, 128);
  P.m_tiles_t = (uint32_t)ceil_div(C, 128);
  P.tiles_t = P.m_tiles_t * (uint32_t)ceil_div(taps * rows, 128);
  P.invalid = d_invalid;
  int grid = 1;
  int rc = capped_grid(P.tiles_t, 8, &grid);
  if (rc) return rc;
  transpose24_kernel<false><<<grid, 256, 0, s>>>(P, Transpose24Phases<1>{});
  SPFY_LAUNCH_OK("transpose24_kernel");
  return SPFY_OK;
}

int spfy_transpose24_conv_bytes(int dtype, size_t m, size_t c, size_t kh, size_t kw, size_t stride, size_t pad,
                                size_t* vals_bytes, size_t* meta_bytes) {
  if (dtype != SPFY_F16 && dtype != SPFY_BF16)
    return fail(SPFY_E_UNSUPPORTED, "transpose24_conv_bytes: dtype %d (need F16/BF16)", dtype);
  Transpose24Phases<MAX_PHASES> T;
  size_t tiles = 0;
  int rc = conv_phase_table("transpose24_conv_bytes", m, c, kh, kw, stride, pad, &T, &tiles);
  if (rc) return rc;
  if (vals_bytes) *vals_bytes = tiles * 16384;
  if (meta_bytes) *meta_bytes = tiles * 2048;
  return SPFY_OK;
}

int spfy_transpose24_conv(int dtype, const void* vals, const void* meta, size_t m, size_t c, size_t kh, size_t kw,
                          size_t stride, size_t pad, void* vals_t, void* meta_t, int* d_invalid, spfy_stream_t stream) {
  if (dtype != SPFY_F16 && dtype != SPFY_BF16)
    return fail(SPFY_E_UNSUPPORTED, "transpose24_conv: dtype %d (need F16/BF16)", dtype);
  Transpose24Phases<MAX_PHASES> T;
  size_t tiles = 0;
  int rc = conv_phase_table("transpose24_conv", m, c, kh, kw, stride, pad, &T, &tiles);
  if (rc) return rc;
  if (!vals || !meta || !vals_t || !meta_t) return fail(SPFY_E_INVALID, "transpose24_conv: null pointer");
  if (misaligned16(vals) || misaligned16(meta) || misaligned16(vals_t) || misaligned16(meta_t))
    return fail(SPFY_E_INVALID, "transpose24_conv: SM100 buffers must be 16-byte aligned");
  cudaStream_t s = (cudaStream_t)stream;
  if (d_invalid) SPFY_CUDA_OK(cudaMemsetAsync(d_invalid, 0, sizeof(int), s));
  Transpose24Params P;
  P.vals = (const uint8_t*)vals;
  P.meta = (const uint8_t*)meta;
  P.vals_t = (uint8_t*)vals_t;
  P.meta_t = (uint8_t*)meta_t;
  P.rows = (uint32_t)m;
  P.C = (uint32_t)c;
  P.taps = (uint32_t)(kh * kw);
  P.m_tiles = (uint32_t)ceil_div(m, 128);
  P.m_tiles_t = (uint32_t)ceil_div(c, 128);
  P.tiles_t = (uint32_t)tiles;
  P.invalid = d_invalid;
  int grid = 1;
  rc = capped_grid(P.tiles_t, 8, &grid);
  if (rc) return rc;
  transpose24_kernel<true><<<grid, 256, 0, s>>>(P, T);
  SPFY_LAUNCH_OK("transpose24_kernel");
  return SPFY_OK;
}

int spfy_recompress24(int in_dtype, const void* in, size_t ld_in, int dtype, size_t rows, size_t cols,
                      const void* meta, void* comp_vals, void* out_masked, size_t ld_out, spfy_stream_t stream) {
  if (in_dtype != SPFY_F32 && in_dtype != SPFY_F16 && in_dtype != SPFY_BF16)
    return fail(SPFY_E_UNSUPPORTED, "recompress24: input dtype %d (need F32/F16/BF16)", in_dtype);
  if (dtype != SPFY_F16 && dtype != SPFY_BF16)
    return fail(SPFY_E_UNSUPPORTED, "recompress24: dtype %d (need F16/BF16)", dtype);
  if (!in || !meta) return fail(SPFY_E_INVALID, "recompress24: null input");
  if (ld_in < cols || (out_masked && ld_out < cols))
    return fail(SPFY_E_INVALID, "recompress24: leading dimension smaller than cols");
  if (rows >= (1ull << 31) || cols >= (1ull << 31) || ld_in >= (1ull << 31) || (out_masked && ld_out >= (1ull << 31)))
    return fail(SPFY_E_UNSUPPORTED, "recompress24: dimension too large");
  if (ceil_div(rows, 128) * ceil_div(cols, 128) >= (1ull << 22))
    return fail(SPFY_E_UNSUPPORTED, "recompress24: more than 2^22 SM100 tiles");
  if (misaligned16(meta) || (comp_vals && misaligned16(comp_vals)))
    return fail(SPFY_E_INVALID, "recompress24: SM100 buffers must be 16-byte aligned");
  const size_t eb = dtype_bytes(in_dtype);
  if ((uintptr_t)in % eb || (uintptr_t)out_masked % eb)
    return fail(SPFY_E_INVALID, "recompress24: in / out_masked are not aligned to their element size");
  if (rows == 0 || cols == 0 || (!comp_vals && !out_masked)) return SPFY_OK;
  Recompress24Params P;
  P.in = in;
  P.ld_in = ld_in;
  P.meta = (const uint8_t*)meta;
  P.comp_vals = (uint8_t*)comp_vals;
  P.out = out_masked;
  P.ld_out = ld_out;
  P.rows = (uint32_t)rows;
  P.cols = (uint32_t)cols;
  P.m_tiles = (uint32_t)ceil_div(rows, 128);
  P.k_tiles = (uint32_t)ceil_div(cols, 128);
  P.vec_in = !misaligned16(in) && (ld_in * eb) % 16 == 0;
  P.vec_out = out_masked && !misaligned16(out_masked) && (ld_out * eb) % 16 == 0;
  int grid = 1;
  int rc = capped_grid(ceil_div((size_t)P.m_tiles * P.k_tiles * 1024, 256), 16, &grid);
  if (rc) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  if (in_dtype == SPFY_F32) launch_recompress24<SPFY_F32>(dtype, grid, P, s);
  else if (in_dtype == SPFY_F16) launch_recompress24<SPFY_F16>(dtype, grid, P, s);
  else launch_recompress24<SPFY_BF16>(dtype, grid, P, s);
  SPFY_LAUNCH_OK("recompress24_kernel");
  return SPFY_OK;
}

}  // extern "C"
