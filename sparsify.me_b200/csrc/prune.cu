// prune.cu -- bandwidth-bound pruning / compression kernels (sm_100a)
//
//   spfy_prune_blocks_ref : exact positional semantics of the reference's
//                           sparsifyme::sparsify (include/sparsify.me/sparsify.hxx:24-82)
//   spfy_prune24          : 2:4 magnitude prune + compress + metadata in ONE pass
//                           (replaces cusparseLtSpMMAPrune/Compress,
//                            include/sparsify.me/spmma.hxx:85-104)
//   spfy_prune24_check    : cusparseLtSpMMAPruneCheck (spmma.hxx:88)
//
// All kernels are HBM-bound byte movers: 128-bit loads/stores, one pass over the
// input, no shared memory (there is no reuse), grid sized in multiples of the SM
// count.  See DESIGN.md for the algorithmic byte counts.
#include "common.cuh"

#include <cstdlib>

namespace spfy {
namespace {

// ------------------------------------------------------------------------
// A1  positional block pruning
// ------------------------------------------------------------------------
struct OffsetList {
  uint16_t off[256];  // offsets (relative to the block start) zeroed per block, in order
  int count;
  int in_block;       // 1 if every offset < blk_size (then a bitmap test is enough)
  uint32_t bitmap[8]; // bit o set  <=>  o in off[] (valid when in_block)
};

template <typename T>
__device__ __forceinline__ void store_zero(T* p) { *p = T(0); }

// which of the 4 elements starting at e0 does the reference zero? (bit i set -> element e0+i)
__device__ __forceinline__ unsigned blocks_ref_zero_bits(size_t e0, size_t total, size_t nblocks, uint32_t blk_size,
                                                        const OffsetList& L) {
  unsigned zero = 0;
  if (L.in_block) {
    // one division per chunk: block and in-block offset of e0, then step
    size_t blk = e0 / blk_size;
    uint32_t o = (uint32_t)(e0 - blk * blk_size);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      if (e0 + i >= total) break;
      if (blk < nblocks && (L.bitmap[o >> 5] >> (o & 31) & 1)) zero |= 1u << i;
      if (++o == blk_size) { o = 0; ++blk; }
    }
  } else {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const size_t e = e0 + i;
      if (e >= total) break;
      for (int j = 0; j < L.count; ++j) {
        const size_t o = L.off[j];
        if (e >= o && (e - o) % blk_size == 0 && (e - o) / blk_size < nblocks) {
          zero |= 1u << i;
          break;
        }
      }
    }
  }
  return zero;
}

// 4 elements of 2 / 4 / 8 bytes as 32-bit words
template <int BYTES> struct Quad { uint32_t w[BYTES]; };
template <int BYTES>
__device__ __forceinline__ Quad<BYTES> quad_load(const void* p) {
  Quad<BYTES> q;
  if (BYTES == 2) { const uint2 v = *reinterpret_cast<const uint2*>(p); q.w[0] = v.x; q.w[1] = v.y; }
  else if (BYTES == 4) { const uint4 v = *reinterpret_cast<const uint4*>(p); q.w[0] = v.x; q.w[1] = v.y; q.w[2] = v.z; q.w[3] = v.w; }
  else {
    const uint4 a = *reinterpret_cast<const uint4*>(p), b = *(reinterpret_cast<const uint4*>(p) + 1);
    q.w[0] = a.x; q.w[1] = a.y; q.w[2] = a.z; q.w[3] = a.w; q.w[4] = b.x; q.w[5] = b.y; q.w[6] = b.z; q.w[7] = b.w;
  }
  return q;
}
template <int BYTES>
__device__ __forceinline__ void quad_zero_store(void* p, Quad<BYTES> q, unsigned zero) {
  if (BYTES == 2) {
    if (zero & 1) q.w[0] &= 0xffff0000u;
    if (zero & 2) q.w[0] &= 0x0000ffffu;
    if (zero & 4) q.w[1] &= 0xffff0000u;
    if (zero & 8) q.w[1] &= 0x0000ffffu;
    *reinterpret_cast<uint2*>(p) = make_uint2(q.w[0], q.w[1]);
  } else if (BYTES == 4) {
#pragma unroll
    for (int i = 0; i < 4; ++i) if (zero >> i & 1) q.w[i] = 0;
    *reinterpret_cast<uint4*>(p) = make_uint4(q.w[0], q.w[1], q.w[2], q.w[3]);
  } else {
#pragma unroll
    for (int i = 0; i < 4; ++i) if (zero >> i & 1) q.w[2 * i] = q.w[2 * i + 1] = 0;
    *reinterpret_cast<uint4*>(p) = make_uint4(q.w[0], q.w[1], q.w[2], q.w[3]);
    *(reinterpret_cast<uint4*>(p) + 1) = make_uint4(q.w[4], q.w[5], q.w[6], q.w[7]);
  }
}

// one chunk = 4 consecutive elements: two 16-byte mask stores + the weights.  The weights are updated
// by a whole-vector read-modify-write (masked partial-sector stores ran at 2.3 TB/s); a thread keeps
// BR_UNROLL chunks in flight so that the reads overlap.
constexpr int BR_UNROLL = 4;
template <typename T>
__global__ void __launch_bounds__(256)
prune_blocks_ref_kernel(T* __restrict__ weights, uint64_t* __restrict__ mask, size_t total,
                        size_t nblocks, uint32_t blk_size, int vec_w, int vec_m,
                        const __grid_constant__ OffsetList L) {
  const size_t nthreads = (size_t)gridDim.x * blockDim.x;
  for (size_t t0 = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t0 * 4 < total; t0 += nthreads * BR_UNROLL) {
    unsigned zero[BR_UNROLL];
    bool full[BR_UNROLL];
    Quad<sizeof(T)> q[BR_UNROLL];
#pragma unroll
    for (int u = 0; u < BR_UNROLL; ++u) {
      const size_t e0 = (t0 + u * nthreads) * 4;
      full[u] = e0 + 4 <= total;
      zero[u] = e0 < total ? blocks_ref_zero_bits(e0, total, nblocks, blk_size, L) : 0u;
      if (vec_w && full[u] && zero[u]) q[u] = quad_load<sizeof(T)>(weights + e0);
    }
#pragma unroll
    for (int u = 0; u < BR_UNROLL; ++u) {
      const size_t e0 = (t0 + u * nthreads) * 4;
      if (e0 >= total) break;
      const unsigned z = zero[u];
      if (full[u]) {
        if (vec_m) {
          *reinterpret_cast<ulonglong2*>(mask + e0) = make_ulonglong2(z & 1 ? 0ull : 1ull, z & 2 ? 0ull : 1ull);
          *reinterpret_cast<ulonglong2*>(mask + e0 + 2) = make_ulonglong2(z & 4 ? 0ull : 1ull, z & 8 ? 0ull : 1ull);
        } else {  // mask only 8-byte aligned (e.g. a slice that starts at an odd word)
#pragma unroll
          for (int i = 0; i < 4; ++i) mask[e0 + i] = (z >> i & 1) ? 0ull : 1ull;
        }
        if (vec_w) {
          if (z) quad_zero_store<sizeof(T)>(weights + e0, q[u], z);
        } else {
#pragma unroll
          for (int i = 0; i < 4; ++i)
            if (z >> i & 1) store_zero(weights + e0 + i);
        }
      } else {
        for (int i = 0; i < 4 && e0 + i < total; ++i) {
          mask[e0 + i] = (z >> i & 1) ? 0ull : 1ull;
          if (z >> i & 1) store_zero(weights + e0 + i);
        }
      }
    }
  }
}

// ------------------------------------------------------------------------
// A2/A3  2:4 magnitude prune + compress (STRIP mode)
// ------------------------------------------------------------------------
struct Prune24Params {
  const uint16_t* in;
  size_t ld_in;
  uint16_t* out_dense;
  size_t ld_out;
  uint8_t* comp_vals;
  uint8_t* meta;
  uint64_t* mask;
  uint32_t rows, cols;
  uint32_t dom_rows;       // rows of the iteration domain (padded to 128 for SM100)
  uint32_t units_per_row;  // 16-column units per row in the iteration domain
  uint32_t G, mb;          // CANONICAL: groups per row, metadata bytes per row
  uint32_t k_tiles;        // SM100: 128-column tiles per row
  uint32_t m_tiles;        // SM100: 128-row tiles per column
  int layout;
  int vec_in, vec_out, vec_cv;  // 16-byte fast paths allowed
  int tile_order;               // iterate in SM100 tile storage order
  int fits32;                   // dom_rows * units_per_row < 2^32
  int fast;                     // every unit is a full, 16-byte aligned 16-column unit and no mask is wanted
};

// Indices i0 < i1 of the two largest magnitudes among the four 16-bit values packed in
// (lo, hi); tie -> lower index.  The 15 magnitude bits are widened to unique 17-bit keys
// (key << 2 | 3 - index: among equal magnitudes the lower index is the larger key), then a
// 4-input max/min network yields the largest and second largest key.
__device__ __forceinline__ void top2of4(uint32_t lo, uint32_t hi, uint32_t& i0, uint32_t& i1) {
  const uint32_t a = ((lo << 2) & 0x1fffcu) | 3u;
  const uint32_t b = ((lo >> 14) & 0x1fffcu) | 2u;
  const uint32_t c = ((hi << 2) & 0x1fffcu) | 1u;
  const uint32_t d = (hi >> 14) & 0x1fffcu;
  const uint32_t m01 = max(a, b), n01 = min(a, b), m23 = max(c, d), n23 = min(c, d);
  const uint32_t top = max(m01, m23);
  const uint32_t second = max(min(m01, m23), m01 > m23 ? n01 : n23);
  const uint32_t ia = 3u - (top & 3u), ib = 3u - (second & 3u);
  i0 = min(ia, ib);
  i1 = max(ia, ib);
}

// streaming 128-bit load.  Not `.nc`: out_dense may alias the input (in-place prune).
__device__ __forceinline__ uint4 ldg_nc_v4(const void* p) {
  uint4 r;
  asm volatile("ld.global.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w)
               : "l"(p));
  return r;
}

// one 16-column unit of one row: load, select, write every requested output
__device__ __forceinline__ void prune24_unit(const Prune24Params& P, size_t t) {
  {
    uint32_t row, unit;
    if (P.tile_order) {
      // SM100 outputs: walk the (128-row x 128-column) tiles in storage order, 8 units per row
      const uint32_t tile = (uint32_t)(t >> 10);
      const uint32_t mt = tile / P.k_tiles;
      row = mt * 128u + ((uint32_t)(t >> 3) & 127u);
      unit = (tile - mt * P.k_tiles) * 8u + ((uint32_t)t & 7u);
    } else if (P.fits32) {
      row = (uint32_t)t / P.units_per_row;
      unit = (uint32_t)t - row * P.units_per_row;
    } else {
      row = (uint32_t)(t / P.units_per_row);
      unit = (uint32_t)(t - (size_t)row * P.units_per_row);
    }
    const uint32_t c0 = unit * 16;

    // ---- load 16 storage words (zeros outside the matrix) ----
    uint32_t w[8] = {0, 0, 0, 0, 0, 0, 0, 0};  // two 16-bit values per word
    const bool row_ok = row < P.rows;
    if (row_ok && c0 < P.cols) {
      const uint16_t* src = P.in + (size_t)row * P.ld_in + c0;
      if (P.vec_in && c0 + 16 <= P.cols) {
        const uint4 a = ldg_nc_v4(src), b = ldg_nc_v4(src + 8);
        w[0] = a.x; w[1] = a.y; w[2] = a.z; w[3] = a.w;
        w[4] = b.x; w[5] = b.y; w[6] = b.z; w[7] = b.w;
      } else {
#pragma unroll
        for (int i = 0; i < 16; ++i)
          if (c0 + i < P.cols) w[i >> 1] |= (uint32_t)src[i] << ((i & 1) * 16);
      }
    }

    // ---- select per group of 4 ----
    uint32_t d[8];       // pruned dense words
    uint32_t cv[4];      // compressed: 2 values per group
    unsigned nibs = 0;   // 4 nibbles
    unsigned keep16 = 0; // keep bit per element
    const bool want_dense = P.out_dense != nullptr || P.mask != nullptr;
#pragma unroll
    for (int g = 0; g < 4; ++g) {
      const uint32_t lo = w[2 * g], hi = w[2 * g + 1];
      uint32_t i0, i1;
      top2of4(lo, hi, i0, i1);
      nibs |= (i0 | i1 << 2) << (4 * g);
      // halfword i of {lo, hi} is bytes (2i, 2i+1): one PRMT gathers the kept pair
      cv[g] = __byte_perm(lo, hi, (i0 + (i1 << 8)) * 0x22u + 0x1010u);
      if (want_dense) {
        const unsigned keep = (1u << i0) | (1u << i1);
        keep16 |= keep << (4 * g);
        d[2 * g] = lo & (((keep & 1u) * 0xffffu) | ((keep >> 1 & 1u) * 0xffff0000u));
        d[2 * g + 1] = hi & (((keep >> 2 & 1u) * 0xffffu) | ((keep >> 3 & 1u) * 0xffff0000u));
      }
    }

    // ---- pruned dense (may alias the input: same thread, same addresses) ----
    if (P.out_dense && row_ok && c0 < P.cols) {
      uint16_t* dst = P.out_dense + (size_t)row * P.ld_out + c0;
      if (P.vec_out && c0 + 16 <= P.cols) {
        *reinterpret_cast<uint4*>(dst) = make_uint4(d[0], d[1], d[2], d[3]);
        *reinterpret_cast<uint4*>(dst + 8) = make_uint4(d[4], d[5], d[6], d[7]);
      } else {
#pragma unroll
        for (int i = 0; i < 16; ++i)
          if (c0 + i < P.cols) dst[i] = (uint16_t)(d[i >> 1] >> ((i & 1) * 16));
      }
    }

    // ---- keep mask (u64 per element, API parity with sparsify.hxx) ----
    if (P.mask && row_ok && c0 < P.cols) {
      uint64_t* mdst = P.mask + (size_t)row * P.cols + c0;
      if (c0 + 16 <= P.cols && ((P.cols & 1) == 0) && ((uintptr_t)P.mask & 15) == 0) {
#pragma unroll
        for (int i = 0; i < 16; i += 2)
          *reinterpret_cast<ulonglong2*>(mdst + i) =
              make_ulonglong2(keep16 >> i & 1, keep16 >> (i + 1) & 1);
      } else {
#pragma unroll
        for (int i = 0; i < 16; ++i)
          if (c0 + i < P.cols) mdst[i] = keep16 >> i & 1;
      }
    }

    // ---- compressed values + metadata ----
    if (P.layout == SPFY_LAYOUT_SM100) {
      const uint32_t r = row & 127, q = (c0 & 127) >> 4;
      const size_t tile = (size_t)(c0 >> 7) * P.m_tiles + (row >> 7);  // k-tile major
      if (P.comp_vals)
        *reinterpret_cast<uint4*>(P.comp_vals + tile * 16384 + r * 128 + ((q ^ (r & 7)) << 4)) =
            make_uint4(cv[0], cv[1], cv[2], cv[3]);
      if (P.meta)
        *reinterpret_cast<uint16_t*>(P.meta + tile * 2048 + (r >> 4) * 256 + (q & 1) * 128 +
                                     (r & 7) * 16 + (q >> 1) * 4 + ((r >> 3) & 1) * 2) =
            (uint16_t)nibs;
    } else if (row_ok) {
      const uint32_t g0 = unit * 4;
      const uint32_t ng = min(4u, P.G - g0);  // groups that exist in this unit
      if (P.comp_vals) {
        uint32_t* dst = reinterpret_cast<uint32_t*>(P.comp_vals) + (size_t)row * P.G + g0;
        if (P.vec_cv && ng == 4) {
          *reinterpret_cast<uint4*>(dst) = make_uint4(cv[0], cv[1], cv[2], cv[3]);
        } else {
#pragma unroll
          for (int g = 0; g < 4; ++g)
            if (g < (int)ng) dst[g] = cv[g];
        }
      }
      if (P.meta) {
        uint8_t* dst = P.meta + (size_t)row * P.mb + g0 / 2;
        // an odd trailing group leaves its partner nibble 0 (CANONICAL contract)
        const unsigned lo = nibs & (ng >= 2 ? 0xffu : 0x0fu);
        dst[0] = (uint8_t)lo;
        if (ng > 2) dst[1] = (uint8_t)((nibs >> 8) & (ng == 4 ? 0xffu : 0x0fu));
      }
    }
  }
}

// ------------------------------------------------------------------------
// Fast path: every 16-column unit is complete and 16-byte aligned (all datasets/*.csv weight
// matrices except the k = 147 first convolution).  The generic unit above spends ~290 warp
// instructions per 16 elements, which makes the kernel integer-ALU-bound at about a third of the
// HBM rate; this one needs ~90.  Two groups of four are selected at once with packed 16-bit
// arithmetic:
//   * the magnitudes of element e of both groups share one word (group g in half g);
//   * x >= y per half is bit 15 / 31 of (x - y + 0x80008000)  (magnitudes are 15 bits wide, so the
//     halves never borrow from each other);
//   * with "earlier beats later on >=" (the documented tie-break: lower index wins) an element is
//     kept iff it loses at most one of its three duels, i.e. a 3-input majority of duel bits --
//     one LOP3 each;
//   * one PRMT in sign-replicate mode widens the keep bits to halfword masks, and bitwise selects
//     pick the first / second kept value and the index nibble.
// ------------------------------------------------------------------------
// prmt.b32 in its default mode: selector nibble bit 3 replicates the sign bit of the selected byte
// (the __byte_perm intrinsic only honours the low three bits)
__device__ __forceinline__ uint32_t prmt(uint32_t a, uint32_t b, uint32_t sel) {
  uint32_t r;
  asm("prmt.b32 %0, %1, %2, %3;" : "=r"(r) : "r"(a), "r"(b), "r"(sel));
  return r;
}
__device__ __forceinline__ uint32_t maj3(uint32_t x, uint32_t y, uint32_t z) { return (x & y) | (x & z) | (y & z); }
__device__ __forceinline__ uint32_t bsel(uint32_t m, uint32_t x, uint32_t y) { return (x & m) | (y & ~m); }

// groups (w0, w1) and (w2, w3) -> their compressed words, nibbles (group 0: bits 0-3, group 1:
// bits 16-19) and, when wanted, the four pruned dense words
template <bool DENSE>
__device__ __forceinline__ void select_two_groups(uint32_t w0, uint32_t w1, uint32_t w2, uint32_t w3,
                                                  uint32_t& cv0, uint32_t& cv1, uint32_t& nib, uint32_t* d) {
  const uint32_t A = __byte_perm(w0, w2, 0x5410), B = __byte_perm(w0, w2, 0x7632);
  const uint32_t C = __byte_perm(w1, w3, 0x5410), D = __byte_perm(w1, w3, 0x7632);
  const uint32_t a = A & 0x7fff7fffu, b = B & 0x7fff7fffu, c = C & 0x7fff7fffu, e = D & 0x7fff7fffu;
  const uint32_t ab = a - b + 0x80008000u, ac = a - c + 0x80008000u, ad = a - e + 0x80008000u;
  const uint32_t bc = b - c + 0x80008000u, bd = b - e + 0x80008000u, cd = c - e + 0x80008000u;
  const uint32_t ka = maj3(ab, ac, ad), kb = maj3(~ab, bc, bd), kc = maj3(~ac, ~bc, cd), kd = maj3(~ad, ~bd, ~cd);
  // bit 15 -> bytes 0,1 ; bit 31 -> bytes 2,3
  const uint32_t MA = prmt(ka, 0, 0xBB99), MB = prmt(kb, 0, 0xBB99);
  const uint32_t MC = prmt(kc, 0, 0xBB99), MD = prmt(kd, 0, 0xBB99);
  const uint32_t first = bsel(MA, A, bsel(MB, B, C));   // a, else b, else c
  const uint32_t second = bsel(MD, D, bsel(MC, C, B));  // d, else c, else b
  cv0 = __byte_perm(first, second, 0x5410);
  cv1 = __byte_perm(first, second, 0x7632);
  // i0 = a ? 0 : b ? 1 : 2  ->  bit0 = ~a & b, bit1 = ~a & ~b ;  i1 = d ? 3 : c ? 2 : 1  ->  bit2 = d | ~c, bit3 = d | c
  const uint32_t n01 = bsel(0x00010001u, ~MA & MB, ~MA & ~MB);
  const uint32_t n23 = bsel(0x00040004u, MD | ~MC, MD | MC);
  nib = (n01 & 0x00030003u) | (n23 & 0x000c000cu);
  if (DENSE) {
    d[0] = w0 & __byte_perm(MA, MB, 0x5410);
    d[1] = w1 & __byte_perm(MC, MD, 0x5410);
    d[2] = w2 & __byte_perm(MA, MB, 0x7632);
    d[3] = w3 & __byte_perm(MC, MD, 0x7632);
  }
}

// 16 elements (8 words) -> 4 compressed words + 16 metadata bits (+ 8 pruned words)
template <bool DENSE>
__device__ __forceinline__ void select_unit(const uint4& x, const uint4& y, uint4& cv, uint32_t& nibs, uint4& dx, uint4& dy) {
  uint32_t n0, n1, d0[4], d1[4];
  select_two_groups<DENSE>(x.x, x.y, x.z, x.w, cv.x, cv.y, n0, d0);
  select_two_groups<DENSE>(y.x, y.y, y.z, y.w, cv.z, cv.w, n1, d1);
  const uint32_t t = n0 | (n1 << 8);  // g0: 0-3, g2: 8-11, g1: 16-19, g3: 24-27
  nibs = (t | (t >> 12)) & 0xffffu;
  if (DENSE) {
    dx = make_uint4(d0[0], d0[1], d0[2], d0[3]);
    dy = make_uint4(d1[0], d1[1], d1[2], d1[3]);
  }
}

constexpr int FAST_UNITS = 4;  // units per thread and pass: all loads are issued before the first select

// SM100 layout: one pass = one (128-row x 128-column) tile = 1024 units.  8 consecutive threads read 256 contiguous bytes of one row and write 128
// contiguous bytes of one swizzled value row.
template <bool DENSE>
__device__ __forceinline__ void prune24_fast_tile_sm100(const Prune24Params& P, uint32_t pass) {
  // passes walk a 128-row block left to right (k-tile fastest): CTAs that run together read
  // neighbouring 256-byte pieces of the same rows (DRAM page locality); the storage index is k-tile major
  const uint32_t mt = pass / P.k_tiles, kt = pass - mt * P.k_tiles;
  const uint32_t tile = kt * P.m_tiles + mt;
  uint4 x[FAST_UNITS], y[FAST_UNITS];
  const uint32_t q = threadIdx.x & 7u, col = kt * 128u + q * 16u;
  const bool col_ok = col < P.cols;
#pragma unroll
  for (int i = 0; i < FAST_UNITS; ++i) {
    const uint32_t r = (threadIdx.x >> 3) + i * 32u, row = mt * 128u + r;
    x[i] = y[i] = make_uint4(0, 0, 0, 0);
    if (col_ok && row < P.rows) {
      const uint16_t* src = P.in + (size_t)row * P.ld_in + col;
      x[i] = ldg_nc_v4(src);
      y[i] = ldg_nc_v4(src + 8);
    }
  }
  uint8_t* vt = P.comp_vals ? P.comp_vals + (size_t)tile * 16384 : nullptr;
  uint8_t* et = P.meta ? P.meta + (size_t)tile * 2048 : nullptr;
#pragma unroll
  for (int i = 0; i < FAST_UNITS; ++i) {
    const uint32_t r = (threadIdx.x >> 3) + i * 32u, row = mt * 128u + r;
    uint4 cv, dx, dy;
    uint32_t nibs;
    select_unit<DENSE>(x[i], y[i], cv, nibs, dx, dy);
    if (DENSE && col_ok && row < P.rows) {
      uint16_t* dst = P.out_dense + (size_t)row * P.ld_out + col;
      *reinterpret_cast<uint4*>(dst) = dx;
      *reinterpret_cast<uint4*>(dst + 8) = dy;
    }
    if (vt) *reinterpret_cast<uint4*>(vt + r * 128u + ((q ^ (r & 7u)) << 4)) = cv;
    if (et)
      *reinterpret_cast<uint16_t*>(et + (r >> 4) * 256u + (q & 1u) * 128u + (r & 7u) * 16u + (q >> 1) * 4u +
                                   ((r >> 3) & 1u) * 2u) = (uint16_t)nibs;
  }
}

// CANONICAL layout: one pass = 1024 consecutive units of the row-major unit order
template <bool DENSE>
__device__ __forceinline__ void prune24_fast_chunk_canonical(const Prune24Params& P, uint32_t chunk) {
  const size_t total = (size_t)P.dom_rows * P.units_per_row;
  uint4 x[FAST_UNITS], y[FAST_UNITS];
  uint32_t rows_[FAST_UNITS], units_[FAST_UNITS];
#pragma unroll
  for (int i = 0; i < FAST_UNITS; ++i) {
    const size_t t = (size_t)chunk * 1024 + i * 256 + threadIdx.x;
    x[i] = y[i] = make_uint4(0, 0, 0, 0);
    rows_[i] = 0xffffffffu;
    units_[i] = 0;
    if (t < total) {
      const uint32_t row = P.fits32 ? (uint32_t)t / P.units_per_row : (uint32_t)(t / P.units_per_row);
      const uint32_t unit = (uint32_t)(t - (size_t)row * P.units_per_row);
      rows_[i] = row;
      units_[i] = unit;
      const uint16_t* src = P.in + (size_t)row * P.ld_in + unit * 16u;
      x[i] = ldg_nc_v4(src);
      y[i] = ldg_nc_v4(src + 8);
    }
  }
#pragma unroll
  for (int i = 0; i < FAST_UNITS; ++i) {
    if (rows_[i] == 0xffffffffu) continue;
    const uint32_t row = rows_[i], unit = units_[i];
    uint4 cv, dx, dy;
    uint32_t nibs;
    select_unit<DENSE>(x[i], y[i], cv, nibs, dx, dy);
    if (DENSE) {
      uint16_t* dst = P.out_dense + (size_t)row * P.ld_out + unit * 16u;
      *reinterpret_cast<uint4*>(dst) = dx;
      *reinterpret_cast<uint4*>(dst + 8) = dy;
    }
    if (P.comp_vals)
      *reinterpret_cast<uint4*>(reinterpret_cast<uint32_t*>(P.comp_vals) + (size_t)row * P.G + unit * 4u) = cv;
    if (P.meta) *reinterpret_cast<uint16_t*>(P.meta + (size_t)row * P.mb + unit * 2u) = (uint16_t)nibs;
  }
}

// number of 1024-unit passes of a matrix
__host__ __device__ inline uint32_t fast_passes(const Prune24Params& P) {
  return P.tile_order ? P.k_tiles * P.m_tiles
                      : (uint32_t)(((size_t)P.dom_rows * P.units_per_row + 1023) / 1024);
}

__device__ __forceinline__ void prune24_fast_pass(const Prune24Params& P, uint32_t pass) {
  if (P.tile_order) {
    if (P.out_dense) prune24_fast_tile_sm100<true>(P, pass); else prune24_fast_tile_sm100<false>(P, pass);
  } else {
    if (P.out_dense) prune24_fast_chunk_canonical<true>(P, pass); else prune24_fast_chunk_canonical<false>(P, pass);
  }
}

__global__ void __launch_bounds__(256)
prune24_fast_kernel(const __grid_constant__ Prune24Params P) {
  const uint32_t passes = fast_passes(P);
  for (uint32_t pass = blockIdx.x; pass < passes; pass += gridDim.x) prune24_fast_pass(P, pass);
}

__global__ void __launch_bounds__(256)
prune24_strip_kernel(const __grid_constant__ Prune24Params P) {
  const size_t total = (size_t)P.dom_rows * P.units_per_row;
  const size_t nthreads = (size_t)gridDim.x * blockDim.x;
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += nthreads)
    prune24_unit(P, t);
}

// Many matrices in one launch (a whole model's weight set: the per-layer matrices are
// <= 4.7 MB, so one launch per layer is launch-latency-bound).  Work is cut into CTA tiles
// of 1024 units (one SM100 tile); every tile belongs to exactly one matrix, so the lookup is CTA-uniform.
constexpr int PRUNE_BATCH_MAX = 96;
struct Prune24Batch {
  Prune24Params item[PRUNE_BATCH_MAX];
  uint32_t tile_prefix[PRUNE_BATCH_MAX + 1];  // tile_prefix[i] = first CTA tile of item i
  int count;
};

__global__ void __launch_bounds__(256)
prune24_batched_kernel(const __grid_constant__ Prune24Batch Bt) {
  const uint32_t tiles = Bt.tile_prefix[Bt.count];
  for (uint32_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    int lo = 0, hi = Bt.count - 1;  // last item with tile_prefix <= tile
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (Bt.tile_prefix[mid] <= tile) lo = mid; else hi = mid - 1;
    }
    const Prune24Params& P = Bt.item[lo];
    const uint32_t pass = tile - Bt.tile_prefix[lo];
    if (P.fast) {
      prune24_fast_pass(P, pass);
    } else {
      const size_t total = (size_t)P.dom_rows * P.units_per_row;
#pragma unroll 1
      for (int i = 0; i < 4; ++i) {
        const size_t t = (size_t)pass * 1024 + i * 256 + threadIdx.x;
        if (t < total) prune24_unit(P, t);
      }
    }
  }
}

// ------------------------------------------------------------------------
// TILE mode (what the reference requests at spmma.hxx:86, CUSPARSELT_PRUNE_SPMMA_TILE): per 4x4 tile
// keep 8 entries, two in every row AND every column, with the largest sum |x|.  The selection below is
// the one cusparseLt 0.7.1 makes -- bit-exact on every tie and every fp32 rounding case of
// tests/golden/tile_*.npz (see oracle/spfy_oracle.cpp:orc_prune24_tile for how it was established):
// the 90 patterns are not scanned one by one but as 19 candidates,
//   pair sums      rp[r][i] = |x[r][c0]| + |x[r][c1]|,  i over the column pairs {01,02,12,03,13,23}
//   complementary  rows (x, ~x, y, ~y): x and y maximised INDEPENDENTLY (first maximum wins)
//   same           rows (x, x, ~x, ~x): first maximum over x
//   mixed          for pairs i < j sharing one column, rows 0/1 hold {j, i} and rows 2/3 hold {~i, ~j}, each
//                  half in the better of its two orders (the listed order wins a tie)
// all sums in fp32 as (row0 + row1) + (row2 + row3); candidates compared in that order, first maximum wins.
// One thread per tile; `VEC`: four aligned 64-bit loads / stores per tile.
// ------------------------------------------------------------------------
// pattern of every candidate, in the order they are compared: 36 complementary (x * 6 + y), 6 same (36 + x),
// 48 mixed (42 + 4 * group + 2 * [rows 0/1 swapped] + [rows 2/3 swapped], groups (i, j) in lexicographic order)
__constant__ uint16_t c_tile_pattern[90] = {
    0xc3c3, 0xa5c3, 0x96c3, 0x69c3, 0x5ac3, 0x3cc3, 0xc3a5, 0xa5a5, 0x96a5, 0x69a5, 0x5aa5, 0x3ca5, 0xc396, 0xa596, 0x9696, 0x6996, 0x5a96, 0x3c96, 0xc369, 0xa569, 0x9669, 0x6969, 0x5a69, 0x3c69, 0xc35a, 0xa55a, 0x965a, 0x695a, 0x5a5a, 0x3c5a, 0xc33c, 0xa53c, 0x963c, 0x693c, 0x5a3c, 0x3c3c, 0xcc33, 0xaa55, 0x9966, 0x6699, 0x55aa, 0x33cc, 0xac35, 0xca35, 0xac53, 0xca53, 0x9c36, 0xc936, 0x9c63, 0xc963, 0x6c39, 0xc639, 0x6c93, 0xc693, 0x5c3a, 0xc53a, 0x5ca3, 0xc5a3, 0x9a56, 0xa956, 0x9a65, 0xa965, 0x6a59, 0xa659, 0x6a95, 0xa695, 0x3a5c, 0xa35c, 0x3ac5, 0xa3c5, 0x596a, 0x956a, 0x59a6, 0x95a6, 0x396c, 0x936c, 0x39c6, 0x93c6, 0x569a, 0x659a, 0x56a9, 0x65a9, 0x369c, 0x639c, 0x36c9, 0x63c9, 0x35ac, 0x53ac, 0x35ca, 0x53ca};

// two fp32 additions in one instruction (FADD2): every sum of the selection exists once for the upper row pair of a
// tile and once for the lower one, so the two travel as the halves of one 64-bit register pair
__device__ __forceinline__ float2 add2(float2 a, float2 b) {
  float2 r;
  asm("{ .reg .b64 ra, rb, rc;\n"
      "  mov.b64 ra, {%2, %3};\n"
      "  mov.b64 rb, {%4, %5};\n"
      "  add.rn.f32x2 rc, ra, rb;\n"
      "  mov.b64 {%0, %1}, rc; }"
      : "=f"(r.x), "=f"(r.y)
      : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));
  return r;
}

// returns the candidate code (index into c_tile_pattern); the selection is tracked as small integers and
// turned into a keep mask once -- the first version carried 16-bit patterns through every compare and was
// integer-ALU bound (600 instructions per tile).  Third version: the 115 fp32 additions are 48 packed ones and 19
// scalar ones -- .x of every pair belongs to rows 0/1, .y to rows 2/3:
//   rpA[i] = (rp[0][i], rp[2][i]),  rpB[i] = (rp[1][i], rp[3][i]),  X(a, b) = rpA[a] + rpB[b] = (rp0[a] + rp1[b], rp2[a] + rp3[b])
__device__ __forceinline__ uint32_t tile_select(const float (&m)[16]) {
  // column-pair index -> (c0, c1); the complement of pair i is pair 5 - i
  constexpr int C0[6] = {0, 0, 1, 0, 1, 2}, C1[6] = {1, 2, 2, 3, 3, 3};
  float2 rpA[6], rpB[6];
#pragma unroll
  for (int i = 0; i < 6; ++i) {
    rpA[i] = add2(make_float2(m[C0[i]], m[8 + C0[i]]), make_float2(m[C1[i]], m[8 + C1[i]]));
    rpB[i] = add2(make_float2(m[4 + C0[i]], m[12 + C0[i]]), make_float2(m[4 + C1[i]], m[12 + C1[i]]));
  }
  // complementary class: x and y maximised independently, first maximum wins
  float2 b = add2(rpA[0], rpB[5]);
  uint32_t x01 = 0, y23 = 0;
#pragma unroll
  for (int x = 1; x < 6; ++x) {
    const float2 g = add2(rpA[x], rpB[5 - x]);
    const bool pg = g.x > b.x, ph = g.y > b.y;
    b.x = pg ? g.x : b.x;
    x01 = pg ? (uint32_t)(6 * x) : x01;
    b.y = ph ? g.y : b.y;
    y23 = ph ? (uint32_t)x : y23;
  }
  float best = __fadd_rn(b.x, b.y);
  uint32_t code = x01 + y23;
  // same class: (rp0[x] + rp1[x]) + (rp2[5-x] + rp3[5-x])
  {
    float2 d[6];
#pragma unroll
    for (int x = 0; x < 6; ++x) d[x] = add2(rpA[x], rpB[x]);
#pragma unroll
    for (int x = 0; x < 6; ++x) {
      const float s = __fadd_rn(d[x].x, d[5 - x].y);
      const bool p = s > best;
      best = p ? s : best;
      code = p ? (uint32_t)(36 + x) : code;
    }
  }
  // mixed class: group (i, j) takes X(j, i).x / X(i, j).x for rows 0/1 and X(5-i, 5-j).y / X(5-j, 5-i).y for rows 2/3
  float2 X[6][6];
#pragma unroll
  for (int a = 0; a < 6; ++a)
#pragma unroll
    for (int c = 0; c < 6; ++c)
      if (a != c && c != 5 - a) X[a][c] = add2(rpA[a], rpB[c]);
  int g = 0;
  float d01 = 0.f, d23 = 0.f;  // stay 0 unless a mixed candidate wins
#pragma unroll
  for (int i = 0; i < 6; ++i)
#pragma unroll
    for (int j = i + 1; j < 6; ++j) {
      if (j == 5 - i) continue;
      const float s1 = X[j][i].x, s2 = X[i][j].x;
      const float t1 = X[5 - i][5 - j].y, t2 = X[5 - j][5 - i].y;
      // The order bits are only needed for the group that wins: the compares are replaced by maxima, and the winner
      // carries s2 - s1 and t2 - t1 along (exact in sign: a difference of distinct floats never rounds to zero).  The
      // kernel is bound by the ALU pipe (compares and selects issue every other cycle); the subtractions go down the
      // FMA pipe, which has room.
      const float s = __fadd_rn(fmaxf(s1, s2), fmaxf(t1, t2));
      const float e01 = __fsub_rn(s2, s1), e23 = __fsub_rn(t2, t1);
      const bool p = s > best;
      best = p ? s : best;
      code = p ? (uint32_t)(42 + 4 * g) : code;
      d01 = p ? e01 : d01;
      d23 = p ? e23 : d23;
      ++g;
    }
  return code + (d01 > 0.f ? 2u : 0u) + (d23 > 0.f ? 1u : 0u);
}

template <bool BF16>
__device__ __forceinline__ float tile_mag(uint32_t bits) {
  const uint32_t ab = bits & 0x7fffu;
  return BF16 ? __uint_as_float(ab << 16) : __half2float(__ushort_as_half((unsigned short)ab));
}

// |x| of both halves of a word as fp32 (one mask for the two signs, no half-word extraction)
template <bool BF16>
__device__ __forceinline__ void tile_mag2(uint32_t w, float& lo, float& hi) {
  if (BF16) {
    lo = __uint_as_float((w << 16) & 0x7fff0000u);
    hi = __uint_as_float(w & 0x7fff0000u);
  } else {
    // (|x| rides on the conversion: HADD2.F32 takes an absolute-value modifier, no mask instruction)
    const float2 f = __half22float2(__habs2(*reinterpret_cast<const __half2*>(&w)));
    lo = f.x;
    hi = f.y;
  }
}

// the candidate -> pattern table in shared memory: the index differs from lane to lane, and a constant-bank read with
// divergent addresses is replayed once per distinct address
struct TilePatterns {
  uint16_t pat[96];
  __device__ __forceinline__ void load() {
    if (threadIdx.x < 90) pat[threadIdx.x] = c_tile_pattern[threadIdx.x];
    __syncthreads();
  }
};

// Keep masks of the four tile rows from the 16-bit pattern.  Row i's nibble k is spread so that its bits sit in the
// sign positions of the four bytes of z[i] (k << 7 | k << 14 | k << 21 | k << 28: bits 7 / 15 / 23 / 31 = b0..b3, one
// multiplication); PRMT's sign-replicate mode then turns (z, z) into a halfword mask, one instruction per word.
struct TileKeep {
  uint32_t z[4];
  __device__ __forceinline__ explicit TileKeep(uint32_t pat) {
    const uint32_t hi = pat >> 8;
    z[0] = (pat & 0xfu) * 0x10204080u;
    z[1] = (pat & 0xf0u) * 0x01020408u;
    z[2] = (hi & 0xfu) * 0x10204080u;
    z[3] = (hi & 0xf0u) * 0x01020408u;
  }
  // (inline PTX: the __byte_perm intrinsic only honours three bits of every selector nibble)
  static __device__ __forceinline__ uint32_t sign_bytes(uint32_t z, uint32_t sel) {
    uint32_t r;
    asm("prmt.b32 %0, %1, %1, %2;" : "=r"(r) : "r"(z), "r"(sel));
    return r;
  }
  __device__ __forceinline__ uint2 row(int i, uint2 w) const {
    return make_uint2(w.x & sign_bytes(z[i], 0x9988u), w.y & sign_bytes(z[i], 0xbbaau));
  }
};

// Block = 32 tile columns (one 256-byte piece of four rows per warp) x 8 tile rows; blockIdx.x walks the tile columns,
// the tile rows are walked with stride 8 * gridDim.y -- no division anywhere (the flat index of the first version paid
// ~60 instructions of a kernel that is issue-bound at ~400 per tile for it).
template <bool BF16, bool VEC>
__global__ void __launch_bounds__(256, VEC ? 3 : 2)  // three blocks per SM: at most 80 registers (four blocks at 64 registers spill 60 bytes: 223 -> 235 us)
prune24_tile_kernel(const uint16_t* in, size_t ld_in, uint16_t* out,  // no __restrict__: out may alias in (in-place prune)
                    size_t ld_out, uint32_t rows, uint32_t cols) {
  __shared__ TilePatterns T;
  T.load();
  const uint32_t tiles_c = (cols + 3) / 4, tiles_r = (rows + 3) / 4;
  const uint32_t tc = blockIdx.x * 32u + (threadIdx.x & 31u);
  if (tc >= tiles_c) return;
  const uint32_t c0 = tc * 4;
  const uint32_t tr_step = gridDim.y * 8u;
  // the next tile of the thread is fetched before the current one is worked on: 32 bytes per thread in flight are a
  // third of what the DRAM latency asks for at three resident blocks per SM (measured: 3.7 TB/s without)
  // (row addresses as column pointer + row * 32-bit byte pitch: one IMAD.WIDE on the FMA pipe instead of a 64-bit add
  // on the ALU pipe, the one this kernel is bound by; the host checks that the pitches fit)
  const uint32_t pitch_in = (uint32_t)ld_in * 2u, pitch_out = (uint32_t)ld_out * 2u;
  const char* in_col = reinterpret_cast<const char*>(in + c0);
  char* out_col = reinterpret_cast<char*>(out + c0);
  auto fetch = [&](uint32_t tr, uint2 (&w)[4]) {
    const uint32_t r0 = tr * 4;
#pragma unroll
    for (int i = 0; i < 4; ++i)
      w[i] = r0 + i < rows ? *reinterpret_cast<const uint2*>(in_col + (uint64_t)(r0 + i) * pitch_in)
                           : make_uint2(0u, 0u);  // (covers tr >= tiles_r)
  };
  uint2 nw[4];
  const uint32_t tr_first = blockIdx.y * 8u + (threadIdx.x >> 5);
  if (VEC) fetch(tr_first, nw);
  for (uint32_t tr = tr_first; tr < tiles_r; tr += tr_step) {
    const uint32_t r0 = tr * 4;
    float mag[16];
    if (VEC) {
      uint2 w[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) w[i] = nw[i];
      fetch(tr + tr_step, nw);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        tile_mag2<BF16>(w[i].x, mag[i * 4 + 0], mag[i * 4 + 1]);
        tile_mag2<BF16>(w[i].y, mag[i * 4 + 2], mag[i * 4 + 3]);
      }
      const TileKeep keep(T.pat[tile_select(mag)]);
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        if (r0 + i >= rows) break;
        *reinterpret_cast<uint2*>(out_col + (uint64_t)(r0 + i) * pitch_out) = keep.row(i, w[i]);
      }
    } else {
      uint16_t v[16];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const bool ok = r0 + i < rows && c0 + j < cols;
          v[i * 4 + j] = ok ? in[(size_t)(r0 + i) * ld_in + c0 + j] : (uint16_t)0;
          mag[i * 4 + j] = tile_mag<BF16>(v[i * 4 + j]);
        }
      const uint32_t pat = T.pat[tile_select(mag)];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j)
          if (r0 + i < rows && c0 + j < cols)
            out[(size_t)(r0 + i) * ld_out + c0 + j] = (pat >> (i * 4 + j) & 1) ? v[i * 4 + j] : (uint16_t)0;
    }
  }
}

// TILE prune + compress in ONE pass (what sparsifyme::spmma runs): the thread that chose a tile's pattern also
// emits, per row, the two kept values and the index nibble exactly as prune24_unit would for the pruned row
// (same top2of4 on the pruned words, so zero-valued survivors resolve to the same indices), in either layout.
// Needs cols % 16 == 0 and 8-byte aligned rows: the four lanes of a 16-column unit are then neighbours
// (quad shuffles assemble the unit's metadata word) and a warp's 32 tiles are one 128-byte line of a value
// tile.  The iteration domain is the padded one of the layout (SM100: 128-row x 128-column tiles; padding is
// read as +0 and comes out as zeros with the neutral nibble 0x4).
// number of 4x4 tiles of the (padded) iteration domain, and tiles per tile row
__device__ __host__ __forceinline__ size_t tile_fused_total(const Prune24Params& P, uint32_t* tiles_c) {
  const uint32_t dom_cols = P.tile_order ? P.k_tiles * 128u : P.cols;
  *tiles_c = dom_cols / 4u;  // % 4 == 0: a quad of lanes never straddles a tile row
  return (size_t)((P.dom_rows + 3u) / 4u) * *tiles_c;
}

// one warp, 32 consecutive tiles of one tile row: lane's tile is (tr, tc) (inactive lanes only take part in the shuffles)
// the four rows of tile (tr, tc); padding of the iteration domain reads as +0
__device__ __forceinline__ void tile_fused_fetch(const Prune24Params& P, uint32_t tr, uint32_t tc, bool active, uint2 (&w)[4]) {
  const uint32_t r0 = tr * 4u, c0 = tc * 4u;
  const bool col_ok = active && c0 < P.cols;
#pragma unroll
  for (int i = 0; i < 4; ++i)
    w[i] = (col_ok && r0 + i < P.rows)
               ? *reinterpret_cast<const uint2*>(reinterpret_cast<const char*>(P.in + c0) + (uint64_t)(r0 + i) * ((uint32_t)P.ld_in * 2u))
               : make_uint2(0u, 0u);
}

// PATTERN (TILE_TRANSPOSABLE): the nibbles are the tile's pattern itself, so they stay two of four along columns even
// where a kept value is +-0 (top2of4 on the pruned words may then name another zero); padding gets the neutral nibble.
template <bool BF16, bool PATTERN>
__device__ __forceinline__ void tile_fused_tiles(const Prune24Params& P, const TilePatterns& T, uint32_t tr, uint32_t tc,
                                                 bool active, uint32_t lane, const uint2 (&w)[4]) {
  {
    const uint32_t r0 = tr * 4u, c0 = tc * 4u;
    const bool col_ok = active && c0 < P.cols;
    float mag[16];
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      tile_mag2<BF16>(w[i].x, mag[i * 4 + 0], mag[i * 4 + 1]);
      tile_mag2<BF16>(w[i].y, mag[i * 4 + 2], mag[i * 4 + 3]);
    }
    const uint32_t pat = T.pat[tile_select(mag)];
    const TileKeep keep(pat);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      const uint32_t row = r0 + i;
      const uint2 kept = keep.row(i, w[i]);
      const uint32_t lo = kept.x, hi = kept.y;
      if (P.out_dense && col_ok && row < P.rows)
        *reinterpret_cast<uint2*>(reinterpret_cast<char*>(P.out_dense + c0) + (uint64_t)row * ((uint32_t)P.ld_out * 2u)) =
            make_uint2(lo, hi);
      uint32_t i0, i1;
      if (PATTERN) {
        const uint32_t nib = (pat >> (4 * i)) & 0xfu;
        const bool pad = !col_ok || row >= P.rows;
        i0 = pad ? 0u : __ffs(nib) - 1u;
        i1 = pad ? 1u : 31u - __clz(nib);
      } else {
        top2of4(lo, hi, i0, i1);
      }
      const uint32_t cv = __byte_perm(lo, hi, (i0 + (i1 << 8)) * 0x22u + 0x1010u);
      // the unit's four nibbles meet in the lane of its first group
      uint32_t nibs = (i0 | i1 << 2) << (4u * (lane & 3u));
      nibs |= __shfl_xor_sync(0xffffffffu, nibs, 1);
      nibs |= __shfl_xor_sync(0xffffffffu, nibs, 2);
      if (!active || row >= P.dom_rows) continue;
      if (P.layout == SPFY_LAYOUT_SM100) {
        const uint32_t r = row & 127u, q = (c0 & 127u) >> 4;
        const size_t tile = (size_t)(c0 >> 7) * P.m_tiles + (row >> 7);
        if (P.comp_vals)
          *reinterpret_cast<uint32_t*>(P.comp_vals + tile * 16384 + r * 128 + ((q ^ (r & 7u)) << 4) + (lane & 3u) * 4u) = cv;
        if (P.meta && (lane & 3u) == 0u)
          *reinterpret_cast<uint16_t*>(P.meta + tile * 2048 + (r >> 4) * 256 + (q & 1u) * 128 + (r & 7u) * 16 +
                                       (q >> 1) * 4 + ((r >> 3) & 1u) * 2) = (uint16_t)nibs;
      } else {
        if (P.comp_vals) reinterpret_cast<uint32_t*>(P.comp_vals)[(size_t)row * P.G + tc] = cv;
        if (P.meta && (lane & 3u) == 0u)
          *reinterpret_cast<uint16_t*>(P.meta + (size_t)row * P.mb + tc / 2u) = (uint16_t)nibs;
      }
    }
  }
}

// 32 consecutive tiles starting at flat index `base` (a multiple of 32; tiles_c is one too, or the row is the last)
template <bool BF16>
__device__ __forceinline__ void tile_fused_warp(const Prune24Params& P, const TilePatterns& T, size_t base, size_t total,
                                                uint32_t tiles_c, uint32_t lane) {
  const size_t t = base + lane;
  const bool active = t < total;
  const uint32_t tr = !active ? 0u : (total >> 32) == 0 ? (uint32_t)t / tiles_c : (uint32_t)(t / tiles_c);
  const uint32_t tc = active ? (uint32_t)(t - (size_t)tr * tiles_c) : 0u;
  uint2 w[4];
  tile_fused_fetch(P, tr, tc, active, w);
  tile_fused_tiles<BF16, false>(P, T, tr, tc, active, lane, w);
}

// grid: x = 32-tile column chunks, y walks the tile rows with stride 8 * gridDim.y (no division, like prune24_tile_kernel)
template <bool BF16, bool PATTERN>
__global__ void __launch_bounds__(256, 3)
prune24_tile_fused_kernel(const __grid_constant__ Prune24Params P) {
  __shared__ TilePatterns T;
  T.load();
  uint32_t tiles_c;
  const size_t total = tile_fused_total(P, &tiles_c);
  const uint32_t tiles_r = (uint32_t)(total / tiles_c);
  const uint32_t lane = threadIdx.x & 31u;
  const uint32_t tc = blockIdx.x * 32u + lane;
  const bool col_in = tc < tiles_c;
  const uint32_t tcc = col_in ? tc : 0u, tr_step = gridDim.y * 8u;
  uint32_t tr = blockIdx.y * 8u + (threadIdx.x >> 5);
  uint2 nw[4];
  tile_fused_fetch(P, tr, tcc, col_in && tr < tiles_r, nw);
  for (; tr < tiles_r; tr += tr_step) {
    uint2 w[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) w[i] = nw[i];
    tile_fused_fetch(P, tr + tr_step, tcc, col_in && tr + tr_step < tiles_r, nw);  // next tile in flight under this one
    tile_fused_tiles<BF16, PATTERN>(P, T, tr, tcc, col_in, lane, w);
  }
}

// TILE prune + compress of many matrices in one launch (what sparsifyme::spmma asks for, spmma.hxx:86, over a whole
// model's weight set): CTA tiles of 1024 4x4 tiles, each belonging to exactly one matrix (binary search as above)
template <bool BF16>
__global__ void __launch_bounds__(256)
prune24_tile_batched_kernel(const __grid_constant__ Prune24Batch Bt) {
  __shared__ TilePatterns T;
  T.load();
  const uint32_t tiles = Bt.tile_prefix[Bt.count];
  const uint32_t lane = threadIdx.x & 31u;
  for (uint32_t tile = blockIdx.x; tile < tiles; tile += gridDim.x) {
    int lo = 0, hi = Bt.count - 1;  // last item with tile_prefix <= tile
    while (lo < hi) {
      const int mid = (lo + hi + 1) >> 1;
      if (Bt.tile_prefix[mid] <= tile) lo = mid; else hi = mid - 1;
    }
    const Prune24Params& P = Bt.item[lo];
    uint32_t tiles_c;
    const size_t total = tile_fused_total(P, &tiles_c);
    const size_t first = (size_t)(tile - Bt.tile_prefix[lo]) * 1024u;
#pragma unroll 1
    for (int i = 0; i < 4; ++i) {
      const size_t base = first + i * 256 + (threadIdx.x & ~31u);
      if (base < total) tile_fused_warp<BF16>(P, T, base, total, tiles_c, lane);
    }
  }
}

// number of non-zero halfwords (sign ignored) in a word: 0, 1 or 2
__device__ __forceinline__ uint32_t nz_halves(uint32_t w) {
  const uint32_t m = w & 0x7fff7fffu;
  return ((m & 0xffffu) != 0u) + ((m >> 16) != 0u);
}

// cusparseLtSpMMAPruneCheck: flag any group of 4 with more than 2 non-zeros.  `vec`: rows are 16-byte
// aligned and cols % 16 == 0 -> a thread checks 16 elements from two 128-bit loads; otherwise one group per
// thread with scalar loads (ragged edges count as zeros).
__global__ void __launch_bounds__(256)
prune24_check_kernel(const uint16_t* __restrict__ in, size_t ld_in, uint32_t rows, uint32_t cols, int vec,
                     int* __restrict__ invalid) {
  const size_t nthreads = (size_t)gridDim.x * blockDim.x;
  bool bad = false;
  if (vec) {
    const uint32_t upr = cols / 16;
    const size_t total = (size_t)rows * upr;
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += nthreads) {
      const uint32_t row = (uint32_t)(t / upr), unit = (uint32_t)(t - (size_t)row * upr);
      const uint16_t* src = in + (size_t)row * ld_in + unit * 16u;
      const uint4 a = ldg_nc_v4(src), b = ldg_nc_v4(src + 8);
      bad |= nz_halves(a.x) + nz_halves(a.y) > 2u;
      bad |= nz_halves(a.z) + nz_halves(a.w) > 2u;
      bad |= nz_halves(b.x) + nz_halves(b.y) > 2u;
      bad |= nz_halves(b.z) + nz_halves(b.w) > 2u;
    }
  } else {
    const uint32_t G = (cols + 3) / 4;
    const size_t total = (size_t)rows * G;
    for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += nthreads) {
      const uint32_t row = (uint32_t)(t / G), g = (uint32_t)(t - (size_t)row * G);
      int nz = 0;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const uint32_t c = g * 4 + i;
        if (c < cols && (in[(size_t)row * ld_in + c] & 0x7fffu)) ++nz;
      }
      bad |= nz > 2;
    }
  }
  if (__any_sync(0xffffffffu, bad) && (threadIdx.x & 31) == 0) atomicExch(invalid, 1);
}

// validate one matrix and fill the kernel's parameter block
int fill_prune24(Prune24Params* out, int layout, const uint16_t* src, size_t ld_src, void* out_dense,
                 size_t ld_out, void* comp_vals, void* meta, uint64_t* mask, size_t rows, size_t cols) {
  Prune24Params P;
  memset(&P, 0, sizeof(P));
  P.in = src;
  P.ld_in = ld_src;
  P.out_dense = (uint16_t*)out_dense;
  P.ld_out = ld_out;
  P.comp_vals = (uint8_t*)comp_vals;
  P.meta = (uint8_t*)meta;
  P.mask = mask;
  P.rows = (uint32_t)rows;
  P.cols = (uint32_t)cols;
  P.layout = layout;
  P.G = (uint32_t)ceil_div(cols, 4);
  P.mb = (uint32_t)ceil_div(P.G, 2);
  P.k_tiles = (uint32_t)ceil_div(cols, 128);
  P.m_tiles = (uint32_t)ceil_div(rows, 128);
  const bool sm100_out = layout == SPFY_LAYOUT_SM100 && (comp_vals || meta);
  P.dom_rows = sm100_out ? (uint32_t)round_up(rows, 128) : (uint32_t)rows;
  P.units_per_row = sm100_out ? P.k_tiles * 8 : (uint32_t)ceil_div(cols, 16);
  P.tile_order = sm100_out ? 1 : 0;
  P.fits32 = (size_t)P.dom_rows * P.units_per_row < (1ull << 32);
  if (sm100_out && ceil_div(rows, 128) * ceil_div(cols, 128) >= (1ull << 22))
    return fail(SPFY_E_UNSUPPORTED, "prune24: more than 2^22 SM100 tiles");
  P.vec_in = ((uintptr_t)src % 16 == 0) && (ld_src % 8 == 0);
  P.vec_out = out_dense && ((uintptr_t)out_dense % 16 == 0) && (ld_out % 8 == 0);
  P.vec_cv = comp_vals && ((uintptr_t)comp_vals % 16 == 0) && (P.G % 4 == 0);
  if (layout == SPFY_LAYOUT_SM100 && ((comp_vals && (uintptr_t)comp_vals % 16) || (meta && (uintptr_t)meta % 16)))
    return fail(SPFY_E_INVALID, "prune24: SM100 outputs must be 16-byte aligned");
  P.fast = !mask && P.vec_in && cols % 16 == 0 && (!out_dense || P.vec_out) &&
           (sm100_out || ((!comp_vals || P.vec_cv) && (uintptr_t)meta % 2 == 0)) &&
           fast_passes(P) < (1u << 31);
  *out = P;
  return SPFY_OK;
}

// the one-pass TILE prune + compress (see prune24_tile_fused_kernel)
template <bool PATTERN>
static int launch_tile_fused(int dtype, int layout, const uint16_t* src, size_t ld_in, void* out_dense, size_t ld_out,
                             void* comp_vals, void* meta, size_t rows, size_t cols, cudaStream_t s) {
  Prune24Params P;
  int rc = fill_prune24(&P, layout, src, ld_in, out_dense, ld_out, comp_vals, meta, nullptr, rows, cols);
  if (rc) return rc;
  const size_t dom_cols = P.tile_order ? (size_t)P.k_tiles * 128 : cols;
  int blocks = 1;
  rc = capped_grid(ceil_div(ceil_div((size_t)P.dom_rows, 4) * (dom_cols / 4), 256), 16, &blocks);
  if (rc) return rc;
  const size_t fx = ceil_div(dom_cols / 4, 32), fy_all = ceil_div(ceil_div((size_t)P.dom_rows, 4), 8);
  size_t fy = ceil_div((size_t)blocks, fx);
  if (fy > fy_all) fy = fy_all;
  if (fy > 65535) fy = 65535;
  if (fy == 0) fy = 1;
  const dim3 grid((unsigned)fx, (unsigned)fy);
  if (dtype == SPFY_BF16) prune24_tile_fused_kernel<true, PATTERN><<<grid, 256, 0, s>>>(P);
  else prune24_tile_fused_kernel<false, PATTERN><<<grid, 256, 0, s>>>(P);
  SPFY_LAUNCH_OK("prune24_tile_fused_kernel");
  return SPFY_OK;
}

}  // namespace
}  // namespace spfy

void spfy::warm_prune_kernels() {
  touch_kernel(prune_blocks_ref_kernel<uint16_t>);
  touch_kernel(prune_blocks_ref_kernel<uint32_t>);
  touch_kernel(prune_blocks_ref_kernel<uint64_t>);
  touch_kernel(prune24_strip_kernel);
  touch_kernel(prune24_fast_kernel);
  touch_kernel(prune24_batched_kernel);
  touch_kernel(prune24_tile_batched_kernel<false>);
  touch_kernel(prune24_tile_batched_kernel<true>);
  touch_kernel(prune24_tile_kernel<false, false>);
  touch_kernel(prune24_tile_kernel<false, true>);
  touch_kernel(prune24_tile_kernel<true, false>);
  touch_kernel(prune24_tile_kernel<true, true>);
  touch_kernel(prune24_tile_fused_kernel<false, false>);
  touch_kernel(prune24_tile_fused_kernel<true, false>);
  touch_kernel(prune24_tile_fused_kernel<false, true>);
  touch_kernel(prune24_tile_fused_kernel<true, true>);
  touch_kernel(prune24_check_kernel);
}

using namespace spfy;

extern "C" {

int spfy_prune_blocks_ref(int dtype, void* weights, uint64_t* mask, size_t m, size_t n,
                          size_t blk_m, size_t blk_n, float sparsity_factor,
                          spfy_stream_t stream) {
  const size_t eb = dtype_bytes(dtype);
  if (!eb) return fail(SPFY_E_INVALID, "prune_blocks_ref: bad dtype %d", dtype);
  if (!weights || !mask) return fail(SPFY_E_INVALID, "prune_blocks_ref: null pointer");
  if (blk_m == 0 || blk_n == 0 || blk_m * blk_n > 256 || blk_m > 16 || blk_n > 16)
    return fail(SPFY_E_UNSUPPORTED, "prune_blocks_ref: block %zux%zu not supported (<=16x16)", blk_m, blk_n);
  const size_t total = m * n;
  if (total == 0) return SPFY_OK;
  const size_t blk_size = blk_m * blk_n;
  const size_t nblocks = (m / blk_m) * (n / blk_n);
  // sparsify.hxx:41 -- the product is evaluated in float
  const size_t nz = (size_t)floorf((float)blk_size * sparsity_factor);
  OffsetList L;
  memset(&L, 0, sizeof(L));
  L.in_block = 1;
  size_t done = 0;
  for (size_t h = 0; h < blk_m; ++h)
    for (size_t w = 0; w < blk_n; ++w) {
      if (done == nz) break;
      size_t o = h + w * blk_n;  // sparsify.hxx:60
      L.off[L.count++] = (uint16_t)o;
      if (o >= blk_size) L.in_block = 0; else L.bitmap[o >> 5] |= 1u << (o & 31);
      ++done;
    }
  int grid = 1;
  int rc = capped_grid(ceil_div(ceil_div(total, 4), 256), 16, &grid);
  if (rc) return rc;
  cudaStream_t s = (cudaStream_t)stream;
  if ((uintptr_t)mask % 8 || (uintptr_t)weights % eb)
    return fail(SPFY_E_INVALID, "prune_blocks_ref: weights / mask are not aligned to their element size");
  const int vec_w = (uintptr_t)weights % (eb == 8 ? 16 : 4 * eb) == 0;  // whole-vector RMW of the weights
  const int vec_m = (uintptr_t)mask % 16 == 0;                          // 16-byte mask stores
  switch (eb) {
    case 2: prune_blocks_ref_kernel<uint16_t><<<grid, 256, 0, s>>>((uint16_t*)weights, mask, total, nblocks, (uint32_t)blk_size, vec_w, vec_m, L); break;
    case 4: prune_blocks_ref_kernel<uint32_t><<<grid, 256, 0, s>>>((uint32_t*)weights, mask, total, nblocks, (uint32_t)blk_size, vec_w, vec_m, L); break;
    default: prune_blocks_ref_kernel<uint64_t><<<grid, 256, 0, s>>>((uint64_t*)weights, mask, total, nblocks, (uint32_t)blk_size, vec_w, vec_m, L); break;
  }
  SPFY_LAUNCH_OK("prune_blocks_ref_kernel");
  return SPFY_OK;
}

int spfy_compressed_bytes(int dtype, size_t rows, size_t cols, int layout, size_t* vals_bytes,
                          size_t* meta_bytes) {
  if (dtype != SPFY_F16 && dtype != SPFY_BF16)
    return fail(SPFY_E_UNSUPPORTED, "compressed_bytes: dtype %d (need F16/BF16)", dtype);
  size_t vb, mb;
  if (layout == SPFY_LAYOUT_CANONICAL) {
    const size_t G = ceil_div(cols, 4);
    vb = rows * G * 2 * 2;
    mb = rows * ceil_div(G, 2);
  } else if (layout == SPFY_LAYOUT_SM100) {
    const size_t tiles = ceil_div(rows, 128) * ceil_div(cols, 128);
    vb = tiles * 16384;
    mb = tiles * 2048;
  } else {
    return fail(SPFY_E_INVALID, "compressed_bytes: bad layout %d", layout);
  }
  if (vals_bytes) *vals_bytes = vb;
  if (meta_bytes) *meta_bytes = mb;
  return SPFY_OK;
}

// can the one-pass prune + compress kernel take these buffers?
static bool tile_fused_shape_ok(const void* in, size_t ld_in, const void* out_dense, size_t ld_out, const void* comp_vals,
                                const void* meta, size_t cols) {
  const bool vec = cols % 4 == 0 && ld_in % 4 == 0 && ld_out % 4 == 0 && (uintptr_t)in % 8 == 0 && (uintptr_t)out_dense % 8 == 0;
  return vec && cols % 16 == 0 && (uintptr_t)meta % 2 == 0 && (uintptr_t)comp_vals % 4 == 0;
}
// can this TILE_MAG request go through the one-pass prune + compress kernel?
static bool tile_fused_ok(const void* in, size_t ld_in, const void* out_dense, size_t ld_out, const void* comp_vals,
                          const void* meta, const uint64_t* mask, size_t cols) {
  return (comp_vals || meta) && !mask && tile_fused_shape_ok(in, ld_in, out_dense, ld_out, comp_vals, meta, cols);
}

int spfy_prune24(int dtype, int mode, int layout, const void* in, size_t ld_in, void* out_dense,
                 size_t ld_out, void* comp_vals, void* meta, uint64_t* mask, size_t rows,
                 size_t cols, spfy_stream_t stream) {
  if (dtype != SPFY_F16 && dtype != SPFY_BF16)
    return fail(SPFY_E_UNSUPPORTED, "prune24: dtype %d (need F16/BF16)", dtype);
  if (layout != SPFY_LAYOUT_CANONICAL && layout != SPFY_LAYOUT_SM100)
    return fail(SPFY_E_INVALID, "prune24: bad layout %d", layout);
  if (!in) return fail(SPFY_E_INVALID, "prune24: null input");
  if (ld_in < cols || (out_dense && ld_out < cols))
    return fail(SPFY_E_INVALID, "prune24: leading dimension smaller than cols");
  if (rows >= (1ull << 31) || cols >= (1ull << 31) || ld_in >= (1ull << 31) || (out_dense && ld_out >= (1ull << 31)))
    return fail(SPFY_E_UNSUPPORTED, "prune24: dimension too large");
  if (rows == 0 || cols == 0) return SPFY_OK;
  cudaStream_t s = (cudaStream_t)stream;

  const uint16_t* src = (const uint16_t*)in;
  size_t ld_src = ld_in;
  if (mode == SPFY_PRUNE_TILE_MAG) {
    if (!out_dense)
      return fail(SPFY_E_INVALID, "prune24: TILE_MAG needs out_dense (it may alias the input)");
    const bool vec = cols % 4 == 0 && ld_in % 4 == 0 && ld_out % 4 == 0 && (uintptr_t)src % 8 == 0 &&
                     (uintptr_t)out_dense % 8 == 0;
    // One pass for weight-sized matrices: the fused kernel saves a launch (every ResNet layer is launch-bound,
    // <= 2.4 M elements) but it is issue-bound and costs 526 us on 16384 x 16384 where the two passes take 445
    static const size_t fused_max = [] {
      const char* e = dev_switch("SPFY_TILE_FUSED_MAX");
      return e ? (size_t)strtoull(e, nullptr, 10) : (size_t)8 << 20;
    }();
    if (tile_fused_ok(src, ld_in, out_dense, ld_out, comp_vals, meta, mask, cols) && rows * cols <= fused_max)
      return launch_tile_fused<false>(dtype, layout, src, ld_in, out_dense, ld_out, comp_vals, meta, rows, cols, s);
    int blocks = 1;
    int rc = capped_grid(ceil_div(ceil_div(rows, 4) * ceil_div(cols, 4), 256), 16, &blocks);  // cap: two waves of resident warps
    if (rc) return rc;
    // 32 tile columns x 8 tile rows per block; the rows are walked with a stride when the cap binds
    const size_t gx = ceil_div(ceil_div(cols, 4), 32), gy_all = ceil_div(ceil_div(rows, 4), 8);
    if (gx >= (1u << 31)) return fail(SPFY_E_UNSUPPORTED, "prune24: too many columns");
    size_t gy = ceil_div((size_t)blocks, gx);
    if (gy > gy_all) gy = gy_all;
    if (gy > 65535) gy = 65535;
    if (gy == 0) gy = 1;
    const dim3 grid((unsigned)gx, (unsigned)gy);
    const uint32_t r32 = (uint32_t)rows, c32 = (uint32_t)cols;
    uint16_t* od = (uint16_t*)out_dense;
    if (dtype == SPFY_BF16) {
      if (vec) prune24_tile_kernel<true, true><<<grid, 256, 0, s>>>(src, ld_in, od, ld_out, r32, c32);
      else prune24_tile_kernel<true, false><<<grid, 256, 0, s>>>(src, ld_in, od, ld_out, r32, c32);
    } else {
      if (vec) prune24_tile_kernel<false, true><<<grid, 256, 0, s>>>(src, ld_in, od, ld_out, r32, c32);
      else prune24_tile_kernel<false, false><<<grid, 256, 0, s>>>(src, ld_in, od, ld_out, r32, c32);
    }
    SPFY_LAUNCH_OK("prune24_tile_kernel");
    if (!comp_vals && !meta && !mask) return SPFY_OK;
    // a valid 2:4 matrix is a fixed point of the strip selection: run it to compress
    src = (const uint16_t*)out_dense;
    ld_src = ld_out;
    out_dense = nullptr;
  } else if (mode == SPFY_PRUNE_TILE_TRANSPOSABLE) {
    if (!out_dense)
      return fail(SPFY_E_INVALID, "prune24: TILE_TRANSPOSABLE needs out_dense (it may alias the input)");
    if (mask) return fail(SPFY_E_UNSUPPORTED, "prune24: TILE_TRANSPOSABLE writes no mask");
    if (!tile_fused_shape_ok(src, ld_in, out_dense, ld_out, comp_vals, meta, cols))
      return fail(SPFY_E_UNSUPPORTED, "prune24: TILE_TRANSPOSABLE needs cols %% 16 == 0 and 8-byte aligned rows");
    return launch_tile_fused<true>(dtype, layout, src, ld_in, out_dense, ld_out, comp_vals, meta, rows, cols, s);
  } else if (mode != SPFY_PRUNE_STRIP_MAG) {
    return fail(SPFY_E_INVALID, "prune24: bad mode %d", mode);
  }

  Prune24Params P;
  int rc = fill_prune24(&P, layout, src, ld_src, out_dense, ld_out, comp_vals, meta, mask, rows, cols);
  if (rc) return rc;
  int grid = 1;
  if (P.fast) {
    rc = capped_grid(fast_passes(P), 16, &grid);
    if (rc) return rc;
    prune24_fast_kernel<<<grid, 256, 0, s>>>(P);
    SPFY_LAUNCH_OK("prune24_fast_kernel");
    return SPFY_OK;
  }
  rc = capped_grid(ceil_div((size_t)P.dom_rows * P.units_per_row, 256), 16, &grid);
  if (rc) return rc;
  prune24_strip_kernel<<<grid, 256, 0, s>>>(P);
  SPFY_LAUNCH_OK("prune24_strip_kernel");
  return SPFY_OK;
}

int spfy_prune24_batched(int dtype, int mode, int layout, const spfy_prune24_item* items, size_t count,
                         spfy_stream_t stream) {
  if (dtype != SPFY_F16 && dtype != SPFY_BF16)
    return fail(SPFY_E_UNSUPPORTED, "prune24_batched: dtype %d (need F16/BF16)", dtype);
  if (mode != SPFY_PRUNE_STRIP_MAG && mode != SPFY_PRUNE_TILE_MAG) return fail(SPFY_E_INVALID, "prune24_batched: bad mode %d", mode);
  if (layout != SPFY_LAYOUT_CANONICAL && layout != SPFY_LAYOUT_SM100)
    return fail(SPFY_E_INVALID, "prune24_batched: bad layout %d", layout);
  if (count && !items) return fail(SPFY_E_INVALID, "prune24_batched: null item table");
  int rc = SPFY_OK;
  cudaStream_t s = (cudaStream_t)stream;
  const bool tile = mode == SPFY_PRUNE_TILE_MAG;
  static thread_local Prune24Batch Bt;  // 10 KB: keep it off the stack
  size_t i = 0;
  while (i < count) {
    Bt.count = 0;
    Bt.tile_prefix[0] = 0;
    for (; i < count && Bt.count < PRUNE_BATCH_MAX; ++i) {
      const spfy_prune24_item& it = items[i];
      if (it.rows == 0 || it.cols == 0) continue;
      if (!it.in) return fail(SPFY_E_INVALID, "prune24_batched: item %zu has a null input", i);
      if (it.ld_in < it.cols || (it.out_dense && it.ld_out < it.cols))
        return fail(SPFY_E_INVALID, "prune24_batched: item %zu leading dimension smaller than cols", i);
      if (it.rows >= (1ull << 31) || it.cols >= (1ull << 31) || it.ld_in >= (1ull << 31) || (it.out_dense && it.ld_out >= (1ull << 31)))
        return fail(SPFY_E_UNSUPPORTED, "prune24_batched: item %zu too large", i);
      if (tile && !it.out_dense)
        return fail(SPFY_E_INVALID, "prune24_batched: item %zu: TILE_MAG needs out_dense (it may alias the input)", i);
      if (tile && !tile_fused_ok(it.in, it.ld_in, it.out_dense, it.ld_out, it.comp_vals, it.meta, nullptr, it.cols)) {
        // ragged / unaligned matrix (k = 147): the general two-pass route, on its own
        rc = spfy_prune24(dtype, mode, layout, it.in, it.ld_in, it.out_dense, it.ld_out, it.comp_vals, it.meta, nullptr,
                          it.rows, it.cols, stream);
        if (rc) return rc;
        continue;
      }
      Prune24Params& P = Bt.item[Bt.count];
      rc = fill_prune24(&P, layout, (const uint16_t*)it.in, it.ld_in, it.out_dense, it.ld_out,
                        it.comp_vals, it.meta, nullptr, it.rows, it.cols);
      if (rc) return rc;
      uint32_t tiles_c = 0;
      const size_t tiles = tile ? ceil_div(tile_fused_total(P, &tiles_c), 1024)
                                : (P.fast ? fast_passes(P) : ceil_div((size_t)P.dom_rows * P.units_per_row, 1024));
      if ((size_t)Bt.tile_prefix[Bt.count] + tiles >= (1ull << 32))
        return fail(SPFY_E_UNSUPPORTED, "prune24_batched: batch too large");
      Bt.tile_prefix[Bt.count + 1] = Bt.tile_prefix[Bt.count] + (uint32_t)tiles;
      ++Bt.count;
    }
    if (Bt.count == 0) continue;
    int grid = 1;
    rc = capped_grid(Bt.tile_prefix[Bt.count], 16, &grid);
    if (rc) return rc;
    if (!tile) {
      prune24_batched_kernel<<<grid, 256, 0, s>>>(Bt);
      SPFY_LAUNCH_OK("prune24_batched_kernel");
    } else {
      if (dtype == SPFY_BF16) prune24_tile_batched_kernel<true><<<grid, 256, 0, s>>>(Bt);
      else prune24_tile_batched_kernel<false><<<grid, 256, 0, s>>>(Bt);
      SPFY_LAUNCH_OK("prune24_tile_batched_kernel");
    }
  }
  return SPFY_OK;
}

int spfy_prune24_check(int dtype, const void* in, size_t ld_in, size_t rows, size_t cols,
                       int* d_invalid, spfy_stream_t stream) {
  if (dtype != SPFY_F16 && dtype != SPFY_BF16)
    return fail(SPFY_E_UNSUPPORTED, "prune24_check: dtype %d (need F16/BF16)", dtype);
  if (!in || !d_invalid) return fail(SPFY_E_INVALID, "prune24_check: null pointer");
  cudaStream_t s = (cudaStream_t)stream;
  SPFY_CUDA_OK(cudaMemsetAsync(d_invalid, 0, sizeof(int), s));
  if (rows == 0 || cols == 0) return SPFY_OK;
  const int vec = cols % 16 == 0 && ld_in % 8 == 0 && (uintptr_t)in % 16 == 0;
  int grid = 1;
  int rc = capped_grid(ceil_div(vec ? rows * (cols / 16) : rows * ceil_div(cols, 4), 256), 16, &grid);
  if (rc) return rc;
  prune24_check_kernel<<<grid, 256, 0, s>>>((const uint16_t*)in, ld_in, (uint32_t)rows, (uint32_t)cols, vec, d_invalid);
  SPFY_LAUNCH_OK("prune24_check_kernel");
  return SPFY_OK;
}

}  // extern "C"
