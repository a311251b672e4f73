// tc_ptx.cuh -- PTX wrappers shared by the tcgen05 kernels (spmma_sm100.cu, gemm_sm100.cu): mbarriers, TMA /
// bulk copies, TMEM allocation, tcgen05.mma / .cp / .ld / .commit, shared-memory matrix descriptors.
#pragma once
#include "common.cuh"

#include <cuda.h>  // CUtensorMap (types only; the encoder is fetched through the runtime)

namespace spfy {
namespace ptx {

constexpr uint64_t HINT_EVICT_FIRST = 0x12F0000000000000ull;
constexpr uint64_t HINT_EVICT_LAST = 0x14F0000000000000ull;
constexpr uint64_t HINT_EVICT_NORMAL = 0x1000000000000000ull;

__device__ __forceinline__ uint32_t smem_u32(const void* p) {
  return (uint32_t)__cvta_generic_to_shared(p);
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint32_t bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.b32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(bar), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ uint64_t globaltimer_ns() {
  uint64_t t;
  asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
  return t;
}
// Bounded wait: a protocol bug must become a trap, not a hung GPU.
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const uint64_t t0 = globaltimer_ns();
  uint32_t spins = 0;
  while (!mbar_try_wait(bar, parity)) {
    if ((++spins & 0x3ff) == 0 && globaltimer_ns() - t0 > 4000000000ull) {
      printf("spfy spmma: mbarrier wait timed out (block %d thread %d bar 0x%x parity %u)\n",
             (int)blockIdx.x, (int)threadIdx.x, bar, parity);
      __trap();
    }
  }
}
__device__ __forceinline__ void fence_barrier_init() {
  asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tma_load_2d(uint32_t dst, const CUtensorMap* map, int c0, int c1,
                                            uint32_t bar, uint64_t hint) {
  asm volatile(
      "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4}], [%2], %5;"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "l"(hint)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, int c0, int c1, int c2,
                                            uint32_t bar, uint64_t hint) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4, %5}], [%2], %6;"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "l"(hint)
      : "memory");
}
// im2col mode (4-D NHWC tensor {C, W, H, N}): `pixels` consecutive output positions starting at base pixel (w, h, n) --
// walking W, then H, then N inside the bounding box of the tensor map -- x `channels` channels from c, at filter tap
// (off_w, off_h); out-of-image taps are zero-filled
__device__ __forceinline__ void tma_load_im2col_4d(uint32_t dst, const CUtensorMap* map, int c, int w, int h, int n,
                                                   uint16_t off_w, uint16_t off_h, uint32_t bar, uint64_t hint) {
  asm volatile(
      "cp.async.bulk.tensor.4d.shared::cluster.global.im2col.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1, {%3, %4, %5, %6}], [%2], {%7, %8}, %9;"
      ::"r"(dst), "l"(map), "r"(bar), "r"(c), "r"(w), "r"(h), "r"(n), "h"(off_w), "h"(off_h), "l"(hint)
      : "memory");
}
__device__ __forceinline__ void bulk_load_1d(uint32_t dst, const void* src, uint32_t bytes,
                                             uint32_t bar, uint64_t hint) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes.L2::cache_hint"
      " [%0], [%1], %2, [%3], %4;"
      ::"r"(dst), "l"(src), "r"(bytes), "r"(bar), "l"(hint)
      : "memory");
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, uint32_t src, int c0, int c1) {
  asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
               ::"l"(map), "r"(src), "r"(c0), "r"(c1)
               : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void bulk_wait_read_all() {
  asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
}
__device__ __forceinline__ void bulk_wait_all() {
  asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
}
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
  asm volatile("prefetch.tensormap [%0];" ::"l"(map) : "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst, uint32_t cols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst),
               "r"(cols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t cols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(cols)
               : "memory");
}
__device__ __forceinline__ void tc_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar)
               : "memory");
}
// metadata: 128 lanes x 128 bits, shared memory -> TMEM (4 columns)
__device__ __forceinline__ void tc_cp_128x128b(uint32_t taddr, uint64_t sdesc) {
  asm volatile("tcgen05.cp.cta_group::1.128x128b [%0], %1;" ::"r"(taddr), "l"(sdesc) : "memory");
}
// D[tmem] (+)= A(2:4)[smem] * B[smem], metadata in TMEM
__device__ __forceinline__ void tc_mma_sp_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b,
                                              uint32_t tmem_e, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %5, 0;\n"
      "tcgen05.mma.sp.cta_group::1.kind::f16 [%0], %1, %2, [%3], %4, p;\n"
      "}\n"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(tmem_e), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_x32(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
      "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]),
        "=r"(r[7]), "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]),
        "=r"(r[14]), "=r"(r[15]), "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]),
        "=r"(r[21]), "=r"(r[22]), "=r"(r[23]), "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]),
        "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_ld_x16(uint32_t taddr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
      "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr)
      : "memory");
}
__device__ __forceinline__ void tmem_wait_ld() {
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void st_shared_v4(uint32_t addr, uint32_t a, uint32_t b, uint32_t c,
                                             uint32_t d) {
  asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d)
               : "memory");
}

__device__ __forceinline__ void st_shared_u16(uint32_t addr, uint32_t v) {
  asm volatile("st.shared.u16 [%0], %1;" ::"r"(addr), "h"((uint16_t)v) : "memory");
}

// shared-memory matrix descriptor (sm_100 format, version 1)
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t saddr, uint32_t lbo_bytes,
                                                   uint32_t sbo_bytes, uint32_t layout_type) {
  return (uint64_t)((saddr >> 4) & 0x3fffu) | (uint64_t)((lbo_bytes >> 4) & 0x3fffu) << 16 |
         (uint64_t)((sbo_bytes >> 4) & 0x3fffu) << 32 | (uint64_t)1 << 46 |
         (uint64_t)layout_type << 61;
}
constexpr uint32_t LAYOUT_SW128 = 2, LAYOUT_NONE = 0;
constexpr uint32_t LAYOUT_SW128_BASE32B = 1;  // 128-byte rows, 32-byte chunks XOR-ed with (row & 3): MN-major 32-bit operands

template <bool BF16>
__device__ __forceinline__ uint32_t pack2(float a, float b) {
  if (BF16) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
  } else {
    __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
  }
}
template <bool BF16>
__device__ __forceinline__ float2 unpack2(uint32_t w) {
  if (BF16) {
    return __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&w));
  } else {
    return __half22float2(*reinterpret_cast<__half2*>(&w));
  }
}

// The producer and MMA roles are executed by a whole, converged warp whose lanes all hold the same
// values; only the instruction that must be issued once sits under `if (leader)`.  ptxas can then keep
// descriptors, coordinates and barrier addresses in uniform registers and feed UTMALDG / UTCHMMA
// directly.  (Running those loops inside `if (lane == 0)` instead makes every operand "possibly
// divergent": each MMA was then preceded by an ELECT + seven R2UR.BROADCAST waterfall, ~25 scalar
// instructions per MMA on the one thread the whole SM waits for.)  Values that come from memory are
// re-broadcast from lane 0 so that the compiler can prove them uniform.
__device__ __forceinline__ uint32_t uni(uint32_t v) { return __shfl_sync(0xffffffffu, v, 0); }
__device__ __forceinline__ uint64_t uni(uint64_t v) {
  return (uint64_t)uni((uint32_t)v) | (uint64_t)uni((uint32_t)(v >> 32)) << 32;
}
template <typename T>
__device__ __forceinline__ const T* uni(const T* p) { return reinterpret_cast<const T*>(uni((uint64_t)(uintptr_t)p)); }
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "elect.sync _|p, 0xffffffff;\n"
      "selp.b32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(pred));
  return pred != 0;
}


// D[tmem] (+)= A[smem] * B[smem], dense: kind::f16 (fp16 / bf16 operands) and kind::tf32 (fp32 containers, the
// tensor core reads the upper 19 bits)
__device__ __forceinline__ void tc_mma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                           uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
      "}\n"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tc_mma_tf32(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                            uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
      "}\n"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// the same with the A operand in tensor memory (lane = row, one 32-bit column per K element)
__device__ __forceinline__ void tc_mma_tf32_ts(uint32_t tmem_d, uint32_t tmem_a, uint64_t desc_b, uint32_t idesc,
                                               uint32_t accumulate) {
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "setp.ne.b32 p, %4, 0;\n"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], [%1], %2, %3, p;\n"
      "}\n"
      ::"r"(tmem_d), "r"(tmem_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
// registers -> tensor memory: the warp writes its 32 lanes x 32 consecutive columns (register j -> column j)
__device__ __forceinline__ void tmem_st_x32(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
      "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]), "r"(r[16]), "r"(r[17]),
        "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]), "r"(r[24]), "r"(r[25]), "r"(r[26]),
        "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
      : "memory");
}
__device__ __forceinline__ void tmem_st_x16(uint32_t taddr, const uint32_t* r) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
      "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]), "r"(r[8]),
        "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
      : "memory");
}
__device__ __forceinline__ void tmem_wait_st() {
  asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t ld_shared_u32(uint32_t addr) {
  uint32_t v;
  asm volatile("ld.shared.u32 %0, [%1];" : "=r"(v) : "r"(addr));
  return v;
}
// 16-byte global -> shared copy that bypasses the registers (zeros when !valid; src is not read then); complete for the
// issuing thread after cp_async_wait_all
__device__ __forceinline__ void cp_async_16(uint32_t dst, const void* src, bool valid) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(dst), "l"(src), "r"(valid ? 16u : 0u) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;" ::: "memory"); }
__device__ __forceinline__ uint32_t ld_shared_u16(uint32_t addr) {
  uint16_t v;
  asm volatile("ld.shared.u16 %0, [%1];" : "=h"(v) : "r"(addr));
  return v;
}
__device__ __forceinline__ uint4 ld_shared_v4(uint32_t addr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr));
  return v;
}

}  // namespace ptx

// cuTensorMapEncodeTiled through the runtime's driver entry point (no -lcuda)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*,
                                  const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                  const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

typedef CUresult (*EncodeIm2colFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                   const cuuint64_t*, const int*, const int*, cuuint32_t, cuuint32_t, const cuuint32_t*,
                                   CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion,
                                   CUtensorMapFloatOOBfill);

inline int get_im2col_encoder(EncodeIm2colFn* out) {
  static std::atomic<void*> cached{nullptr};
  void* fn = cached.load(std::memory_order_acquire);
  if (!fn) {
    cudaDriverEntryPointQueryResult qres;
    SPFY_CUDA_OK(cudaGetDriverEntryPoint("cuTensorMapEncodeIm2col", &fn, cudaEnableDefault, &qres));
    if (qres != cudaDriverEntryPointSuccess || !fn)
      return fail(SPFY_E_CUDA, "cuTensorMapEncodeIm2col not available from this driver");
    cached.store(fn, std::memory_order_release);
  }
  *out = (EncodeIm2colFn)fn;
  return SPFY_OK;
}

inline int get_encoder(EncodeTiledFn* out) {
  static std::atomic<void*> cached{nullptr};
  void* fn = cached.load(std::memory_order_acquire);
  if (!fn) {
    cudaDriverEntryPointQueryResult qres;
    SPFY_CUDA_OK(cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &qres));
    if (qres != cudaDriverEntryPointSuccess || !fn)
      return fail(SPFY_E_CUDA, "cuTensorMapEncodeTiled not available from this driver");
    cached.store(fn, std::memory_order_release);
  }
  *out = (EncodeTiledFn)fn;
  return SPFY_OK;
}

// The encoders need a current context.  A thread that has made no runtime call that needs one -- torch's autograd
// backward threads, for one -- has none and gets CUDA_ERROR_INVALID_CONTEXT: bind the device's primary context (any
// such runtime call does) and encode once more.
template <typename Encode>
inline CUresult encode_with_context(Encode&& encode) {
  CUresult r = encode();
  if (r == CUDA_ERROR_INVALID_CONTEXT && cudaFree(nullptr) == cudaSuccess) r = encode();
  return r;
}

// A tiled tensor map of `rank` <= 3 dimensions, innermost first (`byte_strides` has rank - 1 entries): element strides 1,
// no interleave, L2 promotion in 256-byte lines, out-of-bounds elements read as zero.
inline int encode_tiled(CUtensorMap* map, int dtype, uint32_t rank, const void* base, const cuuint64_t* dims,
                        const cuuint64_t* byte_strides, const cuuint32_t* box, CUtensorMapSwizzle swizzle, const char* who) {
  EncodeTiledFn enc;
  int rc = get_encoder(&enc);
  if (rc) return rc;
  const cuuint32_t estr[3] = {1, 1, 1};
  const CUtensorMapDataType dt = dtype == SPFY_F32    ? CU_TENSOR_MAP_DATA_TYPE_FLOAT32
                                 : dtype == SPFY_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16
                                                      : CU_TENSOR_MAP_DATA_TYPE_FLOAT16;
  const CUresult r = encode_with_context([&] {
    return enc(map, dt, rank, const_cast<void*>(base), dims, byte_strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE, swizzle,
               CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  });
  if (r != CUDA_SUCCESS)
    return fail(SPFY_E_CUDA, "%s: cuTensorMapEncodeTiled failed (%d) for dims %llu x %llu x %llu, row pitch %llu bytes", who,
                (int)r, (unsigned long long)dims[0], (unsigned long long)dims[1],
                (unsigned long long)(rank > 2 ? dims[2] : 1), (unsigned long long)byte_strides[0]);
  return SPFY_OK;
}

// the im2col view of an implicit GEMM's B: NHWC [batch][h][w][c], a kh x kw window whose base pixels run over
// [lo, dim + up) per spatial dimension with `stride` -- the ho x wo output positions of every image
struct Im2col {
  size_t batch, h, w, c, kh, kw, stride;
  int lo_h, lo_w, up_h, up_w;
  size_t ho, wo;
};

// a forward convolution: the bounding box is [-pad, dim + pad - (filter - 1))
inline Im2col im2col_of(const spfy_conv_desc& c) {
  const int p = (int)c.pad;
  return Im2col{c.batch, c.h, c.w, c.c, c.kh, c.kw, c.stride, -p, -p, p - (int)(c.kh - 1), p - (int)(c.kw - 1),
                (c.h + 2 * c.pad - c.kh) / c.stride + 1, (c.w + 2 * c.pad - c.kw) / c.stride + 1};
}

// NHWC activations {C, W, H, N} in im2col mode: one instruction gathers `pixels` consecutive output positions x 64
// channels of one filter tap (128 B swizzle: position j is the 128-byte row j of the box).  The bounding box of base
// pixels (Im2col), walked with the convolution stride, holds exactly the output positions, row by row, image by image.
// (spmma_sm100.cu: 128 positions, the columns of a B stage; gemm_sm100.cu's weight gradient: 64, the k-rows of a stage.)
inline int make_tmap_im2col(CUtensorMap* map, int dtype, const void* x, const Im2col& c, uint32_t pixels) {
  EncodeIm2colFn enc;
  int rc = get_im2col_encoder(&enc);
  if (rc) return rc;
  cuuint64_t dims[4] = {c.c, c.w, c.h, c.batch};
  cuuint64_t strides[3] = {c.c * 2, c.w * c.c * 2, c.h * c.w * c.c * 2};
  int lower[2] = {c.lo_w, c.lo_h};
  int upper[2] = {c.up_w, c.up_h};
  cuuint32_t estr[4] = {1, (cuuint32_t)c.stride, (cuuint32_t)c.stride, 1};
  CUresult r = encode_with_context([&] {
    return enc(map, dtype == SPFY_BF16 ? CU_TENSOR_MAP_DATA_TYPE_BFLOAT16 : CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4,
               const_cast<void*>(x), dims, strides, lower, upper, /*channelsPerPixel*/ 64, /*pixelsPerColumn*/ pixels, estr,
               CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
               CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  });
  if (r != CUDA_SUCCESS)
    return fail(SPFY_E_CUDA, "cuTensorMapEncodeIm2col failed (%d) for NHWC %zu x %zu x %zu x %zu, filter %zu x %zu stride %zu, "
                "corners (%d, %d) / (%d, %d)", (int)r, c.batch, c.h, c.w, c.c, c.kh, c.kw, c.stride, c.lo_h, c.lo_w, c.up_h, c.up_w);
  return SPFY_OK;
}

}  // namespace spfy
