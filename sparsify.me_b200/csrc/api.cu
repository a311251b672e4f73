// api.cu -- library-level entry points of libsparsifyme_b200.so
#include "common.cuh"

namespace spfy {
namespace {

// streaming element-wise conversion: 8 elements per thread per trip when both sides are 16-byte
// aligned, scalar otherwise / for the tail
template <typename S, typename D>
__global__ void __launch_bounds__(256)
convert_kernel(const S* __restrict__ src, D* __restrict__ dst, size_t n, int vec) {
  const size_t tid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  const size_t nthreads = (size_t)gridDim.x * blockDim.x;
  size_t done = 0;
  if (vec) {
    const size_t chunks = n / 8;
    for (size_t c = tid; c < chunks; c += nthreads) {
      S in[8];
      D out[8];
      if (sizeof(S) == 4) {
        *reinterpret_cast<uint4*>(in) = *reinterpret_cast<const uint4*>(src + c * 8);
        *reinterpret_cast<uint4*>(in + 4) = *reinterpret_cast<const uint4*>(src + c * 8 + 4);
      } else {
        *reinterpret_cast<uint4*>(in) = *reinterpret_cast<const uint4*>(src + c * 8);
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) out[i] = from_f32<D>(to_f32(in[i]));
      if (sizeof(D) == 4) {
        *reinterpret_cast<uint4*>(dst + c * 8) = *reinterpret_cast<uint4*>(out);
        *reinterpret_cast<uint4*>(dst + c * 8 + 4) = *reinterpret_cast<uint4*>(out + 4);
      } else {
        *reinterpret_cast<uint4*>(dst + c * 8) = *reinterpret_cast<uint4*>(out);
      }
    }
    done = chunks * 8;
  }
  for (size_t i = done + tid; i < n; i += nthreads) dst[i] = from_f32<D>(to_f32(src[i]));
}

template <typename S, typename D>
int launch_convert(const void* src, void* dst, size_t n, cudaStream_t s) {
  int grid = 1;
  int rc = capped_grid(ceil_div(ceil_div(n, 8), 256), 8, &grid);
  if (rc) return rc;
  const int vec = ((uintptr_t)src % 16 == 0) && ((uintptr_t)dst % 16 == 0);
  convert_kernel<S, D><<<grid, 256, 0, s>>>((const S*)src, (D*)dst, n, vec);
  SPFY_LAUNCH_OK("convert_kernel");
  return SPFY_OK;
}

// conv weights [m][c][kh*kw] -> [m][kh*kw][c]: the K order of the implicit GEMM (spfy_spmma_conv)
__global__ void __launch_bounds__(256)
permute_conv_weights_kernel(const uint16_t* __restrict__ in, uint16_t* __restrict__ out, size_t m, uint32_t c, uint32_t taps) {
  const size_t total = m * c * taps;
  const size_t nthreads = (size_t)gridDim.x * blockDim.x;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += nthreads) {
    const size_t row = i / ((size_t)c * taps);
    const uint32_t r = (uint32_t)(i - row * c * taps), tap = r / c, ch = r - tap * c;  // i walks the OUTPUT
    out[i] = in[row * c * taps + (size_t)ch * taps + tap];
  }
}

}  // namespace
}  // namespace spfy

using namespace spfy;

extern "C" {

int spfy_permute_conv_weights(const void* in, void* out, size_t m, size_t c, size_t kh, size_t kw, spfy_stream_t stream) {
  if (m == 0 || c == 0 || kh == 0 || kw == 0) return SPFY_OK;
  if (!in || !out) return fail(SPFY_E_INVALID, "permute_conv_weights: null pointer");
  if (in == out) return fail(SPFY_E_INVALID, "permute_conv_weights: in place is not supported");
  if (c >= (1ull << 31) || kh * kw >= (1ull << 31)) return fail(SPFY_E_UNSUPPORTED, "permute_conv_weights: too large");
  int grid = 1;
  int rc = capped_grid(ceil_div(m * c * kh * kw, 256), 8, &grid);
  if (rc) return rc;
  permute_conv_weights_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>((const uint16_t*)in, (uint16_t*)out, m, (uint32_t)c,
                                                                      (uint32_t)(kh * kw));
  SPFY_LAUNCH_OK("permute_conv_weights_kernel");
  return SPFY_OK;
}

int spfy_version(void) { return 100; }  // 0.1.0

int spfy_init(void) {
  static std::atomic<int> done[64];
  int dev = 0;
  SPFY_CUDA_OK(cudaGetDevice(&dev));
  if (dev < 0 || dev >= 64) return fail(SPFY_E_CUDA, "device index %d out of range", dev);
  if (done[dev].load(std::memory_order_acquire)) return SPFY_OK;
  DeviceInfo di;
  int rc = device_info(&di);
  if (rc) return rc;
  spfy::warm_prune_kernels();
  spfy::warm_transpose24_kernels();
  spfy::warm_spmma_kernels();
  spfy::warm_spmm_kernels();
  spfy::warm_gemm_kernels();
  spfy::warm_optim24_kernels();
  touch_kernel(convert_kernel<float, __half>);
  touch_kernel(convert_kernel<float, __nv_bfloat16>);
  touch_kernel(convert_kernel<__half, float>);
  touch_kernel(convert_kernel<__nv_bfloat16, float>);
  (void)cudaGetLastError();
  // Loading the code is not all a first call pays (a first spmma launch still took 4-16 ms in the one-shot
  // example drivers: opt-in shared memory, tensor maps, the first allocation of the stream-ordered pool ...), so
  // every entry point the header templates use runs once here on a 128 x 128 scratch problem.
  done[dev].store(1, std::memory_order_release);  // (the calls below may re-enter through the same checks)
  {
    uint8_t* buf = nullptr;
    const size_t mat = 128 * 128 * sizeof(float);
    size_t vb = 0, mb = 0;
    if (spfy_compressed_bytes(SPFY_F16, 128, 128, SPFY_LAYOUT_SM100, &vb, &mb) == SPFY_OK &&
        cudaMalloc(&buf, 4 * mat + vb + mb + 128 * 128 * 8) == cudaSuccess) {
      (void)cudaMemset(buf, 0, 4 * mat + vb + mb + 128 * 128 * 8);
      void *A = buf, *B = buf + mat, *D = buf + 2 * mat, *W = buf + 3 * mat, *vals = buf + 4 * mat, *meta = buf + 4 * mat + vb;
      uint64_t* mask = reinterpret_cast<uint64_t*>(buf + 4 * mat + vb + mb);
      for (int dt = SPFY_F16; dt <= SPFY_BF16; ++dt) {
        (void)spfy_prune24(dt, SPFY_PRUNE_TILE_MAG, SPFY_LAYOUT_SM100, A, 128, A, 128, vals, meta, nullptr, 128, 128, nullptr);
        (void)spfy_prune24(dt, SPFY_PRUNE_STRIP_MAG, SPFY_LAYOUT_SM100, A, 128, A, 128, vals, meta, nullptr, 128, 128, nullptr);
        if (di.cc_major == 10)
          for (int op = SPFY_OP_N; op <= SPFY_OP_T; ++op)
            (void)spfy_spmma(dt, op, 128, 128, 128, 1.f, vals, meta, B, 128, 0.f, nullptr, 0, D, 128, nullptr, 0, nullptr);
      }
      (void)spfy_prune_blocks_ref(SPFY_F32, W, mask, 128, 128, 2, 2, 0.5f, nullptr);
      // unstructured path: W <- 0.747 everywhere, thresholded to a full COO, multiplied through the CSR entry
      // (which launches both SpMM kernels) for a short and a tall A, and through the blocked-ELL entry
      {
        (void)cudaMemset(W, 0x3f, mat);
        int32_t* ri = reinterpret_cast<int32_t*>(A);            // 16384 int32 fit in the 64 KiB of A, B, D each
        int32_t* ci = reinterpret_cast<int32_t*>(B);
        float* va = reinterpret_cast<float*>(D);
        uint8_t* tail = reinterpret_cast<uint8_t*>(mask);       // 128 KiB: nnz, row_ptr, workspaces, pointer tables
        int64_t* nnz = reinterpret_cast<int64_t*>(tail);
        int32_t* rp = reinterpret_cast<int32_t*>(tail + 256);
        uint8_t* ws = tail + 4096;
        float* Bm = reinterpret_cast<float*>(vals);             // >= 8 KiB: reuse the compressed-operand area as B, C
        size_t tws = 0, sws = 0;
        (void)spfy_threshold_workspace_bytes(128, 128, &tws);
        (void)spfy_spmm_workspace_bytes(SPFY_SPMM_ALG_CUDA_CORE, 128, 128, 8, 1, 16384, &sws);
        if (tws <= 32768 && sws <= 32768 && vb >= 2 * 128 * 8 * sizeof(float)) {
          float* Cm = Bm + 128 * 8;
          (void)spfy_threshold_to_coo(SPFY_F32, W, 128, 128, 128, 0.5f, ri, ci, va, 16384, nnz, rp, ws, 32768, nullptr);
          for (size_t mm = 64; mm <= 128; mm += 64)
            (void)spfy_spmm_csr_strided_batched(SPFY_SPMM_ALG_CUDA_CORE, mm, 128, 8, 1, rp, ci, va, Bm, 128, 128 * 8, Cm, mm, mm * 8, 1.f, 0.f, ws, 32768, nullptr);
          const void* hp[3] = {ci /* block-column ids (int64 view of zeros is fine) */, W, Cm};
          void** dp = reinterpret_cast<void**>(tail + 65536);
          (void)cudaMemset(ci, 0, mat);
          (void)cudaMemcpy(dp, hp, sizeof(hp), cudaMemcpyHostToDevice);
          for (size_t mm = 64; mm <= 128; mm += 64)
            (void)spfy_spmm_bell_batched(SPFY_SPMM_ALG_CUDA_CORE, SPFY_F32, mm, 128, 8, 2, 16, 1, reinterpret_cast<const int64_t* const*>(dp),
                                         reinterpret_cast<const void* const*>(dp + 1), Bm, 128,
                                         reinterpret_cast<void* const*>(dp + 2), mm, 1.f, 0.f, ws, 32768, nullptr);
        }
      }
      (void)spfy_convert(SPFY_F32, SPFY_F16, W, A, 128 * 128, nullptr);
      (void)spfy_convert(SPFY_F16, SPFY_F32, A, W, 128 * 128, nullptr);
      if (di.cc_major == 10)  // dense tcgen05 GEMM (batched::gemm and the tensor-core routes of the SpMM entries)
        for (int dt = SPFY_F16; dt <= SPFY_F32; ++dt)
          (void)spfy_gemm_strided_batched(dt, SPFY_GEMM_PRECISE, SPFY_OP_N, SPFY_OP_N, 128, 128, 128, 1.f, A, 128, 0, B, 128,
                                          0, 0.f, D, 128, 0, 1, nullptr, 0, nullptr);
      (void)cudaDeviceSynchronize();
      (void)cudaFree(buf);
    }
    (void)cudaGetLastError();
  }
  return SPFY_OK;
}

const char* spfy_last_error_string(void) { return spfy::err_buf(); }

uint64_t spfy_launch_count(void) { return spfy::launch_counter().load(std::memory_order_relaxed); }

int spfy_convert(int src_dtype, int dst_dtype, const void* src, void* dst, size_t count,
                 spfy_stream_t stream) {
  if (count == 0) return SPFY_OK;
  if (!src || !dst) return fail(SPFY_E_INVALID, "convert: null pointer");
  cudaStream_t s = (cudaStream_t)stream;
  if (src_dtype == SPFY_F32 && dst_dtype == SPFY_F16) return launch_convert<float, __half>(src, dst, count, s);
  if (src_dtype == SPFY_F32 && dst_dtype == SPFY_BF16) return launch_convert<float, __nv_bfloat16>(src, dst, count, s);
  if (src_dtype == SPFY_F16 && dst_dtype == SPFY_F32) return launch_convert<__half, float>(src, dst, count, s);
  if (src_dtype == SPFY_BF16 && dst_dtype == SPFY_F32) return launch_convert<__nv_bfloat16, float>(src, dst, count, s);
  return fail(SPFY_E_UNSUPPORTED, "convert: %d -> %d is not supported (F32 <-> F16/BF16 only)", src_dtype, dst_dtype);
}

// ---------------------------------------------------------------- pruned-layer container (host memory only)
namespace {
struct PackedHeader {
  char magic[8];
  uint32_t version;
  int32_t dtype, layout;
  uint32_t reserved;
  uint64_t rows, cols, vals_bytes, meta_bytes, checksum;
};
static_assert(sizeof(PackedHeader) == SPFY_PACKED_HEADER_BYTES, "container header is 64 bytes");
const char kPackedMagic[8] = {'S', 'P', 'F', 'Y', '2', '4', 0, 0};

uint64_t fnv1a64(const uint8_t* p, size_t n, uint64_t h) {
  for (size_t i = 0; i < n; ++i) h = (h ^ p[i]) * 0x100000001b3ull;
  return h;
}
}  // namespace

int spfy_packed_bytes(int dtype, size_t rows, size_t cols, int layout, size_t* bytes) {
  size_t vb = 0, mb = 0;
  int rc = spfy_compressed_bytes(dtype, rows, cols, layout, &vb, &mb);
  if (rc) return rc;
  if (bytes) *bytes = SPFY_PACKED_HEADER_BYTES + vb + mb;
  return SPFY_OK;
}

int spfy_packed_write(int dtype, int layout, size_t rows, size_t cols, const void* host_vals,
                      const void* host_meta, void* dst, size_t dst_bytes) {
  size_t vb = 0, mb = 0;
  int rc = spfy_compressed_bytes(dtype, rows, cols, layout, &vb, &mb);
  if (rc) return rc;
  if (!dst || (vb && !host_vals) || (mb && !host_meta)) return fail(SPFY_E_INVALID, "packed_write: null pointer");
  if (dst_bytes < SPFY_PACKED_HEADER_BYTES + vb + mb)
    return fail(SPFY_E_WORKSPACE, "packed_write: buffer %zu < %zu bytes", dst_bytes, (size_t)SPFY_PACKED_HEADER_BYTES + vb + mb);
  PackedHeader h;
  memset(&h, 0, sizeof(h));
  memcpy(h.magic, kPackedMagic, 8);
  h.version = 1;
  h.dtype = dtype;
  h.layout = layout;
  h.rows = rows;
  h.cols = cols;
  h.vals_bytes = vb;
  h.meta_bytes = mb;
  h.checksum = fnv1a64((const uint8_t*)host_meta, mb, fnv1a64((const uint8_t*)host_vals, vb, 0xcbf29ce484222325ull));
  uint8_t* out = (uint8_t*)dst;
  memcpy(out, &h, sizeof(h));
  memcpy(out + sizeof(h), host_vals, vb);
  memcpy(out + sizeof(h) + vb, host_meta, mb);
  return SPFY_OK;
}

int spfy_packed_read(const void* src, size_t src_bytes, int* dtype, int* layout, size_t* rows, size_t* cols,
                     size_t* vals_offset, size_t* vals_bytes, size_t* meta_offset, size_t* meta_bytes) {
  if (!src || src_bytes < SPFY_PACKED_HEADER_BYTES) return fail(SPFY_E_INVALID, "packed_read: buffer shorter than a header");
  PackedHeader h;
  memcpy(&h, src, sizeof(h));
  if (memcmp(h.magic, kPackedMagic, 8) != 0) return fail(SPFY_E_INVALID, "packed_read: bad magic");
  if (h.version != 1) return fail(SPFY_E_UNSUPPORTED, "packed_read: container version %u", h.version);
  size_t vb = 0, mb = 0;
  int rc = spfy_compressed_bytes(h.dtype, (size_t)h.rows, (size_t)h.cols, h.layout, &vb, &mb);
  if (rc) return rc;
  if (vb != h.vals_bytes || mb != h.meta_bytes)
    return fail(SPFY_E_INVALID, "packed_read: sizes in the header do not match the shape");
  if (src_bytes < SPFY_PACKED_HEADER_BYTES + vb + mb) return fail(SPFY_E_INVALID, "packed_read: truncated payload");
  const uint8_t* p = (const uint8_t*)src + SPFY_PACKED_HEADER_BYTES;
  if (fnv1a64(p + vb, mb, fnv1a64(p, vb, 0xcbf29ce484222325ull)) != h.checksum)
    return fail(SPFY_E_INVALID, "packed_read: checksum mismatch");
  if (dtype) *dtype = h.dtype;
  if (layout) *layout = h.layout;
  if (rows) *rows = (size_t)h.rows;
  if (cols) *cols = (size_t)h.cols;
  if (vals_offset) *vals_offset = SPFY_PACKED_HEADER_BYTES;
  if (vals_bytes) *vals_bytes = vb;
  if (meta_offset) *meta_offset = SPFY_PACKED_HEADER_BYTES + vb;
  if (meta_bytes) *meta_bytes = mb;
  return SPFY_OK;
}

}  // extern "C"
