/*
 * spfy_b200.h -- C ABI of libsparsifyme_b200.so
 *
 * The B200-native (sm_100a) replacement for the device work behind the
 * header-only `include/sparsify.me` API of owensgroup/sparsify.me.  The
 * reference has no FFI: its "plugin boundary" is five function templates
 * (SURVEY.md section 8b).  Every entry point below is what the corresponding
 * template in our `include/sparsify.me/ *.hxx` forwards to, and each one names
 * the reference call it replaces (file:line under the reference tree).
 *
 * Conventions (all entry points):
 *   - plain C types only: raw device pointers, sizes, enums as int;
 *   - return 0 on success, a negative SPFY_E_* code otherwise; never throw;
 *     `spfy_last_error_string()` returns a thread-local description;
 *   - all device work is enqueued on the caller's stream (a cudaStream_t,
 *     spelled `spfy_stream_t` so that this header needs no CUDA include);
 *   - no hidden allocation on the hot path: temporaries come from a
 *     caller-provided workspace, sized by the matching *_workspace_bytes query;
 *   - there is NO host fallback: without a CUDA device every compute entry
 *     point fails with SPFY_E_CUDA.
 */
#ifndef SPFY_B200_H_
#define SPFY_B200_H_

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#if defined(_WIN32)
#define SPFY_API
#else
#define SPFY_API __attribute__((visibility("default")))
#endif

typedef struct CUstream_st* spfy_stream_t; /* == cudaStream_t */

/* ---- enums (passed as int) --------------------------------------------- */
enum { SPFY_F16 = 0, SPFY_BF16 = 1, SPFY_F32 = 2, SPFY_F64 = 3 };

/* prune24 modes.  STRIP_MAG is the contract mode (top-2-of-4 by |x| along K,
 * tie -> lower index).  TILE_MAG is the 4x4-tile variant the reference asks
 * cusparseLt for at include/sparsify.me/spmma.hxx:86: each 4x4 tile keeps one of
 * the 90 patterns with two of four along rows AND columns; its metadata is what
 * the STRIP compressor makes of the pruned matrix (bit-exact with cusparseLt), so
 * where a kept value is +-0 the recorded index may move to another zero.
 * TILE_TRANSPOSABLE makes the same choice and the same dense output, but records
 * the tile's pattern itself in the metadata: it stays two of four along columns,
 * which spfy_transpose24 needs.  Values and metadata equal TILE_MAG's except in
 * groups where a kept value is +-0; padding rows / columns keep the neutral nibble.
 * Arguments as TILE_MAG (out_dense required, may alias `in`); `mask` is refused
 * and the call needs cols % 16 == 0 and 8-byte aligned rows (SPFY_E_UNSUPPORTED
 * otherwise).  spfy_prune24_batched refuses it. */
enum { SPFY_PRUNE_STRIP_MAG = 0, SPFY_PRUNE_TILE_MAG = 1, SPFY_PRUNE_TILE_TRANSPOSABLE = 2 };

/* layouts of the compressed operand.
 *   CANONICAL : values  [rows][ceil4(cols)/2]   row-major, ascending index
 *               meta    [rows][ceil4(cols)/8]   bytes; group g of a row sits in
 *                       byte g/2, low nibble for even g; nibble = i0 | i1<<2
 *   SM100     : what spfy_spmma consumes.  values and metadata are split into
 *               (128-row x 128-logical-k) tiles; tile (mt,kt) sits at index
 *               kt*m_tiles + mt (k-tile major: the m-tiles of one k-tile are adjacent).
 *               A value tile (16 KiB) is ONE 128-row x 128-byte image, the 128B-swizzled
 *               K-major shared-memory layout the UMMA descriptor reads: row r at r*128,
 *               16-byte chunk c of the row (8 stored values = 16 logical k) at
 *               ((c ^ (r & 7)) << 4).  A metadata tile (2 KiB) is the `tcgen05.cp.128x128b`
 *               source image: the 16-bit word of in-tile row r and 16-column unit q sits at byte
 *               (r>>4)*256 + (q&1)*128 + (r&7)*16 + (q>>1)*4 + ((r>>3)&1)*2.
 *               Padding rows / columns hold +0 and the neutral nibble 0x4.
 *               See DESIGN.md "Data layout in HBM"; pinned by tests/test_boundary.py. */
enum { SPFY_LAYOUT_CANONICAL = 0, SPFY_LAYOUT_SM100 = 1 };

enum { SPFY_OP_N = 0, SPFY_OP_T = 1 }; /* == cusparseOperation_t values */
/* OR-ed into the `opB` argument of spfy_spmma / spfy_spmma_problem: D is written TRANSPOSED, [n][m] row-major with pitch
 * ldd >= m -- for a convolution layer that is NHWC, what spfy_spmma_conv of the next layer reads.  beta must be 0 (except
 * in the _ex entry points, see spfy_epilogue) and m a multiple of 8 (the contiguous dimension of an output always is: n
 * for the row-major one). */
enum { SPFY_OUT_T = 0x10 };

enum {
  SPFY_OK = 0,
  SPFY_E_INVALID = -1,     /* bad argument */
  SPFY_E_UNSUPPORTED = -2, /* valid but not implemented for these arguments */
  SPFY_E_CUDA = -3,        /* CUDA runtime / driver error (see last error)   */
  SPFY_E_WORKSPACE = -4,   /* workspace too small                            */
  SPFY_E_NCCL = -5
};

SPFY_API int spfy_version(void);
/* Loads the library's device code on the current device (CUDA loads kernels lazily at first use, tens of
 * milliseconds for the large ones).  Optional and idempotent; the header templates call it before they start
 * their timers -- the counterpart of the handle / plan creation the reference keeps outside its timers
 * (spmma.hxx:51-80). */
SPFY_API int spfy_init(void);
SPFY_API const char* spfy_last_error_string(void);
/* number of kernels this library launched in this process (bench: gpu_launches) */
SPFY_API uint64_t spfy_launch_count(void);

/* Element-wise dtype conversion between F32 and F16/BF16 (round to nearest even), used by
 * the header templates when a driver instantiates spmma<float> (examples/spmma.cu:24). */
SPFY_API int spfy_convert(int src_dtype, int dst_dtype, const void* src, void* dst, size_t count,
                          spfy_stream_t stream);

/* ------------------------------------------------------------------------
 * A1  sparsifyme::sparsify<BLK_M,BLK_N>          include/sparsify.me/sparsify.hxx:24-82
 * Exact positional semantics of the reference: mask <- 1 (:71); then for each
 * of (m/blk_m)*(n/blk_n) linear blocks zero the first
 * floor(blk_m*blk_n*sparsity_factor) offsets of the sequence h + w*blk_n,
 * h outer / w inner (:53-65), in `weights` and in `mask`.  One fused kernel
 * replaces thrust::fill_n + thrust::transform.  Writes that the reference
 * would issue past m*n (BLK_N > BLK_M instantiations) are dropped.
 * `mask` is an array of m*n 64-bit words (std::size_t in the reference).
 * ---------------------------------------------------------------------- */
SPFY_API int spfy_prune_blocks_ref(int dtype, void* weights, uint64_t* mask,
                                   size_t m, size_t n, size_t blk_m, size_t blk_n,
                                   float sparsity_factor, spfy_stream_t stream);

/* ------------------------------------------------------------------------
 * A2+A3  cusparseLtSpMMAPrune / PruneCheck / CompressedSize / Compress
 *                                               include/sparsify.me/spmma.hxx:85-104
 * One bandwidth-bound kernel: reads `in` (rows x cols, row-major, leading
 * dimension ld_in elements) once and writes any subset of
 *   out_dense : the pruned dense matrix (may alias `in`: in-place like :86)
 *   comp_vals / meta : compressed operand in `layout`
 *   mask      : rows*cols 64-bit keep flags (1 = kept), API parity with A1
 * Null outputs are skipped.  dtype is SPFY_F16 or SPFY_BF16.
 * ---------------------------------------------------------------------- */
SPFY_API int spfy_compressed_bytes(int dtype, size_t rows, size_t cols, int layout,
                                   size_t* vals_bytes, size_t* meta_bytes);
SPFY_API int spfy_prune24(int dtype, int mode, int layout, const void* in, size_t ld_in,
                          void* out_dense, size_t ld_out, void* comp_vals, void* meta,
                          uint64_t* mask, size_t rows, size_t cols, spfy_stream_t stream);
/* Whole-model variant: prune+compress `count` matrices in as few launches as possible (one
 * per 96 matrices).  The per-layer weight matrices of datasets/ *.csv are <= 4.7 MB, so one
 * launch per layer is launch-latency-bound; this is the call the prune GB/s figure is quoted
 * on (mode STRIP_MAG).  TILE_MAG -- the algorithm the reference requests (spmma.hxx:86) --
 * needs out_dense per item (it may alias the input) and takes the one-pass prune + compress
 * kernel for every matrix with cols % 16 == 0 and 8-byte aligned rows; the others (k = 147)
 * go through spfy_prune24 one by one.  `items` is a HOST array; fields as in spfy_prune24
 * (null outputs are skipped). */
typedef struct spfy_prune24_item {
  const void* in;
  size_t ld_in;
  void* out_dense;
  size_t ld_out;
  void* comp_vals;
  void* meta;
  size_t rows, cols;
} spfy_prune24_item;
SPFY_API int spfy_prune24_batched(int dtype, int mode, int layout, const spfy_prune24_item* items,
                                  size_t count, spfy_stream_t stream);
/* A dense matrix obeys 2:4 along its rows iff *d_invalid == 0 afterwards
 * (same convention as cusparseLtSpMMAPruneCheck, spmma.hxx:88-94). */
SPFY_API int spfy_prune24_check(int dtype, const void* in, size_t ld_in, size_t rows,
                                size_t cols, int* d_invalid, spfy_stream_t stream);

/* ------------------------------------------------------------------------
 * 2:4 fine-tuning: the backward pass of a pruned layer and updates under a
 * fixed mask.  No cusparseLt counterpart (a cusparseLt user keeps the dense
 * pruned matrix and prunes and compresses its transpose again).
 *
 * spfy_transpose24 -- A: SM100-layout compressed operand of a rows x cols matrix
 * whose columns are `taps` blocks of cols / taps.  Writes the SM100-layout
 * compressed operand of A' [cols/taps] x [taps*rows]:
 *     A'[ci][t'*rows + r] = A[r][(taps-1-t')*cols/taps + ci]
 * taps = 1: A' = A^T (the data gradient of a Linear layer, dx = dy W, is spfy_spmma
 * of A' with opB = T | SPFY_OUT_T).  taps = kh*kw with A's K in (kh, kw, c) order
 * (spfy_permute_conv_weights): A' is the filter of the data-gradient convolution
 * of a stride-1 layer (taps reversed = kernel flipped in both directions, channels
 * in and out swapped), for spfy_spmma_conv* with pad' = kh - 1 - pad.
 * rows % 8 == 0 and (cols / taps) % 8 == 0, so every 4x4 block of A maps whole onto
 * a 4x4 block of A'.  The kept set comes from A's metadata, not from the values: an
 * A' group keeps the entries A's metadata keeps in that column of the block, with
 * A's stored bits (+-0 included).  When a group of A' does not get exactly two, the
 * mask is not transposable: *d_invalid is set to 1 and the output is unspecified.
 * d_invalid (optional, device int) is zeroed on the stream first; the call never
 * syncs.  Padding rows / columns of A' hold +0 and the neutral nibble 0x4 (the
 * output buffers need not be zeroed); A's padding is never read.  The output must
 * not overlap the input.  Applying the call twice with the same taps gives back
 * the original bytes.  Refusals: dtype not F16/BF16, rows / cols too large or
 * rows % 8, (cols / taps) % 8 (SPFY_E_UNSUPPORTED); taps == 0, cols % taps,
 * null or not 16-byte aligned buffers (SPFY_E_INVALID).
 * ---------------------------------------------------------------------- */
SPFY_API int spfy_transpose24(int dtype, const void* vals, const void* meta, size_t rows, size_t cols, size_t taps,
                              void* vals_t, void* meta_t, int* d_invalid, spfy_stream_t stream);
/* spfy_transpose24_conv -- the filter operands of a STRIDED convolution's data gradient.
 * A: the forward filter, SM100-layout compressed m x (kh*kw*c) in (kh, kw, c) order
 * (spfy_permute_conv_weights, then SPFY_PRUNE_TILE_TRANSPOSABLE).  The data gradient
 * of a stride-s layer splits by output phase (a, b) = (ih mod s, iw mod s).  In one
 * dimension phase a takes the taps T_a = {kh : (a + pad - kh) mod s == 0} in
 * descending order, and
 *     dx[s*i + a] = sum over kh in T_a of dy[i + (a + pad - kh)/s] * W[kh]
 * (dy outside the image counts as 0): a stride-1 correlation of dy.  For each phase
 * with taps in both dimensions, in (a, b) row-major order, the call writes the
 * SM100-layout compressed c x (|T_a|*|T_b|*m) operand
 *     A'_ab[ci][(th*|T_b| + tw)*m + r] = A[r][(kh(th)*kw + kw(tw))*c + ci]
 * (th, tw: positions in T_a, T_b).  The operands lie back to back in vals_t / meta_t,
 * each starting on a tile boundary: phase p at tile sum over earlier phases of
 * ceil(c/128) * ceil(|T_a|*|T_b|*m/128) (16384 value and 2048 metadata bytes per
 * tile); spfy_transpose24_conv_bytes gives the totals.  A phase with no taps gets no
 * operand (1x1 stride 2: three of the four).  For s = 1 the output is byte for byte
 * spfy_transpose24(taps = kh*kw).  With a TILE-transposable mask every tap's slice of
 * the transposed filter is a valid 2:4 operand, so any subset of taps is too: nothing
 * is pruned again.  Otherwise as spfy_transpose24: *d_invalid (optional) is zeroed and
 * set to 1 for a mask that is not transposable, padding is +0 with nibble 0x4, the
 * output buffers need not be zeroed, one launch, no sync.  Refusals: dtype not
 * F16/BF16, m % 8, c % 8, kh or kw > 16, pad > 8, stride > 8 (SPFY_E_UNSUPPORTED);
 * an empty dimension, null or not 16-byte aligned buffers (SPFY_E_INVALID). */
SPFY_API int spfy_transpose24_conv_bytes(int dtype, size_t m, size_t c, size_t kh, size_t kw, size_t stride, size_t pad,
                                         size_t* vals_bytes, size_t* meta_bytes);
SPFY_API int spfy_transpose24_conv(int dtype, const void* vals, const void* meta, size_t m, size_t c, size_t kh,
                                   size_t kw, size_t stride, size_t pad, void* vals_t, void* meta_t, int* d_invalid,
                                   spfy_stream_t stream);
/* spfy_recompress24 -- new values under a fixed mask.
 * in: dense rows x cols (F32, F16 or BF16, row-major, ld_in).  meta: SM100 metadata of
 * a compressed operand of that shape (read only).  comp_vals (may be NULL): that
 * operand's values, `dtype` (F16/BF16), rounded to nearest even from `in` at the kept
 * positions (the bits themselves when in_dtype == dtype); padding +0.  out_masked (may
 * be NULL, may alias in): `in` with every pruned position set to +0, in in's dtype,
 * leading dimension ld_out.  One pass: it refreshes the forward operand from an fp32
 * master after an optimizer step without moving the mask, projects a weight gradient
 * onto the mask, or re-masks the master in place. */
SPFY_API int spfy_recompress24(int in_dtype, const void* in, size_t ld_in, int dtype, size_t rows, size_t cols,
                               const void* meta, void* comp_vals, void* out_masked, size_t ld_out, spfy_stream_t stream);
/* spfy_optim24_step -- one optimizer step over a table of fp32 parameters, the
 * refresh of the 2:4 layers' compressed operands included.
 * algo SPFY_OPTIM_SGD follows torch's _multi_tensor_sgd, SPFY_OPTIM_ADAMW its
 * _multi_tensor_adam with decoupled weight decay (AdamW), operation by operation
 * in fp32; the hyperparameters of item i are groups[items[i].group].
 *   SGD:   g += wd*p;  buf = *first ? g : buf*momentum + (1-dampening)*g;
 *          g = nesterov ? g + momentum*buf : buf;  p -= lr*g
 *          (momentum == 0: no buffer, g is used as is; first: an optional device
 *          float, read and never written, so that a step skipped by found_inf
 *          leaves the first step pending -- the caller clears it once a step
 *          has been applied, e.g. by multiplying it by *found_inf)
 *   AdamW: p *= 1 - lr*wd;  m = lerp(m, g, 1-beta1);  v = v*beta2 + (1-beta2)*g*g;
 *          p -= lr/(1-beta1^t) * m / (sqrt(v)/sqrt(1-beta2^t) + eps)
 *          with t = *step, the item's step count for this step (a device float,
 *          already advanced; the call reads it and never writes it).
 * grad_scale (optional, device float): every gradient is divided by it.
 * found_inf (optional, device float): when *found_inf != 0 nothing is written
 * anywhere (torch.amp.GradScaler's skipped step).  Both are read on the device, so
 * a scaled step needs no host sync.
 * Dense item (meta == NULL): rows * cols contiguous fp32 elements of param, grad
 * and the state(s), updated elementwise (ld is not used).
 * 2:4 item (meta != NULL): param is the fp32 master, rows x cols with leading
 * dimension ld, grad and the states in the same layout; meta, vals: the SM100
 * compressed operand of that shape (`dtype` F16/BF16).  At the positions meta
 * keeps, param and state are updated; at the pruned positions +0 is written to
 * param and state, whatever the gradient holds there (NaN and Inf included).
 * vals receives the new master rounded to nearest even, byte for byte what
 * spfy_recompress24(F32, param, ..., comp_vals = vals) would write.  vals_t
 * (optional) receives byte for byte what spfy_transpose24_conv(vals, meta, rows,
 * cols/(kh*kw), kh, kw, stride, pad) writes from the new vals: kh = kw = stride = 1,
 * pad = 0 is spfy_transpose24(taps = 1), the W^T of a Linear layer.  meta and
 * meta_t are only read and not written (the mask is fixed), nor are the padding
 * bytes of vals and vals_t (they hold +0 since the operand was built).  Every
 * element of param and state is read once and written once, every element of grad
 * read once.  An item with rows * cols == 0 is skipped (its pointers may be NULL).
 * One launch takes up to 192 items and 16 groups (fewer items when the strided
 * convolutions among them bring more than 256 phases); larger tables take further
 * launches, in table order.  The call makes no device allocation, no copy and no
 * sync.
 * Refusals, before any launch: bad algo, null tables, a null param or grad, a
 * missing state (SGD with momentum: state1; AdamW: state1, state2 and step), fp32
 * buffers not 4-byte (dense) or 16-byte (2:4) aligned, SM100 buffers not 16-byte
 * aligned, ld < cols or ld % 4, a group out of range, negative lr or eps, nesterov
 * without momentum or with dampening (SPFY_E_INVALID); a 16-bit dtype other than
 * F16/BF16, rows or cols not multiples of 8, cols not kh*kw*c with c % 8 == 0, kh,
 * kw > 16, pad > 8, stride > 8, items too large (SPFY_E_UNSUPPORTED). */
enum { SPFY_OPTIM_SGD = 0, SPFY_OPTIM_ADAMW = 1 };
typedef struct spfy_optim24_item {
  float* param;
  const float* grad;
  float* state1;     /* SGD: momentum buffer (NULL when momentum == 0); AdamW: exp_avg */
  float* state2;     /* AdamW: exp_avg_sq */
  const float* step; /* AdamW: the step count of this step */
  const float* first; /* SGD (optional, device): nonzero -> torch's first step, buf = g */
  size_t rows, cols, ld;
  size_t group;      /* index into groups */
  int dtype;         /* 2:4 item: F16 / BF16 */
  const void* meta;  /* NULL: dense item */
  void* vals;
  void* vals_t;      /* optional */
  size_t kh, kw, stride, pad;  /* the convolution of vals_t */
} spfy_optim24_item;
typedef struct spfy_optim24_hparams {
  double lr, momentum, dampening, weight_decay; /* SGD: lr, momentum, dampening, weight_decay */
  double beta1, beta2, eps;                     /* AdamW: lr, betas, eps, weight_decay */
  int nesterov;
} spfy_optim24_hparams;
SPFY_API int spfy_optim24_step(int algo, const spfy_optim24_item* items, size_t count,
                               const spfy_optim24_hparams* groups, size_t n_groups, const float* grad_scale,
                               const float* found_inf, spfy_stream_t stream);

/* ------------------------------------------------------------------------
 * A4  cusparseLtMatmul                           include/sparsify.me/spmma.hxx:106-114
 * D = alpha * A(2:4) * op(B) + beta * C, fp32 accumulate on tcgen05.mma.sp.
 * A is the SM100-layout compressed operand of an m x k matrix (from
 * spfy_prune24).  All dense operands are row-major like the reference's
 * descriptors (:56-64): op(B) is k x n.  opB = N: B is k x n, ldb >= n;
 * opB = T: B is n x k, ldb >= k.  C and D are m x n; D may alias C.
 * n, ldb, ldc, ldd must be multiples of 8 elements and all base pointers
 * 16-byte aligned (the reference's own fp16 contract, spmma.hxx:45-49).
 * opB | SPFY_OUT_T: D is n x m (the transpose, pitch ldd >= m), beta must be 0, m % 8 == 0.
 * ---------------------------------------------------------------------- */
SPFY_API int spfy_spmma_workspace_bytes(int dtype, size_t m, size_t n, size_t k,
                                        size_t* bytes);
SPFY_API int spfy_spmma(int dtype, int opB, size_t m, size_t n, size_t k, float alpha,
                        const void* comp_vals, const void* meta, const void* B, size_t ldb,
                        float beta, const void* C, size_t ldc, void* D, size_t ldd,
                        void* workspace, size_t workspace_bytes, spfy_stream_t stream);

/* Implicit GEMM: the step BEFORE the path fused into it (SURVEY.md 8f N2).  The K x N operand of every CSV row
 * is the `unfold` of a convolution input (datasets/get_shapes.py:29-41 of the reference): a 3 x 3 layer reads each
 * activation nine times.  Here B is never materialised: X is the NHWC activation tensor [batch][h][w][c] and the
 * kernel's producer gathers each (128 positions x 64 channels) piece of a B stage with one TMA im2col instruction.
 *     D[m x N] = alpha * A(2:4)[m x K] * im2col(X)[K x N] + beta * C,   N = batch * ho * wo  (image, row, column),
 *     K = kh * kw * c ordered (kh, kw, c): permute the weight columns from PyTorch's (c, kh, kw) BEFORE pruning
 *     (spfy_permute_conv_weights), the 2:4 groups are formed along the new order.
 * c must be a multiple of 64 (every ResNet layer but the first; that one is unfolded explicitly), dilation 1.
 * D is row-major m x N like spfy_spmma (ldd % 8 == 0). */
typedef struct spfy_conv_desc {
  size_t batch, h, w, c; /* NHWC input */
  size_t kh, kw;         /* filter */
  size_t stride, pad;    /* same in both directions */
} spfy_conv_desc;
SPFY_API int spfy_spmma_conv(int dtype, const spfy_conv_desc* conv, size_t m, float alpha,
                             const void* comp_vals, const void* meta, const void* X, float beta,
                             const void* C, size_t ldc, void* D, size_t ldd, spfy_stream_t stream);
/* The same with the output in NHWC: Y[N][m] (pitch ldy >= m, ldy % 8 == 0), i.e. [batch][ho][wo][m] -- the X of the next
 * layer's spfy_spmma_conv, so a chain of convolutions never transposes or unfolds anything.  A unit's 128 positions x m
 * channels are then one contiguous run of Y instead of m rows 2 * N bytes apart.  beta = 0. */
SPFY_API int spfy_spmma_conv_nhwc(int dtype, const spfy_conv_desc* conv, size_t m, float alpha,
                                  const void* comp_vals, const void* meta, const void* X, void* Y, size_t ldy,
                                  spfy_stream_t stream);
/* Epilogue of the _ex entry points (cusparseLt's ALPHA_VECTOR_SCALING, BIAS_POINTER, ACTIVATION_RELU / _GELU): what
 * happens between two layers -- batch norm folded into a per-channel scale and bias, the activation, the shortcut add
 * of a residual block (beta * C) -- done on the accumulators, before the output is written once.  Per output element
 * (i, j), all in fp32, rounded to 16 bit once at the end:
 *     v = (alpha * scale[i]) * acc + beta * C + bias[i],   D = act(v)
 * alpha * scale[i] is formed once per row (exactly alpha when scale is NULL); the product with acc is rounded, then
 * beta * C is added with one fused multiply-add, then bias[i].  SPFY_ACT_GELU_TANH is the tanh form
 * 0.5 v (1 + tanh(sqrt(2/pi) (v + 0.044715 v^3))) -- torch's gelu(approximate="tanh"), cuBLASLt's and cusparseLt's
 * GELU -- with the hardware tanh approximation (relative error ~2^-11).  i is the output row of A: the output channel
 * of a convolution, the output feature of a Linear layer (y = x W^T + b is opB = T with B = x and SPFY_OUT_T).
 * scale / bias are device arrays of m floats, 4-byte aligned; NULL means 1 / 0.  A NULL epilogue pointer, or one with
 * both arrays NULL and SPFY_ACT_NONE, is the identity: the call computes exactly what the plain entry point does.
 * In the _ex entries beta != 0 is also allowed with SPFY_OUT_T: C then has D's layout, [n][m] with ldc >= m,
 * ldc % 8 == 0 and a 16-byte aligned base, and D may alias C (the shortcut add of a bottleneck block, in NHWC). */
enum { SPFY_ACT_NONE = 0, SPFY_ACT_RELU = 1, SPFY_ACT_GELU_TANH = 2 };
typedef struct spfy_epilogue {
  const float* scale; /* [m] device, per output row / channel; NULL = 1 */
  const float* bias;  /* [m] device; NULL = 0 */
  int act;            /* SPFY_ACT_* */
} spfy_epilogue;
/* spfy_spmma with an epilogue (NULL = identity) */
SPFY_API int spfy_spmma_ex(int dtype, int opB, size_t m, size_t n, size_t k, float alpha,
                           const void* comp_vals, const void* meta, const void* B, size_t ldb,
                           float beta, const void* C, size_t ldc, void* D, size_t ldd,
                           void* workspace, size_t workspace_bytes, const spfy_epilogue* epi,
                           spfy_stream_t stream);
/* spfy_spmma_conv / spfy_spmma_conv_nhwc with an epilogue: layout 0 writes D[m][N] (ldd >= N), SPFY_OUT_T writes NHWC
 * D[N][m] (ldd >= m); C, read when beta != 0, has D's layout. */
SPFY_API int spfy_spmma_conv_ex(int dtype, const spfy_conv_desc* conv, size_t m, float alpha,
                                const void* comp_vals, const void* meta, const void* X, float beta,
                                const void* C, size_t ldc, void* D, size_t ldd, int layout,
                                const spfy_epilogue* epi, spfy_stream_t stream);
/* spfy_spmma_conv_dgrad -- the data gradient of a convolution of any stride on sparse tensor cores:
 *     dX = alpha * conv2d_input(W, dY) + beta * dX
 * conv: the FORWARD layer (its h and w say which dX a floor-divided dY belongs to).  dY: NHWC [batch][ho][wo][m];
 * dX: NHWC [batch][h][w][c], contiguous.  vals_t / meta_t: spfy_transpose24_conv of the layer's m x (kh*kw*c) filter.
 * Each phase (a, b) with taps is one implicit GEMM, M = c, K = |T_a|*|T_b|*m, N = batch * H_a * W_b (H_a = ceil((h -
 * a) / s)), whose im2col map walks dY with stride 1 from the phase's first offset, and whose NHWC output rows land on
 * the pixels (s*i + a, s*j + b) of dX.  Every dX element is written: positions no tap reaches get beta * dX (+0 for beta
 * = 0, nothing at all is written for beta = 1).  beta = 1 accumulates in place, e.g. where the shortcut's and the main
 * branch's data gradients meet at a residual block's input.  A phase is one launch (the launches of one call may
 * overlap: they write disjoint pixels); no device allocation, no sync.  Refusals: dtype not F16/BF16, m % 64, c % 8,
 * kh or kw > 16, pad > 8, stride > 8, im2col corners of a phase outside [-128, 127] (SPFY_E_UNSUPPORTED); an empty
 * dimension, a filter larger than the padded image, null or not 16-byte aligned buffers (SPFY_E_INVALID). */
SPFY_API int spfy_spmma_conv_dgrad(int dtype, const spfy_conv_desc* conv, size_t m, float alpha, const void* vals_t,
                                   const void* meta_t, const void* dY, float beta, void* dX, spfy_stream_t stream);
/* spfy_conv_wgrad24 -- the weight gradient of a 2:4 convolution, fp32, masked to the layer's pattern:
 *     dW = alpha * mask(conv2d_weight(X, dY)) + beta * dW
 * conv: the FORWARD layer.  X: NHWC [batch][h][w][c] (F16/BF16); dY: NHWC [batch][ho][wo][m], same dtype.  meta: SM100
 * metadata of the layer's compressed m x (kh*kw*c) filter in (kh, kw, c) order (spfy_permute_conv_weights, then
 * spfy_prune24).  dW: fp32 [m][kh*kw*c] row-major in (kh, kw, c) order -- the storage of a channels_last [m][c][kh][kw]
 * weight.  Positions the metadata prunes are written +0 whatever alpha, beta and dW held; dW is not read when beta = 0.
 * The contraction runs on tcgen05 (kind::f16, fp32 accumulators) with M = kh*kw*c, N = m and K = P = batch*ho*wo output
 * positions, K split into S ranges of k_tiles stages of 64 positions; each split writes an fp32 partial to the
 * workspace, and a second pass sums the partials in ascending split order, applies alpha, beta and the mask.  No atomics:
 * the same inputs give the same bits.  S depends on the shape alone:
 *     tiles   = ceil(kh*kw*c / 128) * ceil(m / 256),   stages = ceil(P / 64)
 *     S0      = max(1, min(floor(148 / tiles), floor(stages / 8)))
 *     k_tiles = ceil(stages / S0),   S = ceil(stages / k_tiles)
 * (one wave of units on the 148 SMs of a B200, at least 8 stages a unit), and the workspace is S * m * kh*kw*c * 4 bytes;
 * the query needs no device.  Two launches, no device allocation, no sync.  Refusals, before any launch: dtype not
 * F16/BF16, c % 64, m % 8, kh or kw > 16, pad > 8, stride > 8 (SPFY_E_UNSUPPORTED); an empty dimension, a filter larger
 * than the padded image, null or not 16-byte aligned buffers (SPFY_E_INVALID); a workspace smaller than the query
 * (SPFY_E_WORKSPACE). */
SPFY_API int spfy_conv_wgrad24_workspace_bytes(int dtype, const spfy_conv_desc* conv, size_t m, size_t* bytes);
SPFY_API int spfy_conv_wgrad24(int dtype, const spfy_conv_desc* conv, size_t m, float alpha, const void* X,
                               const void* dY, const void* meta, float beta, float* dW,
                               void* workspace, size_t workspace_bytes, spfy_stream_t stream);
/* weights [m][c * kh * kw] in (c, kh, kw) column order (what torch's unfold / a flattened conv weight uses)
 * -> [m][kh * kw * c] in (kh, kw, c) order; 16-bit elements */
SPFY_API int spfy_permute_conv_weights(const void* in, void* out, size_t m, size_t c, size_t kh, size_t kw,
                                       spfy_stream_t stream);

/* Many independent problems (the per-layer GEMMs of a datasets/ *.csv table) as ONE plan:
 * tensor maps and the tile schedule are built once (like cusparseLtMatmulPlanInit,
 * spmma.hxx:79, which the reference also keeps outside its timers) and every run issues at
 * most one persistent launch per ring-geometry class (six) and operand orientation that walk all problems' tiles, so neither launch latency
 * nor per-layer wave quantisation is paid per layer.  Problems must not alias each other's
 * outputs.  plan_create allocates a small device table; plan_run never allocates or syncs. */
typedef struct spfy_spmma_problem {
  int opB;                 /* SPFY_OP_N / SPFY_OP_T */
  size_t m, n, k;
  const void* comp_vals;   /* SM100-layout compressed A (spfy_prune24) */
  const void* meta;
  const void* B;
  size_t ldb;
  const void* C;           /* may be null when beta == 0 */
  size_t ldc;
  void* D;
  size_t ldd;
  float alpha, beta;
} spfy_spmma_problem;
typedef struct spfy_spmma_plan_st* spfy_spmma_plan_t;
SPFY_API int spfy_spmma_plan_create(int dtype, const spfy_spmma_problem* problems, size_t count,
                                    spfy_spmma_plan_t* plan);
/* Replicated outputs -- the fused form of the output gather (north_star: the path's only exchange).  Every D tile of
 * problem i is stored, by the same TMA store that writes problems[i].D, to `replicas` further matrices
 * replica_D[i * replicas + r] of the same shape and ldd.  With one process per GPU these are this rank's slab of the
 * gather arena in every PEER GPU's memory (spfy_peer_open mappings, reached over NVLink): the GEMM epilogue is then
 * the all-gather, tile by tile, and no collective follows -- only a barrier among the ranks before anyone reads
 * (completion of the launch on rank r makes rank r's stores visible; it says nothing about the other ranks').
 * replicas <= 15; replica pointers 16-byte aligned; beta != 0 still reads problems[i].C only. */
SPFY_API int spfy_spmma_plan_create_replicated(int dtype, const spfy_spmma_problem* problems, size_t count,
                                               size_t replicas, void* const* replica_D, spfy_spmma_plan_t* plan);
/* A plan whose problems may be convolution layers (a whole network's table with the 3 x 3 layers never unfolded):
 * convs[i] != NULL makes problem i the implicit GEMM of spfy_spmma_conv -- problems[i].B is then the NHWC activation
 * tensor X, n / k follow from the descriptor (problems[i].n, .k, .ldb and the transpose bits of .opB are ignored;
 * SPFY_OUT_T in .opB still selects the NHWC output of spfy_spmma_conv_nhwc), comp_vals / meta hold the weights with K in
 * (kh, kw, c) order.  convs == NULL or convs[i] == NULL: as spfy_spmma_plan_create.  Descriptors are read at creation
 * only.  Results are bitwise those of the single calls. */
SPFY_API int spfy_spmma_plan_create_conv(int dtype, const spfy_spmma_problem* problems,
                                         const spfy_conv_desc* const* convs, size_t count, spfy_spmma_plan_t* plan);
/* A plan with epilogues: as spfy_spmma_plan_create_conv (convs may be NULL), plus epilogues[i] for problem i (the array
 * and its entries may be NULL; read at creation only).  Same launches as without epilogues; every output is bitwise
 * that of the single _ex call. */
SPFY_API int spfy_spmma_plan_create_ex(int dtype, const spfy_spmma_problem* problems,
                                       const spfy_conv_desc* const* convs, const spfy_epilogue* const* epilogues,
                                       size_t count, spfy_spmma_plan_t* plan);
SPFY_API int spfy_spmma_plan_run(spfy_spmma_plan_t plan, spfy_stream_t stream);
SPFY_API int spfy_spmma_plan_launches(spfy_spmma_plan_t plan); /* kernel launches per run */
/* introspection / profiling: run one of the plan's launches, or describe it */
SPFY_API int spfy_spmma_plan_run_launch(spfy_spmma_plan_t plan, int index, spfy_stream_t stream);
SPFY_API int spfy_spmma_plan_launch_info(spfy_spmma_plan_t plan, int index, int* problems, int* units,
                                         int* stages, int* smem_bytes);
SPFY_API int spfy_spmma_plan_destroy(spfy_spmma_plan_t plan);

/* ------------------------------------------------------------------------
 * Pruned-layer container (SURVEY.md 8f N4: the artifact that follows prune + compress).
 * One self-describing HOST buffer per compressed 2:4 operand:
 *   64-byte header {magic "SPFY24\0\0", version, dtype, layout, rows, cols, vals_bytes,
 *   meta_bytes, FNV-1a 64 of the payload} + values + metadata, as spfy_prune24 wrote them
 * (copy them to the host first; these calls touch host memory only, no CUDA).  A reader
 * checks magic / version / sizes against spfy_compressed_bytes and the checksum, then
 * hands back offsets into the buffer, so the payload can go to the device with two copies
 * and be used by spfy_spmma as is.
 * ---------------------------------------------------------------------- */
#define SPFY_PACKED_HEADER_BYTES 64
SPFY_API int spfy_packed_bytes(int dtype, size_t rows, size_t cols, int layout, size_t* bytes);
SPFY_API int spfy_packed_write(int dtype, int layout, size_t rows, size_t cols,
                               const void* host_vals, const void* host_meta, void* dst,
                               size_t dst_bytes);
SPFY_API int spfy_packed_read(const void* src, size_t src_bytes, int* dtype, int* layout,
                              size_t* rows, size_t* cols, size_t* vals_offset,
                              size_t* vals_bytes, size_t* meta_offset, size_t* meta_bytes);

/* ------------------------------------------------------------------------
 * Unstructured path (north_star subsystem 3).  Threshold prune keeps x iff
 * |x| > threshold (compared in fp32) and emits COO sorted by (row, col) or CSR.
 * dtype of `in` is F16/BF16/F32; emitted values are fp32 like the reference's
 * CUDA_R_32F COO (include/sparsify.me/spmm.hxx:165-168).
 * nnz is produced on the device (`d_nnz`, one int64) so the call never syncs.
 * `capacity` bounds the number of entries written.  `d_row_ptr_or_null`
 * (rows+1 int32), when given, receives the CSR row pointer of the same entries.
 * One pass over the input: one memset of the workspace (8 bytes per 4096
 * elements, size from the query; must be 8-byte aligned) + one kernel.
 * rows * cols must be below 2^31.
 * ---------------------------------------------------------------------- */
SPFY_API int spfy_threshold_workspace_bytes(size_t rows, size_t cols, size_t* bytes);
SPFY_API int spfy_threshold_to_coo(int dtype, const void* in, size_t ld_in, size_t rows,
                                   size_t cols, float threshold, int32_t* row_idx,
                                   int32_t* col_idx, float* vals, size_t capacity,
                                   int64_t* d_nnz, int32_t* d_row_ptr_or_null,
                                   void* workspace, size_t workspace_bytes,
                                   spfy_stream_t stream);
/* COO (sorted by row) -> CSR row pointer (rows+1 int32). */
SPFY_API int spfy_coo_to_csr(const int32_t* row_idx, size_t nnz, size_t rows,
                             int32_t* row_ptr, spfy_stream_t stream);

/* ------------------------------------------------------------------------
 * Algorithm of the unstructured SpMM entry points below (first argument).
 *   DEFAULT     : the library chooses.  An A with at least 2 % non-zeros (every pruned ResNet
 *                 weight matrix: 5-50 %) is scattered into a dense matrix in the workspace and
 *                 contracted on tcgen05 (fp32 operands: 3xTF32, fp32-level accuracy, see
 *                 spfy_gemm_*; 16-bit operands: kind::f16) when the operands meet the TMA
 *                 contract (16-byte aligned bases, leading dimensions and batch strides
 *                 multiples of 16 bytes); otherwise, and for sparser A, the CUDA-core kernels run.
 *                 The CSR entry does not know nnz on the host: it launches both candidates and
 *                 a device flag lets exactly one do the work, so it never reads anything back.
 *   CUDA_CORE   : the row-split CUDA-core kernels only.  fp32 sums in ascending k order per
 *                 output element: bit-identical to cuSPARSE 12.5 on exactly representable
 *                 inputs (tests/golden/cusparse_*.npz).
 *   TENSOR      : the tensor-core route or SPFY_E_UNSUPPORTED / SPFY_E_WORKSPACE.
 *   TENSOR_FAST : same with ONE TF32 product per fp32 multiply (10-bit mantissas; the accuracy
 *                 class of cuBLAS's TF32 mode).  16-bit operands: identical to TENSOR.
 * Special values (fp32).  Finite values and their products are handled as by spfy_gemm_* (below)
 * on the tensor-core routes and in IEEE fp32 on the CUDA-core kernels.  Inf and NaN in B follow
 * one of two semantics, by kernel:
 *   stored entries : only the stored entries of A are multiplied (cuSPARSE's semantics), so a
 *                    non-finite B[kk][j] reaches only the rows of C_b that store an entry in
 *                    column kk; IEEE classes (Inf * 0 = NaN for a stored zero).  The per-non-zero
 *                    CUDA-core kernels: CUDA_CORE below 35 % non-zeros and DEFAULT below its
 *                    tensor threshold (CSR, COO), and the blocked-ELL CUDA-core kernel (padding
 *                    ids < 0 store nothing; a stored block multiplies all of its values).
 *   dense image    : A is multiplied as a dense matrix whose structural zeros are real zeros,
 *                    and 0 * Inf = NaN, so a non-finite B[kk][j] makes all of column j of C_b
 *                    non-finite (NaN in the rows that do not store column kk).  Every
 *                    tensor-core route (TENSOR, TENSOR_FAST, DEFAULT from 2 % non-zeros for CSR /
 *                    COO -- 20 % when B needs the padded copy, ldb = k = 147 --, DEFAULT for
 *                    blocked-ELL) and the CUDA-core dense walk (CUDA_CORE from 35 %).
 *                    Blocked-ELL exceptions: a batch chunk in which some block-row repeats an
 *                    id, and DEFAULT without a tensor route (e.g. a workspace sized for
 *                    CUDA_CORE), run on the blocked-ELL CUDA-core kernel: stored entries, IEEE.
 * So DEFAULT switches between the two with the density of A.  Classes of the non-finite outputs:
 * IEEE on the CUDA-core kernels; NaN on TENSOR (and DEFAULT on the tensor route), as PRECISE;
 * on TENSOR_FAST those of SPFY_GEMM_FAST, except that the image of a CSR / COO A is built by fp32
 * additions of the stored values, so a NaN in A stays NaN.  beta = 0: C is written, never read
 * (a NaN in C does not survive), on every route.
 * ---------------------------------------------------------------------- */
enum {
  SPFY_SPMM_ALG_DEFAULT = 0,
  SPFY_SPMM_ALG_CUDA_CORE = 1,
  SPFY_SPMM_ALG_TENSOR = 2,
  SPFY_SPMM_ALG_TENSOR_FAST = 3
};

/* ------------------------------------------------------------------------
 * A6  sparsifyme::batched::strided_coo           include/sparsify.me/spmm.hxx:140-193
 * C_b = alpha * A * B_b + beta * C_b for b in [0, num_batches): ONE sparse A
 * (stride 0, :169) shared by all batches; B_b = B + b*strideB is k x n
 * column-major (ldb >= k, :160,:170); C_b = C + b*strideC is m x n column-major
 * (ldc >= m, :161,:173).  fp32 values, int32 indices, fp32 accumulate.
 * The COO triplets must be sorted by row (any column order; repeated (row, col)
 * entries add, like cuSPARSE); row_ptr is built internally in the workspace.
 * The workspace query takes the algorithm and the batch extent: the tensor-core route keeps
 * the dense m x k fp32 image of A there and, when ldb = k is not a multiple of 16 bytes
 * (k = 147), a padded copy of every B_b (a workspace sized for CUDA_CORE makes DEFAULT
 * take the CUDA-core kernels).
 * ---------------------------------------------------------------------- */
SPFY_API int spfy_spmm_workspace_bytes(int alg, size_t m, size_t k, size_t n, size_t num_batches,
                                       size_t nnz, size_t* bytes);
SPFY_API int spfy_spmm_coo_strided_batched(int alg, size_t m, size_t k, size_t nnz, size_t n,
                                           size_t num_batches, const int32_t* row_idx,
                                           const int32_t* col_idx, const float* vals,
                                           const float* B, size_t ldb, size_t strideB,
                                           float* C, size_t ldc, size_t strideC, float alpha,
                                           float beta, void* workspace, size_t workspace_bytes,
                                           spfy_stream_t stream);
/* Same product with A already in CSR (same workspace query). */
SPFY_API int spfy_spmm_csr_strided_batched(int alg, size_t m, size_t k, size_t n,
                                           size_t num_batches, const int32_t* row_ptr,
                                           const int32_t* col_idx, const float* vals,
                                           const float* B, size_t ldb, size_t strideB, float* C,
                                           size_t ldc, size_t strideC, float alpha, float beta,
                                           void* workspace, size_t workspace_bytes,
                                           spfy_stream_t stream);

/* ------------------------------------------------------------------------
 * A5  sparsifyme::batched::spmm (blocked-ELL)    include/sparsify.me/spmm.hxx:30-138
 * For each batch b: C_b = alpha * A_b * B + beta * C_b.  A_b is blocked-ELL
 * (containers/ell.hxx:24-33): rows x cols, square blocks of `block`,
 * `ell_cols` stored columns per row; col_idx_b[(rows/block) x (ell_cols/block)]
 * block-column ids (int64 here because the reference stores std::size_t,
 * ell.hxx:31; ids < 0 are padding); values_b[rows x ell_cols] row-major.  B is
 * k x n column-major ldb = k shared by all batches (:67); C_b is m x n
 * column-major ldc = m (:63).  `col_idx`, `values`, `Cs` are DEVICE arrays of
 * num_batches device pointers.  dtype is that of values/B/C (F16/BF16/F32);
 * fp32 accumulate (:82).
 * Tensor-core route (DEFAULT when the operands meet the TMA contract): the batch is
 * expanded chunk by chunk into dense row-major matrices in the workspace (every
 * element written once, no atomics) and contracted by the dense tcgen05 GEMM; a
 * block-row that repeats an id (undefined for cuSPARSE; our kernels add the blocks)
 * raises a device flag that hands its chunk to the CUDA-core kernel instead.
 * ---------------------------------------------------------------------- */
SPFY_API int spfy_spmm_bell_workspace_bytes(int alg, int dtype, size_t rows, size_t cols, size_t n,
                                            size_t num_batches, size_t* bytes);
SPFY_API int spfy_spmm_bell_batched(int alg, int dtype, size_t rows, size_t cols, size_t n,
                                    size_t block, size_t ell_cols, size_t num_batches,
                                    const int64_t* const* col_idx, const void* const* values,
                                    const void* B, size_t ldb, void* const* Cs, size_t ldc,
                                    float alpha, float beta, void* workspace,
                                    size_t workspace_bytes, spfy_stream_t stream);

/* ------------------------------------------------------------------------
 * N3  sparsifyme::batched::gemm                  include/sparsify.me/gemm.hxx:25-195
 * Dense batched GEMM on tcgen05 (replaces cublas{H,S}gemmBatched, :51-186), BLAS
 * conventions: column-major, C_b[m x n, ldc] = alpha * op(A_b)[m x k] * op(B_b)[k x n]
 * + beta * C_b.  opX = N: the operand is stored as its op() shape; T: transposed.
 * dtype F16 / BF16: kind::f16, fp32 accumulation in TMEM.  dtype F32:
 *   SPFY_GEMM_PRECISE  3xTF32 -- each operand is split into hi (the 11 significant bits
 *                      the tensor core reads) and lo = x - hi, and hi*lo + lo*hi + hi*hi is
 *                      accumulated in fp32: products exact to ~2^-19.  The long, streamed
 *                      operand is split in registers into tensor memory (hi rounded to
 *                      nearest); the other keeps its raw tile in shared memory as hi (the
 *                      tensor core truncates it) with lo written behind it;
 *   SPFY_GEMM_FAST     one TF32 product.
 * Special values.  beta = 0: C is written, never read (a NaN in C does not survive).  Finite
 * operands whose products and sums stay inside the fp32 range give finite results, except that
 * PRECISE: the streamed operand's hi is rounded to nearest, the other's truncated.  A finite
 * value of the streamed operand with |x| >= 0x7f7ff000 (3.4020e38, the top 2^-11 of the fp32
 * range) rounds to hi = ±Inf, lo = ∓Inf: every output it reaches (its whole row or column of
 * C) is NaN.  In the other operand such values give finite, accurate results.  The streamed
 * operand is op(A) when the kernel maps m onto its 128-row tiles, op(B) when it maps n there
 * (orient() in gemm_sm100.cu: the mapping that issues fewer padded MACs, ties to the larger of
 * m and n); the SpMM tensor routes call it with op(A) = the dense image of A, row-major, and
 * for CSR / COO with n = n * num_batches (the batches of B side by side).
 * Non-finite operands, per mode:
 *   F16 / BF16         IEEE: Inf * finite nonzero = ±Inf, Inf * 0 = NaN, Inf - Inf = NaN, NaN
 *                      stays NaN.
 *   SPFY_GEMM_FAST     IEEE on the operands as the tensor core reads them, truncated to TF32: a
 *                      NaN whose payload lies only in the low 13 mantissa bits reads as ±Inf.
 *   SPFY_GEMM_PRECISE  an Inf or NaN operand splits into hi = ±Inf / NaN and lo = NaN, so every
 *                      output it reaches (row i of C for A[i][kk], column j for B[kk][j]) is
 *                      NaN, also where IEEE gives ±Inf.  Other outputs are unaffected.
 * With non-finite operands (and finite ones below 0x7f7ff000), in every mode an output is
 * non-finite exactly where the IEEE result is.
 * Any other `precision` is refused with SPFY_E_INVALID before any device work, for every dtype.
 * The operands are fetched by TMA, which needs 16-byte aligned bases and lda / ldb /
 * batch strides that are multiples of 16 bytes; an operand that misses this (ldb = k = 147
 * floats, the first conv layer of every ResNet) is first copied into the workspace with
 * padded rows -- one extra pass over that operand, nothing else changes.  The batched form
 * takes HOST arrays of device pointers (what examples/gemm.cu:93-95 holds are device
 * arrays -- the header copies them back once, outside its timer).  Both forms take a
 * device workspace sized by the query (problem table of the batched form + padded copies
 * of the operands whose lda / ldb need them; pass lda = 0 / ldb = 0 to size for a
 * misaligned base pointer as well).
 * ---------------------------------------------------------------------- */
enum { SPFY_GEMM_PRECISE = 0, SPFY_GEMM_FAST = 1 };
SPFY_API int spfy_gemm_workspace_bytes(int dtype, int opA, int opB, size_t m, size_t n, size_t k,
                                       size_t lda, size_t ldb, size_t num_batches, size_t* bytes);
SPFY_API int spfy_gemm_strided_batched(int dtype, int precision, int opA, int opB, size_t m, size_t n,
                                       size_t k, float alpha, const void* A, size_t lda,
                                       size_t strideA, const void* B, size_t ldb, size_t strideB,
                                       float beta, void* C, size_t ldc, size_t strideC,
                                       size_t num_batches, void* workspace, size_t workspace_bytes,
                                       spfy_stream_t stream);
SPFY_API int spfy_gemm_batched(int dtype, int precision, int opA, int opB, size_t m, size_t n, size_t k,
                               float alpha, const void* const* A_ptrs, size_t lda,
                               const void* const* B_ptrs, size_t ldb, float beta,
                               void* const* C_ptrs, size_t ldc, size_t num_batches,
                               void* workspace, size_t workspace_bytes, spfy_stream_t stream);

/* ------------------------------------------------------------------------
 * Multi-GPU (SURVEY.md 8e): the per-layer problems and, inside one GEMM, the N = batch x
 * spatial columns are independent, so the path shards with NO exchange during compute;
 * the only collective is a gather of outputs (north_star).  The reference has no
 * multi-GPU code (examples/spmma.cu:27-28 queries device 0 only).  One process per GPU.
 * NCCL is loaded at run time (libnccl.so.2, or the path in SPFY_NCCL_LIB): without it these
 * calls return SPFY_E_NCCL and nothing else in the library is affected.
 *   bootstrap : rank 0 calls spfy_mg_unique_id (128 bytes), the host program hands the
 *               bytes to every rank (torch.distributed, MPI, a file ...), all call
 *               spfy_mg_create with the current device set.
 *   allgather : N-sharded GEMMs.  Rank r holds D_r [M x N/g] row-major (its images' columns);
 *               the gathered result is [g][M][N/g] -- the ranks' slabs back to back.  In
 *               place when `send` == `recv` + r * bytes_per_rank: let the GEMM write D_r
 *               there and no copy is made at all.
 *   broadcast_many : layer sharding.  Entry i is sent from rank roots[i] to everybody, all
 *               entries as ONE NCCL group (the lists are HOST arrays).
 * All work is enqueued on the caller's stream.
 * ---------------------------------------------------------------------- */
/* Peer memory for the fused gather (spfy_spmma_plan_create_replicated): device memory another process on the same box
 * can map.  spfy_peer_alloc = cudaMalloc + cudaIpcGetMemHandle (the 64 handle bytes travel through the host program,
 * like the NCCL id); spfy_peer_open = cudaIpcOpenMemHandle with lazy peer access, in a DIFFERENT process than the
 * owner; the mapping is an ordinary device pointer for every entry point of this library. */
#define SPFY_PEER_HANDLE_BYTES 64
SPFY_API int spfy_peer_alloc(size_t bytes, void** ptr, void* handle64);
SPFY_API int spfy_peer_free(void* ptr);
SPFY_API int spfy_peer_open(const void* handle64, void** ptr);
SPFY_API int spfy_peer_close(void* ptr);

typedef struct spfy_mg_comm_st* spfy_mg_comm_t;
SPFY_API int spfy_mg_unique_id(void* id128);
SPFY_API int spfy_mg_create(int rank, int world, const void* id128, spfy_mg_comm_t* comm);
SPFY_API int spfy_mg_destroy(spfy_mg_comm_t comm);
SPFY_API int spfy_mg_rank(spfy_mg_comm_t comm);
SPFY_API int spfy_mg_world(spfy_mg_comm_t comm);
SPFY_API int spfy_mg_allgather(spfy_mg_comm_t comm, const void* send, void* recv, size_t bytes_per_rank,
                               spfy_stream_t stream);
SPFY_API int spfy_mg_broadcast_many(spfy_mg_comm_t comm, void* const* buffers, const size_t* bytes,
                                    const int* roots, size_t count, spfy_stream_t stream);

#ifdef __cplusplus
}
#endif
#endif /* SPFY_B200_H_ */
