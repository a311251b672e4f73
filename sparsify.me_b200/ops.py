"""Host-side mirror of the reference's operator API on top of the C ABI (capi).

Names, argument meaning, defaults and return values follow the reference templates:
  sparsify            include/sparsify.me/sparsify.hxx:24-30  (weights, mask, m, n, sparsity_factor=0.5, stream)
  spmma               include/sparsify.me/spmma.hxx:21-33     -> [prune_ms, compress_ms, mul_ms] (:117)
  batched.spmm        include/sparsify.me/spmm.hxx:30-41      -> ms
  batched.strided_coo include/sparsify.me/spmm.hxx:140-153    -> ms
Tensors are torch CUDA tensors used as raw device buffers; all work is enqueued on torch's
current stream.  Nothing here computes on the host.
"""
import ctypes
import sys
import weakref
from dataclasses import dataclass

import torch

from . import capi

_DT = {torch.float16: capi.F16, torch.bfloat16: capi.BF16, torch.float32: capi.F32,
       torch.float64: capi.F64}


def _dtype_code(t):
    try:
        return _DT[t.dtype]
    except KeyError:
        raise capi.SpfyError(capi.E_UNSUPPORTED, "dtype", f"unsupported dtype {t.dtype}")


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)


def _ptr(t):
    if t is None:
        return None
    if not t.is_cuda:
        raise capi.SpfyError(capi.E_INVALID, "device pointer",
                             "operand is not a CUDA tensor (sparsify.me_b200 has no host path)")
    return ctypes.c_void_p(t.data_ptr())


def _workspace(nbytes, device):
    """caller-provided scratch for one call (256-byte aligned like every torch allocation)"""
    return torch.empty(max(int(nbytes), 16), dtype=torch.uint8, device=device)


class _Timer:
    """cudaEvent pair on the current stream -- the reference's util::timer_t
    (include/sparsify.me/util/timer.hxx:24-55): begin/end record + synchronise."""

    def __init__(self):
        self.a = torch.cuda.Event(enable_timing=True)
        self.b = torch.cuda.Event(enable_timing=True)

    def begin(self):
        self.a.record()

    def end(self):
        self.b.record()
        self.b.synchronize()
        return self.a.elapsed_time(self.b)


# ----------------------------------------------------------------------------- A1
def sparsify(weights, mask, m, n, sparsity_factor=0.5, blk=(2, 2)):
    """sparsifyme::sparsify<BLK_M,BLK_N> (sparsify.hxx:24-82), exact positional semantics.
    `weights`: m*n elements (any 2/4/8-byte float type), pruned in place;
    `mask`: m*n int64/uint64 words (std::size_t in the reference)."""
    if mask.element_size() != 8:
        raise capi.SpfyError(capi.E_INVALID, "sparsify", "mask must hold 64-bit words")
    capi.spfy_prune_blocks_ref(_dtype_code(weights), _ptr(weights), _ptr(mask), m, n, blk[0], blk[1],
                               float(sparsity_factor), _stream())


# ------------------------------------------------------------------------- A2 / A3
@dataclass
class Compressed24:
    """The compressed 2:4 operand (what cusparseLtSpMMACompress returns, spmma.hxx:97-104)."""
    vals: torch.Tensor      # uint8 buffer
    meta: torch.Tensor      # uint8 buffer
    rows: int
    cols: int
    dtype: torch.dtype
    layout: int


def compressed_bytes(dtype, rows, cols, layout=capi.LAYOUT_SM100):
    vb, mb = ctypes.c_size_t(), ctypes.c_size_t()
    capi.spfy_compressed_bytes(_DT[dtype], rows, cols, layout, ctypes.byref(vb), ctypes.byref(mb))
    return vb.value, mb.value


def prune24(a, out_dense=None, mask=None, layout=capi.LAYOUT_SM100, mode=capi.PRUNE_STRIP_MAG,
            compress=True, inplace=False, out=None):
    """2:4 magnitude prune (+ compress) of the row-major matrix `a` [rows, cols] in ONE kernel.
    Replaces cusparseLtSpMMAPrune + cusparseLtSpMMACompress (spmma.hxx:85-104).
    Returns a Compressed24 (or None when compress=False)."""
    assert a.dim() == 2 and a.stride(1) == 1
    rows, cols = a.shape
    if inplace:
        out_dense = a
    comp = out
    if compress and comp is None:
        vb, mb = compressed_bytes(a.dtype, rows, cols, layout)
        comp = Compressed24(torch.empty(vb, dtype=torch.uint8, device=a.device),
                            torch.empty(mb, dtype=torch.uint8, device=a.device), rows, cols, a.dtype,
                            layout)
    capi.spfy_prune24(_dtype_code(a), mode, layout, _ptr(a), a.stride(0), _ptr(out_dense),
                      out_dense.stride(0) if out_dense is not None else 0,
                      _ptr(comp.vals) if comp else None, _ptr(comp.meta) if comp else None,
                      _ptr(mask), rows, cols, _stream())
    return comp


def prune24_check(a):
    """cusparseLtSpMMAPruneCheck (spmma.hxx:88-94): 0 iff `a` obeys 2:4 along its rows."""
    flag = torch.empty(1, dtype=torch.int32, device=a.device)
    capi.spfy_prune24_check(_dtype_code(a), _ptr(a), a.stride(0), a.shape[0], a.shape[1], _ptr(flag),
                            _stream())
    return int(flag.item())


def prune24_batched(mats, comps, layout=capi.LAYOUT_SM100, mode=capi.PRUNE_STRIP_MAG, inplace=False):
    """Prune+compress a whole list of weight matrices with as few launches as possible
    (spfy_prune24_batched).  `mats`: 2-D row-major tensors; `comps`: matching Compressed24.
    mode=PRUNE_TILE_MAG (what the reference asks cusparseLt for, spmma.hxx:86) prunes the matrices IN PLACE
    like cusparseLtSpMMAPrune(dA, dA) -- TILE needs the dense pruned matrix as an output; `inplace` asks for the
    same with STRIP."""
    items = (capi.Prune24Item * len(mats))()
    dense = inplace or mode == capi.PRUNE_TILE_MAG
    for i, (a, c) in enumerate(zip(mats, comps)):
        items[i] = capi.Prune24Item(a.data_ptr(), a.stride(0), a.data_ptr() if dense else None, a.stride(0) if dense else 0,
                                    c.vals.data_ptr(), c.meta.data_ptr(), a.shape[0], a.shape[1])
    capi.spfy_prune24_batched(_dtype_code(mats[0]), mode, layout, ctypes.cast(items, ctypes.c_void_p), len(mats),
                              _stream())


def alloc_compressed(dtype, rows, cols, device, layout=capi.LAYOUT_SM100):
    vb, mb = compressed_bytes(dtype, rows, cols, layout)
    return Compressed24(torch.empty(vb, dtype=torch.uint8, device=device),
                        torch.empty(mb, dtype=torch.uint8, device=device), rows, cols, dtype, layout)


def pack_compressed(comp):
    """Compressed24 -> one self-describing host buffer (bytes): the pruned-layer container of spfy_b200.h
    (header + values + metadata, checksummed).  The payload is the device image byte for byte."""
    vals = comp.vals.cpu().contiguous()
    meta = comp.meta.cpu().contiguous()
    n = ctypes.c_size_t()
    capi.spfy_packed_bytes(_DT[comp.dtype], comp.rows, comp.cols, comp.layout, ctypes.byref(n))
    buf = ctypes.create_string_buffer(n.value)
    capi.spfy_packed_write(_DT[comp.dtype], comp.layout, comp.rows, comp.cols, vals.data_ptr(), meta.data_ptr(),
                           ctypes.cast(buf, ctypes.c_void_p), n.value)
    return buf.raw


def unpack_compressed(blob, device):
    """bytes written by pack_compressed -> Compressed24 on `device` (validated: magic, version, sizes, checksum)"""
    buf = ctypes.create_string_buffer(blob, len(blob))
    dt, layout = ctypes.c_int(), ctypes.c_int()
    rows, cols, vo, vb, mo, mb = (ctypes.c_size_t() for _ in range(6))
    capi.spfy_packed_read(ctypes.cast(buf, ctypes.c_void_p), len(blob), ctypes.byref(dt), ctypes.byref(layout),
                          ctypes.byref(rows), ctypes.byref(cols), ctypes.byref(vo), ctypes.byref(vb), ctypes.byref(mo),
                          ctypes.byref(mb))
    raw = torch.frombuffer(bytearray(blob), dtype=torch.uint8)
    tdt = {v: k for k, v in _DT.items()}[dt.value]
    return Compressed24(raw[vo.value: vo.value + vb.value].to(device), raw[mo.value: mo.value + mb.value].to(device),
                        rows.value, cols.value, tdt, layout.value)


_ACTS = {"none": capi.ACT_NONE, "relu": capi.ACT_RELU, "gelu_tanh": capi.ACT_GELU_TANH}


@dataclass
class Epilogue:
    """What the spmma epilogue applies before the output is written (spfy_epilogue, cusparseLt's ALPHA_VECTOR_SCALING /
    BIAS_POINTER / ACTIVATION_*): per output element (i, j), in fp32 and rounded to 16 bit once,
        v = (alpha * scale[i]) * acc + beta * C + bias[i],   D = act(v)
    i is the output row: the output channel of a convolution, the output feature of a Linear layer.  `scale` / `bias`:
    fp32 CUDA tensors of m elements (None: 1 / 0); act: "none", "relu" or "gelu_tanh" (torch's gelu(approximate="tanh")).
    fold_batchnorm turns an inference batch norm into (scale, bias)."""
    scale: torch.Tensor = None
    bias: torch.Tensor = None
    act: str = "none"

    def _c(self, m):
        if self.act not in _ACTS:
            raise ValueError(f"Epilogue: act must be one of {sorted(_ACTS)}, got {self.act!r}")
        for name, t in (("scale", self.scale), ("bias", self.bias)):
            if t is not None and (t.dtype != torch.float32 or not t.is_contiguous() or t.numel() < m):
                raise ValueError(f"Epilogue: {name} must be a contiguous fp32 tensor of at least {m} elements")
        return capi.Epilogue(_ptr(self.scale), _ptr(self.bias), _ACTS[self.act])


def fold_batchnorm(gamma, beta, mean, var, eps=1e-5):
    """An inference batch norm, y = gamma * (x - mean) / sqrt(var + eps) + beta, as the (scale, bias) of an Epilogue
    (fp32 tensors on the device of `gamma`)."""
    scale = gamma.float() / torch.sqrt(var.float() + eps)
    return scale.contiguous(), (beta.float() - mean.float() * scale).contiguous()


class SpmmaPlan:
    """spfy_spmma_plan_*: a list of independent D_i = alpha_i * A_i(2:4) * op(B_i) + beta_i * C_i executed
    by one persistent launch per ring-geometry class present (tensor maps + tile schedule built once, like
    cusparseLtMatmulPlanInit at spmma.hxx:79).  `problems`: dicts with comp, b, out and optional c, alpha,
    beta, op_b, out_t (out is then [n, m], the transposed result; beta must be 0 unless the plan has epilogues) and
    epilogue (an Epilogue: any problem with one makes the plan go through spfy_spmma_plan_create_ex, same launches).
    The plan keeps the tensors alive.
    Optional `replicas` per problem: device addresses (ints) of further copies of `out` (same shape and row pitch) that
    the epilogue stores every tile to as well -- e.g. the slab of this rank in the gather arena of every peer GPU
    (spfy_spmma_plan_create_replicated: the fused output gather); every problem must name the same number of them.
    A problem with `conv=(kh, kw, stride, pad)` is a convolution layer (spfy_spmma_plan_create_conv): `b` is then the
    NHWC activation tensor [batch, h, w, ch] and comp holds the weights with K in (kh, kw, ch) order; the unfolded
    operand is never built.  `out` is [m, batch*ho*wo], or NHWC [batch, ho, wo, m] with out_t."""

    def __init__(self, problems):
        self._keep = problems
        n = len(problems)
        arr = (capi.SpmmaProblem * n)()
        convs = (capi.ConvDesc * max(n, 1))()
        conv_ptrs = (ctypes.c_void_p * max(n, 1))()
        any_conv = False
        epis = (capi.Epilogue * max(n, 1))()
        epi_ptrs = (ctypes.c_void_p * max(n, 1))()
        any_epi = False
        dtype = None
        for i, q in enumerate(problems):
            comp, b, out = q["comp"], q["b"], q["out"]
            c = q.get("c")
            op_b = q.get("op_b", capi.OP_N)
            dtype = comp.dtype
            ldb = b.stride(0)
            ldd = out.stride(0)
            if q.get("conv"):
                kh, kw, stride, pad = q["conv"]
                assert b.dim() == 4 and b.is_contiguous()
                nb, h, w, ch = b.shape
                assert comp.cols == kh * kw * ch
                convs[i] = capi.ConvDesc(nb, h, w, ch, kh, kw, stride, pad)
                conv_ptrs[i] = ctypes.addressof(convs[i])
                any_conv = True
                op_b, ldb = capi.OP_T, comp.cols
                nn = nb * ((h + 2 * pad - kh) // stride + 1) * ((w + 2 * pad - kw) // stride + 1)
                if q.get("out_t"):
                    assert out.is_contiguous()
                    ldd = comp.rows
            else:
                nn = b.shape[1] if op_b == capi.OP_N else b.shape[0]
            if q.get("out_t"):  # `out` is [n, m]: the transposed result
                op_b |= capi.OUT_T
            if q.get("epilogue") is not None:
                epis[i] = q["epilogue"]._c(comp.rows)
                epi_ptrs[i] = ctypes.addressof(epis[i])
                any_epi = True
            arr[i] = capi.SpmmaProblem(op_b, comp.rows, nn, comp.cols, comp.vals.data_ptr(), comp.meta.data_ptr(),
                                       b.data_ptr(), ldb, c.data_ptr() if c is not None else None,
                                       c.stride(-2) if c is not None else 0, out.data_ptr(), ldd,
                                       float(q.get("alpha", 1.0)), float(q.get("beta", 0.0)))
        self._h = ctypes.c_void_p()
        nrep = len(problems[0].get("replicas", ())) if n else 0
        if any(len(q.get("replicas", ())) != nrep for q in problems):
            raise ValueError("SpmmaPlan: every problem needs the same number of replicas")
        if any_epi:
            if nrep:
                raise ValueError("SpmmaPlan: replicas and epilogues cannot be combined")
            capi.spfy_spmma_plan_create_ex(_DT[dtype], ctypes.cast(arr, ctypes.c_void_p),
                                           ctypes.cast(conv_ptrs, ctypes.c_void_p) if any_conv else None,
                                           ctypes.cast(epi_ptrs, ctypes.c_void_p), n, ctypes.byref(self._h))
        elif any_conv:
            if nrep:
                raise ValueError("SpmmaPlan: replicas and convolution problems cannot be combined")
            capi.spfy_spmma_plan_create_conv(_DT[dtype], ctypes.cast(arr, ctypes.c_void_p), ctypes.cast(conv_ptrs, ctypes.c_void_p),
                                             n, ctypes.byref(self._h))
        elif nrep:
            rep = (ctypes.c_void_p * (n * nrep))(*[int(a) for q in problems for a in q["replicas"]])
            capi.spfy_spmma_plan_create_replicated(_DT[dtype], ctypes.cast(arr, ctypes.c_void_p), n, nrep,
                                                   ctypes.cast(rep, ctypes.c_void_p), ctypes.byref(self._h))
        else:
            capi.spfy_spmma_plan_create(_DT[dtype], ctypes.cast(arr, ctypes.c_void_p), n, ctypes.byref(self._h))
        self.replicas = nrep
        self.launches = capi.spfy_spmma_plan_launches(self._h)

    def run(self):
        capi.spfy_spmma_plan_run(self._h, _stream())

    def run_launch(self, index):
        capi.spfy_spmma_plan_run_launch(self._h, index, _stream())

    def launch_info(self, index):
        v = [ctypes.c_int() for _ in range(4)]
        capi.spfy_spmma_plan_launch_info(self._h, index, *[ctypes.byref(x) for x in v])
        return dict(zip(("problems", "units", "stages", "smem_bytes"), (x.value for x in v)))

    def close(self):
        if self._h:
            capi.spfy_spmma_plan_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:  # noqa: BLE001
            pass


# --------------------------------------------------------------------- 2:4 fine-tuning
def transpose24(comp, taps=1, out=None, invalid=None):
    """spfy_transpose24: the compressed operand of A' [cols/taps, taps*rows] from the compressed A [rows, cols],
        A'[ci][t'*rows + r] = A[r][(taps-1-t')*cols/taps + ci].
    taps=1: A' = A^T, the operand of a Linear layer's data gradient, dx = dy W:
        spmma_compressed(transpose24(comp), dy, op_b=OP_T, out_t=True)
    taps=kh*kw (weights permuted with permute_conv_weights before pruning): A' is the flipped, channel-swapped filter
    of a stride-1 convolution's data gradient, with dy and dx in NHWC:
        spmma_conv_nhwc(transpose24(comp, taps=kh * kw), dy, kh, kw, stride=1, pad=kh - 1 - pad)
    A's mask must keep two of four along columns too (PRUNE_TILE_TRANSPOSABLE, or TILE_MAG on weights without zeros).
    `invalid`: optional int32 CUDA tensor, set to 0, or to 1 when the mask is not transposable (the result is then
    unspecified).  Nothing here syncs.  Returns a Compressed24 (== out when given)."""
    assert comp.layout == capi.LAYOUT_SM100
    if comp.cols % taps:
        raise capi.SpfyError(capi.E_INVALID, "transpose24", f"cols {comp.cols} is not a multiple of taps {taps}")
    rows_t, cols_t = comp.cols // taps, taps * comp.rows
    if out is None:
        out = alloc_compressed(comp.dtype, rows_t, cols_t, comp.vals.device)
    assert (out.rows, out.cols, out.dtype, out.layout) == (rows_t, cols_t, comp.dtype, capi.LAYOUT_SM100)
    if invalid is not None:
        assert invalid.dtype == torch.int32 and invalid.is_cuda
    capi.spfy_transpose24(_DT[comp.dtype], _ptr(comp.vals), _ptr(comp.meta), comp.rows, comp.cols, taps,
                          _ptr(out.vals), _ptr(out.meta), _ptr(invalid), _stream())
    return out


def _dgrad_phase(k, s, p, a):
    """the taps of output phase a of a stride-s data gradient in one dimension (spfy_transpose24_conv):
    (filter indices in descending order, dy offset of the first)"""
    taps = [kt for kt in range(k - 1, -1, -1) if (a + p - kt) % s == 0]
    return taps, ((a + p - taps[0]) // s if taps else 0)


@dataclass
class Transpose24Conv:
    """The data-gradient filter operands of a stride-`stride` convolution (spfy_transpose24_conv): one SM100 operand per
    output phase (a, b) with taps, back to back in `vals` / `meta`.  `phases`: [(a, b, taps_h, taps_w, Compressed24)],
    the Compressed24 of each a view of c rows x len(taps_h)*len(taps_w)*m columns (taps in descending filter index)."""
    vals: torch.Tensor
    meta: torch.Tensor
    m: int
    c: int
    kh: int
    kw: int
    stride: int
    pad: int
    dtype: torch.dtype
    phases: list


def transpose24_conv(comp, kh, kw, stride, pad, invalid=None, out=None):
    """spfy_transpose24_conv: the operands of the data gradient of a stride-`stride`, pad-`pad` convolution whose filter
    `comp` is m x kh*kw*c in (kh, kw, c) order (permute_conv_weights, then prune24 with PRUNE_TILE_TRANSPOSABLE).  Phase
    (a, b) holds the dx pixels (s*i + a, s*j + b); its operand is the flipped, channel-swapped sub-filter of the taps
    that reach them.  For stride 1 the one operand is transpose24(comp, taps=kh*kw), byte for byte.
    `invalid`: optional int32 CUDA tensor, 0, or 1 when the mask is not transposable.  `out`: a Transpose24Conv of the
    same layer to refill in place (returned).  Nothing here syncs.  Use it with spmma_conv_dgrad_nhwc."""
    assert comp.layout == capi.LAYOUT_SM100
    if comp.cols % (kh * kw):
        raise capi.SpfyError(capi.E_INVALID, "transpose24_conv", f"cols {comp.cols} is not a multiple of kh*kw {kh * kw}")
    m, c = comp.rows, comp.cols // (kh * kw)
    if invalid is not None:
        assert invalid.dtype == torch.int32 and invalid.is_cuda
    if out is not None:
        assert (out.m, out.c, out.kh, out.kw, out.stride, out.pad, out.dtype) == (m, c, kh, kw, stride, pad, comp.dtype)
        capi.spfy_transpose24_conv(_DT[comp.dtype], _ptr(comp.vals), _ptr(comp.meta), m, c, kh, kw, stride, pad,
                                   _ptr(out.vals), _ptr(out.meta), _ptr(invalid), _stream())
        return out
    vb, mb = ctypes.c_size_t(), ctypes.c_size_t()
    capi.spfy_transpose24_conv_bytes(_DT[comp.dtype], m, c, kh, kw, stride, pad, ctypes.byref(vb), ctypes.byref(mb))
    dev = comp.vals.device
    vals = torch.empty(vb.value, dtype=torch.uint8, device=dev)
    meta = torch.empty(mb.value, dtype=torch.uint8, device=dev)
    capi.spfy_transpose24_conv(_DT[comp.dtype], _ptr(comp.vals), _ptr(comp.meta), m, c, kh, kw, stride, pad,
                               _ptr(vals), _ptr(meta), _ptr(invalid), _stream())
    phases, tile = [], 0
    for a in range(stride):
        for b in range(stride):
            th, tw = _dgrad_phase(kh, stride, pad, a)[0], _dgrad_phase(kw, stride, pad, b)[0]
            if not th or not tw:
                continue
            cols = len(th) * len(tw) * m
            tiles = -(-c // 128) * -(-cols // 128)
            view = Compressed24(vals[tile * 16384:(tile + tiles) * 16384], meta[tile * 2048:(tile + tiles) * 2048], c, cols,
                                comp.dtype, capi.LAYOUT_SM100)
            phases.append((a, b, th, tw, view))
            tile += tiles
    return Transpose24Conv(vals, meta, m, c, kh, kw, stride, pad, comp.dtype, phases)


def spmma_conv_dgrad_nhwc(op, dy, h, w, out=None, alpha=1.0, beta=0.0):
    """spfy_spmma_conv_dgrad: dx = alpha * conv2d_input(W, dy) + beta * out for the forward layer of `op`
    (transpose24_conv), any stride, on sparse tensor cores.  dy: NHWC [batch, ho, wo, m]; h, w: the forward input size
    (a strided layer's ho, wo do not determine it).  Returns dx, NHWC [batch, h, w, c] (== out when given; beta != 0
    needs out, and beta = 1 accumulates into it).  The backward data pass of a strided layer, dy and dx in NHWC:
        w2 = permute_conv_weights(weight.view(m, -1), c, kh, kw)       # (kh, kw, c) order, before pruning
        comp = prune24(w2, mode=PRUNE_TILE_TRANSPOSABLE)
        op = transpose24_conv(comp, kh, kw, stride, pad)              # once per weight update
        dx = spmma_conv_dgrad_nhwc(op, dy, h, w)
    With beta=1 and out = the shortcut's dx, a residual downsample block's two data gradients meet in place.
    The same call is a 2:4 transposed convolution (ConvTranspose2d with stride s, padding pad, output size h x w) of a
    filter pruned in the forward orientation: x_up = spmma_conv_dgrad_nhwc(op, x, h, w)."""
    assert dy.dim() == 4 and dy.is_contiguous() and dy.dtype == op.dtype
    nb, ho, wo, m = dy.shape
    s, p = op.stride, op.pad
    if h + 2 * p < op.kh or w + 2 * p < op.kw or (ho, wo, m) != ((h + 2 * p - op.kh) // s + 1, (w + 2 * p - op.kw) // s + 1,
                                                                  op.m):
        raise capi.SpfyError(capi.E_INVALID, "spmma_conv_dgrad", f"dy {tuple(dy.shape)} does not match a {op.kh}x{op.kw} "
                             f"stride {s} pad {p} layer with {op.m} outputs on {h}x{w} inputs")
    if out is None:
        if beta != 0.0:
            raise capi.SpfyError(capi.E_INVALID, "spmma_conv_dgrad", "beta != 0 needs out")
        out = torch.empty(nb, h, w, op.c, dtype=op.dtype, device=dy.device)
    assert out.is_contiguous() and tuple(out.shape) == (nb, h, w, op.c) and out.dtype == op.dtype
    desc = capi.ConvDesc(nb, h, w, op.c, op.kh, op.kw, s, p)
    capi.spfy_spmma_conv_dgrad(_DT[op.dtype], ctypes.byref(desc), op.m, float(alpha), _ptr(op.vals), _ptr(op.meta),
                               _ptr(dy), float(beta), _ptr(out), _stream())
    return out


def conv_wgrad24_nhwc(comp, x, dy, kh, kw, stride=1, pad=0, out=None, alpha=1.0, beta=0.0):
    """spfy_conv_wgrad24: dW = alpha * mask(conv2d_weight(x, dy)) + beta * out, fp32, for the forward layer whose filter
    `comp` is m x kh*kw*c in (kh, kw, c) order; the mask is comp's, and every position it prunes is +0.  x: NHWC
    [batch, h, w, c]; dy: NHWC [batch, ho, wo, m], both in comp.dtype.  Returns dW (== out when given), fp32 in
    (kh, kw, c) order: a new [m, kh*kw*c] tensor, or `out`, which may be [m, kh*kw*c] row-major or a channels_last
    [m, c, kh, kw] weight (the same storage).  beta != 0 needs out; beta = 1 accumulates into it."""
    assert comp.layout == capi.LAYOUT_SM100
    assert x.dim() == 4 and x.is_contiguous() and dy.dim() == 4 and dy.is_contiguous()
    nb, h, w, c = x.shape
    m, kk = comp.rows, kh * kw * c
    if x.dtype != comp.dtype or dy.dtype != comp.dtype:
        raise TypeError(f"conv_wgrad24_nhwc: x {x.dtype} and dy {dy.dtype} must be the layer dtype {comp.dtype}")
    ho, wo = (h + 2 * pad - kh) // stride + 1, (w + 2 * pad - kw) // stride + 1
    if comp.cols != kk or tuple(dy.shape) != (nb, ho, wo, m):
        raise capi.SpfyError(capi.E_INVALID, "conv_wgrad24", f"x {tuple(x.shape)}, dy {tuple(dy.shape)} do not match a "
                             f"{kh}x{kw} stride {stride} pad {pad} layer with filter {m} x {comp.cols}")
    if out is None:
        if beta != 0.0:
            raise capi.SpfyError(capi.E_INVALID, "conv_wgrad24", "beta != 0 needs out")
        out = torch.empty(m, kk, dtype=torch.float32, device=x.device)
    dense = (out.is_contiguous() and tuple(out.shape) == (m, kk)) or (
        tuple(out.shape) == (m, c, kh, kw) and out.is_contiguous(memory_format=torch.channels_last))
    if out.dtype != torch.float32 or not dense:
        raise ValueError(f"conv_wgrad24_nhwc: out must be fp32, [{m}, {kk}] contiguous or [{m}, {c}, {kh}, {kw}] "
                         f"channels_last; got {out.dtype} {tuple(out.shape)} strides {out.stride()}")
    desc = capi.ConvDesc(nb, h, w, c, kh, kw, stride, pad)
    wb = ctypes.c_size_t()
    capi.spfy_conv_wgrad24_workspace_bytes(_DT[comp.dtype], ctypes.byref(desc), m, ctypes.byref(wb))
    ws = _workspace(wb.value, x.device)
    capi.spfy_conv_wgrad24(_DT[comp.dtype], ctypes.byref(desc), m, float(alpha), _ptr(x), _ptr(dy), _ptr(comp.meta),
                           float(beta), _ptr(out), _ptr(ws), ws.numel(), _stream())
    return out


def recompress24(dense, comp, masked_out=None, values=True):
    """spfy_recompress24: new values under comp's fixed mask.  `dense` [comp.rows, comp.cols] (fp32, fp16 or bf16,
    row-major).  values=True: comp.vals <- dense at the positions comp.meta keeps, rounded to nearest even to comp.dtype
    (the metadata is not touched).  masked_out (may be `dense`): dense with every pruned position set to +0.
    The three jobs of a fine-tuning step: refresh the forward operand from an fp32 master, project a weight gradient
    onto the mask, re-mask the master in place."""
    assert comp.layout == capi.LAYOUT_SM100 and dense.dim() == 2 and dense.stride(1) == 1
    assert tuple(dense.shape) == (comp.rows, comp.cols)
    if masked_out is not None:
        assert masked_out.dtype == dense.dtype and masked_out.shape == dense.shape and masked_out.stride(1) == 1
    capi.spfy_recompress24(_dtype_code(dense), _ptr(dense), dense.stride(0), _DT[comp.dtype], comp.rows, comp.cols,
                           _ptr(comp.meta), _ptr(comp.vals) if values else None, _ptr(masked_out),
                           masked_out.stride(0) if masked_out is not None else 0, _stream())


# the Linear24 / Conv2d24 that owns a weight Parameter, by id(weight): how SGD24 / AdamW24 find a 2:4 layer's operands
_LAYERS24 = weakref.WeakValueDictionary()


class _Linear24Fn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x2, weight, bias, layer):
        del weight  # the forward operand is layer.comp; weight is an input so that its gradient reaches it
        ctx.layer = layer
        ctx.save_for_backward(x2)
        ctx.has_bias = bias is not None
        return spmma_compressed(layer.comp, x2, op_b=capi.OP_T, out_t=True,
                                epilogue=Epilogue(bias=bias.detach()) if bias is not None else None)

    @staticmethod
    def backward(ctx, dy):
        (x2,) = ctx.saved_tensors
        layer = ctx.layer
        dy = dy.to(layer.dtype).contiguous()
        tokens, out_f = dy.shape
        in_f = x2.shape[1]
        dx = None
        if ctx.needs_input_grad[0]:
            dx = spmma_compressed(layer.comp_t, dy, op_b=capi.OP_T, out_t=True)  # dy W on sparse tensor cores
        dw = None
        if ctx.needs_input_grad[1]:
            # dW [out, in] = dy^T x: column-major m = in, n = out, k = tokens on the dense tcgen05 GEMM, then masked
            dt = _DT[layer.dtype]
            dw = torch.empty(out_f, in_f, dtype=layer.dtype, device=dy.device)
            wb = ctypes.c_size_t()
            capi.spfy_gemm_workspace_bytes(dt, capi.OP_N, capi.OP_T, in_f, out_f, tokens, in_f, out_f, 1, ctypes.byref(wb))
            ws = _workspace(wb.value, dy.device)
            capi.spfy_gemm_strided_batched(dt, capi.GEMM_PRECISE, capi.OP_N, capi.OP_T, in_f, out_f, tokens, 1.0,
                                           _ptr(x2), in_f, 0, _ptr(dy), out_f, 0, 0.0, _ptr(dw), in_f, 0, 1,
                                           _ptr(ws), ws.numel(), _stream())
            recompress24(dw, layer.comp, masked_out=dw, values=False)
            dw = dw.float()
        db = dy.float().sum(0) if ctx.has_bias and ctx.needs_input_grad[2] else None
        return dx, dw, db, None


class Linear24(torch.nn.Module):
    """A 2:4 Linear layer for fine-tuning with a fixed mask, y = x W^T + b, on sparse tensor cores forward and backward.
    State: `weight`, the fp32 master [out, in], kept masked; `bias` (fp32, optional); `comp` and `comp_t`, the 16-bit
    compressed W and W^T.  The mask is chosen once, by PRUNE_TILE_TRANSPOSABLE, so that W^T is a 2:4 operand as well.
      forward : spmma(comp, x) with the bias in the epilogue; x is [..., in] in `dtype`, and the flattened leading
                dimensions must be a multiple of 8
      backward: dx = dy W through comp_t (sparse tensor cores); dW = dy^T x on the dense tcgen05 GEMM, masked, fp32;
                db = sum of dy
    After optimizer.step(), call refresh(): it re-masks the master in place and rebuilds comp and comp_t from it (the
    mask does not move).  forward refuses to run on a weight changed since the last refresh.  An NHWC 1x1 stride-1
    convolution is this layer applied to the [..., channels] activation."""

    def __init__(self, weight, bias, comp, comp_t, dtype):
        super().__init__()
        self.weight = torch.nn.Parameter(weight)
        self.bias = torch.nn.Parameter(bias) if bias is not None else None
        self.comp, self.comp_t, self.dtype = comp, comp_t, dtype
        self._synced_version = self.weight._version
        _LAYERS24[id(self.weight)] = self

    @classmethod
    def from_dense(cls, w, b=None, dtype=torch.float16):
        """Prune `w` [out, in] (out and in multiples of 8, in a multiple of 16) with PRUNE_TILE_TRANSPOSABLE in
        `dtype`.  Raises ValueError if the mask is not transposable (one sync, here only)."""
        with torch.no_grad():
            w16 = w.detach().to(dtype).contiguous()
            comp = prune24(w16, inplace=True, mode=capi.PRUNE_TILE_TRANSPOSABLE)
            master = w.detach().float().contiguous().clone()
            recompress24(master, comp, masked_out=master, values=False)
            invalid = torch.empty(1, dtype=torch.int32, device=w.device)
            comp_t = transpose24(comp, invalid=invalid)
            if int(invalid.item()):
                raise ValueError("Linear24: the pruned mask is not transposable")
            bias = b.detach().float().contiguous().clone() if b is not None else None
        return cls(master, bias, comp, comp_t, dtype)

    @torch.no_grad()
    def refresh(self):
        """master -> comp.vals (mask fixed), master re-masked in place, comp -> comp_t.  No sync."""
        recompress24(self.weight, self.comp, masked_out=self.weight)
        transpose24(self.comp, out=self.comp_t)
        self._synced_version = self.weight._version

    def forward(self, x):
        if self.weight._version != self._synced_version:
            raise RuntimeError("Linear24: weight changed since the last refresh(); call refresh() after optimizer.step()")
        in_f = self.comp.cols
        x2 = x.reshape(-1, in_f).contiguous()
        if x2.dtype != self.dtype:
            raise TypeError(f"Linear24: input dtype {x2.dtype}, layer dtype {self.dtype}")
        y = _Linear24Fn.apply(x2, self.weight, self.bias, self)
        return y.view(*x.shape[:-1], self.comp.rows)


class _Conv2d24Fn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, x, weight, bias, layer):
        del weight  # the forward operand is layer.comp; weight is an input so that its gradient reaches it
        ctx.layer = layer
        ctx.save_for_backward(x)
        ctx.has_bias = bias is not None
        y = spmma_conv_nhwc(layer.comp, x.permute(0, 2, 3, 1), layer.kh, layer.kw, layer.stride, layer.padding,
                            epilogue=Epilogue(bias=bias.detach()) if bias is not None else None)
        return y.permute(0, 3, 1, 2)  # [N, M, Ho, Wo], channels_last

    @staticmethod
    def backward(ctx, dy):
        (x,) = ctx.saved_tensors
        layer = ctx.layer
        xh = x.permute(0, 2, 3, 1)
        dyh = dy.to(layer.dtype).permute(0, 2, 3, 1).contiguous()  # no copy when dy is channels_last in the layer dtype
        dx = dw = db = None
        if ctx.needs_input_grad[0]:
            dx = spmma_conv_dgrad_nhwc(layer.op_t, dyh, x.shape[2], x.shape[3]).permute(0, 3, 1, 2)
        if ctx.needs_input_grad[1]:
            dw = conv_wgrad24_nhwc(layer.comp, xh, dyh, layer.kh, layer.kw, layer.stride, layer.padding,
                                   out=torch.empty_like(layer.weight, memory_format=torch.channels_last))
        if ctx.has_bias and ctx.needs_input_grad[2]:
            db = dyh.float().sum((0, 1, 2))
        return dx, dw, db, None


class Conv2d24(torch.nn.Module):
    """A 2:4 convolution for fine-tuning with a fixed mask, the convolutional twin of Linear24: forward and both
    gradients on tcgen05, activations channels_last.  The filter is pruned in (kh, kw, c) order with
    PRUNE_TILE_TRANSPOSABLE, so that the data gradient's flipped filter is a 2:4 operand as well.
    State: `weight`, the fp32 master [m, c, kh, kw] in torch.channels_last, kept masked -- its storage is the (kh, kw, c)
    order of the operand, so optimizers work on it unchanged and dW is written straight into a tensor of its layout;
    `bias` (fp32, optional); `comp`, the 16-bit compressed filter; `op_t`, the data gradient's phase operands.
      forward : spmma_conv_nhwc(comp, x) with the bias in the epilogue; x is [N, c, H, W] in `dtype` and channels_last
                with N * Ho * Wo a multiple of 8, the result [N, m, Ho, Wo] channels_last
      backward: dx = spmma_conv_dgrad_nhwc(op_t, dy) (any stride); dW = conv_wgrad24_nhwc, fp32, masked; db = sum of dy
    After optimizer.step(), call refresh(): it re-masks the master in place and refills comp and op_t from it (the mask
    does not move).  forward refuses to run on a weight changed since the last refresh."""

    def __init__(self, weight, bias, comp, op_t, dtype, stride, padding):
        super().__init__()
        self.weight = torch.nn.Parameter(weight)
        self.bias = torch.nn.Parameter(bias) if bias is not None else None
        self.comp, self.op_t, self.dtype = comp, op_t, dtype
        self.m, self.c, self.kh, self.kw = weight.shape
        self.stride, self.padding = stride, padding
        self._synced_version = self.weight._version
        _LAYERS24[id(self.weight)] = self

    @classmethod
    def from_dense(cls, weight, bias=None, stride=1, padding=0, dtype=torch.float16, groups=1, dilation=1):
        """Prune `weight` [m, c, kh, kw] (c a multiple of 64, m a multiple of 64) in `dtype`.  Raises ValueError for
        groups or dilation other than 1, for c or m off those multiples, and when the pruned mask is not transposable
        (one sync, here only)."""
        m, c, kh, kw = weight.shape
        if groups != 1 or dilation != 1:
            raise ValueError("Conv2d24: grouped and dilated convolutions are not supported")
        if c % 64 or m % 64:
            raise ValueError(f"Conv2d24: in and out channels must be multiples of 64 (got c = {c}, m = {m})")
        with torch.no_grad():
            master = weight.detach().float().contiguous(memory_format=torch.channels_last).clone(
                memory_format=torch.channels_last)
            w2 = master.permute(0, 2, 3, 1).reshape(m, kh * kw * c)  # a view: the (kh, kw, c) storage
            w16 = w2.to(dtype).contiguous()
            comp = prune24(w16, inplace=True, mode=capi.PRUNE_TILE_TRANSPOSABLE)
            recompress24(w2, comp, masked_out=w2, values=False)
            invalid = torch.empty(1, dtype=torch.int32, device=weight.device)
            op_t = transpose24_conv(comp, kh, kw, stride, padding, invalid=invalid)
            if int(invalid.item()):
                raise ValueError("Conv2d24: the pruned mask is not transposable")
            b = bias.detach().float().contiguous().clone() if bias is not None else None
        return cls(master, b, comp, op_t, dtype, stride, padding)

    def _w2d(self):
        """the master as the [m, kh*kw*c] matrix of its storage"""
        if not self.weight.is_contiguous(memory_format=torch.channels_last):
            raise RuntimeError("Conv2d24: the weight is no longer channels_last")
        return self.weight.permute(0, 2, 3, 1).reshape(self.m, -1)

    @torch.no_grad()
    def refresh(self):
        """master -> comp.vals (mask fixed), master re-masked in place, comp -> op_t (in place).  No sync."""
        w2 = self._w2d()
        recompress24(w2, self.comp, masked_out=w2)
        transpose24_conv(self.comp, self.kh, self.kw, self.stride, self.padding, out=self.op_t)
        self._synced_version = self.weight._version

    def forward(self, x):
        if self.weight._version != self._synced_version:
            raise RuntimeError("Conv2d24: weight changed since the last refresh(); call refresh() after optimizer.step()")
        if x.dtype != self.dtype:
            raise TypeError(f"Conv2d24: input dtype {x.dtype}, layer dtype {self.dtype}: convert with x.to({self.dtype})")
        if x.dim() != 4 or not x.is_contiguous(memory_format=torch.channels_last):
            raise ValueError("Conv2d24: the input must be a 4-D channels_last tensor: convert with "
                             "x.contiguous(memory_format=torch.channels_last)")
        return _Conv2d24Fn.apply(x, self.weight, self.bias, self)


def _non_overlapping_dense(t):
    expected = 1
    for size, stride in sorted(zip(t.shape, t.stride()), key=lambda e: e[1]):
        if size != 1:
            if stride != expected:
                return False
            expected *= size
    return True


def _layer24_of(p):
    layer = _LAYERS24.get(id(p))
    return layer if layer is not None and layer.weight is p else None


class _Optim24(torch.optim.Optimizer):
    """spfy_optim24_step behind torch.optim.Optimizer: one step() updates every parameter that has a gradient in one
    library launch (up to 192 parameters and 16 parameter groups per launch; more take further launches).  The weight of a Linear24 / Conv2d24 is a 2:4 item: updated at
    the kept positions, re-masked, and the layer's compressed operands refilled in the same pass, so no refresh() is
    needed.  Every other parameter must be a non-overlapping, dense fp32 tensor; it is updated elementwise.  State
    tensors carry torch's names and the parameter's layout, so state_dict() moves to and from the torch optimizer.
    GradScaler: grad_scale and found_inf are read on the device (no sync); a step with found_inf != 0 writes nothing."""
    _ALGO = None
    _step_supports_amp_scaling = True

    def __init__(self, params, defaults):
        for k in ("amsgrad", "maximize", "foreach", "fused", "differentiable"):
            if defaults.get(k):
                raise ValueError(f"{type(self).__name__}: {k}=True is not supported")
        super().__init__(params, defaults)

    def add_param_group(self, param_group):
        super().add_param_group(param_group)
        group = self.param_groups[-1]
        try:
            self._check_group(group)
            device = None
            for g in self.param_groups:
                for p in g["params"]:
                    if p.dtype != torch.float32:
                        raise TypeError(f"{type(self).__name__}: parameters must be fp32, got {p.dtype}")
                    if not _non_overlapping_dense(p):
                        raise ValueError(f"{type(self).__name__}: a parameter of strides {p.stride()} is not dense")
                    if device is not None and p.device != device:
                        raise ValueError(f"{type(self).__name__}: parameters on {device} and {p.device}")
                    device = p.device
        except (TypeError, ValueError):
            self.param_groups.pop()
            raise

    def _check_group(self, group):
        if group["lr"] < 0.0:
            raise ValueError(f"Invalid learning rate: {group['lr']}")
        for k in ("amsgrad", "maximize", "foreach", "fused", "differentiable"):
            if group.get(k):
                raise ValueError(f"{type(self).__name__}: {k}=True is not supported")

    def _table(self):
        """The item table of the parameters with a gradient: (ctypes items, ctypes hparams, params, layers, keep-alive
        tensors, AdamW step counts, SGD first-step flags as (param, flag)).  Creates missing state; needs no device."""
        items, params, layers, keep, steps, firsts = [], [], [], [], [], []
        hps = (capi.Optim24Hparams * len(self.param_groups))()
        for gi, group in enumerate(self.param_groups):
            self._hparams(group, hps[gi])
            for p in group["params"]:
                g = p.grad
                if g is None:
                    continue
                if g.is_sparse:
                    raise TypeError(f"{type(self).__name__} does not support sparse gradients")
                if g.stride() != p.stride():
                    g = torch.empty_like(p).copy_(g)  # the kernel reads the gradient in the parameter's layout
                    keep.append(g)
                state = self.state[p]
                it = capi.Optim24Item(param=p.data_ptr(), grad=g.data_ptr(), rows=1, cols=p.numel(), ld=p.numel(),
                                      group=gi)
                for k, s in self._states(p, state, it, firsts):
                    if s.stride() != p.stride() or s.device != p.device:
                        s = state[k] = torch.empty_like(p).copy_(s)
                    setattr(it, "state1" if k in ("momentum_buffer", "exp_avg") else "state2", s.data_ptr())
                if "step" in state:
                    st = state["step"]
                    if st.device != p.device or st.dtype != torch.float32:
                        st = state["step"] = st.to(device=p.device, dtype=torch.float32)
                    it.step = st.data_ptr()
                    steps.append(st)
                layer = _layer24_of(p)
                if layer is not None:
                    self._item24(layer, it)
                    layers.append(layer)
                items.append(it)
                params.append(p)
        return (capi.Optim24Item * len(items))(*items), hps, params, layers, keep, steps, firsts

    @staticmethod
    def _item24(layer, it):
        comp = layer.comp
        op_t = layer.op_t if isinstance(layer, Conv2d24) else layer.comp_t
        if any(t.device != layer.weight.device for t in (comp.vals, comp.meta, op_t.vals)):
            raise ValueError(f"{type(layer).__name__}: the compressed operands are not on the weight's device")
        it.rows, it.cols, it.dtype = comp.rows, comp.cols, _DT[layer.dtype]
        it.meta, it.vals = comp.meta.data_ptr(), comp.vals.data_ptr()
        if isinstance(layer, Conv2d24):
            it.ld = layer._w2d().stride(0)
            it.vals_t = layer.op_t.vals.data_ptr()
            it.kh, it.kw, it.stride, it.pad = layer.kh, layer.kw, layer.stride, layer.padding
        else:
            w = layer.weight
            if tuple(w.shape) != (comp.rows, comp.cols) or w.stride(1) != 1:
                raise ValueError("Linear24: the weight is no longer a row-major [out, in] matrix")
            it.ld = w.stride(0)
            it.vals_t = layer.comp_t.vals.data_ptr()
            it.kh = it.kw = it.stride = 1

    @torch.no_grad()
    def step(self, closure=None):
        loss = None
        if closure is not None:
            with torch.enable_grad():
                loss = closure()
        for group in self.param_groups:  # the table holds raw addresses: refuse host memory before anything changes
            for p in group["params"]:
                if p.grad is not None and not p.is_cuda:
                    raise capi.SpfyError(capi.E_INVALID, type(self).__name__, f"a parameter on {p.device}: "
                                         "sparsify.me_b200 has no host path")
        items, hps, params, layers, keep, steps, firsts = self._table()
        if not params:
            return loss
        grad_scale = getattr(self, "grad_scale", None)
        found_inf = getattr(self, "found_inf", None)
        if grad_scale is not None:
            grad_scale = grad_scale.to(device=params[0].device, dtype=torch.float32)
            keep.append(grad_scale)
        if found_inf is not None:
            found_inf = found_inf.to(device=params[0].device, dtype=torch.float32)
            keep.append(found_inf)
        inc = 1.0 if found_inf is None else 1.0 - found_inf.reshape(())
        if steps:  # AdamW: the count advances by 1 - found_inf, on the stream, before the kernel reads it
            torch._foreach_add_(steps, inc)
        try:
            capi.spfy_optim24_step(self._ALGO, items, len(items), hps, len(hps), _ptr(grad_scale), _ptr(found_inf),
                                   _stream())
        except capi.SpfyError:
            if steps:  # refused before any launch: the state is as it was
                torch._foreach_sub_(steps, inc)
            raise
        if firsts:  # SGD: a first step is done once it was applied; a skipped one (found_inf != 0) stays pending
            if found_inf is None:
                for p, _ in firsts:
                    del self._first[p]
            else:
                torch._foreach_mul_([f for _, f in firsts], found_inf.reshape(()))
        torch.autograd.graph.increment_version(params)
        for layer in layers:
            layer._synced_version = layer.weight._version  # its operands were refilled by the same launch
        return loss


class SGD24(_Optim24):
    """torch.optim.SGD for models with Linear24 / Conv2d24 layers: the update of torch's _multi_tensor_sgd in fp32,
    the 2:4 layers refreshed by the same launch.  maximize, foreach, fused and differentiable are not supported.
        opt = SGD24(model.parameters(), lr=0.1, momentum=0.9)
        loss.backward(); opt.step()          # no refresh()"""
    _ALGO = capi.OPTIM_SGD

    def __init__(self, params, lr=1e-3, momentum=0.0, dampening=0.0, weight_decay=0.0, nesterov=False, *,
                 maximize=False, foreach=None, differentiable=False, fused=None):
        if lr < 0.0:
            raise ValueError(f"Invalid learning rate: {lr}")
        if momentum < 0.0:
            raise ValueError(f"Invalid momentum value: {momentum}")
        if weight_decay < 0.0:
            raise ValueError(f"Invalid weight_decay value: {weight_decay}")
        if nesterov and (momentum <= 0 or dampening != 0):
            raise ValueError("Nesterov momentum requires a momentum and zero dampening")
        # param -> device float, 1 while torch's first step (buf = grad) is still to be applied to the parameter
        self._first = {}
        super().__init__(params, dict(lr=lr, momentum=momentum, dampening=dampening, weight_decay=weight_decay,
                                      nesterov=nesterov, maximize=maximize, foreach=foreach,
                                      differentiable=differentiable, fused=fused))

    def _check_group(self, group):
        super()._check_group(group)
        if group["nesterov"] and (group["momentum"] <= 0 or group["dampening"] != 0):
            raise ValueError("Nesterov momentum requires a momentum and zero dampening")

    @staticmethod
    def _hparams(group, h):
        h.lr, h.momentum, h.dampening = group["lr"], group["momentum"], group["dampening"]
        h.weight_decay, h.nesterov = group["weight_decay"], int(bool(group["nesterov"]))

    def load_state_dict(self, state_dict):
        super().load_state_dict(state_dict)
        self._first.clear()  # a loaded momentum buffer has seen its first step

    def _states(self, p, state, it, firsts):
        if self.param_groups[it.group]["momentum"] == 0:
            return []
        if state.get("momentum_buffer") is None:
            state["momentum_buffer"] = torch.zeros_like(p, memory_format=torch.preserve_format)
            self._first[p] = torch.ones((), dtype=torch.float32, device=p.device)
        flag = self._first.get(p)
        if flag is not None:
            it.first = flag.data_ptr()
            firsts.append((p, flag))
        return [("momentum_buffer", state["momentum_buffer"])]


class AdamW24(_Optim24):
    """torch.optim.AdamW for models with Linear24 / Conv2d24 layers: the update of torch's _multi_tensor_adam with
    decoupled weight decay in fp32, the 2:4 layers refreshed by the same launch.  The bias corrections come from the
    `step` state, a device float, so a step needs no host value.  amsgrad, maximize, foreach, fused and differentiable
    are not supported."""
    _ALGO = capi.OPTIM_ADAMW

    def __init__(self, params, lr=1e-3, betas=(0.9, 0.999), eps=1e-8, weight_decay=1e-2, amsgrad=False, *,
                 maximize=False, foreach=None, capturable=False, differentiable=False, fused=None):
        if lr < 0.0:
            raise ValueError(f"Invalid learning rate: {lr}")
        if eps < 0.0:
            raise ValueError(f"Invalid epsilon value: {eps}")
        if not 0.0 <= betas[0] < 1.0 or not 0.0 <= betas[1] < 1.0:
            raise ValueError(f"Invalid beta parameters: {betas}")
        if weight_decay < 0.0:
            raise ValueError(f"Invalid weight_decay value: {weight_decay}")
        super().__init__(params, dict(lr=lr, betas=tuple(betas), eps=eps, weight_decay=weight_decay, amsgrad=amsgrad,
                                      maximize=maximize, foreach=foreach, capturable=capturable,
                                      differentiable=differentiable, fused=fused, decoupled_weight_decay=True))

    def _check_group(self, group):
        super()._check_group(group)
        if group["eps"] < 0.0:
            raise ValueError(f"Invalid epsilon value: {group['eps']}")

    @staticmethod
    def _hparams(group, h):
        h.lr, h.weight_decay, h.eps = group["lr"], group["weight_decay"], group["eps"]
        h.beta1, h.beta2 = group["betas"]

    def _states(self, p, state, it, firsts):
        if "step" not in state:
            state["step"] = torch.zeros((), dtype=torch.float32, device=p.device)
            state["exp_avg"] = torch.zeros_like(p, memory_format=torch.preserve_format)
            state["exp_avg_sq"] = torch.zeros_like(p, memory_format=torch.preserve_format)
        return [("exp_avg", state["exp_avg"]), ("exp_avg_sq", state["exp_avg_sq"])]


# ----------------------------------------------------------------------------- A4
def spmma_compressed(comp, b, c=None, out=None, alpha=1.0, beta=0.0, op_b=capi.OP_N, out_t=False, epilogue=None):
    """D = alpha * A(2:4) * op(B) + beta * C on tcgen05.mma.sp (cusparseLtMatmul, spmma.hxx:106-114).
    All dense operands row-major.  Returns D (== out, or a new tensor); out_t: D is [n, m], the transposed result
    (SPFY_OUT_T: NHWC for a convolution layer; beta must be 0 without an epilogue).
    epilogue: an Epilogue (per-row scale / bias, activation) applied before D is written (spfy_spmma_ex); with one,
    out_t also takes beta * C with C as [n, m] like D.  A Linear layer y = act(x W^T + b) is
    spmma_compressed(comp(W), x, op_b=OP_T, out_t=True, epilogue=Epilogue(bias=b, act=...))."""
    assert comp.layout == capi.LAYOUT_SM100
    m, k = comp.rows, comp.cols
    n = b.shape[1] if op_b == capi.OP_N else b.shape[0]
    assert (b.shape[0] if op_b == capi.OP_N else b.shape[1]) == k
    if out is None:
        out = torch.empty((n, m) if out_t else (m, n), dtype=comp.dtype, device=b.device)
    if out_t:
        op_b |= capi.OUT_T
    if epilogue is None:
        capi.spfy_spmma(_DT[comp.dtype], op_b, m, n, k, float(alpha), _ptr(comp.vals), _ptr(comp.meta),
                        _ptr(b), b.stride(0), float(beta), _ptr(c), c.stride(0) if c is not None else 0,
                        _ptr(out), out.stride(0), None, 0, _stream())
    else:
        epi = epilogue._c(m)
        capi.spfy_spmma_ex(_DT[comp.dtype], op_b, m, n, k, float(alpha), _ptr(comp.vals), _ptr(comp.meta),
                           _ptr(b), b.stride(0), float(beta), _ptr(c), c.stride(0) if c is not None else 0,
                           _ptr(out), out.stride(0), None, 0, ctypes.byref(epi), _stream())
    return out


def permute_conv_weights(w, c, kh, kw):
    """[m, c*kh*kw] conv weights in (c, kh, kw) column order (a flattened torch conv weight, the K order of `unfold`)
    -> [m, kh*kw*c] in (kh, kw, c) order, the K order of spmma_conv.  Do this BEFORE pruning."""
    out = torch.empty_like(w)
    capi.spfy_permute_conv_weights(_ptr(w), _ptr(out), w.shape[0], c, kh, kw, _stream())
    return out


def spmma_conv(comp, x, kh, kw, stride=1, pad=0, c=None, out=None, alpha=1.0, beta=0.0, epilogue=None):
    """Implicit GEMM (spfy_spmma_conv): D[m, batch*ho*wo] = alpha * A(2:4) * im2col(x) + beta * C with x the NHWC
    activation tensor [batch, h, w, ch] -- the unfolded K x N operand of datasets/get_shapes.py:29-41 is never built.
    `comp`: compressed weights whose K is ordered (kh, kw, ch) (permute_conv_weights before prune24).
    epilogue: an Epilogue applied before D is written (spfy_spmma_conv_ex)."""
    assert x.dim() == 4 and x.is_contiguous()
    nb, h, w, ch = x.shape
    ho, wo = (h + 2 * pad - kh) // stride + 1, (w + 2 * pad - kw) // stride + 1
    assert comp.cols == kh * kw * ch
    n = nb * ho * wo
    if out is None:
        out = torch.empty(comp.rows, n, dtype=comp.dtype, device=x.device)
    desc = capi.ConvDesc(nb, h, w, ch, kh, kw, stride, pad)
    if epilogue is None:
        capi.spfy_spmma_conv(_DT[comp.dtype], ctypes.byref(desc), comp.rows, float(alpha), _ptr(comp.vals),
                             _ptr(comp.meta), _ptr(x), float(beta), _ptr(c), c.stride(0) if c is not None else 0, _ptr(out),
                             out.stride(0), _stream())
    else:
        epi = epilogue._c(comp.rows)
        capi.spfy_spmma_conv_ex(_DT[comp.dtype], ctypes.byref(desc), comp.rows, float(alpha), _ptr(comp.vals),
                                _ptr(comp.meta), _ptr(x), float(beta), _ptr(c), c.stride(0) if c is not None else 0,
                                _ptr(out), out.stride(0), 0, ctypes.byref(epi), _stream())
    return out


def spmma_conv_nhwc(comp, x, kh, kw, stride=1, pad=0, out=None, alpha=1.0, c=None, beta=0.0, epilogue=None):
    """spfy_spmma_conv_nhwc: the same implicit GEMM with the result in NHWC, [batch, ho, wo, m] -- the `x` of the next
    layer, so a chain of convolutions never transposes or unfolds anything.
    epilogue (an Epilogue), c / beta (beta * C with C in NHWC like the result, e.g. the shortcut of a residual block; `c`
    may be `out`) go through spfy_spmma_conv_ex: conv + batch norm + shortcut + ReLU in one pass over the output."""
    assert x.dim() == 4 and x.is_contiguous()
    nb, h, w, ch = x.shape
    ho, wo = (h + 2 * pad - kh) // stride + 1, (w + 2 * pad - kw) // stride + 1
    assert comp.cols == kh * kw * ch
    if out is None:
        out = torch.empty(nb, ho, wo, comp.rows, dtype=comp.dtype, device=x.device)
    assert out.is_contiguous() and out.numel() == nb * ho * wo * comp.rows
    desc = capi.ConvDesc(nb, h, w, ch, kh, kw, stride, pad)
    if epilogue is None and c is None and beta == 0.0:
        capi.spfy_spmma_conv_nhwc(_DT[comp.dtype], ctypes.byref(desc), comp.rows, float(alpha), _ptr(comp.vals),
                                  _ptr(comp.meta), _ptr(x), _ptr(out), comp.rows, _stream())
        return out
    if c is not None:
        assert c.shape[-1] == comp.rows and c.numel() == out.numel()
        c = c if c.dim() == 2 else c.view(-1, comp.rows)
    epi = (epilogue or Epilogue())._c(comp.rows)
    capi.spfy_spmma_conv_ex(_DT[comp.dtype], ctypes.byref(desc), comp.rows, float(alpha), _ptr(comp.vals), _ptr(comp.meta),
                            _ptr(x), float(beta), _ptr(c), c.stride(0) if c is not None else 0, _ptr(out), comp.rows,
                            capi.OUT_T, ctypes.byref(epi), _stream())
    return out


def spmma(a, b, c, m, n, k, batch_size=1, transpose_a=capi.OP_N, transpose_b=capi.OP_N, alpha=1.0,
          beta=0.0, prune_mode=capi.PRUNE_TILE_MAG):
    """sparsifyme::spmma (spmma.hxx:21-118): prune A in place (2:4 magnitude), compress, multiply
    into C (D aliases C, :52-53).  Returns [prune_ms, compress_ms, mul_ms] like :117.  Like the header
    (include/sparsify.me/spmma.hxx) it prunes with TILE_MAG, the algorithm the reference requests from
    cusparseLt (:86); prune_mode=PRUNE_STRIP_MAG is the header's -DSPARSIFYME_PRUNE_STRIP.  Prune and
    compress are timed together under `prune`; `compress` only times the (empty) remainder;
    batch_size is accepted and unused exactly like the reference (:29)."""
    del batch_size
    if transpose_a != capi.OP_N:
        raise capi.SpfyError(capi.E_UNSUPPORTED, "spmma", "transpose_a is not supported")
    if m % 8 or n % 8 or k % 8:  # spmma.hxx:45-49 (warning only, execution continues)
        print("Invalid matrix sizes for data type __half. Rows and columns must be divisible by 8.", file=sys.stderr)
    a2 = a.view(-1)[: m * k].view(m, k)
    b2 = b.view(-1)[: k * n].view(k, n) if transpose_b == capi.OP_N else b.view(-1)[: k * n].view(n, k)
    c2 = c.view(-1)[: m * n].view(m, n)
    vb, mb = compressed_bytes(a.dtype, m, k)
    t = _Timer()
    t.begin()
    comp = Compressed24(torch.empty(vb, dtype=torch.uint8, device=a.device),
                        torch.empty(mb, dtype=torch.uint8, device=a.device), m, k, a.dtype,
                        capi.LAYOUT_SM100)
    prune24(a2, inplace=True, out=comp, mode=prune_mode)
    prune_ms = t.end()
    t.begin()
    compress_ms = t.end()
    t.begin()
    spmma_compressed(comp, b2, c=c2 if beta != 0.0 else None, out=c2, alpha=alpha, beta=beta,
                     op_b=transpose_b)
    mul_ms = t.end()
    return [prune_ms, compress_ms, mul_ms]


# ------------------------------------------------------------------- unstructured path
def threshold_to_coo(a, threshold, capacity=None, want_csr=False, sync=True):
    """Unstructured magnitude prune: keep x iff |x| > threshold; COO sorted by (row, col),
    fp32 values, int32 indices (the operand format of spmm.hxx:165-168).
    Returns (row_idx, col_idx, vals, nnz[, row_ptr]); index/value tensors are trimmed to nnz.
    sync=False skips the nnz read-back: the arrays keep their full capacity, nnz is a device tensor and
    row_ptr is always returned (feed it to batched.csr, which needs no host-side nnz)."""
    rows, cols = a.shape
    cap = rows * cols if capacity is None else capacity
    dev = a.device
    ri = torch.empty(cap, dtype=torch.int32, device=dev)
    ci = torch.empty(cap, dtype=torch.int32, device=dev)
    va = torch.empty(cap, dtype=torch.float32, device=dev)
    nnz = torch.zeros(1, dtype=torch.int64, device=dev)
    rp = torch.empty(rows + 1, dtype=torch.int32, device=dev)
    wb = ctypes.c_size_t()
    capi.spfy_threshold_workspace_bytes(rows, cols, ctypes.byref(wb))
    ws = torch.empty(max(wb.value, 16), dtype=torch.uint8, device=dev)
    capi.spfy_threshold_to_coo(_dtype_code(a), _ptr(a), a.stride(0), rows, cols, float(threshold),
                               _ptr(ri), _ptr(ci), _ptr(va), cap, _ptr(nnz), _ptr(rp), _ptr(ws),
                               ws.numel(), _stream())
    if not sync:
        return ri, ci, va, nnz, rp
    n = int(nnz.item())
    kept = min(n, cap)
    res = (ri[:kept], ci[:kept], va[:kept], n)
    return res + (rp,) if want_csr else res


def coo_to_csr(row_idx, rows):
    rp = torch.empty(rows + 1, dtype=torch.int32, device=row_idx.device)
    capi.spfy_coo_to_csr(_ptr(row_idx), row_idx.numel(), rows, _ptr(rp), _stream())
    return rp


class batched:
    """namespace sparsifyme::batched"""

    @staticmethod
    def strided_coo(a_num_rows, a_num_cols, a_nnz, b_num_rows, b_num_cols, num_batches, a_rows, a_cols,
                    a_values, b, c, alpha=1.0, beta=0.0, alg=capi.SPMM_ALG_DEFAULT):
        """batched::strided_coo (spmm.hxx:140-193): C_b = alpha*A*B_b + beta*C_b with ONE COO A
        (row-sorted), B_b = b[i] k x n column-major (ldb = k), C_b m x n column-major (ldc = m);
        b and c are single slabs strided by ldb*n / ldc*n (:172,:175 intent).  Returns ms.
        `alg`: SPMM_ALG_* of spfy_b200.h (DEFAULT: tensor cores when A is dense enough to pay)."""
        assert b_num_rows == a_num_cols
        ldb, ldc = b_num_rows, a_num_rows
        wb = ctypes.c_size_t()
        capi.spfy_spmm_workspace_bytes(alg, a_num_rows, a_num_cols, b_num_cols, num_batches, a_nnz, ctypes.byref(wb))
        ws = _workspace(wb.value, b.device)
        t = _Timer()
        t.begin()
        capi.spfy_spmm_coo_strided_batched(alg, a_num_rows, a_num_cols, a_nnz, b_num_cols, num_batches,
                                           _ptr(a_rows), _ptr(a_cols), _ptr(a_values), _ptr(b), ldb,
                                           ldb * b_num_cols, _ptr(c), ldc, ldc * b_num_cols,
                                           float(alpha), float(beta), _ptr(ws), ws.numel(), _stream())
        return t.end()

    @staticmethod
    def csr(m, k, n, num_batches, row_ptr, col_idx, vals, b, c, alpha=1.0, beta=0.0, alg=capi.SPMM_ALG_DEFAULT):
        wb = ctypes.c_size_t()
        capi.spfy_spmm_workspace_bytes(alg, m, k, n, num_batches, col_idx.numel(), ctypes.byref(wb))
        ws = _workspace(wb.value, b.device)
        capi.spfy_spmm_csr_strided_batched(alg, m, k, n, num_batches, _ptr(row_ptr), _ptr(col_idx),
                                           _ptr(vals), _ptr(b), k, k * n, _ptr(c), m, m * n,
                                           float(alpha), float(beta), _ptr(ws), ws.numel(), _stream())

    @staticmethod
    def spmm(col_idx_list, values_list, b, c_list, m, n, k, block, ell_cols, alpha=1.0, beta=0.0,
             alg=capi.SPMM_ALG_DEFAULT):
        """batched::spmm (spmm.hxx:30-138): per batch C_b = alpha*A_b*B + beta*C_b, A_b blocked-ELL
        (containers/ell.hxx:24-33), B k x n column-major shared, C_b m x n column-major.
        One launch covers every batch element (the reference fans out one host thread +
        stream per batch, :94-115).  Returns ms."""
        dev = b.device
        nb = len(values_list)
        ci = torch.tensor([t.data_ptr() for t in col_idx_list], dtype=torch.int64, device=dev)
        va = torch.tensor([t.data_ptr() for t in values_list], dtype=torch.int64, device=dev)
        cs = torch.tensor([t.data_ptr() for t in c_list], dtype=torch.int64, device=dev)
        wb = ctypes.c_size_t()
        capi.spfy_spmm_bell_workspace_bytes(alg, _dtype_code(b), m, k, n, nb, ctypes.byref(wb))
        ws = _workspace(wb.value, dev)
        t = _Timer()
        t.begin()
        capi.spfy_spmm_bell_batched(alg, _dtype_code(b), m, k, n, block, ell_cols, nb, _ptr(ci), _ptr(va),
                                    _ptr(b), k, _ptr(cs), m, float(alpha), float(beta), _ptr(ws), ws.numel(),
                                    _stream())
        return t.end()


    @staticmethod
    def gemm(a, b, c, m, n, k, transpose_a=capi.OP_N, transpose_b=capi.OP_N, alpha=1.0, beta=0.0,
             precision=capi.GEMM_PRECISE, strided=True):
        """batched::gemm (gemm.hxx:25-195): column-major C_i[m x n] = alpha*op(A_i)*op(B_i) + beta*C_i on tcgen05
        (fp16 / bf16: kind::f16; fp32: 3xTF32, or one TF32 product with precision=GEMM_FAST).
        a: [nb, ...] slab of column-major operands (or a single matrix shared by the batch), same for b;
        c: [nb, n, m] slab (column-major m x n per batch).  lda = m (k if transposed), ldb = k (n), ldc = m (:79-81).
        strided=False goes through the pointer-array entry (what the header template calls).  Returns ms."""
        nb = c.shape[0]
        lda = m if transpose_a == capi.OP_N else k
        ldb = k if transpose_b == capi.OP_N else n
        sa = a.stride(0) if a.dim() == 3 and a.shape[0] == nb and nb > 1 else 0
        sb = b.stride(0) if b.dim() == 3 and b.shape[0] == nb and nb > 1 else 0
        t = _Timer()
        wb = ctypes.c_size_t()
        capi.spfy_gemm_workspace_bytes(_dtype_code(c), transpose_a, transpose_b, m, n, k, lda, ldb, nb, ctypes.byref(wb))
        ws = _workspace(wb.value, c.device)
        if strided:
            t.begin()
            capi.spfy_gemm_strided_batched(_dtype_code(c), precision, transpose_a, transpose_b, m, n, k, float(alpha),
                                           _ptr(a), lda, sa, _ptr(b), ldb, sb, float(beta), _ptr(c), m, c.stride(0), nb,
                                           _ptr(ws), ws.numel(), _stream())
            return t.end()
        es = a.element_size()
        pa = (ctypes.c_void_p * nb)(*[a.data_ptr() + i * sa * es for i in range(nb)])
        pb = (ctypes.c_void_p * nb)(*[b.data_ptr() + i * sb * es for i in range(nb)])
        pc = (ctypes.c_void_p * nb)(*[c.data_ptr() + i * c.stride(0) * es for i in range(nb)])
        t.begin()
        capi.spfy_gemm_batched(_dtype_code(c), precision, transpose_a, transpose_b, m, n, k, float(alpha),
                               ctypes.cast(pa, ctypes.c_void_p), lda, ctypes.cast(pb, ctypes.c_void_p), ldb, float(beta),
                               ctypes.cast(pc, ctypes.c_void_p), m, nb, _ptr(ws), ws.numel(), _stream())
        return t.end()
