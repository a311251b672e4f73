"""The 2:4 fine-tuning path at the shapes and values where its kernels can go wrong.

transpose24: c != m filters, 5x5 and 7x7 taps, a tap boundary inside a 16-column unit, 8-row operands, and the validity
flag when the unbalanced block sits in a tile after the first wave of CTAs.  Data gradients of stride-1 convolutions and
ragged Linear layers against fp64.  recompress24: all six (input, operand) dtype pairs on infinities, overflow, subnormals,
ties, signed zeros and NaNs, strided, misaligned and in-place.  Linear24 per element against fp64, including the 16-bit
rounding of dW, its overflow to inf and torch.amp.GradScaler skipping that step.

Every arithmetic result is checked per element against fp64 computed from the exact 16-bit operands the kernel read:
    |got - ref| <= u |ref| + K 2^-23 (|A| |B|) + eta
u: one rounding of the output (2^-11 fp16, 2^-8 bf16, 2^-24 fp32); K: the reduction length, with a bias counted as one
more term; the K term bounds fp32 accumulation even when every addition truncates; eta: half the smallest subnormal of
the output type, for results that underflow.  Byte-level results are compared with the CPU oracle."""
import functools

import numpy as np
import pytest
import torch

from test_gpu_parity import bits_of, to_dev
from test_gpu_transpose24 import operand_from_mask, poisoned_out, prune_dev, zero_free
from test_transpose24 import expected_sm100, move_kept_pair

pytestmark = pytest.mark.gpu

TDT = {0: torch.float16, 1: torch.bfloat16}
U = {torch.float16: 2.0 ** -11, torch.bfloat16: 2.0 ** -8, torch.float32: 2.0 ** -24}
ETA = {torch.float16: 2.0 ** -25, torch.bfloat16: 2.0 ** -134, torch.float32: 2.0 ** -150}


def assert_bound(got, ref, absprod, k, dtype, what):
    """|got - ref| <= U[dtype] |ref| + k 2^-23 absprod + ETA[dtype], element by element (a NaN fails)"""
    got = got.detach().double()
    assert got.shape == ref.shape, what
    bound = U[dtype] * ref.abs() + k * 2.0 ** -23 * absprod + ETA[dtype]
    err = (got - ref).abs()
    bad = ~(err <= bound)
    if bool(bad.any()):
        i = int(torch.nan_to_num(err / bound, nan=float("inf")).flatten().argmax())
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} elements outside the bound; worst: got "
                             f"{got.flatten()[i].item()!r}, fp64 {ref.flatten()[i].item()!r}, "
                             f"bound {bound.flatten()[i].item()!r}")


# ------------------------------------------------------------------ transpose24
def padding_of(orc, rows, cols):
    """(value bytes, metadata nibbles) that are padding in the SM100 image of a rows x cols operand"""
    g = cols // 4
    pv, pm = orc.pack_sm100(np.full((rows, 2 * g), 0xFFFF, np.uint16), np.full((rows, (g + 1) // 2), 0xFF, np.uint8),
                            rows, cols)
    return pv == 0, np.stack([pm & 0xF, pm >> 4]) == 4


def nibbles(meta):
    return np.stack([meta & 0xF, meta >> 4])


# (rows, cols, taps): A is rows x taps*C.  Filters with c != m; 5x5 and 7x7; rows = 8 (mod 16) with taps > 1, so one
# 16-column unit of A' takes its four groups from two taps; the smallest operands.
TRANSPOSE_CASES = [(128, 9 * 64, 9), (64, 9 * 128, 9), (72, 9 * 64, 9), (200, 9 * 136, 9), (136, 9 * 64, 9),
                   (64, 25 * 64, 25), (64, 49 * 64, 49), (8, 8, 1), (8, 16, 1), (8, 16, 2)]


@pytest.mark.parametrize("rows,cols,taps", TRANSPOSE_CASES)
@pytest.mark.parametrize("dt", [0, 1])
def test_transpose24_edges_byte_exact(spfy, orc, cuda, rows, cols, taps, dt):
    """A' byte-exact against the oracle from a poisoned output: padding +0 with nibble 0x4; twice gives A back"""
    bits = zero_free(orc, dt, (rows, cols), seed=rows * 7 + cols + taps + dt)
    comp, dense = prune_dev(spfy, bits, dt, cuda, spfy.PRUNE_TILE_MAG)
    want_dense, _ = orc.prune24_tile(dt, bits)
    assert np.array_equal(bits_of(dense), want_dense)
    inv = torch.full((1,), 7, dtype=torch.int32, device=cuda)
    out = spfy.transpose24(comp, taps=taps, out=poisoned_out(spfy, comp, taps, cuda), invalid=inv)
    assert int(inv.item()) == 0
    got_v, got_m = out.vals.cpu().numpy(), out.meta.cpu().numpy()
    pv, pm = padding_of(orc, cols // taps, taps * rows)
    assert (got_v[pv] == 0).all() and (nibbles(got_m)[pm] == 4).all()
    ov, om = expected_sm100(orc, dt, want_dense, taps)
    assert np.array_equal(got_v, ov) and np.array_equal(got_m, om)
    back = spfy.transpose24(out, taps=taps, out=poisoned_out(spfy, out, taps, cuda))
    assert torch.equal(back.vals, comp.vals) and torch.equal(back.meta, comp.meta)


def oracle_compressed(spfy, orc, dt, dense, dev):
    """SM100 operand of a matrix that is 2:4 along its rows, compressed by the oracle (STRIP keeps its nonzeros)"""
    rows, cols = dense.shape
    ref = orc.prune24_strip(dt, dense, want_mask=False)
    assert np.array_equal(ref["dense"], dense)
    ov, om = orc.pack_sm100(ref["vals"], ref["meta"], rows, cols)
    return spfy.Compressed24(torch.from_numpy(ov).to(dev), torch.from_numpy(om).to(dev), rows, cols, TDT[dt],
                             spfy.LAYOUT_SM100)


@functools.lru_cache(maxsize=2)
def _tile_pruned(orc, rows, cols, seed):
    bits = zero_free(orc, 0, (rows, cols), seed=seed)
    return bits, orc.prune24_tile(0, bits)[0]


@pytest.mark.parametrize("rows,cols,row,group", [
    (4096, 8192, 4095, 2047),  # A' has 2048 tiles, more than one wave (8 CTAs per SM): the block is in the last one
    (4096, 8192, 0, 0),        # the first A' tile: its CTA goes on to a tile of the second wave
    (200, 136, 199, 33),       # ragged: the last row and the last group
])
def test_transpose24_flags_one_unbalanced_block(spfy, orc, cuda, rows, cols, row, group):
    """one row of one 4x4 block keeps the other two positions: the rows stay 2:4, the columns do not; the flag is 1
    wherever that block sits, and 0 for the matrix before the move"""
    bits, dense = _tile_pruned(orc, rows, cols, seed=rows + cols)
    inv = torch.full((1,), 7, dtype=torch.int32, device=cuda)
    good, _ = prune_dev(spfy, bits, 0, cuda, spfy.PRUNE_TILE_MAG)
    spfy.transpose24(good, invalid=inv)
    assert int(inv.item()) == 0
    bad = oracle_compressed(spfy, orc, 0, move_kept_pair(dense, bits, row, group), cuda)
    spfy.transpose24(bad, invalid=inv)
    assert int(inv.item()) == 1


# ------------------------------------------------------------------ data gradients
# (m, c, k, pad, h, w): forward m output and c input channels, k x k filter, stride 1, h x w input.  The data gradient
# reads dy with m channels (a multiple of 64) and writes dx with c.
CONV_CASES = [(128, 64, 3, 1, 9, 7), (64, 72, 3, 1, 13, 11), (64, 64, 3, 0, 11, 9), (64, 64, 5, 2, 7, 9),
              (64, 64, 7, 3, 9, 9)]


@pytest.mark.parametrize("m,c,k,pad,h,w", CONV_CASES)
@pytest.mark.parametrize("dt", [0, 1])
def test_conv_data_gradient_fp64(spfy, orc, cuda, m, c, k, pad, h, w, dt):
    """dx = spmma_conv_nhwc(transpose24(comp, taps=k*k), dy, pad=k-1-pad) against fp64 conv2d_input of the pruned dense
    weight (not of the transposed operand); K = k*k*m"""
    tdt, nb = TDT[dt], 8  # n = nb * h * w, a multiple of 8
    wt = to_dev(zero_free(orc, dt, (m, c * k * k), seed=m + c + k + pad + dt), dt, cuda)
    comp, dense = prune_dev(spfy, bits_of(spfy.permute_conv_weights(wt, c, k, k)), dt, cuda, spfy.PRUNE_TILE_MAG)
    inv = torch.full((1,), 7, dtype=torch.int32, device=cuda)
    comp_t = spfy.transpose24(comp, taps=k * k, invalid=inv)
    ho, wo = h + 2 * pad - k + 1, w + 2 * pad - k + 1
    g = torch.Generator(device="cpu").manual_seed(h * w + m)
    dy = torch.randn(nb, ho, wo, m, generator=g).to(tdt).to(cuda)
    dx = spfy.spmma_conv_nhwc(comp_t, dy, k, k, stride=1, pad=k - 1 - pad)
    assert int(inv.item()) == 0 and dx.shape == (nb, h, w, c) and dx.dtype == tdt
    w_nchw = dense.double().view(m, k, k, c).permute(0, 3, 1, 2)
    dy_nchw = dy.double().permute(0, 3, 1, 2)
    ref = torch.nn.grad.conv2d_input((nb, c, h, w), w_nchw, dy_nchw, padding=pad)
    absprod = torch.nn.grad.conv2d_input((nb, c, h, w), w_nchw.abs(), dy_nchw.abs(), padding=pad)
    assert_bound(dx.permute(0, 3, 1, 2), ref, absprod, k * k * m, tdt, "dx")


def test_conv_data_gradient_refuses_channels_not_a_multiple_of_64(spfy, orc, cuda):
    """a layer with 72 output channels: its data gradient would read dy with 72 channels, which the im2col gather
    cannot take; refused before any launch"""
    m, c = 72, 64
    comp, _ = prune_dev(spfy, zero_free(orc, 0, (m, 9 * c), seed=5), 0, cuda, spfy.PRUNE_TILE_MAG)
    comp_t = spfy.transpose24(comp, taps=9)
    dy = torch.zeros(8, 7, 7, m, dtype=torch.float16, device=cuda)
    before = spfy.launch_count()
    with pytest.raises(spfy.SpfyError) as e:
        spfy.spmma_conv_nhwc(comp_t, dy, 3, 3, stride=1, pad=1)
    assert e.value.code == spfy.capi.E_UNSUPPORTED and spfy.launch_count() == before


LINEAR_CASES = [(136, 208, 200), (8, 48, 72)]  # (tokens, in, out): neither width a multiple of 128


@pytest.mark.parametrize("tokens,in_f,out_f", LINEAR_CASES)
@pytest.mark.parametrize("dt", [0, 1])
def test_linear_data_gradient_fp64(spfy, orc, cuda, tokens, in_f, out_f, dt):
    """dx = dy W through transpose24(comp) against fp64; K = out"""
    tdt = TDT[dt]
    comp, dense = prune_dev(spfy, zero_free(orc, dt, (out_f, in_f), seed=tokens + in_f + dt), dt, cuda,
                            spfy.PRUNE_TILE_TRANSPOSABLE)
    g = torch.Generator(device="cpu").manual_seed(tokens)
    dy = torch.randn(tokens, out_f, generator=g).to(tdt).to(cuda)
    dx = spfy.spmma_compressed(spfy.transpose24(comp), dy, op_b=spfy.OP_T, out_t=True)
    assert dx.shape == (tokens, in_f) and dx.dtype == tdt
    wd, dyd = dense.double(), dy.double()
    assert_bound(dx, dyd @ wd, dyd.abs() @ wd.abs(), out_f, tdt, "dx")


# ------------------------------------------------------------------ recompress24
F32_SPECIAL = [
    0x7F800000, 0xFF800000,                                      # +-inf
    0x477FE000, 0x477FEFFF, 0x477FF000, 0xC77FF000, 0x47800000,  # fp16: 65504, just below the tie to inf, the tie, 2^16
    0x7F7F7FFF, 0x7F7F8000, 0x7F7FFFFF, 0xFF7F7FFF,              # bf16: below max, the tie to inf, FLT_MAX
    0x33800000, 0x33000000, 0x33000001, 0x33C00000, 0xB3C00000,  # fp16 subnormals: 2^-24, ties at 2^-25 and 3 2^-25
    0x387FC000, 0x2EDBE6FF,                                      # the largest fp16 subnormal; 1e-10 -> 0
    0x00012345, 0x00008000, 0x00018000, 0x80018000, 0x00000001,  # fp32 subnormals: bf16 subnormals, ties, 0
    0x3F801000, 0x3F803000, 0x3F808000, 0x3F818000, 0xBF818000,  # ties: fp16 down, fp16 up, bf16 down, bf16 up
    0x80000000, 0x00000000,                                      # -0, +0
    0x7FC00000, 0xFFC00000, 0x7F800001, 0x7F800100, 0xFF80FFFF, 0x7FFFFFFF,  # NaNs, some with payload in the low half
]
F16_SPECIAL = [
    0x7C00, 0xFC00, 0x7BFF, 0xFBFF, 0x7BFE,          # +-inf, +-max (bf16: rounds up to 2^16)
    0x0001, 0x8001, 0x0003, 0x03FF, 0x0201,          # subnormals
    0x3C04, 0x3C0C, 0xBC0C,                          # ties for bf16
    0x8000, 0x0000,
    0x7E00, 0xFE00, 0x7C01, 0xFC01, 0x7C10, 0x7FFF,  # NaNs
]
BF16_SPECIAL = [
    0x7F80, 0xFF80, 0x7F7F, 0x477F, 0xC77F, 0x4780,  # +-inf, max, fp16: just below 65504, 2^16 -> inf
    0x3380, 0x3300, 0x3340, 0x33C0, 0xB3C0, 0x387F,  # fp16 subnormals, ties at 2^-25 and 3 2^-25
    0x0001, 0x8001, 0x2EDC, 0x3F81,                  # bf16 subnormals and 1e-10 flush to +-0 in fp16
    0x8000, 0x0000,
    0x7FC0, 0xFFC0, 0x7F81, 0xFF81, 0x7FFF,          # NaNs
]
SPECIAL = {torch.float32: np.array(F32_SPECIAL, np.uint32), torch.float16: np.array(F16_SPECIAL, np.uint16),
           torch.bfloat16: np.array(BF16_SPECIAL, np.uint16)}


def raw_of(t):
    """the bits of a tensor (fp32 -> uint32, 16-bit -> uint16) as numpy"""
    if t.dtype == torch.float32:
        return t.contiguous().view(torch.int32).cpu().numpy().view(np.uint32)
    return bits_of(t)


def from_raw(raw, dtype):
    if dtype == torch.float32:
        return torch.from_numpy(raw.view(np.int32).copy()).view(torch.float32)
    return torch.from_numpy(raw.view(np.int16).copy()).view(dtype)


def raw_to_f32(raw, dtype):
    """exact: every fp16 and bf16 value is an fp32 value"""
    if dtype == torch.float32:
        return raw.view(np.float32)
    if dtype == torch.float16:
        return raw.view(np.float16).astype(np.float32)
    return (raw.astype(np.uint32) << 16).view(np.float32)


def rne16(x32, dtype):
    """fp32 -> fp16 / bf16 bits, round to nearest even; a NaN stays a NaN"""
    if dtype == torch.float16:
        with np.errstate(over="ignore", invalid="ignore"):
            return x32.astype(np.float16).view(np.uint16)
    b = x32.view(np.uint32).astype(np.uint64)
    r = ((b + 0x7FFF + ((b >> 16) & 1)) >> 16).astype(np.uint16)
    return np.where(np.isnan(x32), np.uint16(0x7FC0), r)


def canon_nan(bits16, dtype):
    """every fp16 / bf16 NaN -> one pattern: a NaN must stay a NaN, its payload and sign are not compared"""
    exp, man, nan = (0x7C00, 0x03FF, 0x7E00) if dtype == torch.float16 else (0x7F80, 0x007F, 0x7FC0)
    return np.where(((bits16 & exp) == exp) & ((bits16 & man) != 0), np.uint16(nan), bits16)


def special_input(dtype, keep, seed):
    """zero-free values with every special value of `dtype` at a kept and at a pruned position, and at a quarter of
    the rest at random"""
    rows, cols = keep.shape
    rng = np.random.default_rng(seed)
    base = rng.uniform(0.25, 1.0, keep.shape) * rng.choice([-1.0, 1.0], keep.shape)
    raw = raw_of(torch.from_numpy(base.astype(np.float32)).to(dtype)).copy()
    pool = SPECIAL[dtype]
    pick = rng.random(keep.shape) < 0.25
    raw[pick] = pool[rng.integers(0, len(pool), int(pick.sum()))]
    flat = raw.reshape(-1)
    flat[np.flatnonzero(keep.reshape(-1))[: len(pool)]] = pool
    flat[np.flatnonzero(~keep.reshape(-1))[: len(pool)]] = pool
    return raw


RC_PAIRS = [(torch.float32, 0), (torch.float32, 1), (torch.float16, 0), (torch.float16, 1), (torch.bfloat16, 0),
            (torch.bfloat16, 1)]
RC_LAYOUTS = ["contiguous", "column_slice", "offset_by_one", "small", "in_place"]


@pytest.mark.parametrize("layout", RC_LAYOUTS)
@pytest.mark.parametrize("in_dtype,dt", RC_PAIRS, ids=["f32-f16", "f32-bf16", "f16-f16", "f16-bf16", "bf16-f16",
                                                      "bf16-bf16"])
def test_recompress24_special_values(spfy, orc, cuda, in_dtype, dt, layout):
    """The mask of a zero-free TILE prune; then values and masked copy of a different input full of special values.
    comp.vals == pack_sm100(operand_from_mask(input rounded to nearest even, keep)), byte for byte (the input's own bits
    when the dtypes match, NaNs compared as NaNs otherwise), padding +0 over a poisoned buffer, metadata untouched;
    masked_out == the input's bits with +0 at every pruned position (a kept -0 stays -0, a pruned -0 becomes +0).
    Layouts: ld_in > cols, a base one element off 16 bytes (the scalar path), ragged rows and cols, and values and
    masked_out in one aliased call, as Linear24.refresh() makes it."""
    tdt = TDT[dt]
    rows, cols = (8, 24) if layout == "small" else (130, 260)
    mbits = zero_free(orc, dt, (rows, cols), seed=rows + cols + 3 * dt)
    comp, dense = prune_dev(spfy, mbits, dt, cuda, spfy.PRUNE_TILE_MAG)
    want_dense, mask = orc.prune24_tile(dt, mbits)
    assert np.array_equal(bits_of(dense), want_dense)
    keep = mask.astype(bool)
    meta0 = comp.meta.clone()
    raw = special_input(in_dtype, keep, seed=rows * cols + dt + 17 * len(layout))
    x_cpu = from_raw(raw, in_dtype)
    fence = None
    if layout == "column_slice":
        x = torch.full((rows, cols + 40), 7.0, dtype=in_dtype, device=cuda)[:, 16:16 + cols]
        fence = torch.full((rows, cols + 24), 5.0, dtype=in_dtype, device=cuda)
        out = fence[:, 8:8 + cols]
    elif layout == "offset_by_one":
        x = torch.full((rows * cols + 1,), 7.0, dtype=in_dtype, device=cuda)[1:].view(rows, cols)
        fence = torch.full((rows * cols + 1,), 5.0, dtype=in_dtype, device=cuda)
        out = fence[1:].view(rows, cols)
    else:
        x = torch.empty(rows, cols, dtype=in_dtype, device=cuda)
        out = x if layout == "in_place" else torch.full_like(x, 5.0)
    x.copy_(x_cpu)
    comp.vals.fill_(0xAB)
    spfy.recompress24(x, comp, masked_out=out)
    conv = raw if in_dtype == tdt else rne16(raw_to_f32(raw, in_dtype), tdt)
    ov, om = orc.pack_sm100(*operand_from_mask(conv, keep), rows, cols)
    got = comp.vals.cpu().numpy()
    if in_dtype == tdt:
        assert np.array_equal(got, ov)
    else:
        assert np.array_equal(canon_nan(got.view(np.uint16), tdt), canon_nan(ov.view(np.uint16), tdt))
    assert torch.equal(comp.meta, meta0) and np.array_equal(meta0.cpu().numpy(), om)
    assert np.array_equal(raw_of(out), np.where(keep, raw, 0).astype(raw.dtype))
    if layout != "in_place":
        assert np.array_equal(raw_of(x), raw)
    if fence is not None:  # nothing written outside masked_out
        f = raw_of(fence)
        five = raw_of(torch.full((1,), 5.0, dtype=in_dtype))[0]
        rest = f.copy()
        if layout == "column_slice":
            rest[:, 8:8 + cols] = five
        else:
            rest[1:] = five
        assert (rest == five).all()


# ------------------------------------------------------------------ Linear24
def make_layer(spfy, cuda, in_f, out_f, tdt, bias, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    w = torch.randn(out_f, in_f, generator=g) * 0.05
    b = torch.randn(out_f, generator=g).to(cuda) if bias else None
    return spfy.Linear24.from_dense(w.to(cuda), b, dtype=tdt), g


def w16(layer):
    """the dense weight the kernels read: the masked fp32 master rounded to the layer's dtype (what comp holds)"""
    return layer.weight.detach().to(layer.dtype).double()


def assert_weight_grad(layer, dyd, xd, what):
    """dW = mask * 16-bit(dy^T x), then fp32: per element against fp64 (K = tokens), exactly +0 where pruned"""
    keep = layer.weight.detach() != 0
    gw = layer.weight.grad
    assert gw.dtype == torch.float32
    assert torch.equal(gw, gw.to(layer.dtype).float()), f"{what}: dW is not a {layer.dtype} value"
    ref = torch.where(keep, dyd.T @ xd, torch.zeros((), dtype=torch.float64, device=xd.device))
    assert_bound(gw, ref, dyd.abs().T @ xd.abs(), dyd.shape[0], layer.dtype, what)
    assert bool((gw[~keep] == 0).all()) and not bool(torch.signbit(gw[~keep]).any())


@pytest.mark.parametrize("bias", [True, False])
@pytest.mark.parametrize("dt", [0, 1])
@pytest.mark.parametrize("tokens,in_f,out_f", LINEAR_CASES)
def test_linear24_per_element(spfy, cuda, tokens, in_f, out_f, dt, bias):
    """y, dx, dW and db of Linear24 per element against fp64 (K = in + 1 with the bias, out, tokens, tokens)"""
    tdt = TDT[dt]
    layer, g = make_layer(spfy, cuda, in_f, out_f, tdt, bias, seed=tokens + dt)
    x = torch.randn(2, tokens // 2, in_f, generator=g).to(tdt).to(cuda).requires_grad_(True)
    y = layer(x)
    assert y.shape == (2, tokens // 2, out_f) and y.dtype == tdt
    wd, xd = w16(layer), x.detach().double().reshape(tokens, in_f)
    bd = layer.bias.detach().double() if bias else torch.zeros(out_f, dtype=torch.float64, device=cuda)
    assert_bound(y.reshape(tokens, out_f), xd @ wd.T + bd, xd.abs() @ wd.abs().T + bd.abs(), in_f + 1, tdt, "y")
    dy = torch.randn(y.shape, generator=g).to(tdt).to(cuda)
    y.backward(dy)
    dyd = dy.double().reshape(tokens, out_f)
    assert_bound(x.grad.reshape(tokens, in_f), dyd @ wd, dyd.abs() @ wd.abs(), out_f, tdt, "dx")
    assert_weight_grad(layer, dyd, xd, "dW")
    if bias:
        assert_bound(layer.bias.grad, dyd.sum(0), dyd.abs().sum(0), tokens, torch.float32, "db")


@pytest.mark.parametrize("dt", [0, 1])
def test_linear24_gradient_combinations(spfy, cuda, dt):
    """a frozen weight gets dx only, an x without grad dW only: each backward launches exactly the kernels of the
    gradients it returns"""
    tokens, in_f, out_f = 136, 208, 200
    tdt = TDT[dt]
    layer, g = make_layer(spfy, cuda, in_f, out_f, tdt, True, seed=11 + dt)
    x = torch.randn(tokens, in_f, generator=g).to(tdt).to(cuda)
    dy = torch.randn(tokens, out_f, generator=g).to(tdt).to(cuda)
    wd, xd, dyd = w16(layer), x.double(), dy.double()

    def backward(x_in):
        y = layer(x_in)
        before = spfy.launch_count()
        y.backward(dy)
        return spfy.launch_count() - before

    before = spfy.launch_count()
    spfy.spmma_compressed(layer.comp_t, dy, op_b=spfy.OP_T, out_t=True)
    n_dx = spfy.launch_count() - before

    layer.weight.requires_grad_(False)
    xg = x.clone().requires_grad_(True)
    assert backward(xg) == n_dx
    assert layer.weight.grad is None
    assert_bound(xg.grad, dyd @ wd, dyd.abs() @ wd.abs(), out_f, tdt, "dx, frozen weight")
    assert_bound(layer.bias.grad, dyd.sum(0), dyd.abs().sum(0), tokens, torch.float32, "db, frozen weight")

    layer.weight.requires_grad_(True)
    layer.bias.grad = None
    n_dw = backward(x)
    assert x.grad is None
    assert_weight_grad(layer, dyd, xd, "dW, x without grad")

    layer.weight.grad = None
    xg = x.clone().requires_grad_(True)
    assert backward(xg) == n_dx + n_dw
    assert_bound(xg.grad, dyd @ wd, dyd.abs() @ wd.abs(), out_f, tdt, "dx")
    assert_weight_grad(layer, dyd, xd, "dW")


@pytest.mark.parametrize("dt", [0, 1])
def test_linear24_non_contiguous(spfy, cuda, dt):
    """x a strided view; dy the expanded ones of y.sum(), then the gradient of a strided slice of y"""
    tokens, in_f, out_f = 136, 208, 200
    tdt = TDT[dt]
    layer, g = make_layer(spfy, cuda, in_f, out_f, tdt, True, seed=23 + dt)
    xbig = torch.randn(2, tokens // 2, 2 * in_f, generator=g).to(tdt).to(cuda).requires_grad_(True)
    x = xbig[..., ::2]
    assert not x.is_contiguous()
    wd, xd = w16(layer), x.detach().double().reshape(tokens, in_f)
    picked = torch.zeros(tokens, out_f, dtype=torch.float64, device=cuda)
    r = torch.randn(picked[::2, 1::3].shape, generator=g).to(tdt).to(cuda)
    picked[::2, 1::3] = r.double()
    for name, loss_of, dyd in (
            ("y.sum()", lambda y: y.sum(), torch.ones(tokens, out_f, dtype=torch.float64, device=cuda)),
            ("strided slice of y", lambda y: (y.reshape(tokens, out_f)[::2, 1::3] * r).sum(), picked)):
        xbig.grad = layer.weight.grad = layer.bias.grad = None
        loss_of(layer(x)).backward()
        gx = xbig.grad.reshape(tokens, 2 * in_f)
        assert_bound(gx[:, ::2], dyd @ wd, dyd.abs() @ wd.abs(), out_f, tdt, f"dx, {name}")
        assert bool((gx[:, 1::2] == 0).all())
        assert_weight_grad(layer, dyd, xd, f"dW, {name}")
        assert_bound(layer.bias.grad, dyd.sum(0), dyd.abs().sum(0), tokens, torch.float32, f"db, {name}")


def kept_and_pruned(keep_row):
    row = keep_row.tolist()
    return row.index(True), row.index(False)


def test_linear24_weight_gradient_overflow(spfy, cuda):
    """fp16: dy^T x of +-131072 becomes +-inf in dW at kept positions (not 65504, not finite) and exactly +0 at
    pruned ones; with an inf in dy, the inf * 0 = NaN of a pruned position becomes +0 as well"""
    tokens, in_f, out_f = 8, 48, 72
    layer, g = make_layer(spfy, cuda, in_f, out_f, torch.float16, False, seed=3)
    keep = layer.weight.detach() != 0
    o, o2 = 5, 11
    ik, ip = kept_and_pruned(keep[o])
    x = torch.zeros(tokens, in_f, dtype=torch.float16, device=cuda)
    x[:, ik] = x[:, ip] = 256.0
    dy = torch.zeros(tokens, out_f, dtype=torch.float16, device=cuda)
    dy[:, o], dy[:, o2] = 64.0, -64.0
    layer(x).backward(dy)
    gw = layer.weight.grad
    ref = dy.double().T @ x.double()  # +-131072 at rows o, o2 and columns ik, ip; 0 elsewhere
    want = torch.where(keep, ref.half().float(), torch.zeros((), device=cuda))
    assert gw[o, ik].item() == float("inf") and gw[o, ip].item() == 0.0
    assert torch.equal(gw, want) and not bool(torch.signbit(gw[~keep]).any())

    layer.weight.grad = None
    x = torch.randn(tokens, in_f, generator=g).half().to(cuda)
    x[0, ip] = 0.0
    dy = torch.zeros(tokens, out_f, dtype=torch.float16, device=cuda)
    dy[0, o] = float("inf")
    layer(x).backward(dy)
    gw = layer.weight.grad
    ref = dy.double().T @ x.double()  # row o: inf * x[0], NaN where x[0] is 0
    assert bool(torch.isnan(ref[o, ip]))
    want = torch.where(keep, ref.half().float(), torch.zeros((), device=cuda))
    torch.testing.assert_close(gw, want, rtol=0, atol=0, equal_nan=True)
    assert gw[o, ip].item() == 0.0 and not bool(torch.signbit(gw[~keep]).any())


def test_linear24_grad_scaler(spfy, cuda):
    """torch.amp.GradScaler with 2^40 as the first scale: the scaled dy overflows fp16, the step is skipped, the master,
    comp and comp_t stay byte-identical and the forward runs without refresh(); the scale drops, and the next steps
    track torch in fp32 on the masked weight"""
    tokens, in_f, out_f = 136, 208, 200
    layer, g = make_layer(spfy, cuda, in_f, out_f, torch.float16, True, seed=41)
    keep = layer.weight.detach() != 0
    w_ref = layer.weight.detach().clone().requires_grad_(True)
    b_ref = layer.bias.detach().clone().requires_grad_(True)
    opt = torch.optim.SGD([layer.weight, layer.bias], lr=0.5)
    opt_ref = torch.optim.SGD([w_ref, b_ref], lr=0.5)
    scaler = torch.amp.GradScaler("cuda", init_scale=2.0 ** 40, backoff_factor=2.0 ** -30, growth_interval=1000)
    x = torch.randn(tokens, in_f, generator=g).half().to(cuda)
    target = torch.randn(tokens, out_f, generator=g).to(cuda)

    def state():
        return [layer.weight.detach().view(torch.int32).clone(), layer.bias.detach().clone(), layer.comp.vals.clone(),
                layer.comp.meta.clone(), layer.comp_t.vals.clone(), layer.comp_t.meta.clone()]

    for step in range(4):
        before = state()
        scale = scaler.get_scale()
        opt.zero_grad()
        loss = ((layer(x).float() - target) ** 2).mean()
        scaler.scale(loss).backward()
        scaler.step(opt)
        scaler.update()
        if step == 0:
            assert not bool(torch.isfinite(layer.weight.grad).all())
            assert scaler.get_scale() < scale
            assert all(torch.equal(a, b) for a, b in zip(before, state()))
            continue  # no refresh(): the next forward runs on the unchanged operands
        assert scaler.get_scale() == scale
        layer.refresh()
        opt_ref.zero_grad()
        loss_ref = ((torch.nn.functional.linear(x.float(), w_ref, b_ref) - target) ** 2).mean()
        loss_ref.backward()
        w_ref.grad.mul_(keep)
        opt_ref.step()
        assert abs(loss.item() - loss_ref.item()) <= 1e-2 * abs(loss_ref.item())
        assert bool((layer.weight.detach()[~keep] == 0).all())
        for got, want in ((layer.weight, w_ref), (layer.bias, b_ref)):
            d = (got.detach() - want.detach()).abs().max().item()
            assert d <= 1e-2 * want.detach().abs().max().item()
