"""Data gradients of strided 2:4 convolutions on the GPU: spfy_transpose24_conv byte-exact against the numpy statement of
test_conv_dgrad.py (and against transpose24 for stride 1), its validity flag, and spfy_spmma_conv_dgrad per element
against fp64 conv2d_input of the pruned dense filter -- the strided ResNet-50 layers, odd images, other strides and
filters, c != m, ragged and multi-wave grids, beta = 0 over a poisoned dX, beta = 1 in place, alpha != 1, stride 1
bitwise against the stride-1 path, and the refusals."""
import ctypes

import numpy as np
import pytest
import torch

from test_conv_dgrad import phase_order, phase_tiles
from test_gpu_parity import bits_of, to_dev
from test_gpu_train24_edges import ETA, U, assert_bound
from test_gpu_transpose24 import prune_dev, zero_free
from test_transpose24 import expected_sm100, move_kept_pair

pytestmark = pytest.mark.gpu

TDT = {0: torch.float16, 1: torch.bfloat16}


def pruned_filter(spfy, orc, cuda, m, c, k, dt, seed):
    """a TILE-transposable pruned m x (kh*kw*c) filter in (kh, kw, c) order, k = kh = kw or k = (kh, kw): (comp, dense
    bits, fp64 NCHW weight).  The values are zero-free, so TILE_MAG keeps what PRUNE_TILE_TRANSPOSABLE keeps; it stands in
    where that mode's one-pass kernel refuses the width (kh*kw*c % 16, e.g. c = 72)."""
    kh, kw = k if isinstance(k, tuple) else (k, k)
    wt = to_dev(zero_free(orc, dt, (m, c * kh * kw), seed=seed), dt, cuda)
    mode = spfy.PRUNE_TILE_TRANSPOSABLE if (c * kh * kw) % 16 == 0 else spfy.PRUNE_TILE_MAG
    comp, dense = prune_dev(spfy, bits_of(spfy.permute_conv_weights(wt, c, kh, kw)), dt, cuda, mode)
    return comp, bits_of(dense), dense.double().view(m, kh, kw, c).permute(0, 3, 1, 2)


def rand_nhwc(shape, dt, cuda, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    return torch.randn(*shape, generator=g).to(TDT[dt]).to(cuda)


def reference(w, dy, h, wd, s, p):
    """fp64 conv2d_input of w (NCHW) and dy (NHWC): (ref, |w| * |dy|), both NCHW"""
    nb, c = dy.shape[0], w.shape[1]
    dyn = dy.double().permute(0, 3, 1, 2)
    ref = torch.nn.grad.conv2d_input((nb, c, h, wd), w, dyn, stride=s, padding=p)
    absprod = torch.nn.grad.conv2d_input((nb, c, h, wd), w.abs(), dyn.abs(), stride=s, padding=p)
    return ref, absprod


def poisoned_phase_operands(spfy, comp, k, s, p, invalid):
    """spfy_transpose24_conv into buffers filled with 0xAB / 0xCD"""
    capi = spfy.capi
    m, c = comp.rows, comp.cols // (k * k)
    vb, mb = ctypes.c_size_t(), ctypes.c_size_t()
    capi.spfy_transpose24_conv_bytes(capi.F16 if comp.dtype == torch.float16 else capi.BF16, m, c, k, k, s, p,
                                     ctypes.byref(vb), ctypes.byref(mb))
    vals = torch.full((vb.value,), 0xAB, dtype=torch.uint8, device=comp.vals.device)
    meta = torch.full((mb.value,), 0xCD, dtype=torch.uint8, device=comp.vals.device)
    capi.spfy_transpose24_conv(capi.F16 if comp.dtype == torch.float16 else capi.BF16, comp.vals.data_ptr(),
                               comp.meta.data_ptr(), m, c, k, k, s, p, vals.data_ptr(), meta.data_ptr(),
                               invalid.data_ptr(), torch.cuda.current_stream().cuda_stream)
    return vals, meta


# ------------------------------------------------------------------ phase operands
# (m, c, k, stride, pad)
OPERAND_CASES = [(64, 64, 3, 2, 1), (128, 72, 3, 2, 1), (64, 128, 1, 2, 0), (72, 64, 5, 2, 2), (64, 64, 3, 3, 1),
                 (64, 64, 2, 2, 0), (64, 64, 7, 2, 3), (136, 64, 1, 3, 1), (64, 200, 3, 1, 1)]


@pytest.mark.parametrize("m,c,k,s,p", OPERAND_CASES)
@pytest.mark.parametrize("dt", [0, 1])
def test_phase_operands_byte_exact(spfy, orc, cuda, m, c, k, s, p, dt):
    comp, dense, _ = pruned_filter(spfy, orc, cuda, m, c, k, dt, seed=m + c + k * 10 + s + p + dt)
    inv = torch.full((1,), 7, dtype=torch.int32, device=cuda)
    vals, meta = poisoned_phase_operands(spfy, comp, k, s, p, inv)
    assert int(inv.item()) == 0
    got_v, got_m = vals.cpu().numpy(), meta.cpu().numpy()
    for _, _, order, first, n in phase_tiles(m, c, k, k, s, p):
        rev = np.concatenate([dense[:, t * c:(t + 1) * c] for t in order[::-1]], axis=1)
        ov, om = expected_sm100(orc, dt, rev, len(order))
        assert np.array_equal(got_v[first * 16384:(first + n) * 16384], ov)
        assert np.array_equal(got_m[first * 2048:(first + n) * 2048], om)
    op = spfy.transpose24_conv(comp, k, k, s, p)
    assert torch.equal(op.vals, vals) and torch.equal(op.meta, meta)
    # the per-phase views: the statement's phases, taps, byte ranges and shapes
    tiles = phase_tiles(m, c, k, k, s, p)
    assert len(op.phases) == len(tiles)
    for (a, b, th, tw, view), (ta, tb, order, first, n) in zip(op.phases, tiles):
        assert (a, b) == (ta, tb) and phase_order(k, k, th, tw) == order
        assert (view.rows, view.cols, view.dtype) == (c, len(order) * m, comp.dtype)
        assert view.vals.data_ptr() - op.vals.data_ptr() == first * 16384 and view.vals.numel() == n * 16384
        assert view.meta.data_ptr() - op.meta.data_ptr() == first * 2048 and view.meta.numel() == n * 2048


@pytest.mark.parametrize("k,p", [(3, 1), (5, 2), (1, 0)])
@pytest.mark.parametrize("dt", [0, 1])
def test_stride_one_is_transpose24(spfy, orc, cuda, k, p, dt):
    comp, _, _ = pruned_filter(spfy, orc, cuda, 128, 64, k, dt, seed=k + dt)
    inv = torch.full((1,), 7, dtype=torch.int32, device=cuda)
    vals, meta = poisoned_phase_operands(spfy, comp, k, 1, p, inv)
    t = spfy.transpose24(comp, taps=k * k)
    assert int(inv.item()) == 0 and torch.equal(vals, t.vals) and torch.equal(meta, t.meta)


def test_invalid_flag(spfy, orc, cuda):
    """one moved kept pair raises the flag; the filter before the move does not"""
    m, c, k = 64, 64, 3
    bits = zero_free(orc, 0, (m, k * k * c), seed=3)
    dense = orc.prune24_tile(0, bits)[0]
    inv = torch.full((1,), 7, dtype=torch.int32, device=cuda)
    good, _ = prune_dev(spfy, bits, 0, cuda, spfy.PRUNE_TILE_TRANSPOSABLE)
    spfy.transpose24_conv(good, k, k, 2, 1, invalid=inv)
    assert int(inv.item()) == 0
    moved = move_kept_pair(dense, bits, 37, 5 * (c // 4) + 3)  # tap 5 = (kh 1, kw 2): phase (0, 1)
    ref = orc.prune24_strip(0, moved, want_mask=False)
    ov, om = orc.pack_sm100(ref["vals"], ref["meta"], m, k * k * c)
    bad = spfy.Compressed24(torch.from_numpy(ov).to(cuda), torch.from_numpy(om).to(cuda), m, k * k * c, torch.float16,
                            spfy.LAYOUT_SM100)
    spfy.transpose24_conv(bad, k, k, 2, 1, invalid=inv)
    assert int(inv.item()) == 1


# ------------------------------------------------------------------ data gradients
# (m, c, k, stride, pad, h, w, batch): forward m output and c input channels on an h x w input
DGRAD_CASES = [
    # the strided layers of torchvision's ResNet-50: 3x3 stride 2 (c = m) and the 1x1 stride-2 downsample projections
    (128, 128, 3, 2, 1, 56, 56, 2), (256, 256, 3, 2, 1, 28, 28, 2), (512, 512, 3, 2, 1, 14, 14, 2),
    (512, 256, 1, 2, 0, 56, 56, 2), (1024, 512, 1, 2, 0, 28, 28, 2), (2048, 1024, 1, 2, 0, 14, 14, 2),
    # odd and non-square images
    (64, 64, 3, 2, 1, 7, 9, 3), (128, 64, 3, 2, 1, 13, 7, 1), (64, 128, 1, 2, 0, 9, 13, 2),
    # other filters and strides
    (64, 64, 5, 2, 2, 11, 10, 2), (64, 64, 3, 3, 1, 13, 10, 2), (64, 128, 2, 2, 0, 8, 9, 2), (64, 64, 7, 2, 3, 15, 15, 1),
    # c != m, c = 72 (not a multiple of 64 or of the 128-row tile)
    (64, 72, 3, 2, 1, 13, 11, 2), (192, 72, 1, 2, 0, 9, 9, 3),
    # a batch whose last unit is ragged (N = 5 * 14 * 14 = 980 per phase), and one with more than one wave of units
    (128, 128, 3, 2, 1, 28, 28, 5), (128, 256, 3, 2, 1, 56, 56, 32),
]


@pytest.mark.parametrize("m,c,k,s,p,h,w,nb", DGRAD_CASES)
@pytest.mark.parametrize("dt", [0, 1])
def test_dgrad_fp64(spfy, orc, cuda, m, c, k, s, p, h, w, nb, dt):
    comp, _, wd = pruned_filter(spfy, orc, cuda, m, c, k, dt, seed=m + c + k + s + p + h + dt)
    op = spfy.transpose24_conv(comp, k, k, s, p)
    ho, wo = (h + 2 * p - k) // s + 1, (w + 2 * p - k) // s + 1
    dy = rand_nhwc((nb, ho, wo, m), dt, cuda, seed=h * w + m + nb)
    dx = spfy.spmma_conv_dgrad_nhwc(op, dy, h, w)
    assert dx.shape == (nb, h, w, c) and dx.dtype == TDT[dt]
    ref, absprod = reference(wd, dy, h, w, s, p)
    assert_bound(dx.permute(0, 3, 1, 2), ref, absprod, k * k * m, TDT[dt], "dx")


@pytest.mark.parametrize("dt", [0, 1])
def test_beta0_overwrites_a_poisoned_dx(spfy, orc, cuda, dt):
    """1x1 stride 2: the odd rows and columns of dX get no tap; they come back as +0 over a NaN-filled dX"""
    m, c, h, w, nb = 128, 64, 14, 13, 2
    comp, _, wd = pruned_filter(spfy, orc, cuda, m, c, 1, dt, seed=21 + dt)
    op = spfy.transpose24_conv(comp, 1, 1, 2, 0)
    dy = rand_nhwc((nb, 7, 7, m), dt, cuda, seed=5)
    out = torch.full((nb, h, w, c), float("nan"), dtype=TDT[dt], device=cuda)
    dx = spfy.spmma_conv_dgrad_nhwc(op, dy, h, w, out=out, beta=0.0)
    assert dx.data_ptr() == out.data_ptr() and bool(torch.isfinite(dx).all())
    bits = dx.view(torch.int16)
    for sl in ((slice(None), slice(1, None, 2)), (slice(None), slice(None), slice(1, None, 2))):
        assert bool((bits[sl] == 0).all())  # +0, not -0
    ref, absprod = reference(wd, dy, h, w, 2, 0)
    assert_bound(dx.permute(0, 3, 1, 2), ref, absprod, m, TDT[dt], "dx")


@pytest.mark.parametrize("dt", [0, 1])
def test_beta_scales_dx_where_no_tap_reaches(spfy, orc, cuda, dt):
    """1x1 stride 2, beta = 0.5 over a known dX: the pixels no tap reaches get 0.5 * dX (the fill), the others
    0.5 * dX + the gradient (C read at the scattered rows), against fp64"""
    m, c, h, w, nb = 128, 64, 14, 13, 2
    comp, _, wd = pruned_filter(spfy, orc, cuda, m, c, 1, dt, seed=23 + dt)
    op = spfy.transpose24_conv(comp, 1, 1, 2, 0)
    dy = rand_nhwc((nb, 7, 7, m), dt, cuda, seed=10)
    dx0 = rand_nhwc((nb, h, w, c), dt, cuda, seed=11)
    got = spfy.spmma_conv_dgrad_nhwc(op, dy, h, w, out=dx0.clone(), beta=0.5)
    r, absprod = reference(wd, dy, h, w, 2, 0)
    c0 = dx0.permute(0, 3, 1, 2).double()
    ref = r + 0.5 * c0
    # one rounding of the result, the fp32 accumulation, and one fp32 rounding of the beta * C term
    bound = U[TDT[dt]] * ref.abs() + 2.0 ** -23 * (m * absprod + 0.5 * c0.abs()) + ETA[TDT[dt]]
    err = (got.permute(0, 3, 1, 2).double() - ref).abs()
    assert bool((err <= bound).all()), f"{int((~(err <= bound)).sum())} elements outside the bound"
    # the odd rows: 0.5 * dX in fp32, rounded to nearest even, bit for bit
    want = (0.5 * dx0.float()).to(TDT[dt])
    assert torch.equal(got[:, 1::2].view(torch.int16), want[:, 1::2].view(torch.int16))


@pytest.mark.parametrize("dt", [0, 1])
def test_beta1_downsample_block_in_place(spfy, orc, cuda, dt):
    """a residual downsample block's input gradient: the main branch's 3x3 stride-2 layer, then the 1x1 stride-2
    shortcut accumulated into the same dX with beta = 1"""
    cin, mid, cout, h, w, nb = 128, 128, 256, 28, 28, 2
    comp3, _, w3 = pruned_filter(spfy, orc, cuda, mid, cin, 3, dt, seed=31 + dt)
    comp1, _, w1 = pruned_filter(spfy, orc, cuda, cout, cin, 1, dt, seed=32 + dt)
    dy3 = rand_nhwc((nb, 14, 14, mid), dt, cuda, seed=6)
    dy1 = rand_nhwc((nb, 14, 14, cout), dt, cuda, seed=7)
    dx = spfy.spmma_conv_dgrad_nhwc(spfy.transpose24_conv(comp3, 3, 3, 2, 1), dy3, h, w)
    got = spfy.spmma_conv_dgrad_nhwc(spfy.transpose24_conv(comp1, 1, 1, 2, 0), dy1, h, w, out=dx, beta=1.0)
    assert got.data_ptr() == dx.data_ptr()
    r3, a3 = reference(w3, dy3, h, w, 2, 1)
    r1, a1 = reference(w1, dy1, h, w, 2, 0)
    # the main branch's rounded dX (its own bound) plus the shortcut's, and one more rounding of the sum
    ref = r3 + r1
    bound = U[TDT[dt]] * (ref.abs() + r3.abs()) + 2.0 ** -23 * (9 * mid * a3 + cout * a1 + ref.abs()) + 2 * ETA[TDT[dt]]
    err = (got.permute(0, 3, 1, 2).double() - ref).abs()
    assert bool((err <= bound).all()), f"{int((~(err <= bound)).sum())} elements outside the bound"


@pytest.mark.parametrize("dt", [0, 1])
def test_alpha(spfy, orc, cuda, dt):
    m, c, k, s, p, h, w, nb = 128, 64, 3, 2, 1, 15, 12, 2
    comp, _, wd = pruned_filter(spfy, orc, cuda, m, c, k, dt, seed=41 + dt)
    dy = rand_nhwc((nb, 8, 6, m), dt, cuda, seed=8)
    dx = spfy.spmma_conv_dgrad_nhwc(spfy.transpose24_conv(comp, k, k, s, p), dy, h, w, alpha=-0.375)
    ref, absprod = reference(wd, dy, h, w, s, p)
    assert_bound(dx.permute(0, 3, 1, 2), -0.375 * ref, 0.375 * absprod, k * k * m, TDT[dt], "dx")


@pytest.mark.parametrize("k,p,c", [(3, 1, 64), (5, 2, 72), (3, 0, 128)])
@pytest.mark.parametrize("dt", [0, 1])
def test_stride_one_matches_the_stride_one_path(spfy, orc, cuda, k, p, c, dt):
    """stride 1: bit for bit spmma_conv_nhwc(transpose24(comp, taps), dy, pad = k - 1 - pad)"""
    m, h, w, nb = 128, 9, 11, 8
    comp, _, _ = pruned_filter(spfy, orc, cuda, m, c, k, dt, seed=51 + k + dt)
    ho, wo = h + 2 * p - k + 1, w + 2 * p - k + 1
    dy = rand_nhwc((nb, ho, wo, m), dt, cuda, seed=9)
    got = spfy.spmma_conv_dgrad_nhwc(spfy.transpose24_conv(comp, k, k, 1, p), dy, h, w)
    want = spfy.spmma_conv_nhwc(spfy.transpose24(comp, taps=k * k), dy, k, k, stride=1, pad=k - 1 - p)
    assert torch.equal(got.view(torch.int16), want.view(torch.int16))


def test_refusals_on_device(spfy, orc, cuda):
    comp, _, _ = pruned_filter(spfy, orc, cuda, 128, 64, 3, 0, seed=61)
    op = spfy.transpose24_conv(comp, 3, 3, 2, 1)
    before = spfy.launch_count()
    for shape in ((2, 7, 8, 128), (2, 8, 8, 64)):  # a 15 x 15 input gives 8 x 8 x 128
        with pytest.raises(spfy.SpfyError) as e:
            spfy.spmma_conv_dgrad_nhwc(op, torch.zeros(*shape, dtype=torch.float16, device=cuda), 15, 15)
        assert e.value.code == spfy.capi.E_INVALID
    assert spfy.launch_count() == before
    # 72 output channels: dY would be the im2col operand with 72 channels
    comp72, _, _ = pruned_filter(spfy, orc, cuda, 72, 64, 3, 0, seed=62)
    op72 = spfy.transpose24_conv(comp72, 3, 3, 2, 1)
    before = spfy.launch_count()
    with pytest.raises(spfy.SpfyError) as e:
        spfy.spmma_conv_dgrad_nhwc(op72, torch.zeros(2, 8, 8, 72, dtype=torch.float16, device=cuda), 15, 15)
    assert e.value.code == spfy.capi.E_UNSUPPORTED and spfy.launch_count() == before
