"""The 2:4 convolution training path at the filter, stride and padding geometries that spfy_b200.h admits and the other
suites never reach: rectangular filters (the source-tap walk and the weight gradient's tap split are symmetric in kh
and kw for a square one), strides larger than the filter (phases without taps, in sets that are not symmetric in a
and b), pad >= filter (output positions that see only padding), images smaller than the stride (phases with taps but
no dX pixels, between phases that have both), the contract's maxima (16x16 filters, stride 8, 11x11 at stride 4), an
output row wider than 128 positions and a tall image of width <= 4.

One table of geometries feeds every section: the forward implicit GEMM, spfy_transpose24_conv, spfy_spmma_conv_dgrad,
spfy_conv_wgrad24, the fused optimizer step (with a table of more than 256 phases) and the Conv2d24 layer.  Arithmetic
results are checked per element against fp64 computed from the exact 16-bit operands (test_gpu_train24_edges.assert_bound),
byte-level results against the numpy statement of test_conv_dgrad.py and the CPU oracle.  The CPU tests at the top
check that the table holds each of these properties and that the phase rule reproduces fp64 conv2d_input on it."""
import numpy as np
import pytest
import torch
import torch.nn.functional as F

from test_conv_dgrad import PHASE_CASES, dgrad_by_phases, phase_order, phase_taps, phase_tiles
from test_conv_wgrad import split_count
from test_gpu_conv import explicit_b
from test_gpu_conv_dgrad import pruned_filter, rand_nhwc
from test_gpu_conv_dgrad import reference as dgrad_reference
from test_gpu_conv_wgrad import inputs, pruned_layer
from test_gpu_conv_wgrad import reference as wgrad_reference
from test_gpu_optim24 import make_opt, mask_of, metas_of, operand_refs, set_grads, state2d, twin
from test_gpu_train24_edges import ETA, U, assert_bound
from test_transpose24 import expected_sm100

gpu = pytest.mark.gpu
TDT = {0: torch.float16, 1: torch.bfloat16}

# (m, c, kh, kw, stride, pad, batch, h, w): m output and c input channels, multiples of 64 (what Conv2d24 and the data
# gradient's im2col take); the batch makes batch * ho * wo a multiple of 8 (the forward pass's N)
GEOMS = [
    # rectangular filters both ways, pad 1 on both dimensions (pad >= filter along the 1-tap one)
    (64, 64, 1, 3, 1, 1, 2, 6, 7), (64, 64, 3, 1, 1, 1, 2, 7, 6),
    # 7x1 at stride 2 (the 1-tap dimension with pad 3: phase b = 0 has no tap), 3x5 at stride 3 with c != m, 2x1 at
    # stride 2 without padding (phase b = 1 has no tap)
    (128, 64, 7, 1, 2, 3, 1, 11, 9), (64, 128, 3, 5, 3, 2, 2, 10, 13), (64, 64, 2, 1, 2, 0, 2, 9, 8),
    # stride greater than the filter: 15, 7 and 21 of the phases have no tap
    (64, 64, 1, 1, 4, 0, 8, 9, 10), (64, 64, 3, 3, 4, 1, 2, 13, 10), (64, 64, 2, 2, 5, 0, 4, 12, 11),
    # pad >= filter
    (64, 64, 1, 1, 1, 1, 2, 5, 6), (64, 64, 3, 3, 1, 3, 1, 5, 4),
    # images smaller than the stride: on 3 x 5, phase a = 3 has a tap and no rows and phase a = 2 rows and no tap; on
    # 5 x 3 the phase (0, 3) without columns comes before phases with pixels
    (64, 64, 3, 3, 4, 1, 4, 3, 5), (64, 64, 3, 3, 4, 1, 4, 5, 3),
    # the contract's maxima: 256 taps; 64 phases of 4 taps (on a 6-wide image, 16 of them without columns); 11x11 at
    # stride 4
    (64, 64, 16, 16, 1, 8, 4, 6, 5), (64, 64, 16, 16, 8, 8, 4, 17, 12), (64, 64, 16, 16, 8, 8, 8, 17, 6),
    (128, 64, 11, 11, 4, 2, 2, 19, 15),
    # an output row of 150 positions (more than one 128-position im2col load, and more than 64: the weight gradient's
    # step is dw = 64 in one row), and a tall image with 120 positions of width 3 (dn = 0, dh = 21)
    (64, 64, 3, 3, 1, 1, 4, 5, 150), (64, 64, 3, 3, 1, 1, 2, 40, 3),
]
LAYERS = sorted({g[:6] for g in GEOMS})  # (m, c, kh, kw, stride, pad): the layers of the table


def gid(g):
    m, c, kh, kw, s, p, nb, h, w = g
    return f"m{m}c{c}_{kh}x{kw}s{s}p{p}_{nb}x{h}x{w}"


def out_size(kh, kw, s, p, h, w):
    return (h + 2 * p - kh) // s + 1, (w + 2 * p - kw) // s + 1


def no_tap_phases(kh, kw, s, p):
    """the phases (a, b) that no filter tap reaches"""
    return {(a, b) for a in range(s) for b in range(s) if not phase_taps(kh, s, p, a)[0] or not phase_taps(kw, s, p, b)[0]}


def unreached(h, w, kh, kw, s, p):
    """[h, w] bool: the dX pixels of those phases"""
    hole = np.zeros((h, w), bool)
    for a, b in no_tap_phases(kh, kw, s, p):
        hole[a::s, b::s] = True
    return torch.from_numpy(hole)


def phases_with_pixels(kh, kw, s, p, h, w):
    """for each phase with taps, in spfy_transpose24_conv's order: whether it has dX pixels"""
    return [a < h and b < w for a, b, *_ in phase_tiles(64, 64, kh, kw, s, p)]


# ------------------------------------------------------------------ the table, without a GPU
def test_geometry_table_has_every_property():
    """computed from phase_taps and the shapes: the geometries below are there, and so is each property the module
    docstring names"""
    layers = {(kh, kw, s, p) for _, _, kh, kw, s, p, *_ in GEOMS}
    for want in ((1, 3, 1, 1), (3, 1, 1, 1), (3, 3, 4, 1), (16, 16, 1, 8), (16, 16, 8, 8), (11, 11, 4, 2)):
        assert want in layers
    assert any(kh == 7 and kw == 1 and s == 2 for kh, kw, s, p in layers)
    assert any(kh == 3 and kw == 5 and s == 3 for kh, kw, s, p in layers)
    assert (2, 1, 2, 0) in layers
    for k, s in ((1, 4), (3, 4), (2, 5)):  # stride greater than the filter
        assert any(kh == kw == k and st == s for kh, kw, st, p in layers)
    for k in (1, 3):  # pad >= filter
        assert any(kh == kw == k and p >= k for kh, kw, s, p in layers)
    empties = [no_tap_phases(kh, kw, s, p) for kh, kw, s, p in layers]
    assert sum(len(e) > 0 for e in empties) >= 4
    assert any(e != {(b, a) for a, b in e} for e in empties)  # a set of empty phases that is not symmetric
    for m, c, kh, kw, s, p, nb, h, w in GEOMS:
        assert m % 64 == 0 and c % 64 == 0 and h + 2 * p >= kh and w + 2 * p >= kw
        ho, wo = out_size(kh, kw, s, p, h, w)
        assert (nb * ho * wo) % 8 == 0
    # an image smaller than the stride: a phase with a tap and no rows, one with rows and no tap; and a phase with taps
    # but no pixels that comes before phases with pixels
    small = [(kh, kw, s, p, h, w) for _, _, kh, kw, s, p, _, h, w in GEOMS if h < s or w < s]
    assert any(any(phase_taps(kh, s, p, a)[0] for a in range(h, s)) and
               any(not phase_taps(kh, s, p, a)[0] for a in range(h)) for kh, kw, s, p, h, w in small)
    orders = [phases_with_pixels(kh, kw, s, p, h, w) for kh, kw, s, p, h, w in small]
    assert any(not f and any(o[i + 1:]) for o in orders for i, f in enumerate(o))
    # the maxima: 256 taps in one phase, 64 phases of 4 taps
    assert any(len(o) == 256 for *_, kh, kw, s, p in LAYERS for _, _, o, _, _ in phase_tiles(64, 64, kh, kw, s, p))
    assert any(len(t) == 64 and all(len(o) == 4 for _, _, o, _, _ in t)
               for t in (phase_tiles(64, 64, kh, kw, s, p) for *_, kh, kw, s, p in LAYERS))
    # wide and tall outputs; the weight gradient with one split and with many
    sizes = [(nb, *out_size(kh, kw, s, p, h, w)) for _, _, kh, kw, s, p, nb, h, w in GEOMS]
    assert any(wo > 128 for _, _, wo in sizes)
    assert any(ho * wo > 64 and wo <= 4 for _, ho, wo in sizes)
    splits = [split_count(nb, h, w, c, kh, kw, s, p, m) for m, c, kh, kw, s, p, nb, h, w in GEOMS]
    assert 1 in splits and max(splits) > 1
    # each dimension's (taps, stride, pad) is a case of test_conv_dgrad's CPU phase tests
    assert {(k, s, p) for kh, kw, s, p in layers for k in (kh, kw)} <= set(PHASE_CASES)


@pytest.mark.parametrize("g", GEOMS, ids=gid)
def test_phase_rule_is_conv2d_input(g):
    """the phase decomposition with the table's rectangular filters and image sizes, against fp64 conv2d_input"""
    _, _, kh, kw, s, p, nb, h, w = g
    rng = np.random.default_rng(sum(g))
    m, c = 3, 2
    ho, wo = out_size(kh, kw, s, p, h, w)
    wt = rng.standard_normal((m, c, kh, kw))
    dy = rng.standard_normal((1, m, ho, wo))
    ref = torch.nn.grad.conv2d_input((1, c, h, w), torch.from_numpy(wt), torch.from_numpy(dy), stride=s, padding=p)
    np.testing.assert_allclose(dgrad_by_phases(wt, dy, h, w, s, p), ref.numpy(), rtol=1e-12, atol=1e-12)


# ------------------------------------------------------------------ forward, phase operands, data and weight gradients
@gpu
@pytest.mark.parametrize("g", GEOMS, ids=gid)
@pytest.mark.parametrize("dt", [0, 1])
def test_forward(spfy, orc, cuda, g, dt):
    """spmma_conv_nhwc: bit for bit spmma_compressed on the explicit unfold, and within the fp64 bound of conv2d of the
    pruned filter (K = kh*kw*c)"""
    m, c, kh, kw, s, p, nb, h, w = g
    comp, _, wd = pruned_filter(spfy, orc, cuda, m, c, (kh, kw), dt, seed=sum(g) + dt)
    x = rand_nhwc((nb, h, w, c), dt, cuda, seed=sum(g) + 1)
    y = spfy.spmma_conv_nhwc(comp, x, kh, kw, stride=s, pad=p)
    want = spfy.spmma_compressed(comp, explicit_b(x, kh, kw, s, p))
    assert torch.equal(y.view(-1, m).view(torch.int16), want.t().view(torch.int16))
    xd = x.double().permute(0, 3, 1, 2)
    ref = F.conv2d(xd, wd, stride=s, padding=p)
    absref = F.conv2d(xd.abs(), wd.abs(), stride=s, padding=p)
    assert_bound(y.permute(0, 3, 1, 2), ref, absref, kh * kw * c, TDT[dt], "y")


@gpu
@pytest.mark.parametrize("layer", LAYERS, ids=lambda t: "m{}c{}_{}x{}s{}p{}".format(*t))
@pytest.mark.parametrize("dt", [0, 1])
def test_phase_operands(spfy, orc, cuda, layer, dt):
    """spfy_transpose24_conv refilling a poisoned output: every phase byte-exact against expected_sm100 of its
    sub-filter, the phase views at the statement's offsets and shapes, the invalid flag 0"""
    m, c, kh, kw, s, p = layer
    comp, dense, _ = pruned_filter(spfy, orc, cuda, m, c, (kh, kw), dt, seed=sum(layer) + dt)
    op = spfy.transpose24_conv(comp, kh, kw, s, p)
    op.vals.fill_(0xAB)
    op.meta.fill_(0xCD)
    inv = torch.full((1,), 7, dtype=torch.int32, device=cuda)
    assert spfy.transpose24_conv(comp, kh, kw, s, p, invalid=inv, out=op) is op
    assert int(inv.item()) == 0
    tiles = phase_tiles(m, c, kh, kw, s, p)
    total = sum(n for *_, n in tiles)
    assert (op.vals.numel(), op.meta.numel()) == (total * 16384, total * 2048)
    assert len(op.phases) == len(tiles)
    got_v, got_m = op.vals.cpu().numpy(), op.meta.cpu().numpy()
    for (a, b, th, tw, view), (ta, tb, order, first, n) in zip(op.phases, tiles):
        assert (a, b) == (ta, tb) and phase_order(kh, kw, th, tw) == order
        assert (view.rows, view.cols, view.dtype) == (c, len(order) * m, comp.dtype)
        assert view.vals.data_ptr() - op.vals.data_ptr() == first * 16384 and view.vals.numel() == n * 16384
        assert view.meta.data_ptr() - op.meta.data_ptr() == first * 2048 and view.meta.numel() == n * 2048
        rev = np.concatenate([dense[:, t * c:(t + 1) * c] for t in order[::-1]], axis=1)
        ov, om = expected_sm100(orc, dt, rev, len(order))
        assert np.array_equal(got_v[first * 16384:(first + n) * 16384], ov), f"phase ({a}, {b}): values"
        assert np.array_equal(got_m[first * 2048:(first + n) * 2048], om), f"phase ({a}, {b}): metadata"


@gpu
@pytest.mark.parametrize("g", GEOMS, ids=gid)
@pytest.mark.parametrize("dt", [0, 1])
def test_data_gradient(spfy, orc, cuda, g, dt):
    """spmma_conv_dgrad_nhwc against fp64 conv2d_input (K = kh*kw*m): with beta = 0 over a NaN-filled dX, every pixel no
    tap reaches is +0; with beta = 0.5 over a known dX, those pixels are 0.5 * dX rounded once, bit for bit"""
    m, c, kh, kw, s, p, nb, h, w = g
    tdt = TDT[dt]
    comp, _, wd = pruned_filter(spfy, orc, cuda, m, c, (kh, kw), dt, seed=sum(g) + 2 * dt)
    op = spfy.transpose24_conv(comp, kh, kw, s, p)
    ho, wo = out_size(kh, kw, s, p, h, w)
    dy = rand_nhwc((nb, ho, wo, m), dt, cuda, seed=sum(g) + 3)
    ref, absprod = dgrad_reference(wd, dy, h, w, s, p)
    hole = unreached(h, w, kh, kw, s, p).to(cuda)
    dx = spfy.spmma_conv_dgrad_nhwc(op, dy, h, w, out=torch.full((nb, h, w, c), float("nan"), dtype=tdt, device=cuda))
    assert_bound(dx.permute(0, 3, 1, 2), ref, absprod, kh * kw * m, tdt, "dx, beta 0 over NaN")
    assert bool((dx.view(torch.int16)[:, hole] == 0).all())  # +0, not -0
    dx0 = rand_nhwc((nb, h, w, c), dt, cuda, seed=sum(g) + 4)
    got = spfy.spmma_conv_dgrad_nhwc(op, dy, h, w, out=dx0.clone(), beta=0.5)
    c0 = dx0.permute(0, 3, 1, 2).double()
    want = ref + 0.5 * c0
    # one rounding of the result, the fp32 accumulation, and one fp32 rounding of the beta * C term
    bound = U[tdt] * want.abs() + 2.0 ** -23 * (kh * kw * m * absprod + 0.5 * c0.abs()) + ETA[tdt]
    err = (got.permute(0, 3, 1, 2).double() - want).abs()
    assert bool((err <= bound).all()), f"dx, beta 0.5: {int((~(err <= bound)).sum())} elements outside the bound"
    half = (0.5 * dx0.float()).to(tdt)
    assert torch.equal(got.view(torch.int16)[:, hole], half.view(torch.int16)[:, hole])


@gpu
@pytest.mark.parametrize("g", GEOMS, ids=gid)
@pytest.mark.parametrize("dt", [0, 1])
def test_weight_gradient(spfy, cuda, g, dt):
    """conv_wgrad24_nhwc against fp64 conv2d_weight masked to the layer's pattern (K = batch*ho*wo); +0 at every pruned
    position; two calls give the same bits"""
    m, c, kh, kw, s, p, nb, h, w = g
    comp, mask = pruned_layer(spfy, cuda, m, c, kh, kw, TDT[dt], seed=sum(g) + dt)
    x, dy = inputs(cuda, nb, h, w, c, m, kh, kw, s, p, TDT[dt], seed=sum(g) + 5)
    got = spfy.conv_wgrad24_nhwc(comp, x, dy, kh, kw, s, p)
    ref, absprod = wgrad_reference(x, dy, kh, kw, s, p)
    ho, wo = out_size(kh, kw, s, p, h, w)
    assert_bound(got, ref * mask, absprod * mask, nb * ho * wo, torch.float32, "dW")
    assert bool((got.view(torch.int32)[mask == 0] == 0).all())
    again = spfy.conv_wgrad24_nhwc(comp, x, dy, kh, kw, s, p)
    assert torch.equal(got.view(torch.int32), again.view(torch.int32))


# ------------------------------------------------------------------ the fused optimizer step
def conv_layer(spfy, cuda, layer, dtype, seed, scale=1.0, bias=True):
    m, c, kh, kw, s, p = layer
    g = torch.Generator(device="cpu").manual_seed(seed)
    w = (torch.randn(m, c, kh, kw, generator=g) * scale).to(cuda)
    b = torch.randn(m, generator=g).to(cuda) if bias else None
    return spfy.Conv2d24.from_dense(w, b, stride=s, padding=p, dtype=dtype), g


@gpu
@pytest.mark.parametrize("layer", LAYERS, ids=lambda t: "m{}c{}_{}x{}s{}p{}".format(*t))
@pytest.mark.parametrize("dtype", [torch.float16, torch.bfloat16], ids=["fp16", "bf16"])
@pytest.mark.parametrize("rule", ["sgd_momentum_dampening", "adamw"])
def test_optimizer_step_refills_the_operands(spfy, cuda, layer, dtype, rule):
    """two SGD24 (momentum) or AdamW24 steps with NaN / Inf at the pruned positions of the gradient: comp.vals byte-equal
    to recompress24 of the new master, op_t.vals to transpose24_conv of the new comp, metadata unchanged, master and
    state +0 at pruned positions"""
    conv, _ = conv_layer(spfy, cuda, layer, dtype, seed=sum(layer))
    mk = mask_of(conv)
    mm, mt = metas_of(conv)
    opt = make_opt(spfy, rule, list(conv.parameters()))
    for step in range(2):
        set_grads([conv], 300 + step, poison=True)
        opt.step()
        vals, vt = operand_refs(spfy, conv)
        assert torch.equal(conv.comp.vals, vals), f"step {step}: comp.vals"
        assert torch.equal(conv.op_t.vals, vt), f"step {step}: op_t.vals"
        assert torch.equal(conv.comp.meta, mm) and torch.equal(conv.op_t.meta, mt)
        assert bool((conv._w2d().detach().view(torch.int32)[~mk] == 0).all())
        for k, v in opt.state[conv.weight].items():
            if k != "step":
                assert bool((state2d(conv, v).view(torch.int32)[~mk] == 0).all()), f"step {step}: {k} not +0"


SPLIT_TABLE = [(64, 64, 16, 16, 8, 8)] * 5 + [(64, 64, 3, 5, 1, 2)]  # 5 x 64 phases, then a stride-1 layer


def test_split_table_has_more_than_256_phases():
    """spfy_optim24_step carries at most 256 phases in one launch"""
    assert sum(len(phase_tiles(m, c, kh, kw, s, p)) for m, c, kh, kw, s, p in SPLIT_TABLE) > 256


@gpu
def test_optimizer_splits_more_than_256_phases(spfy, cuda):
    """five 16x16 stride-8 layers and a stride-1 layer: one SGD24 step takes more than one launch and writes, byte for
    byte, what one step per parameter writes"""
    layers = [conv_layer(spfy, cuda, t, torch.float16, seed=i)[0] for i, t in enumerate(SPLIT_TABLE)]
    twins = [twin(spfy, layer) for layer in layers]
    params = [p for layer in layers for p in layer.parameters()]
    params2 = [p for layer in twins for p in layer.parameters()]
    opt = spfy.SGD24(params, lr=0.1, momentum=0.9, weight_decay=1e-4)
    opts = [spfy.SGD24([q], lr=0.1, momentum=0.9, weight_decay=1e-4) for q in params2]
    g = torch.Generator(device="cpu").manual_seed(5)
    for step in range(2):
        for p, q in zip(params, params2):
            q.grad = torch.randn(p.shape, generator=g).to(cuda).contiguous(
                memory_format=torch.channels_last if p.dim() == 4 else torch.contiguous_format)
            p.grad = q.grad.clone(memory_format=torch.preserve_format)
        n0 = spfy.launch_count()
        opt.step()
        assert spfy.launch_count() - n0 > 1
        for o in opts:
            o.step()
        for p, q, o in zip(params, params2, opts):
            assert torch.equal(p.detach(), q.detach())
            assert torch.equal(opt.state[p]["momentum_buffer"], o.state[q]["momentum_buffer"])
        for layer, t in zip(layers, twins):
            assert torch.equal(layer.comp.vals, t.comp.vals) and torch.equal(layer.op_t.vals, t.op_t.vals)


# ------------------------------------------------------------------ Conv2d24
def conv2d24_and_input(spfy, cuda, g, tdt, bias, seed):
    m, c, kh, kw, s, p, nb, h, w = g
    layer, gen = conv_layer(spfy, cuda, g[:6], tdt, seed, scale=0.1, bias=bias)
    x = torch.randn(nb, c, h, w, generator=gen).to(tdt).to(cuda).contiguous(memory_format=torch.channels_last)
    return layer, x, gen


@gpu
@pytest.mark.parametrize("g", GEOMS, ids=gid)
@pytest.mark.parametrize("dt", [0, 1])
@pytest.mark.parametrize("bias", [True, False])
def test_conv2d24_against_fp64_autograd(spfy, cuda, g, dt, bias):
    """y, x.grad, weight.grad and bias.grad against fp64 autograd of the masked master rounded to the layer's dtype"""
    m, c, kh, kw, s, p, nb, h, w = g
    tdt = TDT[dt]
    layer, x, gen = conv2d24_and_input(spfy, cuda, g, tdt, bias, seed=sum(g) + dt)
    x.requires_grad_(True)
    y = layer(x)
    assert y.is_contiguous(memory_format=torch.channels_last) and y.dtype == tdt
    w16 = layer.weight.detach().to(tdt).double()
    mask = (layer.weight.detach() != 0).double()
    xd = x.detach().double()
    bd = layer.bias.detach().double() if bias else None
    ref = F.conv2d(xd, w16, bd, stride=s, padding=p)
    absref = F.conv2d(xd.abs(), w16.abs(), bd.abs() if bias else None, stride=s, padding=p)
    assert_bound(y, ref, absref, kh * kw * c + int(bias), tdt, "y")
    dy = torch.randn(y.shape, generator=gen).to(tdt).to(cuda).contiguous(memory_format=torch.channels_last)
    y.backward(dy)
    dyd = dy.double()
    dx = torch.nn.grad.conv2d_input(x.shape, w16, dyd, stride=s, padding=p)
    adx = torch.nn.grad.conv2d_input(x.shape, w16.abs(), dyd.abs(), stride=s, padding=p)
    assert_bound(x.grad, dx, adx, kh * kw * m, tdt, "x.grad")
    dw = torch.nn.grad.conv2d_weight(xd, w16.shape, dyd, stride=s, padding=p) * mask
    adw = torch.nn.grad.conv2d_weight(xd.abs(), w16.shape, dyd.abs(), stride=s, padding=p) * mask
    K = nb * dy.shape[2] * dy.shape[3]
    assert layer.weight.grad.dtype == torch.float32
    assert_bound(layer.weight.grad, dw, adw, K, torch.float32, "weight.grad")
    assert bool((layer.weight.grad.view(torch.int32)[mask == 0] == 0).all())
    if bias:
        assert_bound(layer.bias.grad, dyd.sum((0, 2, 3)), dyd.abs().sum((0, 2, 3)), K, torch.float32, "bias.grad")


@gpu
@pytest.mark.parametrize("g", GEOMS, ids=gid)
@pytest.mark.parametrize("dt", [0, 1])
def test_conv2d24_gradient_combinations_and_dy_layouts(spfy, cuda, g, dt):
    """a dy that is NCHW-contiguous, and one that arrives through an fp32 loss, give the bits of a channels_last dy; a
    frozen weight launches no weight-gradient kernel and an input without grad no data-gradient kernel"""
    m, c, kh, kw, s, p, nb, h, w = g
    tdt = TDT[dt]
    layer, x, gen = conv2d24_and_input(spfy, cuda, g, tdt, True, seed=sum(g) + 7 + dt)
    ho, wo = out_size(kh, kw, s, p, h, w)
    dy = torch.randn(nb, m, ho, wo, generator=gen).to(tdt).to(cuda).contiguous(memory_format=torch.channels_last)
    n0 = spfy.launch_count()
    spfy.spmma_conv_dgrad_nhwc(layer.op_t, dy.permute(0, 2, 3, 1), h, w)
    n_dx = spfy.launch_count() - n0
    n0 = spfy.launch_count()
    spfy.conv_wgrad24_nhwc(layer.comp, x.permute(0, 2, 3, 1), dy.permute(0, 2, 3, 1), kh, kw, s, p)
    n_dw = spfy.launch_count() - n0

    def backward(x_in, go):
        layer.weight.grad = layer.bias.grad = None
        y = layer(x_in)
        n0 = spfy.launch_count()
        go(y)
        return spfy.launch_count() - n0

    def bits(t):
        return t.view(torch.int16 if t.dtype != torch.float32 else torch.int32).clone()

    xg = x.clone().requires_grad_(True)
    assert backward(xg, lambda y: y.backward(dy)) == n_dx + n_dw
    want = [bits(xg.grad), bits(layer.weight.grad), bits(layer.bias.grad)]
    for name, go in (("NCHW dy", lambda y: y.backward(dy.contiguous())),
                     ("fp32 loss", lambda y: (y.float() * dy.float()).sum().backward())):
        xg = x.clone().requires_grad_(True)
        backward(xg, go)
        got = [bits(xg.grad), bits(layer.weight.grad), bits(layer.bias.grad)]
        assert all(torch.equal(a, b) for a, b in zip(got, want)), name
    layer.weight.requires_grad_(False)
    xg = x.clone().requires_grad_(True)
    assert backward(xg, lambda y: y.backward(dy)) == n_dx
    assert layer.weight.grad is None and torch.equal(bits(xg.grad), want[0]) and torch.equal(bits(layer.bias.grad), want[2])
    layer.weight.requires_grad_(True)
    assert backward(x, lambda y: y.backward(dy)) == n_dw
    assert x.grad is None and torch.equal(bits(layer.weight.grad), want[1])


@gpu
@pytest.mark.parametrize("g", GEOMS, ids=gid)
def test_conv2d24_grad_scaler_overflow(spfy, cuda, g):
    """fp16, torch.amp.GradScaler with 2^40 as the first scale and SGD24: the scaled dy overflows, the step is skipped
    and master, bias, comp and op_t stay byte-identical; weight.grad is +0 at every pruned position, where the unmasked
    gradient is inf or NaN"""
    m, c, kh, kw, s, p, nb, h, w = g
    layer, x, gen = conv2d24_and_input(spfy, cuda, g, torch.float16, True, seed=sum(g) + 11)
    opt = spfy.SGD24(layer.parameters(), lr=0.5, momentum=0.9)
    scaler = torch.amp.GradScaler("cuda", init_scale=2.0 ** 40, backoff_factor=2.0 ** -30, growth_interval=1000)
    ho, wo = out_size(kh, kw, s, p, h, w)
    target = torch.randn(nb, m, ho, wo, generator=gen).to(cuda)
    before = [layer.weight.detach().view(torch.int32).clone(), layer.bias.detach().clone(), layer.comp.vals.clone(),
              layer.comp.meta.clone(), layer.op_t.vals.clone(), layer.op_t.meta.clone()]
    seen = []
    y = layer(x)
    y.register_hook(lambda gr: seen.append(gr.detach().clone()))
    scaler.scale(((y.float() - target) ** 2).mean()).backward()
    scaler.step(opt)
    scaler.update()
    assert scaler.get_scale() < 2.0 ** 40
    after = [layer.weight.detach().view(torch.int32), layer.bias.detach(), layer.comp.vals, layer.comp.meta,
             layer.op_t.vals, layer.op_t.meta]
    assert all(torch.equal(a, b) for a, b in zip(before, after))
    keep = layer.weight.detach() != 0
    gw = layer.weight.grad
    assert not bool(torch.isfinite(seen[0]).all()) and not bool(torch.isfinite(gw[keep]).all())
    unmasked = torch.nn.grad.conv2d_weight(x.double(), gw.shape, seen[0].double(), stride=s, padding=p)
    assert not bool(torch.isfinite(unmasked[~keep]).all())
    assert bool((gw.view(torch.int32)[~keep] == 0).all())
    layer(x)  # the skipped step left the operands in sync: no refresh() needed
