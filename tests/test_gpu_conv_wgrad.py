"""Weight gradients of 2:4 convolutions on the GPU (spfy_conv_wgrad24) and the Conv2d24 layer.

Every element is checked against fp64 conv2d_weight of the exact 16-bit X and dY the kernel read, masked to the layer's
pattern, with the bound of test_gpu_train24_edges.assert_bound: u = 2^-24 (fp32 output) and K = batch * ho * wo, the
reduction length (plus one term each for alpha's and beta's products where they apply)."""
import sys

import pytest
import torch

from test_conv_wgrad import RESNET50, split_count
from test_gpu_train24_edges import assert_bound

pytestmark = pytest.mark.gpu

DT = {0: torch.float16, 1: torch.bfloat16}


def pruned_layer(spfy, cuda, m, c, kh, kw, dtype, seed):
    """(comp, mask [m, kh*kw*c] fp64) of a random filter pruned in (kh, kw, c) order"""
    g = torch.Generator(device="cpu").manual_seed(seed)
    w2 = torch.randn(m, kh * kw * c, generator=g).to(cuda).to(dtype)
    comp = spfy.prune24(w2, inplace=True, mode=spfy.PRUNE_TILE_TRANSPOSABLE)
    ones = torch.ones(m, kh * kw * c, device=cuda)
    spfy.recompress24(ones, comp, masked_out=ones, values=False)
    return comp, ones.double()


def inputs(cuda, nb, h, w, c, m, kh, kw, s, p, dtype, seed):
    g = torch.Generator(device="cpu").manual_seed(seed)
    ho, wo = (h + 2 * p - kh) // s + 1, (w + 2 * p - kw) // s + 1
    x = torch.randn(nb, h, w, c, generator=g).to(cuda).to(dtype)
    dy = torch.randn(nb, ho, wo, m, generator=g).to(cuda).to(dtype)
    return x, dy


def reference(x, dy, kh, kw, s, p):
    """fp64 conv2d_weight of NHWC x, dy in (kh, kw, c) order, and the same of |x|, |dy|: [m, kh*kw*c] each"""
    c, m = x.shape[3], dy.shape[3]

    def wg(a, b):
        r = torch.nn.grad.conv2d_weight(a.permute(0, 3, 1, 2), (m, c, kh, kw), b.permute(0, 3, 1, 2), stride=s, padding=p)
        return r.permute(0, 2, 3, 1).reshape(m, -1)
    xd, dyd = x.double(), dy.double()
    return wg(xd, dyd), wg(xd.abs(), dyd.abs())


# (nb, h, w, c, m, k, stride, pad): 5x5 and 7x7 filters with stride 3; odd and non-square images; c != m; m = 72 and 200
# (an n-tile with rows past m); c = 192 (a 128-row tile across two filter taps); K = nb*ho*wo not a multiple of 64; shapes
# with one split (one stage, and seven) and with many
EDGE = [(2, 19, 23, 64, 64, 5, 3, 2), (3, 17, 15, 128, 72, 7, 3, 3), (3, 13, 9, 64, 200, 3, 1, 1),
        (2, 11, 7, 192, 64, 3, 2, 1), (2, 9, 13, 64, 8, 3, 1, 0), (1, 8, 8, 64, 64, 1, 1, 0), (1, 20, 20, 64, 64, 3, 1, 1),
        (4, 15, 17, 256, 136, 1, 2, 0), (8, 28, 28, 128, 256, 3, 1, 1)]


def check(spfy, cuda, nb, h, w, c, m, k, s, p, dt, seed):
    dtype = DT[dt]
    comp, mask = pruned_layer(spfy, cuda, m, c, k, k, dtype, seed)
    x, dy = inputs(cuda, nb, h, w, c, m, k, k, s, p, dtype, seed + 1)
    got = spfy.conv_wgrad24_nhwc(comp, x, dy, k, k, s, p)
    ref, absprod = reference(x, dy, k, k, s, p)
    K = dy.shape[0] * dy.shape[1] * dy.shape[2]
    assert_bound(got, ref * mask, absprod * mask, K, torch.float32, f"wgrad {nb}x{h}x{w}x{c} -> {m}, {k}x{k} s{s} p{p}")
    assert bool((got[mask == 0] == 0).all())


@pytest.mark.parametrize("c,m,hw,k,s,p", RESNET50)
def test_wgrad_resnet50_against_fp64(spfy, cuda, c, m, hw, k, s, p):
    check(spfy, cuda, 32, hw, hw, c, m, k, s, p, 0, seed=c + m + hw + k + s)


@pytest.mark.parametrize("nb,h,w,c,m,k,s,p", EDGE)
@pytest.mark.parametrize("dt", [0, 1])
def test_wgrad_edges_against_fp64(spfy, cuda, nb, h, w, c, m, k, s, p, dt):
    check(spfy, cuda, nb, h, w, c, m, k, s, p, dt, seed=nb * 7 + h + w + c + m + k + dt)


def test_edge_cases_cover_one_and_many_splits():
    splits = [split_count(nb, h, w, c, k, k, s, p, m) for nb, h, w, c, m, k, s, p in EDGE]
    assert 1 in splits and max(splits) > 1
    assert any((nb * ((h + 2 * p - k) // s + 1) * ((w + 2 * p - k) // s + 1)) % 64 for nb, h, w, c, m, k, s, p in EDGE)


@pytest.mark.parametrize("dt", [0, 1])
def test_mask_beta_alpha(spfy, cuda, dt):
    """beta = 0 over NaN: pruned positions bitwise +0, the rest finite; beta = 1 accumulates; beta = 0.5 with alpha = -1.5
    against fp64 of the two, pruned positions +0 where the old dW was not"""
    dtype = DT[dt]
    nb, h, w, c, m, k, s, p = 4, 14, 14, 128, 128, 3, 2, 1
    comp, mask = pruned_layer(spfy, cuda, m, c, k, k, dtype, 11 + dt)
    x, dy = inputs(cuda, nb, h, w, c, m, k, k, s, p, dtype, 12 + dt)
    ref, absprod = reference(x, dy, k, k, s, p)
    K = nb * 7 * 7
    out = torch.full((m, k * k * c), float("nan"), device=cuda)
    spfy.conv_wgrad24_nhwc(comp, x, dy, k, k, s, p, out=out)
    pruned = mask == 0
    assert bool((out[pruned] == 0).all()) and not bool(torch.signbit(out[pruned]).any())
    assert bool(torch.isfinite(out[~pruned]).all())
    old = torch.randn(m, k * k * c, device=cuda)
    acc = old.clone()
    spfy.conv_wgrad24_nhwc(comp, x, dy, k, k, s, p, out=acc, beta=1.0)
    assert_bound(acc, old.double() * mask + ref * mask, (old.double().abs() + absprod) * mask, K + 1, torch.float32, "beta 1")
    assert bool((acc[pruned] == 0).all())
    acc = old.clone()
    spfy.conv_wgrad24_nhwc(comp, x, dy, k, k, s, p, out=acc, alpha=-1.5, beta=0.5)
    want = (0.5 * old.double() - 1.5 * ref) * mask
    assert_bound(acc, want, (0.5 * old.double().abs() + 1.5 * absprod) * mask, K + 2, torch.float32, "alpha -1.5 beta 0.5")
    assert bool((acc[pruned] == 0).all()) and not bool(torch.signbit(acc[pruned]).any())
    with pytest.raises(spfy.SpfyError):
        spfy.conv_wgrad24_nhwc(comp, x, dy, k, k, s, p, beta=1.0)  # beta != 0 needs out


def test_wgrad_is_deterministic(spfy, cuda):
    nb, hw, c, m, k, s, p = 32, 28, 128, 128, 3, 1, 1
    assert split_count(nb, hw, hw, c, k, k, s, p, m) > 1
    comp, _ = pruned_layer(spfy, cuda, m, c, k, k, torch.float16, 3)
    x, dy = inputs(cuda, nb, hw, hw, c, m, k, k, s, p, torch.float16, 4)
    a = spfy.conv_wgrad24_nhwc(comp, x, dy, k, k, s, p)
    b = spfy.conv_wgrad24_nhwc(comp, x, dy, k, k, s, p)
    assert torch.equal(a.view(torch.int32), b.view(torch.int32))


def test_wgrad_writes_a_channels_last_weight(spfy, cuda):
    """out may be the channels_last [m, c, kh, kw] weight itself: the same bits as the [m, kh*kw*c] result"""
    nb, hw, c, m, k, s, p = 2, 10, 64, 64, 3, 1, 1
    comp, _ = pruned_layer(spfy, cuda, m, c, k, k, torch.float16, 5)
    x, dy = inputs(cuda, nb, hw, hw, c, m, k, k, s, p, torch.float16, 6)
    flat = spfy.conv_wgrad24_nhwc(comp, x, dy, k, k, s, p)
    w4 = torch.empty(m, c, k, k, device=cuda, memory_format=torch.channels_last)
    spfy.conv_wgrad24_nhwc(comp, x, dy, k, k, s, p, out=w4)
    assert torch.equal(w4.permute(0, 2, 3, 1).reshape(m, -1), flat)
    with pytest.raises(ValueError):
        spfy.conv_wgrad24_nhwc(comp, x, dy, k, k, s, p, out=torch.empty(m, c, k, k, device=cuda))  # NCHW storage


# ------------------------------------------------------------------ Conv2d24
@pytest.mark.parametrize("m,c,k,s,p,hw", [(128, 64, 3, 1, 1, 14), (64, 128, 3, 2, 1, 15), (256, 128, 1, 2, 0, 14),
                                          (128, 128, 1, 1, 0, 9)])
def test_conv2d24_against_fp64_autograd(spfy, cuda, m, c, k, s, p, hw):
    g = torch.Generator(device="cpu").manual_seed(m + c + k + s)
    nb = 8  # nb * ho * wo a multiple of 8, as spmma_conv_nhwc needs
    w = (torch.randn(m, c, k, k, generator=g) * 0.1).to(cuda)
    b = torch.randn(m, generator=g).to(cuda)
    layer = spfy.Conv2d24.from_dense(w, b, stride=s, padding=p)
    assert layer.weight.is_contiguous(memory_format=torch.channels_last) and layer.weight.dtype == torch.float32
    x = torch.randn(nb, c, hw, hw, generator=g).to(cuda).half().contiguous(memory_format=torch.channels_last)
    x.requires_grad_(True)
    y = layer(x)
    assert y.is_contiguous(memory_format=torch.channels_last) and y.dtype == torch.float16
    # the forward is spmma_conv_nhwc with the bias in the epilogue, bit for bit
    direct = spfy.spmma_conv_nhwc(layer.comp, x.detach().permute(0, 2, 3, 1), k, k, s, p,
                                  epilogue=spfy.Epilogue(bias=layer.bias.detach()))
    assert torch.equal(y.detach().permute(0, 2, 3, 1), direct)
    w16 = layer.weight.detach().half().double()  # the operand: the masked master rounded to fp16
    mask = (layer.weight.detach() != 0).double()
    xd = x.detach().double()
    ref = torch.nn.functional.conv2d(xd, w16, layer.bias.detach().double(), stride=s, padding=p)
    absref = torch.nn.functional.conv2d(xd.abs(), w16.abs(), layer.bias.detach().double().abs(), stride=s, padding=p)
    assert_bound(y, ref, absref, k * k * c + 1, torch.float16, "forward")
    dy = torch.randn(y.shape, generator=g).to(cuda).half().contiguous(memory_format=torch.channels_last)
    y.backward(dy)
    dyd = dy.double()
    dx = torch.nn.grad.conv2d_input(x.shape, w16, dyd, stride=s, padding=p)
    adx = torch.nn.grad.conv2d_input(x.shape, w16.abs(), dyd.abs(), stride=s, padding=p)
    assert_bound(x.grad, dx, adx, k * k * m, torch.float16, "input gradient")
    dw = torch.nn.grad.conv2d_weight(xd, w.shape, dyd, stride=s, padding=p) * mask
    adw = torch.nn.grad.conv2d_weight(xd.abs(), w.shape, dyd.abs(), stride=s, padding=p) * mask
    K = dy.shape[0] * dy.shape[2] * dy.shape[3]
    assert layer.weight.grad.dtype == torch.float32
    assert_bound(layer.weight.grad, dw, adw, K, torch.float32, "weight gradient")
    assert bool((layer.weight.grad[mask == 0] == 0).all())
    assert_bound(layer.bias.grad, dyd.sum((0, 2, 3)), dyd.abs().sum((0, 2, 3)), K, torch.float32, "bias gradient")


def test_conv2d24_refuses_inputs_and_shapes(spfy, cuda):
    layer = spfy.Conv2d24.from_dense(torch.randn(64, 64, 3, 3, device=cuda), padding=1)
    x = torch.randn(2, 64, 8, 8, device=cuda).half()
    with pytest.raises(ValueError, match="channels_last"):
        layer(x)  # NCHW
    with pytest.raises(TypeError, match="dtype"):
        layer(x.float().contiguous(memory_format=torch.channels_last))
    layer(x.contiguous(memory_format=torch.channels_last))
    for bad in (dict(weight=torch.randn(64, 48, 3, 3, device=cuda)), dict(weight=torch.randn(72, 64, 1, 1, device=cuda)),
                dict(weight=torch.randn(64, 64, 3, 3, device=cuda), groups=2),
                dict(weight=torch.randn(64, 64, 3, 3, device=cuda), dilation=2)):
        with pytest.raises(ValueError):
            spfy.Conv2d24.from_dense(**bad)


def test_conv2d24_refuses_a_mask_that_is_not_transposable(spfy, cuda, monkeypatch):
    """from_dense raises when transpose24_conv flags the mask (here: a STRIP-pruned mask, which keeps 2 of 4 along rows
    only)"""
    ops = sys.modules[spfy.Conv2d24.__module__]
    real = ops.prune24
    monkeypatch.setattr(ops, "prune24", lambda a, **kw: real(a, inplace=True, mode=spfy.PRUNE_STRIP_MAG))
    g = torch.Generator(device="cpu").manual_seed(9)
    with pytest.raises(ValueError, match="transposable"):
        spfy.Conv2d24.from_dense(torch.randn(128, 128, 3, 3, generator=g).to(cuda))


def test_bottleneck_sgd_tracks_torch(spfy, cuda):
    """five SGD-with-momentum steps of a bottleneck block (1x1, 3x3 stride 2, 1x1, projection 1x1 stride 2) of Conv2d24
    layers with torch BatchNorm / ReLU: the losses track an fp32 torch replica on the masked weights; the masks never move
    (comp.meta and op_t.meta byte-identical after every step); pruned master entries stay 0; forward without refresh()
    raises"""
    g = torch.Generator(device="cpu").manual_seed(7)
    nb, c, mid, out, hw = 8, 64, 64, 256, 16
    specs = [(mid, c, 1, 1, 0), (mid, mid, 3, 2, 1), (out, mid, 1, 1, 0), (out, c, 1, 2, 0)]
    convs = [spfy.Conv2d24.from_dense((torch.randn(m, ci, k, k, generator=g) * (2.0 / (ci * k * k)) ** 0.5).to(cuda),
                                      torch.zeros(m, device=cuda), stride=s, padding=p) for m, ci, k, s, p in specs]
    bns = [torch.nn.BatchNorm2d(m).to(cuda) for m, *_ in specs]
    bns_ref = [torch.nn.BatchNorm2d(m).to(cuda) for m, *_ in specs]
    ref = [(cv.weight.detach().clone().requires_grad_(True), cv.bias.detach().clone().requires_grad_(True)) for cv in convs]
    masks = [cv.weight.detach() != 0 for cv in convs]
    metas = [(cv.comp.meta.clone(), cv.op_t.meta.clone()) for cv in convs]
    params = [q for cv in convs for q in (cv.weight, cv.bias)] + [q for bn in bns for q in bn.parameters()]
    params_ref = [q for pair in ref for q in pair] + [q for bn in bns_ref for q in bn.parameters()]
    opt = torch.optim.SGD(params, lr=0.05, momentum=0.9)
    opt_ref = torch.optim.SGD(params_ref, lr=0.05, momentum=0.9)
    x = torch.randn(nb, c, hw, hw, generator=g).to(cuda).half().contiguous(memory_format=torch.channels_last)
    target = torch.randn(nb, out, hw // 2, hw // 2, generator=g).to(cuda)

    def block(xin, conv, bn):
        h = torch.relu(bn[0](conv[0](xin)))
        h = torch.relu(bn[1](conv[1](h)))
        return torch.relu(bn[2](conv[2](h)) + bn[3](conv[3](xin)))

    def conv_ref(i):
        w, b = ref[i]
        s, p = specs[i][3], specs[i][4]
        return lambda t: torch.nn.functional.conv2d(t, w, b, stride=s, padding=p)

    for step in range(5):
        opt.zero_grad()
        loss = ((block(x, convs, bns).float() - target) ** 2).mean()
        loss.backward()
        opt.step()
        opt_ref.zero_grad()
        loss_ref = ((block(x.float(), [conv_ref(i) for i in range(4)], bns_ref) - target) ** 2).mean()
        loss_ref.backward()
        for (w, _), mk in zip(ref, masks):
            w.grad.mul_(mk)
        opt_ref.step()
        assert abs(loss.item() - loss_ref.item()) <= 1e-2 * abs(loss_ref.item()), (step, loss.item(), loss_ref.item())
        if step == 0:
            with pytest.raises(RuntimeError, match="refresh"):
                convs[0](x)
        for cv in convs:
            cv.refresh()
        for cv, (mm, mt), mk in zip(convs, metas, masks):
            assert torch.equal(cv.comp.meta, mm) and torch.equal(cv.op_t.meta, mt)
            assert bool((cv.weight.detach()[~mk] == 0).all())
            assert cv.weight.is_contiguous(memory_format=torch.channels_last)
