"""2:4 fine-tuning on the GPU: spfy_transpose24 byte-exact against the oracle (A^T and the flipped 3x3 filter), its
validity flag, PRUNE_TILE_TRANSPOSABLE, spfy_recompress24, the backward data pass through the transposed operand
(Linear and 3x3 stride-1 convolutions) and the Linear24 layer against torch autograd."""
import numpy as np
import pytest
import torch

from test_gpu_parity import REL_TOL, bits_of, rel_err, to_dev
from test_transpose24 import expected_sm100

pytestmark = pytest.mark.gpu

TDT = {0: torch.float16, 1: torch.bfloat16}


def zero_free(orc, dt, shape, seed):
    """magnitudes in [0.25, 1), random signs: no zeros, so the kept set of a TILE prune is the nonzero set"""
    rng = np.random.default_rng(seed)
    x = rng.uniform(0.25, 1.0, shape) * rng.choice([-1.0, 1.0], shape)
    return orc.from_f32(dt, x.astype(np.float32))


def half_zero(orc, dt, shape, seed):
    """half of the entries exactly +-0: zero-valued survivors in many groups"""
    rng = np.random.default_rng(seed)
    x = rng.uniform(0.25, 1.0, shape) * rng.choice([-1.0, 1.0], shape)
    x[rng.random(shape) < 0.5] = 0.0
    x = np.copysign(x, rng.choice([-1.0, 1.0], shape))
    return orc.from_f32(dt, x.astype(np.float32))


def prune_dev(spfy, bits, dt, dev, mode, layout=None):
    a = to_dev(bits, dt, dev)
    dense = torch.empty_like(a)
    comp = spfy.prune24(a, out_dense=dense, mode=mode, layout=layout if layout is not None else spfy.LAYOUT_SM100)
    return comp, dense


def poisoned_out(spfy, comp, taps, dev):
    out = spfy.alloc_compressed(comp.dtype, comp.cols // taps, taps * comp.rows, dev)
    out.vals.fill_(0xAB)
    out.meta.fill_(0xCD)
    return out


def operand_from_mask(bits, keep):
    """canonical vals / meta of the operand that keeps exactly `keep` (two per group of four)"""
    rows, cols = bits.shape
    kq = keep.reshape(rows, cols // 4, 4).astype(bool)
    assert (kq.sum(-1) == 2).all()
    order = np.argsort(~kq, axis=-1, kind="stable")[..., :2]
    vals = np.take_along_axis(bits.reshape(rows, cols // 4, 4), order, -1).reshape(rows, -1)
    nib = (order[..., 0] | (order[..., 1] << 2)).astype(np.uint8)
    meta = nib[:, 0::2].copy()  # an odd last group: low nibble only
    meta[:, : nib.shape[1] // 2] |= nib[:, 1::2] << 4
    return vals, meta


# ------------------------------------------------------------------ transpose24
@pytest.mark.parametrize("rows,cols", [(128, 128), (200, 72), (64, 576), (256, 2304), (1024, 4608), (2048, 512)])
@pytest.mark.parametrize("dt", [0, 1])
def test_transpose24_byte_exact(spfy, orc, cuda, rows, cols, dt):
    bits = zero_free(orc, dt, (rows, cols), seed=rows + 7 * cols + dt)
    comp, dense = prune_dev(spfy, bits, dt, cuda, spfy.PRUNE_TILE_MAG)
    want_dense, _ = orc.prune24_tile(dt, bits)
    assert np.array_equal(bits_of(dense), want_dense)
    inv = torch.full((1,), 7, dtype=torch.int32, device=cuda)
    out = spfy.transpose24(comp, out=poisoned_out(spfy, comp, 1, cuda), invalid=inv)
    ov, om = expected_sm100(orc, dt, want_dense, 1)
    assert int(inv.item()) == 0
    assert np.array_equal(out.vals.cpu().numpy(), ov) and np.array_equal(out.meta.cpu().numpy(), om)
    back = spfy.transpose24(out, out=poisoned_out(spfy, out, 1, cuda))
    assert torch.equal(back.vals, comp.vals) and torch.equal(back.meta, comp.meta)


@pytest.mark.parametrize("ch", [64, 128, 256, 512])
@pytest.mark.parametrize("dt", [0, 1])
def test_transpose24_conv_taps(spfy, orc, cuda, ch, dt):
    """ResNet-50 3x3 filters (c = m): A in (kh, kw, c) order -> the flipped, channel-swapped filter, byte-exact"""
    m = c = ch
    w = to_dev(zero_free(orc, dt, (m, c * 9), seed=ch + dt), dt, cuda)
    wp = spfy.permute_conv_weights(w, c, 3, 3)
    comp, dense = prune_dev(spfy, bits_of(wp), dt, cuda, spfy.PRUNE_TILE_MAG)
    want_dense, _ = orc.prune24_tile(dt, bits_of(wp))
    assert np.array_equal(bits_of(dense), want_dense)
    out = spfy.transpose24(comp, taps=9, out=poisoned_out(spfy, comp, 9, cuda))
    ov, om = expected_sm100(orc, dt, want_dense, 9)
    assert np.array_equal(out.vals.cpu().numpy(), ov) and np.array_equal(out.meta.cpu().numpy(), om)
    back = spfy.transpose24(out, taps=9, out=poisoned_out(spfy, out, 9, cuda))
    assert torch.equal(back.vals, comp.vals) and torch.equal(back.meta, comp.meta)


def test_transpose24_invalid_flag(spfy, orc, cuda):
    inv = torch.full((1,), 5, dtype=torch.int32, device=cuda)
    bits = zero_free(orc, 0, (256, 512), seed=11)
    tile, _ = prune_dev(spfy, bits, 0, cuda, spfy.PRUNE_TILE_MAG)
    spfy.transpose24(tile, invalid=inv)
    assert int(inv.item()) == 0
    trans, _ = prune_dev(spfy, bits, 0, cuda, spfy.PRUNE_TILE_TRANSPOSABLE)
    spfy.transpose24(trans, invalid=inv)
    assert int(inv.item()) == 0
    strip = spfy.prune24(to_dev(bits, 0, cuda))
    spfy.transpose24(strip, invalid=inv)
    assert int(inv.item()) == 1
    spfy.transpose24(tile, invalid=inv)  # the next clean call resets it
    assert int(inv.item()) == 0


# ------------------------------------------------------------------ PRUNE_TILE_TRANSPOSABLE
@pytest.mark.parametrize("shape", [(128, 128), (256, 2304), (130, 256), (64, 576)])
@pytest.mark.parametrize("dt", [0, 1])
def test_tile_transposable_equals_tile_mag_without_zeros(spfy, orc, cuda, shape, dt):
    bits = zero_free(orc, dt, shape, seed=3 * shape[0] + shape[1] + dt)
    for layout in (spfy.LAYOUT_SM100, spfy.LAYOUT_CANONICAL):
        c1, d1 = prune_dev(spfy, bits, dt, cuda, spfy.PRUNE_TILE_MAG, layout)
        before = spfy.launch_count()
        c2, d2 = prune_dev(spfy, bits, dt, cuda, spfy.PRUNE_TILE_TRANSPOSABLE, layout)
        assert spfy.launch_count() - before == 1
        assert torch.equal(d1, d2) and torch.equal(c1.vals, c2.vals) and torch.equal(c1.meta, c2.meta)


@pytest.mark.parametrize("dt", [0, 1])
def test_tile_transposable_with_zeros(spfy, orc, cuda, dt):
    rows, cols = 256, 512
    flagged = 0
    for seed in range(4):
        bits = half_zero(orc, dt, (rows, cols), seed=100 + seed)
        want_dense, keep = orc.prune24_tile(dt, bits)
        c1, d1 = prune_dev(spfy, bits, dt, cuda, spfy.PRUNE_TILE_MAG)
        c2, d2 = prune_dev(spfy, bits, dt, cuda, spfy.PRUNE_TILE_TRANSPOSABLE)
        assert torch.equal(d1, d2) and np.array_equal(bits_of(d2), want_dense)
        vals, meta = operand_from_mask(want_dense, keep)  # nibbles = the oracle's TILE pattern
        ov, om = orc.pack_sm100(vals, meta, rows, cols)
        assert np.array_equal(c2.vals.cpu().numpy(), ov) and np.array_equal(c2.meta.cpu().numpy(), om)
        # in place, like TILE_MAG
        a = to_dev(bits, dt, cuda)
        c3 = spfy.prune24(a, inplace=True, mode=spfy.PRUNE_TILE_TRANSPOSABLE)
        assert torch.equal(a, d2) and torch.equal(c3.vals, c2.vals) and torch.equal(c3.meta, c2.meta)
        inv = torch.zeros(1, dtype=torch.int32, device=cuda)
        spfy.transpose24(c2, invalid=inv)
        assert int(inv.item()) == 0
        spfy.transpose24(c1, invalid=inv)
        flagged += int(inv.item())
    # zero-valued survivors move TILE_MAG's recorded indices: its metadata stops being column-balanced
    assert flagged > 0


# ------------------------------------------------------------------ recompress24
@pytest.mark.parametrize("shape", [(256, 512), (200, 72), (130, 260)])
@pytest.mark.parametrize("dt", [0, 1])
def test_recompress24(spfy, orc, cuda, shape, dt):
    rows, cols = shape
    tdt = TDT[dt]
    bits = zero_free(orc, dt, shape, seed=rows + cols + 50 * dt)
    a = to_dev(bits, dt, cuda)
    comp = spfy.prune24(a, out_dense=torch.empty_like(a), mode=spfy.PRUNE_TILE_MAG)
    dense = torch.empty_like(a)
    spfy.prune24(a, out_dense=dense, mode=spfy.PRUNE_TILE_MAG, compress=False)
    meta0 = comp.meta.clone()
    # from the pruned 16-bit matrix: the same values, byte for byte; the metadata untouched
    fresh = spfy.Compressed24(torch.full_like(comp.vals, 0x5A), comp.meta, rows, cols, tdt, comp.layout)
    spfy.recompress24(dense, fresh)
    assert torch.equal(fresh.vals, comp.vals) and torch.equal(comp.meta, meta0)
    keep = dense != 0
    # from fp32: torch's round to nearest even at the kept positions
    g = torch.Generator(device="cpu").manual_seed(rows)
    master = torch.randn(rows, cols, generator=g).to(cuda)
    spfy.recompress24(master, fresh)
    ref = spfy.Compressed24(torch.full_like(comp.vals, 0x33), comp.meta, rows, cols, tdt, comp.layout)
    spfy.recompress24(master.to(tdt), ref)  # 16-bit input of the operand's dtype: its bits are copied
    assert torch.equal(fresh.vals, ref.vals)
    assert torch.equal(spfy.prune24(torch.where(keep, master.to(tdt), torch.zeros((), dtype=tdt, device=cuda))).vals,
                       ref.vals)  # == compressing the rounded, masked master from scratch
    # masked copies: in with every pruned position +0, for fp32 / fp16 / bf16, out of place and in place
    for src in (master, master.to(torch.float16), master.to(torch.bfloat16)):
        want = torch.where(keep, src, torch.zeros((), dtype=src.dtype, device=cuda))
        out = torch.full_like(src, 3.0)
        spfy.recompress24(src, comp, masked_out=out, values=False)
        assert torch.equal(out.view(torch.uint8), want.view(torch.uint8))
        inplace = src.clone()
        spfy.recompress24(inplace, comp, masked_out=inplace, values=False)
        assert torch.equal(inplace.view(torch.uint8), want.view(torch.uint8))
    assert torch.equal(comp.meta, meta0)


# ------------------------------------------------------------------ data gradients
@pytest.mark.parametrize("tokens,in_f,out_f", [(64, 256, 128), (512, 1024, 512), (136, 512, 2048), (1024, 768, 3072)])
def test_linear_data_gradient(spfy, orc, cuda, tokens, in_f, out_f):
    """dx = dy W through comp_t on sparse tensor cores, against fp64"""
    comp, dense = prune_dev(spfy, zero_free(orc, 0, (out_f, in_f), seed=tokens + in_f), 0, cuda,
                            spfy.PRUNE_TILE_TRANSPOSABLE)
    dy = torch.randn(tokens, out_f, device=cuda).to(torch.float16)
    dx = spfy.spmma_compressed(spfy.transpose24(comp), dy, op_b=spfy.OP_T, out_t=True)
    want = dy.double() @ dense.double()
    assert rel_err(dx.double().cpu().numpy(), want.cpu().numpy()) < REL_TOL


@pytest.mark.parametrize("ch,hw", [(64, 56), (128, 28), (256, 14), (512, 7)])
def test_conv3x3_data_gradient(spfy, orc, cuda, ch, hw):
    """dx of a 3x3 stride-1 pad-1 convolution: spmma_conv_nhwc of dy with the transposed, flipped filter"""
    nb, m, c = 8, ch, ch  # n = nb * hw * hw must be a multiple of 8
    w = to_dev(zero_free(orc, 0, (m, c * 9), seed=ch), 0, cuda)
    comp, dense = prune_dev(spfy, bits_of(spfy.permute_conv_weights(w, c, 3, 3)), 0, cuda,
                            spfy.PRUNE_TILE_TRANSPOSABLE)
    dy = torch.randn(nb, hw, hw, m, device=cuda).to(torch.float16)  # NHWC
    dx = spfy.spmma_conv_nhwc(spfy.transpose24(comp, taps=9), dy, 3, 3, stride=1, pad=3 - 1 - 1)
    w_nchw = dense.double().view(m, 3, 3, c).permute(0, 3, 1, 2)
    want = torch.nn.grad.conv2d_input((nb, c, hw, hw), w_nchw, dy.double().permute(0, 3, 1, 2), padding=1)
    assert rel_err(dx.double().permute(0, 3, 1, 2).cpu().numpy(), want.cpu().numpy()) < REL_TOL


# ------------------------------------------------------------------ Linear24
def close(got, want, tol=1e-2):
    """max |got - want| <= tol * max |want|: the layer runs on the 16-bit copy of the fp32 master"""
    got, want = got.detach().double(), want.detach().double()
    return float((got - want).abs().max()) <= tol * float(want.abs().max())


def _torch_ref(layer):
    w = layer.weight.detach().clone().requires_grad_(True)
    b = layer.bias.detach().clone().requires_grad_(True) if layer.bias is not None else None
    return w, b


@pytest.mark.parametrize("tokens,in_f,out_f", [(256, 512, 256), (1024, 1024, 4096)])
def test_linear24_forward_backward(spfy, cuda, tokens, in_f, out_f):
    g = torch.Generator(device="cpu").manual_seed(tokens)
    layer = spfy.Linear24.from_dense(torch.randn(out_f, in_f, generator=g).to(cuda) * 0.05,
                                     torch.randn(out_f, generator=g).to(cuda))
    pruned = layer.weight.detach() == 0
    assert bool((pruned.view(out_f, -1, 4).sum(-1) == 2).all())
    x = (torch.randn(4, tokens // 4, in_f, generator=g) * 0.5).to(cuda).half().requires_grad_(True)
    y = layer(x)
    w, b = _torch_ref(layer)
    xr = x.detach().float().requires_grad_(True)
    yr = torch.nn.functional.linear(xr, w, b)
    assert y.shape == yr.shape and y.dtype == torch.float16
    assert close(y, yr)
    dy = torch.randn(y.shape, generator=g).to(cuda).half()
    y.backward(dy)
    yr.backward(dy.float())
    assert close(x.grad, xr.grad)
    assert close(layer.weight.grad, torch.where(pruned, torch.zeros_like(w.grad), w.grad))
    assert bool((layer.weight.grad[pruned] == 0).all()) and layer.weight.grad.dtype == torch.float32
    assert close(layer.bias.grad, b.grad)


def test_linear24_mlp_sgd_tracks_torch(spfy, cuda):
    """five SGD-with-momentum steps of a two-layer MLP: the same losses and weights as torch on the masked fp32 weights;
    the mask never moves (comp.meta / comp_t.meta byte-identical after every step); forward without refresh() raises"""
    g = torch.Generator(device="cpu").manual_seed(5)
    d_in, d_hid, d_out, tokens = 256, 512, 128, 512
    l1 = spfy.Linear24.from_dense(torch.randn(d_hid, d_in, generator=g).to(cuda) * 0.06, torch.zeros(d_hid, device=cuda))
    l2 = spfy.Linear24.from_dense(torch.randn(d_out, d_hid, generator=g).to(cuda) * 0.04, torch.zeros(d_out, device=cuda))
    ref = [(lay.weight.detach().clone().requires_grad_(True), lay.bias.detach().clone().requires_grad_(True))
           for lay in (l1, l2)]
    masks = [lay.weight.detach() != 0 for lay in (l1, l2)]
    metas = [(lay.comp.meta.clone(), lay.comp_t.meta.clone()) for lay in (l1, l2)]
    params = [p for lay in (l1, l2) for p in (lay.weight, lay.bias)]
    opt = torch.optim.SGD(params, lr=0.05, momentum=0.9)
    opt_ref = torch.optim.SGD([p for pair in ref for p in pair], lr=0.05, momentum=0.9)
    x = torch.randn(tokens, d_in, generator=g).to(cuda).half()
    target = torch.randn(tokens, d_out, generator=g).to(cuda)
    for step in range(5):
        opt.zero_grad()
        h = torch.relu(l1(x))
        loss = ((l2(h).float() - target) ** 2).mean()
        loss.backward()
        opt.step()
        opt_ref.zero_grad()
        hr = torch.relu(torch.nn.functional.linear(x.float(), *ref[0]))
        loss_ref = ((torch.nn.functional.linear(hr, *ref[1]) - target) ** 2).mean()
        loss_ref.backward()
        for (w, _), m in zip(ref, masks):
            w.grad.mul_(m)
        opt_ref.step()
        assert abs(loss.item() - loss_ref.item()) <= 1e-2 * abs(loss_ref.item())
        if step == 0:
            with pytest.raises(RuntimeError, match="refresh"):
                l1(x)
        for lay in (l1, l2):
            lay.refresh()
        for lay, (m, mt), (w, _), mask in zip((l1, l2), metas, ref, masks):
            assert torch.equal(lay.comp.meta, m) and torch.equal(lay.comp_t.meta, mt)
            assert bool((lay.weight.detach()[~mask] == 0).all())
            assert close(lay.weight, w)
