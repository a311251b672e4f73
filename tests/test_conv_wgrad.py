"""Weight gradients of 2:4 convolutions without a GPU: spfy_conv_wgrad24 and its workspace query are declared, exported
and bound; the query follows its documented formula (the split count over every ResNet-50 convolution but the stem); every
refusal is returned before any device work; and the layout contract of Conv2d24 holds: the channels_last master's storage
is the (kh, kw, c) order of permute_conv_weights, and the (kh, kw, c) contraction dY^T im2col(X) the kernel computes is
fp64 conv2d_weight in that storage.  The GPU tests (test_gpu_conv_wgrad.py) check the kernels against fp64."""
import ctypes

import numpy as np
import pytest

NEW = ["spfy_conv_wgrad24_workspace_bytes", "spfy_conv_wgrad24"]

# every unique ResNet-50 convolution but the 3-channel stem (torchvision v1.5: the stride sits on the 3x3), b = 32:
# (c, m, input size, k, stride, pad)
RESNET50 = [
    (64, 64, 56, 1, 1, 0), (64, 64, 56, 3, 1, 1), (64, 256, 56, 1, 1, 0), (256, 64, 56, 1, 1, 0),
    (256, 128, 56, 1, 1, 0), (128, 128, 56, 3, 2, 1), (128, 512, 28, 1, 1, 0), (256, 512, 56, 1, 2, 0),
    (512, 128, 28, 1, 1, 0), (128, 128, 28, 3, 1, 1),
    (512, 256, 28, 1, 1, 0), (256, 256, 28, 3, 2, 1), (256, 1024, 14, 1, 1, 0), (512, 1024, 28, 1, 2, 0),
    (1024, 256, 14, 1, 1, 0), (256, 256, 14, 3, 1, 1),
    (1024, 512, 14, 1, 1, 0), (512, 512, 14, 3, 2, 1), (512, 2048, 7, 1, 1, 0), (1024, 2048, 14, 1, 2, 0),
    (2048, 512, 7, 1, 1, 0), (512, 512, 7, 3, 1, 1),
]


def cdiv(a, b):
    return -(-a // b)


def split_count(nb, h, w, c, kh, kw, s, p, m):
    """S of spfy_b200.h: one wave of (split, m-tile, n-tile) units on 148 SMs, at least 8 stages of 64 positions each"""
    ho, wo = (h + 2 * p - kh) // s + 1, (w + 2 * p - kw) // s + 1
    tiles = cdiv(kh * kw * c, 128) * cdiv(m, 256)
    stages = cdiv(nb * ho * wo, 64)
    s0 = max(1, min(148 // tiles, stages // 8))
    return cdiv(stages, cdiv(stages, s0))


def query(spfy, nb, h, w, c, kh, kw, s, p, m, dtype=None):
    capi = spfy.capi
    cd = capi.ConvDesc(nb, h, w, c, kh, kw, s, p)
    sz = ctypes.c_size_t(12345)
    capi.spfy_conv_wgrad24_workspace_bytes(capi.F16 if dtype is None else dtype, ctypes.byref(cd), m, ctypes.byref(sz))
    return sz.value


def test_new_symbols_are_declared_exported_and_bound(spfy):
    from test_boundary import declared_symbols
    names = declared_symbols()
    lib = ctypes.CDLL(spfy.capi.LIB_PATH)
    for n in NEW:
        assert n in names and hasattr(lib, n) and n in spfy.capi.SIGNATURES
    for n in ("conv_wgrad24_nhwc", "Conv2d24"):
        assert n in spfy.__all__ and callable(getattr(spfy, n))


@pytest.mark.parametrize("c,m,hw,k,s,p", RESNET50)
def test_workspace_is_the_documented_formula_on_resnet50(spfy, c, m, hw, k, s, p):
    splits = split_count(32, hw, hw, c, k, k, s, p, m)
    before = spfy.launch_count()
    for dtype in (spfy.capi.F16, spfy.capi.BF16):
        assert query(spfy, 32, hw, hw, c, k, k, s, p, m, dtype) == splits * m * k * k * c * 4
    assert spfy.launch_count() == before
    ho = (hw + 2 * p - k) // s + 1
    tiles = cdiv(k * k * c, 128) * cdiv(m, 256)
    assert splits * tiles <= max(148, tiles)                           # never more than one wave of units
    assert splits == 1 or cdiv(cdiv(32 * ho * ho, 64), splits) >= 8  # and at least 8 stages a unit when split


def test_split_counts_at_both_ends(spfy):
    """the splits of layers at both ends: the 1x1 64->64 layer at 56^2 (one tile, K = 100352 positions) takes 143 splits
    of 11 stages; the 3x3 512->512 layer at 7^2 (72 tiles) two; a layer of one stage none; and odd shapes"""
    assert split_count(32, 56, 56, 64, 1, 1, 1, 0, 64) == 143
    assert split_count(32, 56, 56, 64, 3, 3, 1, 1, 64) == 29
    assert split_count(32, 7, 7, 512, 3, 3, 1, 1, 512) == 2
    assert split_count(32, 7, 7, 512, 1, 1, 1, 0, 2048) == 3
    assert split_count(1, 8, 8, 64, 1, 1, 1, 0, 64) == 1  # one stage: no split
    for args in ((2, 9, 7, 64, 5, 5, 3, 2, 72), (3, 11, 13, 128, 7, 7, 3, 3, 200), (1, 5, 6, 64, 3, 3, 1, 1, 8)):
        nb, h, w, c, kh, kw, s, p, m = args
        assert query(spfy, nb, h, w, c, kh, kw, s, p, m) == split_count(*args) * m * kh * kw * c * 4


def _code(spfy, call):
    before = spfy.launch_count()
    with pytest.raises(spfy.SpfyError) as e:
        call()
    assert spfy.launch_count() == before
    return e.value.code


def test_refusals_need_no_device(spfy):
    capi = spfy.capi
    P = ctypes.c_void_p
    x, dy, meta, dw, ws = P(1 << 20), P(2 << 20), P(3 << 20), P(4 << 20), P(5 << 20)  # aligned, never dereferenced
    big = 1 << 40
    sz = ctypes.c_size_t()

    def args(dtype=capi.F16, nb=2, h=14, w=14, ch=128, kh=3, kw=3, s=2, p=1, m=128, desc=True):
        cd = capi.ConvDesc(nb, h, w, ch, kh, kw, s, p)
        return dtype, (ctypes.byref(cd) if desc else None), m, cd

    def q(**kw):
        dtype, d, m, cd = args(**kw)
        return lambda: (cd, capi.spfy_conv_wgrad24_workspace_bytes(dtype, d, m, ctypes.byref(sz)))

    def g(X=x, DY=dy, META=meta, DW=dw, WS=ws, wsb=big, **kw):
        dtype, d, m, cd = args(**kw)
        return lambda: (cd, capi.spfy_conv_wgrad24(dtype, d, m, 1.0, X, DY, META, 0.0, DW, WS, wsb, None))

    for f in (q, g):
        assert _code(spfy, f(dtype=capi.F32)) == capi.E_UNSUPPORTED
        assert _code(spfy, f(dtype=capi.F64)) == capi.E_UNSUPPORTED
        assert _code(spfy, f(ch=96)) == capi.E_UNSUPPORTED                 # c % 64
        assert _code(spfy, f(m=68)) == capi.E_UNSUPPORTED                  # m % 8
        assert _code(spfy, f(kh=17, h=20)) == capi.E_UNSUPPORTED
        assert _code(spfy, f(kw=17, w=20)) == capi.E_UNSUPPORTED
        assert _code(spfy, f(p=9)) == capi.E_UNSUPPORTED
        assert _code(spfy, f(s=9)) == capi.E_UNSUPPORTED
        assert _code(spfy, f(desc=False)) == capi.E_INVALID
        for empty in ("nb", "h", "w", "ch", "kh", "kw", "s", "m"):
            assert _code(spfy, f(**{empty: 0})) == capi.E_INVALID, empty
        assert _code(spfy, f(h=1, p=0)) == capi.E_INVALID                  # filter larger than the padded image
        assert _code(spfy, f(w=2, p=0)) == capi.E_INVALID
    for name in ("X", "DY", "META", "DW", "WS"):
        assert _code(spfy, g(**{name: None})) == capi.E_INVALID, name
        assert _code(spfy, g(**{name: P((6 << 20) + 8)})) == capi.E_INVALID, name  # 16-byte alignment
    need = query(spfy, 2, 14, 14, 128, 3, 3, 2, 1, 128)
    assert _code(spfy, g(wsb=need - 1)) == capi.E_WORKSPACE
    assert _code(spfy, g(wsb=0)) == capi.E_WORKSPACE


def permute_rule(w2, c, kh, kw):
    """spfy_permute_conv_weights as stated in spfy_b200.h: column (ci, i, j) of a flattened torch weight -> (i, j, ci)"""
    m = w2.shape[0]
    out = np.empty_like(w2)
    for i in range(kh):
        for j in range(kw):
            for ci in range(c):
                out[:, (i * kw + j) * c + ci] = w2[:, (ci * kh + i) * kw + j]
    return out.reshape(m, -1)


def wgrad_khkwc(x, dy, kh, kw, s, p):
    """what the kernel computes, in numpy: dW[r][(i*kw + j)*c + ci] = sum over output positions (n, oh, ow) of
    dy[n, oh, ow, r] * x[n, oh*s - p + i, ow*s - p + j, ci] (x outside the image = 0); x, dy NHWC"""
    nb, h, w, c = x.shape
    _, ho, wo, m = dy.shape
    xp = np.zeros((nb, h + 2 * p + s * ho, w + 2 * p + s * wo, c))
    xp[:, p:p + h, p:p + w] = x
    out = np.zeros((m, kh * kw * c))
    d2 = dy.reshape(-1, m)
    for i in range(kh):
        for j in range(kw):
            cols = xp[:, i:i + s * ho:s, j:j + s * wo:s][:, :ho, :wo].reshape(-1, c)
            out[:, (i * kw + j) * c:(i * kw + j + 1) * c] = d2.T @ cols
    return out


@pytest.mark.parametrize("m,c,kh,kw,s,p,h,w", [(8, 16, 3, 3, 1, 1, 7, 9), (16, 8, 1, 1, 2, 0, 9, 8),
                                               (8, 8, 5, 5, 3, 2, 11, 13), (4, 12, 3, 2, 2, 1, 6, 5)])
def test_conv2d24_layout_contract(m, c, kh, kw, s, p, h, w):
    """the channels_last master's storage is permute_conv_weights of the NCHW weight, and fp64 conv2d_weight in that
    storage is the (kh, kw, c) contraction the kernel computes"""
    import torch
    rng = np.random.default_rng(m * 1000 + c * 10 + kh + s)
    wt = torch.from_numpy(rng.standard_normal((m, c, kh, kw)))
    master = wt.contiguous(memory_format=torch.channels_last)
    w2 = master.permute(0, 2, 3, 1).reshape(m, kh * kw * c)
    assert w2.data_ptr() == master.data_ptr() and w2.is_contiguous()  # a view: optimizers and dW share the storage
    assert np.array_equal(w2.numpy(), permute_rule(wt.reshape(m, -1).numpy(), c, kh, kw))
    nb = 2
    ho, wo = (h + 2 * p - kh) // s + 1, (w + 2 * p - kw) // s + 1
    x = torch.from_numpy(rng.standard_normal((nb, c, h, w)))
    dy = torch.from_numpy(rng.standard_normal((nb, m, ho, wo)))
    ref = torch.nn.grad.conv2d_weight(x, wt.shape, dy, stride=s, padding=p)
    got = wgrad_khkwc(x.permute(0, 2, 3, 1).numpy(), dy.permute(0, 2, 3, 1).numpy(), kh, kw, s, p)
    np.testing.assert_allclose(got, ref.contiguous(memory_format=torch.channels_last).permute(0, 2, 3, 1)
                               .reshape(m, -1).numpy(), rtol=1e-12, atol=1e-12)
