"""Data gradients of strided 2:4 convolutions without a GPU: spfy_transpose24_conv, its size query and
spfy_spmma_conv_dgrad are declared, exported and bound; every argument refusal is returned before any device work; the
phase decomposition reproduces fp64 conv2d_input; and each phase operand, stated in numpy on the canonical layout,
equals the oracle's STRIP compression of the explicitly built sub-filter of a TILE-pruned filter.  The GPU tests
(test_gpu_conv_dgrad.py) check the kernels against the same statement and against fp64."""
import ctypes

import numpy as np
import pytest

from test_transpose24 import expected_sm100, flip_transpose, tile_pruned, transpose24_canonical

NEW = ["spfy_transpose24_conv_bytes", "spfy_transpose24_conv", "spfy_spmma_conv_dgrad"]


def phase_taps(k, s, p, a):
    """filter indices of output phase a, descending: the taps kt with (a + p - kt) % s == 0; dy offset of the first"""
    taps = [kt for kt in range(k - 1, -1, -1) if (a + p - kt) % s == 0]
    return taps, ((a + p - taps[0]) // s if taps else 0)


def phase_order(kh, kw, th, tw):
    """forward tap index (kh * kw_dim + kw) of every column tap t' = i * len(tw) + j of a phase operand"""
    return [h * kw + w for h in th for w in tw]


def phase_subfilter(dense, c, order):
    """the phase operand [c, T*m] built explicitly: S[ci][t'*m + r] = W[r][order[t']*c + ci]"""
    m = dense.shape[0]
    s = np.empty((c, len(order) * m), dtype=dense.dtype)
    for t, src in enumerate(order):
        s[:, t * m:(t + 1) * m] = dense[:, src * c:(src + 1) * c].T
    return s


def phase_canonical(vals, meta, c, order):
    """the transpose rule on the canonical layout, applied to the taps of one phase: A's compressed columns of those taps,
    in reversed phase order (flip_transpose reverses them again) -> (vals', meta', invalid)"""
    rows = vals.shape[0]
    rev = order[::-1]
    sv = np.concatenate([vals[:, t * c // 2:(t + 1) * c // 2] for t in rev], axis=1)
    sm = np.concatenate([meta[:, t * c // 8:(t + 1) * c // 8] for t in rev], axis=1)
    return transpose24_canonical(sv, sm, rows, len(order) * c, len(order))


def phase_tiles(m, c, kh, kw, s, p):
    """(a, b, order, first tile, tiles) of every phase with taps, in (a, b) row-major order"""
    out, tile = [], 0
    for a in range(s):
        for b in range(s):
            th, tw = phase_taps(kh, s, p, a)[0], phase_taps(kw, s, p, b)[0]
            if th and tw:
                n = -(-c // 128) * -(-(len(th) * len(tw) * m) // 128)
                out.append((a, b, phase_order(kh, kw, th, tw), tile, n))
                tile += n
    return out


def dgrad_by_phases(w, dy, h, wd, s, p):
    """dx [nb, c, h, w] of a stride-s, pad-p convolution from w [m, c, kh, kw] and dy [nb, m, ho, wo] (fp64 numpy), phase
    by phase: dx[s*i + a][s*j + b] = sum over the phase's taps of dy[i + dh][j + dw] W[kh][kw], dy outside = 0"""
    m, c, kh, kw = w.shape
    nb, _, ho, wo = dy.shape
    dx = np.zeros((nb, c, h, wd))
    for a in range(s):
        for b in range(s):
            (th, dh0), (tw, dw0) = phase_taps(kh, s, p, a), phase_taps(kw, s, p, b)
            ha, wb = len(range(a, h, s)), len(range(b, wd, s))
            for ih, khi in enumerate(th):
                for iw, kwi in enumerate(tw):
                    for i in range(ha):
                        oh = i + dh0 + ih
                        if not 0 <= oh < ho:
                            continue
                        for j in range(wb):
                            ow = j + dw0 + iw
                            if 0 <= ow < wo:
                                dx[:, :, s * i + a, s * j + b] += dy[:, :, oh, ow] @ w[:, :, khi, kwi]
    return dx


def test_new_symbols_are_declared_exported_and_bound(spfy):
    from test_boundary import declared_symbols
    names = declared_symbols()
    lib = ctypes.CDLL(spfy.capi.LIB_PATH)
    for n in NEW:
        assert n in names and hasattr(lib, n) and n in spfy.capi.SIGNATURES
    for n in ("transpose24_conv", "spmma_conv_dgrad_nhwc", "Transpose24Conv"):
        assert n in spfy.__all__ and callable(getattr(spfy, n))


def _code(spfy, call):
    before = spfy.launch_count()
    with pytest.raises(spfy.SpfyError) as e:
        call()
    assert spfy.launch_count() == before
    return e.value.code


def test_refusals_need_no_device(spfy):
    capi = spfy.capi
    P = ctypes.c_void_p
    a, b, c, d = P(1 << 20), P(2 << 20), P(3 << 20), P(4 << 20)  # 16-byte aligned, never dereferenced
    sz = ctypes.c_size_t()

    def q(dtype=capi.F16, m=64, ch=64, kh=3, kw=3, s=2, p=1):
        return lambda: capi.spfy_transpose24_conv_bytes(dtype, m, ch, kh, kw, s, p, ctypes.byref(sz), ctypes.byref(sz))

    def t(dtype=capi.F16, vals=a, meta=b, m=64, ch=64, kh=3, kw=3, s=2, p=1, vt=c, mt=d):
        return lambda: capi.spfy_transpose24_conv(dtype, vals, meta, m, ch, kh, kw, s, p, vt, mt, None, None)

    for f in (q, t):
        assert _code(spfy, f(dtype=capi.F32)) == capi.E_UNSUPPORTED
        assert _code(spfy, f(m=60)) == capi.E_UNSUPPORTED                  # m % 8
        assert _code(spfy, f(ch=12)) == capi.E_UNSUPPORTED                 # c % 8
        assert _code(spfy, f(kh=17)) == capi.E_UNSUPPORTED
        assert _code(spfy, f(s=9)) == capi.E_UNSUPPORTED
        assert _code(spfy, f(p=9)) == capi.E_UNSUPPORTED
        assert _code(spfy, f(s=0)) == capi.E_INVALID
        assert _code(spfy, f(kw=0)) == capi.E_INVALID
    assert _code(spfy, t(vals=None)) == capi.E_INVALID
    assert _code(spfy, t(mt=None)) == capi.E_INVALID
    assert _code(spfy, t(meta=P((2 << 20) + 8))) == capi.E_INVALID        # SM100 buffers 16-byte aligned
    assert _code(spfy, t(vt=P((3 << 20) + 4))) == capi.E_INVALID

    def g(dtype=capi.F16, nb=2, h=14, w=14, ch=128, kh=3, kw=3, s=2, p=1, m=128, vt=a, mt=b, dy=c, dx=d, desc=True):
        cd = capi.ConvDesc(nb, h, w, ch, kh, kw, s, p)
        return lambda: capi.spfy_spmma_conv_dgrad(dtype, ctypes.byref(cd) if desc else None, m, 1.0, vt, mt, dy, 0.0,
                                                  dx, None)

    assert _code(spfy, g(dtype=capi.F32)) == capi.E_UNSUPPORTED
    assert _code(spfy, g(m=72)) == capi.E_UNSUPPORTED                      # dY is the im2col operand: m % 64
    assert _code(spfy, g(ch=12)) == capi.E_UNSUPPORTED                     # c % 8
    assert _code(spfy, g(s=9)) == capi.E_UNSUPPORTED
    assert _code(spfy, g(p=9)) == capi.E_UNSUPPORTED
    assert _code(spfy, g(kh=17, h=20)) == capi.E_UNSUPPORTED
    assert _code(spfy, g(desc=False)) == capi.E_INVALID
    assert _code(spfy, g(nb=0)) == capi.E_INVALID
    assert _code(spfy, g(h=1, p=0)) == capi.E_INVALID                      # filter larger than the padded image
    assert _code(spfy, g(vt=None)) == capi.E_INVALID
    assert _code(spfy, g(dx=None)) == capi.E_INVALID
    assert _code(spfy, g(dy=P((3 << 20) + 8))) == capi.E_INVALID
    assert _code(spfy, g(dx=P((4 << 20) + 2))) == capi.E_INVALID
    assert _code(spfy, g(mt=P((2 << 20) + 4))) == capi.E_INVALID


# (kh = kw, stride, pad): s in {1, 2, 3}, k in {1, 2, 3, 5, 7}; first dy offsets negative (pad < k - 1), zero and positive
# (1x1 with pad 1: phase 1 reads dy one position ahead).  Then each dimension of the geometries of
# test_gpu_conv24_geometry.py: pad >= filter, stride > filter (phases without taps), 1 x k filters' 1-tap dimension with
# pad 3, and the contract's maxima (16 taps with pad 8 at stride 1 and 8, 11 taps at stride 4)
PHASE_CASES = [(3, 1, 1), (5, 1, 0), (1, 2, 0), (1, 2, 1), (2, 2, 0), (3, 2, 1), (3, 2, 0), (5, 2, 2), (7, 2, 3),
               (1, 3, 1), (2, 3, 2), (3, 3, 1), (5, 3, 0), (7, 3, 3), (3, 3, 4),
               (1, 1, 1), (3, 1, 3), (1, 2, 3), (3, 3, 2), (5, 3, 2), (1, 4, 0), (3, 4, 1), (2, 5, 0), (11, 4, 2),
               (16, 1, 8), (16, 8, 8)]


@pytest.mark.parametrize("k,s,p", PHASE_CASES)
def test_phase_decomposition_is_conv2d_input(k, s, p):
    """the phase rule against torch's fp64 conv2d_input, on odd and non-square images"""
    import torch
    rng = np.random.default_rng(k * 100 + s * 10 + p)
    m, c, nb = 3, 2, 2
    for h, wd in ((7, 9), (k + 2 * s, k + 1)):
        if h + 2 * p < k or wd + 2 * p < k:
            continue
        ho, wo = (h + 2 * p - k) // s + 1, (wd + 2 * p - k) // s + 1
        w = rng.standard_normal((m, c, k, k))
        dy = rng.standard_normal((nb, m, ho, wo))
        ref = torch.nn.grad.conv2d_input((nb, c, h, wd), torch.from_numpy(w), torch.from_numpy(dy), stride=s,
                                         padding=p).numpy()
        np.testing.assert_allclose(dgrad_by_phases(w, dy, h, wd, s, p), ref, rtol=1e-12, atol=1e-12)


def test_phase_offsets():
    """first dy offsets of the cases above: negative, zero and positive all occur"""
    offs = {phase_taps(k, s, p, a)[1] for k, s, p in PHASE_CASES for a in range(s) if phase_taps(k, s, p, a)[0]}
    assert min(offs) < 0 and 0 in offs and max(offs) > 0


@pytest.mark.parametrize("k,s,p", PHASE_CASES)
@pytest.mark.parametrize("m,c", [(16, 24), (8, 8)])
@pytest.mark.parametrize("dtype", [0, 1])
def test_phase_operands_match_the_oracle(spfy, orc, k, s, p, m, c, dtype):
    """every phase operand: the transpose rule on the phase's taps == STRIP compression of the explicit sub-filter; the
    size query covers exactly the phases' tiles"""
    dense = tile_pruned(orc, dtype, m, k * k * c, seed=k * 1000 + s * 100 + p * 10 + m + c + dtype)
    a = orc.prune24_strip(dtype, dense, want_mask=False)
    phases = phase_tiles(m, c, k, k, s, p)
    assert phases
    for _, _, order, _, _ in phases:
        sub = phase_subfilter(dense, c, order)
        rev = np.concatenate([dense[:, t * c:(t + 1) * c] for t in order[::-1]], axis=1)
        assert np.array_equal(flip_transpose(rev, len(order)), sub)
        vt, mt, invalid = phase_canonical(a["vals"], a["meta"], c, order)
        assert invalid == 0
        got = orc.pack_sm100(vt, mt, c, len(order) * m)
        want = expected_sm100(orc, dtype, rev, len(order))
        assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
    if s == 1:  # one phase, the taps of transpose24(taps = k*k)
        assert phases[0][2] == list(range(k * k - 1, -1, -1))
    vb, mb = ctypes.c_size_t(), ctypes.c_size_t()
    spfy.capi.spfy_transpose24_conv_bytes(dtype, m, c, k, k, s, p, ctypes.byref(vb), ctypes.byref(mb))
    tiles = sum(n for *_, n in phases)
    assert (vb.value, mb.value) == (tiles * 16384, tiles * 2048)
