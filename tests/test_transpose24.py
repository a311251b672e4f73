"""2:4 fine-tuning entry points without a GPU: spfy_transpose24 / spfy_recompress24 and PRUNE_TILE_TRANSPOSABLE are
declared, exported and bound; every argument refusal is returned before any device work; and the transpose rule, stated
here in numpy on the canonical layout, agrees with the oracle's STRIP compression of the explicitly transposed
TILE-pruned matrix.  The GPU tests (test_gpu_transpose24.py) check the kernels against the same statement."""
import ctypes

import numpy as np
import pytest

NEW = ["spfy_transpose24", "spfy_recompress24"]


def tile_pruned(orc, dtype, rows, cols, seed):
    """TILE-pruned (oracle) rows x cols matrix of zero-free values: magnitudes in [0.25, 1), random signs"""
    rng = np.random.default_rng(seed)
    x = rng.uniform(0.25, 1.0, (rows, cols)) * rng.choice([-1.0, 1.0], (rows, cols))
    return orc.prune24_tile(dtype, orc.from_f32(dtype, x.astype(np.float32)))[0]


def flip_transpose(a, taps):
    """A [rows, taps*C] -> A' [C, taps*rows],  A'[ci][t'*rows + r] = A[r][(taps-1-t')*C + ci]"""
    rows, cols = a.shape
    c = cols // taps
    return a.reshape(rows, taps, c)[:, ::-1, :].transpose(2, 1, 0).reshape(c, taps * rows)


def transpose24_canonical(vals, meta, rows, cols, taps):
    """The transpose rule on the CANONICAL layout: the kept set of each group of A' is what A's metadata keeps in that
    column of the 4x4 block, values carried bit for bit.  -> (vals', meta', invalid)"""
    G = cols // 4
    nib = np.empty((rows, G), dtype=np.uint8)
    nib[:, 0::2] = meta[:, : (G + 1) // 2] & 0xF
    nib[:, 1::2] = meta[:, : G // 2] >> 4
    v = vals.reshape(rows, G, 2)
    bits = np.zeros((rows, cols), dtype=np.uint16)
    kept = np.zeros((rows, cols), dtype=bool)
    g = np.arange(G)
    for slot, idx in ((0, nib & 3), (1, nib >> 2)):
        bits[np.arange(rows)[:, None], 4 * g + idx] = v[:, :, slot]
        kept[np.arange(rows)[:, None], 4 * g + idx] = True
    bt, kt = flip_transpose(bits, taps), flip_transpose(kept, taps)
    rt, ct = bt.shape
    kq = kt.reshape(rt, ct // 4, 4)
    invalid = int((kq.sum(-1) != 2).any())
    order = np.argsort(~kq, axis=-1, kind="stable")[..., :2]  # the two kept positions, ascending
    vt = np.take_along_axis(bt.reshape(rt, ct // 4, 4), order, -1).reshape(rt, -1)
    nt = (order[..., 0] | (order[..., 1] << 2)).astype(np.uint8)
    mt = np.zeros((rt, (ct // 4 + 1) // 2), dtype=np.uint8)
    mt[:, : (ct // 4 + 1) // 2] = nt[:, 0::2]
    mt[:, : ct // 8] |= nt[:, 1::2] << 4
    return vt, mt, invalid


def expected_sm100(orc, dtype, dense, taps):
    """oracle: STRIP prune + pack_sm100 of the explicitly transposed TILE-pruned matrix"""
    t = flip_transpose(dense, taps)
    ref = orc.prune24_strip(dtype, t, want_mask=False)
    return orc.pack_sm100(ref["vals"], ref["meta"], *t.shape)


def move_kept_pair(dense, bits, row, group):
    """TILE-pruned zero-free `dense` with row `row` of group `group` keeping the other two of its four positions (their
    values from `bits`, zero-free): the row stays 2:4, but two columns of that 4x4 block now keep three and two keep
    one, so the mask is no longer transposable."""
    out = dense.copy()
    cs = slice(4 * group, 4 * group + 4)
    kept = out[row, cs] != 0
    assert kept.sum() == 2 and (bits[row, cs] != 0).all()
    out[row, cs] = np.where(kept, 0, bits[row, cs])
    return out


def test_new_symbols_are_declared_exported_and_bound(spfy):
    from test_boundary import declared_symbols
    names = declared_symbols()
    lib = ctypes.CDLL(spfy.capi.LIB_PATH)
    for n in NEW:
        assert n in names and hasattr(lib, n) and n in spfy.capi.SIGNATURES
    assert spfy.PRUNE_TILE_TRANSPOSABLE == 2
    for n in ("transpose24", "recompress24", "Linear24"):
        assert n in spfy.__all__ and callable(getattr(spfy, n))


def _code(call):
    import __graft_entry__ as ge
    spfy = ge.load_package()
    with pytest.raises(spfy.SpfyError) as e:
        call()
    return e.value.code


def test_refusals_need_no_device(spfy):
    capi = spfy.capi
    P = ctypes.c_void_p
    a, b, c, d = P(1 << 20), P(2 << 20), P(3 << 20), P(4 << 20)  # 16-byte aligned, never dereferenced

    def t24(dtype=capi.F16, vals=a, meta=b, rows=64, cols=64, taps=1, vt=c, mt=d):
        return lambda: capi.spfy_transpose24(dtype, vals, meta, rows, cols, taps, vt, mt, None, None)

    assert _code(t24(dtype=capi.F32)) == capi.E_UNSUPPORTED
    assert _code(t24(taps=0)) == capi.E_INVALID
    assert _code(t24(vals=None)) == capi.E_INVALID
    assert _code(t24(mt=None)) == capi.E_INVALID
    assert _code(t24(cols=64, taps=3)) == capi.E_INVALID                # cols % taps
    assert _code(t24(rows=60)) == capi.E_UNSUPPORTED                    # rows % 8
    assert _code(t24(cols=9 * 12, taps=9)) == capi.E_UNSUPPORTED        # (cols / taps) % 8
    assert _code(t24(rows=1 << 31)) == capi.E_UNSUPPORTED
    assert _code(t24(meta=P((2 << 20) + 8))) == capi.E_INVALID          # SM100 buffers 16-byte aligned
    assert _code(t24(vt=P((3 << 20) + 4))) == capi.E_INVALID

    def rc24(in_dt=capi.F32, inp=a, ld=64, dt=capi.F16, rows=64, cols=64, meta=b, vals=c, out=None, ldo=0):
        return lambda: capi.spfy_recompress24(in_dt, inp, ld, dt, rows, cols, meta, vals, out, ldo, None)

    assert _code(rc24(in_dt=capi.F64)) == capi.E_UNSUPPORTED
    assert _code(rc24(dt=capi.F32)) == capi.E_UNSUPPORTED
    assert _code(rc24(inp=None)) == capi.E_INVALID
    assert _code(rc24(meta=None)) == capi.E_INVALID
    assert _code(rc24(ld=63)) == capi.E_INVALID
    assert _code(rc24(out=d, ldo=32)) == capi.E_INVALID
    assert _code(rc24(cols=1 << 31, ld=1 << 31)) == capi.E_UNSUPPORTED
    assert _code(rc24(meta=P((2 << 20) + 2))) == capi.E_INVALID
    assert _code(rc24(vals=P((3 << 20) + 8))) == capi.E_INVALID
    assert _code(rc24(inp=P((1 << 20) + 2))) == capi.E_INVALID          # fp32 input not 4-byte aligned

    mode = capi.PRUNE_TILE_TRANSPOSABLE

    def pr(out_dense=c, mask=None, cols=64, ld=64):
        return lambda: capi.spfy_prune24(capi.F16, mode, capi.LAYOUT_SM100, a, ld, out_dense, ld, b, d, mask, 64, cols, None)

    assert _code(pr(out_dense=None)) == capi.E_INVALID
    assert _code(pr(mask=P(5 << 20))) == capi.E_UNSUPPORTED
    assert _code(pr(cols=72, ld=72)) == capi.E_UNSUPPORTED              # the one-pass kernel needs cols % 16 == 0
    assert _code(pr(ld=66, cols=64)) == capi.E_UNSUPPORTED              # rows not 8-byte aligned
    items = (capi.Prune24Item * 1)(capi.Prune24Item(a.value, 64, a.value, 64, b.value, d.value, 64, 64))
    assert _code(lambda: capi.spfy_prune24_batched(capi.F16, mode, capi.LAYOUT_SM100,
                                                   ctypes.cast(items, ctypes.c_void_p), 1, None)) == capi.E_INVALID


@pytest.mark.parametrize("rows,cols,taps", [(8, 8, 1), (200, 72, 1), (64, 576, 1), (64, 576, 9), (136, 9 * 24, 9),
                                            (256, 512, 4), (8, 16, 1), (8, 16, 2), (128, 9 * 64, 9), (72, 9 * 64, 9),
                                            (64, 9 * 128, 9), (64, 25 * 64, 25), (64, 49 * 64, 49)])
@pytest.mark.parametrize("dtype", [0, 1])
def test_transpose_rule_matches_the_oracle(orc, rows, cols, taps, dtype):
    dense = tile_pruned(orc, dtype, rows, cols, seed=rows * 31 + cols + taps)
    a = orc.prune24_strip(dtype, dense, want_mask=False)
    vt, mt, invalid = transpose24_canonical(a["vals"], a["meta"], rows, cols, taps)
    assert invalid == 0
    got = orc.pack_sm100(vt, mt, cols // taps, taps * rows)
    want = expected_sm100(orc, dtype, dense, taps)
    assert np.array_equal(got[0], want[0]) and np.array_equal(got[1], want[1])
    # twice with the same taps: the original operand
    v2, m2, inv2 = transpose24_canonical(vt, mt, cols // taps, taps * rows, taps)
    assert inv2 == 0 and np.array_equal(v2, a["vals"]) and np.array_equal(m2, a["meta"])


def test_transpose_rule_flags_a_strip_mask(orc):
    rng = np.random.default_rng(3)
    bits = orc.from_f32(0, rng.uniform(0.25, 1.0, (64, 64)).astype(np.float32))
    a = orc.prune24_strip(0, bits, want_mask=False)
    assert transpose24_canonical(a["vals"], a["meta"], 64, 64, 1)[2] == 1


@pytest.mark.parametrize("rows,cols,row,group", [(64, 64, 0, 0), (64, 64, 37, 9), (200, 136, 199, 33)])
def test_transpose_rule_flags_one_moved_pair(orc, rows, cols, row, group):
    """one row of one 4x4 block keeping the other two positions: still 2:4 along rows, flagged by the rule"""
    rng = np.random.default_rng(rows + row)
    bits = orc.from_f32(0, (rng.uniform(0.25, 1.0, (rows, cols)) * rng.choice([-1.0, 1.0], (rows, cols)))
                        .astype(np.float32))
    dense = orc.prune24_tile(0, bits)[0]
    moved = move_kept_pair(dense, bits, row, group)
    assert orc.prune24_check(0, moved) == 0
    a = orc.prune24_strip(0, moved, want_mask=False)
    assert np.array_equal(a["dense"], moved)
    assert transpose24_canonical(a["vals"], a["meta"], rows, cols, 1)[2] == 1
