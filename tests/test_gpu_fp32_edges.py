"""The fp32 tensor-core paths at the edges of the fp32 range, against a plain fp64 reference that follows IEEE rules.

Every fp32 product of the library that runs on tensor cores goes through the 3xTF32 splitter of gemm_sm100.cu
(batched::gemm fp32 PRECISE, the COO / CSR and blocked-ELL tensor routes) or through one TF32 product (FAST); these
tests give them what the parity tests never do: values next to FLT_MAX, power-of-two scales out to the subnormal range,
Inf and NaN operands, non-finite B next to structural zeros of a sparse A, and a NaN-filled C with beta = 0.  The
special-value contract they pin is the one written next to SPFY_SPMM_ALG_* and SPFY_GEMM_* in include/spfy_b200.h.

The references form every fp64 product explicitly and sum over k (no BLAS: reference BLAS skips B == 0 terms and so
hides 0 * Inf).  The sparse "stored entries" reference is the CPU oracle's loop over stored entries.  For finite outputs
the bounds are those of tests/test_gpu_tensor.py: |err| <= 4e-6 * sum_k |a||b| (3xTF32), 2e-3 * sum_k |a||b| (one TF32
product), 2e-5 * sum_k |a||b| (CUDA-core fp32 sums); every other output is compared by class: finite, +Inf, -Inf, NaN."""
import ctypes

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

F32_TOL = 4e-6
TF32_TOL = 2e-3
CORE_TOL = 2e-5

QNAN = 0x7FC00000
LOW_NAN = 0x7F800001  # NaN whose payload lies only in the 13 bits TF32 drops: truncated, it reads as +Inf
NONFINITE = {"+inf": 0x7F800000, "-inf": 0xFF800000, "qnan": QNAN, "low_nan": LOW_NAN}

TA_TB = [(0, 0), (1, 0), (0, 1), (1, 1)]
# ragged with nb > 1; k = 147 (ldb not a multiple of 16 bytes: the padded-copy repack path); a plain square-ish tile
# (op(A) is the streamed operand of the 3xTF32 kernel in the first three, op(B) in the last: 40 < 264)
GEMM_SHAPES = [(200, 72, 104, 3), (70, 33, 147, 2), (128, 64, 64, 1), (40, 264, 96, 2)]
# ragged with nb > 1; k = 147 (padded copy of B); a layer of the benchmarked COO workload (resnet50 3x3, 256 x 2304)
SPMM_SHAPES = [(130, 332, 70, 2), (64, 147, 96, 2), (256, 2304, 49, 2)]


def f32(bits):
    return np.array(bits, dtype=np.uint32).view(np.float32)


def classes(x):
    """0 finite, 1 +Inf, 2 -Inf, 3 NaN"""
    c = np.zeros(x.shape, np.int8)
    c[np.isposinf(x)] = 1
    c[np.isneginf(x)] = 2
    c[np.isnan(x)] = 3
    return c


def tf32_read(x):
    """fp32 operand as the tensor core reads it in one TF32 product, for the special values only (finite values stay as
    they are: their truncation is what the 2e-3 bound covers): the low 13 mantissa bits are dropped"""
    bits = np.array(x, dtype=np.float32).view(np.uint32).copy()
    nf = (bits & 0x7F800000) == 0x7F800000
    bits[nf] &= 0xFFFFE000
    return bits.view(np.float32)


def dense_ref(A, B):
    """IEEE fp64 products summed over k: A [nb, m, k], B [nb, k, n] -> [nb, m, n] (chunked over m)"""
    A = np.asarray(A, np.float64)
    B = np.asarray(B, np.float64)
    nb, m, k = A.shape
    out = np.empty((nb, m, B.shape[2]))
    rows = max(1, (1 << 22) // max(1, k * B.shape[2]))
    with np.errstate(invalid="ignore", over="ignore"):
        for b in range(nb):
            for i in range(0, m, rows):
                out[b, i:i + rows] = (A[b, i:i + rows, :, None] * B[b, None]).sum(1)
    return out


def check(got, want, bound, tol, special, what, absolute=0.0, nan_at=None):
    """finite outputs within tol * bound (+ absolute); the others by class.  special: 'ieee' -- the class of every
    non-finite output is the reference's; 'nan' -- every output the reference makes non-finite is NaN.  nan_at: outputs
    that must be NaN although the reference is finite (PRECISE, a streamed value >= 0x7f7ff000: spfy_b200.h)"""
    if nan_at is not None:
        assert nan_at.any() and np.isnan(got[nan_at]).all(), (what, "expected NaN", int((~np.isnan(got[nan_at])).sum()))
        got = np.where(nan_at, want, got)
    with np.errstate(invalid="ignore", over="ignore"):
        _check(got, want, bound, tol, special, what, absolute)


def _check(got, want, bound, tol, special, what, absolute):
    fin = np.isfinite(want)
    bad = np.isfinite(got) != fin
    assert not bad.any(), (what, "finite / non-finite mismatch", int(bad.sum()), tuple(np.argwhere(bad)[0]),
                           got[bad][:4], want[bad][:4])
    allowed = tol(want, bound) if callable(tol) else tol * bound
    err = np.abs(got - want)
    over = fin & ~(err <= allowed + absolute)
    assert not over.any(), (what, "error bound", int(over.sum()), float(np.max(err[fin] / np.maximum(bound[fin], 1e-300))))
    nf = ~fin
    if special == "ieee":
        assert np.array_equal(classes(got)[nf], classes(want)[nf]), (what, "class", classes(got)[nf][:8], classes(want)[nf][:8])
    else:
        assert np.all(np.isnan(got[nf])), (what, "non-finite outputs that are not NaN", classes(got)[nf][:8])


# ------------------------------------------------------------------ dense batched::gemm
def half_tol(eps):
    # fp32 accumulation of exact products, one rounding to the 16-bit output type (tests/test_gpu_tensor.py)
    return lambda want, bound: eps * np.abs(want) + 1e-4 * bound


# name -> (torch dtype, precision name, special-value rule, tolerance)
MODES = {
    "f32_precise": (torch.float32, "GEMM_PRECISE", "nan", F32_TOL),
    "f32_fast": (torch.float32, "GEMM_FAST", "ieee", TF32_TOL),
    "f16": (torch.float16, "GEMM_PRECISE", "ieee", half_tol(2.0 ** -11)),
    "bf16": (torch.bfloat16, "GEMM_PRECISE", "ieee", half_tol(2.0 ** -8)),
}


def run_gemm(spfy, cuda, A, B, ta, tb, mode, strided=True, alpha=1.0):
    """C = alpha * op(A) op(B) with beta = 0 over a NaN-filled C.  A [nb, m, k], B [nb, k, n]: logical op() shapes in
    float32 (bit patterns kept), converted to the mode's type.  Returns (got, want, bound) in fp64, [nb, m, n]; the
    reference is formed from the operands as the GPU received them (as the tensor core reads them for FAST)."""
    tdt, prec = MODES[mode][0], getattr(spfy, MODES[mode][1])
    nb, m, k = A.shape
    n = B.shape[2]
    tA, tB = torch.from_numpy(np.ascontiguousarray(A)).to(tdt), torch.from_numpy(np.ascontiguousarray(B)).to(tdt)
    # storage: column-major op() shape, or its transpose when the flag says T
    dA = (tA.transpose(1, 2) if ta == spfy.OP_N else tA).contiguous().to(cuda)
    dB = (tB.transpose(1, 2) if tb == spfy.OP_N else tB).contiguous().to(cuda)
    dC = torch.full((nb, n, m), float("nan"), dtype=tdt, device=cuda)
    spfy.batched.gemm(dA, dB, dC, m, n, k, transpose_a=ta, transpose_b=tb, alpha=alpha, beta=0.0, precision=prec,
                      strided=strided)
    got = dC.double().cpu().numpy().transpose(0, 2, 1)
    A64, B64 = tA.double().numpy(), tB.double().numpy()
    if mode == "f32_fast":
        A64, B64 = tf32_read(A).astype(np.float64), tf32_read(B).astype(np.float64)
    want = alpha * dense_ref(A64, B64)
    bound = abs(alpha) * dense_ref(np.abs(A64), np.abs(B64))
    return got, want, bound


EDGE = float(np.array([0x7F7FF000], np.uint32).view(np.float32)[0])  # from here PRECISE may round hi into Inf


def near_edge(x):
    """finite entries with |x| >= EDGE"""
    return np.isfinite(x) & (np.abs(x) >= EDGE)


def streamed_is_a(m, n, ta, tb):
    """whether the 3xTF32 kernel streams op(A) (rounds its hi) or op(B): orient() of gemm_sm100.cu with 128-column tiles
    -- the mapping that issues fewer padded MACs, ties to the larger of m and n"""
    def split(nu, gran):
        tiles = -(-nu // 128)
        b = min(-(-(-(-nu // tiles)) // gran) * gran, 128)
        return b * -(-nu // b)
    p0 = -(-m // 128) * 128 * split(n, 32 if tb == 1 else 16)  # m along the tiles: op(A) streamed
    p1 = -(-n // 128) * 128 * split(m, 32 if ta == 0 else 16)
    return p0 < p1 if p0 != p1 else m >= n


def precise_nan_at(A, B, ta, tb):
    """[nb, m, n]: the outputs PRECISE makes NaN from finite operands -- the whole row (column) of C of a row of op(A)
    (column of op(B)) that holds a value >= 0x7f7ff000, if that operand is the streamed one; None if there are none"""
    nb, m, _ = A.shape
    n = B.shape[2]
    out = np.zeros((nb, m, n), bool)
    if streamed_is_a(m, n, ta, tb):
        out |= near_edge(A).any(2)[:, :, None]
    else:
        out |= near_edge(B).any(1)[:, None, :]
    return out if out.any() else None


def big_values(mode):
    """the largest finite values of the operand type, including (fp32) the rounding edge of the 3xTF32 split: from
    0x7f7ff000 up, rounding x to the nearest TF32 carries into the Inf exponent"""
    if mode.startswith("f32"):
        bits = [0x7F7FFFFF, 0x7F7FF000, 0x7F7FEFFF]
    elif mode == "bf16":
        bits = [0x7F7F0000, 0x7F7E0000, 0x7F700000]
    else:
        return [65504.0, 65472.0, 65440.0, -65504.0, -65472.0, -65440.0]
    v = f32(bits).astype(np.float64)
    return list(v) + list(-v)


@pytest.mark.parametrize("m,n,k,nb", GEMM_SHAPES)
@pytest.mark.parametrize("ta,tb", TA_TB)
@pytest.mark.parametrize("mode", list(MODES))
def test_gemm_near_overflow_stays_finite(spfy, cuda, mode, ta, tb, m, n, k, nb):
    """Single entries at FLT_MAX (0x7f7fffff), at the split's rounding edge 0x7f7ff000, just below it (0x7f7fefff) and
    their negatives, on the A side and on the B side, times partners of about 2^-11 (|x * b| <= 2^118, at most three of
    them in one row): every exact sum lies far inside the fp32 range, so every output is finite and within the mode's
    bound -- except on PRECISE, where a value with |x| >= 0x7f7ff000 in the streamed operand (spfy_b200.h: its hi is
    rounded to nearest and carries into the Inf exponent) makes its whole row or column of C NaN, and in the other operand
    (hi truncated) stays finite and accurate.  0x7f7fefff is finite everywhere.
    (The 16-bit control uses the largest values of its own type.)"""
    rng = np.random.default_rng(m + n + k + 17 * ta + 5 * tb)
    bigs = big_values(mode)
    kks = [0, k // 2, k - 1]
    for side in ("A", "B"):
        A = rng.uniform(-1, 1, (nb, m, k)).astype(np.float32)
        B = rng.uniform(-1, 1, (nb, k, n)).astype(np.float32)
        small = (2.0 ** -11 * rng.uniform(1, 2, (nb, len(kks), max(m, n))) * rng.choice([-1, 1], (nb, len(kks), max(m, n))))
        if side == "A":
            B[:, kks, :] = small[:, :, :n]
            for t, i in enumerate(range(0, m, max(1, m // 12))):
                A[:, i, kks[t % 3]] = bigs[t % len(bigs)]
            A[:, m - 1, kks[0]], A[:, m - 1, kks[2]] = bigs[0], bigs[len(bigs) // 2]  # two in one row
        else:
            A[:, :, kks] = small[:, :, :m].transpose(0, 2, 1)
            for t, j in enumerate(range(0, n, max(1, n // 12))):
                B[:, kks[t % 3], j] = bigs[t % len(bigs)]
            B[:, kks[1], n - 1], B[:, kks[2], n - 1] = bigs[1], bigs[len(bigs) // 2 + 1]
        got, want, bound = run_gemm(spfy, cuda, A, B, ta, tb, mode)
        assert np.isfinite(want).all() and np.abs(want).max() < 2.0 ** 122
        nan_at = precise_nan_at(A, B, ta, tb) if mode == "f32_precise" else None
        check(got, want, bound, MODES[mode][3], MODES[mode][2], (mode, side), nan_at=nan_at)


# p, q: A scaled by 2^p, B by 2^q.  Operands are drawn with magnitudes in [1/2, 1), so every hi lies in [2^-1, 1],
# every nonzero lo in [2^-24, 2^-10] and the products of the split in [2^-25, 1]: all of them stay normal while
# p, q >= -102 and p + q >= -101 (the bound that binds: a hi * lo product).
SCALES_NORMAL = [(0, 0), (60, 0), (0, 60), (100, 20), (-100, 100), (100, -100), (-50, -51), (-101, 0), (0, -101),
                 (120, -2), (-30, -60)]
# subnormal lo parts and products, where the fp64 bound alone was measured to hold on a B200 (below)
SCALES_BOUND = [(-102, 0), (0, -103), (-110, 0), (0, -112), (-56, -56), (-60, -60), (-62, -58)]
# lo parts, products, results or whole operands far below 2^-126: the bound needs its absolute term
SCALES_SUBNORMAL = [(-120, 0), (0, -122), (-126, 0), (0, -126), (-126, 10), (-130, 20), (-66, -66), (-70, -55),
                    (-80, -80)]


def unit_magnitudes(rng, shape):
    return (rng.uniform(0.5, 1.0, shape) * rng.choice([-1, 1], shape)).astype(np.float32)


@pytest.mark.parametrize("m,n,k,nb", GEMM_SHAPES)
@pytest.mark.parametrize("ta,tb", TA_TB)
@pytest.mark.parametrize("mode", ["f32_precise", "f32_fast"])
def test_gemm_power_of_two_scaling(spfy, cuda, mode, ta, tb, m, n, k, nb):
    """gemm(2^p A, 2^q B) == 2^(p+q) gemm(A, B) bit for bit while every hi, lo and product of the split is normal
    (SCALES_NORMAL, derived above): the split works on mantissa bits, and neither the tensor core nor the fp32
    accumulation depends on a power-of-two scale shared by all terms.

    Measured on a B200 (1000 W limit), shapes 200x72x104 and 128x64x64: bitwise scaling holds further down, to p = -112
    (q = 0) and p = q = -57 for PRECISE, p = -125 and p = q = -63 for FAST -- tcgen05 kind::tf32 reads subnormal TF32
    inputs (spacing 2^-136) and keeps subnormal products instead of flushing them.  The fp64 bound alone holds to
    p = -119 and p = q = -65 (PRECISE), p = -128 (FAST), and fails from p = -120, p = q = -66 and p = -129.  So the bound
    is asserted alone down to SCALES_BOUND (p, q >= -112, p + q >= -120: a margin of five or more binades), and
    below that (SCALES_SUBNORMAL) with an absolute term.  Read as TF32, a piece (hi or lo) below 2^-126 loses less than
    the subnormal spacing 2^-136, and it multiplies at most two partner pieces of magnitude <= 2|partner|: per k less
    than 2^-134 (|a_k| + |b_k|).  Each of the three products per k and each addition of the fp32 accumulation rounds to
    the subnormal spacing 2^-149 at worst, and the result once more.  Per output:
        |err| <= tol * sum_k |a_k||b_k| + 2^-134 * sum_k (|a_k| + |b_k|) + 2^-149 * (3k + 1)
    in the scaled values (measured: at most 1/10 of that term)."""
    rng = np.random.default_rng(3 * m + n + k + ta + 2 * tb)
    A = unit_magnitudes(rng, (nb, m, k))
    B = unit_magnitudes(rng, (nb, k, n))
    base, _, _ = run_gemm(spfy, cuda, A, B, ta, tb, mode)
    tol = MODES[mode][3]
    for p, q in SCALES_NORMAL + SCALES_BOUND + SCALES_SUBNORMAL:
        As = (A.astype(np.float64) * 2.0 ** p).astype(np.float32)
        Bs = (B.astype(np.float64) * 2.0 ** q).astype(np.float32)
        got, want, bound = run_gemm(spfy, cuda, As, Bs, ta, tb, mode)
        absolute = 0.0
        if (p, q) in SCALES_NORMAL:
            assert np.array_equal(got, base * 2.0 ** (p + q)), (p, q, float(np.max(np.abs(got - base * 2.0 ** (p + q)))))
        elif (p, q) in SCALES_SUBNORMAL:
            sa = np.abs(As.astype(np.float64)).sum(2)[:, :, None]  # [nb, m, 1]
            sb = np.abs(Bs.astype(np.float64)).sum(1)[:, None, :]  # [nb, 1, n]
            absolute = 2.0 ** -134 * (sa + sb) + 2.0 ** -149 * (3 * k + 1)
        check(got, want, bound, tol, "ieee", (p, q), absolute=absolute)


@pytest.mark.parametrize("m,n,k,nb", GEMM_SHAPES)
@pytest.mark.parametrize("ta,tb", TA_TB)
@pytest.mark.parametrize("mode", list(MODES))
def test_gemm_nonfinite_operands(spfy, cuda, mode, ta, tb, m, n, k, nb):
    """+Inf, -Inf, a quiet NaN and a NaN with payload only in the low 13 bits (0x7f800001), on the A side and on the B
    side, against finite nonzero, zero, +Inf and -Inf partners, and in a row (column) that also holds its negative.  In
    every mode an output is non-finite exactly where the IEEE reference's is.  f16 / bf16: the IEEE class as well.  FAST:
    the IEEE class of the operands as the tensor core reads them (0x7f800001 truncated reads as +Inf).  PRECISE: NaN
    wherever the reference is non-finite, ±Inf included (the split of an Inf or NaN has lo = NaN)."""
    rng = np.random.default_rng(m * n + k + 3 * ta + tb)
    for name, bits in NONFINITE.items():
        s = f32([bits])[0]
        neg = f32([bits ^ 0x80000000])[0]
        for side in ("A", "B"):
            A = rng.uniform(-1, 1, (nb, m, k)).astype(np.float32)
            B = rng.uniform(-1, 1, (nb, k, n)).astype(np.float32)
            k0, k1 = 1, k - 2
            if side == "A":
                A[:, 0, k0] = s                                 # row 0: against B row k0
                A[:, m - 1, k0], A[:, m - 1, k1] = s, neg       # a row with x and -x
                B[:, k0, 1] = 0.0
                B[:, k0, 2], B[:, k0, n - 1] = np.inf, -np.inf
            else:
                B[:, k0, 0] = s
                B[:, k0, n - 1], B[:, k1, n - 1] = s, neg
                A[:, 1, k0] = 0.0
                A[:, 2, k0], A[:, m - 1, k0] = np.inf, -np.inf
            got, want, bound = run_gemm(spfy, cuda, A, B, ta, tb, mode)
            check(got, want, bound, MODES[mode][3], MODES[mode][2], (mode, name, side))


@pytest.mark.parametrize("strided", [True, False])
@pytest.mark.parametrize("mode", list(MODES))
def test_gemm_beta_zero_never_reads_c(spfy, cuda, mode, strided):
    """beta = 0 over a NaN-filled C, every GEMM kernel and both entries (strided, pointer array): C is written without
    being read, as BLAS does -- every output is finite and within the bound"""
    rng = np.random.default_rng(4)
    for m, n, k, nb in GEMM_SHAPES:
        for ta, tb in TA_TB:
            A = rng.uniform(-1, 1, (nb, m, k)).astype(np.float32)
            B = rng.uniform(-1, 1, (nb, k, n)).astype(np.float32)
            got, want, bound = run_gemm(spfy, cuda, A, B, ta, tb, mode, strided=strided, alpha=0.75)
            check(got, want, bound, MODES[mode][3], MODES[mode][2], (mode, m, n, k, ta, tb))


# ------------------------------------------------------------------ unstructured SpMM: COO / CSR, blocked-ELL
def dense_walk_density():
    return 0.35   # CUDA_CORE takes the dense walk from this fraction of non-zeros (spfy_b200.h)


def tensor_density(k):
    return 0.2 if (k * 4) % 16 else 0.02  # DEFAULT: tensor route from 2 %, 20 % when B needs the padded copy


def coo_semantics(alg, density, k):
    """(semantics, special-value rule, tolerance) of a CSR / COO route, as spfy_b200.h documents them"""
    if alg == "DEFAULT":
        alg = "TENSOR" if density >= tensor_density(k) else "CUDA_CORE"
    if alg == "CUDA_CORE":
        return ("dense" if density >= dense_walk_density() else "stored"), "ieee", CORE_TOL
    return "dense", ("nan" if alg == "TENSOR" else "ieee"), (F32_TOL if alg == "TENSOR" else TF32_TOL)


def BELL_SEMANTICS(alg):
    if alg == "CUDA_CORE":
        return "stored", "ieee", CORE_TOL
    return "dense", ("ieee" if alg == "TENSOR_FAST" else "nan"), (TF32_TOL if alg == "TENSOR_FAST" else F32_TOL)


def coo_matrix(rng, m, k, density):
    """row-sorted COO with exactly round(density * m * k) distinct entries, values in +-[1/2, 1)"""
    nnz = max(1, int(round(density * m * k)))
    flat = np.sort(rng.choice(m * k, nnz, replace=False))
    ri, ci = (flat // k).astype(np.int32), (flat % k).astype(np.int32)
    return ri, ci, unit_magnitudes(rng, nnz)


def coo_refs(orc, m, k, n, nb, ri, ci, va, B, fast):
    """{"stored": oracle over stored entries, "dense": IEEE over the dense image}, bounds, all [nb, n, m] fp64"""
    if fast:  # (A's image is built by fp32 adds of the stored values, which quiet every NaN: only B is read truncated)
        B = tf32_read(B)
    stored = orc.spmm_coo_batched_f64(m, k, n, nb, ri, ci, va, B)
    bound = orc.spmm_coo_batched_f64(m, k, n, nb, ri, ci, np.abs(va), np.abs(B))
    dense = np.zeros((m, k))
    np.add.at(dense, (ri, ci), va.astype(np.float64))
    img = dense_ref(np.broadcast_to(dense, (nb, m, k)), B.transpose(0, 2, 1)).transpose(0, 2, 1)
    return {"stored": stored, "dense": img}, bound


def run_coo(spfy, cuda, fmt, alg, m, k, n, nb, ri, ci, va, B, C=None, alpha=1.0, beta=0.0):
    dri, dci, dva, dB = (torch.from_numpy(np.ascontiguousarray(x)).to(cuda) for x in (ri, ci, va, B))
    dC = (torch.full((nb, n, m), float("nan"), device=cuda) if C is None else torch.from_numpy(C.copy()).to(cuda))
    algc = getattr(spfy, "SPMM_ALG_" + alg)
    if fmt == "coo":
        spfy.batched.strided_coo(m, k, ri.size, k, n, nb, dri, dci, dva, dB, dC, alpha=alpha, beta=beta, alg=algc)
    else:
        spfy.batched.csr(m, k, n, nb, spfy.coo_to_csr(dri, m), dci, dva, dB, dC, alpha=alpha, beta=beta, alg=algc)
    return dC.double().cpu().numpy()


def spmm_check(spfy, orc, cuda, fmt, m, k, n, nb, density, ri, ci, va, B, what, nan_at=None):
    refs = {}
    for alg in ("CUDA_CORE", "TENSOR", "TENSOR_FAST", "DEFAULT"):
        sem, special, tol = coo_semantics(alg, density, k)
        fast = alg == "TENSOR_FAST"
        if fast not in refs:
            refs[fast] = coo_refs(orc, m, k, n, nb, ri, ci, va, B, fast)
        want, bound = refs[fast][0][sem], refs[fast][1]
        got = run_coo(spfy, cuda, fmt, alg, m, k, n, nb, ri, ci, va, B)
        check(got, want, bound, tol, special, (fmt, alg, density, sem) + what,
              nan_at=nan_at if special == "nan" else None)


@pytest.mark.parametrize("m,k,n,nb", SPMM_SHAPES)
@pytest.mark.parametrize("fmt", ["coo", "csr"])
def test_coo_csr_near_overflow_stays_finite(spfy, orc, cuda, fmt, m, k, n, nb):
    """stored values at 0x7f7fffff, 0x7f7ff000, 0x7f7fefff and their negatives, times B entries of about 2^-11, with
    A at 10 % non-zeros: every route (CUDA_CORE, TENSOR, TENSOR_FAST, DEFAULT) gives finite outputs within its bound,
    except that the PRECISE tensor routes make NaN the rows of C that store a value with |x| >= 0x7f7ff000 when they
    stream A's image, which they do when m >= n * nb here (256 x 2304; in the other two B is streamed and every output
    stays finite)"""
    rng = np.random.default_rng(m + k + n)
    ri, ci, va = coo_matrix(rng, m, k, 0.1)
    B = unit_magnitudes(rng, (nb, n, k))
    bigs = big_values("f32")
    cols = np.unique(ci[::max(1, ri.size // 12)])[:6]
    B[:, :, cols] *= 2.0 ** -11
    for t, c in enumerate(cols):
        e = np.nonzero(ci == c)[0]
        va[e] = bigs[t % len(bigs)]
    nan_at = None
    # the tensor routes multiply the row-major dense image of A (op = T) by the batches of B side by side (op = N)
    if streamed_is_a(m, n * nb, 1, 0):
        nan_at = np.zeros((nb, n, m), bool)
        nan_at[:, :, ri[near_edge(va)]] = True
    spmm_check(spfy, orc, cuda, fmt, m, k, n, nb, 0.1, ri, ci, va, B, ("near overflow",), nan_at=nan_at)


@pytest.mark.parametrize("m,k,n,nb", SPMM_SHAPES)
@pytest.mark.parametrize("fmt", ["coo", "csr"])
def test_coo_csr_nonfinite_stored_values(spfy, orc, cuda, fmt, m, k, n, nb):
    """+Inf, -Inf, a quiet NaN and 0x7f800001 as stored values of A (10 % non-zeros), against finite, zero and ±Inf
    entries of B.  A stored entry is part of both semantics, so every route makes the same outputs non-finite as the
    IEEE reference; CUDA_CORE with the IEEE class, TENSOR_FAST with the IEEE class of A's image (built by adding the
    stored values, so 0x7f800001 in A stays NaN) times B truncated to TF32, TENSOR (and DEFAULT at this density, except
    for k = 147 where it takes the CUDA-core kernel) with NaN."""
    rng = np.random.default_rng(7 * m + k + n)
    ri, ci, va0 = coo_matrix(rng, m, k, 0.1)
    for name, bits in NONFINITE.items():
        va = va0.copy()
        B = unit_magnitudes(rng, (nb, n, k))
        e0, e1 = 0, ri.size - 1                   # first entry of the first stored row, last of the last
        va[e0] = va[e1] = f32([bits])[0]
        B[:, 1, ci[e0]] = 0.0
        B[:, 2, ci[e0]], B[:, n - 1, ci[e1]] = np.inf, -np.inf
        spmm_check(spfy, orc, cuda, fmt, m, k, n, nb, 0.1, ri, ci, va, B, (name,))


@pytest.mark.parametrize("m,k,n,nb", SPMM_SHAPES)
@pytest.mark.parametrize("density", [0.01, 0.1, 0.5])
@pytest.mark.parametrize("fmt", ["coo", "csr"])
def test_coo_csr_nonfinite_b_next_to_structural_zeros(spfy, orc, cuda, fmt, density, m, k, n, nb):
    """a non-finite B[kk][j] (+Inf, -Inf, quiet NaN, 0x7f800001) in a column kk that some rows store (one of them a
    stored zero) and most do not.  Per spfy_b200.h: the per-non-zero CUDA-core kernels (CUDA_CORE below 35 %, DEFAULT
    below 2 % -- 20 % for k = 147) follow the stored entries, so only the rows that store column kk are reached, IEEE
    classes; the dense routes (every tensor route, the CUDA-core dense walk at 50 %) multiply the dense image, so all of
    column j of C_b is non-finite, NaN in the rows that do not store kk.  Run at 1 %, 10 % and 50 % non-zeros: DEFAULT on
    each side of 2 %, CUDA_CORE on each side of 35 %."""
    rng = np.random.default_rng(m + 3 * k + n + int(density * 100))
    ri, ci, va0 = coo_matrix(rng, m, k, density)
    counts = np.bincount(ci, minlength=k)
    kk = int(np.argmax((counts > 1) & (counts < m)))  # stored by some rows, not all
    assert 1 < counts[kk] < m
    va0[np.nonzero(ci == kk)[0][0]] = 0.0              # a stored zero in column kk
    for name, bits in NONFINITE.items():
        B = unit_magnitudes(rng, (nb, n, k))
        B[0, 0, kk] = f32([bits])[0]
        B[nb - 1, n - 1, kk] = f32([bits ^ 0x80000000])[0]
        spmm_check(spfy, orc, cuda, fmt, m, k, n, nb, ri.size / (m * k), ri, ci, va0, B, (name,))


def bell_matrix(rng, m, k, block, ell_cols):
    """blocked-ELL with ids in ascending order, every fifth id a padding id -1 (stores nothing)"""
    bcols = ell_cols // block
    ci = np.stack([np.sort(rng.choice(-(-k // block), bcols, replace=False)) for _ in range(-(-m // block))]).astype(np.int64)
    ci[:, ::5] = -1
    return ci, unit_magnitudes(rng, (m, ell_cols))


def bell_dense(m, k, block, ell_cols, ci, va):
    """dense image of one blocked-ELL matrix (padding ids store nothing)"""
    rows = np.repeat(np.arange(m), ell_cols).reshape(m, ell_cols)
    e = np.arange(ell_cols)[None, :]
    bc = ci[rows // block, e // block]
    cols = bc * block + e % block
    keep = (bc >= 0) & (cols < k)
    d = np.zeros((m, k))
    np.add.at(d, (rows[keep], cols[keep]), va[keep].astype(np.float64))
    return d


def run_bell(spfy, cuda, alg, m, n, k, block, ell_cols, cis, vas, B, cs=None, beta=0.0, ws_alg=None):
    """ws_alg: size the workspace for this algorithm instead of `alg` (DEFAULT with a CUDA_CORE workspace has no tensor
    route)"""
    cs = cs if cs is not None else [torch.full((n, m), float("nan"), device=cuda) for _ in cis]
    if ws_alg is not None:
        capi = spfy.capi
        wb = ctypes.c_size_t()
        capi.spfy_spmm_bell_workspace_bytes(getattr(capi, "SPMM_ALG_" + ws_alg), capi.F32, m, k, n, len(cis), ctypes.byref(wb))
        ws = torch.empty(wb.value, dtype=torch.uint8, device=cuda)
        keep = [torch.from_numpy(c).to(cuda) for c in cis], [torch.from_numpy(v).to(cuda) for v in vas]
        tab = [torch.tensor([t.data_ptr() for t in lst], dtype=torch.int64, device=cuda) for lst in (keep[0], keep[1], cs)]
        dB = torch.from_numpy(B).to(cuda)
        capi.spfy_spmm_bell_batched(getattr(capi, "SPMM_ALG_" + alg), capi.F32, m, k, n, block, ell_cols, len(cis),
                                    tab[0].data_ptr(), tab[1].data_ptr(), dB.data_ptr(), k, tab[2].data_ptr(), m, 1.0, beta,
                                    ws.data_ptr(), ws.numel(), None)
        return [c.double().cpu().numpy() for c in cs]
    spfy.batched.spmm([torch.from_numpy(c).to(cuda) for c in cis], [torch.from_numpy(v).to(cuda) for v in vas],
                      torch.from_numpy(B).to(cuda), cs, m, n, k, block, ell_cols, beta=beta,
                      alg=getattr(spfy, "SPMM_ALG_" + alg))
    return [c.double().cpu().numpy() for c in cs]


BELL_SHAPES = [(200, 152, 448, 3, 4), (130, 40, 147, 2, 3), (64, 48, 128, 2, 2)]


@pytest.mark.parametrize("m,n,k,nb,block", BELL_SHAPES)
@pytest.mark.parametrize("case", ["near_overflow", "nonfinite_values", "nonfinite_b", "nonfinite_b_fallback"])
def test_blocked_ell_edges(spfy, orc, cuda, case, m, n, k, nb, block):
    """fp32 blocked-ELL (padding ids included), every route:
    near_overflow   : block values at 0x7f7fffff, 0x7f7ff000, 0x7f7fefff and negatives times B rows of about 2^-11 --
                      finite, within the bound -- TENSOR / DEFAULT stream A's image here, so its rows that hold
                      |x| >= 0x7f7ff000 are NaN (spfy_b200.h);
    nonfinite_values: ±Inf, NaN, 0x7f800001 as block values -- non-finite exactly where the IEEE reference is;
    nonfinite_b     : a non-finite B[kk][j] in a block column some block rows store and others do not (or only through
                      a padding id) -- CUDA_CORE follows the stored entries (IEEE classes; a stored zero gives NaN), the
                      tensor routes (TENSOR, TENSOR_FAST, DEFAULT) the dense image: all of column j non-finite;
    nonfinite_b_fallback: the same with a block-row of batch 0 that repeats an id -- the chunk runs on the CUDA-core
                      kernel on every route, stored entries and IEEE classes -- and DEFAULT given a workspace sized for
                      CUDA_CORE (no tensor route): the same.
    Classes: CUDA_CORE IEEE, TENSOR_FAST IEEE of the operands truncated to TF32, TENSOR / DEFAULT NaN."""
    rng = np.random.default_rng(m + n + k + block + len(case))
    ell_cols = (k // 2) // block * block
    vals = [("+inf", 0x7F800000), ("-inf", 0xFF800000), ("qnan", QNAN), ("low_nan", LOW_NAN)]
    for name, bits in (vals if case != "near_overflow" else [("big", None)]):
        cis, vas = zip(*[bell_matrix(rng, m, k, block, ell_cols) for _ in range(nb)])
        cis, vas = list(cis), [v.copy() for v in vas]
        B = unit_magnitudes(rng, (n, k))
        if case == "near_overflow":
            bigs = big_values("f32")
            B[:, : 2 * block] *= 2.0 ** -11
            for b in range(nb):
                for br in range(cis[b].shape[0]):
                    hit = np.nonzero((cis[b][br] >= 0) & (cis[b][br] < 2))[0]
                    if hit.size:
                        e = hit[0] * block + br % block
                        vas[b][br * block, e] = bigs[(br + b) % len(bigs)]
        elif case == "nonfinite_values":
            for b in range(nb):
                vas[b][0, block] = f32([bits])[0]
                vas[b][m - 1, ell_cols - 1] = f32([bits ^ 0x80000000])[0]
            B[1, :] = np.where(np.arange(k) % 3 == 0, 0.0, B[1, :])
            B[2, k // 2], B[n - 1, 0] = np.inf, -np.inf
        else:
            stored = np.concatenate([c.ravel() for c in cis])
            bc = int(np.bincount(stored[stored >= 0]).argmax())
            kk = bc * block
            for b in range(nb):
                r, e = np.argwhere(cis[b] == bc)[0]
                vas[b][r * block, e * block] = 0.0  # a stored zero in column kk
            B[0, kk] = f32([bits])[0]
            B[n - 1, kk] = f32([bits ^ 0x80000000])[0]
        runs = [(alg, None) for alg in ("CUDA_CORE", "TENSOR", "TENSOR_FAST", "DEFAULT")]
        fallback = case == "nonfinite_b_fallback"
        if fallback:
            own = cis[0][3, 2]
            cis[0][3, 2] = cis[0][3, 1]  # a repeated id: the chunk goes to the CUDA-core stand-in
            runs.append(("DEFAULT", "CUDA_CORE"))
        for alg, ws_alg in runs:
            if ws_alg is not None:  # (without the repeated id: only the missing tensor route makes it CUDA-core)
                cis[0][3, 2] = own
            sem, special, tol = ("stored", "ieee", CORE_TOL) if fallback else BELL_SEMANTICS(alg)
            fast = alg == "TENSOR_FAST" and not fallback
            Bu = tf32_read(B) if fast else B
            gots = run_bell(spfy, cuda, alg, m, n, k, block, ell_cols, cis, vas, B, ws_alg=ws_alg)
            for b in range(nb):
                va = tf32_read(vas[b]) if fast else vas[b]
                bound = orc.spmm_bell_f64(m, k, n, block, ell_cols, cis[b], np.abs(va), np.abs(Bu))
                if sem == "stored":
                    want = orc.spmm_bell_f64(m, k, n, block, ell_cols, cis[b], va, Bu)
                else:
                    d = bell_dense(m, k, block, ell_cols, cis[b], va)
                    want = dense_ref(d[None], Bu.T[None].astype(np.float64))[0].T
                nan_at = None
                if special == "nan" and streamed_is_a(m, n, 1, 0):
                    rows = bell_dense(m, k, block, ell_cols, cis[b], near_edge(vas[b]).astype(np.float32)).any(1)
                    nan_at = np.zeros((n, m), bool)
                    nan_at[:, rows] = True
                    nan_at = nan_at if rows.any() else None
                check(gots[b], want, bound, tol, special, (case, name, alg, ws_alg, b), nan_at=nan_at)


# ------------------------------------------------------------------ beta = 0 over a NaN-filled C, every SpMM route
@pytest.mark.parametrize("fmt", ["coo", "csr"])
def test_coo_csr_beta_zero_never_reads_c(spfy, orc, cuda, fmt):
    """beta = 0 over a NaN-filled C on every route and density, including the gated CSR pair (the device flag picks
    the per-non-zero kernel or scatter + tcgen05 on either side of 2 %): C is written without being read"""
    for m, k, n, nb in SPMM_SHAPES:
        for density in (0.005, 0.1, 0.5):
            rng = np.random.default_rng(m + k + int(density * 1000))
            ri, ci, va = coo_matrix(rng, m, k, density)
            B = unit_magnitudes(rng, (nb, n, k))
            want = orc.spmm_coo_batched_f64(m, k, n, nb, ri, ci, va, B, None, 0.5, 0.0)
            bound = 0.5 * orc.spmm_coo_batched_f64(m, k, n, nb, ri, ci, np.abs(va), np.abs(B))
            for alg in ("CUDA_CORE", "TENSOR", "TENSOR_FAST", "DEFAULT"):
                got = run_coo(spfy, cuda, fmt, alg, m, k, n, nb, ri, ci, va, B, alpha=0.5)
                tol = coo_semantics(alg, density, k)[2]
                check(got, want, bound, tol, "ieee", (fmt, alg, m, k, density))


def test_blocked_ell_beta_zero_never_reads_c(spfy, orc, cuda):
    """beta = 0 over NaN-filled C_b on every blocked-ELL route, with a repeated id (the block-row goes to the gated
    CUDA-core stand-in) and through the chunked path (a workspace that holds one dense image at a time)"""
    m, n, k, nb, block = 264, 64, 320, 5, 4
    ell_cols = k // 2
    rng = np.random.default_rng(12)
    cis, vas = zip(*[bell_matrix(rng, m, k, block, ell_cols) for _ in range(nb)])
    cis = [c.copy() for c in cis]
    cis[1][3, 2] = cis[1][3, 1] if cis[1][3, 1] >= 0 else cis[1][3, 3]  # a repeated id
    B = unit_magnitudes(rng, (n, k))
    wants = [orc.spmm_bell_f64(m, k, n, block, ell_cols, cis[b], vas[b], B) for b in range(nb)]
    bounds = [orc.spmm_bell_f64(m, k, n, block, ell_cols, cis[b], np.abs(vas[b]), np.abs(B)) for b in range(nb)]
    for alg in ("CUDA_CORE", "TENSOR", "TENSOR_FAST", "DEFAULT"):
        tol = BELL_SEMANTICS(alg)[2]
        gots = run_bell(spfy, cuda, alg, m, n, k, block, ell_cols, cis, vas, B)
        for b in range(nb):
            check(gots[b], wants[b], bounds[b], tol, "ieee", (alg, b))
    # chunked: room for the dense image of one batch element at a time
    capi = spfy.capi
    small = ctypes.c_size_t()
    capi.spfy_spmm_bell_workspace_bytes(capi.SPMM_ALG_TENSOR, capi.F32, m, k, n, 1, ctypes.byref(small))
    ws = torch.empty(small.value + 100, dtype=torch.uint8, device=cuda)
    dci = [torch.from_numpy(c).to(cuda) for c in cis]
    dva = [torch.from_numpy(v).to(cuda) for v in vas]
    cs = [torch.full((n, m), float("nan"), device=cuda) for _ in range(nb)]
    dB = torch.from_numpy(B).to(cuda)
    tab = [torch.tensor([t.data_ptr() for t in lst], dtype=torch.int64, device=cuda) for lst in (dci, dva, cs)]
    capi.spfy_spmm_bell_batched(capi.SPMM_ALG_TENSOR, capi.F32, m, k, n, block, ell_cols, nb, tab[0].data_ptr(),
                                tab[1].data_ptr(), dB.data_ptr(), k, tab[2].data_ptr(), m, 1.0, 0.0, ws.data_ptr(),
                                ws.numel(), None)
    for b in range(nb):
        check(cs[b].double().cpu().numpy(), wants[b], bounds[b], F32_TOL, "ieee", ("chunked", b))
