"""GPU parity tests of the dense tcgen05 GEMM (spfy_gemm_*, the replacement for cublas*gemmBatched behind
sparsifyme::batched::gemm, reference include/sparsify.me/gemm.hxx:25-195) and of the tensor-core routes of the
unstructured SpMM entry points built on it (spmm.hxx:30-193).

Tolerances (written next to each assert):
  fp32 operands, 3xTF32 (default): |err| <= 4e-6 * sum_k |a||b|   -- fp32-level (each product exact to ~2^-21)
  fp32 operands, one TF32 product:  |err| <= 2e-3 * sum_k |a||b|   -- 10-bit mantissas (cuBLAS TF32 class)
  fp16 / bf16 operands:             max relative error 1e-2 (north_star), fp32 accumulation
  inputs exact in TF32 (small integers, multiples of 1/64): bit-identical to the fp64 oracle / cuSPARSE goldens"""
import glob
import os
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

REL_TOL = 1e-2
F32_TOL = 4e-6
TF32_TOL = 2e-3


def colmajor(x):
    """numpy [r, c] -> the same matrix stored column-major, as a contiguous torch-ready array [c, r]"""
    return np.ascontiguousarray(x.T)


def gemm_case(spfy, cuda, tdt, m, n, k, nb, ta, tb, alpha, beta, shared_a, shared_b, precision, strided, seed, ints=False):
    rng = np.random.default_rng(seed)
    gen = (lambda *s: rng.integers(-4, 5, s).astype(np.float32)) if ints else (lambda *s: rng.uniform(-1, 1, s).astype(np.float32))
    na, nbb = (1 if shared_a else nb), (1 if shared_b else nb)
    A = gen(na, m, k)   # op(A_b), logical
    B = gen(nbb, k, n)  # op(B_b), logical
    C0 = gen(nb, m, n)
    tA = torch.from_numpy(A).to(tdt)
    tB = torch.from_numpy(B).to(tdt)
    tC = torch.from_numpy(C0).to(tdt)
    A64, B64, C64 = tA.double().numpy(), tB.double().numpy(), tC.double().numpy()
    # storage: column-major op() shape, or its transpose when the flag says T
    sa = np.stack([colmajor(x) if ta == spfy.OP_N else np.ascontiguousarray(x) for x in tA.float().numpy()])
    sb = np.stack([colmajor(x) if tb == spfy.OP_N else np.ascontiguousarray(x) for x in tB.float().numpy()])
    dA = torch.from_numpy(sa).to(cuda).to(tdt)
    dB = torch.from_numpy(sb).to(cuda).to(tdt)
    dC = torch.from_numpy(np.stack([colmajor(x) for x in tC.float().numpy()])).to(cuda).to(tdt)  # [nb, n, m]
    a_arg = dA[0] if shared_a else dA
    b_arg = dB[0] if shared_b else dB
    ms = spfy.batched.gemm(a_arg, b_arg, dC, m, n, k, transpose_a=ta, transpose_b=tb, alpha=alpha, beta=beta,
                           precision=precision, strided=strided)
    assert ms >= 0
    got = dC.double().cpu().numpy().transpose(0, 2, 1)  # [nb, m, n]
    Ab = np.broadcast_to(A64, (nb, m, k))
    Bb = np.broadcast_to(B64, (nb, k, n))
    want = alpha * (Ab @ Bb) + beta * C64
    bound = abs(alpha) * (np.abs(Ab) @ np.abs(Bb)) + abs(beta) * np.abs(C64)
    return got, want, bound


GEMM_SHAPES = [(128, 128, 64, 1), (200, 72, 104, 3), (64, 392, 256, 2), (520, 264, 1000, 2), (136, 8, 40, 1),
               (8, 136, 2304, 2)]


@pytest.mark.parametrize("m,n,k,nb", GEMM_SHAPES)
@pytest.mark.parametrize("ta,tb", [(0, 0), (1, 0), (0, 1), (1, 1)])
def test_gemm_f32_3xtf32_is_fp32_accurate(spfy, cuda, m, n, k, nb, ta, tb):
    got, want, bound = gemm_case(spfy, cuda, torch.float32, m, n, k, nb, ta, tb, 1.0, 0.0, False, nb > 1, spfy.GEMM_PRECISE,
                                 True, seed=m + n + k)
    err = np.abs(got - want)
    assert np.all(err <= F32_TOL * bound + 1e-30), float(np.max(err / np.maximum(bound, 1e-30)))


@pytest.mark.parametrize("tdt", [torch.float16, torch.bfloat16])
@pytest.mark.parametrize("m,n,k,nb", GEMM_SHAPES)
@pytest.mark.parametrize("ta,tb", [(0, 0), (1, 0), (0, 1), (1, 1)])
def test_gemm_half_matches_fp64(spfy, cuda, tdt, m, n, k, nb, ta, tb):
    got, want, bound = gemm_case(spfy, cuda, tdt, m, n, k, nb, ta, tb, 1.0, 0.0, False, nb > 1, spfy.GEMM_PRECISE, True,
                                 seed=m * 3 + n + k)
    # fp32 accumulation of exact products, one rounding to the 16-bit output type
    eps = 2.0 ** -11 if tdt == torch.float16 else 2.0 ** -8
    assert np.all(np.abs(got - want) <= eps * np.abs(want) + 1e-4 * bound + 1e-30)
    scale = np.maximum(np.abs(want), 1e-2 * np.abs(want).max())
    assert float(np.max(np.abs(got - want) / scale)) <= REL_TOL


@pytest.mark.parametrize("tdt", [torch.float16, torch.bfloat16, torch.float32])
@pytest.mark.parametrize("m,n,k,nb", [(200, 72, 104, 3), (520, 264, 1000, 2), (64, 392, 256, 2), (784, 256, 2304, 2),
                                      (1000, 520, 72, 1), (300, 16, 40, 2)])
@pytest.mark.parametrize("ta,tb", [(0, 0), (1, 0), (0, 1), (1, 1)])
def test_gemm_single_product_alpha_beta_matches_fp64(spfy, cuda, tdt, m, n, k, nb, ta, tb):
    """the shared-memory kernel (fp16 / bf16, fp32 as one TF32 product) with alpha = 0.5, beta = 0.25: odd tile counts,
    ragged edges, every major-ness, within the fp64 bound"""
    prec = spfy.GEMM_FAST if tdt == torch.float32 else spfy.GEMM_PRECISE
    got, want, bound = gemm_case(spfy, cuda, tdt, m, n, k, nb, ta, tb, 0.5, 0.25, False, nb > 1, prec, True, seed=m + 7 * n + k)
    tol = TF32_TOL if tdt == torch.float32 else 2.0 ** -7
    assert np.all(np.abs(got - want) <= tol * bound + 1e-30)


@pytest.mark.parametrize("tdt", [torch.float16, torch.bfloat16, torch.float32])
@pytest.mark.parametrize("strided", [True, False])
def test_gemm_refuses_unknown_precision(spfy, cuda, tdt, strided):
    """precision is PRECISE or FAST for every dtype; anything else (0x10 once selected an opt-in kernel, 2 was read as
    FAST for fp32 and ignored for 16-bit operands) is SPFY_E_INVALID with no launch and C untouched"""
    m, n, k, nb = 200, 72, 104, 2
    a = torch.rand(nb, k, m, device=cuda).to(tdt)
    b = torch.rand(nb, n, k, device=cuda).to(tdt)
    c = torch.rand(nb, n, m, device=cuda).to(tdt)
    c0 = c.clone()
    torch.cuda.synchronize()
    for prec in (0x10, 2, spfy.GEMM_FAST | 0x10, -1):
        before = spfy.launch_count()
        with pytest.raises(spfy.SpfyError) as e:
            spfy.batched.gemm(a, b, c, m, n, k, beta=0.5, precision=prec, strided=strided)
        assert e.value.code == spfy.capi.E_INVALID and "precision" in str(e.value)
        assert spfy.launch_count() == before
    torch.cuda.synchronize()
    assert torch.equal(c.view(torch.int8), c0.view(torch.int8))


@pytest.mark.parametrize("strided", [True, False])
@pytest.mark.parametrize("shared_a,shared_b", [(False, True), (True, False), (False, False)])
def test_gemm_alpha_beta_sharing_and_pointer_arrays(spfy, cuda, strided, shared_a, shared_b):
    """the pointer-array entry is what the header template calls (examples/gemm.cu passes per-batch A and one shared B)"""
    got, want, bound = gemm_case(spfy, cuda, torch.float32, 264, 72, 200, 4, 0, 0, 0.75, -0.5, shared_a, shared_b,
                                 spfy.GEMM_PRECISE, strided, seed=5)
    assert np.all(np.abs(got - want) <= F32_TOL * bound + 1e-30)


def test_gemm_single_tf32_product_and_exact_integers(spfy, cuda):
    got, want, bound = gemm_case(spfy, cuda, torch.float32, 256, 128, 512, 2, 0, 0, 1.0, 0.0, False, True, spfy.GEMM_FAST,
                                 True, seed=9)
    err = np.abs(got - want)
    assert np.all(err <= TF32_TOL * bound + 1e-30)
    assert float(np.max(err / np.maximum(bound, 1e-30))) > F32_TOL  # it really is the single-product mode
    for prec in (spfy.GEMM_PRECISE, spfy.GEMM_FAST):  # small integers are exact in TF32: every mode gives the exact sum
        got, want, _ = gemm_case(spfy, cuda, torch.float32, 136, 200, 300, 2, 1, 0, 1.0, 0.0, False, False, prec, True,
                                 seed=10, ints=True)
        assert np.array_equal(got, want)


def test_gemm_resnet_layer_full_size(spfy, cuda):
    """one datasets/resnet50.csv row as the reference's gemm driver runs it (m, n, k, b) = (3136, 128, 1152, 32):
    per-image A, shared B; checked on sampled rows / columns against fp64 with the 3xTF32 bound"""
    m, n, k, nb = 3136, 128, 1152, 32
    gen = torch.Generator(device=cuda)
    gen.manual_seed(3)
    dA = torch.rand(nb, k, m, device=cuda, generator=gen) * 2 - 1   # m x k column-major per batch
    dB = torch.rand(n, k, device=cuda, generator=gen) * 2 - 1       # k x n column-major
    dC = torch.empty(nb, n, m, device=cuda)
    spfy.batched.gemm(dA, dB, dC, m, n, k)
    rows = torch.tensor([0, 1, 127, 128, 1000, m - 129, m - 1], device=cuda)
    for b in (0, 17, nb - 1):
        a = dA[b][:, rows].double()                                  # [k, rows]
        want = dB.double() @ a                                       # [n, rows]
        bound = dB.double().abs() @ a.abs()
        got = dC[b][:, rows].double()
        assert bool(((got - want).abs() <= F32_TOL * bound).all())


@pytest.mark.parametrize("tdt", [torch.float32, torch.float16])
@pytest.mark.parametrize("m,n,k,nb,ta,tb", [(12544 // 8, 64, 147, 3, 0, 0), (70, 33, 147, 2, 1, 1), (6, 10, 100, 3, 0, 1)])
def test_gemm_operands_tma_cannot_address_are_repacked(spfy, cuda, tdt, m, n, k, nb, ta, tb):
    """ldb = k = 147 (the first conv layer of every ResNet through the reference's gemm driver), odd m / n: leading
    dimensions that are not multiples of 16 bytes -- the operand is copied once with padded rows, same results"""
    got, want, bound = gemm_case(spfy, cuda, tdt, m, n, k, nb, ta, tb, 1.0, 0.0, False, True, spfy.GEMM_PRECISE, True,
                                 seed=k + m)
    tol = F32_TOL if tdt == torch.float32 else 2.0 ** -10
    assert np.all(np.abs(got - want) <= tol * bound + 1e-30)


def test_gemm_rejects_unsupported_types(spfy, cuda):
    a = torch.zeros(3, 100, 8, device=cuda, dtype=torch.float64)
    b = torch.zeros(3, 10, 100, device=cuda, dtype=torch.float64)
    c = torch.zeros(3, 10, 8, device=cuda, dtype=torch.float64)
    with pytest.raises(spfy.SpfyError) as e:  # no fp64 tensor-core path (the header keeps cublasDgemmBatched for double)
        spfy.batched.gemm(a, b, c, 8, 10, 100)
    assert e.value.code == spfy.capi.E_UNSUPPORTED


# ------------------------------------------------------------------ tensor-core routes of the unstructured SpMM
def coo_problem(orc, m, k, n, nb, density, seed, ints=False):
    rng = np.random.default_rng(seed)
    if ints:
        w = rng.integers(-4, 5, (m, k)).astype(np.float32)
        thr = float(np.quantile(np.abs(w), 1.0 - density)) - 0.5
        B = rng.integers(-3, 4, (nb, n, k)).astype(np.float32)
    else:
        w = rng.uniform(-1, 1, (m, k)).astype(np.float32)
        thr = float(np.quantile(np.abs(w), 1.0 - density))
        B = rng.uniform(-1, 1, (nb, n, k)).astype(np.float32)
    ri, ci, va, _ = orc.threshold_to_coo(2, w, thr)
    return ri, ci, va, B


def abs_bound(orc, m, k, n, nb, ri, ci, va, B):
    return orc.spmm_coo_batched_f64(m, k, n, nb, ri, ci, np.abs(va), np.abs(B))


@pytest.mark.parametrize("m,k,n,nb,density", [(64, 576, 200, 3, 0.5), (128, 1152, 196, 4, 0.1), (256, 2304, 49, 4, 0.05),
                                              (512, 512, 64, 2, 0.1), (40, 64, 24, 2, 0.3), (130, 332, 70, 2, 0.5)])
@pytest.mark.parametrize("alg", ["TENSOR", "TENSOR_FAST", "DEFAULT"])
def test_coo_spmm_tensor_route_matches_oracle(spfy, orc, cuda, m, k, n, nb, density, alg):
    algc = getattr(spfy, "SPMM_ALG_" + alg)
    ri, ci, va, B = coo_problem(orc, m, k, n, nb, density, seed=m + k + n)
    rng = np.random.default_rng(1)
    C0 = rng.uniform(-1, 1, (nb, n, m)).astype(np.float32)
    for alpha, beta in [(1.0, 0.0), (0.75, 0.5)]:
        want = orc.spmm_coo_batched_f64(m, k, n, nb, ri, ci, va, B, C0, alpha, beta)
        bound = abs(alpha) * abs_bound(orc, m, k, n, nb, ri, ci, va, B) + abs(beta) * np.abs(C0)
        dC = torch.from_numpy(C0.copy()).to(cuda)
        before = spfy.launch_count()
        spfy.batched.strided_coo(m, k, ri.size, k, n, nb, torch.from_numpy(ri).to(cuda), torch.from_numpy(ci).to(cuda),
                                 torch.from_numpy(va).to(cuda), torch.from_numpy(B).to(cuda), dC, alpha=alpha, beta=beta,
                                 alg=algc)
        tol = TF32_TOL if alg == "TENSOR_FAST" else F32_TOL
        err = np.abs(dC.cpu().numpy().astype(np.float64) - want)
        assert np.all(err <= tol * bound + 1e-30), float(np.max(err / np.maximum(bound, 1e-30)))
        assert spfy.launch_count() - before == 3  # coo_to_csr + scatter + tcgemm: no CUDA-core SpMM kernel ran


def test_coo_spmm_tensor_route_exact_on_integers_and_duplicates(spfy, orc, cuda):
    """integers are exact in TF32, so the tensor route must return the exact sums; a duplicated (row, col) entry and
    columns in any order inside a row add up like cuSPARSE COO"""
    m, k, n, nb = 132, 336, 70, 2
    ri, ci, va, B = coo_problem(orc, m, k, n, nb, 0.5, seed=5, ints=True)
    rng = np.random.default_rng(2)
    ri, ci, va = (np.concatenate([x, x[-3:]]) for x in (ri, ci, va))
    for r in range(0, m, 3):
        sel = np.nonzero(ri == r)[0]
        pm = rng.permutation(sel.size)
        ci[sel], va[sel] = ci[sel][pm], va[sel][pm]
    want = orc.spmm_coo_batched_f64(m, k, n, nb, ri, ci, va, B)
    for alg in (spfy.SPMM_ALG_TENSOR, spfy.SPMM_ALG_CUDA_CORE, spfy.SPMM_ALG_DEFAULT):
        dC = torch.full((nb, n, m), 7.0, dtype=torch.float32, device=cuda)
        spfy.batched.strided_coo(m, k, ri.size, k, n, nb, torch.from_numpy(ri).to(cuda), torch.from_numpy(ci).to(cuda),
                                 torch.from_numpy(va).to(cuda), torch.from_numpy(B).to(cuda), dC, alg=alg)
        assert np.array_equal(dC.cpu().numpy().astype(np.float64), want), alg


def test_coo_spmm_first_conv_layer_runs_on_a_padded_copy(spfy, orc, cuda):
    """k = 147 (the first conv layer): ldb = 147 floats is not a multiple of 16 bytes, so TMA cannot address B_b.  The
    tensor-core route then runs on a padded copy of B in the workspace; a workspace without room for it makes TENSOR
    fail loudly (SPFY_E_WORKSPACE) and DEFAULT take the CUDA-core kernels."""
    import ctypes
    m, k, n, nb = 64, 147, 96, 2
    ri, ci, va, B = coo_problem(orc, m, k, n, nb, 0.5, seed=3)
    dri, dci, dva, dB = (torch.from_numpy(x).to(cuda) for x in (ri, ci, va, B))
    want = orc.spmm_coo_batched_f64(m, k, n, nb, ri, ci, va, B)
    bound = abs_bound(orc, m, k, n, nb, ri, ci, va, B)
    for alg in (spfy.SPMM_ALG_TENSOR, spfy.SPMM_ALG_DEFAULT):
        dC = torch.zeros(nb, n, m, device=cuda)
        before = spfy.launch_count()
        spfy.batched.strided_coo(m, k, ri.size, k, n, nb, dri, dci, dva, dB, dC, alg=alg)
        assert spfy.launch_count() - before == 4  # coo_to_csr + scatter + repack + tcgemm
        err = np.abs(dC.cpu().numpy().astype(np.float64) - want)
        assert np.all(err <= F32_TOL * bound + 1e-30)
    capi = spfy.capi
    small = ctypes.c_size_t()
    capi.spfy_spmm_workspace_bytes(capi.SPMM_ALG_TENSOR, m, k, n, 0, ri.size, ctypes.byref(small))  # sized for no batch at all
    ws = torch.empty(small.value, dtype=torch.uint8, device=cuda)
    dC = torch.zeros(nb, n, m, device=cuda)
    args = (m, k, ri.size, n, nb, dri.data_ptr(), dci.data_ptr(), dva.data_ptr(), dB.data_ptr(), k, k * n, dC.data_ptr(), m,
            m * n, 1.0, 0.0, ws.data_ptr(), ws.numel(), None)
    with pytest.raises(spfy.SpfyError) as e:
        capi.spfy_spmm_coo_strided_batched(capi.SPMM_ALG_TENSOR, *args)
    assert e.value.code == capi.E_WORKSPACE
    capi.spfy_spmm_coo_strided_batched(capi.SPMM_ALG_DEFAULT, *args)
    assert np.allclose(dC.cpu().numpy(), want, rtol=2e-4, atol=2e-4)


@pytest.mark.parametrize("density,route", [(0.3, "tensor"), (0.004, "cuda-core")])
def test_csr_entry_chooses_between_tensor_and_cuda_cores_on_the_device(spfy, orc, cuda, density, route):
    """the CSR entry does not know nnz on the host: the per-non-zero kernel and the scatter + tcgen05 GEMM are both
    launched, and a device flag (nnz >= 2 % of m*k) lets exactly one of them write C"""
    m, k, n, nb = 200, 1000, 64, 3
    ri, ci, va, B = coo_problem(orc, m, k, n, nb, density, seed=77)
    rng = np.random.default_rng(3)
    C0 = rng.uniform(-1, 1, (nb, n, m)).astype(np.float32)
    want = orc.spmm_coo_batched_f64(m, k, n, nb, ri, ci, va, B, C0, 0.5, 2.0)
    bound = 0.5 * abs_bound(orc, m, k, n, nb, ri, ci, va, B) + 2.0 * np.abs(C0)
    dri = torch.from_numpy(ri).to(cuda)
    rp = spfy.coo_to_csr(dri, m)
    dC = torch.from_numpy(C0.copy()).to(cuda)
    spfy.batched.csr(m, k, n, nb, rp, torch.from_numpy(ci).to(cuda), torch.from_numpy(va).to(cuda),
                     torch.from_numpy(B).to(cuda), dC, alpha=0.5, beta=2.0)  # beta = 2: a double write would show
    err = np.abs(dC.cpu().numpy().astype(np.float64) - want)
    assert np.all(err <= 2e-5 * bound + 1e-30), route


def bell_problem(orc, rng, m, n, k, nb, block, ell_cols, order="sorted", ints=False):
    bcols = ell_cols // block
    B = rng.integers(-3, 4, (n, k)).astype(np.float32) if ints else rng.uniform(-1, 1, (n, k)).astype(np.float32)
    cis, vas, wants, bounds = [], [], [], []
    for b in range(nb):
        ci = np.stack([np.sort(rng.choice(-(-k // block), bcols, replace=False)) for _ in range(-(-m // block))]).astype(np.int64)
        if order == "shuffled":
            ci = np.stack([rng.permutation(r) for r in ci])
        elif order == "padded":
            ci[:, ::5] = -1
        elif order == "duplicated":
            ci[3, 1] = ci[3, 0]
        va = (rng.integers(-3, 4, (m, ell_cols)) if ints else rng.uniform(-1, 1, (m, ell_cols))).astype(np.float32)
        wants.append(orc.spmm_bell_f64(m, k, n, block, ell_cols, ci, va, B))
        bounds.append(orc.spmm_bell_f64(m, k, n, block, ell_cols, ci, np.abs(va), np.abs(B)))
        cis.append(ci)
        vas.append(va)
    return B, cis, vas, wants, bounds


@pytest.mark.parametrize("order", ["sorted", "shuffled", "padded", "duplicated"])
@pytest.mark.parametrize("m,n,k,nb,block", [(200, 152, 448, 3, 4), (64, 48, 128, 2, 2), (392, 64, 576, 4, 2),
                                            (130, 40, 96, 2, 3), (256, 264, 512, 2, 16)])
def test_blocked_ell_tensor_route_matches_oracle(spfy, orc, cuda, order, m, n, k, nb, block):
    """fp32 blocked-ELL through expand + tcgen05 (DEFAULT / TENSOR): ascending, shuffled and padded ids are expanded
    as they are; a repeated id raises the device flag and the chunk is recomputed by the CUDA-core kernel (both
    add the blocks, like the oracle).  (392, 64, 576, 4, 2) is the reference driver's construction."""
    ell_cols = (k // 2) // block * block
    rng = np.random.default_rng(m + n + k + block)
    B, cis, vas, wants, bounds = bell_problem(orc, rng, m, n, k, nb, block, ell_cols, order)
    for alg in (spfy.SPMM_ALG_DEFAULT, spfy.SPMM_ALG_TENSOR):
        cs = [torch.full((n, m), 3.0, dtype=torch.float32, device=cuda) for _ in range(nb)]
        spfy.batched.spmm([torch.from_numpy(c).to(cuda) for c in cis], [torch.from_numpy(v).to(cuda) for v in vas],
                          torch.from_numpy(B).to(cuda), cs, m, n, k, block, ell_cols, alg=alg)
        for c, want, bound in zip(cs, wants, bounds):
            err = np.abs(c.cpu().numpy().astype(np.float64) - want)
            assert np.all(err <= 2e-5 * bound + 1e-30), (order, float(np.max(err / np.maximum(bound, 1e-30))))


@pytest.mark.parametrize("tdt", [torch.float16, torch.bfloat16])
def test_blocked_ell_half_precision_runs_on_tensor_cores(spfy, orc, cuda, tdt):
    """16-bit blocked-ELL (the type the reference's descriptor declares, spmm.hxx:60): kind::f16 with fp32
    accumulation; small integers make the result exact, alpha / beta applied in fp32"""
    m, n, k, nb, block = 136, 72, 256, 3, 4
    ell_cols = k // 2
    rng = np.random.default_rng(8)
    B, cis, vas, wants, _ = bell_problem(orc, rng, m, n, k, nb, block, ell_cols, "shuffled", ints=True)
    cs = [torch.zeros(n, m, dtype=tdt, device=cuda) for _ in range(nb)]
    before = spfy.launch_count()
    spfy.batched.spmm([torch.from_numpy(c).to(cuda) for c in cis], [torch.from_numpy(v).to(cuda).to(tdt) for v in vas],
                      torch.from_numpy(B).to(cuda).to(tdt), cs, m, n, k, block, ell_cols)
    assert spfy.launch_count() - before == 3  # expand + tcgemm + (gated off) row-split stand-in
    for c, want in zip(cs, wants):  # the exact sum, rounded once to the 16-bit output type
        assert torch.equal(c.cpu(), torch.from_numpy(want).to(tdt))


def test_blocked_ell_chunked_batches_and_beta(spfy, orc, cuda):
    """a workspace that holds the dense image of only one batch element at a time: the batch is processed chunk by
    chunk, and beta != 0 shows that every C_b is written exactly once"""
    import ctypes
    m, n, k, nb, block = 264, 64, 320, 5, 4
    ell_cols = k // 2
    rng = np.random.default_rng(12)
    B, cis, vas, _, _ = bell_problem(orc, rng, m, n, k, nb, block, ell_cols)
    C0 = rng.uniform(-1, 1, (nb, n, m)).astype(np.float32)
    dci = [torch.from_numpy(c).to(cuda) for c in cis]
    dva = [torch.from_numpy(v).to(cuda) for v in vas]
    dB = torch.from_numpy(B).to(cuda)
    cs = [torch.from_numpy(C0[b].copy()).to(cuda) for b in range(nb)]
    capi = spfy.capi
    small = ctypes.c_size_t()
    capi.spfy_spmm_bell_workspace_bytes(capi.SPMM_ALG_TENSOR, capi.F32, m, k, n, 1, ctypes.byref(small))
    ws = torch.empty(small.value + 100, dtype=torch.uint8, device=cuda)  # room for one dense matrix, not two
    tab = [torch.tensor([t.data_ptr() for t in lst], dtype=torch.int64, device=cuda) for lst in (dci, dva, cs)]
    capi.spfy_spmm_bell_batched(capi.SPMM_ALG_TENSOR, capi.F32, m, k, n, block, ell_cols, nb, tab[0].data_ptr(),
                                tab[1].data_ptr(), dB.data_ptr(), k, tab[2].data_ptr(), m, 0.5, 2.0, ws.data_ptr(),
                                ws.numel(), None)
    for b in range(nb):
        want = orc.spmm_bell_f64(m, k, n, block, ell_cols, cis[b], vas[b], B, C0[b], 0.5, 2.0)
        assert np.allclose(cs[b].cpu().numpy().astype(np.float64), want, rtol=1e-5, atol=1e-5)


@pytest.mark.parametrize("alg", ["CUDA_CORE", "DEFAULT", "TENSOR"])
def test_unstructured_routes_bit_exact_with_cusparse_golden(spfy, cuda, alg):
    """what cuSPARSE returned for the reference's call sequences (tests/golden/cusparse_*.npz; inputs are multiples
    of 1/64, exact in fp32 AND in TF32, so every route must reproduce the same bits)"""
    gold = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    sys.path.insert(0, gold)
    from make_golden import gen_f32
    algc = getattr(spfy, "SPMM_ALG_" + alg)
    for path in sorted(glob.glob(os.path.join(gold, "cusparse_coo_*.npz"))):
        z = np.load(path)
        m, k, n, nb = int(z["m"]), int(z["k"]), int(z["n"]), int(z["nb"])
        a = torch.from_numpy(gen_f32(1, m * k).reshape(m, k)).to(cuda)
        B = torch.from_numpy(gen_f32(2, nb * n * k).reshape(nb, n, k)).to(cuda)
        C = torch.from_numpy(gen_f32(3, nb * n * m).reshape(nb, n, m).copy()).to(cuda)
        ri, ci, va, nnz = spfy.threshold_to_coo(a, float(z["thr"]))
        spfy.batched.strided_coo(m, k, nnz, k, n, nb, ri, ci, va, B, C, alpha=float(z["alpha"]), beta=float(z["beta"]),
                                 alg=algc)
        assert np.array_equal(C.cpu().numpy(), z["c"]), os.path.basename(path)
    for path in sorted(glob.glob(os.path.join(gold, "cusparse_bell_*.npz"))):
        z = np.load(path)
        m, k, n, nb, block, ell_cols = (int(z[x]) for x in ("m", "k", "n", "nb", "block", "ell_cols"))
        V = gen_f32(4, nb * m * ell_cols).reshape(nb, m, ell_cols)
        B = torch.from_numpy(gen_f32(5, n * k).reshape(n, k)).to(cuda)
        cis = [torch.from_numpy(np.ascontiguousarray(z["col_idx"][b])).to(cuda) for b in range(nb)]
        vas = [torch.from_numpy(np.ascontiguousarray(V[b])).to(cuda) for b in range(nb)]
        cs = [torch.zeros(n, m, dtype=torch.float32, device=cuda) for _ in range(nb)]
        spfy.batched.spmm(cis, vas, B, cs, m, n, k, block, ell_cols, alg=algc)
        for b in range(nb):
            assert np.array_equal(cs[b].cpu().numpy(), z["c"][b]), os.path.basename(path)
