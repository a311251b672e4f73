"""GPU tests of the C++ header layer (`include/sparsify.me/*.hxx`), i.e. of the drop-in boundary itself.

* tests/cpp/header_parity.cu (ours) calls the five operator templates the way the reference's drivers do, on
  deterministic inputs, and dumps inputs and outputs; the dumps are checked here against the CPU oracle.
* examples/bin/* and profiling/* (our drivers with the reference's command lines) must run on the B200.
The binaries are built by __graft_entry__.build()."""
import os
import subprocess

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
DRIVER = os.path.join(ROOT, "tests", "cpp", "bin", "header_parity")
REL_TOL = 1e-2


def rel_err(got, want):
    scale = np.maximum(np.abs(want), 1e-2 * max(np.abs(want).max(), 1e-30))
    return float(np.max(np.abs(got - want) / scale))


@pytest.fixture(scope="module")
def dumps(tmp_path_factory, cuda):
    assert os.path.exists(DRIVER), "tests/cpp/bin/header_parity is missing: run __graft_entry__.build()"
    out = tmp_path_factory.mktemp("header_parity")
    r = subprocess.run([DRIVER, str(out)], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, (r.stdout + r.stderr)[-2000:]
    assert "sparsify.me:" not in r.stderr, r.stderr[-2000:]  # the header glue reports C-ABI failures on stderr
    meta = {}
    for line in open(out / "meta.txt"):
        f = line.split()
        meta[f[0]] = f[1:]

    def load(name, dtype):
        return np.fromfile(out / (name + ".bin"), dtype=dtype)

    return meta, load


def test_header_sparsify_matches_oracle(dumps, orc):
    meta, load = dumps
    m, n = (int(x) for x in meta["sparsify"][:2])
    w_in = load("sparsify_in", np.float32)
    want_w, want_mask = orc.prune_blocks_ref(w_in.copy(), m, n)
    assert np.array_equal(load("sparsify_out", np.float32), want_w)
    assert np.array_equal(load("sparsify_mask", np.uint64), want_mask.astype(np.uint64))


def test_header_spmma_half_prunes_like_cusparselt_tile_and_multiplies(dumps, orc):
    meta, load = dumps
    m, n, k = (int(x) for x in meta["spmma_f16"][:3])
    assert meta["spmma_f16"][-1] == "3"  # {prune, compress, multiply} ms (spmma.hxx:117)
    a_in = load("spmma_f16_a_in", np.uint16).reshape(m, k)
    b = load("spmma_f16_b", np.uint16).reshape(k, n)
    pruned, _ = orc.prune24_tile(0, a_in)
    assert np.array_equal(load("spmma_f16_a_out", np.uint16).reshape(m, k), pruned)  # in place, bit-exact
    want = orc.spmma_f64(0, pruned, b)
    got = load("spmma_f16_c", np.float16).reshape(m, n).astype(np.float64)
    assert rel_err(got, want) <= REL_TOL


def test_header_spmma_float_instantiation(dumps, orc):
    """the reference driver instantiates spmma<float> (examples/spmma.cu:24): fp16 images are pruned and multiplied,
    A comes back pruned, C comes back as float"""
    meta, load = dumps
    m, n, k = (int(x) for x in meta["spmma_f32"][:3])
    a16 = orc.from_f32(0, load("spmma_f32_a_in", np.float32).reshape(m, k))
    b16 = orc.from_f32(0, load("spmma_f32_b", np.float32).reshape(k, n))
    pruned, _ = orc.prune24_tile(0, a16)
    assert np.array_equal(orc.from_f32(0, load("spmma_f32_a_out", np.float32).reshape(m, k)), pruned)
    want = orc.spmma_f64(0, pruned, b16)
    assert rel_err(load("spmma_f32_c", np.float32).reshape(m, n).astype(np.float64), want) <= REL_TOL


def test_header_blocked_ell_spmm(dumps, orc):
    meta, load = dumps
    m, n, k, nb = (int(x) for x in meta["spmm"][:4])
    block, ell_cols = 2, k // 2
    B = load("spmm_b", np.float32).reshape(n, k)  # k x n column-major
    for b in range(nb):
        ids = load(f"spmm_ids_{b}", np.uint64).astype(np.int64).reshape(m // block, ell_cols // block)
        vals = load(f"spmm_vals_{b}", np.float32).reshape(m, ell_cols)
        want = orc.spmm_bell_f64(m, k, n, block, ell_cols, ids, vals, B)
        got = load(f"spmm_c_{b}", np.float32).reshape(n, m).astype(np.float64)  # m x n column-major
        assert np.allclose(got, want, rtol=2e-5, atol=2e-5)


def test_header_strided_coo(dumps, orc):
    meta, load = dumps
    m, n, k, nb = (int(x) for x in meta["coo"][:4])
    ri, ci, va = load("coo_rows", np.int32), load("coo_cols", np.int32), load("coo_vals", np.float32)
    assert ri.size == int(meta["coo"][5])
    B = load("coo_b", np.float32).reshape(nb, n, k)
    want = orc.spmm_coo_batched_f64(m, k, n, nb, ri, ci, va, B)
    got = load("coo_c", np.float32).reshape(nb, n, m).astype(np.float64)
    assert np.allclose(got, want, rtol=2e-5, atol=2e-5)


@pytest.mark.parametrize("tag,np_dt,tol", [("f32", np.float32, 4e-6), ("f16", np.float16, 2e-3)])
def test_header_batched_gemm(dumps, tag, np_dt, tol):
    """batched::gemm: column-major, per-batch A, one shared B (examples/gemm.cu:60-95); fp32 must hold fp32-level
    accuracy (3xTF32): |err| <= 4e-6 * sum_k |a||b|"""
    meta, load = dumps
    m, n, k, nb = (int(x) for x in meta["gemm_" + tag][:4])
    A = load(f"gemm_{tag}_a", np_dt).astype(np.float64).reshape(nb, k, m)  # m x k column-major per batch
    B = load(f"gemm_{tag}_b", np_dt).astype(np.float64).reshape(n, k)      # k x n column-major
    C = load(f"gemm_{tag}_c", np_dt).astype(np.float64).reshape(nb, n, m)  # m x n column-major
    for b in range(nb):
        want = B @ A[b]                     # [n, m] = (A^T)[m,k] ... column-major result
        bound = np.abs(B) @ np.abs(A[b])
        assert np.all(np.abs(C[b] - want) <= tol * bound + 1e-30), float(np.max(np.abs(C[b] - want) / bound))


@pytest.mark.parametrize("name,argv", [("sparsify", ["3136", "576"]), ("spmma", ["128", "256", "512", "1"]),
                                       ("spmm", ["196", "64", "128", "4"]), ("batched_coo", ["128", "96", "160", "2"]),
                                       ("gemm", ["392", "64", "128", "4"])])
def test_our_example_drivers_run(cuda, name, argv):
    """examples/bin/* (our copies of the five drivers' command lines): exit 0 and print their timings"""
    exe = os.path.join(ROOT, "examples", "bin", name)
    assert os.path.exists(exe), "examples/bin is missing: run __graft_entry__.build()"
    r = subprocess.run([exe] + argv, capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, (r.stdout + r.stderr)[-2000:]
    assert "sparsify.me:" not in r.stderr, r.stderr[-2000:]
    assert r.stdout.strip()


def test_profiling_drivers_keep_the_reference_command_lines(cuda, tmp_path):
    """profiling/gemm_timing <f|h|d> out.csv [shapes.csv] -> "m,n,k,b,elapsed" rows (reference profiling/gemm_timing.cu:38-43,110);
    profiling/spmm_timing m n k b -> "prune, compress, multiply" ms (profiling/spmm_timing.cu:64-66)"""
    gt, st = os.path.join(ROOT, "profiling", "gemm_timing"), os.path.join(ROOT, "profiling", "spmm_timing")
    assert os.path.exists(gt) and os.path.exists(st), "profiling/ is not built: run __graft_entry__.build()"
    table = tmp_path / "shapes.csv"
    table.write_text("m,n,k,b\r\n392,64,147,4\r\n196,128,256,4\r\n")
    for prec in ("f", "h"):
        out = tmp_path / f"gemm_{prec}.csv"
        r = subprocess.run([gt, prec, str(out), str(table)], capture_output=True, text=True, timeout=300)
        assert r.returncode == 0 and "sparsify.me:" not in r.stderr, (r.stdout + r.stderr)[-2000:]
        rows = out.read_text().strip().splitlines()
        assert rows[0] == "m,n,k,b,elapsed" and len(rows) == 3
        assert rows[1].startswith("392,64,147,4,") and float(rows[1].split(",")[4]) > 0
    r = subprocess.run([st, "128", "256", "512", "1"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0 and "sparsify.me:" not in r.stderr, (r.stdout + r.stderr)[-2000:]
    assert len([float(x) for x in r.stdout.strip().split(",")]) == 3
