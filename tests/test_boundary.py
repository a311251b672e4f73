"""The drop-in boundary without a GPU: the C-ABI library loads and exports every symbol that
include/spfy_b200.h declares, argument validation fails loudly (never falls back to the host), and the
shape tables match the reference's."""
import ctypes
import hashlib
import os
import re
import subprocess

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def declared_symbols():
    text = open(os.path.join(ROOT, "include", "spfy_b200.h")).read()
    return sorted(set(re.findall(r"SPFY_API\s+[\w\s\*]+?\b(spfy_\w+)\s*\(", text)))


def test_library_exports_every_declared_symbol(spfy):
    names = declared_symbols()
    assert len(names) >= 18
    lib = ctypes.CDLL(spfy.capi.LIB_PATH)
    missing = [n for n in names if not hasattr(lib, n)]
    assert not missing, f"declared in include/spfy_b200.h but not exported: {missing}"
    assert sorted(spfy.capi.SIGNATURES) == names  # the Python binding covers the whole ABI
    assert spfy.version() == 100


def test_no_cusparse_or_cusparselt_dependency(spfy):
    out = subprocess.run(["ldd", spfy.capi.LIB_PATH], capture_output=True, text=True).stdout
    assert "cusparse" not in out.lower() and "cublas" not in out.lower()


def test_argument_errors_do_not_fall_back(spfy):
    capi = spfy.capi
    vb, mb = ctypes.c_size_t(), ctypes.c_size_t()
    with pytest.raises(spfy.SpfyError) as e:
        capi.spfy_compressed_bytes(capi.F32, 8, 8, capi.LAYOUT_SM100, ctypes.byref(vb), ctypes.byref(mb))
    assert e.value.code == capi.E_UNSUPPORTED and "F16/BF16" in str(e.value)
    capi.spfy_compressed_bytes(capi.F16, 130, 260, capi.LAYOUT_SM100, ctypes.byref(vb), ctypes.byref(mb))
    assert (vb.value, mb.value) == (2 * 3 * 16384, 2 * 3 * 2048)
    capi.spfy_compressed_bytes(capi.F16, 5, 147, capi.LAYOUT_CANONICAL, ctypes.byref(vb), ctypes.byref(mb))
    assert (vb.value, mb.value) == (5 * 37 * 4, 5 * 19)
    with pytest.raises(spfy.SpfyError) as e:
        capi.spfy_prune24(capi.F16, 0, 0, None, 8, None, 0, None, None, None, 8, 8, None)
    assert e.value.code == capi.E_INVALID
    with pytest.raises(spfy.SpfyError) as e:
        capi.spfy_spmma(capi.F32, 0, 8, 8, 8, 1.0, None, None, None, 8, 0.0, None, 8, None, 8, None, 0, None)
    assert e.value.code == capi.E_UNSUPPORTED
    with pytest.raises(spfy.SpfyError):
        capi.spfy_convert(capi.F64, capi.F16, ctypes.c_void_p(16), ctypes.c_void_p(16), 4, None)


def test_host_tensors_are_rejected(spfy):
    import torch
    a = torch.zeros(8, 8, dtype=torch.float16)
    with pytest.raises(spfy.SpfyError) as e:
        spfy.prune24(a, compress=False, inplace=True)
    assert "no host path" in str(e.value)


def test_shape_tables_and_reader(spfy):
    sh = spfy.shapes
    counts = {"resnet18.csv": 17, "resnet34.csv": 33, "resnet50.csv": 49, "resnet101.csv": 100, "resnet152.csv": 151,
              "shapes.csv": 49}
    for name, n in counts.items():
        rows = sh.read_shapes(name)
        assert len(rows) == n and all(r.b == 32 for r in rows)
    assert sh.read_shapes("resnet18.csv")[0] == sh.Shape(12544, 64, 147, 32)  # datasets/resnet18.csv:2
    assert sh.read_shapes("shapes.csv") == sh.read_shapes("resnet50.csv")     # SURVEY.md 0.7
    g = sh.to_gemm(sh.Shape(196, 512, 4608, 32))
    assert g == sh.Gemm(M=512, N=6272, K=4608)
    assert sh.to_gemm(sh.Shape(196, 512, 4608, 32), "ref") == sh.Gemm(M=196, N=512, K=4608)
    assert sh.to_gemm(sh.Shape(196, 512, 4608, 32), batch=256).N == 196 * 256
    assert sh.spmma_flops(g) == 2.0 * 512 * 6272 * 4608
    assert sh.spmma_bytes(g) == 2 * 4608 * 6272 + 2 * 512 * 6272 + 512 * 4608 + 512 * 4608 // 8
    assert sh.prune24_bytes(512, 4608) == int(512 * 4608 * 3.125)


def test_dataset_csvs_are_byte_identical_to_the_reference():
    """tests/golden/reference_datasets.md5 holds the md5 of each of the reference's datasets/*.csv (md5sum -c format).
    The hashes were taken with md5sum from this repository's datasets/*.csv, which were checked byte for byte against
    the reference tree's copies while it was at hand and have not changed since: the test pins the tables to them."""
    want = dict(line.split()[::-1] for line in open(os.path.join(ROOT, "tests", "golden", "reference_datasets.md5")))
    assert sorted(want) == sorted(f"datasets/{n}.csv" for n in
                                  ["resnet18", "resnet34", "resnet50", "resnet101", "resnet152", "shapes"])
    for path, md5 in want.items():
        assert hashlib.md5(open(os.path.join(ROOT, path), "rb").read()).hexdigest() == md5, path


def test_packed_container_roundtrip_on_the_host(spfy):
    """the pruned-layer container is host-only code: write, read back, and refuse every kind of damage"""
    import ctypes
    import numpy as np
    capi = spfy.capi
    rows, cols = 130, 576
    for layout in (capi.LAYOUT_CANONICAL, capi.LAYOUT_SM100):
        vb, mb, n = ctypes.c_size_t(), ctypes.c_size_t(), ctypes.c_size_t()
        capi.spfy_compressed_bytes(capi.F16, rows, cols, layout, ctypes.byref(vb), ctypes.byref(mb))
        capi.spfy_packed_bytes(capi.F16, rows, cols, layout, ctypes.byref(n))
        assert n.value == 64 + vb.value + mb.value
        rng = np.random.default_rng(layout)
        vals = rng.integers(0, 256, vb.value, dtype=np.uint8)
        meta = rng.integers(0, 256, mb.value, dtype=np.uint8)
        buf = np.zeros(n.value, dtype=np.uint8)
        capi.spfy_packed_write(capi.F16, layout, rows, cols, vals.ctypes.data, meta.ctypes.data, buf.ctypes.data, buf.size)
        assert bytes(buf[:6]) == b"SPFY24"

        def read(b):
            dt, lo = ctypes.c_int(), ctypes.c_int()
            out = [ctypes.c_size_t() for _ in range(6)]
            capi.spfy_packed_read(b.ctypes.data, b.size, ctypes.byref(dt), ctypes.byref(lo), *[ctypes.byref(x) for x in out])
            return (dt.value, lo.value) + tuple(x.value for x in out)

        dt, lo, r, c, vo, vbytes, mo, mbytes = read(buf)
        assert (dt, lo, r, c) == (capi.F16, layout, rows, cols) and (vo, vbytes, mo, mbytes) == (64, vb.value, 64 + vb.value, mb.value)
        assert np.array_equal(buf[vo: vo + vbytes], vals) and np.array_equal(buf[mo: mo + mbytes], meta)
        for damage in ("payload", "magic", "truncate", "shape"):
            b = buf.copy()
            if damage == "payload":
                b[64 + 5] ^= 1
            elif damage == "magic":
                b[0] = ord("X")
            elif damage == "truncate":
                b = b[:-1].copy()
            else:
                b[24] ^= 2  # rows
            with pytest.raises(spfy.SpfyError):
                read(b)
        small = np.zeros(n.value - 1, dtype=np.uint8)
        with pytest.raises(spfy.SpfyError):
            capi.spfy_packed_write(capi.F16, layout, rows, cols, vals.ctypes.data, meta.ctypes.data, small.ctypes.data, small.size)
