"""spmma epilogue (spfy_spmma_ex / spfy_spmma_conv_ex / spfy_spmma_plan_create_ex): per-row scale and bias, ReLU / GELU
and beta * C with the transposed (NHWC) output, applied to the accumulators before the output is written.

Parity bar: an identity epilogue is the plain entry point bit for bit in every launch class; ReLU, a 16-bit-exact bias and
the transposed C are bitwise against compositions of plain calls; scale and GELU against fp64 within the suite's 1e-2
relative bound; a ResNet-50 bottleneck block and a Linear + GELU layer end to end against torch in fp32."""
import ctypes

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from test_gpu_parity import CLASS_SHAPES, REL_TOL, rand_bits, rel_err, to_dev

pytestmark = pytest.mark.gpu

TDT = {0: torch.float16, 1: torch.bfloat16}


def rnd(gen, *shape, lo=-1.0, hi=1.0, dtype=torch.float32):
    return (torch.rand(*shape, device="cuda", generator=gen) * (hi - lo) + lo).to(dtype)


def spmma_ex_null(spfy, comp, b, out, alpha=1.0, beta=0.0, c=None, op_b=0, out_t=False):
    """spfy_spmma_ex with epi == NULL"""
    capi = spfy.capi
    m, k = comp.rows, comp.cols
    n = b.shape[1] if op_b == capi.OP_N else b.shape[0]
    capi.spfy_spmma_ex(capi.F16 if comp.dtype == torch.float16 else capi.BF16, op_b | (capi.OUT_T if out_t else 0), m, n, k,
                       float(alpha), comp.vals.data_ptr(), comp.meta.data_ptr(), b.data_ptr(), b.stride(0), float(beta),
                       c.data_ptr() if c is not None else None, c.stride(0) if c is not None else 0, out.data_ptr(),
                       out.stride(0), None, 0, None, ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    return out


# ------------------------------------------------------------------------------------------------ identity
@pytest.mark.parametrize("M,K,N", CLASS_SHAPES)
def test_identity_epilogue_is_the_plain_call_bitwise(spfy, orc, cuda, M, K, N):
    """epi = NULL and an all-NULL / NONE epilogue equal the plain entry point bit for bit: every launch class, both opB,
    both output layouts (with alpha != 1 on the transposed one), fp16 and bf16 on alternating shapes"""
    dt = CLASS_SHAPES.index((M, K, N)) % 2
    comp = spfy.prune24(to_dev(rand_bits(orc, dt, (M, K), seed=M * 5 + K), dt, cuda))
    b = to_dev(rand_bits(orc, dt, (K, N), seed=N + 3), dt, cuda)
    ops = [(spfy.OP_N, b)] + ([(spfy.OP_T, b.t().contiguous())] if K % 8 == 0 else [])
    for op_b, bb in ops:
        for out_t, alpha in [(False, 1.0)] + ([(True, 1.0), (True, 0.5)] if M % 8 == 0 else []):
            want = spfy.spmma_compressed(comp, bb, op_b=op_b, out_t=out_t, alpha=alpha)
            got_null = spmma_ex_null(spfy, comp, bb, torch.empty_like(want), alpha=alpha, op_b=op_b, out_t=out_t)
            got_id = spfy.spmma_compressed(comp, bb, op_b=op_b, out_t=out_t, alpha=alpha, epilogue=spfy.Epilogue())
            torch.cuda.synchronize()
            assert torch.equal(got_null, want), (op_b, out_t, alpha)
            assert torch.equal(got_id, want), (op_b, out_t, alpha)


def test_identity_epilogue_with_c_is_the_plain_call_bitwise(spfy, orc, cuda):
    """row-major beta * C through the _ex entry: the plain call's alpha / beta code, bit for bit"""
    M, K, N = 300, 264, 9480
    comp = spfy.prune24(to_dev(rand_bits(orc, 0, (M, K), seed=1), 0, cuda))
    b = to_dev(rand_bits(orc, 0, (K, N), seed=2), 0, cuda)
    c = to_dev(rand_bits(orc, 0, (M, N), seed=3), 0, cuda)
    want = spfy.spmma_compressed(comp, b, c=c, alpha=0.5, beta=0.25)
    got = spfy.spmma_compressed(comp, b, c=c, alpha=0.5, beta=0.25, epilogue=spfy.Epilogue())
    torch.cuda.synchronize()
    assert torch.equal(got, want)


CONV_CASES = [(4, 56, 56, 64, 64, 3, 3, 1, 1), (2, 28, 28, 128, 256, 3, 3, 2, 1), (2, 56, 56, 64, 128, 1, 1, 2, 0),
              (3, 10, 12, 64, 72, 3, 3, 1, 1)]


@pytest.mark.parametrize("case", CONV_CASES, ids=lambda c: "x".join(str(v) for v in c))
@pytest.mark.parametrize("tdt", [torch.float16, torch.bfloat16], ids=["fp16", "bf16"])
def test_identity_epilogue_conv_both_layouts_bitwise(spfy, cuda, case, tdt):
    nb, h, w, c, cout, kh, kw, stride, pad = case
    gen = torch.Generator(device=cuda)
    gen.manual_seed(sum(case) + 9)
    x = rnd(gen, nb, h, w, c, dtype=tdt)
    comp = spfy.prune24(spfy.permute_conv_weights(rnd(gen, cout, c * kh * kw, dtype=tdt), c, kh, kw))
    want = spfy.spmma_conv(comp, x, kh, kw, stride=stride, pad=pad)
    want_t = spfy.spmma_conv_nhwc(comp, x, kh, kw, stride=stride, pad=pad)
    got = spfy.spmma_conv(comp, x, kh, kw, stride=stride, pad=pad, epilogue=spfy.Epilogue())
    got_t = spfy.spmma_conv_nhwc(comp, x, kh, kw, stride=stride, pad=pad, epilogue=spfy.Epilogue())
    torch.cuda.synchronize()
    assert torch.equal(got, want)
    assert torch.equal(got_t, want_t)


# ------------------------------------------------------------------------------------- ReLU, bias: bitwise
@pytest.mark.parametrize("M,K,N", [(64, 147, 19008), (200, 72, 19080), (512, 200, 9600), (128, 1152, 2048), (384, 640, 12752)])
def test_relu_is_relu_of_the_plain_output(spfy, orc, cuda, M, K, N):
    """rounding to 16 bit commutes with max(., 0): bitwise, both layouts"""
    comp = spfy.prune24(to_dev(rand_bits(orc, 0, (M, K), seed=M + 11), 0, cuda))
    b = to_dev(rand_bits(orc, 0, (K, N), seed=N + 12), 0, cuda)
    want = spfy.spmma_compressed(comp, b, alpha=0.75).relu()
    got = spfy.spmma_compressed(comp, b, alpha=0.75, epilogue=spfy.Epilogue(act="relu"))
    got_t = spfy.spmma_compressed(comp, b, alpha=0.75, out_t=True, epilogue=spfy.Epilogue(act="relu"))
    torch.cuda.synchronize()
    assert torch.equal(got, want)
    assert torch.equal(got_t, want.t())


@pytest.mark.parametrize("M,K,N,dt", [(64, 147, 19008, 0), (256, 64, 19200, 1), (1024, 256, 4800, 0), (96, 2304, 1000, 1),
                                      (256, 384, 25088, 0)])
def test_bias_equals_beta_c_with_the_bias_broadcast(spfy, orc, cuda, M, K, N, dt):
    """alpha = 1 and 16-bit-exact bias values: the bias epilogue is the plain call with C = bias broadcast, beta = 1"""
    comp = spfy.prune24(to_dev(rand_bits(orc, dt, (M, K), seed=M + 21), dt, cuda))
    b = to_dev(rand_bits(orc, dt, (K, N), seed=N + 22), dt, cuda)
    gen = torch.Generator(device=cuda)
    gen.manual_seed(M)
    bias16 = rnd(gen, M, lo=-2, hi=2, dtype=TDT[dt])
    want = spfy.spmma_compressed(comp, b, c=bias16[:, None].expand(M, N).contiguous(), beta=1.0)
    epi = spfy.Epilogue(bias=bias16.float())
    got = spfy.spmma_compressed(comp, b, epilogue=epi)
    got_t = spfy.spmma_compressed(comp, b, out_t=True, epilogue=epi)
    torch.cuda.synchronize()
    assert torch.equal(got, want)
    assert torch.equal(got_t, want.t())


@pytest.mark.parametrize("M,K,N", [(104, 576, 19000), (200, 72, 19080), (512, 200, 9600), (1024, 256, 9600), (136, 260, 264)])
@pytest.mark.parametrize("dt", [0, 1])
def test_transposed_c_is_the_transpose_of_the_row_major_c(spfy, orc, cuda, M, K, N, dt):
    """SPFY_OUT_T with C as [n][m]: bitwise the transpose of the row-major result with C as [m][n] -- identity and full
    epilogues, a pitched C, D aliasing C, m not a multiple of 32"""
    comp = spfy.prune24(to_dev(rand_bits(orc, dt, (M, K), seed=M + 31), dt, cuda))
    b = to_dev(rand_bits(orc, dt, (K, N), seed=N + 32), dt, cuda)
    c = to_dev(rand_bits(orc, dt, (M, N), seed=N + 33), dt, cuda)
    gen = torch.Generator(device=cuda)
    gen.manual_seed(N)
    full = spfy.Epilogue(scale=rnd(gen, M, lo=0.5, hi=1.5), bias=rnd(gen, M), act="relu")
    ld = (M + 15) // 8 * 8
    for epi in (spfy.Epilogue(), full):
        want = spfy.spmma_compressed(comp, b, c=c, alpha=0.5, beta=0.75, epilogue=epi)
        ct = torch.full((N, ld), 3.0, dtype=c.dtype, device=cuda)
        ct[:, :M] = c.t()
        got = spfy.spmma_compressed(comp, b, c=ct[:, :M], alpha=0.5, beta=0.75, out_t=True, epilogue=epi)
        alias = ct.clone()
        spfy.spmma_compressed(comp, b, c=alias[:, :M], out=alias[:, :M], alpha=0.5, beta=0.75, out_t=True, epilogue=epi)
        torch.cuda.synchronize()
        assert torch.equal(got, want.t())
        assert torch.equal(alias[:, :M], want.t())
        assert bool((alias[:, M:] == 3.0).all())  # nothing written beyond column m


# ---------------------------------------------------------------------------------- scale, GELU: fp64
def gelu_tanh64(v):
    return 0.5 * v * (1.0 + np.tanh(np.sqrt(2.0 / np.pi) * (v + 0.044715 * v ** 3)))


@pytest.mark.parametrize("M,K,N", [(64, 147, 19008), (200, 40, 19080), (512, 200, 9600), (128, 1152, 2048), (256, 384, 25088)])
@pytest.mark.parametrize("dt", [0, 1])
def test_scale_bias_gelu_against_fp64(spfy, orc, cuda, M, K, N, dt):
    a_bits = rand_bits(orc, dt, (M, K), seed=M + 41)
    b_bits = rand_bits(orc, dt, (K, N), seed=N + 42)
    acc = orc.spmma_f64(dt, orc.prune24_strip(dt, a_bits, want_mask=False)["dense"], b_bits)
    comp = spfy.prune24(to_dev(a_bits, dt, cuda))
    b = to_dev(b_bits, dt, cuda)
    gen = torch.Generator(device=cuda)
    gen.manual_seed(M + N)
    scale, bias = rnd(gen, M, lo=0.25, hi=2.0), rnd(gen, M)
    s64, b64 = scale.double().cpu().numpy()[:, None], bias.double().cpu().numpy()[:, None]
    for act, f in (("none", lambda v: v), ("gelu_tanh", gelu_tanh64)):
        want = f(0.5 * s64 * acc + b64)
        for out_t in (False, True):
            got = spfy.spmma_compressed(comp, b, alpha=0.5, out_t=out_t, epilogue=spfy.Epilogue(scale, bias, act))
            got = got.t() if out_t else got
            assert rel_err(got.double().cpu().numpy(), want) <= REL_TOL, (act, out_t)


# ------------------------------------------------------------------------------- end to end: ResNet, Linear
def bn_params(gen, c):
    return (rnd(gen, c, lo=0.5, hi=1.5), rnd(gen, c, lo=-0.5, hi=0.5), rnd(gen, c, lo=-0.1, hi=0.1),
            rnd(gen, c, lo=0.5, hi=1.5))


def pruned_conv(spfy, gen, cout, cin, k, tdt):
    wt = (rnd(gen, cout, cin * k * k) * (1.0 / (cin * k * k) ** 0.5) * 2).to(tdt)
    wp = spfy.permute_conv_weights(wt, cin, k, k)
    dense = torch.empty_like(wp)
    comp = spfy.prune24(wp, out_dense=dense)
    return comp, dense.view(cout, k, k, cin).permute(0, 3, 1, 2).float()  # torch layout [cout, cin, k, k]


@pytest.mark.parametrize("cin,mid,cout,stride", [(256, 64, 256, 1), (256, 128, 512, 2)], ids=["identity", "projection"])
@pytest.mark.parametrize("tdt", [torch.float16, torch.bfloat16], ids=["fp16", "bf16"])
def test_resnet50_bottleneck_block_in_nhwc(spfy, cuda, cin, mid, cout, stride, tdt):
    """1x1 -> 3x3 -> 1x1 + shortcut, batch norm folded, ReLU, all NHWC: three calls (four with the projection), no
    elementwise pass.  Every call against torch's conv2d / batch_norm / relu in fp32 on the pruned weights, fed the
    16-bit tensors that call was fed (a chain of independent references drifts apart by whole bf16 ulps wherever
    the two sides round a value near a rounding boundary differently)"""
    gen = torch.Generator(device=cuda)
    gen.manual_seed(cin + cout + stride)
    nb, hw = 4, 28
    x = rnd(gen, nb, hw, hw, cin, dtype=tdt)
    k1, f1 = pruned_conv(spfy, gen, mid, cin, 1, tdt)
    k2, f2 = pruned_conv(spfy, gen, mid, mid, 3, tdt)
    k3, f3 = pruned_conv(spfy, gen, cout, mid, 1, tdt)
    bn1, bn2, bn3 = bn_params(gen, mid), bn_params(gen, mid), bn_params(gen, cout)
    e1 = spfy.Epilogue(*spfy.fold_batchnorm(*bn1), act="relu")
    e2 = spfy.Epilogue(*spfy.fold_batchnorm(*bn2), act="relu")
    e3 = spfy.Epilogue(*spfy.fold_batchnorm(*bn3), act="relu")
    y1 = spfy.spmma_conv_nhwc(k1, x, 1, 1, epilogue=e1)
    y2 = spfy.spmma_conv_nhwc(k2, y1, 3, 3, stride=stride, pad=1, epilogue=e2)
    if stride == 1:
        shortcut = x
    else:
        kp, fp = pruned_conv(spfy, gen, cout, cin, 1, tdt)
        bnp = bn_params(gen, cout)
        shortcut = spfy.spmma_conv_nhwc(kp, x, 1, 1, stride=stride, epilogue=spfy.Epilogue(*spfy.fold_batchnorm(*bnp)))
    y3 = spfy.spmma_conv_nhwc(k3, y2, 1, 1, c=shortcut, beta=1.0, epilogue=e3)
    torch.cuda.synchronize()

    def bn(t, p):
        g, b, m, v = p
        return F.batch_norm(t, m, v, g, b, training=False, eps=1e-5)

    def nchw(t):
        return t.permute(0, 3, 1, 2).float()

    def close(got, ref):
        ref = ref.permute(0, 2, 3, 1)
        assert got.shape == ref.shape
        scale = torch.clamp(ref.abs(), min=1e-2 * float(ref.abs().max()))
        return float(((got.float() - ref).abs() / scale).max())

    tf32 = torch.backends.cudnn.allow_tf32
    torch.backends.cudnn.allow_tf32 = False  # a fp32 reference (cuDNN's default would round the operands to TF32)
    try:
        errs = [close(y1, F.relu(bn(F.conv2d(nchw(x), f1), bn1))),
                close(y2, F.relu(bn(F.conv2d(nchw(y1), f2, stride=stride, padding=1), bn2))),
                close(y3, F.relu(bn(F.conv2d(nchw(y2), f3), bn3) + nchw(shortcut)))]
        if stride != 1:
            errs.append(close(shortcut, bn(F.conv2d(nchw(x), fp, stride=stride), bnp)))
    finally:
        torch.backends.cudnn.allow_tf32 = tf32
    assert max(errs) <= 1e-2, errs

@pytest.mark.parametrize("tdt", [torch.float16, torch.bfloat16], ids=["fp16", "bf16"])
def test_linear_bias_gelu(spfy, cuda, tdt):
    """y = gelu(x W^T + b): opB = T with B = x and the transposed output, bias per row of A (output feature)"""
    gen = torch.Generator(device=cuda)
    gen.manual_seed(3)
    tokens, fin, fout = 1000, 768, 3072
    x = rnd(gen, tokens, fin, dtype=tdt)
    w = (rnd(gen, fout, fin) * (3.0 / fin) ** 0.5).to(tdt)
    bias = rnd(gen, fout)
    wd = torch.empty_like(w)
    comp = spfy.prune24(w, out_dense=wd)
    y = spfy.spmma_compressed(comp, x, op_b=spfy.OP_T, out_t=True, epilogue=spfy.Epilogue(bias=bias, act="gelu_tanh"))
    ref = F.gelu(F.linear(x.float(), wd.float(), bias), approximate="tanh")
    torch.cuda.synchronize()
    assert y.shape == (tokens, fout)
    scale = torch.clamp(ref.abs(), min=1e-2 * float(ref.abs().max()))
    assert float(((y.float() - ref).abs() / scale).max()) <= 1e-2


# ------------------------------------------------------------------------------------------------ plans
def test_plan_with_epilogues_matches_single_calls(spfy, cuda):
    """matrix and convolution problems, both layouts, with and without epilogues (and an NHWC shortcut add): every
    output bitwise the single _ex call's, and the same launches as the plan without epilogues"""
    tdt = torch.float16
    gen = torch.Generator(device=cuda)
    gen.manual_seed(99)
    problems, wants = [], []
    for i, (nb, h, w, c, cout, kh, kw, stride, pad, nhwc) in enumerate([
            (4, 56, 56, 64, 64, 3, 3, 1, 1, True), (2, 28, 28, 128, 256, 3, 3, 2, 1, False),
            (8, 7, 7, 512, 512, 3, 3, 1, 1, True), (2, 56, 56, 64, 128, 1, 1, 2, 0, True), (3, 10, 12, 64, 72, 3, 3, 1, 1, False)]):
        x = rnd(gen, nb, h, w, c, dtype=tdt)
        comp = spfy.prune24(spfy.permute_conv_weights(rnd(gen, cout, c * kh * kw, dtype=tdt), c, kh, kw))
        epi = spfy.Epilogue(rnd(gen, cout, lo=0.5, hi=1.5), rnd(gen, cout), act=("relu", "gelu_tanh")[i % 2]) if i != 1 else None
        ho, wo = (h + 2 * pad - kh) // stride + 1, (w + 2 * pad - kw) // stride + 1
        q = dict(comp=comp, b=x, conv=(kh, kw, stride, pad), out_t=nhwc)
        if nhwc:
            cc = rnd(gen, nb, ho, wo, cout, dtype=tdt) if i == 0 else None
            want = spfy.spmma_conv_nhwc(comp, x, kh, kw, stride=stride, pad=pad, c=cc, beta=1.0 if cc is not None else 0.0,
                                        epilogue=epi)
            q.update(out=torch.zeros_like(want), c=cc, beta=1.0 if cc is not None else 0.0)
        else:
            want = spfy.spmma_conv(comp, x, kh, kw, stride=stride, pad=pad, epilogue=epi)
            q.update(out=torch.zeros_like(want))
        if epi is not None:
            q["epilogue"] = epi
        problems.append(q)
        wants.append(want)
    for i, (M, K, N) in enumerate([(64, 147, 19008), (512, 200, 1600), (256, 2304, 392), (128, 1152, 520), (256, 64, 19200)]):
        a = rnd(gen, M, K, dtype=tdt)
        op_t = i % 2 == 1 and K % 8 == 0
        b = rnd(gen, *((N, K) if op_t else (K, N)), dtype=tdt)
        comp = spfy.prune24(a)
        op_b = spfy.OP_T if op_t else spfy.OP_N
        epi = spfy.Epilogue(rnd(gen, M, lo=0.5, hi=1.5), rnd(gen, M), act="relu") if i != 2 else None
        out_t = i >= 3
        want = spfy.spmma_compressed(comp, b, op_b=op_b, out_t=out_t, epilogue=epi)
        q = dict(comp=comp, b=b, out=torch.zeros_like(want), op_b=op_b, out_t=out_t)
        if epi is not None:
            q["epilogue"] = epi
        problems.append(q)
        wants.append(want)
    plan = spfy.SpmmaPlan(problems)
    plan.run()
    plan.run()
    torch.cuda.synchronize()
    for j, (q, want) in enumerate(zip(problems, wants)):
        assert torch.equal(q["out"], want), j
    plain = spfy.SpmmaPlan([{k: v for k, v in q.items() if k not in ("epilogue", "c", "beta")} for q in problems])
    assert plan.launches == plain.launches
    plan.close()
    plain.close()


# ------------------------------------------------------------------------------------------------ refusals
def test_bad_epilogues_are_refused(spfy, cuda):
    capi = spfy.capi
    M, K, N = 128, 128, 256
    comp = spfy.prune24(torch.ones(M, K, dtype=torch.float16, device=cuda))
    b = torch.ones(K, N, dtype=torch.float16, device=cuda)
    d = torch.empty(M, N, dtype=torch.float16, device=cuda)
    s = torch.ones(M + 1, dtype=torch.float32, device=cuda)
    stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def call(epi):
        return capi.spfy_spmma_ex.raw(capi.F16, capi.OP_N, M, N, K, 1.0, comp.vals.data_ptr(), comp.meta.data_ptr(),
                                      b.data_ptr(), N, 0.0, None, 0, d.data_ptr(), N, None, 0, ctypes.byref(epi), stream)

    assert call(capi.Epilogue(None, None, 3)) == capi.E_INVALID
    assert call(capi.Epilogue(None, None, -1)) == capi.E_INVALID
    assert call(capi.Epilogue(s.data_ptr() + 2, None, capi.ACT_RELU)) == capi.E_INVALID
    assert call(capi.Epilogue(None, s.data_ptr() + 2, capi.ACT_NONE)) == capi.E_INVALID
    assert call(capi.Epilogue(s.data_ptr() + 4, s.data_ptr(), capi.ACT_GELU_TANH)) == capi.OK
    with pytest.raises(ValueError):
        spfy.spmma_compressed(comp, b, epilogue=spfy.Epilogue(act="swish"))
    # the plain entry points keep their contract: no beta * C with the transposed output
    with pytest.raises(spfy.SpfyError):
        spfy.spmma_compressed(comp, b, c=d.t().contiguous(), beta=1.0, out_t=True)
    torch.cuda.synchronize()
