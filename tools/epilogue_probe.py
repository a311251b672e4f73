#!/usr/bin/env python3
"""What the spmma epilogue costs, and what it saves: every unique convolution layer of a datasets/*.csv table (the
3-channel first layer excepted) as an NHWC implicit GEMM at batch b, cold (L2 flushed before every launch, median of 7):

  a          spfy_spmma_conv_nhwc, the plain call
  b          spfy_spmma_conv_ex with an identity epilogue (must be a, same code)
  c          spfy_spmma_conv_ex with per-channel scale + bias + ReLU (conv + folded batch norm + ReLU)
  d          a followed by torch's (y * s + b).relu_(), the unfused alternative
  gelu       spfy_spmma_conv_ex with scale + bias + GELU (tanh form)
  gelu_torch a followed by torch's gelu(y * s + b, approximate="tanh")

The CSV records m = Ho * Wo, n = C_out, k = kh * kw * C_in but not the stride: a layer is run with stride 1 and
"same" padding, which gives the GEMM the table lists.  Then one ResNet-50 bottleneck block per stage with the identity
shortcut, fused (three calls: BN folded, ReLU, the shortcut added by the last call's beta * C in NHWC) against the
same three plain calls each followed by torch's elementwise pass; and a Linear + bias + GELU layer.

    python tools/epilogue_probe.py [--csv resnet50.csv] [--batch 32] [--out profiles/r03_epilogue.csv]
"""
import argparse
import collections
import math
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import __graft_entry__ as ge  # noqa: E402


def card():
    """name and power limit of GPU 0, read with the measurement"""
    try:
        q = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=name,power.limit", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=30).stdout.strip()
        return q or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--csv", default="resnet50.csv")
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--out", default=None, help="CSV file (default: stdout only)")
    args = ap.parse_args()
    import torch
    import torch.nn.functional as F
    spfy = ge.load_package()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn):
        fn()  # warm: module load, first launch
        ts = []
        for _ in range(7):
            flush.zero_()
            e0.record()
            fn()
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e3)
        return statistics.median(ts)

    def max_rel(got, want):
        want = want.float()
        scale = torch.clamp(want.abs(), min=1e-2 * float(want.abs().max()))
        return float(((got.float() - want).abs() / scale).max())

    rows = []
    gpu = card()
    head = f"# {gpu}; {args.csv} at batch {args.batch}; cold (L2 flushed before every launch), median of 7, microseconds"
    cols = ("kind,kh,Ho,C_in,C_out,count,out_MB,a_plain_us,b_identity_us,c_scale_bias_relu_us,d_plain_plus_torch_us,"
            "gelu_us,gelu_torch_us,b_identical,c_vs_fp32_epilogue_of_a_max_rel,gelu_vs_fp32_epilogue_of_a_max_rel")
    print(head)
    print(cols, flush=True)

    def emit(s):
        rows.append(s)
        print(s, flush=True)

    shapes = spfy.shapes.read_shapes(args.csv)
    layers = collections.Counter()
    for s in shapes:
        if s.k % 9 == 0 and (s.k // 9) % 64 == 0:
            layers[(3, s.m, s.k // 9, s.n)] += 1
        elif s.k % 64 == 0:
            layers[(1, s.m, s.k, s.n)] += 1
    tot = collections.Counter()
    nb = args.batch
    for (kh, m, cin, cout), cnt in sorted(layers.items(), key=lambda kv: (-kv[0][1], kv[0][0], kv[0][2])):
        ho = math.isqrt(m)
        pad = kh // 2
        gen = torch.Generator(device=dev)
        gen.manual_seed(m + cin + cout)
        x = (torch.rand(nb, ho, ho, cin, device=dev, generator=gen) * 2 - 1).half()
        w = ((torch.rand(cout, kh * kh * cin, device=dev, generator=gen) * 2 - 1) / math.sqrt(kh * kh * cin)).half()
        comp = spfy.prune24(w)
        scale = torch.rand(cout, device=dev, generator=gen) + 0.5
        bias = torch.rand(cout, device=dev, generator=gen) - 0.5
        s16, b16 = scale.half(), bias.half()
        y = torch.empty(nb, ho, ho, cout, dtype=torch.float16, device=dev)
        yb, yc, yg = torch.empty_like(y), torch.empty_like(y), torch.empty_like(y)
        relu = spfy.Epilogue(scale, bias, "relu")
        gelu = spfy.Epilogue(scale, bias, "gelu_tanh")
        res = {}

        def plain():
            spfy.spmma_conv_nhwc(comp, x, kh, kh, pad=pad, out=y)

        res["a"] = timed(plain)
        res["b"] = timed(lambda: spfy.spmma_conv_nhwc(comp, x, kh, kh, pad=pad, out=yb, epilogue=spfy.Epilogue()))
        res["c"] = timed(lambda: spfy.spmma_conv_nhwc(comp, x, kh, kh, pad=pad, out=yc, epilogue=relu))
        unfused = {}

        def plain_relu():
            plain()
            unfused["d"] = (y * s16 + b16).relu_()

        def plain_gelu():
            plain()
            unfused["g"] = F.gelu(y * s16 + b16, approximate="tanh")

        res["d"] = timed(plain_relu)
        res["g"] = timed(lambda: spfy.spmma_conv_nhwc(comp, x, kh, kh, pad=pad, out=yg, epilogue=gelu))
        res["gt"] = timed(plain_gelu)
        plain()
        ident = bool(torch.equal(y, yb))
        ref_c = torch.relu(y.float() * scale + bias)
        ref_g = F.gelu(y.float() * scale + bias, approximate="tanh")
        out_mb = y.numel() * 2 / 1e6
        emit(f"conv,{kh},{ho},{cin},{cout},{cnt},{out_mb:.1f},{res['a']:.1f},{res['b']:.1f},{res['c']:.1f},{res['d']:.1f},"
             f"{res['g']:.1f},{res['gt']:.1f},{ident},{max_rel(yc, ref_c):.2e},{max_rel(yg, ref_g):.2e}")
        for key in res:
            tot[key] += res[key] * cnt
        del x, w, comp, y, yb, yc, yg, unfused
    emit(f"total_weighted_by_count,,,,,,,{tot['a']:.0f},{tot['b']:.0f},{tot['c']:.0f},{tot['d']:.0f},{tot['g']:.0f},"
         f"{tot['gt']:.0f},,,")

    # ---- bottleneck blocks (identity shortcut), NHWC: fused vs plain calls + torch elementwise
    print("kind,Ho,C_in,mid,batch,fused_us,unfused_us,unfused_over_fused,max_rel_fused_vs_unfused")
    rows.append("kind,Ho,C_in,mid,batch,fused_us,unfused_us,unfused_over_fused,max_rel_fused_vs_unfused")
    for ho, cin, mid in [(56, 256, 64), (28, 512, 128), (14, 1024, 256), (7, 2048, 512)]:
        gen = torch.Generator(device=dev)
        gen.manual_seed(ho + cin)
        x = (torch.rand(nb, ho, ho, cin, device=dev, generator=gen) * 2 - 1).half()
        ks, eps, tch = [], [], []
        for co, ci, k in [(mid, cin, 1), (mid, mid, 3), (cin, mid, 1)]:
            w = ((torch.rand(co, k * k * ci, device=dev, generator=gen) * 2 - 1) / math.sqrt(k * k * ci)).half()
            ks.append((spfy.prune24(w), k))
            s = torch.rand(co, device=dev, generator=gen) + 0.5
            b = torch.rand(co, device=dev, generator=gen) - 0.5
            eps.append(spfy.Epilogue(s, b, "relu"))
            tch.append((s.half(), b.half()))
        f = [torch.empty(nb, ho, ho, c, dtype=torch.float16, device=dev) for c in (mid, mid, cin)]
        u = [torch.empty_like(t) for t in f]
        outs = {}

        def fused():
            spfy.spmma_conv_nhwc(ks[0][0], x, 1, 1, out=f[0], epilogue=eps[0])
            spfy.spmma_conv_nhwc(ks[1][0], f[0], 3, 3, pad=1, out=f[1], epilogue=eps[1])
            spfy.spmma_conv_nhwc(ks[2][0], f[1], 1, 1, out=f[2], c=x, beta=1.0, epilogue=eps[2])

        def unfused():
            spfy.spmma_conv_nhwc(ks[0][0], x, 1, 1, out=u[0])
            a1 = (u[0] * tch[0][0] + tch[0][1]).relu_()
            spfy.spmma_conv_nhwc(ks[1][0], a1, 3, 3, pad=1, out=u[1])
            a2 = (u[1] * tch[1][0] + tch[1][1]).relu_()
            spfy.spmma_conv_nhwc(ks[2][0], a2, 1, 1, out=u[2])
            outs["u"] = (u[2] * tch[2][0] + tch[2][1] + x).relu_()

        tf, tu = timed(fused), timed(unfused)
        fused()
        unfused()
        torch.cuda.synchronize()
        line = f"bottleneck,{ho},{cin},{mid},{nb},{tf:.1f},{tu:.1f},{tu / tf:.2f},{max_rel(f[2], outs['u']):.2e}"
        emit(line)
        del x, f, u, outs

    # ---- Linear + bias + GELU (y = gelu(x W^T + b): opB = T, B = x, transposed output)
    print("kind,tokens,in,out,fused_us,unfused_us,unfused_over_fused,max_rel_fused_vs_torch")
    rows.append("kind,tokens,in,out,fused_us,unfused_us,unfused_over_fused,max_rel_fused_vs_torch")
    for tokens, fin, fout in [(16384, 1024, 4096), (16384, 4096, 1024)]:
        gen = torch.Generator(device=dev)
        gen.manual_seed(tokens + fin)
        x = (torch.rand(tokens, fin, device=dev, generator=gen) * 2 - 1).half()
        w = ((torch.rand(fout, fin, device=dev, generator=gen) * 2 - 1) * math.sqrt(3.0 / fin)).half()
        b = torch.rand(fout, device=dev, generator=gen) - 0.5
        b16 = b.half()
        comp = spfy.prune24(w)
        yf, yp = torch.empty(tokens, fout, dtype=torch.float16, device=dev), torch.empty(tokens, fout, dtype=torch.float16, device=dev)
        epi = spfy.Epilogue(bias=b, act="gelu_tanh")
        outs = {}

        def fused():
            spfy.spmma_compressed(comp, x, op_b=spfy.OP_T, out_t=True, out=yf, epilogue=epi)

        def unfused():
            spfy.spmma_compressed(comp, x, op_b=spfy.OP_T, out_t=True, out=yp)
            outs["u"] = F.gelu(yp + b16, approximate="tanh")

        tf, tu = timed(fused), timed(unfused)
        fused()
        plain = spfy.spmma_compressed(comp, x, op_b=spfy.OP_T, out_t=True)
        ref = F.gelu(plain.float() + b, approximate="tanh")
        emit(f"linear_gelu,{tokens},{fin},{fout},{tf:.1f},{tu:.1f},{tu / tf:.2f},{max_rel(yf, ref):.2e}")
        del x, w, comp, yf, yp, outs
    if args.out:
        with open(args.out, "w") as fh:
            fh.write(head + "\n" + cols + "\n" + "\n".join(rows) + "\n")


if __name__ == "__main__":
    main()
