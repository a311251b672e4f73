#!/usr/bin/env python3
"""What 2:4 fine-tuning costs on the GPU (fp16, L2 flushed before every timed call, median of 7 CUDA-event timings):

  transpose24   spfy_transpose24 on a TILE-pruned 16384 x 16384 operand, and summed over the ResNet-50 weight set
                (every unique conv weight of datasets/resnet50.csv but the 3-channel first layer, taps = 1).
                Bytes: 1.125 per element read (values + metadata) + 1.125 written.  Bound: HBM.
  recompress24  spfy_recompress24 from an fp32 master (4 bytes read per element + 0.125 metadata, 1 written), the
                compressed values only; same shapes.  Bound: HBM.
  linear24      forward + backward of Linear24 layers (an MLP in -> hidden -> in at `tokens` tokens) against
                torch.nn.functional.linear with the dense masked fp16 weights and torch autograd.
  conv3x3_dx    the data gradient of the ResNet-50 3x3 stride-1 layers at batch b: spfy_spmma_conv_nhwc of dy with the
                transposed, flipped filter (transpose24 not included) against torch.nn.grad.conv2d_input (cuDNN, NCHW).

    python tools/train24_probe.py [--out profiles/r03_train24.csv] [--tokens 8192] [--mlp 4096,16384] [--batch 32]
"""
import argparse
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
    ap.add_argument("--out", default=None)
    ap.add_argument("--tokens", type=int, default=8192)
    ap.add_argument("--mlp", default="4096,16384")
    ap.add_argument("--batch", type=int, default=32)
    args = ap.parse_args()
    import torch
    import torch.nn.functional as F
    spfy = ge.load_package()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn):
        fn()  # warm: module load, first launch, torch's algorithm choice
        ts = []
        for _ in range(7):
            flush.zero_()
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e3)
        return statistics.median(ts)

    gpu = card()
    rows = []

    def row(kind, shape, ours, ref=None, nbytes=None):
        gbs = nbytes / (ours * 1e-6) / 1e9 if nbytes else None
        rows.append((kind, shape, ours, ref, gbs))
        print(f"{kind:13s} {shape:28s} {ours:10.1f} us" + (f"  torch {ref:10.1f} us  x{ref / ours:5.2f}" if ref else "") +
              (f"  {gbs:7.0f} GB/s" if gbs else ""), flush=True)

    def pruned(m, k):
        w = torch.randn(m, k, device=dev).half()
        return spfy.prune24(w, inplace=True, mode=spfy.PRUNE_TILE_TRANSPOSABLE), w

    # ---- the two new kernels
    weights = [(16384, 16384)]
    seen = set()
    for s in spfy.shapes.read_shapes("resnet50.csv"):
        g = spfy.shapes.to_gemm(s)
        if g.K % 8 == 0 and (g.M, g.K) not in seen:
            seen.add((g.M, g.K))
            weights.append((g.M, g.K))
    sums = {"transpose24": [0.0, 0], "recompress24": [0.0, 0]}
    for i, (m, k) in enumerate(weights):
        comp, _ = pruned(m, k)
        comp_t = spfy.alloc_compressed(torch.float16, k, m, dev)
        master = torch.randn(m, k, device=dev)
        tt = timed(lambda: spfy.transpose24(comp, out=comp_t))
        tr = timed(lambda: spfy.recompress24(master, comp))
        bt, br = int(2.25 * m * k), int((4 + 0.125 + 1) * m * k)
        if i == 0:
            row("transpose24", f"{m}x{k}", tt, nbytes=bt)
            row("recompress24", f"{m}x{k} fp32", tr, nbytes=br)
        else:
            for key, t, b in (("transpose24", tt, bt), ("recompress24", tr, br)):
                sums[key][0] += t
                sums[key][1] += b
        del comp, comp_t, master
    for key, (t, b) in sums.items():
        row(key, f"resnet50 sum ({len(weights) - 1})", t, nbytes=b)

    # ---- Linear24 MLP forward + backward against dense torch
    d_in, d_hid = (int(v) for v in args.mlp.split(","))
    t = args.tokens
    l1 = spfy.Linear24.from_dense(torch.randn(d_hid, d_in, device=dev) * 0.02, torch.zeros(d_hid, device=dev))
    l2 = spfy.Linear24.from_dense(torch.randn(d_in, d_hid, device=dev) * 0.02, torch.zeros(d_in, device=dev))
    w1 = l1.weight.detach().half().requires_grad_(True)
    w2 = l2.weight.detach().half().requires_grad_(True)
    b1 = torch.zeros(d_hid, device=dev, dtype=torch.half, requires_grad=True)
    b2 = torch.zeros(d_in, device=dev, dtype=torch.half, requires_grad=True)
    x = torch.randn(t, d_in, device=dev).half().requires_grad_(True)
    dy = torch.randn(t, d_in, device=dev).half()

    def ours():
        l2(l1(x)).backward(dy)

    def dense():
        F.linear(F.linear(x, w1, b1), w2, b2).backward(dy)

    row("linear24", f"{t} tok {d_in}-{d_hid}-{d_in} f+b", timed(ours), timed(dense))
    del l1, l2, w1, w2

    # ---- 3x3 stride-1 data gradient
    for ch, hw in ((64, 56), (128, 28), (256, 14), (512, 7)):
        nb = args.batch
        comp, dense_w = pruned(ch, ch * 9)
        comp_t = spfy.transpose24(comp, taps=9)
        dy_nhwc = torch.randn(nb, hw, hw, ch, device=dev).half()
        dx = torch.empty(nb, hw, hw, ch, device=dev).half()
        w_nchw = dense_w.view(ch, 3, 3, ch).permute(0, 3, 1, 2).contiguous()
        dy_nchw = dy_nhwc.permute(0, 3, 1, 2).contiguous()
        ta = timed(lambda: spfy.spmma_conv_nhwc(comp_t, dy_nhwc, 3, 3, stride=1, pad=1, out=dx))
        tb = timed(lambda: torch.nn.grad.conv2d_input((nb, ch, hw, hw), w_nchw, dy_nchw, padding=1))
        row("conv3x3_dx", f"c=m={ch} {hw}x{hw} b={nb}", ta, tb)

    if args.out:
        with open(args.out, "w") as f:
            f.write(f"# {gpu}; fp16; L2 flushed before every call; median of 7 CUDA-event timings (tools/train24_probe.py)\n")
            f.write("kernel,shape,ours_us,torch_us,speedup,gb_per_s\n")
            for kind, shape, a, b, gbs in rows:
                f.write(f"{kind},{shape},{a:.1f},{'' if b is None else f'{b:.1f}'},"
                        f"{'' if b is None else f'{b / a:.2f}'},{'' if gbs is None else f'{gbs:.0f}'}\n")
    print(f"# {gpu}")


if __name__ == "__main__":
    main()
