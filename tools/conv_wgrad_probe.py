#!/usr/bin/env python3
"""The weight gradient of every ResNet-50 convolution but the stem on the GPU (b = 32, fp16, random NHWC X and dY, L2
flushed before every timed call, median of 9 CUDA-event timings), two ways:

  ours   spfy_conv_wgrad24: the split-K implicit GEMM on tcgen05 plus the pass that sums the splits and masks, fp32 out
  cudnn  torch.ops.aten.convolution_backward (weight only) on channels_last fp16, then the multiply by the 2:4 mask

with the bytes each moves at least, the fp16 tensor-core and HBM bounds of ours (data-sheet figures, 2250 TFLOP/s and 7.7
TB/s: a share of them, not a claim that they were reached) and which of the two is the larger.  One more row: a bottleneck
block (1x1, 3x3 stride 2, 1x1, projection 1x1 stride 2, torch BatchNorm / ReLU) of Conv2d24 layers, forward and backward,
against the same block with dense fp16 channels_last torch convolutions.

A layer reads "k x k s stride, c -> m, input h x w".

    python tools/conv_wgrad_probe.py [--out profiles/r03_conv_wgrad.csv]
"""
import argparse
import ctypes
import os
import statistics
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.path.insert(0, os.path.join(ROOT, "tests"))
import __graft_entry__ as ge  # noqa: E402
from test_conv_wgrad import RESNET50, split_count  # noqa: E402
from train24_probe import card  # noqa: E402

HBM = 7.7e12
TC16 = 2250e12
NB = 32


def make_timer(torch, dev, reps=9):
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn):
        fn()
        fn()  # warm: module load, first launch, torch's algorithm choice
        ts = []
        for _ in range(reps):
            flush.zero_()
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            ts.append(e0.elapsed_time(e1) * 1e3)
        return statistics.median(ts)
    return timed


def layer_row(spfy, torch, dev, timed, c, m, hw, k, s, p):
    capi = spfy.capi
    ho = (hw + 2 * p - k) // s + 1
    kk = k * k * c
    w2 = torch.randn(m, kk, device=dev).half()
    comp = spfy.prune24(w2, inplace=True, mode=spfy.PRUNE_TILE_TRANSPOSABLE)
    x = torch.randn(NB, hw, hw, c, device=dev).half()
    dy = torch.randn(NB, ho, ho, m, device=dev).half()
    out = torch.empty(m, kk, device=dev)
    desc = capi.ConvDesc(NB, hw, hw, c, k, k, s, p)
    wb = ctypes.c_size_t()
    capi.spfy_conv_wgrad24_workspace_bytes(capi.F16, ctypes.byref(desc), m, ctypes.byref(wb))
    ws = torch.empty(wb.value, dtype=torch.uint8, device=dev)
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def ours():
        capi.spfy_conv_wgrad24(capi.F16, ctypes.byref(desc), m, 1.0, ctypes.c_void_p(x.data_ptr()),
                               ctypes.c_void_p(dy.data_ptr()), ctypes.c_void_p(comp.meta.data_ptr()), 0.0,
                               ctypes.c_void_p(out.data_ptr()), ctypes.c_void_p(ws.data_ptr()), ws.numel(), st)

    # the same layer in torch: NCHW-shaped channels_last views of the same data, mask as a channels_last fp16 weight
    xc, dyc = x.permute(0, 3, 1, 2), dy.permute(0, 3, 1, 2)
    ones = torch.ones(m, kk, device=dev)
    spfy.recompress24(ones, comp, masked_out=ones, values=False)
    mask = ones.half().view(m, k, k, c).permute(0, 3, 1, 2)
    weight = torch.empty(m, c, k, k, device=dev, dtype=torch.float16, memory_format=torch.channels_last)

    def cudnn():
        gw = torch.ops.aten.convolution_backward(dyc, xc, weight, None, [s, s], [p, p], [1, 1], False, [0, 0], 1,
                                                 [False, True, False])[1]
        return gw * mask

    t_ours, t_cudnn = timed(ours), timed(cudnn)
    splits = split_count(NB, hw, hw, c, k, k, s, p, m)
    positions = NB * ho * ho
    flops = 2.0 * m * kk * positions
    # at least: X and dY once, the split partials written and read, the metadata, dW written
    bytes_ours = x.numel() * 2 + dy.numel() * 2 + 2 * splits * m * kk * 4 + m * kk // 8 + m * kk * 4
    bytes_cudnn = x.numel() * 2 + dy.numel() * 2 + m * kk * 2 * 4  # ... dW fp16 written, read, masked and written
    t_hbm, t_tc = bytes_ours / HBM, flops / TC16
    return {"layer": f"{k}x{k} s{s} {c}->{m} {hw}x{hw}", "splits": splits, "ours_us": round(t_ours, 1),
            "cudnn_us": round(t_cudnn, 1), "speedup_vs_cudnn": round(t_cudnn / t_ours, 2), "ours_bytes": bytes_ours,
            "cudnn_bytes": bytes_cudnn, "gflop": round(flops / 1e9, 2),
            "hbm_share": round(t_hbm * 1e6 / t_ours, 3), "tc_share": round(t_tc * 1e6 / t_ours, 3),
            "bound": "hbm" if t_hbm > t_tc else "tensor"}


def block_row(spfy, torch, dev, timed):
    """stage-2 entry block of ResNet-50: 256 -> (128, 128 s2, 512) + projection 256 -> 512 s2, input 56 x 56"""
    c, mid, out, hw = 256, 128, 512, 56
    specs = [(mid, c, 1, 1, 0), (mid, mid, 3, 2, 1), (out, mid, 1, 1, 0), (out, c, 1, 2, 0)]
    ws = [torch.randn(m, ci, k, k, device=dev) * (2.0 / (ci * k * k)) ** 0.5 for m, ci, k, _, _ in specs]
    ours = [spfy.Conv2d24.from_dense(w, torch.zeros(w.shape[0], device=dev), stride=s, padding=p)
            for w, (_, _, _, s, p) in zip(ws, specs)]
    dense = []
    for w, (m, ci, k, s, p) in zip(ws, specs):
        cv = torch.nn.Conv2d(ci, m, k, stride=s, padding=p).to(dev).half().to(memory_format=torch.channels_last)
        with torch.no_grad():
            cv.weight.copy_(w)
        dense.append(cv)
    bns = [torch.nn.BatchNorm2d(m).to(dev) for m, *_ in specs]
    x = torch.randn(NB, c, hw, hw, device=dev).half().contiguous(memory_format=torch.channels_last).requires_grad_(True)
    g = torch.randn(NB, out, hw // 2, hw // 2, device=dev).half().contiguous(memory_format=torch.channels_last)

    def block(conv):
        h = torch.relu(bns[0](conv[0](x)))
        h = torch.relu(bns[1](conv[1](h)))
        return torch.relu(bns[2](conv[2](h)) + bns[3](conv[3](x)))

    def step(conv):
        return lambda: block(conv).backward(g)

    t_ours, t_torch = timed(step(ours)), timed(step(dense))
    return {"layer": "bottleneck 256->128->128 s2->512 + proj s2 56x56 fwd+bwd", "splits": "", "ours_us": round(t_ours, 1),
            "cudnn_us": round(t_torch, 1), "speedup_vs_cudnn": round(t_torch / t_ours, 2), "ours_bytes": "",
            "cudnn_bytes": "", "gflop": "", "hbm_share": "", "tc_share": "", "bound": ""}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_conv_wgrad.csv"))
    args = ap.parse_args()
    spfy = ge.load_package()
    import torch
    if not torch.cuda.is_available():
        raise SystemExit("conv_wgrad_probe: no CUDA device (this measurement runs on the GPU only)")
    dev = torch.device("cuda:0")
    torch.backends.cudnn.benchmark = True
    timed = make_timer(torch, dev)
    rows = [layer_row(spfy, torch, dev, timed, *layer) for layer in RESNET50]
    tot = {"layer": "resnet50 sum (22)", "splits": "", "ours_us": round(sum(r["ours_us"] for r in rows), 1),
           "cudnn_us": round(sum(r["cudnn_us"] for r in rows), 1), "ours_bytes": sum(r["ours_bytes"] for r in rows),
           "cudnn_bytes": sum(r["cudnn_bytes"] for r in rows), "gflop": round(sum(r["gflop"] for r in rows), 2),
           "hbm_share": "", "tc_share": "", "bound": ""}
    tot["speedup_vs_cudnn"] = round(tot["cudnn_us"] / tot["ours_us"], 2)
    rows += [tot, block_row(spfy, torch, dev, timed)]
    cols = ["layer", "splits", "ours_us", "cudnn_us", "speedup_vs_cudnn", "ours_bytes", "cudnn_bytes", "gflop", "hbm_share",
            "tc_share", "bound"]
    head = (f"# {card()}; fp16, b = {NB}; L2 flushed before every call; median of 9 CUDA-event timings "
            f"(tools/conv_wgrad_probe.py); shares of 7.7 TB/s and 2250 TFLOP/s (data sheet)")
    text = "\n".join([head, ",".join(cols)] + [",".join(str(r[k]) for k in cols) for r in rows]) + "\n"
    os.makedirs(os.path.dirname(args.out), exist_ok=True)
    with open(args.out, "w") as f:
        f.write(text)
    print(text)


if __name__ == "__main__":
    main()
