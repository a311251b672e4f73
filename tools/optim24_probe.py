#!/usr/bin/env python3
"""What an optimizer step of a 2:4 model costs on the GPU (L2 flushed before every timed step, median of 7 CUDA-event
timings, the card's name and power limit in the header):

  resnet50  Conv2d24 for every convolution past the stem, a Linear24 fc (2048 -> 1000), the fp32 stem and BatchNorm:
            161 parameter tensors, 53 of them 2:4 layers
  mlp       Linear24 4096 -> 16384 -> 4096 with biases

For each: torch.optim.SGD (momentum 0.9, torch's default foreach path) plus refresh() of every 2:4 layer against
SGD24, and torch.optim.AdamW(fused=True) plus refresh() against AdamW24.  `kernel` rows time spfy_optim24_step alone on
a table built once (what step() adds on the host is the difference).  Launches: spfy_launch_count per step (the
library's kernels only; torch's own are not counted).  GB/s: the algorithmic bytes over the time, the same bytes for
both sides: per fp32 element, SGD with momentum reads p, g, buf and writes p, buf (20 B), AdamW reads p, g, m, v and
writes p, m, v (28 B); a 2:4 weight adds 1 B of values, 1 B of transposed values and 1/8 B of metadata.

    python tools/optim24_probe.py [--out profiles/r03_optim24.csv]
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


def resnet50(spfy, torch, dev):
    """(2:4 layers, dense fp32 parameters) of ResNet-50 (torchvision v1.5: the stride on the 3x3 convolution)"""
    g = torch.Generator(device="cpu").manual_seed(0)
    layers = []
    dense = [torch.nn.Parameter(torch.randn(64, 3, 7, 7, generator=g).to(dev))]
    dense += [torch.nn.Parameter(torch.randn(64, generator=g).to(dev)) for _ in range(2)]
    cin = 64
    for width, blocks, stride in ((64, 3, 1), (128, 4, 2), (256, 6, 2), (512, 3, 2)):
        for b in range(blocks):
            s = stride if b == 0 else 1
            specs = [(width, cin, 1, 1, 0), (width, width, 3, s, 1), (4 * width, width, 1, 1, 0)]
            if b == 0:
                specs.append((4 * width, cin, 1, s, 0))
            for m, c, k, st, p in specs:
                layers.append(spfy.Conv2d24.from_dense(torch.randn(m, c, k, k, generator=g).to(dev) * 0.05, None,
                                                       stride=st, padding=p))
                dense += [torch.nn.Parameter(torch.randn(m, generator=g).to(dev)) for _ in range(2)]
            cin = 4 * width
    layers.append(spfy.Linear24.from_dense(torch.randn(1000, 2048, generator=g).to(dev) * 0.02,
                                           torch.randn(1000, generator=g).to(dev)))
    return layers, dense


def mlp(spfy, torch, dev):
    g = torch.Generator(device="cpu").manual_seed(1)
    return [spfy.Linear24.from_dense(torch.randn(16384, 4096, generator=g).to(dev) * 0.02, torch.zeros(16384, device=dev)),
            spfy.Linear24.from_dense(torch.randn(4096, 16384, generator=g).to(dev) * 0.02, torch.zeros(4096, device=dev))], []


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    import torch
    spfy = ge.load_package()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    flush = torch.empty(512 << 20, dtype=torch.uint8, device=dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)

    def timed(fn):
        fn()  # warm: module load, state allocation, first launch
        ts, launches = [], []
        for _ in range(7):
            flush.zero_()
            n0 = spfy.launch_count()
            e0.record()
            fn()
            e1.record()
            e1.synchronize()
            launches.append(spfy.launch_count() - n0)
            ts.append(e0.elapsed_time(e1) * 1e3)
        return statistics.median(ts), max(launches)

    gpu = card()
    rows = []
    for name, build in (("resnet50", resnet50), ("mlp 4096-16384-4096", mlp)):
        layers, dense = build(spfy, torch, dev)
        params = [p for layer in layers for p in layer.parameters()] + dense
        for p in params:
            p.grad = torch.randn_like(p) * 1e-3
        n24 = sum(layer.weight.numel() for layer in layers)
        n = sum(p.numel() for p in params)
        for algo, per_el, make_ref, make_ours in (
                ("sgd", 20, lambda ps: torch.optim.SGD(ps, lr=1e-3, momentum=0.9),
                 lambda ps: spfy.SGD24(ps, lr=1e-3, momentum=0.9)),
                ("adamw", 28, lambda ps: torch.optim.AdamW(ps, lr=1e-4, fused=True),
                 lambda ps: spfy.AdamW24(ps, lr=1e-4))):
            nbytes = per_el * n + 2.125 * n24
            ref, ours = make_ref(params), make_ours(params)

            def torch_step():
                ref.step()
                for layer in layers:
                    layer.refresh()

            tr, lr_ = timed(torch_step)
            to, lo = timed(ours.step)
            # the kernel alone, on the table step() builds
            items, hps, *_ = ours._table()
            stream = spfy.ops._stream()
            tk, lk = timed(lambda: spfy.capi.spfy_optim24_step(ours._ALGO, items, len(items), hps, len(hps), None, None,
                                                               stream))
            shape = f"{name} ({len(params)} tensors; {n / 1e6:.1f} M)"
            for method, t, la in ((f"torch {algo} + refresh", tr, lr_), (f"{algo}24 step()", to, lo),
                                  (f"{algo}24 kernel", tk, lk)):
                gbs = nbytes / (t * 1e-6) / 1e9
                rows.append((shape, method, t, la, gbs, tr / t))
                print(f"{shape:40s} {method:24s} {t:9.1f} us  {la:4d} launches  {gbs:6.0f} GB/s  x{tr / t:5.2f}",
                      flush=True)
            del ref, ours
        del layers, dense, params
        torch.cuda.empty_cache()
    if args.out:
        with open(args.out, "w") as f:
            f.write(f"# {gpu}; L2 flushed before every step; median of 7 CUDA-event timings (tools/optim24_probe.py)\n")
            f.write("workload,method,us,spfy_launches,gb_per_s,speedup_vs_torch\n")
            for shape, method, t, la, gbs, sp in rows:
                f.write(f"{shape},{method},{t:.1f},{la},{gbs:.0f},{sp:.2f}\n")
    print(f"# {gpu}")


if __name__ == "__main__":
    main()
