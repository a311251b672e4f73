#!/usr/bin/env python3
"""The data gradient of the strided ResNet-50 layers on the GPU (fp16, L2 flushed before every timed call, median of 7
CUDA-event timings), three ways:

  ours         spfy_spmma_conv_dgrad: one stride-1 implicit GEMM per output phase, scattered into dx (transpose24_conv
               not included)
  zero_insert  dy upsampled with zeros in torch, then the stride-1 path (spmma_conv_nhwc of transpose24(comp, taps) with
               pad k - 1 - pad), the upsampling included
  cudnn        torch.nn.grad.conv2d_input on the dense masked filter (NCHW)

and the launch form of the phases: `chained` (each phase's launch may start while the previous one runs, what the
library does) against `serial` (plain stream order, the SPFY_SPMMA_NO_OVERLAP switch of the dev build), both on the
dev library (python sparsify.me_b200/build.py --dev) in a subprocess, alternated three times, medians taken.

A layer reads "k x k, stride, dx channels <- dy channels, input h x w, batch".

    python tools/conv_dgrad_probe.py [--out profiles/r03_conv_dgrad.csv] [--batch 32]
"""
import argparse
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))
import __graft_entry__ as ge  # noqa: E402
from train24_probe import card  # noqa: E402

# (m, c, k, stride, pad, input h = w): the six strided layers of torchvision's ResNet-50 past its stem
LAYERS = [(128, 128, 3, 2, 1, 56), (256, 256, 3, 2, 1, 28), (512, 512, 3, 2, 1, 14),
          (512, 256, 1, 2, 0, 56), (1024, 512, 1, 2, 0, 28), (2048, 1024, 1, 2, 0, 14)]


DEV_LIB = os.path.join(ROOT, "sparsify.me_b200", "lib_dev", "libsparsifyme_b200.so")


def make_timer(torch, dev):
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
    return timed


def layer(spfy, torch, dev, m, c, k, s, p, hw, nb):
    """(pruned filter, comp, op, dy, dx) of one layer, fp16"""
    w = torch.randn(m, k * k * c, device=dev).half()
    comp = spfy.prune24(w, inplace=True, mode=spfy.PRUNE_TILE_TRANSPOSABLE)  # w: the pruned filter, (kh, kw, c)
    op = spfy.transpose24_conv(comp, k, k, s, p)
    ho = (hw + 2 * p - k) // s + 1
    return w, comp, op, torch.randn(nb, ho, ho, m, device=dev).half(), torch.empty(nb, hw, hw, c, device=dev).half()


def phase_launches(nb):
    """(runs on the dev library) one JSON line per layer: chained and serial phase launches, alternated"""
    import torch
    spfy = ge.load_package()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    timed = make_timer(torch, dev)
    for m, c, k, s, p, hw in LAYERS:
        _, _, op, dy, dx = layer(spfy, torch, dev, m, c, k, s, p, hw, nb)
        chained, serial = [], []
        for _ in range(3):
            os.environ.pop("SPFY_SPMMA_NO_OVERLAP", None)
            chained.append(timed(lambda: spfy.spmma_conv_dgrad_nhwc(op, dy, hw, hw, out=dx)))
            os.environ["SPFY_SPMMA_NO_OVERLAP"] = "1"
            serial.append(timed(lambda: spfy.spmma_conv_dgrad_nhwc(op, dy, hw, hw, out=dx)))
        os.environ.pop("SPFY_SPMMA_NO_OVERLAP", None)
        print(json.dumps({"chained": statistics.median(chained), "serial": statistics.median(serial)}), flush=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=None)
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--phase-launches", action="store_true", help=argparse.SUPPRESS)
    args = ap.parse_args()
    if args.phase_launches:
        return phase_launches(args.batch)
    if not os.path.exists(DEV_LIB):
        sys.exit(f"{DEV_LIB} is missing: build it with `python sparsify.me_b200/build.py --dev`")
    import torch
    spfy = ge.load_package()
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    timed = make_timer(torch, dev)

    gpu = card()
    nb = args.batch
    rows = []
    for m, c, k, s, p, hw in LAYERS:
        w, comp, op, dy, dx = layer(spfy, torch, dev, m, c, k, s, p, hw, nb)
        comp_t = spfy.transpose24(comp, taps=k * k)
        ho = dy.shape[1]
        up = hw - k + 1 + 2 * p  # the zero-inserted dy: a stride-1 layer with pad k - 1 - p maps it onto h x w
        dy_up = torch.zeros(nb, up, up, m, device=dev).half()

        def zero_insert():
            dy_up.zero_()
            dy_up[:, : (ho - 1) * s + 1: s, : (ho - 1) * s + 1: s] = dy
            spfy.spmma_conv_nhwc(comp_t, dy_up, k, k, stride=1, pad=k - 1 - p, out=dx)

        w_nchw = w.view(m, k, k, c).permute(0, 3, 1, 2).contiguous()
        dy_nchw = dy.permute(0, 3, 1, 2).contiguous()
        ta = timed(lambda: spfy.spmma_conv_dgrad_nhwc(op, dy, hw, hw, out=dx))
        tz = timed(zero_insert)
        tc = timed(lambda: torch.nn.grad.conv2d_input((nb, c, hw, hw), w_nchw, dy_nchw, stride=s, padding=p))
        shape = f"{k}x{k} s{s} {c}<-{m} {hw}x{hw} b={nb}"
        rows.append((shape, ta, tz, tc))
        print(f"{shape:32s} ours {ta:8.1f} us  zero-insert {tz:8.1f} us  cudnn {tc:8.1f} us  x{tc / ta:5.2f} vs cudnn",
              flush=True)
        del w, comp, op, comp_t, dy, dx, dy_up, w_nchw, dy_nchw
    del timed
    torch.cuda.empty_cache()
    sub = subprocess.run([sys.executable, os.path.abspath(__file__), "--phase-launches", "--batch", str(nb)],
                         env=dict(os.environ, SPFY_LIB=DEV_LIB), capture_output=True, text=True, timeout=900)
    if sub.returncode:
        sys.exit(f"phase-launch comparison failed:\n{sub.stderr}")
    launches = [json.loads(ln) for ln in sub.stdout.splitlines() if ln.startswith("{")]
    assert len(launches) == len(rows)
    for i, ln in enumerate(launches):
        rows[i] += (ln["chained"], ln["serial"])
        print(f"{rows[i][0]:32s} phases chained {ln['chained']:8.1f} us  serial {ln['serial']:8.1f} us", flush=True)
    if args.out:
        with open(args.out, "w") as f:
            f.write(f"# {gpu}; fp16; L2 flushed before every call; median of 7 CUDA-event timings "
                    "(tools/conv_dgrad_probe.py)\n")
            f.write("layer,ours_us,zero_insert_us,cudnn_us,speedup_vs_cudnn,speedup_vs_zero_insert,"
                    "dev_chained_us,dev_serial_us\n")
            for shape, ta, tz, tc, ch, se in rows:
                f.write(f"{shape},{ta:.1f},{tz:.1f},{tc:.1f},{tc / ta:.2f},{tz / ta:.2f},{ch:.1f},{se:.1f}\n")
    print(f"# {gpu}")


if __name__ == "__main__":
    main()
