#!/usr/bin/env python3
"""bench.py -- the hot path of sparsify.me on B200: 2:4 magnitude prune+compress of every weight
matrix of a ResNet shape table, then the 2:4 sparse GEMM (spmma) of every layer.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]

One STEP = one pass over one batch of synthetic input: ONE batched prune+compress launch over all
layers' weights (spfy_prune24_batched) + the spmma of every layer through one plan
(spfy_spmma_plan_run: one persistent launch per ring-geometry class that walks all layers' tiles; the plan -- tensor maps
and tile schedule -- is built once outside the timed region, like cusparseLtMatmulPlanInit in the
reference, spmma.hxx:51-80), weights orientation M = C_out, K = C_in*kh*kw, N = H*W*b (SURVEY.md 8).  Workload = BASELINE.json
configs[1]: all of datasets/resnet50.csv, fp16, b = 32 images per GPU.  Every layer has its own
B / D buffers (7.4 GB per step, far larger than the 126 MB L2), so nothing is re-read from L2
between layers or steps.

value  : dense-equivalent TFLOP/s (2*M*N*K summed over layers and ranks / step time), inputs
         resident in HBM, device-timed with CUDA events, max over ranks.
e2e    : the same metric through the reference-shaped public call `spmma(A, B, C, m, n, k, b)`
         with HOST (pinned) buffers: H2D of A and B, prune+compress+multiply, D2H of C, per layer,
         all inside the timed region.
N > 1  : weak scaling -- every rank runs the same table on its own 32 images (the global batch is
         sharded on image boundaries; no data-path collective).
--impl reference : the CPU oracle port of the same math on the host cores (the reference has no
         CPU path of its own and its cusparseLt build is closed source; when oracle/_ref holds the
         cusparseLt comparator its B200 timing is added under "cusparselt").
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time


def claim_stdout():
    """stdout carries the one JSON line only.  NCCL prints its version banner to fd 1 whatever NCCL_DEBUG_FILE
    says, so multi-rank runs keep a private duplicate of the real stdout for the JSON line and point fd 1 at
    stderr for everything else (libraries included)."""
    sys.stdout.flush()
    out = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    return out


ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
import __graft_entry__ as ge  # noqa: E402

METRIC = "2:4 spmma TFLOP/s over ResNet-50 GEMM shapes (dense-equivalent 2MNK, prune+compress included)"
UNIT = "TFLOP/s"


def read_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            d = json.load(f)
        return float(d["hbm_gbs"]), float(d["bf16_tflops"]), float(d.get("bf16_tflops_sustained", d["bf16_tflops"])), "measured"
    return 6650.0, 1590.0, 1400.0, "fallback"


def ncu_traffic():
    """DRAM bytes per step of the spmma launches from the committed `ncu --set full` summary
    (profiles/rNN_spmma_ncu.csv: dram__bytes_read.sum + dram__bytes_write.sum over the launches of one
    step), or None when no capture is committed."""
    import csv
    import glob
    files = sorted(glob.glob(os.path.join(ROOT, "profiles", "r*_spmma_ncu.csv")))
    if not files:
        return None, None
    scale = {"byte": 1.0, "Kbyte": 1e3, "Mbyte": 1e6, "Gbyte": 1e9, "Tbyte": 1e12}
    total = 0.0
    try:
        with open(files[-1]) as f:
            for row in csv.reader(f):
                if row and row[0] in ("dram__bytes_read.sum", "dram__bytes_write.sum"):
                    total += sum(float(x) for x in row[2:]) * scale.get(row[1], 1.0)
    except (OSError, ValueError):
        return None, None
    return (total or None), os.path.relpath(files[-1], ROOT)


class ClockSampler:
    """SM clock and throttle reasons sampled DURING the timed region.

    The timed region is tens of milliseconds, so the sampler polls NVML directly (nvidia_ml_py) about
    once per millisecond from a thread; `nvidia-smi -lms` is only the fallback when NVML cannot be loaded.
    """
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index, uuid=None):
        self.index = index
        self.uuid = uuid
        self.rows = []       # nvidia-smi fallback lines
        self.samples = []    # (sm_mhz, reasons bitmask) from NVML
        self.proc = None
        self.nvml = None
        self.handle = None
        self.sm_max = None
        self.power = []
        self._stop = threading.Event()
        try:
            import pynvml
            pynvml.nvmlInit()
            h = None
            if uuid:
                try:
                    h = pynvml.nvmlDeviceGetHandleByUUID(uuid if uuid.startswith("GPU-") else "GPU-" + uuid)
                except Exception:  # noqa: BLE001
                    h = None
            if h is None:
                h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.sm_max = float(pynvml.nvmlDeviceGetMaxClockInfo(h, pynvml.NVML_CLOCK_SM))
            self.nvml, self.handle = pynvml, h
        except Exception:  # noqa: BLE001
            self.nvml = None

    def _poll(self):
        nv, h = self.nvml, self.handle
        while not self._stop.is_set():
            try:
                mhz = nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)
                try:
                    rs = nv.nvmlDeviceGetCurrentClocksEventReasons(h)
                except Exception:  # noqa: BLE001
                    rs = nv.nvmlDeviceGetCurrentClocksThrottleReasons(h)
                self.samples.append((float(mhz), int(rs)))
                if len(self.samples) % 16 == 1:
                    self.power.append(nv.nvmlDeviceGetPowerUsage(h) / 1000.0)
            except Exception:  # noqa: BLE001
                pass
            time.sleep(0.001)

    def start(self):
        if self.nvml:
            self.t = threading.Thread(target=self._poll, daemon=True)
            self.t.start()
            return
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except OSError:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if self.nvml:
            self._stop.set()
            self.t.join(timeout=2)
            nv = self.nvml
            names = (("hw_slowdown", "nvmlClocksEventReasonHwSlowdown", 0x8),
                     ("hw_thermal_slowdown", "nvmlClocksEventReasonHwThermalSlowdown", 0x40),
                     ("sw_thermal_slowdown", "nvmlClocksEventReasonSwThermalSlowdown", 0x20),
                     ("sw_power_cap", "nvmlClocksEventReasonSwPowerCap", 0x4))
            reasons = set()
            for mhz, rs in self.samples:
                for name, attr, dflt in names:
                    if rs & int(getattr(nv, attr, dflt)):
                        reasons.add(name)
            sm = [s[0] for s in self.samples]
            return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": self.sm_max, "samples": len(sm),
                    "reasons": sorted(reasons), "power_w_max": max(self.power) if self.power else None,
                    "source": "nvml"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "samples": 0, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons), "source": "nvidia-smi"}


def bind_near_gpu(local, ngpus):
    """Pin this process (and so the pages its pinned host buffers are first touched on) to the NUMA node of its GPU.
    With every rank left on node 0 the staging buffers of all GPUs share one socket's memory controllers (round 1:
    e2e 8.5 -> 19.5 TFLOP/s from 1 to 8 GPUs).  The node comes from sysfs; when the platform does not report one, the
    GPUs are spread evenly over the nodes in index order."""
    try:
        import torch
        nodes = sorted(int(d[4:]) for d in os.listdir("/sys/devices/system/node") if d.startswith("node") and d[4:].isdigit())
        if len(nodes) < 2:
            return {"node": nodes[0] if nodes else 0, "source": "single node"}
        p = torch.cuda.get_device_properties(local)
        node, src = -1, "sysfs"
        try:
            path = f"/sys/bus/pci/devices/{p.pci_domain_id:04x}:{p.pci_bus_id:02x}:{p.pci_device_id:02x}.0/numa_node"
            node = int(open(path).read().strip())
        except Exception:  # noqa: BLE001
            node = -1
        if node not in nodes:
            node, src = nodes[min(len(nodes) - 1, local * len(nodes) // max(ngpus, 1))], "even spread (no node in sysfs)"
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        allowed = cpus & os.sched_getaffinity(0)
        if allowed:
            os.sched_setaffinity(0, allowed)
        return {"node": node, "source": src, "cpus": len(allowed)}
    except Exception as e:  # noqa: BLE001
        return {"node": None, "source": f"not bound: {e}"[:120]}


def layer_table(spfy, csv, batch):
    shapes = spfy.shapes.read_shapes(csv)
    return [spfy.shapes.to_gemm(s, "weights", batch) for s in shapes]


# ------------------------------------------------------------------------------ CPU baseline
_CPU_INPUTS = {}


def cpu_baseline(spfy, orc, gemms, dtype_code, seconds_target=20.0, ncols=8192):
    """The oracle port (fp32 accumulate over the CANONICAL compressed operand, OpenMP over rows) on a
    bounded sample of the same workload: every layer of the table, first `ncols` columns of N.
    Inputs are generated once per unique shape (outside the timed regions) and reused by later calls."""
    import numpy as np
    flops = 0.0
    t_total = 0.0
    done = 0
    for g in gemms:
        n = min(ncols, g.N)
        key = (dtype_code, g.M, g.K, n)
        if key not in _CPU_INPUTS:
            rng = np.random.default_rng(0x5EED + g.M * 7 + g.K)
            _CPU_INPUTS[key] = (orc.from_f32(dtype_code, rng.uniform(-1, 1, (g.M, g.K)).astype(np.float32)),
                                orc.from_f32(dtype_code, rng.uniform(-1, 1, (g.K, n)).astype(np.float32)))
        a_bits, b_bits = _CPU_INPUTS[key]
        t0 = time.perf_counter()
        pr = orc.prune24_strip(dtype_code, a_bits, want_mask=False)
        orc.spmma_compressed_f32(dtype_code, pr["vals"], pr["meta"], g.M, g.K, b_bits)
        t_total += time.perf_counter() - t0
        flops += 2.0 * g.M * n * g.K
        done += 1
        if t_total > seconds_target:
            break
    return {"value": flops / t_total / 1e12, "unit": UNIT, "cores": orc.num_threads(), "kind": "port", "seconds": t_total,
            "sample": f"prune24+spmma of the first {done} of {len(gemms)} layers, first {ncols} columns of N each, "
                      f"{t_total:.1f} s of host time (oracle/spfy_oracle.cpp, OpenMP, fp32 accumulate)"}


def cusparselt_comparator(csv, batch):
    exe = os.path.join(ROOT, "oracle", "_ref", "cusparselt_ref")
    if not os.path.exists(exe):
        return None
    try:
        out = subprocess.run([exe, "sweep", os.path.join(ROOT, "datasets", csv), str(batch)], capture_output=True,
                             text=True, timeout=600)
        for line in out.stdout.splitlines()[::-1]:
            if line.startswith("{"):
                return json.loads(line)
        return {"error": (out.stderr or out.stdout)[-300:]}
    except Exception as e:  # noqa: BLE001
        return {"error": str(e)[:300]}


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    # the reference arm runs none of the product: the shape table is loaded by path (not through the package, which
    # would map libsparsifyme_b200.so into this process), the arithmetic is the oracle port on ALL host cores
    # (torchrun exports OMP_NUM_THREADS=1 to its workers; rank 0 is the only one that works here)
    class _Pkg:
        shapes = ge._load_by_path("spfy_shapes_only", os.path.join(ge.PKG_DIR, "shapes.py"))
    spfy = _Pkg
    orc = ge.load_oracle()
    orc.set_num_threads(len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1))
    gemms = layer_table(spfy, args.csv, args.batch)
    dt = 0 if args.dtype == "fp16" else 1
    vals, secs, best = [], [], None
    for i in range(args.warmup + args.steps):
        # the whole run stays within a couple of minutes whatever --steps / --warmup the driver passes
        budget = min(5.0, max(0.2, 90.0 / (args.warmup + args.steps)))
        r = cpu_baseline(spfy, orc, gemms, dt, seconds_target=budget, ncols=4096)
        if i >= args.warmup:
            vals.append(r["value"])
            secs.append(r["seconds"])
            best = r
    v = statistics.mean(vals)
    flops_step = sum(spfy.shapes.spmma_flops(g) for g in gemms)
    step_ms = statistics.mean(secs) * 1e3  # what one step of this arm really took: the bounded sample
    line = {"impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": step_ms, "full_workload_ms_extrapolated": flops_step / (v * 1e12) * 1e3,
            "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f16" if dt == 0 else "bf16", "data": "synthetic",
            "config": config_dict(args, len(gemms)),
            "cpu_baseline": dict(best, value=v),
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "gpu_launches": 0,
            "note": "the reference has no CPU path (SURVEY.md 0.3): this is the oracle port of the same math on the host "
                    "cores, each step a bounded sample of the workload (value = its FLOPs / its time; ms_per_step = its time; the full "
                    "workload at that rate would take full_workload_ms_extrapolated)"}
    cmp_ = cusparselt_comparator(args.csv, args.batch)
    if cmp_ is not None:
        line["cusparselt"] = cmp_
    print(json.dumps(line))
    return 0


def config_dict(args, nlayers, launches=None):
    how = f"one plan, {launches} persistent launches" if launches else "one plan of persistent launches"
    return {"workload": f"datasets/{args.csv}: all {nlayers} layers, weights orientation (M=C_out, K=C_in*kh*kw, "
                        f"N=H*W*b), b={args.batch} images per GPU, 2:4 magnitude prune+compress (one batched launch) "
                        f"+ spmma of every layer ({how})",
            "csv": args.csv, "batch_per_gpu": args.batch, "global_batch": args.batch * args.gpus,
            "l2_policy": "inputs larger than L2 (7.4 GB of distinct B/D buffers per step vs 126 MB L2)",
            "parallelism": f"batch-sharded x{args.gpus}, no data-path collective"}


# ------------------------------------------------------------------------------ unstructured workload
def run_coo(args):
    """BASELINE.json configs[2]/[3]: magnitude-threshold prune of every layer's weights to COO, then the batched COO
    SpMM of every layer (A = W shared by the batch, B_b = [K x H*W] column-major per image, fp32 -- the operand
    types of spmm.hxx:165-180).  The batch of `--batch` images is sharded on image boundaries across the ranks
    (STRONG scaling: the job is fixed), no data-path collective.  One step = threshold->COO + SpMM of all layers."""
    import collections
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (sparsify.me_b200 has no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    json_out = claim_stdout() if world > 1 else sys.stdout
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    spfy = ge.load_package()
    csv = args.csv if args.csv != "resnet50.csv" else "resnet101.csv"
    shapes = spfy.shapes.read_shapes(csv)
    lo, hi = spfy.multigpu.shard_batch(args.batch, world, rank)
    nb = hi - lo
    hbm_peak, _, _, peak_src = read_peaks()
    cnt = collections.Counter((s.n, s.k, s.m) for s in shapes)  # (M, K, n = H*W) -> layers of that shape
    gen = torch.Generator(device=dev)
    gen.manual_seed(0x5EED)  # same weights on every rank (replicated, pruned redundantly)
    gen_b = torch.Generator(device=dev)
    gen_b.manual_seed(0xB0 + rank)  # every rank its own images
    work = []
    for (M, K, n), c in cnt.items():
        w = torch.rand(M, K, device=dev, generator=gen) * 2 - 1
        kth = max(1, min(M * K, int(args.sparsity * M * K)))
        thr = float(torch.kthvalue(w.abs().flatten(), kth).values)
        per_set = 4 * (K + M) * n * max(nb, 1)
        nsets = max(1, min(4, -(-300_000_000 // max(per_set, 1))))  # rotate so that nothing is served from L2
        bs = [torch.rand(max(nb, 1), n, K, device=dev, generator=gen_b) * 2 - 1 for _ in range(nsets)]
        cs = [torch.empty(max(nb, 1), n, M, device=dev) for _ in range(nsets)]
        nnz = int((w.abs() > thr).sum())
        work.append(dict(M=M, K=K, n=n, count=c, w=w, thr=thr, b=bs, c=cs, nnz=nnz, cap=nnz + 16))

    def prune_step():
        """threshold -> COO of every layer (weights are replicated: every rank prunes all of them)"""
        coos = []
        for x in work:
            for rep in range(x["count"]):
                coos.append(spfy.threshold_to_coo(x["w"], x["thr"], capacity=x["cap"], sync=False))
        return coos

    def spmm_step(it, coos):
        fl = by = 0.0
        i = 0
        for x in work:
            for rep in range(x["count"]):
                ri, ci, va, _, rp = coos[i]  # no host read-back: the CSR entry point takes row_ptr from the device
                i += 1
                nnz = x["nnz"]
                if nb:
                    j = (it * x["count"] + rep) % len(x["b"])
                    spfy.batched.csr(x["M"], x["K"], x["n"], nb, rp, ci, va, x["b"][j], x["c"][j])
                fl += 2.0 * nnz * x["n"] * nb
                by += 12 * nnz + 4.0 * (x["K"] + x["M"]) * x["n"] * nb
        return fl, by

    for i in range(args.warmup):
        spmm_step(i, prune_step())
    torch.cuda.synchronize()
    steps = args.steps

    # The step is ~600 short launches with no host read-back anywhere, i.e. bound by how fast the host can
    # launch (and with eight ranks on one box, by the host cores they share): capture it once per operand
    # rotation in CUDA graphs -- one for the prune phase, one per rotation for the SpMM phase -- and replay.
    graphs = None
    import math
    period = 1
    for x in work:
        period = math.lcm(period, len(x["b"]))  # the operand set of a launch depends on the step modulo this
    launches_per_step = None
    if not args.no_graph:
        try:
            side = torch.cuda.Stream(dev)
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                l0 = spfy.launch_count()
                g_prune = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g_prune, stream=side):
                    coos_g = prune_step()
                g_spmm = []
                for it in range(period):
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g, stream=side):
                        fl, by = spmm_step(it, coos_g)
                    g_spmm.append(g)
            torch.cuda.current_stream().wait_stream(side)
            torch.cuda.synchronize()
            graphs = (g_prune, g_spmm)
        except Exception as e:  # noqa: BLE001 -- capture is an optimisation of the harness, not of the product
            print(f"bench.py: CUDA graph capture failed ({e}); timing eager launches", file=sys.stderr)
            graphs = None
            torch.cuda.synchronize()
    if graphs:  # launches of one eager step (replays do not pass through the library's counter)
        l0 = spfy.launch_count()
        spmm_step(0, prune_step())
        torch.cuda.synchronize()
        launches_per_step = spfy.launch_count() - l0
        for it in range(period):  # warm the replays
            graphs[0].replay()
            graphs[1][it].replay()
        torch.cuda.synchronize()
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(steps)]
    launches0 = spfy.launch_count()
    sampler = ClockSampler(local, str(torch.cuda.get_device_properties(local).uuid))
    if world > 1:
        dist.barrier()
    torch.cuda.synchronize()
    if rank == 0:
        sampler.start()
    for i in range(steps):
        ev[i][0].record()
        if graphs:
            graphs[0].replay()
        else:
            coos = prune_step()
        ev[i][1].record()
        if graphs:
            graphs[1][i % period].replay()
        else:
            fl, by = spmm_step(i, coos)
        ev[i][2].record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    clocks = sampler.stop() if rank == 0 else None
    prune_ms = sum(e[0].elapsed_time(e[1]) for e in ev) / steps
    spmm_ms = sum(e[1].elapsed_time(e[2]) for e in ev) / steps
    t = torch.tensor([ev[0][0].elapsed_time(ev[-1][2]) / steps, prune_ms, spmm_ms, fl, by], dtype=torch.float64, device=dev)
    if world > 1:
        tmax = t.clone()
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        t[:3] = tmax[:3]
    ms, prune_ms, spmm_ms, fl_all, by_all = (float(x) for x in t.tolist())
    if args.dump_outputs and rank == 0:
        # the last step: every layer's C (this rank's images; a layer's operand set depends on the step), and the COO /
        # CSR weights of every shape (the layers of one shape share them)
        arrays, coos, i = {}, (coos_g if graphs else coos), 0
        for xi, x in enumerate(work):
            ri, ci, va, nnz, rp = coos[i]
            n = int(nnz.item())
            arrays.update({f"coo_rows_{xi:03d}": ri[:n], f"coo_cols_{xi:03d}": ci[:n], f"coo_vals_{xi:03d}": va[:n],
                           f"csr_row_ptr_{xi:03d}": rp})
            for rep in range(x["count"]):
                if nb:
                    arrays[f"c_{i:03d}"] = x["c"][((steps - 1) * x["count"] + rep) % len(x["c"])]
                i += 1
        dump_outputs(args.dump_outputs, arrays)
    if rank == 0:
        print(json.dumps({
            "metric": "batched COO SpMM TFLOP/s (2*nnz*N) over a ResNet table, threshold prune included", "value": fl_all / ms / 1e9,
            "unit": UNIT, "n_gpus": world, "steps": steps, "warmup": args.warmup, "ms_per_step": ms,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"datasets/{csv}: all {len(shapes)} layers, weights kept above the {args.sparsity:.2f} magnitude "
                                   f"quantile -> COO, batched COO SpMM over {args.batch} images sharded across {world} rank(s)",
                       "csv": csv, "global_batch": args.batch, "sparsity": args.sparsity,
                       "l2_policy": "operand sets rotated so that a launch never finds B in L2",
                       "parallelism": f"batch-sharded x{world}, no data-path collective"},
            "clocks": clocks,
            "gpu_launches": launches_per_step * steps if graphs else spfy.launch_count() - launches0,
            "launch_mode": ("CUDA graphs: one for the prune phase, one per operand rotation for the SpMM phase; gpu_launches = "
                            "kernel launches of one eager step x steps") if graphs else "eager",
            "phases": {"threshold_to_coo_ms": prune_ms, "spmm_ms": spmm_ms, "spmm_tflops": fl_all / spmm_ms / 1e9,
                       "note": "the threshold prune is replicated on every rank; no host read-back (CSR row_ptr stays on the device)"},
            "roofline": {"bound": "hbm", "kernel": "coo_scatter_kernel + tcgemm_ts_kernel (3xTF32, A in tensor memory; k = 147 on a padded "
                                                   "copy of B)", "achieved": by_all / spmm_ms / 1e6, "peak": hbm_peak * world,
                         "unit": "GB/s", "frac": by_all / spmm_ms / 1e6 / (hbm_peak * world), "traffic": None,
                         "peak_source": peak_src,
                         "note": "bytes are the SPARSE algorithmic ones (12 nnz + 4KN + 4MN per batch); the dense contraction is "
                                 "bound by the traffic into the SMs and the 3x tensor work, not by HBM (DESIGN.md 4)"}}),
              file=json_out, flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


# ------------------------------------------------------------------------------ our arm
# ------------------------------------------------------------------------------ strong scaling with the output gather
def run_strong(args):
    """BASELINE.json configs[4]: the 2:4 spmma sweep over datasets/resnet152.csv at a FIXED global batch (256 images),
    N-sharded on image boundaries across the ranks (rank r owns b/g images of every layer = columns [r*N/g, (r+1)*N/g)
    of B and D; weights replicated and pruned redundantly), followed by the path's only collective: the gather of every
    layer's output onto every rank (north_star: "NCCL used only to gather outputs").

    Each rank's GEMMs write D_r [M x N/g] straight into slab r of a per-chunk gather arena; the arena's other slabs are
    filled by ONE in-place ncclAllGather per chunk (spfy_mg_allgather: layout [g][M][N/g] per layer, no transpose, no
    copy) on a second stream, so the gather of chunk c runs under the GEMMs of chunk c+1.  Reported: compute-only,
    gather-only and the overlapped whole; `value` is the whole job (compute + gather)."""
    import torch
    import torch.distributed as dist
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (sparsify.me_b200 has no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    json_out = claim_stdout() if world > 1 else sys.stdout
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    spfy = ge.load_package()
    csv = args.csv if args.csv != "resnet50.csv" else "resnet152.csv"
    gbatch = args.batch if args.batch != 32 else 256
    lo, hi = spfy.multigpu.shard_batch(gbatch, world, rank)
    nb = hi - lo
    if gbatch % world:
        raise SystemExit("bench.py --strong: the global batch must be divisible by the number of GPUs (equal slabs)")
    tdt = torch.float16 if args.dtype == "fp16" else torch.bfloat16
    shapes = spfy.shapes.read_shapes(csv)
    gemms = [spfy.shapes.to_gemm(s, "weights", nb) for s in shapes]          # this rank's shard
    gemms_global = [spfy.shapes.to_gemm(s, "weights", gbatch) for s in shapes]
    hbm_peak, _, tc_sust, peak_src = read_peaks()
    need = sum((g.K * g.N + (2 if world > 1 and not args.no_fused else 1) * world * g.M * g.N) * 2 for g in gemms)
    if need > 150e9:
        raise SystemExit(f"bench.py --strong: {need/1e9:.0f} GB per GPU do not fit; use more GPUs")

    nchunks = max(1, min(args.chunks, len(gemms)))
    bounds = [len(gemms) * c // nchunks for c in range(nchunks + 1)]
    gen_w = torch.Generator(device=dev)
    gen_w.manual_seed(0x5EED)          # same weights on every rank
    gen_b = torch.Generator(device=dev)
    gen_b.manual_seed(0xB0 + rank)     # every rank its own images
    layers, arenas, plans = [], [], []
    for c in range(nchunks):
        idx = range(bounds[c], bounds[c + 1])
        elems = sum(gemms[i].M * gemms[i].N for i in idx)
        elems = -(-elems // 64) * 64
        arena = torch.zeros(world, elems, dtype=tdt, device=dev)
        arenas.append(arena)
        off, probs = 0, []
        for i in idx:
            g = gemms[i]
            w = (torch.rand(g.M, g.K, device=dev, generator=gen_w) * 2 - 1).to(tdt)
            b = (torch.rand(g.K, g.N, device=dev, generator=gen_b) * 2 - 1).to(tdt)
            d = arena[rank, off: off + g.M * g.N].view(g.M, g.N)
            off += g.M * g.N
            comp = spfy.alloc_compressed(tdt, g.M, g.K, dev)
            comp.vals.zero_()  # padding bytes prune24 leaves alone are the same in every run (--dump-outputs)
            comp.meta.zero_()
            layers.append((g, w, b, d, comp, c, off - g.M * g.N))
            probs.append(dict(comp=comp, b=b, out=d))
        plans.append(spfy.SpmmaPlan(probs))
    gather = spfy.multigpu.OutputGather() if world > 1 else None
    s_comm = torch.cuda.Stream(dev)
    # the fused gather: a second set of arenas every rank can store into (peer mappings) and plans whose epilogue
    # writes every D tile to slab `rank` of ALL of them -- the GEMM is the all-gather, no collective follows
    fused = world > 1 and not args.no_fused
    peer_arenas, fplans = [], []
    if fused:
        for c in range(nchunks):
            pa = spfy.multigpu.PeerArena(arenas[c][0].numel() * arenas[c].element_size())
            peer_arenas.append(pa)
            mine = pa.local[rank].view(tdt)
            probs = []
            for (g, w, b, d, comp, cc, off) in layers:
                if cc == c:
                    probs.append(dict(comp=comp, b=b, out=mine[off: off + g.M * g.N].view(g.M, g.N),
                                      replicas=pa.replica_addresses(off * arenas[c].element_size())))
            fplans.append(spfy.SpmmaPlan(probs))

    def prune_all():
        spfy.prune24_batched([l[1] for l in layers], [l[4] for l in layers])

    def step(do_compute, do_gather):
        cur = torch.cuda.current_stream()
        if do_compute:
            prune_all()
        for c in range(nchunks):
            if do_compute:
                plans[c].run()
            if do_gather and gather is not None:
                s_comm.wait_event(cur.record_event())
                gather.allgather(arenas[c], stream=s_comm)
        if do_gather:
            cur.wait_event(s_comm.record_event())

    def step_fused(*_):
        prune_all()
        for c in range(nchunks):
            fplans[c].run()
        peer_arenas[0].barrier()  # 4-byte all-reduce on the compute stream: every rank's stores have landed

    def timed(do_compute, do_gather, steps, step=step):
        for _ in range(max(1, args.warmup // 2)):
            step(do_compute, do_gather)
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            step(do_compute, do_gather)
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / steps], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    for _ in range(args.warmup):
        step(True, True)
    torch.cuda.synchronize()
    sampler = ClockSampler(local, str(torch.cuda.get_device_properties(local).uuid))
    launches0 = spfy.launch_count()
    if rank == 0:
        sampler.start()
    both_ms = timed(True, True, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    launches = (spfy.launch_count() - launches0) // (args.steps + max(1, args.warmup // 2))
    compute_ms = timed(True, False, args.steps)
    gather_ms = timed(False, True, args.steps) if world > 1 else 0.0
    fused_ms = timed(True, True, args.steps, step=step_fused) if fused else None

    # ---- the gathered slabs are what the other ranks computed: per-rank checksums travel by all_gather and are compared
    #      with the sums of the slabs received (and the local slab against a torch fp32 matmul, first and last layer)
    step(True, True)
    torch.cuda.synchronize()
    def slab_sum(t, piece=1 << 26):  # fp64 sum of a 16-bit slab without materialising a wide copy of it
        flat = t.reshape(-1)
        return torch.stack([flat[i: i + piece].double().sum() for i in range(0, flat.numel(), piece)]).sum()

    sums = torch.stack([torch.stack([slab_sum(a[r]) for r in range(world)]) for a in arenas])  # [chunks, world] as seen here
    mine = sums[:, rank].clone()                                                                # [chunks] my own slab
    ok_gather = True
    if world > 1:
        allmine = [torch.empty_like(mine) for _ in range(world)]
        dist.all_gather(allmine, mine)
        for r in range(world):
            ok_gather &= bool(torch.allclose(sums[:, r], allmine[r], rtol=1e-9, atol=1e-6))
    worst = 0.0
    for i in (0, len(layers) - 1):
        g, w, b, d, comp, c, off = layers[i]
        pruned = torch.empty_like(w)
        spfy.prune24(w, out_dense=pruned, compress=False)
        n1 = min(g.N, 50176)
        want = pruned.float() @ b[:, :n1].float()
        scale = torch.clamp(want.abs(), min=1e-2 * float(want.abs().max()))
        worst = max(worst, float(((d[:, :n1].float() - want).abs() / scale).max()))
    ok_fused = True
    if fused:
        for pa in peer_arenas:
            pa.local.zero_()
        torch.cuda.synchronize()
        dist.barrier()
        step_fused()
        torch.cuda.synchronize()
        for c in range(nchunks):  # bit-identical to GEMM + ncclAllGather
            used = sum(l[0].M * l[0].N for l in layers if l[5] == c)  # (the alignment tail of an arena is never written)
            ok_fused &= bool(torch.equal(peer_arenas[c].local.view(tdt)[:, :used], arenas[c][:, :used]))
    ok_gather = ok_gather and ok_fused
    flag = torch.tensor([1.0 if (ok_gather and worst <= 1e-2) else 0.0], device=dev)
    if world > 1:
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
    if float(flag.item()) != 1.0:
        raise SystemExit(f"bench.py --strong: verification failed on some rank (gather ok {ok_gather}, max rel err {worst:.3e})")
    if args.dump_outputs and rank == 0:
        # the step above is the timed step once more (compute + gather): every layer's output as gathered onto this rank,
        # [world][M][N / world], and the compressed weights
        arrays = {}
        for i, (g, w, b, d, comp, c, off) in enumerate(layers):
            arrays[f"d_{i:03d}"] = arenas[c][:, off: off + g.M * g.N]
            arrays.update(compressed_arrays(i, comp))
        dump_outputs(args.dump_outputs, arrays)

    if rank == 0:
        flops = sum(spfy.shapes.spmma_flops(g) for g in gemms_global)
        bytes_rank = sum(spfy.shapes.spmma_bytes(g) for g in gemms)
        recv = sum(a[0].numel() * a.element_size() for a in arenas) * (world - 1)
        best_ms = min(both_ms, fused_ms) if fused else both_ms
        line = {
            "metric": METRIC, "value": flops / (best_ms * 1e-3) / 1e12, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": best_ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
            "dtype": "f16" if args.dtype == "fp16" else "bf16", "data": "synthetic",
            "config": {"workload": f"datasets/{csv}: all {len(gemms)} layers, 2:4 prune+compress + spmma at GLOBAL batch {gbatch} "
                                   f"(BASELINE.json configs[4]), N-sharded on image boundaries: {nb} images per GPU; every layer's "
                                   f"output gathered onto every GPU ([g][M][N/g], in-place ncclAllGather per chunk of layers, "
                                   f"{nchunks} chunks, overlapped with the next chunk's GEMMs)",
                       "csv": csv, "global_batch": gbatch, "batch_per_gpu": nb, "chunks": nchunks,
                       "l2_policy": "inputs larger than L2", "parallelism": f"N-sharded x{world} + output all-gather"},
            "clocks": clocks, "gpu_launches": launches,
            "compute_only": {"ms_per_step": compute_ms, "tflops": flops / (compute_ms * 1e-3) / 1e12,
                             "hbm_frac": bytes_rank / (compute_ms * 1e-3) / 1e9 / hbm_peak},
            "gather_only": {"ms_per_step": gather_ms, "bytes_received_per_rank": recv,
                            "algbw_GBs_per_rank": recv / (gather_ms * 1e-3) / 1e9 if gather_ms else None,
                            "collective": "ncclAllGather via spfy_mg_allgather (NCCL loaded at run time), in place"},
            "compute_plus_gather": {"ms_per_step": both_ms, "overlap_saved_ms": compute_ms + gather_ms - both_ms},
            "fused_gather": None if not fused else {
                "ms_per_step": fused_ms, "tflops": flops / (fused_ms * 1e-3) / 1e12,
                "bytes_stored_to_peers_per_rank": recv, "nvlink_out_GBs_per_rank": recv / (fused_ms * 1e-3) / 1e9,
                "how": "spfy_spmma_plan_create_replicated: the epilogue's TMA store of every D tile goes to slab `rank` of "
                       "every GPU's arena (cudaIpc peer mappings over NVLink); completion = one 4-byte all-reduce",
                "bit_identical_to_nccl_gather": ok_fused},
            "value_is": "fused_gather" if fused and fused_ms <= both_ms else "compute_plus_gather",
            "verified": {"gather_checksums_match": ok_gather, "max_rel_err_local": worst, "tolerance": 1e-2},
        }
        print(json.dumps(line), file=json_out, flush=True)
    for pl in fplans:
        pl.close()
    for pa in peer_arenas:
        pa.close()
    if gather is not None:
        gather.close()
    if world > 1:
        dist.destroy_process_group()
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--csv", default="resnet50.csv")
    ap.add_argument("--batch", type=int, default=32)
    ap.add_argument("--dtype", default="fp16", choices=["fp16", "bf16"])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="coo workload: eager launches instead of CUDA graph replays")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-implicit", action="store_true", help="skip the implicit-GEMM variants (plan and e2e)")
    ap.add_argument("--no-prune-large", action="store_true", help="skip the large-matrix prune24 measurement")
    ap.add_argument("--e2e-steps", type=int, default=3)
    ap.add_argument("--per-layer", action="store_true", help="also print a per-layer table to stderr")
    ap.add_argument("--workload", default="spmma", choices=["spmma", "coo"],
                    help="spmma: the headline (BASELINE.json configs[1]); coo: unstructured threshold prune + batched COO "
                         "SpMM over a table, batch-sharded across ranks (configs[2]/[3])")
    ap.add_argument("--sparsity", type=float, default=0.9, help="--workload coo: fraction of the weights dropped")
    ap.add_argument("--strong", action="store_true",
                    help="BASELINE.json configs[4]: fixed global batch (256) over resnet152.csv, N-sharded across the ranks, "
                         "outputs all-gathered onto every rank (compute-only / gather-only / overlapped are all reported)")
    ap.add_argument("--chunks", type=int, default=6, help="--strong: groups of layers per gather")
    ap.add_argument("--no-fused", action="store_true", help="--strong: skip the fused gather (epilogue stores to peer memory)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write what the last timed step computed (every layer's output and its compressed or COO weights) "
                         "to DIR/<name>.npy; not with --impl reference")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs: the reference arm times a bounded CPU sample, not the whole step")
    if args.impl == "reference":
        return run_reference(args)
    if args.workload == "coo":
        return run_coo(args)
    if args.strong:
        return run_strong(args)

    import ctypes
    import numpy as np
    import torch
    import torch.distributed as dist

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (sparsify.me_b200 has no CPU fallback)")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    json_out = claim_stdout() if world > 1 else sys.stdout
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    spfy = ge.load_package()
    tdt = torch.float16 if args.dtype == "fp16" else torch.bfloat16
    dcode = spfy.F16 if args.dtype == "fp16" else spfy.BF16
    gemms = layer_table(spfy, args.csv, args.batch)
    hbm_peak, tc_burst, tc_sust, peak_src = read_peaks()

    # ---- resident synthetic inputs: per layer W [M,K], B [K,N], D [M,N], compressed operand ----
    gen = torch.Generator(device=dev)
    gen.manual_seed(0x5EED + rank)
    layers = []
    for g in gemms:
        w = (torch.rand(g.M, g.K, device=dev, generator=gen) * 2 - 1).to(tdt)
        b = (torch.rand(g.K, g.N, device=dev, generator=gen) * 2 - 1).to(tdt)
        d = torch.empty(g.M, g.N, device=dev, dtype=tdt)
        vb, mb = spfy.compressed_bytes(tdt, g.M, g.K)
        # zero-filled, so that bytes of the padded tiles that prune24 leaves alone are the same in every run (--dump-outputs)
        comp = spfy.Compressed24(torch.zeros(vb, dtype=torch.uint8, device=dev),
                                 torch.zeros(mb, dtype=torch.uint8, device=dev), g.M, g.K, tdt, spfy.LAYOUT_SM100)
        layers.append((g, w, b, d, comp))

    def prune_all():
        spfy.prune24_batched([l[1] for l in layers], [l[4] for l in layers])

    plan = spfy.SpmmaPlan([dict(comp=comp, b=b, out=d) for g, w, b, d, comp in layers])

    def spmma_all():
        plan.run()

    flops_step = sum(spfy.shapes.spmma_flops(g) for g in gemms)
    spmma_bytes_step = sum(spfy.shapes.spmma_bytes(g) for g in gemms)
    prune_bytes_step = sum(spfy.shapes.prune24_bytes(g.M, g.K) for g in gemms)

    def barrier():
        if world > 1:
            dist.barrier()

    for _ in range(args.warmup):
        prune_all()
        spmma_all()
    torch.cuda.synchronize()
    sampler = ClockSampler(local, str(torch.cuda.get_device_properties(local).uuid))
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(args.steps)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    launches0 = spfy.launch_count()
    barrier()
    torch.cuda.synchronize()
    if rank == 0:
        sampler.start()
    e0.record()
    for s in range(args.steps):
        ev[s][0].record()
        prune_all()
        ev[s][1].record()
        spmma_all()
        ev[s][2].record()
    e1.record()
    torch.cuda.synchronize()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    launches = spfy.launch_count() - launches0
    total_ms = e0.elapsed_time(e1)
    prune_ms = sum(ev[s][0].elapsed_time(ev[s][1]) for s in range(args.steps)) / args.steps
    spmma_ms = sum(ev[s][1].elapsed_time(ev[s][2]) for s in range(args.steps)) / args.steps
    t = torch.tensor([total_ms, prune_ms, spmma_ms], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    total_ms, prune_ms, spmma_ms = (float(x) for x in t.tolist())
    ms_per_step = total_ms / args.steps
    value = flops_step * world / (ms_per_step * 1e-3) / 1e12
    if args.dump_outputs and rank == 0:
        arrays = {}
        for i, (g, w, b, d, comp) in enumerate(layers):
            arrays[f"d_{i:03d}"] = d
            arrays.update(compressed_arrays(i, comp))
        dump_outputs(args.dump_outputs, arrays)

    # ---- the timed outputs are checked, not just produced: D of the last timed step against a torch fp32 matmul of
    #      the pruned weights (decoded by the same prune kernel family), first / middle / last / largest-K layers, every
    #      column (outside the timed region; tests/test_gpu_fullsize.py checks all layers against the CPU oracle too)
    verified = None
    if rank == 0:
        picks = sorted({0, len(layers) // 2, len(layers) - 1, max(range(len(layers)), key=lambda i: layers[i][0].K)})
        worst = 0.0
        for i in picks:
            g, w, b, d, comp = layers[i]
            pruned = torch.empty_like(w)
            spfy.prune24(w, out_dense=pruned, compress=False)
            pf = pruned.float()
            for c0 in range(0, g.N, 50176):
                want = pf @ b[:, c0:c0 + 50176].float()
                scale = torch.clamp(want.abs(), min=1e-2 * float(want.abs().max()))
                worst = max(worst, float(((d[:, c0:c0 + 50176].float() - want).abs() / scale).max()))
            del pruned, pf
        verified = {"layers": picks, "columns": "all", "max_rel_err": worst, "tolerance": 1e-2, "ok": worst <= 1e-2,
                    "against": "torch fp32 matmul of the 2:4-pruned weights on the same GPU"}
        if not verified["ok"]:
            raise SystemExit(f"bench.py: timed outputs are wrong (max relative error {worst:.3e} > 1e-2)")

    # ---- the same table with the 3 x 3 layers as implicit GEMMs (SURVEY.md 8f N2): ONE plan in which those layers read
    #      their NHWC activations through TMA im2col instead of the unfolded K x N operand (spfy_spmma_plan_create_conv).
    #      Same FLOPs, same outputs (checked below); reported beside the headline, which multiplies the CSV's matrices.
    conv_geom = {}
    for g in gemms:
        hw = g.N // args.batch
        ho = math.isqrt(hw)
        if g.K % 9 == 0 and (g.K // 9) % 64 == 0 and ho * ho == hw and hw * args.batch == g.N:
            conv_geom[g] = (ho, g.K // 9)  # 3 x 3, pad 1, stride 1 (the CSV does not record strides)
    xdev, xl, implicit_plan = {}, {}, None
    if conv_geom and not args.no_implicit:
        for g, (ho, cin) in conv_geom.items():
            xdev[g] = (torch.rand(args.batch, ho, ho, cin, device=dev, generator=gen) * 2 - 1).to(tdt)
        xl = {id(l[3]): xdev[l[0]].clone() for l in layers if l[0] in conv_geom}  # one x per layer: nothing is shared through L2
        plan_i = spfy.SpmmaPlan([dict(comp=comp, b=xl[id(d)], out=d, conv=(3, 3, 1, 1)) if g in conv_geom else
                                 dict(comp=comp, b=b, out=d) for g, w, b, d, comp in layers])
        for _ in range(args.warmup):
            prune_all()
            plan_i.run()
        barrier()
        torch.cuda.synchronize()
        evi = [[torch.cuda.Event(enable_timing=True) for _ in range(2)] for _ in range(args.steps)]
        e0.record()
        for s_ in range(args.steps):
            prune_all()
            evi[s_][0].record()
            plan_i.run()
            evi[s_][1].record()
        e1.record()
        torch.cuda.synchronize()
        ti = torch.tensor([e0.elapsed_time(e1) / args.steps, sum(a.elapsed_time(b_) for a, b_ in evi) / args.steps],
                          dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(ti, op=dist.ReduceOp.MAX)
        step_i, spmma_i = (float(v) for v in ti.tolist())
        if rank == 0:
            import torch.nn.functional as F
            same = True
            for g0 in sorted(conv_geom, key=lambda q: q.K)[-2:]:  # the two largest-K conv shapes: every column, bit for bit
                li = next(i for i, l in enumerate(layers) if l[0] == g0)
                _, _, _, d0, comp0 = layers[li]
                ho, cin = conv_geom[g0]
                cols = F.unfold(xl[id(d0)].permute(0, 3, 1, 2).float(), 3, padding=1).view(args.batch, cin, 9, ho * ho)
                bx = cols.permute(2, 1, 0, 3).reshape(g0.K, g0.N).to(tdt).contiguous()
                del cols
                same = same and bool(torch.equal(spfy.spmma_compressed(comp0, bx), d0))
                del bx
            if not same:
                raise SystemExit("bench.py: the implicit-GEMM plan's outputs differ from the explicit operand's")
            bytes_i = sum((spfy.shapes.spmma_bytes(g) - 2 * g.K * g.N + 2 * xdev[g].numel()) if g in conv_geom
                          else spfy.shapes.spmma_bytes(g) for g in gemms)
            implicit_plan = {
                "ms_per_step": step_i, "spmma_ms_per_step": spmma_i, "value": flops_step * world / (step_i * 1e-3) / 1e12, "unit": UNIT,
                "conv_layers": sum(1 for g in gemms if g in conv_geom), "launches_per_step": plan_i.launches,
                "algorithmic_bytes_per_step": bytes_i, "achieved_GBs": bytes_i / (spmma_i * 1e-3) / 1e9,
                "frac_of_hbm_on_its_own_bytes": bytes_i / (spmma_i * 1e-3) / 1e9 / hbm_peak,
                "explicit_spmma_ms_per_step": spmma_ms, "identical_to_explicit_operand": same,
                "note": "3 x 3 layers (pad 1, stride 1 assumed: the CSV has no strides) read NHWC activations through TMA im2col; "
                        "HBM bytes drop, the bytes entering the SMs do not (DESIGN.md 4), so the gain is bounded by the L2 -> SM path"}
        plan_i.close()

    # ---- end to end through the reference-shaped call with host buffers ----
    e2e = None
    if not args.no_e2e:
        numa = bind_near_gpu(local, torch.cuda.device_count())
        hostbuf = {}

        def pinned(key, shape):
            if key not in hostbuf:
                hostbuf[key] = torch.empty(shape, dtype=tdt).pin_memory()
            return hostbuf[key]

        for g, w, b, d, comp in layers:  # host images of the inputs, one per unique shape
            if ("w", g) not in hostbuf:
                pinned(("w", g), (g.M, g.K)).copy_(w)
                pinned(("b", g), (g.K, g.N)).copy_(b)
                pinned(("d", g), (g.M, g.N))
        h2d = sum((g.M * g.K + g.K * g.N) * 2 for g in gemms)
        d2h = sum(g.M * g.N * 2 for g in gemms)

        # three streams so that PCIe runs full duplex and the GPU works under the copies: layer i+1's
        # H2D and layer i-1's D2H overlap layer i's prune+compress+multiply
        s_in, s_run, s_out = torch.cuda.Stream(dev), torch.cuda.Stream(dev), torch.cuda.Stream(dev)

        # (spmma() synchronises on its event pairs like the reference's timer_t, so the copies of ALL layers are queued
        # first -- every layer has its own device buffers -- and the copy engine never waits for the host)
        def e2e_step():
            ready = []
            with torch.cuda.stream(s_in):
                for g, w, b, d, comp in layers:
                    w.copy_(hostbuf[("w", g)], non_blocking=True)
                    b.copy_(hostbuf[("b", g)], non_blocking=True)
                    ready.append(s_in.record_event())
            for (g, w, b, d, comp), rdy in zip(layers, ready):
                with torch.cuda.stream(s_run):
                    s_run.wait_event(rdy)
                    spfy.spmma(w, b, d, g.M, g.N, g.K, args.batch)
                    done = s_run.record_event()
                with torch.cuda.stream(s_out):
                    s_out.wait_event(done)
                    hostbuf[("d", g)].copy_(d, non_blocking=True)
            torch.cuda.synchronize()

        e2e_step()
        barrier()
        torch.cuda.synchronize()
        e0.record()
        for _ in range(args.e2e_steps):
            e2e_step()
        e1.record()
        torch.cuda.synchronize()
        te = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e_ms = float(te.item()) / args.e2e_steps
        e2e = {"value": flops_step * world / (e2e_ms * 1e-3) / 1e12, "unit": UNIT, "h2d_bytes_per_step": h2d,
               "d2h_bytes_per_step": d2h, "ms_per_step": e2e_ms, "steps": args.e2e_steps,
               "pcie_GBs_per_rank": {"h2d": h2d / (e2e_ms * 1e-3) / 1e9, "d2h": d2h / (e2e_ms * 1e-3) / 1e9},
               "host_numa": numa,
               "api": "spmma(A, B, C, m, n, k, b) per layer: pinned H2D of A and B, TILE prune in place (as spmma.hxx:86) + compress + "
                      "tcgen05 matmul, D2H of C; copy-in / compute / copy-out on three streams, the step's H2D copies queued ahead of the calls"}
        # ---- the same step with the bytes shrunk: the 3 x 3 layers' unfolded K x N operand (9 copies of every
        #      activation, datasets/get_shapes.py:29-41) never exists on the host either -- the NHWC activations travel and
        #      spfy_spmma_conv gathers the operand with TMA im2col (weights stored (kh, kw, c)-major, a layout chosen once
        #      at export).  Reported BESIDE e2e, not instead of it: the reference's call takes the unfolded matrix.
        if xl:
            for g in conv_geom:
                hostbuf[("x", g)] = torch.empty(xdev[g].shape, dtype=tdt).pin_memory()
                hostbuf[("x", g)].copy_(xdev[g])
            h2d_i = sum((g.M * g.K + (xdev[g].numel() if g in conv_geom else g.K * g.N)) * 2 for g in gemms)

            def e2e_implicit_step():
                ready = []
                with torch.cuda.stream(s_in):
                    for g, w, b, d, comp in layers:
                        w.copy_(hostbuf[("w", g)], non_blocking=True)
                        if g in conv_geom:
                            xl[id(d)].copy_(hostbuf[("x", g)], non_blocking=True)
                        else:
                            b.copy_(hostbuf[("b", g)], non_blocking=True)
                        ready.append(s_in.record_event())
                for (g, w, b, d, comp), rdy in zip(layers, ready):
                    with torch.cuda.stream(s_run):
                        s_run.wait_event(rdy)
                        if g in conv_geom:
                            spfy.prune24(w, inplace=True, out=comp, mode=spfy.PRUNE_TILE_MAG)
                            spfy.spmma_conv(comp, xl[id(d)], 3, 3, stride=1, pad=1, out=d)
                        else:
                            spfy.spmma(w, b, d, g.M, g.N, g.K, args.batch)
                        done = s_run.record_event()
                    with torch.cuda.stream(s_out):
                        s_out.wait_event(done)
                        hostbuf[("d", g)].copy_(d, non_blocking=True)
                torch.cuda.synchronize()

            e2e_implicit_step()
            barrier()
            torch.cuda.synchronize()
            e0.record()
            for _ in range(args.e2e_steps):
                e2e_implicit_step()
            e1.record()
            torch.cuda.synchronize()
            te = torch.tensor([e0.elapsed_time(e1)], dtype=torch.float64, device=dev)
            if world > 1:
                dist.all_reduce(te, op=dist.ReduceOp.MAX)
            ei_ms = float(te.item()) / args.e2e_steps
            # the implicit result is the explicit one bit for bit: largest conv layer, unfolded operand in (kh, kw, c) order
            same = None
            if rank == 0:
                import torch.nn.functional as F
                g0 = max(conv_geom, key=lambda q: q.K)
                li = next(i for i, l in enumerate(layers) if l[0] == g0)
                _, w0, _, d0, comp0 = layers[li]
                ho, cin = conv_geom[g0]
                cols = F.unfold(xdev[g0].permute(0, 3, 1, 2).float(), 3, padding=1).view(args.batch, cin, 9, ho * ho)
                bx = cols.permute(2, 1, 0, 3).reshape(g0.K, g0.N).to(tdt).contiguous()
                del cols
                same = bool(torch.equal(spfy.spmma_compressed(comp0, bx), d0)) and \
                    bool(torch.equal(hostbuf[("d", g0)], d0.cpu()))
                del bx
                if not same:
                    raise SystemExit("bench.py: implicit-GEMM e2e output differs from the explicit operand's")
            e2e["implicit"] = {
                "value": flops_step * world / (ei_ms * 1e-3) / 1e12, "unit": UNIT, "ms_per_step": ei_ms,
                "h2d_bytes_per_step": h2d_i, "d2h_bytes_per_step": d2h, "steps": args.e2e_steps,
                "conv_layers": sum(1 for g in gemms if g in conv_geom), "identical_to_explicit_operand": same,
                "pcie_GBs_per_rank": {"h2d": h2d_i / (ei_ms * 1e-3) / 1e9, "d2h": d2h / (ei_ms * 1e-3) / 1e9},
                "api": "as e2e, but the 3 x 3 layers go through spfy_spmma_conv: host NHWC activations in, the K x N operand "
                       "(9 x the activation bytes) is never built on either side of PCIe; same outputs, same FLOPs counted"}
        # restore the resident weights for anything that follows
        del hostbuf

    # ---- prune24 on a matrix large enough to be bandwidth- rather than ramp-bound (the weight set of one
    #      model is 47 MB: a 15-20 us launch) -- the "prune GB/s" half of the metric
    prune_large = None
    if rank == 0 and not args.no_prune_large:
        rows = cols = 16384
        big = (torch.rand(rows, cols, device=dev, generator=gen) * 2 - 1).to(tdt)
        bcomp = spfy.alloc_compressed(tdt, rows, cols, dev)
        for _ in range(3):
            spfy.prune24(big, out=bcomp)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(10):
            spfy.prune24(big, out=bcomp)
        e1.record()
        torch.cuda.synchronize()
        pl_ms = e0.elapsed_time(e1) / 10
        pl_bytes = spfy.shapes.prune24_bytes(rows, cols)
        prune_large = {"kernel": "prune24_fast_kernel", "case": f"{rows}x{cols} {args.dtype} -> SM100 layout", "ms": pl_ms,
                       "gbs": pl_bytes / (pl_ms * 1e-3) / 1e9, "frac": pl_bytes / (pl_ms * 1e-3) / 1e9 / hbm_peak,
                       "algorithmic_bytes": pl_bytes}
        del big, bcomp

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0

    achieved = spmma_bytes_step / (spmma_ms * 1e-3) / 1e9
    traffic, traffic_src = ncu_traffic() if args.csv == "resnet50.csv" and args.batch == 32 else (None, None)
    line = {
        "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "f16" if args.dtype == "fp16" else "bf16", "data": "synthetic",
        "config": config_dict(args, len(gemms), plan.launches),
        "clocks": clocks, "gpu_launches": launches,
        "roofline": {"bound": "hbm", "kernel": f"spmma_kernel (tcgen05.mma.sp, {plan.launches} persistent launches per step)", "achieved": achieved, "peak": hbm_peak,
                     "unit": "GB/s", "frac": achieved / hbm_peak, "traffic": traffic, "traffic_source": traffic_src,
                     "peak_source": peak_src,
                     "algorithmic_bytes_per_step": spmma_bytes_step, "launches_per_step": plan.launches, "layers_per_step": len(layers),
                     "ms_per_step": spmma_ms,
                     "tflops": flops_step / (spmma_ms * 1e-3) / 1e12,
                     "frac_of_sparse_tensor_peak": flops_step / (spmma_ms * 1e-3) / 1e12 / (2 * tc_sust)},
        "prune": {"kernel": "prune24_batched_kernel", "gbs": prune_bytes_step / (prune_ms * 1e-3) / 1e9,
                  "frac": prune_bytes_step / (prune_ms * 1e-3) / 1e9 / hbm_peak, "ms_per_step": prune_ms,
                  "algorithmic_bytes_per_step": prune_bytes_step,
                  "note": "all layers' weights in one launch; 23.5 M elements, 3.125 B/element"},
    }
    if verified:
        line["verified"] = verified
    if prune_large:
        line["prune_large"] = prune_large
    if e2e:
        line["e2e"] = e2e
    if implicit_plan:
        line["implicit_plan"] = implicit_plan
    if not args.no_cpu and world == 1:
        orc = ge.load_oracle()
        line["cpu_baseline"] = cpu_baseline(spfy, orc, gemms, 0 if args.dtype == "fp16" else 1)
    # the drop-in call is ONE spmma per layer: its cost next to the plan's (and next to cusparseLt's single_ms / back_to_back_ms
    # of the reference arm, which are taken the same two ways)
    single_ms = per_layer_report(spfy, layers, hbm_peak, tc_sust, quiet=not args.per_layer)
    line["single_call"] = {"ms_sum_over_layers": single_ms, "frac_of_hbm": spmma_bytes_step / (single_ms * 1e-3) / 1e9 / hbm_peak,
                           "timing": "spfy_spmma per layer, median of 5 launches, L2 flushed before each",
                           "plan_ms": spmma_ms}
    print(json.dumps(line), file=json_out, flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


DUMP_BYTES = 48 << 20


def dump_outputs(out_dir, arrays):
    """`arrays` ({name: tensor}, in a fixed order) to out_dir/<name>.npy, DUMP_BYTES in all whatever the table:
    float32, or float64 for int32 indices so that they stay exact.  An array larger than its share is written as a
    1-D sample at sorted positions drawn with its position in `arrays` as seed, so two builds run with the same
    arguments write the same positions."""
    import numpy as np
    import torch
    os.makedirs(out_dir, exist_ok=True)
    cap = DUMP_BYTES // 8 // len(arrays)
    for i, (name, a) in enumerate(arrays.items()):
        if a.numel() > cap:
            idx = np.sort(np.random.default_rng(i).choice(a.numel(), cap, replace=False))
            a = a.reshape(-1)[torch.from_numpy(idx).to(a.device)]
        a = a.double() if a.dtype == torch.int32 else a.float()
        np.save(os.path.join(out_dir, name + ".npy"), a.cpu().numpy())


def compressed_arrays(i, comp):
    """the compressed operand prune24_batched hands its caller: values (in the weights' dtype) and metadata bytes"""
    return {f"vals_{i:03d}": comp.vals.view(comp.dtype), f"meta_{i:03d}": comp.meta}


def per_layer_report(spfy, layers, hbm_peak, tc_peak, quiet=False):
    """Per-shape timing of the SINGLE call spfy_spmma (what one sparsifyme::spmma issues), cold operands (L2 flushed
    before every launch, median of 5): a stderr table for profiles/, and the sum over all layers of the table -- the
    figure to put beside cusparseLt's `single_ms` (oracle/cusparselt_ref.cu sweep times each layer the same way)."""
    import torch
    seen = {}
    total = 0.0
    for g, w, b, d, comp in layers:
        if g in seen:
            total += seen[g]
            continue
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        flush = torch.empty(256 << 20, dtype=torch.uint8, device=b.device)
        ts = []
        for _ in range(5):
            flush.zero_()
            e0.record()
            spfy.spmma_compressed(comp, b, out=d)
            e1.record()
            torch.cuda.synchronize()
            ts.append(e0.elapsed_time(e1))
        ms = statistics.median(ts)
        by = spfy.shapes.spmma_bytes(g)
        fl = spfy.shapes.spmma_flops(g)
        seen[g] = ms
        total += ms
        if not quiet:
            print(f"layer M={g.M:5d} K={g.K:5d} N={g.N:7d}  {ms*1e3:8.1f} us  {by/ms/1e6:7.0f} GB/s ({by/ms/1e6/hbm_peak:5.2f} of HBM)"
                  f"  {fl/ms/1e9:7.1f} TFLOP/s ({fl/ms/1e9/(2*tc_peak):5.2f} of sparse TC)", file=sys.stderr)
    return total


if __name__ == "__main__":
    sys.exit(main())
