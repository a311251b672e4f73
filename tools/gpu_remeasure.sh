#!/bin/bash
# per-call (event pair per call) timings: dense GEMM beside cuBLAS, COO SpMM table
T=${1:-rm}; O=gpurun_out; mkdir -p $O
export SPFY_LIB=$PWD/sparsify.me_b200/lib_dev/libsparsifyme_b200.so
timeout 300 python tools/gemm_probe.py --time --dtype f16 >> $O/${T}_gemm.log 2>&1
timeout 300 python tools/gemm_probe.py --time --dtype f32 >> $O/${T}_gemm.log 2>&1
cat $O/${T}_gemm.log
unset SPFY_LIB
timeout 900 python tools/spmm_sweep.py --csv resnet34.csv --no-cusparse --tag $T > $O/${T}_spmm_sweep.csv 2> $O/${T}_spmm_sweep.err; echo "sweep rc=$?"
grep "^#" $O/${T}_spmm_sweep.csv
