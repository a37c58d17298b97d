#!/bin/bash
# Round 3, run A (CTA-pair GEMM): the pair tests and the GEMM suite first; then the GEMM microbenchmark at T = 65536 for two
# epilogue-warp variants of the new kernel (run B measures the default and the parent in the same call).  The variants are built
# beforehand with DLE_GEMM_EW16_EPILOGUES set:
#   python -c "from deeplearningexamples_b200.csrc import build as b; b.build_variant('ew16gelu', ['-DDLE_GEMM_EW16_EPILOGUES=0xAu'], only=['gemm_sm100.cu'])"
#   (and 'ew16all' with 0xFFu)
# Usage: tools/gpu_run_r3a.sh OUT_DIR.  Exits 1 when a test fails, so that `gpu_run_r3a.sh D && gpu_run_r3b.sh D` measures only a correct tree.
cd "$(dirname "$0")/.."
OUT="${1:?output directory}"
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT/r3a_gpu.txt" 2>&1; cat "$OUT/r3a_gpu.txt"
timeout -k 10 400 python -m pytest tests/test_gemm_pair_gpu.py tests/test_gemm_gpu.py -m gpu -x -q > "$OUT/r3a_pytest_gemm.log" 2>&1; rc=$?
echo "pytest rc=$rc"; tail -15 "$OUT/r3a_pytest_gemm.log"
[ $rc -ne 0 ] && exit 1
for v in ew16gelu ew16all; do
    DLE_LIB_PATH=deeplearningexamples_b200/libdle_b200_$v.so T=65536 timeout -k 10 300 python tools/bench_gemm.py > "$OUT/r3a_gemm_$v.log" 2>&1
    echo "bench_gemm $v rc=$?"
done
exit 0
