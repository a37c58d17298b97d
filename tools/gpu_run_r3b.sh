#!/bin/bash
# Round 3, run B (CTA-pair GEMM, final tree): whole-step A/B against the parent commit's build (exported and built beforehand:
# git archive HEAD~1 | tar -x -C build/parent, then build() there), three runs each, interleaved, every run also dumping what its last
# step computed; the dumps compared (tools/compare_outputs.py); the GEMM microbenchmark at T = 65536 from both trees; the GPU suite and
# smoke() on the new tree.  Usage: tools/gpu_run_r3b.sh OUT_DIR
cd "$(dirname "$0")/.."
OUT="${1:?output directory}"
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > "$OUT/r3b_gpu.txt" 2>&1; cat "$OUT/r3b_gpu.txt"
for i in 1 2 3; do
    for v in parent new; do
        d=.; [ $v = parent ] && d=build/parent
        timeout -k 10 900 python $d/bench.py --gpus 1 --no-cpu-baseline --no-reference-gpu --dump-outputs "$OUT/r3b_dump_${v}_$i" \
            > "$OUT/r3b_bench_${v}_$i.json" 2> "$OUT/r3b_bench_${v}_$i.err"; echo "bench $v $i rc=$?"
        python -c "import json,sys; l=[json.loads(x) for x in open(sys.argv[1]) if x.startswith('{')][-1]; print(sys.argv[1], l.get('training_sequences_per_second'))" "$OUT/r3b_bench_${v}_$i.json"
    done
done
python tools/compare_outputs.py "$OUT"/r3b_dump_parent_{1,2,3} -- "$OUT"/r3b_dump_new_{1,2,3} > "$OUT/r3b_compare_outputs.log" 2>&1
echo "compare rc=$?"; cat "$OUT/r3b_compare_outputs.log"
for v in parent new; do
    d=.; [ $v = parent ] && d=build/parent
    T=65536 timeout -k 10 300 python $d/tools/bench_gemm.py > "$OUT/r3b_gemm_$v.log" 2>&1; echo "bench_gemm $v rc=$?"
done
timeout -k 10 900 python -m pytest tests -m gpu -q > "$OUT/r3b_pytest_gpu.log" 2>&1; echo "pytest rc=$?"; tail -5 "$OUT/r3b_pytest_gpu.log"
timeout -k 10 300 python -c "import __graft_entry__ as g; g.smoke()" > "$OUT/r3b_smoke.log" 2>&1; echo "smoke rc=$?"; tail -5 "$OUT/r3b_smoke.log"
exit 0
