#!/bin/bash
# tools/capture_round.sh TAG — one-GPU evidence of a round: GPU tests, every bench workload (never under a profiler),
# the reference arm, then the ncu launch list and the `--set full` captures of the dominant kernels.
# Run through gpurun; outputs land in gpurun_out/ and are copied into profiles/ by hand.
TAG=${1:-rX}
O=gpurun_out
mkdir -p $O
timeout 600 python -m pytest tests -m gpu -x -q > $O/pytest_$TAG.log 2>&1; tail -2 $O/pytest_$TAG.log
python bench.py > $O/bench_$TAG.json 2> $O/bench_$TAG.err
python bench.py --impl reference --steps 2 --warmup 1 > $O/bench_ref_$TAG.json 2>/dev/null
python bench.py --workload cfg1_n50 --steps 50 > $O/bench_cfg1_$TAG.json 2>/dev/null
python bench.py --workload cfg3_batch4096 > $O/bench_cfg3_$TAG.json 2>/dev/null
python bench.py --workload cfg4_n2000 --steps 8 --no-cpu-baseline > $O/bench_cfg4_$TAG.json 2>/dev/null
python bench.py --workload cfg5_match > $O/bench_cfg5_$TAG.json 2>/dev/null
python bench.py --full-square --no-cpu-baseline > $O/bench_full_$TAG.json 2>/dev/null
# matcher evidence: DP4A / IMAD issue rates of this GPU
[ -x tools/idp_rate_probe ] || nvcc -gencode arch=compute_100a,code=sm_100a -O3 -o tools/idp_rate_probe tools/idp_rate_probe.cu
./tools/idp_rate_probe > $O/idp_rate_probe_$TAG.txt 2>&1
ncu --metrics gpu__time_duration.sum --clock-control none -c 4000 --csv --log-file $O/launches_$TAG.csv \
    python bench.py --steps 2 --warmup 3 --no-cpu-baseline --no-sharded --no-parity > $O/ncu_$TAG.log 2>&1
ncu --set full --clock-control none --import-source on \
    -k regex:"k_gemm_nt_sub|k_blk_factor|k_blk_V|k_blk_gather|k_match_filter|k_blk_S|k_blk_Gx|k_ransac|k_predict" -s 60 -c 40 -o $O/top_$TAG \
    python bench.py --steps 1 --warmup 3 --no-cpu-baseline > $O/ncu_full_$TAG.log 2>&1
for f in $O/bench_*_$TAG.json $O/bench_$TAG.json; do echo $f; python - "$f" <<'PY'
import json, sys
d = json.loads(open(sys.argv[1]).read().strip().splitlines()[-1])
print({k: d.get(k) for k in ("value", "ms_per_step", "gpu_launches")}, d.get("e2e", {}).get("value"), d.get("roofline", {}).get("frac"), d.get("cpu_baseline", {}).get("value"))
PY
done
# the warp tile matcher inside a batch of filters (8 waves of 148 filters)
ncu --set full --clock-control none --import-source on -k regex:"k_match_filter_batch_warp2" -s 3 -c 1 -o $O/warp2_$TAG \
    python bench.py --workload cfg3_batch4096 --filters 1184 --steps 1 --warmup 3 --no-cpu-baseline --no-parity > $O/ncu_warp2_$TAG.log 2>&1
