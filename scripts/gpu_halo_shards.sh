#!/bin/bash
# One B200: the sharded halo exchange's tests, the whole GPU suite, smoke(), bench.py and scripts/halo_bench.py.
#   bash scripts/gpu_halo_shards.sh <output directory>
OUT=${1:?usage: gpu_halo_shards.sh <output directory>}
mkdir -p "$OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader | tee "$OUT/halo_gpu_info.txt"
timeout 300 python -m pytest tests/test_gpu_halo_shards.py -m gpu -q > "$OUT/halo_pytest_shards.log" 2>&1; echo "shards pytest rc=$?"; tail -3 "$OUT/halo_pytest_shards.log"
timeout 300 python scripts/halo_bench.py --out "$OUT/halo_bench_1gpu.json" > "$OUT/halo_bench_1gpu.log" 2>&1; echo "halo_bench rc=$?"; tail -c 1500 "$OUT/halo_bench_1gpu.log"
timeout 400 python -m pytest tests -m gpu -q > "$OUT/halo_pytest_gpu.log" 2>&1; echo "pytest rc=$?"; tail -2 "$OUT/halo_pytest_gpu.log"
timeout 120 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -1
timeout 300 python bench.py --gpus 1 --steps 20 --warmup 5 > "$OUT/halo_bench_py.json" 2> "$OUT/halo_bench_py.err"; echo "bench rc=$?"; tail -c 600 "$OUT/halo_bench_py.json"
