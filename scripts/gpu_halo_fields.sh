#!/bin/bash
# One B200: the halo scatter / gather tests, scripts/halo_bench.py, the whole GPU suite, smoke() and bench.py.
#   bash scripts/gpu_halo_fields.sh <output directory>
OUT=${1:?usage: gpu_halo_fields.sh <output directory>}
mkdir -p "$OUT"
python -c "import __graft_entry__ as g; g.build()" > "$OUT/fields_build.log" 2>&1; echo "build rc=$?"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader | tee "$OUT/fields_gpu_info.txt"
timeout 600 python -m pytest tests/test_gpu_halo_fields.py -m gpu -q > "$OUT/fields_pytest.log" 2>&1; echo "fields pytest rc=$?"; tail -3 "$OUT/fields_pytest.log"
timeout 600 python scripts/halo_bench.py --out "$OUT/halo_bench_1gpu.json" > "$OUT/halo_bench_1gpu.log" 2>&1; echo "halo_bench rc=$?"; tail -c 3000 "$OUT/halo_bench_1gpu.log"
timeout 900 python -m pytest tests -m gpu -q > "$OUT/pytest_gpu.log" 2>&1; echo "pytest rc=$?"; tail -2 "$OUT/pytest_gpu.log"
timeout 120 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -1
timeout 300 python bench.py --gpus 1 --steps 20 --warmup 5 > "$OUT/bench_py.json" 2> "$OUT/bench_py.err"; echo "bench rc=$?"; tail -c 600 "$OUT/bench_py.json"
