#!/bin/bash
# One B200: the wide-halo tests, scripts/halo_bench.py at widths 1 2 4, the whole GPU suite, smoke() and bench.py.
#   bash scripts/gpu_halo_width.sh <output directory>
OUT=${1:?usage: gpu_halo_width.sh <output directory>}
mkdir -p "$OUT"
python -c "import __graft_entry__ as g; g.build()" > "$OUT/width_build.log" 2>&1; echo "build rc=$?"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader | tee "$OUT/width_gpu_info.txt"
timeout 1200 python -m pytest tests/test_gpu_halo_width.py -m gpu -q > "$OUT/width_pytest.log" 2>&1; echo "width pytest rc=$?"; tail -3 "$OUT/width_pytest.log"
timeout 900 python scripts/halo_bench.py --widths 1 2 4 --out "$OUT/halo_bench_widths_1gpu.json" > "$OUT/halo_bench_widths_1gpu.log" 2>&1; echo "halo_bench rc=$?"
timeout 1500 python -m pytest tests -m gpu -q > "$OUT/pytest_gpu.log" 2>&1; echo "pytest rc=$?"; tail -2 "$OUT/pytest_gpu.log"
timeout 120 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -1
timeout 300 python bench.py --gpus 1 --steps 20 --warmup 5 > "$OUT/bench_py.json" 2> "$OUT/bench_py.err"; echo "bench rc=$?"; tail -c 600 "$OUT/bench_py.json"
