#!/bin/bash
# One B200: the cut kernels past their level tables (tests/test_gpu_many_leaves.py), the whole GPU suite, smoke() and bench.py.
#   bash scripts/gpu_many_leaves.sh <output directory>
OUT=${1:?usage: gpu_many_leaves.sh <output directory>}
mkdir -p "$OUT"
python -c "import __graft_entry__ as g; g.build()" > "$OUT/many_leaves_build.log" 2>&1; echo "build rc=$?"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader | tee "$OUT/many_leaves_gpu_info.txt"
timeout 1200 python -m pytest tests/test_gpu_many_leaves.py -m gpu -q --durations=0 > "$OUT/many_leaves_pytest.log" 2>&1; echo "many-leaves pytest rc=$?"; tail -3 "$OUT/many_leaves_pytest.log"
timeout 1800 python -m pytest tests -m gpu -q > "$OUT/pytest_gpu.log" 2>&1; echo "pytest rc=$?"; tail -2 "$OUT/pytest_gpu.log"
timeout 120 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -1
timeout 300 python bench.py --gpus 1 --steps 20 --warmup 5 > "$OUT/bench_py.json" 2> "$OUT/bench_py.err"; echo "bench rc=$?"; tail -c 600 "$OUT/bench_py.json"
