#!/bin/bash
# One B200: the byte-mask tests (tests/test_gpu_mask_bytes.py), the torchrun worker on the GPUs there are, the byte-mask
# benchmark, smoke(), bench.py and the whole GPU suite.
#   bash scripts/gpu_mask_bytes.sh <output directory>
OUT=${1:?usage: gpu_mask_bytes.sh <output directory>}
mkdir -p "$OUT"
python -c "import __graft_entry__ as g; g.build()" > "$OUT/mask_bytes_build.log" 2>&1; echo "build rc=$?"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader | tee "$OUT/mask_bytes_gpu_info.txt"
timeout 900 python -m pytest tests/test_gpu_mask_bytes.py -m gpu -q --durations=0 > "$OUT/mask_bytes_pytest.log" 2>&1; echo "mask-bytes pytest rc=$?"; tail -3 "$OUT/mask_bytes_pytest.log"
G=$(nvidia-smi -L | wc -l)
timeout 600 python -m torch.distributed.run --nnodes=1 --nproc-per-node "$G" --master-addr 127.0.0.1 --master-port 29541 \
    tests/mask_bytes_worker.py --big > "$OUT/mask_bytes_worker_${G}gpu.log" 2>&1; echo "worker G=$G rc=$?"; tail -2 "$OUT/mask_bytes_worker_${G}gpu.log"
timeout 900 python scripts/mask_bytes_bench.py --out "$OUT/mask_bytes_bench_1gpu.json" > "$OUT/mask_bytes_bench_1gpu.log" 2>&1; echo "mask-bytes bench rc=$?"; cat "$OUT/mask_bytes_bench_1gpu.log" | cut -c1-400
timeout 120 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -1
timeout 300 python bench.py --gpus 1 --steps 20 --warmup 5 > "$OUT/bench_py.json" 2> "$OUT/bench_py.err"; echo "bench rc=$?"; tail -c 300 "$OUT/bench_py.json"
timeout 1800 python -m pytest tests -m gpu -q > "$OUT/pytest_gpu.log" 2>&1; echo "pytest rc=$?"; tail -2 "$OUT/pytest_gpu.log"
