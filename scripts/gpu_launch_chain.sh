#!/bin/bash
# B200: this tree against a built checkout of its parent commit, alternated in one job -- bench.py at C5, C4, C3 and
# C2, three rounds, the order of the two builds swapped every round -- then smoke() and the GPU suite; with two GPUs
# or more also the torchrun parity worker and bench.py on 2 GPUs for both builds.
#   bash scripts/gpu_launch_chain.sh <output directory> <built checkout of the parent commit>
OUT=${1:?usage: gpu_launch_chain.sh <output directory> <parent checkout>}
PARENT=${2:?usage: gpu_launch_chain.sh <output directory> <parent checkout>}
mkdir -p "$OUT"
OUT=$(cd "$OUT" && pwd)
PARENT=$(cd "$PARENT" && pwd)
BRANCH=$(pwd)
python -c "import __graft_entry__ as g; g.build()" > "$OUT/build.log" 2>&1; echo "build rc=$?"
(cd "$PARENT" && python -c "import __graft_entry__ as g; g.build()") > "$OUT/build_parent.log" 2>&1; echo "parent build rc=$?"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv,noheader | tee "$OUT/gpu_info.txt"
G=$(nvidia-smi -L | wc -l)
line() { # ms per step, parity and digest of a bench.py output
    python -c "import json, sys; d = json.loads(open(sys.argv[1]).read().strip().splitlines()[-1]); \
print('%.4f ms' % d['ms_per_step'], 'parity', d['parity']['passed'], d['parity']['digest'][:16])" "$1" 2>/dev/null || echo "no result"
}
for round in 1 2 3; do
    arms="parent branch"
    [ $((round % 2)) = 0 ] && arms="branch parent"
    for w in C5_32768x32768_p16384 C4_8192x8192_p4096 C3_4096x4096_p1024 C2_528x522_p64; do
        for arm in $arms; do
            dir=$BRANCH
            [ $arm = parent ] && dir=$PARENT
            f="$OUT/ab_${w%%_*}_${arm}_r${round}"
            (cd "$dir" && timeout 300 python bench.py --gpus 1 --steps 20 --warmup 5 --workload $w --no-e2e --no-cpu) > "$f.json" 2> "$f.err"
            echo "r$round ${w%%_*} $arm rc=$? $(line "$f.json")"
        done
    done
done
timeout 120 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -1
timeout 300 python bench.py --gpus 1 --steps 20 --warmup 5 > "$OUT/bench_py.json" 2> "$OUT/bench_py.err"; echo "bench rc=$? $(line "$OUT/bench_py.json")"
timeout 1800 python -m pytest tests -m gpu -q > "$OUT/pytest_gpu.log" 2>&1; echo "pytest rc=$?"; tail -2 "$OUT/pytest_gpu.log"
if [ "$G" -ge 2 ]; then
    TR="python -m torch.distributed.run --nnodes=1 --nproc-per-node 2 --master-addr 127.0.0.1"
    timeout 900 $TR --master-port 29541 tests/mgpu_worker.py --big > "$OUT/mgpu2_parity.log" 2>&1; echo "parity rc=$?"
    grep -E "MISMATCH|PARITY|Error|error" "$OUT/mgpu2_parity.log" | head -5
    for round in 1 2; do
        for arm in parent branch; do
            dir=$BRANCH
            [ $arm = parent ] && dir=$PARENT
            f="$OUT/ab2_C5_${arm}_r${round}"
            (cd "$dir" && timeout 300 $TR --master-port 29542 bench.py --gpus 2 --steps 20 --warmup 5 --no-e2e --no-cpu) > "$f.json" 2> "$f.err"
            echo "2 GPUs r$round C5 $arm rc=$? $(line "$f.json")"
        done
    done
else
    echo "one GPU: the 2-GPU parity worker and bench.py --gpus 2 were not run"
fi
