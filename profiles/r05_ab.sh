#!/bin/bash
# Round 5 A/B on one B200 (or more): the parent build (a copy of the previous commit with its library built, in
# $PARENT) against this tree, whose one-GPU streamed passes keep partner sums and S in adjacency order.  Outputs
# must be byte-identical; then alternating timed runs, the GPU tests, smoke() and, with 2+ GPUs, the multi-GPU check
# over both exchanges.
#   PARENT=<dir> OUT=<dir> bash profiles/r05_ab.sh        (writes <OUT>/r05_*)
set -u
PARENT=${PARENT:?directory of the parent build}
mkdir -p "${OUT:?directory for the results}"
OUT=$(cd "$OUT" && pwd)
here=$(pwd)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $OUT/r05_gpu.txt
ngpu=$(nvidia-smi -L | wc -l)
echo "gpus: $ngpu" | tee -a $OUT/r05_gpu.txt

run() {   # run <tree> <tag> <bench args...>: last JSON line -> $OUT/r05_<tag>.json
    local tree=$1 tag=$2
    shift 2
    (cd $tree && python bench.py "$@" > $OUT/r05_$tag.json 2> $OUT/r05_$tag.err)
    python - $OUT/r05_$tag.json $tag <<'PY'
import json, sys
try:
    j = json.loads(open(sys.argv[1]).read().strip().splitlines()[-1])
    s = j.get("stages_ms", {})
    print("%-22s ms_per_step %8.2f  pass1 %.4f  pass2 %.4f  comm %.4f  parity %s" % (
        sys.argv[2], j["ms_per_step"], s.get("pgd_pass1_ms", 0), s.get("pgd_pass2_ms", 0), s.get("pgd_comm_ms", 0),
        j.get("parity", {}).get("ok") if isinstance(j.get("parity"), dict) else None))
except Exception as e:
    print(sys.argv[2], "FAILED", e)
PY
}

# 1. outputs: byte-identical S_vec / R_est at every streamed / blocked workload
dump=$(mktemp -d)
for wl in cfg4 cfg2 cfg3 cfg5; do
    rm -rf $dump/p $dump/b
    run $PARENT dump_${wl}_parent --workload $wl --steps 3 --warmup 1 --no-cpu --no-side --dump-outputs $dump/p
    run $here dump_${wl}_branch --workload $wl --steps 3 --warmup 1 --no-cpu --no-side --dump-outputs $dump/b
    for f in $dump/p/*.npy; do
        b=$(basename $f)
        if cmp -s $f $dump/b/$b; then echo "$wl $b identical"; else echo "$wl $b DIFFERENT"; fi
    done
done 2>&1 | tee $OUT/r05_outputs_cmp.log
rm -rf $dump

# 2. speed: cfg 4 alternating parent / branch, then cfg 2 / 3 / 5
{
for k in 1 2 3; do
    run $PARENT cfg4_parent_$k --workload cfg4 --steps 10 --warmup 3 --no-cpu --no-side
    run $here cfg4_branch_$k --workload cfg4 --steps 10 --warmup 3 --no-cpu --no-side
done
for wl in cfg2 cfg3 cfg5; do
    for k in 1 2; do
        run $PARENT ${wl}_parent_$k --workload $wl --steps 10 --warmup 3 --no-cpu --no-side
        run $here ${wl}_branch_$k --workload $wl --steps 10 --warmup 3 --no-cpu --no-side
    done
done
if [ "$ngpu" -ge 8 ]; then
    run $here cfg4_n8_branch --workload cfg4 --gpus 8 --steps 10 --warmup 3 --no-cpu --no-side
fi
} 2>&1 | tee $OUT/r05_ab.log

# 3. tests, smoke, and the multi-GPU check over the default (peer) and the NCCL point-to-point exchange
python -m pytest -q -m gpu tests -p no:cacheprovider > $OUT/r05_gpu_tests.log 2>&1
tail -5 $OUT/r05_gpu_tests.log
python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2 | tee $OUT/r05_smoke.log
if [ "$ngpu" -ge 2 ]; then
    for comm in peer p2p; do
        DESC_B200_COMM=$comm python -m torch.distributed.run --nnodes=1 --nproc-per-node $ngpu --master-addr 127.0.0.1 \
            --master-port 29521 tests/multi_gpu_check.py --full > $OUT/r05_multi_gpu_check_$comm.log 2>&1
        echo "multi-GPU check ($comm): $(grep -c MULTI_GPU_OK $OUT/r05_multi_gpu_check_$comm.log) MULTI_GPU_OK"
    done
fi
