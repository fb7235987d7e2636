#!/bin/bash
# Round 3 A/B on one B200: the parent build (a copy of the previous commit with its library built, in $PARENT)
# against this tree.  Outputs must be byte-identical; then alternating timed runs, the knob sweep, the GPU tests.
#   PARENT=<dir> OUT=<dir> bash profiles/r03_ab.sh        (writes <OUT>/r03_*)
set -u
PARENT=${PARENT:?directory of the parent build}
mkdir -p "${OUT:?directory for the results}"
OUT=$(cd "$OUT" && pwd)
here=$(pwd)
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $OUT/r03_gpu.txt
ngpu=$(nvidia-smi -L | wc -l)
echo "gpus: $ngpu" | tee -a $OUT/r03_gpu.txt

run() {   # run <tree> <tag> <bench args...>: last JSON line -> $OUT/r03_<tag>.json
    local tree=$1 tag=$2
    shift 2
    (cd $tree && python bench.py "$@" > $OUT/r03_$tag.json 2> $OUT/r03_$tag.err)
    python - $OUT/r03_$tag.json $tag <<'PY'
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
for wl in cfg4 cfg2 cfg3 cfg5; do
    rm -rf /tmp/r03_dump_p /tmp/r03_dump_b
    run $PARENT dump_${wl}_parent --workload $wl --steps 3 --warmup 1 --no-cpu --no-side --dump-outputs /tmp/r03_dump_p
    run $here dump_${wl}_branch --workload $wl --steps 3 --warmup 1 --no-cpu --no-side --dump-outputs /tmp/r03_dump_b
    for f in /tmp/r03_dump_p/*.npy; do
        b=$(basename $f)
        if cmp -s $f /tmp/r03_dump_b/$b; then echo "$wl $b identical"; else echo "$wl $b DIFFERENT"; fi
    done
done 2>&1 | tee $OUT/r03_outputs_cmp.log

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
# 3. knobs at cfg 4 (branch): pass-1 launch shape, pass-2 warps per CTA
for st in 8,2,2,3 8,4,2,2 8,2,2,4; do
    DESC_B200_ST=$st run $here cfg4_st_$st --workload cfg4 --steps 10 --warmup 3 --no-cpu --no-side
done
for pw in 4 8; do
    DESC_B200_PB_WARPS=$pw run $here cfg4_pbw_$pw --workload cfg4 --steps 10 --warmup 3 --no-cpu --no-side
done
if [ "$ngpu" -ge 8 ]; then
    run $here cfg4_n8_branch --workload cfg4 --gpus 8 --steps 10 --warmup 3 --no-cpu --no-side
fi
} 2>&1 | tee $OUT/r03_ab.log

# 4. tests
python -m pytest -q -m gpu tests -p no:cacheprovider > $OUT/r03_gpu_tests.log 2>&1
tail -5 $OUT/r03_gpu_tests.log
if [ "$ngpu" -ge 2 ]; then
    python tests/multi_gpu_check.py --full > $OUT/r03_multi_gpu_check.log 2>&1
    tail -2 $OUT/r03_multi_gpu_check.log
fi
python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2 | tee $OUT/r03_smoke.log
