#!/usr/bin/env bash
# A/B of this tree against another build of the project (PARENT=<its root>, built), in one session on one GPU:
#   the GPU suite and smoke() of this tree, bench.py alternating between the two builds, the output dumps of both compared
#   (profiles/compare_dumps.py, with a second dump of the parent for the run-to-run spread of the float atomics) and the
#   step timelines of one and of two groups per build.  ARMS adds arms that run this tree with extra environment, e.g.
#   ARMS="fwd:D3H_ZERO_IN_FORWARD=1".  Everything lands under OUT=<directory>.
set -u
cd "$(dirname "$0")/.."
NEW=$(pwd)
PARENT=$(cd "${PARENT:?set PARENT to the root of the other build}" && pwd)
RUNS=${RUNS:-3}
ARMS=${ARMS:-}
mkdir -p "${OUT:?set OUT to the directory for the results}"
OUT=$(cd "$OUT" && pwd)
BENCH_FLAGS="--no-e2e --no-cold --no-cpu-baseline --no-torch-baseline --no-sdf-query --no-lbs-stage --no-mesh-stage"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee "$OUT/ab_gpu.csv"
echo "== GPU suite (this tree)"
timeout 1500 python -m pytest tests -m gpu -q -p no:cacheprovider > "$OUT/ab_pytest.log" 2>&1
tail -3 "$OUT/ab_pytest.log"
echo "== smoke"
timeout 300 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -1
echo "== bench, alternating parent / new"
for r in $(seq 1 "$RUNS"); do
  for spec in parent new $ARMS; do
    arm=${spec%%:*}; envs=""; [ "$spec" != "$arm" ] && envs=${spec#*:}
    root=$PARENT; [ "$arm" != parent ] && root=$NEW
    (cd "$root" && env $envs timeout 600 python bench.py $BENCH_FLAGS) > "$OUT/ab_bench_${arm}_${r}.json" 2> "$OUT/ab_bench_${arm}_${r}.err"
    python - "$OUT/ab_bench_${arm}_${r}.json" "$arm" <<'PY'
import json, sys
d = json.loads(open(sys.argv[1]).read().strip().splitlines()[-1])
print(sys.argv[2], 'ms_per_step', round(d['ms_per_step'], 4), 'blocks', d['ms_per_step_blocks'], 'single ms/frame',
      round(d['single_call']['ms_per_frame'], 4), 'clocks', d.get('clocks', {}).get('sm_mhz'))
PY
  done
done
echo "== output dumps"
(cd "$PARENT" && timeout 600 python bench.py $BENCH_FLAGS --steps 20 --dump-outputs "$OUT/dump_parent") > /dev/null 2> "$OUT/dump_parent.err"
(cd "$PARENT" && timeout 600 python bench.py $BENCH_FLAGS --steps 20 --dump-outputs "$OUT/dump_parent2") > /dev/null 2> "$OUT/dump_parent2.err"
(cd "$NEW" && timeout 600 python bench.py $BENCH_FLAGS --steps 20 --dump-outputs "$OUT/dump_new") > /dev/null 2> "$OUT/dump_new.err"
python profiles/compare_dumps.py "$OUT/dump_parent" "$OUT/dump_new" "$OUT/dump_parent2" | tee "$OUT/ab_compare_dumps.txt"
rm -rf "$OUT/dump_parent" "$OUT/dump_parent2" "$OUT/dump_new"
echo "== step timelines (one group, two groups)"
for g in 1 2; do
  (cd "$PARENT" && NGROUPS=$g timeout 300 python profiles/step_timeline.py) > "$OUT/ab_timeline_${g}g_parent.txt" 2>&1
  (cd "$NEW" && NGROUPS=$g timeout 300 python profiles/step_timeline.py) > "$OUT/ab_timeline_${g}g_new.txt" 2>&1
  grep -v "Warn\|warn" "$OUT/ab_timeline_${g}g_parent.txt" | grep "zero\|adjoint\|step" | cut -c1-60
  grep -v "Warn\|warn" "$OUT/ab_timeline_${g}g_new.txt" | grep "zero\|adjoint\|step" | cut -c1-60
done
