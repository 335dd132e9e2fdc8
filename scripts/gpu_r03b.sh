#!/bin/bash
# Round 3, GPU call B (1 GPU): two-class SWAR words.  Card, whole suite and smoke, then the parent build
# (skywalking-banyandb_b200/variants/parent.so, built from the parent commit) against this one: scan-kernel times at 1e9 in one
# process, and bench.py three times per build, alternating, each dumping its outputs for a byte-for-byte comparison.
# Usage: scripts/gpu_r03b.sh [tag] [output directory]
TAG=${1:-r03b}
OUT=${2:-bench_outputs}  # results directory
mkdir -p $OUT
PARENT=$PWD/skywalking-banyandb_b200/variants/parent.so
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $OUT/${TAG}_card.txt
python -c "import __graft_entry__ as g; g.build(); g.smoke()" 2>&1 | tail -2 | tee $OUT/${TAG}_smoke.log
echo "== pytest -m gpu"
timeout 1200 python -m pytest tests -m gpu -q 2>&1 | grep -E "FAILED|ERROR|passed|failed|^E  " | head -30 | tee $OUT/${TAG}_pytest.log
echo "== variants (1e9)"
timeout 900 python tools/time_variants.py variants/parent.so libbydbgpu.so --series 10000 --steps 30 2>&1 | grep -v "^$" | tail -4 | tee $OUT/${TAG}_variants.log
summ() {
python -c "
import json,sys
j=json.loads(open(sys.argv[1]).read().strip().splitlines()[-1])
cb=j.get('cpu_baseline') or j.get('vs_baseline') or {}
print(sys.argv[2],'value',j['value'],'ms/step',round(j['ms_per_step'],4),'scan',round(j['scan_kernel_ms'],4),'c2',round(j['c2_query']['ms_per_step'],4),'keyed',round(j['stored_tag_group_by']['ms_per_step'],4),
      'agrees', cb.get('agrees_with_gpu') if isinstance(cb,dict) else None)
" $1 $2 | tee -a $OUT/${TAG}_bench_summary.txt
}
for rep in 1 2 3; do
  EXTRA=""
  [ $rep -gt 1 ] && EXTRA="--no-cpu --no-e2e"
  for arm in parent new; do
    echo "== bench $arm $rep $EXTRA"
    if [ $arm = parent ]; then export BYDB_GPU_LIB=$PARENT; else unset BYDB_GPU_LIB; fi
    timeout 900 python bench.py --gpus 1 --steps 20 --warmup 3 $EXTRA --dump-outputs $OUT/dump_${arm}_$rep > $OUT/${TAG}_bench_${arm}_$rep.json 2>$OUT/${TAG}_bench_${arm}_$rep.err
    summ $OUT/${TAG}_bench_${arm}_$rep.json "$arm$rep"
  done
  unset BYDB_GPU_LIB
  cmp -s <(cd $OUT/dump_parent_$rep && cat $(ls)) <(cd $OUT/dump_new_$rep && cat $(ls)) && [ "$(ls $OUT/dump_parent_$rep)" = "$(ls $OUT/dump_new_$rep)" ] \
    && echo "dumps $rep identical ($(ls $OUT/dump_new_$rep | tr '\n' ' '))" | tee -a $OUT/${TAG}_bench_summary.txt \
    || echo "dumps $rep DIFFER" | tee -a $OUT/${TAG}_bench_summary.txt
done
