#!/bin/bash
# Round 3, pre-split GroupNorm outputs (DPB200_PRESPLIT): full GPU suite (with tests/test_presplit_gpu.py), smoke(), then an A/B of the
# plan with the fp32 operands (DPB200_PRESPLIT=0) against the split operands in ONE box, arms alternating: 3 C1 bench lines per arm,
# --dump-outputs of both arms compared, one per-layer table per arm (DPB200_LAYERS_OUT).  With LEGS=1 instead: one line per arm of
# the default run's finetune and LSUN-256 legs and one c5 line per arm.  Card name / power limit are read first: they belong beside
# every number.  Results go to $OUT (default: a fresh temporary directory).
set -u
OUT=${OUT:-$(mktemp -d)}
mkdir -p "$OUT"
echo "results in $OUT"
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv | tee $OUT/card.txt
python -c "import __graft_entry__ as g; g.build()" || exit 1
if [ "${LEGS:-0}" = 1 ]; then
  for arm in 0 1; do
    DPB200_PRESPLIT=$arm timeout 400 python bench.py --no-cpu --steps 10 > $OUT/bench_legs_$arm.json 2> $OUT/bench_legs_$arm.err
    echo "== legs arm $arm rc=$?"
    DPB200_PRESPLIT=$arm timeout 300 python bench.py --no-cpu --no-finetune --no-c3 --config c5 --steps 10 > $OUT/bench_c5_$arm.json 2> $OUT/bench_c5_$arm.err
    echo "== c5 arm $arm rc=$?"
  done
  OUT="$OUT" python - <<'PY'
import json, os
OUT = os.environ['OUT']
for arm in (0, 1):
    d = json.loads(open(f'{OUT}/bench_legs_{arm}.json').read().strip().split('\n')[-1])
    print(f'arm {arm} c1', d['ms_per_step'], {k: d[k]['ms_per_step'] for k in ('finetune', 'finetune_bf16', 'config3') if k in d})
    c5 = json.loads(open(f'{OUT}/bench_c5_{arm}.json').read().strip().split('\n')[-1])
    print(f'arm {arm} c5', c5['ms_per_step'])
PY
  exit 0
fi
timeout 240 python -m pytest tests -q -m gpu -rs --timeout=200 > $OUT/pytest_gpu.log 2>&1
echo "== gpu suite rc=$?"; grep -n "^FAILED\|^ERROR\|passed\|failed" $OUT/pytest_gpu.log | head -30
timeout 60 python -m pytest tests/test_presplit_gpu.py -q -s -k "groupnorm_split_output or plan" > $OUT/presplit_bounds.log 2>&1
grep -n "log2\|split GroupNorm" $OUT/presplit_bounds.log | head -40
python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -2
for i in 1 2 3; do
  for arm in 0 1; do
    extra=""
    if [ "$i" = 1 ]; then extra="--dump-outputs $OUT/dump_$arm"; export DPB200_LAYERS_OUT=$OUT/layers_$arm.txt; else unset DPB200_LAYERS_OUT; fi
    DPB200_PRESPLIT=$arm timeout 300 python bench.py --no-cpu --no-finetune --no-c3 --steps 20 $extra > $OUT/bench_c1_${arm}_$i.json 2> $OUT/bench_c1_${arm}_$i.err
    echo "== c1 arm $arm run $i rc=$?"
  done
done
unset DPB200_LAYERS_OUT
OUT="$OUT" python - <<'PY'
import json, os, statistics as stt
OUT = os.environ['OUT']
import numpy as np
def last(p):
    return json.loads(open(p).read().strip().split('\n')[-1])
for arm in (0, 1):
    rs = [last(f'{OUT}/bench_c1_{arm}_{i}.json') for i in (1, 2, 3)]
    ms = [r['ms_per_step'] for r in rs]
    print(f'arm {arm} c1 ms_per_step', ms, 'median', stt.median(ms), 'spread', max(ms) - min(ms))
    r = rs[0]['roofline']
    print('  breakdown_ms', r.get('breakdown_ms'), 'conv_ms', r.get('conv_ms'))
    print('  other_launches_ms', r.get('other_launches_ms'))
    print('  top_layers_ms', r.get('top_layers_ms'))
for f in ('loss.npy', 'grad_sample.npy'):
    a, b = np.load(f'{OUT}/dump_0/{f}'), np.load(f'{OUT}/dump_1/{f}')
    d = np.abs(a.astype(np.float64) - b)
    print(f, 'equal' if np.array_equal(a, b) else f'max|diff| {d.max():.3e} max|ref| {np.abs(a).max():.3e} rel {d.max() / max(np.abs(a).max(), 1e-30):.3e}')
PY
