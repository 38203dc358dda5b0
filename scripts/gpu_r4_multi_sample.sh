# K samples per pocket (DESIGN.md 7b) on the GPU.  PART (default: all three, in order):
#   tests  the new tests on the product and the debug build, the whole GPU suite, smoke()
#   ab     K = 1 against the parent commit: final logits of bench.py --dump-outputs, then bench.py alternately, three runs each
#   bench  scripts/multi_sample_bench.py and the per-kernel attribution (scripts/loop_kernel_profile.py 50 8)
# BASE_TREE = a checkout of the parent commit with its library built (python e3-invaraint-diffusion-model_b200/build.py there); the
# debug library comes from SEQDIFF_DEBUG_BOUNDS=1 python e3-invaraint-diffusion-model_b200/build.py.  OUT = directory for the
# results (default: a new temporary directory).
set +e
export OUT=$(realpath -m ${OUT:-$(mktemp -d)})
mkdir -p "$OUT"
BASE_TREE=${BASE_TREE:-_parent}
PART=${PART:-tests ab bench}
CARD="nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv"
if [[ " $PART " == *" tests "* ]]; then
  S=$OUT/multi_sample_suite_r04.log
  $CARD >> $S
  timeout 1200 python -m pytest tests/test_multi_sample.py -q -rf -m gpu -p no:cacheprovider 2>&1 | tail -4 | sed 's/^/multi_sample : /' >> $S
  SEQDIFF_DEBUG_BOUNDS=1 timeout 1200 python -m pytest tests/test_multi_sample.py -q -rf -m gpu -p no:cacheprovider 2>&1 | tail -4 |
    sed 's/^/debug build (SEQDIFF_DEBUG_BOUNDS=1) multi_sample : /' >> $S
  [ -n "$SKIP_SUITE" ] || timeout 1800 python -m pytest tests -q -rf -m gpu -p no:cacheprovider 2>&1 | tail -4 | sed 's/^/whole GPU suite : /' >> $S
  r=$(timeout 600 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -1); echo "smoke : $r" >> $S
  cat $S
fi
if [[ " $PART " == *" ab "* ]]; then
  L=$OUT/multi_sample_ab_r04.log
  $CARD > $L
  # the final logits of the padded and the packed sampling, parent against this build
  (cd $BASE_TREE && timeout 600 python bench.py --steps 1 --warmup 1 --no-cpu-baseline --no-extras --dump-outputs $OUT/dump_base > /dev/null 2>&1)
  timeout 600 python bench.py --steps 1 --warmup 1 --no-cpu-baseline --no-extras --dump-outputs $OUT/dump_new > /dev/null 2>&1
  python - >> $L 2>&1 <<'PY'
import os
import numpy as np
OUT = os.environ["OUT"]
for n in ("final_logits", "final_logits_packed"):
    a, b = np.load(f"{OUT}/dump_base/{n}.npy"), np.load(f"{OUT}/dump_new/{n}.npy")
    print(n, a.shape, "byte-identical" if a.tobytes() == b.tobytes() else f"DIFFERENT (max |d| {np.abs(a - b).max()})")
PY
  # speed: bench.py's headline line, the two builds alternately
  for i in 1 2 3; do
    (cd $BASE_TREE && timeout 600 python bench.py --no-cpu-baseline --no-extras > $OUT/ab_base.json 2> /dev/null)
    timeout 600 python bench.py --no-cpu-baseline --no-extras > $OUT/ab_new.json 2> /dev/null
    for v in base new; do
      python -c "import json; d=json.load(open('$OUT/ab_$v.json')); print('$v', round(d['value']), round(d['packed']['value']), 'sm clock', d['clocks'])" >> $L 2>&1
    done
  done
  python - >> $L <<'PY'
import os, statistics
rows = [l.split() for l in open(os.environ["OUT"] + "/multi_sample_ab_r04.log") if l.startswith(("base ", "new "))]
for v in ("base", "new"):
    p = [float(r[1]) for r in rows if r[0] == v]; q = [float(r[2]) for r in rows if r[0] == v]
    print(v, "median value", statistics.median(p), "median packed", statistics.median(q), "runs", len(p))
PY
  cat $L
fi
if [[ " $PART " == *" bench "* ]]; then
  # P = 8 pockets x K = 8 samples against the replicated 64-graph batch
  timeout 1500 python scripts/multi_sample_bench.py --runs 3 > $OUT/multi_sample_bench_r04.log 2>&1
  tail -60 $OUT/multi_sample_bench_r04.log
  # device time per kernel of the step, replicated and shared (a separate profiler run)
  timeout 900 python scripts/loop_kernel_profile.py 50 8 > $OUT/multi_sample_kernels_r04.json 2> /dev/null
fi
exit 0
