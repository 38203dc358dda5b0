# Padded sampling loop on the valid receptor rows only (DESIGN.md 7b) on the GPU.  PART (default: all three, in order):
#   tests  tests/test_receptor_rows.py and the whole GPU suite on the product and the debug build, smoke() on both
#   ab     against the parent commit: final logits of bench.py --dump-outputs, then bench.py alternately, three runs each
#   prof   per-position device time of the cfg-2 step, parent and this build (scripts/loop_kernel_profile.py 50)
# BASE_LIB = the parent commit's library (python e3-invaraint-diffusion-model_b200/build.py in a checkout of it, copied next to
# the product library; the Python side is the same).  The debug library comes from SEQDIFF_DEBUG_BOUNDS=1 python
# e3-invaraint-diffusion-model_b200/build.py.  OUT = directory for the results (default: a new temporary directory).
set +e
export OUT=$(realpath -m ${OUT:-$(mktemp -d)})
mkdir -p "$OUT"
BASE_LIB=$(realpath ${BASE_LIB:-e3-invaraint-diffusion-model_b200/libseqdiff_b200_parent.so})
PART=${PART:-tests ab prof}
CARD="nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv"
if [[ " $PART " == *" tests "* ]]; then
  S=$OUT/receptor_rows_suite_r07.log
  $CARD >> $S
  timeout 900 python -m pytest tests/test_receptor_rows.py -q -rf -m gpu -p no:cacheprovider 2>&1 | tail -6 | sed 's/^/receptor_rows : /' >> $S
  SEQDIFF_DEBUG_BOUNDS=1 timeout 900 python -m pytest tests/test_receptor_rows.py -q -rf -m gpu -p no:cacheprovider 2>&1 | tail -6 |
    sed 's/^/debug build (SEQDIFF_DEBUG_BOUNDS=1) receptor_rows : /' >> $S
  timeout 1200 python -m pytest tests -q -rf -m gpu -p no:cacheprovider 2>&1 | tail -8 | sed 's/^/whole GPU suite : /' >> $S
  SEQDIFF_DEBUG_BOUNDS=1 timeout 1200 python -m pytest tests -q -rf -m gpu -p no:cacheprovider 2>&1 | tail -8 |
    sed 's/^/debug build (SEQDIFF_DEBUG_BOUNDS=1) whole GPU suite : /' >> $S
  r=$(timeout 600 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -1); echo "smoke : $r" >> $S
  r=$(SEQDIFF_DEBUG_BOUNDS=1 timeout 600 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -1); echo "debug build smoke : $r" >> $S
  cat $S
fi
if [[ " $PART " == *" ab "* ]]; then
  L=$OUT/receptor_rows_ab_r07.log
  $CARD > $L
  # the final logits of the padded and the packed sampling, parent against this build
  SEQDIFF_LIB=$BASE_LIB timeout 600 python bench.py --steps 1 --warmup 1 --no-cpu-baseline --no-extras --dump-outputs $OUT/dump_base > /dev/null 2>&1
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
    SEQDIFF_LIB=$BASE_LIB timeout 600 python bench.py --no-cpu-baseline --no-extras > $OUT/ab_base_$i.json 2> /dev/null
    timeout 600 python bench.py --no-cpu-baseline --no-extras > $OUT/ab_new_$i.json 2> /dev/null
    for v in base new; do
      python -c "import json; d=json.load(open('$OUT/ab_${v}_$i.json')); print('$v', round(d['value']), round(d['packed']['value']), 'launches', d['gpu_launches'], 'sm clock', d['clocks'])" >> $L 2>&1
    done
  done
  python - >> $L <<'PY'
import os, statistics
rows = [l.split() for l in open(os.environ["OUT"] + "/receptor_rows_ab_r07.log") if l.startswith(("base ", "new "))]
for v in ("base", "new"):
    p = [float(r[1]) for r in rows if r[0] == v]; q = [float(r[2]) for r in rows if r[0] == v]
    print(v, "value median", statistics.median(p), "range", min(p), max(p), "| packed median", statistics.median(q), "range", min(q), max(q), "| runs", len(p))
PY
  cat $L
fi
if [[ " $PART " == *" prof "* ]]; then
  # device time per kernel and per position of the step (a separate profiler run per library)
  SEQDIFF_LIB=$BASE_LIB timeout 900 python scripts/loop_kernel_profile.py 50 > $OUT/receptor_rows_kernels_base_r07.json 2> $OUT/prof_base.err
  timeout 900 python scripts/loop_kernel_profile.py 50 > $OUT/receptor_rows_kernels_r07.json 2> $OUT/prof_new.err
  python - <<'PY' 2>&1 | tee $OUT/receptor_rows_attribution_r07.txt
import json, os
OUT = os.environ["OUT"]
a, b = (json.load(open(f"{OUT}/{n}.json")) for n in ("receptor_rows_kernels_base_r07", "receptor_rows_kernels_r07"))
for mode in ("padded", "packed"):
    pa, pb = a[mode]["by_position"], b[mode]["by_position"]
    print(mode, "us/step", a[mode]["us_per_step"], "->", b[mode]["us_per_step"], "| positions", len(pa), len(pb))
    if mode == "padded" and len(pa) == len(pb):
        for i, (x, y) in enumerate(zip(pa, pb)):
            if abs(x["us"] - y["us"]) > 1.5:
                print(f"  {i:3d} {x['kernel']:28s} {str(x['grid']):16s} {x['us']:8.2f} -> {str(y['grid']):16s} {y['us']:8.2f}")
PY
fi
exit 0
