# Sampling-loop invariants (DESIGN.md 7b): the parent commit's library against this one, alternately in one GPU session.
# BASE = the parent's library, built from its checkout with SEQDIFF_VARIANT=base (python e3-invaraint-diffusion-model_b200/build.py)
# and copied next to the product build.  OUT = directory for the results (default: a new temporary directory).
set +e
export OUT=${OUT:-$(mktemp -d)}
mkdir -p "$OUT"
BASE=${BASE:-e3-invaraint-diffusion-model_b200/libseqdiff_b200_base.so}
L=$OUT/loop_invariants_ab_r03.log
nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv > $L
# outputs: the final logits of the padded and the packed sampling, old against new
for v in base new; do
  if [ $v = base ]; then export SEQDIFF_LIB=$BASE; else unset SEQDIFF_LIB; fi
  timeout 600 python bench.py --steps 1 --warmup 1 --no-cpu-baseline --no-extras --dump-outputs $OUT/dump_$v > /dev/null 2>&1
done
unset SEQDIFF_LIB
python - >> $L 2>&1 <<'PY'
import os
import numpy as np
OUT = os.environ["OUT"]
for n in ("final_logits", "final_logits_packed"):
    a, b = np.load(f"{OUT}/dump_base/{n}.npy"), np.load(f"{OUT}/dump_new/{n}.npy")
    print(n, a.shape, "byte-identical" if a.tobytes() == b.tobytes() else f"DIFFERENT (max |d| {np.abs(a - b).max()})")
PY
# speed: headline line, the two libraries alternately
for i in 1 2 3 4; do
  for v in base new; do
    if [ $v = base ]; then export SEQDIFF_LIB=$BASE; else unset SEQDIFF_LIB; fi
    timeout 600 python bench.py --no-cpu-baseline --no-extras > $OUT/ab_$v.json 2> /dev/null
    python -c "import json; d=json.load(open('$OUT/ab_$v.json')); print('$v', round(d['value']), round(d['packed']['value']), 'ms/step', round(d['ms_per_step'] / 500, 4), round(d['packed']['ms_per_step'] / 500, 4), 'launches/step', d['gpu_launches'] / d['steps'] / 500, 'sm clock', d['clocks'])" >> $L 2>&1
  done
done
unset SEQDIFF_LIB
python - >> $L <<'PY'
import os, statistics
rows = [l.split() for l in open(os.environ["OUT"] + "/loop_invariants_ab_r03.log") if l.startswith(("base ", "new "))]
for v in ("base", "new"):
    p = [float(r[1]) for r in rows if r[0] == v]; q = [float(r[2]) for r in rows if r[0] == v]
    print(v, "median value", statistics.median(p), "median packed", statistics.median(q), "runs", len(p))
PY
# per-kernel device time of the loop's step (padded and packed), both libraries
SEQDIFF_LIB=$BASE timeout 600 python scripts/loop_kernel_profile.py 50 > $OUT/loop_kernels_base_r03.json 2> /dev/null
timeout 600 python scripts/loop_kernel_profile.py 50 > $OUT/loop_kernels_r03.json 2> /dev/null
cat $L
