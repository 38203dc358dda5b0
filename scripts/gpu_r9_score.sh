# Sequence score (DESIGN.md 7b) on the GPU.  PART (default: all, in order):
#   tests  tests/test_score.py on the product and the debug build, then the whole GPU suite and smoke() on both
#   ab     against the parent commit: outputs of bench.py --workload cfg2 --dump-outputs (parent twice, this build once), flagship bench
#          alternately, two runs each
#   bench  scripts/score_bench.py (cfg-2 padded / packed, P = 8 x K = 8; plain-PyTorch arm)
# BASE_TREE = a checkout of the parent commit with its library built (python e3-invaraint-diffusion-model_b200/build.py there).  The debug
# library comes from SEQDIFF_DEBUG_BOUNDS=1 python e3-invaraint-diffusion-model_b200/build.py.  OUT = directory for the results (default:
# a new temporary directory).
set +e
export OUT=$(realpath -m ${OUT:-$(mktemp -d)})
mkdir -p "$OUT"
BASE_TREE=$(realpath ${BASE_TREE:-.parent_tree})
PART=${PART:-tests ab bench}
CARD="nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv"
S=$OUT/score_r09.log
$CARD >> $S
if [[ " $PART " == *" tests "* ]]; then
  timeout 1200 python -m pytest tests/test_score.py -q -rf -m gpu -p no:cacheprovider -s 2>&1 | grep -E "score |passed|failed|Error|error" | sed 's/^/score : /' >> $S
  SEQDIFF_DEBUG_BOUNDS=1 timeout 1200 python -m pytest tests/test_score.py -q -rf -m gpu -p no:cacheprovider 2>&1 | tail -6 |
    sed 's/^/debug build (SEQDIFF_DEBUG_BOUNDS=1) score : /' >> $S
  timeout 1800 python -m pytest tests -q -rf -m gpu -p no:cacheprovider 2>&1 | tail -8 | sed 's/^/whole GPU suite : /' >> $S
  SEQDIFF_DEBUG_BOUNDS=1 timeout 1800 python -m pytest tests -q -rf -m gpu -p no:cacheprovider 2>&1 | tail -8 |
    sed 's/^/debug build (SEQDIFF_DEBUG_BOUNDS=1) whole GPU suite : /' >> $S
  r=$(timeout 600 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -1); echo "smoke : $r" >> $S
  r=$(SEQDIFF_DEBUG_BOUNDS=1 timeout 600 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -1); echo "debug build smoke : $r" >> $S
fi
if [[ " $PART " == *" ab "* ]]; then
  (cd $BASE_TREE && timeout 600 python bench.py --workload cfg2 --steps 2 --warmup 2 --no-cpu-baseline --no-extras --dump-outputs $OUT/cfg2_base1 > $OUT/cfg2_base1.json 2>&1)
  timeout 600 python bench.py --workload cfg2 --steps 2 --warmup 2 --no-cpu-baseline --no-extras --dump-outputs $OUT/cfg2_new > $OUT/cfg2_new.json 2>&1
  (cd $BASE_TREE && timeout 600 python bench.py --workload cfg2 --steps 2 --warmup 2 --no-cpu-baseline --no-extras --dump-outputs $OUT/cfg2_base2 > $OUT/cfg2_base2.json 2>&1)
  python - >> $S 2>&1 <<'PY'
import glob, os
import numpy as np
OUT = os.environ["OUT"]
for p in sorted(glob.glob(f"{OUT}/cfg2_base1/*.npy")):
    n = os.path.basename(p)
    a, b, c = np.load(p), np.load(f"{OUT}/cfg2_base2/{n}"), np.load(f"{OUT}/cfg2_new/{n}")
    print(f"cfg2 {n} {a.shape}: parent runs identical {np.array_equal(a, b)}; this build identical to the parent {np.array_equal(c, a)}")
PY
  for i in 1 2; do
    echo "bench parent: $(cd $BASE_TREE && timeout 900 python bench.py --gpus 1 --steps 5 --warmup 3 --no-cpu-baseline 2>/dev/null | tail -n 1 | cut -c1-160)" >> $S
    echo "bench this  : $(timeout 900 python bench.py --gpus 1 --steps 5 --warmup 3 --no-cpu-baseline 2>/dev/null | tail -n 1 | cut -c1-160)" >> $S
  done
fi
if [[ " $PART " == *" bench "* ]]; then
  timeout 1200 python scripts/score_bench.py --T 500 --runs 3 --torch-T 10 --out $OUT/score_bench_r09.json > $OUT/score_bench_r09.log 2>&1
  echo "score_bench: $(grep -E '^(cfg2|P8|torch)' $OUT/score_bench_r09.log)" >> $S
fi
cat $S
