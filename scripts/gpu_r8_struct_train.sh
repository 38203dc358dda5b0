# Structure-model training step (DESIGN.md 5b) on the GPU.  PART (default: all, in order):
#   tests  tests/test_struct_train.py on the product and the debug build, tests/test_train.py, the structure sampling tests
#   ab     against the parent commit: outputs of bench.py --workload cfg4 --dump-outputs (parent twice, this build once), flagship bench
#   bench  scripts/struct_train_bench.py (B = 64 and 128)
#   suite  the whole GPU suite and smoke()
# BASE_TREE = a checkout of the parent commit with its library built (python e3-invaraint-diffusion-model_b200/build.py there).  The debug library comes from SEQDIFF_DEBUG_BOUNDS=1 python
# e3-invaraint-diffusion-model_b200/build.py.  OUT = directory for the results (default: a new temporary directory).
set +e
export OUT=$(realpath -m ${OUT:-$(mktemp -d)})
mkdir -p "$OUT"
BASE_TREE=$(realpath ${BASE_TREE:-.parent_tree})
PART=${PART:-tests ab bench suite}
CARD="nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv"
S=$OUT/struct_train_r08.log
$CARD >> $S
if [[ " $PART " == *" tests "* ]]; then
  timeout 1200 python -m pytest tests/test_struct_train.py -q -rf -m gpu -p no:cacheprovider -s 2>&1 | grep -E "rel err|cosine|losses|resume|passed|failed|Error|error" | sed 's/^/struct_train : /' >> $S
  SEQDIFF_DEBUG_BOUNDS=1 timeout 1200 python -m pytest tests/test_struct_train.py -q -rf -m gpu -p no:cacheprovider 2>&1 | tail -6 |
    sed 's/^/debug build (SEQDIFF_DEBUG_BOUNDS=1) struct_train : /' >> $S
  timeout 1200 python -m pytest tests/test_train.py tests/test_structure_model.py tests/test_struct_packed.py tests/test_struct_multi_sample.py -q -rf -m gpu \
    -p no:cacheprovider 2>&1 | tail -6 | sed 's/^/train + structure sampling : /' >> $S
fi
if [[ " $PART " == *" ab "* ]]; then
  (cd $BASE_TREE && timeout 600 python bench.py --workload cfg4 --steps 2 --warmup 2 --no-cpu-baseline --no-extras --dump-outputs $OUT/cfg4_base1 > $OUT/cfg4_base1.json 2>&1)
  timeout 600 python bench.py --workload cfg4 --steps 2 --warmup 2 --no-cpu-baseline --no-extras --dump-outputs $OUT/cfg4_new > $OUT/cfg4_new.json 2>&1
  (cd $BASE_TREE && timeout 600 python bench.py --workload cfg4 --steps 2 --warmup 2 --no-cpu-baseline --no-extras --dump-outputs $OUT/cfg4_base2 > $OUT/cfg4_base2.json 2>&1)
  python - >> $S 2>&1 <<'PY'
import glob, os
import numpy as np
OUT = os.environ["OUT"]
for p in sorted(glob.glob(f"{OUT}/cfg4_base1/*.npy")):
    n = os.path.basename(p)
    a, b, c = np.load(p), np.load(f"{OUT}/cfg4_base2/{n}"), np.load(f"{OUT}/cfg4_new/{n}")
    f = lambda x, y: float(np.abs(x.astype(np.float64) - y.astype(np.float64)).max()) if x.size else 0.0
    print(f"cfg4 {n} {a.shape}: parent vs parent max |d| {f(a, b):.3e}; this build vs parent runs {f(c, a):.3e} / {f(c, b):.3e}")
PY
  for f in cfg4_base1 cfg4_new cfg4_base2; do echo "$f: $(tail -n 1 $OUT/$f.json | cut -c1-200)" >> $S; done
  for i in 1 2; do
    echo "bench parent: $(cd $BASE_TREE && timeout 900 python bench.py --gpus 1 --steps 5 --warmup 3 2>/dev/null | tail -n 1 | cut -c1-160)" >> $S
    echo "bench this  : $(timeout 900 python bench.py --gpus 1 --steps 5 --warmup 3 2>/dev/null | tail -n 1 | cut -c1-160)" >> $S
  done
fi
if [[ " $PART " == *" bench "* ]]; then
  timeout 1200 python scripts/struct_train_bench.py --steps 10 --warmup 3 > $OUT/struct_train_bench_r08.json 2> $OUT/struct_train_bench_r08.err
  echo "struct_train_bench: $(tail -n 1 $OUT/struct_train_bench_r08.json)" >> $S
  echo "GPUs visible: $(nvidia-smi -L | wc -l)" >> $S
fi
if [[ " $PART " == *" suite "* ]]; then
  timeout 2400 python -m pytest tests -q -rf -m gpu -p no:cacheprovider 2>&1 | tail -8 | sed 's/^/whole GPU suite : /' >> $S
  r=$(timeout 600 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -1); echo "smoke : $r" >> $S
fi
cat $S
