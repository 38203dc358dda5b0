# Backbone score (DESIGN.md 7b) on the GPU.  PART (default: all, in order):
#   tests  tests/test_struct_score.py on the product and the debug build, then the whole GPU suite and smoke() on both
#   ab     the structure sampler against the parent commit: final angles of p_sample_loop (64 complexes, padded and packed, T = 1000)
#          byte for byte, scripts/struct_packed_bench.py (workload a) alternately, two runs each, and the flagship bench.py alternately
#   bench  scripts/struct_score_bench.py (64 complexes padded / packed, P = 8 x K = 8; plain-PyTorch arm)
# BASE_TREE = a checkout of the parent commit with its library built (python e3-invaraint-diffusion-model_b200/build.py there).  The debug
# library comes from SEQDIFF_DEBUG_BOUNDS=1 python e3-invaraint-diffusion-model_b200/build.py.  OUT = directory for the results (default:
# a new temporary directory).
set +e
export OUT=$(realpath -m ${OUT:-$(mktemp -d)})
mkdir -p "$OUT"
BASE_TREE=$(realpath ${BASE_TREE:-.parent_tree})
PART=${PART:-tests ab bench}
CARD="nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv"
S=$OUT/struct_score_r10.log
$CARD >> $S
if [[ " $PART " == *" tests "* ]]; then
  timeout 1200 python -m pytest tests/test_struct_score.py -q -rf -m gpu -p no:cacheprovider -s 2>&1 |
    grep -E "struct score|design backbone|passed|failed|Error|error|assert" | sed 's/^/struct score : /' >> $S
  SEQDIFF_DEBUG_BOUNDS=1 timeout 1200 python -m pytest tests/test_struct_score.py -q -rf -m gpu -p no:cacheprovider 2>&1 | tail -6 |
    sed 's/^/debug build (SEQDIFF_DEBUG_BOUNDS=1) struct score : /' >> $S
  timeout 1800 python -m pytest tests -q -rf -m gpu -p no:cacheprovider 2>&1 | tail -8 | sed 's/^/whole GPU suite : /' >> $S
  SEQDIFF_DEBUG_BOUNDS=1 timeout 1800 python -m pytest tests -q -rf -m gpu -p no:cacheprovider 2>&1 | tail -8 |
    sed 's/^/debug build (SEQDIFF_DEBUG_BOUNDS=1) whole GPU suite : /' >> $S
  r=$(timeout 600 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -1); echo "smoke : $r" >> $S
  r=$(SEQDIFF_DEBUG_BOUNDS=1 timeout 600 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -1); echo "debug build smoke : $r" >> $S
fi
if [[ " $PART " == *" ab "* ]]; then
  DUMP='
import os, sys, numpy as np, torch
sys.path.insert(0, os.getcwd()); sys.path.insert(0, os.path.join(os.getcwd(), "scripts"))
import seqdiff_b200 as sd, struct_packed_bench as B
SM = sd.structure_model
torch.manual_seed(0)
common = dict(max_position_embeddings=64, intermediate_size=1024, num_hidden_layers=12, position_embedding_type="relative_key")
m = SM.ConditionalBertForDiffusionBase(sd.BertConfig(**common), sd.BertConfig(**common, is_decoder=True, add_cross_attention=True), 8)
for blk in (m.receptor_emb, m.timestep_emb):
    torch.nn.init.xavier_uniform_(blk.adaLN_modulation[0].weight)
m = m.eval().to("cuda:0"); m.precision = "bf16"
lm, rm, rseq, rang, x_T = (t.cuda() for t in B.inputs(64, (5, 64), (16, 64), 3))
for packed in (False, True):
    f = SM.p_sample_loop(m, lm, x_T, rseq, rm, rang, 1000, SM.cosine_beta_schedule(1000), seed=5, graph_id0=0, keep_history=False, packed=packed)
    np.save(os.path.join(sys.argv[1], f"final_{int(packed)}.npy"), f.numpy())
'
  mkdir -p $OUT/base1 $OUT/new $OUT/base2
  (cd $BASE_TREE && timeout 600 python -c "$DUMP" $OUT/base1 > $OUT/base1.log 2>&1)
  timeout 600 python -c "$DUMP" $OUT/new > $OUT/new.log 2>&1
  (cd $BASE_TREE && timeout 600 python -c "$DUMP" $OUT/base2 > $OUT/base2.log 2>&1)
  python - >> $S 2>&1 <<'PY'
import glob, os
import numpy as np
OUT = os.environ["OUT"]
for p in sorted(glob.glob(f"{OUT}/base1/*.npy")):
    n = os.path.basename(p)
    a, b, c = np.load(p), np.load(f"{OUT}/base2/{n}"), np.load(f"{OUT}/new/{n}")
    print(f"struct sampler {n} {a.shape}: parent runs identical {a.tobytes() == b.tobytes()}; this build byte-identical to the parent {c.tobytes() == a.tobytes()}")
PY
  for i in 1 2; do
    echo "struct_packed_bench parent: $(cd $BASE_TREE && timeout 900 python scripts/struct_packed_bench.py --runs 3 --workloads a 2>&1 | grep '"a"' | python -c 'import json,sys; d=json.loads(sys.stdin.read())["a"]; print({k: d[k] for k in ("padded_graph_steps_per_s", "packed_graph_steps_per_s", "kernels_per_step")})')" >> $S
    echo "struct_packed_bench this  : $(timeout 900 python scripts/struct_packed_bench.py --runs 3 --workloads a 2>&1 | grep '"a"' | python -c 'import json,sys; d=json.loads(sys.stdin.read())["a"]; print({k: d[k] for k in ("padded_graph_steps_per_s", "packed_graph_steps_per_s", "kernels_per_step")})')" >> $S
  done
  for i in 1 2; do
    echo "bench parent: $(cd $BASE_TREE && timeout 900 python bench.py --gpus 1 --steps 5 --warmup 3 --no-cpu-baseline 2>/dev/null | tail -n 1 | cut -c1-200)" >> $S
    echo "bench this  : $(timeout 900 python bench.py --gpus 1 --steps 5 --warmup 3 --no-cpu-baseline 2>/dev/null | tail -n 1 | cut -c1-200)" >> $S
  done
fi
if [[ " $PART " == *" bench "* ]]; then
  timeout 1200 python scripts/struct_score_bench.py --T 1000 --runs 3 --torch-T 5 --out $OUT/struct_score_bench_r10.json > $OUT/struct_score_bench_r10.log 2>&1
  echo "struct_score_bench: $(grep -E '^(c64|P8|torch)' $OUT/struct_score_bench_r10.log)" >> $S
fi
cat $S
