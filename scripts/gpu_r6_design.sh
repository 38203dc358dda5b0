# K backbones per pocket in the structure sampler and the design call (DESIGN.md 7b, 9) on the GPU.  PART (default: all three, in order):
#   tests  tests/test_struct_multi_sample.py and tests/test_design.py on the product and the debug build, the whole GPU suite, smoke()
#   ab     K = 1 against the parent commit: bench.py --dump-outputs files, seeded padded and packed structure p_sample_loop histories
#          at the struct_bench.py default, then bench.py and scripts/struct_packed_bench.py (workloads a, b) alternately, three runs each
#   bench  scripts/design_bench.py: P = 8 x K1 = 8 (x K2 = 8), three alternating runs each
# BASE_TREE = a checkout of the parent commit with its library built (python e3-invaraint-diffusion-model_b200/build.py there); the
# debug library comes from SEQDIFF_DEBUG_BOUNDS=1 python e3-invaraint-diffusion-model_b200/build.py.  OUT = directory for the
# results (default: a new temporary directory).
set +e
export OUT=$(realpath -m ${OUT:-$(mktemp -d)})
mkdir -p "$OUT"
BASE_TREE=$(realpath -m ${BASE_TREE:-_parent})
PART=${PART:-tests ab bench}
CARD="nvidia-smi --query-gpu=name,power.limit,clocks.max.sm --format=csv"
NEW_TESTS="tests/test_struct_multi_sample.py tests/test_design.py"
if [[ " $PART " == *" tests "* ]]; then
  S=$OUT/design_suite_r06.log
  $CARD >> $S
  timeout 1200 python -m pytest $NEW_TESTS -q -rf -m gpu -p no:cacheprovider 2>&1 | tail -8 | sed 's/^/new GPU tests : /' >> $S
  SEQDIFF_DEBUG_BOUNDS=1 timeout 1200 python -m pytest $NEW_TESTS -q -rf -m gpu -p no:cacheprovider 2>&1 | tail -8 |
    sed 's/^/debug build (SEQDIFF_DEBUG_BOUNDS=1) new GPU tests : /' >> $S
  [ -n "$SKIP_SUITE" ] || timeout 1800 python -m pytest tests -q -rf -m gpu -p no:cacheprovider 2>&1 | tail -8 | sed 's/^/whole GPU suite : /' >> $S
  r=$(timeout 600 python -c "import __graft_entry__ as g; g.smoke()" 2>&1 | tail -1); echo "smoke : $r" >> $S
  cat $S
fi
if [[ " $PART " == *" ab "* ]]; then
  L=$OUT/design_ab_r06.log
  $CARD > $L
  (cd $BASE_TREE && timeout 600 python bench.py --steps 1 --warmup 1 --no-cpu-baseline --no-extras --dump-outputs $OUT/dump_base > /dev/null 2>&1)
  timeout 600 python bench.py --steps 1 --warmup 1 --no-cpu-baseline --no-extras --dump-outputs $OUT/dump_new > /dev/null 2>&1
  python - >> $L 2>&1 <<'PY'
import os
OUT = os.environ["OUT"]
names = sorted(os.listdir(f"{OUT}/dump_base"))
assert names == sorted(os.listdir(f"{OUT}/dump_new")), "different dump file sets"
for n in names:
    a, b = open(f"{OUT}/dump_base/{n}", "rb").read(), open(f"{OUT}/dump_new/{n}", "rb").read()
    print("bench.py --dump-outputs", n, "byte-identical" if a == b else "DIFFERENT")
PY
  # the structure loop at the struct_bench.py default (64 complexes, L = 64, 12 + 12 layers, T = 1000, bf16, seeded Philox)
  for v in base new; do
    d=$([ $v = base ] && echo $BASE_TREE || echo .)
    (cd $d && timeout 600 python - > $OUT/struct_hist_$v.txt 2>&1 <<'PY'
import hashlib, math, sys, os
sys.path.insert(0, os.getcwd())
import torch
import seqdiff_b200 as sd
SM = sd.structure_model
B, L, T, Fs = 64, 64, 1000, 8
torch.manual_seed(0)
common = dict(max_position_embeddings=L, intermediate_size=1024, num_hidden_layers=12, position_embedding_type="relative_key")
m = SM.ConditionalBertForDiffusionBase(sd.BertConfig(**common), sd.BertConfig(**common, is_decoder=True, add_cross_attention=True), Fs)
for blk in (m.receptor_emb, m.timestep_emb):
    torch.nn.init.xavier_uniform_(blk.adaLN_modulation[0].weight)
m = m.eval().to("cuda:0")
m.precision = "bf16"
g = torch.Generator().manual_seed(3)
nl, nr = torch.randint(5, L + 1, (B,), generator=g), torch.randint(16, L + 1, (B,), generator=g)
pos = torch.arange(L)[None, :]
lm, rm = (pos < nl[:, None]).float(), (pos < nr[:, None]).float()
rseq = torch.nn.functional.one_hot(torch.randint(0, 20, (B, L), generator=g), 20).float() * rm[..., None]
rang = ((torch.rand(B, L, Fs, generator=g) * 2 - 1) * math.pi) * rm[..., None]
x_T = SM.modulo_with_wrapped_range(torch.randn(B, L, Fs, generator=g))
for packed in (False, True):
    h = SM.p_sample_loop(m, lm, x_T, rseq, rm, rang, T, SM.cosine_beta_schedule(T), seed=5, graph_id0=0, packed=packed)
    print("packed" if packed else "padded", tuple(h.shape), hashlib.sha256(h.numpy().tobytes()).hexdigest())
PY
    )
  done
  for mode in padded packed; do
    a=$(grep "^$mode " $OUT/struct_hist_base.txt); b=$(grep "^$mode " $OUT/struct_hist_new.txt)
    echo "structure p_sample_loop history: base $a | new $b | $([ -n "$a" ] && [ "$a" = "$b" ] && echo bitwise-equal || echo DIFFERENT)" >> $L
  done
  # speed: bench.py's headline line and struct_packed_bench.py, the two builds alternately
  for i in 1 2 3; do
    (cd $BASE_TREE && timeout 600 python bench.py --no-cpu-baseline --no-extras > $OUT/ab_base.json 2> /dev/null)
    timeout 600 python bench.py --no-cpu-baseline --no-extras > $OUT/ab_new.json 2> /dev/null
    for v in base new; do
      python -c "import json; d=json.load(open('$OUT/ab_$v.json')); print('$v', round(d['value']), round(d['packed']['value']), 'sm clock', d['clocks'])" >> $L 2>&1
    done
  done
  for i in 1 2 3; do
    (cd $BASE_TREE && timeout 600 python scripts/struct_packed_bench.py --runs 1 --workloads ab > $OUT/sp_base.log 2>&1)
    timeout 600 python scripts/struct_packed_bench.py --runs 1 --workloads ab > $OUT/sp_new.log 2>&1
    for v in base new; do
      python - $v $OUT/sp_$v.log >> $L 2>&1 <<'PY'
import json, sys
for line in open(sys.argv[2]):
    d = json.loads(line)
    for k, w in d.items():
        if k != "gpu":
            print("struct_packed_bench", sys.argv[1], k, round(w["padded_graph_steps_per_s"]), round(w["packed_graph_steps_per_s"]))
PY
    done
  done
  python - >> $L <<'PY'
import os, statistics
lines = open(os.environ["OUT"] + "/design_ab_r06.log").read().splitlines()
rows = [l.split() for l in lines if l.startswith(("base ", "new "))]
for v in ("base", "new"):
    p = [float(r[1]) for r in rows if r[0] == v]; q = [float(r[2]) for r in rows if r[0] == v]
    print(v, "bench.py median value", statistics.median(p), "median packed", statistics.median(q), "runs", len(p))
sp = [l.split() for l in lines if l.startswith("struct_packed_bench ")]
for v in ("base", "new"):
    for w in sorted({r[2] for r in sp}):
        p = [float(r[3]) for r in sp if r[1] == v and r[2] == w]; q = [float(r[4]) for r in sp if r[1] == v and r[2] == w]
        print(v, "struct_packed_bench", w, "median padded", statistics.median(p), "median packed", statistics.median(q), "runs", len(p))
PY
  cat $L
fi
if [[ " $PART " == *" bench "* ]]; then
  timeout 1500 python scripts/design_bench.py --runs 3 --out $OUT > $OUT/design_bench_r06.log 2>&1
  tail -20 $OUT/design_bench_r06.log
fi
exit 0
