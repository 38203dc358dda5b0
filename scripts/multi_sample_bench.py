"""K sequences per pocket: P pockets x K samples through seqdiff_sample_multi (denoise_tensors(num_samples=K)) against the same
P*K graphs as one replicated batch through seqdiff_sample_ex, bf16, padded and packed.

    python scripts/multi_sample_bench.py [--pockets 8] [--samples 8] [--T 500] [--runs 3]

Shapes: "cfg2" = bench.py's synthetic_workload pockets (n_lig ~ U{5..64}, n_rec ~ U{16..128}, L = 128); "design" = peptides of
10-20 residues in pockets of 80-128 residues (L = 128).  Each form runs on its own model handle (same weights), so each keeps its
own captured step graph; every (shape, mode, form) is warmed up once, then the two forms alternate, --runs times each, timed with
CUDA events around a whole T-step sampling (the per-sampling receptor work included).  The outputs of the two forms are compared
at the timed sizes (padded: every position, packed: the valid ones).  Prints the card name, its power limit and the SM clock, one
line per run and a JSON summary with the medians in graph-steps/s (P*K graphs x T steps / time)."""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402
import seqdiff_b200 as sd  # noqa: E402

SHAPES = {"cfg2": dict(n_lig=(5, 64), n_rec=(16, 128)), "design": dict(n_lig=(10, 20), n_rec=(80, 128))}


def smi(q):
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return r.stdout.strip()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pockets", type=int, default=8)
    ap.add_argument("--samples", type=int, default=8)
    ap.add_argument("--T", type=int, default=500)
    ap.add_argument("--runs", type=int, default=3)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("multi_sample_bench.py needs a CUDA device")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    P, K, T = a.pockets, a.samples, a.T
    bench.L = 128
    print("card:", smi("name,power.limit,clocks.max.sm"), flush=True)
    torch.manual_seed(0)
    common = dict(max_position_embeddings=128, intermediate_size=bench.I, num_hidden_layers=bench.NL, position_embedding_type="relative_key")
    models = {}
    for form in ("replicated", "shared"):
        m = sd.ConditionalBertForDiffusionBase(sd.BertConfig(**common), sd.BertConfig(**common, is_decoder=True, add_cross_attention=True), 20)
        if models:
            m.load_state_dict(models["replicated"].state_dict())
        models[form] = m.eval().to(dev)
        models[form].precision = "bf16"
    sched, trans = sd.PredefinedNoiseScheduleDiscrete("cosine", T), sd.BlosumTransition(x_classes=20, timestep=500)
    cases = []
    for shape, kw in SHAPES.items():
        pockets, _ = bench.synthetic_workload(P, **kw)
        pockets.pop("structure_ids")
        x_T = torch.nn.functional.one_hot(torch.randint(0, 20, (P * K, 128), generator=torch.Generator().manual_seed(9)), 20).float().to(dev)
        shared = {k: v.to(dev) for k, v in pockets.items()}
        replicated = {k: v.repeat_interleave(K, dim=0) for k, v in shared.items()}
        for packed in (False, True):
            cases.append((shape, packed, shared, replicated, x_T))

    def run(form, case):
        shape, packed, shared, replicated, x_T = case
        b, k = (shared, K) if form == "shared" else (replicated, 1)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        out = sd.denoise_tensors(b, models[form], sched, trans, True, timesteps=T, x_T=x_T, seed=5, graph_id0=0, packed=packed, num_samples=k)
        e1.record()
        torch.cuda.synchronize()
        return out, e0.elapsed_time(e1)

    summary = {"card": smi("name,power.limit"), "P": P, "K": K, "T": T, "precision": "bf16", "cases": {}}
    for case in cases:
        shape, packed = case[0], case[1]
        name = f"{shape}_{'packed' if packed else 'padded'}"
        outs = {form: run(form, case)[0] for form in ("replicated", "shared")}  # warm-up: captures both step graphs
        if packed:
            valid = case[3]["ligand_attn_mask"].bool()
            equal = torch.equal(outs["shared"][valid], outs["replicated"][valid]) and bool((outs["shared"][~valid] == 0).all())
        else:
            equal = torch.equal(outs["shared"], outs["replicated"])
        ms = {"replicated": [], "shared": []}
        for i in range(a.runs):
            for form in ("replicated", "shared"):
                out, t = run(form, case)
                ms[form].append(t)
                print(f"{name} run {i} {form}: {t:.1f} ms  {P * K * T / t * 1e3:.0f} graph-steps/s  sm clock {smi('clocks.sm')}", flush=True)
        med = {f: statistics.median(v) for f, v in ms.items()}
        rate = {f: P * K * T / med[f] * 1e3 for f in med}
        summary["cases"][name] = {"outputs_equal": equal, "median_ms": {f: round(v, 2) for f, v in med.items()},
                                  "graph_steps_per_s": {f: round(v) for f, v in rate.items()},
                                  "speedup": round(rate["shared"] / rate["replicated"], 3), "runs": a.runs}
        print(name, "outputs equal:", equal, "median graph-steps/s replicated", round(rate["replicated"]), "shared", round(rate["shared"]),
              "speed-up", round(rate["shared"] / rate["replicated"], 3), flush=True)
    print(json.dumps(summary, indent=1))


if __name__ == "__main__":
    main()
