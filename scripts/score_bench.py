"""Sequence scoring (seqdiff_score_multi through score_tensors) against sampling (denoise_tensors) on the same batches, bf16, and a
plain-PyTorch arm: the oracle's score loop (tests/score_oracle.py) on the same GPU under bf16 autocast.

    python scripts/score_bench.py [--T 500] [--runs 3] [--torch-T 10] [--out profiles/score_bench_r09.json]

Cases: bench.py's cfg-2 batch (64 pockets, n_lig ~ U{5..64}, n_rec ~ U{16..128}, L = 128) padded and packed, and P = 8 pockets x K = 8
candidate sequences per pocket (packed).  One model handle serves both calls, so the score's and the sampler's step graphs are cached
side by side; every case is warmed up once per call, then the two calls alternate, --runs times each, timed with CUDA events around
the whole T-step loop (the per-call receptor work included).  Launches per step = library kernel launches of a warm call / T.  The
PyTorch arm runs --torch-T steps of the loop (x_t, forward, per-residue terms; seconds, not minutes) on the cfg-2 batch.  The card's
name and power limit are read in the same run; the JSON goes to --out."""
import argparse
import json
import os
import statistics
import subprocess
import sys

import torch
import torch.nn.functional as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import bench  # noqa: E402
import score_oracle as SO  # noqa: E402
import seqdiff_b200 as sd  # noqa: E402
from helpers import O, make_model  # noqa: E402


def smi(q):
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return r.stdout.strip()


def torch_score_steps(state, cfg, batch, x0, sched, tr, T, steps, dev):
    """the oracle's score loop on the device under bf16 autocast, steps k = T-1 .. T-steps; returns (ms, terms)"""
    B, L, C = x0.shape
    g = torch.Generator(device=dev).manual_seed(1)
    terms = torch.zeros((B * L, 2), dtype=torch.float64, device=dev)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for k in range(T - 1, T - 1 - steps, -1):
        t, s, Qt, Qsb, Qtb = (x.to(dev) for x in SO.step_tables(k, T, B, sched, tr))
        x_t = SO.q_sample(x0, Qtb, torch.empty(B * L, C, device=dev).exponential_(1, generator=g))
        with torch.autocast("cuda", dtype=torch.bfloat16):
            logits = O.denoiser_forward(state, cfg, k * torch.ones((B, 1), device=dev), x_t, batch["ligand_angles"], batch["ligand_attn_mask"],
                                        batch["receptor_seq"], batch["receptor_angles"], batch["receptor_attn_mask"]).float()
        a = x0.reshape(B * L, C).argmax(-1)
        ce = -F.log_softmax(logits.reshape(B * L, C).double(), -1).gather(1, a[:, None]).squeeze(1)
        p = SO.posterior_probs(F.softmax(logits.reshape(B * L, C), -1), x_t, Qt, Qsb, Qtb)
        q = SO.posterior_probs(F.one_hot(a, C).float(), x_t, Qt, Qsb, Qtb)
        terms[:, 0] += SO.kl_terms(q, p) if k > 0 else ce
        terms[:, 1] += ce
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1), terms


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--T", type=int, default=500)
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--torch-T", type=int, default=10)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "score_bench_r09.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("score_bench.py needs a CUDA device")
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    T = a.T
    bench.L = 128
    card = smi("name,power.limit,clocks.max.sm")
    print("card:", card, flush=True)
    cfg = O.OracleConfig(max_position_embeddings=128, relative_key=True)
    state = O.init_state_dict(cfg, 1, "B")
    m = make_model(sd, cfg, state, "bf16")
    sched, trans = sd.PredefinedNoiseScheduleDiscrete("cosine", T), sd.BlosumTransition(x_classes=20, timestep=500)
    lib = sd.lib()
    cases = []
    cfg2, _ = bench.synthetic_workload(64)
    cfg2.pop("structure_ids")
    cfg2 = {k: v.to(dev) for k, v in cfg2.items()}
    cases += [("cfg2_padded", cfg2, 1, False), ("cfg2_packed", cfg2, 1, True)]
    pk8, _ = bench.synthetic_workload(8, seed_offset=1)
    pk8.pop("structure_ids")
    cases.append(("P8xK8_packed", {k: v.to(dev) for k, v in pk8.items()}, 8, True))

    def run(kind, case):
        _, b, K, packed = case
        P, L = b["ligand_seq"].shape[:2]
        torch.cuda.synchronize()
        n0 = lib.seqdiff_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        if kind == "score":
            seqs = b["ligand_seq"] if K == 1 else F.one_hot(torch.randint(0, 20, (P * K, L), generator=torch.Generator().manual_seed(3)),
                                                            20).float().to(dev)
            sd.score_tensors(b, m, sched, trans, sequences=seqs, timesteps=T, seed=5, graph_id0=0, packed=packed, num_samples=K)
        else:
            x_T = F.one_hot(torch.randint(0, 20, (P * K, L), generator=torch.Generator().manual_seed(9)), 20).float().to(dev)
            sd.denoise_tensors(b, m, sched, trans, True, timesteps=T, x_T=x_T, seed=5, graph_id0=0, packed=packed, num_samples=K)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), (lib.seqdiff_launch_count() - n0) / T

    summary = {"card": card, "T": T, "precision": "bf16", "model": "H 768, 6 decoder layers, relative_key, L 128", "cases": {}}
    for case in cases:
        name, b, K = case[0], case[1], case[2]
        G = b["ligand_seq"].shape[0] * K
        for kind in ("sample", "score"):
            run(kind, case)  # warm-up: captures the step graph of each kind
        ms, launches = {"sample": [], "score": []}, {}
        for i in range(a.runs):
            for kind in ("sample", "score"):
                t, n = run(kind, case)
                ms[kind].append(t)
                launches[kind] = n
                print(f"{name} run {i} {kind}: {t:.1f} ms  {G * T / t * 1e3:.0f} graph-steps/s  {n:.2f} launches/step  sm clock {smi('clocks.sm')}",
                      flush=True)
        med = {k: statistics.median(v) for k, v in ms.items()}
        rate = {k: G * T / med[k] * 1e3 for k in med}
        summary["cases"][name] = {"graphs": G, "median_ms": {k: round(v, 2) for k, v in med.items()},
                                  "graph_steps_per_s": {k: round(v) for k, v in rate.items()},
                                  "score_over_sample_time": round(med["score"] / med["sample"], 3),
                                  "launches_per_step": {k: round(v, 2) for k, v in launches.items()},
                                  "spread_ms": {k: [round(min(v), 2), round(max(v), 2)] for k, v in ms.items()}, "runs": a.runs}
        print(name, json.dumps(summary["cases"][name]), flush=True)
    # plain PyTorch: the oracle's loop on the device, bf16 autocast, on the cfg-2 batch
    gstate = {k: v.to(dev) for k, v in state.items()}
    osched, otr = O.NoiseScheduleDiscrete("cosine", T), O.BlosumTransition()
    with torch.no_grad():
        torch_score_steps(gstate, cfg, cfg2, cfg2["ligand_seq"], osched, otr, T, 2, dev)  # warm-up
        t, _ = torch_score_steps(gstate, cfg, cfg2, cfg2["ligand_seq"], osched, otr, T, a.torch_T, dev)
    G = cfg2["ligand_seq"].shape[0]
    summary["torch_arm"] = {"what": "tests/score_oracle.py loop on the GPU, bf16 autocast, cfg2 batch (padded)", "steps": a.torch_T,
                            "ms": round(t, 1), "graph_steps_per_s": round(G * a.torch_T / t * 1e3)}
    summary["torch_arm"]["cuda_score_speedup"] = round(summary["cases"]["cfg2_padded"]["graph_steps_per_s"]["score"] /
                                                       summary["torch_arm"]["graph_steps_per_s"], 1)
    print("torch arm:", json.dumps(summary["torch_arm"]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(summary, f, indent=1)
    print(json.dumps(summary, indent=1))


if __name__ == "__main__":
    main()
