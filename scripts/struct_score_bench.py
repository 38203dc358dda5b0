#!/usr/bin/env python
"""Backbone scoring (seqdiff_struct_score_multi through structure_model.score_backbones_tensors) against structure sampling
(p_sample_loop_tensors) on the same batches, bf16, and a plain-PyTorch arm: the oracle's score loop (tests/struct_score_oracle.py) on the
same GPU under bf16 autocast.

    python scripts/struct_score_bench.py [--T 1000] [--runs 3] [--torch-T 5] [--out profiles/struct_score_bench_r10.json]

Model: scripts/struct_bench.py's (12 + 12 layers, H 768, relative_key, 8 angle features, L = 64, no SELayer is an identity).  Cases:
struct_bench's default batch of 64 complexes (ligand lengths U(5..64), receptor lengths U(16..64)) padded and packed, and the design
shape of P = 8 pockets x K = 8 backbones per pocket (packed).  One model handle serves both calls, so the score's and the sampler's step
graphs are cached side by side; every case is warmed up once per call, then the two calls alternate, --runs times each, each timed with
CUDA events around the whole call (the per-call receptor branch included; sampling keeps only the final angles).  Kernels per step =
library kernel launches of a warm call // T (the receptor branch, run once per call, adds fewer than T launches).  The PyTorch arm runs
--torch-T steps of the oracle loop (q-sample, forward, per-element terms) on the 64-complex batch.  The card's name and power limit
are read in the same run; the JSON goes to --out."""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys

import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import struct_score_oracle as SSO  # noqa: E402
from oracle import structdiff_oracle as S  # noqa: E402

L, FS = 64, 8


def smi(q):
    r = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader", "-i", "0"], capture_output=True, text=True)
    return r.stdout.strip()


def inputs(P, K, nl_rng, nr_rng, seed):
    """ligand mask [P*K, L], receptor mask / seq / angles of the P pockets, backbones x0 [P*K, L, F] (wrapped uniform angles)"""
    g = torch.Generator().manual_seed(seed)
    nl = torch.randint(nl_rng[0], nl_rng[1] + 1, (P * K,), generator=g)
    nr = torch.randint(nr_rng[0], nr_rng[1] + 1, (P,), generator=g)
    pos = torch.arange(L)[None, :]
    lm, rm = (pos < nl[:, None]).float(), (pos < nr[:, None]).float()
    rseq = torch.nn.functional.one_hot(torch.randint(0, 20, (P, L), generator=g), 20).float() * rm[..., None]
    rang = ((torch.rand(P, L, FS, generator=g) * 2 - 1) * math.pi) * rm[..., None]
    x0 = (torch.rand(P * K, L, FS, generator=g) * 2 - 1) * math.pi
    return lm, rm, rseq, rang, x0


def torch_score_steps(state, cfg, x0, lm, rseq, rang, rm, betas, steps, dev):
    """the oracle's loop on the device under bf16 autocast, steps k = T-1 .. T-steps; returns ms"""
    T = betas.shape[0]
    qs = SSO.qs_table(betas).to(dev)
    g = torch.Generator(device=dev).manual_seed(1)
    terms = torch.zeros(x0.shape, dtype=torch.float64, device=dev)
    valid = (lm != 0)[..., None]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    enc = None
    for k in range(T - 1, T - 1 - steps, -1):
        eps = torch.randn(x0.shape, device=dev, generator=g)
        x_k = SSO.q_sample(x0, qs[k], eps)
        with torch.autocast("cuda", dtype=torch.bfloat16):
            if enc is None:  # the receptor branch once, as the CUDA loop does
                enc = S.struct_encode(state, cfg, rseq, rang, rm)
            pred = S.struct_forward(state, cfg, torch.full((x0.shape[0],), k, dtype=torch.long, device=dev), x_k, lm, rseq, rang, rm,
                                    encoder_outputs=enc).float()
        terms += torch.where(valid, SSO.smooth_l1_terms(eps, pred).double(), torch.zeros((), dtype=torch.float64, device=dev))
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--T", type=int, default=1000)
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--torch-T", type=int, default=5)
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "struct_score_bench_r10.json"))
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("struct_score_bench.py needs a CUDA device")
    import seqdiff_b200 as sd
    SM = sd.structure_model
    dev = torch.device("cuda:0")
    torch.cuda.set_device(dev)
    T = a.T
    card = smi("name,power.limit,clocks.max.sm")
    print("card:", card, flush=True)
    torch.manual_seed(0)
    common = dict(max_position_embeddings=L, intermediate_size=1024, num_hidden_layers=12, position_embedding_type="relative_key")
    m = SM.ConditionalBertForDiffusionBase(sd.BertConfig(**common), sd.BertConfig(**common, is_decoder=True, add_cross_attention=True), FS)
    for blk in (m.receptor_emb, m.timestep_emb):  # as struct_bench.py: no SELayer is an identity
        torch.nn.init.xavier_uniform_(blk.adaLN_modulation[0].weight)
    m = m.eval().to(dev)
    m.precision = "bf16"
    betas = SM.cosine_beta_schedule(T)
    lib = sd.lib()
    cases = []
    b64 = [t.to(dev) for t in inputs(64, 1, (5, 64), (16, 64), 3)]
    cases += [("c64_padded", b64, 1, False), ("c64_packed", b64, 1, True)]
    cases.append(("P8xK8_packed", [t.to(dev) for t in inputs(8, 8, (10, 20), (40, 64), 4)], 8, True))

    def run(kind, case):
        _, (lm, rm, rseq, rang, x0), K, packed = case
        torch.cuda.synchronize()
        n0 = lib.seqdiff_launch_count()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        if kind == "score":
            SM.score_backbones_tensors(m, lm, x0, rseq, rm, rang, T, betas, seed=5, graph_id0=0, packed=packed, num_samples=K)
        else:
            SM.p_sample_loop_tensors(m, lm, x0, rseq, rm, rang, T, betas, seed=5, graph_id0=0, keep_history=False, packed=packed, num_samples=K)
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1), (lib.seqdiff_launch_count() - n0) // T

    summary = {"card": card, "T": T, "precision": "bf16", "model": "12 + 12 layers, H 768, relative_key, F 8, L 64", "cases": {}}
    for case in cases:
        name, K = case[0], case[2]
        G = case[1][4].shape[0]
        for kind in ("sample", "score"):
            run(kind, case)  # warm-up: captures the step graph of each kind
        ms, kernels = {"sample": [], "score": []}, {}
        for i in range(a.runs):
            for kind in ("sample", "score"):
                t, n = run(kind, case)
                ms[kind].append(t)
                kernels[kind] = n
                print(f"{name} run {i} {kind}: {t:.1f} ms  {G * T / t * 1e3:.0f} graph-steps/s  {n} kernels/step  sm clock {smi('clocks.sm')}",
                      flush=True)
        med = {k: statistics.median(v) for k, v in ms.items()}
        rate = {k: G * T / med[k] * 1e3 for k in med}
        summary["cases"][name] = {"graphs": G, "pockets": G // K, "median_ms": {k: round(v, 2) for k, v in med.items()},
                                  "graph_steps_per_s": {k: round(v) for k, v in rate.items()},
                                  "score_over_sample_time": round(med["score"] / med["sample"], 3), "kernels_per_step": kernels,
                                  "spread_ms": {k: [round(min(v), 2), round(max(v), 2)] for k, v in ms.items()}, "runs": a.runs}
        print(name, json.dumps(summary["cases"][name]), flush=True)
    # plain PyTorch: the oracle's loop on the device, bf16 autocast, on the 64-complex batch (padded)
    cfg = S.OracleConfig(max_position_embeddings=L, num_hidden_layers=12, feature_size=FS, relative_key=True)
    state = {k: v.detach().float() for k, v in m.state_dict().items()}
    lm, rm, rseq, rang, x0 = b64
    G = x0.shape[0]
    try:
        with torch.no_grad():
            torch_score_steps(state, cfg, x0, lm, rseq, rang, rm, betas, 2, dev)  # warm-up
            t = torch_score_steps(state, cfg, x0, lm, rseq, rang, rm, betas, a.torch_T, dev)
        summary["torch_arm"] = {"what": "tests/struct_score_oracle.py loop on the GPU, bf16 autocast, receptor branch once, 64 complexes (padded)",
                                "steps": a.torch_T, "ms": round(t, 1), "graph_steps_per_s": round(G * a.torch_T / t * 1e3)}
        summary["torch_arm"]["cuda_score_speedup"] = round(summary["cases"]["c64_padded"]["graph_steps_per_s"]["score"] /
                                                           summary["torch_arm"]["graph_steps_per_s"], 1)
    except Exception as e:  # a failing arm is recorded; the CUDA cases stay
        summary["torch_arm"] = {"error": repr(e)}
    print("torch arm:", json.dumps(summary["torch_arm"]), flush=True)
    os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
    with open(a.out, "w") as f:
        json.dump(summary, f, indent=1)
    print(json.dumps(summary, indent=1))


if __name__ == "__main__":
    main()
