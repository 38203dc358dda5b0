#!/usr/bin/env python
"""Peptide design on one GPU: P pockets x K1 backbones x K2 sequences, in alternating runs (bf16, medians of --runs).

  a  structure sampler, 12 + 12 layers, L = 64, T = 1000, ligand lengths U(5..64), receptor lengths U(16..64):
     p_sample_loop(num_samples=K1) on P pockets against p_sample_loop on the 64-complex batch with every pocket repeated K1 times,
     padded and packed.  Times one whole sampling (CUDA events, final angles only) and checks the two final tensors equal; reports
     the receptor-side rows and bytes from the shapes (encoder rows, cross K|V block of every decoder layer).
  b  design: design() (device hand-off, K1 backbones x K2 sequences per pocket) against the host composition it replaces --
     p_sample_loop on the replicated batch (the [T,B,L,F] history copied to the host), sample()'s numpy trim, load_generated_angles,
     denoise on the batch with every (pocket, backbone) repeated K2 times.  Sequence model: sample.py's CONFIG (6 layers, L = 64,
     T = 50), DiscreteUniformTransition(20).  Both paths are packed and get the same start states, seeds and graph ids; the
     sequences must be equal.  Reports the wall time of every leg (host clock around work that ends in a device synchronise).

    python scripts/design_bench.py [--runs 3] [--pockets 8] [--backbones 8] [--sequences 8] [--timesteps 1000] [--parts ab] [--out DIR]
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

L, FS = 64, 8


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm,clocks.sm", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()
        info["power_limit, max_sm_clock, sm_clock"] = q[0] if q else None
    except (OSError, subprocess.SubprocessError):
        info["power_limit, max_sm_clock, sm_clock"] = None
    return info


def pockets(P, seed):
    """a sequence-model batch of P complexes (L = 64), ligand U(5..64), receptor U(16..64)"""
    g = torch.Generator().manual_seed(seed)
    nl = torch.randint(5, L + 1, (P,), generator=g)
    nr = torch.randint(16, L + 1, (P,), generator=g)
    pos = torch.arange(L)[None, :]
    lm, rm = (pos < nl[:, None]).float(), (pos < nr[:, None]).float()
    oh = lambda m: torch.nn.functional.one_hot(torch.randint(0, 20, (P, L), generator=g), 20).float() * m[..., None]  # noqa: E731
    ang = lambda m: ((torch.rand(P, L, FS, generator=g) * 2 - 1) * math.pi) * m[..., None]  # noqa: E731
    return {"ligand_seq": oh(lm), "ligand_angles": ang(lm), "ligand_attn_mask": lm, "receptor_seq": oh(rm), "receptor_angles": ang(rm),
            "receptor_attn_mask": rm, "structure_ids": {"pdb_id": [f"s{i:03d}" for i in range(P)], "ligand_chain": ["A"] * P}}


def rep(batch, K):
    out = {k: v.repeat_interleave(K, dim=0) for k, v in batch.items() if torch.is_tensor(v)}
    out["structure_ids"] = {k: [x for x in v for _ in range(K)] for k, v in batch["structure_ids"].items()}
    return out


def timed(fn):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    out = fn()
    torch.cuda.synchronize()
    return out, time.perf_counter() - t0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--pockets", type=int, default=8)
    ap.add_argument("--backbones", type=int, default=8)
    ap.add_argument("--sequences", type=int, default=8)
    ap.add_argument("--timesteps", type=int, default=1000)
    ap.add_argument("--parts", default="ab")
    ap.add_argument("--out", default=None, help="directory for design_bench.json")
    a = ap.parse_args()
    import seqdiff_b200 as sd
    SM = sd.structure_model
    dev = torch.device("cuda:0")
    sd.sample.DEVICE = dev
    P, K1, K2, T = a.pockets, a.backbones, a.sequences, a.timesteps
    torch.manual_seed(0)
    common = dict(max_position_embeddings=L, intermediate_size=1024, num_hidden_layers=12, position_embedding_type="relative_key")
    st = SM.ConditionalBertForDiffusionBase(sd.BertConfig(**common), sd.BertConfig(**common, is_decoder=True, add_cross_attention=True), FS)
    for blk in (st.receptor_emb, st.timestep_emb):  # as struct_bench.py: no SELayer is an identity
        torch.nn.init.xavier_uniform_(blk.adaLN_modulation[0].weight)
    st = st.eval().to(dev)
    st.precision = "bf16"
    betas = SM.cosine_beta_schedule(T)
    H, NL = st.decoder_config.hidden_size, st.decoder_config.num_hidden_layers
    batch = pockets(P, 3)
    g = torch.Generator().manual_seed(4)
    x_T = SM.modulo_with_wrapped_range(torch.randn(P * K1, L, FS, generator=g))
    res = {"gpu": gpu_info(), "dtype": "bf16", "pockets": P, "backbones": K1, "sequences": K2, "struct_timesteps": T, "runs": a.runs}

    if "a" in a.parts:
        args = lambda b: (b["ligand_attn_mask"][:, :L].to(dev), x_T.to(dev), b["receptor_seq"].to(dev), b["receptor_attn_mask"].to(dev),  # noqa: E731
                          b["receptor_angles"].to(dev), T, betas)
        rb = rep(batch, K1)
        part = {}
        for packed in (False, True):
            kw = dict(seed=5, graph_id0=0, keep_history=False, packed=packed)
            shared = lambda: SM.p_sample_loop_tensors(st, *args(batch), num_samples=K1, **kw)[1]  # noqa: E731
            repl = lambda: SM.p_sample_loop_tensors(st, *args(rb), **kw)[1]  # noqa: E731
            timed(repl), timed(shared)  # warm-up: captures each variant's step graph
            times = {"replicated": [], "shared": []}
            for _ in range(a.runs):
                want, t_r = timed(repl)
                got, t_s = timed(shared)
                if not torch.equal(got, want):
                    raise SystemExit(f"part a (packed={packed}): shared-pocket result differs from the replicated batch")
                times["replicated"].append(t_r)
                times["shared"].append(t_s)
            rows = {"replicated": int(rb["receptor_attn_mask"].sum()) if packed else P * K1 * L,
                    "shared": int(batch["receptor_attn_mask"].sum()) if packed else P * L}
            med = {k: statistics.median(v) for k, v in times.items()}
            part["packed" if packed else "padded"] = {
                "s_per_sampling": times, "median_s": med, "ms_per_step": {k: 1e3 * v / T for k, v in med.items()},
                "graph_steps_per_s": {k: P * K1 * T / v for k, v in med.items()}, "change": med["replicated"] / med["shared"] - 1,
                "receptor_rows": rows, "cross_kv_bytes": {k: v * NL * 2 * H * 2 for k, v in rows.items()},
                "encoder_row_bytes_bf16": {k: v * H * 2 for k, v in rows.items()}, "equal": True}
            print(json.dumps({"a": {"packed" if packed else "padded": part["packed" if packed else "padded"]}}), flush=True)
        res["a_structure"] = part

    if "b" in a.parts:
        sc = sd.sample.CONFIG
        qc = dict(max_position_embeddings=sc["max_seq_len"], num_attention_heads=sc["num_heads"], hidden_size=sc["hidden_size"],
                  intermediate_size=sc["intermediate_size"], num_hidden_layers=sc["num_hidden_layers"],
                  position_embedding_type=sc["position_embedding_type"])
        sq = sd.ConditionalBertForDiffusionBase(sd.BertConfig(**qc), sd.BertConfig(**qc, is_decoder=True, add_cross_attention=True), 20)
        sq = sq.eval().to(dev)
        sq.precision = "bf16"
        Tq = sc["timesteps"]
        sched, tr = sd.PredefinedNoiseScheduleDiscrete(sc["noise_schedule"], Tq), sd.DiscreteUniformTransition(20)
        seq_x_T = sd.generate_discrete_noise(P * K1 * K2, L, device=torch.device("cpu"))
        ids = dict(seed=5, graph_id0=1000, seq_graph_id0=20000)

        def design():
            return sd.design.design(st, sq, batch, K1, K2, packed=True, struct_betas=betas, noise_schedule=sched, transition=tr,
                                    timesteps=Tq, x_T=x_T, seq_x_T=seq_x_T, **ids)

        def host():
            legs = {}
            sb = rep(batch, K1)
            hist, legs["structure (history to host)"] = timed(lambda: SM.p_sample_loop(
                st, sb["ligand_attn_mask"], x_T, sb["receptor_seq"], sb["receptor_attn_mask"], sb["receptor_angles"], T, betas,
                seed=ids["seed"], graph_id0=ids["graph_id0"], packed=True))
            t0 = time.perf_counter()
            lens = sb["ligand_attn_mask"].sum(dim=1).int()
            trimmed = [hist[:, i, :int(l), :].numpy() for i, l in enumerate(lens)]
            gen = sd.load_generated_angles([x[-1] for x in trimmed], max_seq_len=L, batch_size=P * K1)[0]
            qb = rep(batch, K1 * K2)
            qb["ligand_angles"] = gen.repeat_interleave(K2, dim=0)
            legs["trim + load_generated_angles (host)"] = time.perf_counter() - t0
            out, legs["sequence + decode"] = timed(lambda: sd.denoise(qb, sq, sched, tr, True, timesteps=Tq, x_T=seq_x_T, seed=ids["seed"],
                                                                      graph_id0=ids["seq_graph_id0"], packed=True))
            return out, legs

        def design_legs():
            legs = {}
            _, legs["structure (final angles on the device)"] = timed(lambda: SM.p_sample_loop_tensors(
                st, batch["ligand_attn_mask"], x_T, batch["receptor_seq"], batch["receptor_attn_mask"], batch["receptor_angles"], T, betas,
                seed=ids["seed"], graph_id0=ids["graph_id0"], keep_history=False, packed=True, num_samples=K1))
            out, legs["design() total"] = timed(design)
            return out, legs

        host(), design_legs()  # warm-up
        times = {"host": [], "design": []}
        for _ in range(a.runs):
            want, lh = host()
            got, ld = design_legs()
            if (got[0], got[3], got[4], got[5]) != tuple(want):
                raise SystemExit("part b: design() sequences differ from the host composition")
            lh["total"] = sum(lh.values())
            times["host"].append(lh)
            times["design"].append(ld)
        med = {k: {leg: statistics.median(r[leg] for r in v) for leg in v[0]} for k, v in times.items()}
        res["b_design"] = {"sequences_total": P * K1 * K2, "seq_timesteps": Tq, "runs_s": times, "median_s": med, "equal": True,
                           "history_bytes_copied_by_host_path": T * P * K1 * L * FS * 4}
        print(json.dumps({"b": {"median_s": med}}), flush=True)
    print(json.dumps({"gpu": res["gpu"]}))
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "design_bench.json"), "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
