#!/usr/bin/env python
"""Structure sampler, padded vs ragged-packed (p_sample_loop(packed=True)) on one GPU, in alternating runs.

Workloads (bf16, 12 + 12 layers, relative_key, 8 angle features, in-kernel Philox noise, L = 64):
  a  scripts/struct_bench.py's default: 64 complexes, ligand lengths U(5..64), receptor lengths U(16..64)
  b  design shape: 64 complexes, peptides of 10-20 residues in pockets of 40-64
  c  256 complexes of shape a
Every run times one whole p_sample_loop call (CUDA events, device-resident inputs, final angles only) in each mode, padded first,
and checks that the two final tensors are equal at every valid position and that the packed one is 0 at the padded positions.
Unit: graph-steps/s (one complex through one step = denoiser forward + Gaussian update + wrap).  Kernels per step = launches of a
warm call // T (the receptor branch, run once per call, adds fewer than T launches).

    python scripts/struct_packed_bench.py [--runs 3] [--timesteps 1000] [--workloads abc] [--out DIR]
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

WORKLOADS = {  # name: (complexes, ligand length range, receptor length range)
    "a": (64, (5, 64), (16, 64)),
    "b": (64, (10, 20), (40, 64)),
    "c": (256, (5, 64), (16, 64)),
}
L, FS = 64, 8


def gpu_info():
    info = {"name": torch.cuda.get_device_name(0)}
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True,
                           timeout=30).stdout.strip().splitlines()
        info["power_limit, max_sm_clock"] = q[0] if q else None
    except (OSError, subprocess.SubprocessError):
        info["power_limit, max_sm_clock"] = None
    return info


def inputs(B, nl_rng, nr_rng, seed):
    g = torch.Generator().manual_seed(seed)
    nl = torch.randint(nl_rng[0], nl_rng[1] + 1, (B,), generator=g)
    nr = torch.randint(nr_rng[0], nr_rng[1] + 1, (B,), generator=g)
    pos = torch.arange(L)[None, :]
    lm, rm = (pos < nl[:, None]).float(), (pos < nr[:, None]).float()
    rseq = torch.nn.functional.one_hot(torch.randint(0, 20, (B, L), generator=g), 20).float() * rm[..., None]
    rang = ((torch.rand(B, L, FS, generator=g) * 2 - 1) * math.pi) * rm[..., None]
    x_T = ((torch.rand(B, L, FS, generator=g) * 2 - 1) * math.pi)
    return lm, rm, rseq, rang, x_T


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--runs", type=int, default=3)
    ap.add_argument("--timesteps", type=int, default=1000)
    ap.add_argument("--workloads", default="abc")
    ap.add_argument("--out", default=None, help="directory for struct_packed_bench.json")
    a = ap.parse_args()
    import seqdiff_b200 as sd
    SM = sd.structure_model
    dev = torch.device("cuda:0")
    T = a.timesteps
    torch.manual_seed(0)
    common = dict(max_position_embeddings=L, intermediate_size=1024, num_hidden_layers=12, position_embedding_type="relative_key")
    m = SM.ConditionalBertForDiffusionBase(sd.BertConfig(**common), sd.BertConfig(**common, is_decoder=True, add_cross_attention=True), FS)
    for blk in (m.receptor_emb, m.timestep_emb):  # as struct_bench.py: no SELayer is an identity
        torch.nn.init.xavier_uniform_(blk.adaLN_modulation[0].weight)
    m = m.eval().to(dev)
    m.precision = "bf16"
    betas = SM.cosine_beta_schedule(T)
    lib = sd.lib()
    res = {"gpu": gpu_info(), "timesteps": T, "runs": a.runs, "dtype": "bf16", "layers": "12 + 12", "L": L, "workloads": {}}
    for name in a.workloads:
        B, nl_rng, nr_rng = WORKLOADS[name]
        lm, rm, rseq, rang, x_T = inputs(B, nl_rng, nr_rng, 3)
        args = dict(model=m, ligand_mask=lm.to(dev), ligand_angle_noise=x_T.to(dev), receptor_seq=rseq.to(dev), receptor_mask=rm.to(dev),
                    receptor_angle=rang.to(dev), total_timesteps=T, betas=betas, seed=5, graph_id0=0, keep_history=False)
        valid = lm.bool().to(dev)[:, :, None].expand(B, L, FS)

        def run(packed):
            torch.cuda.synchronize()
            n0 = lib.seqdiff_launch_count()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            out = SM.p_sample_loop(**args, packed=packed)
            e1.record()
            torch.cuda.synchronize()
            return out[0], e0.elapsed_time(e1), lib.seqdiff_launch_count() - n0

        times = {False: [], True: []}
        kernels = {}
        run(False), run(True)  # warm-up: captures each mode's step graph
        for _ in range(a.runs):
            ref, ms_pad, n_pad = run(False)
            got, ms_pk, n_pk = run(True)
            if not (torch.equal(got.to(dev)[valid], ref.to(dev)[valid]) and bool((got.to(dev)[~valid] == 0).all())):
                raise SystemExit(f"workload {name}: packed result differs from the padded one at a valid position")
            times[False].append(ms_pad)
            times[True].append(ms_pk)
            kernels = {"padded": n_pad // T, "packed": n_pk // T}
        med = {k: statistics.median(v) for k, v in times.items()}
        rate = {k: B * T / (v * 1e-3) for k, v in med.items()}
        res["workloads"][name] = {
            "complexes": B, "ligand_lengths": list(nl_rng), "receptor_lengths": list(nr_rng),
            "valid_rows": {"ligand": int(lm.sum()), "receptor": int(rm.sum()), "padded_each": B * L},
            "padded_graph_steps_per_s": rate[False], "packed_graph_steps_per_s": rate[True], "speedup": rate[True] / rate[False],
            "ms_per_call": {"padded": times[False], "packed": times[True]}, "kernels_per_step": kernels, "equal_at_valid_positions": True}
        print(json.dumps({name: res["workloads"][name]}), flush=True)
    print(json.dumps({"gpu": res["gpu"]}))
    if a.out:
        os.makedirs(a.out, exist_ok=True)
        with open(os.path.join(a.out, "struct_packed_bench.json"), "w") as f:
            json.dump(res, f, indent=1)


if __name__ == "__main__":
    main()
