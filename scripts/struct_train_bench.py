#!/usr/bin/env python
"""Structure-model training step on one GPU: forward (dropout 0.1) + wrapped smooth-L1 loss + full backward + clip + AdamW.

Configuration (the struct_bench one): 12 + 12 layers, hidden 768, intermediate 1024, relative_key, L 64 (ligand and receptor), 8 angle
features, bf16 operands, synthetic NoisedAnglesDataset-style batches, at B = 64 and 128 complexes.  Timed with CUDA events around K
steps of `training_step` + `FlatAdamW.step` after W warm-up steps; launches counted by the library over the timed steps.  The
comparison arm is plain PyTorch on the same GPU: autograd through the oracle (oracle/structdiff_oracle.py, objective: tests/struct_train_oracle.py) under bf16 autocast, then
torch's clip_grad_norm_ and AdamW.  The card's name and power limit are read in the same run.

    python scripts/struct_train_bench.py [--steps 10] [--warmup 3] [--batches 64,128] [--no-torch]
"""
import argparse
import json
import math
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch  # noqa: E402

L, NL, FS = 64, 12, 8


def batch_for(B, seed, dev):
    from oracle import seqdiff_oracle as O
    from oracle import structdiff_oracle as S
    b = O.synthetic_batch(B, L, (5, L), (16, L), seed)
    g = torch.Generator().manual_seed(seed + 1)
    ab = S.compute_alphas(S.cosine_beta_schedule(1000))
    t = torch.randint(0, 1000, (B,), generator=g)
    noise = torch.randn(B, L, FS, generator=g)
    corrupted = S.modulo_with_wrapped_range(ab["sqrt_alphas_cumprod"][t][:, None, None] * b["ligand_angles"] +
                                            ab["sqrt_one_minus_alphas_cumprod"][t][:, None, None] * noise)
    out = {"corrupted": corrupted, "t": t, "known_noise": noise, "ligand_attn_mask": b["ligand_attn_mask"], "receptor_seq": b["receptor_seq"],
           "receptor_angles": b["receptor_angles"], "receptor_attn_mask": b["receptor_attn_mask"]}
    return {k: v.to(dev) for k, v in out.items()}


def time_steps(step, steps, warmup):
    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        step()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / steps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--batches", default="64,128")
    ap.add_argument("--no-torch", action="store_true")
    a = ap.parse_args()
    import seqdiff_b200 as sd
    from oracle import structdiff_oracle as S
    import struct_train_oracle as T
    if not torch.cuda.is_available():
        raise SystemExit("struct_train_bench.py measures on a CUDA device")
    dev = torch.device("cuda:0")
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    common = dict(max_position_embeddings=L, intermediate_size=1024, num_hidden_layers=NL, position_embedding_type="relative_key")
    cfgs = (sd.BertConfig(**common), sd.BertConfig(**common, is_decoder=True, add_cross_attention=True))
    cfg = S.OracleConfig(max_position_embeddings=L, num_hidden_layers=NL, feature_size=FS, relative_key=True)
    state = S.init_struct_state_dict(cfg, 0)
    lib = sd.lib()
    res = {"metric": "structure-model training step (forward + loss + backward + clip + AdamW)", "unit": "ms per step", "n_gpus": 1,
           "steps": a.steps, "warmup": a.warmup, "dtype": "bf16", "data": "synthetic", "card": card,
           "config": {"layers": "12 + 12", "hidden": 768, "intermediate": 1024, "position_embedding_type": "relative_key", "L_lig": L, "L_rec": L,
                      "features": FS, "dropout": 0.1},
           "results": []}
    for B in [int(x) for x in a.batches.split(",")]:
        batch = batch_for(B, 7, dev)
        m = sd.structure_model.ConditionalBertForDiffusion(*cfgs, FS)
        m.load_state_dict(state, strict=True)
        m = m.to(dev).train()
        m.precision = "bf16"
        opt = m.configure_optimizers()["optimizer"]
        it = [0]

        def step():
            it[0] += 1
            m.training_step(batch, it[0])
            opt.step()

        for _ in range(a.warmup):
            step()
        torch.cuda.synchronize()
        n0 = lib.seqdiff_launch_count()
        ms = time_steps(step, a.steps, 0)
        launches = (lib.seqdiff_launch_count() - n0) / a.steps
        loss = float(m.last_log["train_loss"])
        row = {"B": B, "ms_per_step": ms, "graphs_per_s": B / (ms * 1e-3), "launches_per_step": launches, "last_loss": loss}
        m.release()
        del m, opt
        if not a.no_torch:
            leaf = {k: v.detach().clone().to(dev).requires_grad_(k != "timestep_projector.W") for k, v in state.items()}
            params = [v for k, v in leaf.items() if v.requires_grad]
            topt = torch.optim.AdamW(params, lr=5e-5, weight_decay=0.0)

            def tstep():
                topt.zero_grad(set_to_none=True)
                with torch.autocast("cuda", dtype=torch.bfloat16):
                    pred = S.struct_forward(leaf, cfg, batch["t"], batch["corrupted"], batch["ligand_attn_mask"], batch["receptor_seq"],
                                            batch["receptor_angles"], batch["receptor_attn_mask"])
                loss_, _ = T.angle_loss(pred.float(), batch["known_noise"], batch["ligand_attn_mask"])
                loss_.backward()
                torch.nn.utils.clip_grad_norm_(params, 1.0)
                topt.step()

            tms = time_steps(tstep, a.steps, a.warmup)
            row["torch_autograd"] = {"ms_per_step": tms, "graphs_per_s": B / (tms * 1e-3), "speedup": tms / ms,
                                     "what": "oracle forward under bf16 autocast + autograd + clip_grad_norm_ + torch.optim.AdamW, dropout off"}
            del leaf, params, topt
            torch.cuda.empty_cache()
        res["results"].append(row)
    print(json.dumps(res))


if __name__ == "__main__":
    main()
