#!/usr/bin/env python
"""bench.py -- headline benchmark of the sequence-denoiser hot path (BASELINE.json configs[1]):
full reverse-diffusion sampling (T=500) of 64 synthetic pocket graphs (L=128) per GPU, bf16 tensor-core
operands, on N B200s of one node (one process per GPU, graphs sharded across ranks, no collective on the
data path: weak scaling).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this repository's CUDA path
    python bench.py --impl reference [--steps K] [--warmup W]      # the reference algorithm on host CPU cores
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py ... --dump-outputs DIR     # also write what the last timed step computed as DIR/<name>.npy

The inputs and weights are seeded, so two builds run with the same arguments can be compared output for output.

Vocabulary.  graph-step = one pocket graph through one denoiser forward + one reverse-diffusion step
(sequence_model/sample.py:199-207).  One bench "step" = one complete T-step sampling of the rank's batch
= B*T graph-steps.  denoised pocket-graphs/s = value / T;  edge msgs/s (attended query-key pairs) =
value * 15 * L^2 (SURVEY.md section 8d).  One JSON line is printed by rank 0.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "denoiser graph-steps/s (forward + reverse-diffusion step per pocket graph; cfg2: 64 pockets x 500 steps, L=128)"
UNIT = "graph-steps/s"
H, I, NL = 768, 1024, 6
L = 128  # set by the workload in main()
# algorithmic FLOPs per graph-step (BASELINE.md section 3) and the reference's own sizes per workload
WORKLOADS = {
    "cfg2": dict(L=128, T=500, batch=64, scaling="weak", n_lig=(5, 64), n_rec=(16, 128), flops=18.369e9,
                 text="BASELINE configs[1]: full reverse-diffusion sampling (T={T}) of {B} synthetic pockets per GPU, L=128, ragged "
                      "n_lig~U[5,64] n_rec~U[16,128], diverse=True, random-init weights, relative_key attention"),
    "cfg3": dict(L=512, T=50, batch=256, scaling="strong", n_lig=(48, 48), n_rec=(464, 464), flops=85.229e9,
                 text="BASELINE configs[2]: ext-neighbour pockets, 256 graphs of 512 residues (n_lig=48, n_rec=464) sharded over the GPUs, "
                      "T={T} (reference default), {B} graphs on this rank, diverse=True, random-init weights"),
    "cfg4": dict(L=128, T=50, batch=128, scaling="strong", n_lig=(5, 64), n_rec=(16, 128), flops=3 * 18.369e9,
                 text="BASELINE configs[3]: training step, global batch 128 graphs over the GPUs ({B} on this rank), L=128, T={T}, dropout 0.1, "
                      "AdamW + clip, one NCCL gradient all-reduce per step"),
}


# ----------------------------------------------------------------------------------------------------
def synthetic_workload(B, seed_offset=0, n_lig=(5, 64), n_rec=(16, 128)):
    """SURVEY.md section 8d cfg 2: n_lig ~ U{5..64}, n_rec ~ U{16..128} (seed 3), angles ~ U(-pi, pi), zero padding,
    prefix-ones masks; x_T one-hot of randint (seed 4).  Plain torch on the host -- no oracle import here."""
    g = torch.Generator().manual_seed(3 + seed_offset)
    nl = torch.randint(n_lig[0], n_lig[1] + 1, (B,), generator=g)
    nr = torch.randint(n_rec[0], n_rec[1] + 1, (B,), generator=g)
    pos = torch.arange(L)[None, :]
    lm, rm = (pos < nl[:, None]).float(), (pos < nr[:, None]).float()

    def side(mask):
        seq = torch.nn.functional.one_hot(torch.randint(0, 20, (B, L), generator=g), 20).float() * mask[..., None]
        ang = ((torch.rand(B, L, 8, generator=g) * 2 - 1) * math.pi) * mask[..., None]
        return seq, ang

    lseq, lang = side(lm)
    rseq, rang = side(rm)
    g4 = torch.Generator().manual_seed(4 + seed_offset)
    x_T = torch.nn.functional.one_hot(torch.randint(0, 20, (B, L), generator=g4), 20).float()
    batch = {"ligand_seq": lseq, "ligand_angles": lang, "ligand_attn_mask": lm, "receptor_seq": rseq, "receptor_angles": rang,
             "receptor_attn_mask": rm, "structure_ids": {"pdb_id": [f"s{i:04d}" for i in range(B)], "ligand_chain": ["A"] * B}}
    return batch, x_T


def gemm_flops_per_forward(B):
    """2*M*N*K summed over the 50 GEMM launches of one forward (DESIGN.md section 'Kernels')."""
    Ml = Mr = B * L
    Mt = Ml + Mr
    macs = 19 * Mt * H * H                      # ligand_feature_emb over [lig|rec]: ada0, ada2(6), qkv(3), out, mlp(4+4)
    macs += 2 * NL * Mr * H * H                 # stacked cross K|V projection
    macs += NL * Ml * (6 * H * H + 2 * I * H)   # decoder layers: qkv(3) out cq cout + FFN up/down
    macs += 12 * Ml * H * H + 7 * B * H * H     # decoder_normalize (adaLN on B rows only)
    macs += Ml * H * H                          # predictor dense1
    return 2 * macs




class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled every 200 ms while the timed region runs."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown," \
        "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, gpu_index):
        self.idx, self.rows, self.proc = gpu_index, [], None

    def __enter__(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i",
                                          str(self.idx)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._pump, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None
        return self

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def __exit__(self, *a):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self):
        sm, mx, reasons = [], [], set()
        for r in self.rows:
            try:
                sm.append(float(r[1]))
                mx.append(float(r[2]))
            except Exception:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        return {"sm_mhz": statistics.median(sm), "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


DUMP_BYTES = 64 << 20  # all arrays of one --dump-outputs directory together


def dump_outputs(out_dir, arrays):
    """Writes {name: tensor} as out_dir/<name>.npy (float64 stays float64, everything else becomes float32), DUMP_BYTES in all.  Going
    from the smallest array up, one larger than an even share of what is left is replaced by a fixed sample of its flattened elements
    (seeded, ascending indices), so runs with the same arguments dump the same positions."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: (t.detach().cpu().double() if t.dtype == torch.float64 else t.detach().cpu().float()) for k, t in arrays.items()}
    left = DUMP_BYTES - 256 * len(arrays)  # room for the .npy headers
    for i, (name, t) in enumerate(sorted(arrays.items(), key=lambda kv: kv[1].numel() * kv[1].element_size())):
        n = left // (len(arrays) - i) // t.element_size()
        if t.numel() > n:
            t = t.reshape(-1)[torch.randperm(t.numel(), generator=torch.Generator().manual_seed(0))[:n].sort().values]
        left -= t.numel() * t.element_size()
        np.save(os.path.join(out_dir, f"{name}.npy"), t.numpy())


def training_outputs(sd, opt, loss, n_sample=1 << 20):
    """What a caller holds after one optimizer step of the training path: the loss, the gradient norm the clip measured, and the same
    fixed seeded sample of the flat gradient and of the updated fp32 weights (live parameters in name order)."""
    import ctypes
    flat = opt.flat
    lib = sd.lib()
    names = sorted(flat.table)
    grads = torch.cat([flat.grads[flat.table[k][0]:flat.table[k][0] + flat.table[k][1]] for k in names])
    weights = torch.empty_like(grads)
    pos = 0
    with torch.cuda.device(flat.device):
        stream = ctypes.c_void_p(torch.cuda.current_stream(flat.device).cuda_stream)
        for k in names:
            n = flat.table[k][1]
            sd._cabi.check(lib.seqdiff_model_get_tensor(flat.handle, k.encode(), sd._cabi.ptr(weights[pos:pos + n]), n, stream))
            pos += n
    idx = torch.randperm(grads.numel(), generator=torch.Generator().manual_seed(0))[:n_sample].sort().values.to(grads.device)
    return {"loss": loss.reshape(1), "grad_norm": opt.grad_norm, "grads_sample": grads[idx], "weights_sample": weights[idx]}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("bf16_tflops_sustained", d.get("bf16_tflops")), "measured (MEASURED_PEAKS.json bf16_tflops_sustained)", d.get("hbm_gbs")
    return 1400.0, "fallback (B200_PROFILING.md sustained 1.4 PFLOP/s)", 6650.0


# ----------------------------------------------------------------------------------------------------
def cpu_reference_steps(state, batch, x_T, T, n_steps, n_warm, threads, outputs=None):
    """The reference algorithm on host cores ("port": oracle/seqdiff_oracle.py, which restates
    sequence_model/model.py:200-237 + sample.py:141-179 incl. its Python multinomial loop).
    One step = forward + reverse step over the whole batch at s_int = T-1, T-2, ...
    `outputs` (a dict) receives the logits and the sampled x of the last step."""
    from oracle import seqdiff_oracle as O
    torch.set_num_threads(threads)
    cfg = O.OracleConfig(max_position_embeddings=L)
    sched, trans = O.NoiseScheduleDiscrete("cosine", T), O.BlosumTransition(timestep=500)
    B = x_T.shape[0]
    x = x_T.clone()
    times = []
    with torch.no_grad():
        for i in range(n_warm + n_steps):
            s_int = T - 1 - i
            t0 = time.perf_counter()
            s_array = s_int * torch.ones((B, 1))
            logits = O.denoiser_forward(state, cfg, s_array, x, batch["ligand_angles"], batch["ligand_attn_mask"], batch["receptor_seq"],
                                        batch["receptor_angles"], batch["receptor_attn_mask"])
            x = O.reverse_step_python_loop((s_array + 1) / T, s_array / T, x, logits, sched, trans, True, False)
            dt = time.perf_counter() - t0
            if i >= n_warm:
                times.append(dt)
    if outputs is not None:
        outputs.update(logits=logits, x=x)
    return times


def workload_config(wl, B, T, world):
    """The `config` object of the JSON line: static description of the workload only, identical on the product and the reference arm
    (what the reference arm samples of it is said in its `cpu_baseline.sample` / `sample` keys; derived rates live in `derived`)."""
    return {"workload": wl["text"].format(T=T, B=B), "batch_per_gpu": B, "L": L, "timesteps": T,
            "sharding": f"graphs x{world} (no data-path collective)",
            "l2": "per-step working set of activations (0.9 GB at cfg2, ~10 GB at cfg3) >> 126 MB L2 (no explicit flush needed)"}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    import seqdiff_b200 as sd  # host-side module tree only (weights); no CUDA call is made on this arm
    torch.manual_seed(0)
    common = dict(max_position_embeddings=L, intermediate_size=I, num_hidden_layers=NL, position_embedding_type="relative_key")
    model = sd.ConditionalBertForDiffusionBase(sd.BertConfig(**common), sd.BertConfig(**common, is_decoder=True, add_cross_attention=True), 20)
    state = {k: v.detach().clone() for k, v in model.state_dict().items()}
    cpu_b = args.batch if args.workload == "cfg2" else 4  # L=512: a 4-graph sample keeps a step at a few seconds
    batch, x_T = synthetic_workload(cpu_b, n_lig=args.wl["n_lig"], n_rec=args.wl["n_rec"])
    cfg_obj = workload_config(args.wl, args.batch, args.timesteps, int(os.environ.get("WORLD_SIZE", "1")))  # the product arm's config
    args.batch = cpu_b
    threads = os.cpu_count() or 1
    outputs = {} if args.dump_outputs else None
    times = cpu_reference_steps(state, batch, x_T, args.timesteps, args.steps, args.warmup, threads, outputs)
    if outputs is not None:
        dump_outputs(args.dump_outputs, outputs)
    total = sum(times)
    value = args.batch * len(times) / total
    out = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
           "warmup": args.warmup, "ms_per_step": 1e3 * total / len(times), "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
           "dtype": "f32", "data": "synthetic",
           "config": cfg_obj,
           "sample": f"each bench step = ONE denoise step (forward + reverse step) of a {args.batch}-pocket batch on the host CPU; the metric is "
                     "normalised per graph-step, so it compares with the product arm's full samplings (SURVEY.md section 8d)",
           "cpu_baseline": {"value": value, "unit": UNIT, "cores": threads, "kind": "port",
                            "sample": f"{len(times)} denoise steps x {args.batch} graphs (of {args.timesteps} steps); oracle port incl. the reference's Python multinomial loop"},
           "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out))
    return 0


# ----------------------------------------------------------------------------------------------------
def cfg3_strong_record(sd, dev, world, rank, barrier, precision, steps=2, warmup=1):
    """BASELINE configs[2] on the ranks of this job: 256 ext-pocket graphs of 512 residues (n_lig 48, n_rec 464), T = 50, block-
    partitioned over the GPUs (strong scaling: 256 / world graphs per rank, no data-path collective).  Device-resident inputs, CUDA
    events, max over ranks.  Returned as the `cfg3_strong` record of the main JSON line so that the driver's 1/2/4/8-GPU scaling run
    carries the numbers of the NAMED strong-scaling configuration next to the cfg-2 value."""
    import torch.distributed as dist
    global L
    keep_L, wl = L, WORKLOADS["cfg3"]
    L = wl["L"]
    try:
        total, T = wl["batch"], wl["T"]
        lo, hi = sd.shard_bounds(total, world, rank)
        Bl = hi - lo
        torch.manual_seed(0)
        common = dict(max_position_embeddings=L, intermediate_size=I, num_hidden_layers=NL, position_embedding_type="relative_key")
        model = sd.ConditionalBertForDiffusionBase(sd.BertConfig(**common), sd.BertConfig(**common, is_decoder=True, add_cross_attention=True), 20)
        model = model.eval().to(dev)
        model.precision = precision
        sched, trans = sd.PredefinedNoiseScheduleDiscrete("cosine", T), sd.BlosumTransition(x_classes=20, timestep=500)
        batch, x_T = synthetic_workload(total, n_lig=wl["n_lig"], n_rec=wl["n_rec"])  # the SAME 256 graphs for every world size
        dbatch = {k: (v[lo:hi].to(dev) if torch.is_tensor(v) else v) for k, v in batch.items()}
        dx_T = x_T[lo:hi].to(dev)
        run = lambda: sd.denoise_tensors(dbatch, model, sched, trans, True, timesteps=T, x_T=dx_T, seed=5, graph_id0=lo)
        for _ in range(warmup):
            run()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            out = run()
        e1.record()
        barrier()
        ms_rank = e0.elapsed_time(e1)
        ms = torch.tensor([ms_rank], device=dev)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        ms = ms.item()
        ok = bool(torch.isfinite(out).all())
        value = total * T * steps / (ms * 1e-3)
        peak, _, _ = measured_peaks()
        packed_value = None
        if precision != "fp32":
            runp = lambda: sd.denoise_tensors(dbatch, model, sched, trans, True, timesteps=T, x_T=dx_T, seed=5, graph_id0=lo, packed=True)
            outp = runp()
            barrier()
            e0.record()
            for _ in range(steps):
                outp = runp()
            e1.record()
            barrier()
            msp = torch.tensor([e0.elapsed_time(e1)], device=dev)
            if world > 1:
                dist.all_reduce(msp, op=dist.ReduceOp.MAX)
            vm = dbatch["ligand_attn_mask"].bool()
            packed_value = {"value": total * T * steps / (msp.item() * 1e-3), "ms_per_sampling": msp.item() / steps,
                            "identical_to_padded_at_valid_positions": bool(torch.equal(outp[vm], out[vm]))}
        model.release()
        del model
        torch.cuda.empty_cache()
        return {"workload": wl["text"].format(T=T, B=Bl), "scaling": "strong", "graphs_total": total, "graphs_per_gpu": Bl, "L": L, "timesteps": T,
                "value": value, "unit": UNIT, "ms_per_sampling": ms / steps, "ms_this_rank": ms_rank / steps, "steps": steps, "warmup": warmup,
                "finite": ok, "whole_step_model_flops_frac": (value / world) * wl["flops"] / 1e12 / peak, "dtype": precision, "packed": packed_value}
    finally:
        L = keep_L


def cfg4_train_record(sd, dev, world, rank, barrier, precision, steps=10, warmup=10, global_batch=128, grad_comm="fp32", weak=False,
                      outputs=None):
    """BASELINE configs[3]: one optimizer step of the sequence denoiser on a GLOBAL batch of 128 graphs (L = 128, T = 50, dropout 0.1,
    AdamW lr 5e-5 wd 0.1, clip 1.0: train_model.py:17-33), data-parallel over the ranks (128 / world graphs each), ONE gradient
    all-reduce per step over NCCL (61.06 M live parameters).  Reports whole steps (training_step + all-reduce + clip + AdamW), the
    same without the all-reduce, and the all-reduce alone => exposed-communication fraction and achieved bus bandwidth.
    `outputs` (a dict) receives training_outputs() of the last whole step."""
    import torch.distributed as dist
    global L
    keep_L = L
    L = 128
    try:
        T = 50
        if weak:  # Lightning-DDP reading of "batch 128": the DataLoader batch size is per process (train_model.py:38,50), global = 128 x world
            global_batch = global_batch * world
        lo, hi = sd.shard_bounds(global_batch, world, rank)
        Bl = hi - lo
        torch.manual_seed(0)
        common = dict(max_position_embeddings=L, intermediate_size=I, num_hidden_layers=NL, position_embedding_type="relative_key",
                      hidden_dropout_prob=0.1, attention_probs_dropout_prob=0.1)
        model = sd.PeptideDiff(sd.BertConfig(**common), sd.BertConfig(**common, is_decoder=True, add_cross_attention=True), list(sd.AA_VOCAB),
                               torch.nn.CrossEntropyLoss(), "cosine", T, max_epochs=150, lr_scheduler="LinearWarmup", l2_lambda=0.1, learning_rate=5e-5)
        model = model.to(dev).train()
        model.precision = precision
        batch, _ = synthetic_workload(global_batch, n_lig=(5, 64), n_rec=(16, 128))
        dbatch = {k: (v[lo:hi].to(dev) if torch.is_tensor(v) else v) for k, v in batch.items()}
        opt = model.configure_optimizers(grad_comm=grad_comm)["optimizer"]

        def step(i, skip=False, overlap=True):
            opt.overlap = overlap and not skip
            loss = model.training_step(dbatch, i)
            opt.step(skip_all_reduce=skip)
            return loss

        def timed(fn, n):
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for i in range(n):
                r = fn(i)
            e1.record()
            barrier()
            ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
            if world > 1:
                dist.all_reduce(ms, op=dist.ReduceOp.MAX)
            return ms.item() / n, r

        # ten warm-up steps by default: three 14 ms steps right after the GEMM tuner's host-bound first step are ~50 ms of GPU work, and the
        # first timed steps were seen at 2.3 x their steady time once in a while (32.6 vs 14.0 ms, profiles/bench_r02_final2_outlier.json)
        for i in range(warmup):
            step(i)
        n0 = sd.lib().seqdiff_launch_count()  # counted over the timed steps (the warm-up steps also hold the GEMM tuner's candidate launches)
        ms_full, loss = timed(lambda i: step(i), steps)                       # bucketed all-reduce under the backward pass
        launches_per_step = (sd.lib().seqdiff_launch_count() - n0) // max(steps, 1)
        if outputs is not None:  # outside the timed loops: timed() ends in a synchronise and the next one starts with one
            outputs.update({k: v.cpu() for k, v in training_outputs(sd, opt, loss).items()})
        ms_block, _ = timed(lambda i: step(i, overlap=False), steps) if world > 1 else (ms_full, None)  # all-reduce after the backward pass
        ms_nocomm, _ = timed(lambda i: step(i, skip=True), steps)
        opt.overlap = True
        ms_ar, _ = timed(lambda i: opt.all_reduce_grads(), steps) if world > 1 else (0.0, None)
        nbytes = opt.last_allreduce_bytes
        flops = 3 * 18.369e9 * global_batch  # forward + backward ~ 3x the forward's algorithmic FLOPs
        peak, _, _ = measured_peaks()
        rec = {"workload": f"BASELINE configs[3]: training step, global batch {global_batch} graphs ({Bl} on this rank), L=128, T=50, dropout 0.1, "
                           "AdamW lr 5e-5 wd 0.1, clip 1.0, one NCCL gradient all-reduce per step",
               "scaling": "weak" if weak else "strong", "global_batch": global_batch, "graphs_per_gpu": Bl, "dtype": precision,
               "value": global_batch / (ms_full * 1e-3), "unit": "graphs/s (training)", "steps_per_s": 1e3 / ms_full, "ms_per_step": ms_full,
               "ms_per_step_without_allreduce": ms_nocomm, "ms_per_step_allreduce_after_backward": ms_block, "ms_allreduce_alone": ms_ar,
               "allreduce": "4 buckets in backward order on a communication stream, each behind the CUDA event the backward pass records "
                            "when that bucket is final (seqdiff_train_set_bucket_events)",
               "exposed_allreduce_frac": max(0.0, (ms_full - ms_nocomm) / ms_full) if world > 1 else 0.0,
               "exposed_allreduce_frac_without_overlap": max(0.0, (ms_block - ms_nocomm) / ms_block) if world > 1 else 0.0,
               "allreduce_bytes": int(nbytes), "grad_comm": grad_comm, "live_parameters": int(opt.flat.live_numel),
               "allreduce_bus_GBps": (2.0 * (world - 1) / world * nbytes / (ms_ar * 1e-3) / 1e9) if (world > 1 and ms_ar > 0) else None,
               "train_flops_frac_of_peak": flops / world / (ms_full * 1e-3) / 1e12 / peak, "launches_per_step": int(launches_per_step),
               "loss_last": float(loss), "steps": steps, "warmup": warmup}
        model.release()
        del model, opt
        torch.cuda.empty_cache()
        return rec
    finally:
        L = keep_L


# ----------------------------------------------------------------------------------------------------
def main():
    def positive_int(s):
        v = int(s)
        if v < 1:
            raise argparse.ArgumentTypeError(f"needs at least 1, got {v}")
        return v

    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=positive_int, default=5, help="timed steps")
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=0, help="pocket graphs per GPU (default: the workload's)")
    ap.add_argument("--timesteps", type=int, default=0, help="T (default: the workload's; smaller only for profiling runs)")
    ap.add_argument("--precision", default="bf16", choices=["bf16", "fp16", "fp32"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--workload", default="cfg2", choices=["cfg2", "cfg3", "cfg4"], help="cfg2 = headline (B=64/GPU, L=128); cfg3 = 256 ext-pockets of 512 residues sharded over the GPUs (strong scaling)")
    ap.add_argument("--no-extras", action="store_true", help="skip e2e / roofline / cpu legs (profiling runs)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed (rank 0) as DIR/<name>.npy, "
                                                          f"{DUMP_BYTES >> 20} MB at most")
    args = ap.parse_args()
    global L
    wl = WORKLOADS[args.workload]
    L = wl["L"]
    world_env = int(os.environ.get("WORLD_SIZE", "1"))
    if not args.batch:
        args.batch = wl["batch"] if wl["scaling"] == "weak" else max(1, wl["batch"] // world_env)
    if not args.timesteps:
        args.timesteps = wl["T"]
    args.wl = wl
    if args.impl == "reference":
        return run_reference_arm(args)

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    # stdout carries exactly ONE line (the JSON): anything a library writes to fd 1 meanwhile (NCCL prints its version
    # banner there when NCCL_DEBUG is set) is sent to stderr; fd 1 is restored just before the result is printed
    sys.stdout.flush()
    _saved_stdout_fd = os.dup(1)
    os.dup2(2, 1)

    def emit(obj):
        sys.stdout.flush()
        os.dup2(_saved_stdout_fd, 1)
        print(json.dumps(obj), flush=True)

    if not torch.cuda.is_available():
        emit({"error": "no CUDA device: this benchmark has no CPU fallback (use --impl reference for the CPU arm)"})
        return 1
    torch.cuda.set_device(local)
    dev = torch.device(f"cuda:{local}")
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=dev)

    import seqdiff_b200 as sd
    lib = sd.lib()
    sd.sample.DEVICE = dev

    def barrier0():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    if args.workload == "cfg4":  # the training configuration on its own: one line whose value is training graphs/s
        outputs = {} if args.dump_outputs else None
        with ClockSampler(local) as clk:
            rec = cfg4_train_record(sd, dev, world, rank, barrier0, args.precision, steps=args.steps, warmup=max(args.warmup, 3), outputs=outputs)
        if rank == 0 and outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
        if rank == 0:
            emit({"metric": "training graphs/s (forward + backward + gradient all-reduce + clip + AdamW; cfg4: global batch 128, L=128)",
                  "value": rec["value"], "unit": rec["unit"], "n_gpus": world, "steps": rec["steps"], "warmup": rec["warmup"],
                  "ms_per_step": rec["ms_per_step"], "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": args.precision,
                  "data": "synthetic", "config": {"workload": rec["workload"], "l2": "activations + 244 MB of gradients per step >> 126 MB L2"},
                  "clocks": clk.summary(), "gpu_launches": rec["launches_per_step"] * rec["steps"], "cfg4_train": rec})
        if world > 1:
            dist.destroy_process_group()
        return 0
    sd.sample.CONFIG.update(timesteps=args.timesteps, max_seq_len=L, batch_size=args.batch)
    B, T = args.batch, args.timesteps
    torch.manual_seed(0)  # identical random-init weights on every rank (replicated model, 145 MB bf16)
    common = dict(max_position_embeddings=L, intermediate_size=I, num_hidden_layers=NL, position_embedding_type="relative_key")
    model = sd.ConditionalBertForDiffusionBase(sd.BertConfig(**common), sd.BertConfig(**common, is_decoder=True, add_cross_attention=True), 20)
    # reference init leaves decoder_normalize an exact identity (gates 0); same FLOPs either way, keep the reference init
    model = model.eval().to(dev)
    model.precision = args.precision
    sched = sd.PredefinedNoiseScheduleDiscrete("cosine", T)
    trans = sd.BlosumTransition(x_classes=20, timestep=500)
    batch, x_T = synthetic_workload(B, seed_offset=1000 * rank, n_lig=wl["n_lig"], n_rec=wl["n_rec"])
    gid0 = rank * B  # global graph ids key the Philox noise: results do not depend on the sharding
    dbatch = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in batch.items()}
    dx_T = x_T.to(dev)

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize(dev)

    def one_sampling():
        return sd.denoise_tensors(dbatch, model, sched, trans, True, timesteps=T, x_T=dx_T, seed=5, graph_id0=gid0)

    # ---- device-resident throughput: K full T-step samplings, CUDA events on the launching stream -------
    for _ in range(args.warmup):
        one_sampling()
    barrier()
    n0 = lib.seqdiff_launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    prof_range = os.environ.get("SEQDIFF_PROFILER_RANGE") == "1"  # ncu --profile-from-start off: capture the timed region only
    if prof_range:
        torch.cuda.cudart().cudaProfilerStart()
    with ClockSampler(local) as clk:
        e0.record()
        for _ in range(args.steps):
            out = one_sampling()
        e1.record()
        barrier()
    if prof_range:
        torch.cuda.cudart().cudaProfilerStop()
    launches = lib.seqdiff_launch_count() - n0
    ms = torch.tensor([e0.elapsed_time(e1)], device=dev)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms = ms.item()
    value = world * B * T * args.steps / (ms * 1e-3)
    assert torch.isfinite(out).all()
    # denoise_tensors returns the final [B, L, 20] logits of the sampling (raw logits of the last step, as the reference's denoise)
    outputs = {"final_logits": out.cpu()} if args.dump_outputs else None

    # ---- the same samplings with ragged packing (valid prefixes only; bit-identical at every position denoise() reads) ----
    packed_rec = None
    if args.precision != "fp32":
        run_packed = lambda: sd.denoise_tensors(dbatch, model, sched, trans, True, timesteps=T, x_T=dx_T, seed=5, graph_id0=gid0, packed=True)
        for _ in range(max(1, args.warmup // 2)):
            outp = run_packed()
        barrier()
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record()
        for _ in range(args.steps):
            outp = run_packed()
        p1.record()
        barrier()
        pms = torch.tensor([p0.elapsed_time(p1)], device=dev)
        if world > 1:
            dist.all_reduce(pms, op=dist.ReduceOp.MAX)
        vmask = dbatch["ligand_attn_mask"].bool()
        tok = (dbatch["ligand_attn_mask"].sum() + dbatch["receptor_attn_mask"].sum()).item() / (2.0 * B * L)
        packed_rec = {"value": world * B * T * args.steps / (pms.item() * 1e-3), "unit": UNIT, "ms_per_step": pms.item() / args.steps,
                      "valid_token_frac": tok, "identical_to_padded_at_valid_positions": bool(torch.equal(outp[vmask], out[vmask])),
                      "note": "ragged packing (seqdiff_sample_ex flag 1): M = sum of lengths; `value` above is the padded computation"}
        if outputs is not None:
            outputs["final_logits_packed"] = outp.cpu()
    if rank == 0 and outputs is not None:
        dump_outputs(args.dump_outputs, outputs)

    result = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
              "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": wl["scaling"], "vs_baseline": None, "dtype": args.precision,
              "data": "synthetic",
              "config": workload_config(wl, B, T, world),
              "derived": {"pocket_graphs_per_s": value / T, "edge_msgs_per_s": value * 15 * L * L},
              "clocks": clk.summary(), "gpu_launches": int(launches)}
    if packed_rec is not None:
        result["packed"] = packed_rec

    if not args.no_extras and args.workload == "cfg2":
        # ---- the two other multi-GPU configurations BASELINE.json names, on the ranks of THIS job (all ranks take part) ----
        for key, fn in (("cfg3_strong", cfg3_strong_record), ("cfg4_train", cfg4_train_record)):
            try:
                result[key] = fn(sd, dev, world, rank, barrier, args.precision)
            except Exception as ex:  # extras never cost the headline line
                result[key] = {"error": f"{type(ex).__name__}: {str(ex)[:300]}"}
                barrier()
        if world > 1 and "error" not in result["cfg4_train"]:
            # the per-process reading of the same configuration (128 graphs on EVERY GPU, as Lightning DDP shards a DataLoader)
            try:
                result["cfg4_train"]["weak_128_per_gpu"] = cfg4_train_record(sd, dev, world, rank, barrier, args.precision, weak=True)
            except Exception as ex:
                result["cfg4_train"]["weak_128_per_gpu"] = {"error": f"{type(ex).__name__}: {str(ex)[:300]}"}
                barrier()

    if not args.no_extras:
        # ---- end to end through the public API: denoise(batch_on_host, ...) -> decoded sequences on the host ----
        pinned = {k: (v.pin_memory() if torch.is_tensor(v) else v) for k, v in batch.items()}
        px_T = x_T.pin_memory()
        # loop inputs + x_T + the [T,3,20,20] tables; the decode kernel also takes the true sequence and the mask on the device
        h2d = sum(v.numel() * v.element_size() for k, v in pinned.items() if torch.is_tensor(v))
        h2d += pinned["ligand_attn_mask"].numel() * 4 + px_T.numel() * 4 + T * 3 * 400 * 4
        d2h = 2 * B * L + B * 2 * 8  # decode kernel output: pred / true indices (u8) + per-graph (matches, valid) counts (i64)
        import contextlib
        import io
        with contextlib.redirect_stdout(io.StringIO()):
            sd.denoise(pinned, model, sched, trans, True, timesteps=T, x_T=px_T, seed=5, graph_id0=gid0)
            barrier()
            t0 = time.perf_counter()
            for _ in range(args.steps):
                ids, true_seq, pred_seq, rates = sd.denoise(pinned, model, sched, trans, True, timesteps=T, x_T=px_T, seed=5, graph_id0=gid0)
            barrier()
            dt = torch.tensor([time.perf_counter() - t0], device=dev)
        if world > 1:
            dist.all_reduce(dt, op=dist.ReduceOp.MAX)
        result["e2e"] = {"value": world * B * T * args.steps / dt.item(), "unit": UNIT, "h2d_bytes_per_step": int(h2d),
                         "d2h_bytes_per_step": int(d2h), "api": "denoise(batch_on_pinned_host, model, noise_schedule, transition, diverse)"}
        if packed_rec is not None:
            with contextlib.redirect_stdout(io.StringIO()):
                sd.denoise(pinned, model, sched, trans, True, timesteps=T, x_T=px_T, seed=5, graph_id0=gid0, packed=True)
                barrier()
                t0 = time.perf_counter()
                for _ in range(args.steps):
                    ids_p, true_p, pred_p, rates_p = sd.denoise(pinned, model, sched, trans, True, timesteps=T, x_T=px_T, seed=5, graph_id0=gid0, packed=True)
                barrier()
                dtp = torch.tensor([time.perf_counter() - t0], device=dev)
            if world > 1:
                dist.all_reduce(dtp, op=dist.ReduceOp.MAX)
            result["packed"]["e2e"] = {"value": world * B * T * args.steps / dtp.item(), "unit": UNIT,
                                       "same_decoded_sequences_as_padded": bool(pred_p == pred_seq and rates_p == rates),
                                       "api": "denoise(batch_on_pinned_host, ..., packed=True)"}

        # ---- roofline of the dominant kernel (tcgen05 GEMM), timed live with CUDA events (library profiler) ----
        if rank == 0:
            t_arr = torch.full((B, 1), float(T - 1), device=dev)
            fwd_args = (t_arr, dx_T, dbatch["ligand_angles"], dbatch["ligand_attn_mask"], dbatch["receptor_seq"], dbatch["receptor_angles"],
                        dbatch["receptor_attn_mask"])
            with torch.no_grad():
                for _ in range(2):
                    model(*fwd_args)
                torch.cuda.synchronize(dev)
                reps = 5
                prof = sd._cabi.profile(lambda: [model(*fwd_args) for _ in range(reps)])
            total_ms = sum(v[0] for v in prof.values())
            gemm_ms = sum(v[0] for k, v in prof.items() if k.startswith("gemm_tcgen05"))  # 1-CTA and CTA-pair variants
            gemm_n = sum(v[1] for k, v in prof.items() if k.startswith("gemm_tcgen05"))
            peak, peak_src, hbm = measured_peaks()
            flops = gemm_flops_per_forward(B) * reps
            achieved = flops / (gemm_ms * 1e-3) / 1e12 if gemm_ms > 0 else 0.0
            traffic = None
            tp = os.path.join(ROOT, "profiles", "roofline_traffic.json")
            if os.path.exists(tp):
                traffic = json.load(open(tp)).get("gemm_tcgen05_dram_bytes_per_launch")
            result["roofline"] = {"kernel": "gemm_tcgen05_kernel (50 launches per forward; 1-CTA and cta_group::2 variants)", "bound": "tensor", "achieved": achieved, "peak": peak,
                                  "unit": "TFLOP/s", "frac": achieved / peak, "traffic": traffic, "peak_source": peak_src,
                                  "flops_per_launch_avg": flops / max(gemm_n, 1), "avg_launch_us": 1e3 * gemm_ms / max(gemm_n, 1),
                                  "share_of_forward": gemm_ms / total_ms if total_ms else None,
                                  "kernel_ms_per_forward": {k: v[0] / reps for k, v in sorted(prof.items())},
                                  "whole_step_model_flops_frac": (value / world) * wl["flops"] / 1e12 / peak}
            # ---- the same GEMM shapes timed alone: every (M, N, K, epilogue) of the forward as 20 launches in a captured CUDA
            #      graph (no CPU launch gaps, no other kernels between them), CUDA events around the replay; against the BURST
            #      peak, which is the denominator for a kernel timed in isolation ----
            try:
                import ctypes as _ct
                Ml_, Mt_ = B * L, 2 * B * L
                shapes = [(1, Mt_, H, H, 2, False), (1, Mt_, 6 * H, H, 0, False), (1, Mt_, 3 * H, H, 0, False), (1, Mt_, H, H, 0, True),
                          (1, Mt_, 4 * H, H, 1, False), (1, Mt_, H, 4 * H, 0, True), (1, Ml_, 2 * NL * H, H, 0, False),
                          (NL + 1, Ml_, 3 * H, H, 0, False), (2 * NL + 1, Ml_, H, H, 0, True), (NL + 1, Ml_, H, H, 0, False),
                          (NL, Ml_, I, H, 1, False), (NL, Ml_, H, I, 0, True), (1, Ml_, 4 * H, H, 1, False), (1, Ml_, H, 4 * H, 0, True)]
                pp = sd._cabi.ptr
                iso_us, iso_fl, bound_us, per_shape = 0.0, 0.0, 0.0, []
                burst0 = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("bf16_tflops", 1590.0) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else 1590.0
                for cnt, M_, N_, K_, epi_, res_ in shapes:
                    A_ = torch.randn(M_, K_, device=dev).bfloat16()
                    W_ = (torch.randn(N_, K_, device=dev) / math.sqrt(K_)).bfloat16()
                    b_ = torch.randn(N_, device=dev)
                    R_ = torch.randn(M_, N_, device=dev) if res_ else None
                    C_ = torch.empty(M_, N_, device=dev, dtype=torch.float32 if res_ else torch.bfloat16)
                    call_ = lambda st_: lib.seqdiff_op_gemm(1, M_, N_, K_, pp(A_), pp(W_), pp(b_), pp(R_), epi_, pp(C_), st_)
                    assert call_(_ct.c_void_p(torch.cuda.current_stream(dev).cuda_stream)) == 0  # first call: tile tuner
                    torch.cuda.synchronize(dev)
                    gr_ = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(gr_):
                        cs_ = _ct.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
                        for _ in range(20):
                            assert call_(cs_) == 0
                    gr_.replay()
                    g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    torch.cuda.synchronize(dev)
                    g0.record()
                    gr_.replay()
                    g1.record()
                    torch.cuda.synchronize(dev)
                    us_ = g0.elapsed_time(g1) / 20 * 1e3
                    iso_us += cnt * us_
                    iso_fl += cnt * 2.0 * M_ * N_ * K_
                    # the two floors of this launch: tensor pipe at the burst peak, and its compulsory HBM bytes (16-bit A and W once,
                    # fp32 residual in + fp32 C out for the residual form, else 16-bit C out) at the measured copy rate
                    by_ = 2.0 * M_ * K_ + 2.0 * N_ * K_ + (8.0 * M_ * N_ if res_ else 2.0 * M_ * N_)
                    t_mma, t_mem = 2.0 * M_ * N_ * K_ / burst0 / 1e6, by_ / hbm / 1e3
                    bound_us += cnt * max(t_mma, t_mem)
                    per_shape.append({"M": M_, "N": N_, "K": K_, "resid_fp32": bool(res_), "count": cnt, "us": round(us_, 2), "tflops": round(2e-6 * M_ * N_ * K_ / us_, 1),
                                      "floor_us_tensor": round(t_mma, 2), "floor_us_hbm": round(t_mem, 2), "frac_of_floor": round(max(t_mma, t_mem) / us_, 3)})
                    del gr_
                burst = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))).get("bf16_tflops", 1590.0) if os.path.exists(os.path.join(ROOT, "MEASURED_PEAKS.json")) else 1590.0
                result["roofline_isolated"] = {"kernel": "gemm_tcgen05_kernel, each shape of the forward as 20 launches in a captured graph", "bound": "tensor",
                                               "achieved": iso_fl / iso_us / 1e6, "peak": burst, "unit": "TFLOP/s", "frac": iso_fl / iso_us / 1e6 / burst,
                                               "gemm_us_per_forward": iso_us, "flops_per_forward": iso_fl,
                                               "two_floor_bound_us_per_forward": bound_us, "frac_of_two_floor_bound": bound_us / iso_us,
                                               "two_floor_note": "per launch max(FLOPs / burst tensor peak, compulsory HBM bytes / measured copy rate): the fp32-residual "
                                                                 "GEMMs (N = 768) are HBM-bound at 153 FLOP/B, so the tensor peak alone overstates what they can reach",
                                               "per_shape": per_shape,
                                               "peak_source": "MEASURED_PEAKS.json bf16_tflops (burst: kernel timed alone)"}
            except Exception as ex:  # the isolated sweep is an extra; never fail the bench line over it
                result["roofline_isolated"] = {"error": str(ex)[:200]}
            # ---- the HBM-bound kernel of the path: reverse step at a size that streams (256 graphs x 512 residues) ----
            RB, RL = 256, 512
            rx = torch.nn.functional.one_hot(torch.randint(0, 20, (RB, RL), device=dev), 20).float()
            rlg = torch.randn(RB, RL, 20, device=dev)
            rs = torch.full((RB, 1), float(T // 2))
            call = lambda: sd.sample_p_zs_given_zt_discrete((rs + 1) / T, rs / T, rx, rlg, sched, trans, True, False)
            for _ in range(3):
                call()
            tabs = sd.utils.step_tables((rs + 1) / T, rs / T, sched, trans).to(dev)
            import ctypes
            rout = torch.empty_like(rx)
            stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            p = sd._cabi.ptr
            raw = lambda st=stream: lib.seqdiff_reverse_step(p(tabs), RB, RB, RL, p(rx), p(rlg), 1, None, 5, 0, 1, p(rout), None, st)
            for _ in range(3):
                raw()
            torch.cuda.synchronize(dev)
            # device time per launch: 50 launches captured in a CUDA graph (50 eager launches from Python are bound by the
            # interpreter, not by the 10 us kernel), CUDA events around the replay on the launching stream
            gr = torch.cuda.CUDAGraph()
            with torch.cuda.graph(gr):
                cst = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
                for _ in range(50):
                    assert raw(cst) == 0
            gr.replay()
            r0, r1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize(dev)
            r0.record()
            gr.replay()
            r1.record()
            torch.cuda.synchronize(dev)
            rus = r0.elapsed_time(r1) / 50 * 1e3
            rbytes = RB * RL * 240
            result["reverse_step_roofline"] = {"kernel": "reverse_step_kernel", "bound": "hbm", "residues": RB * RL, "bytes_per_residue": 240,
                                               "avg_launch_us": rus, "achieved": rbytes / rus / 1e3, "peak": hbm, "unit": "GB/s",
                                               "frac": rbytes / rus / 1e3 / hbm, "note": "31 MB per launch fits L2 (126 MB): back-to-back launches re-hit L2, so this is an upper bound on the HBM-resident rate"}

        # ---- BASELINE configs[0] shape on the GPU: ONE 128-slot pocket + peptide graph (latency; SURVEY.md section 8d cfg 1) ----
        if rank == 0:
            try:
                b1, x1 = synthetic_workload(1, n_lig=(30, 30), n_rec=(98, 98))
                d1 = {k: (v.to(dev) if torch.is_tensor(v) else v) for k, v in b1.items()}
                dx1 = x1.to(dev)
                a1 = (torch.full((1, 1), 7.0, device=dev), dx1, d1["ligand_angles"], d1["ligand_attn_mask"], d1["receptor_seq"], d1["receptor_angles"],
                      d1["receptor_attn_mask"])
                with torch.no_grad():
                    for _ in range(5):
                        model(*a1)
                    torch.cuda.synchronize(dev)
                    c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                    c0.record()
                    for _ in range(20):
                        model(*a1)
                    c1.record()
                    torch.cuda.synchronize(dev)
                    fwd_us = c0.elapsed_time(c1) / 20 * 1e3
                    T1 = 100
                    s1 = sd.PredefinedNoiseScheduleDiscrete("cosine", T1)
                    run1 = lambda: sd.denoise_tensors(d1, model, s1, trans, True, timesteps=T1, x_T=dx1, seed=5, graph_id0=0)
                    run1()
                    torch.cuda.synchronize(dev)
                    c0.record()
                    for _ in range(3):
                        run1()
                    c1.record()
                    torch.cuda.synchronize(dev)
                    step_us = c0.elapsed_time(c1) / (3 * T1) * 1e3
                result["cfg1_latency"] = {"workload": f"BASELINE configs[0] shape: one graph, L=128 slots (30 peptide + 98 pocket residues valid), {args.precision}",
                                          "forward_call_us": fwd_us, "forward_note": "model(...) from Python: ~60 eager launches + ctypes, device-timed over 20 calls",
                                          "sampling_step_us": step_us, "sampling_note": f"forward + reverse step inside the replayed CUDA graph of denoise (T={T1})",
                                          "weight_streaming_floor_us": 145e6 / hbm / 1e3}
            except Exception as ex:
                result["cfg1_latency"] = {"error": f"{type(ex).__name__}: {str(ex)[:200]}"}

        # ---- the reference algorithm on this box's host cores (reported baseline, not the target) ----
        if rank == 0 and world == 1 and not args.no_cpu_baseline:
            state = {k: v.detach().cpu().clone() for k, v in model.state_dict().items()}
            threads = os.cpu_count() or 1
            cb = B if args.workload == "cfg2" else 4
            cbatch = {k: (v[:cb] if torch.is_tensor(v) else v) for k, v in batch.items()}
            times = cpu_reference_steps(state, cbatch, x_T[:cb], T, 3, 1, threads)
            result["cpu_baseline"] = {"value": cb * len(times) / sum(times), "unit": UNIT, "cores": threads, "kind": "port",
                                      "sample": f"{len(times)} denoise steps x {cb} graphs (of {T}); oracle port incl. the reference's Python multinomial loop"}

    if rank == 0:
        emit(result)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
