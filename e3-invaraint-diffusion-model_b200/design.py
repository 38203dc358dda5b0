"""Peptide design in one call: P pockets x K1 backbones from the structure sampler x K2 sequences per backbone from the sequence sampler.

The reference runs this pipeline as two scripts: structure_model/sample.py writes the generated backbone angles to a pickle (every
complex trimmed to its ligand length), and sample_by_generated_angles.py reads them back, zero-pads them to the sequence model's
length (load_generated_angles) and samples one sequence per backbone.  Here both samplers run on the device and the hand-off is a few
torch ops on the final angles:
  * structure: `p_sample_loop_tensors(num_samples=K1)` -- the pocket's receptor branch runs once for its K1 backbones, and only the
    final angles are kept (no [T,B,L,F] history, no host copy);
  * hand-off: the positions at or beyond each ligand length are zeroed -- exactly what the trim of structure_model.sample() followed
    by the zero pad of load_generated_angles produces -- then the angles are padded from the structure length to the sequence
    length and every backbone is repeated K2 times;
  * sequence: `denoise_tensors(num_samples=K1*K2)` with one ligand-angle entry per sample -- the pocket's receptor rows run once per
    step for its K1*K2 sequences.
Sample k of backbone j of pocket p is sequence graph (p*K1 + j)*K2 + k; backbone j of pocket p is structure graph p*K1 + j.  The
results equal, bit for bit, the host composition on the batch with every pocket repeated (tests/test_design.py).
"""
from __future__ import annotations

from typing import Optional

import torch
from torch.nn import functional as F

from . import _cabi
from . import structure_model as SM
from .model import AA_VOCAB
from .sample import CONFIG, check_num_samples, decode_batch, denoise_tensors, score
from .utils import DiscreteUniformTransition, PredefinedNoiseScheduleDiscrete

STRUCT_KEYS = ("ligand_attn_mask", "receptor_seq", "receptor_angles", "receptor_attn_mask")


def _prefix_lengths(mask: torch.Tensor, name: str) -> torch.Tensor:
    """valid lengths of a {0,1} mask whose rows are prefixes of ones (ValueError otherwise)"""
    m = mask.detach().float().cpu()
    n = (m != 0).sum(dim=1)
    prefix = (torch.arange(m.shape[1])[None, :] < n[:, None]).float()
    if not torch.equal(m, prefix):
        raise ValueError(f"{name} must be a prefix of ones in every row")
    return n


def structure_inputs(batch, Ls: int):
    """The structure model's inputs from a sequence-model batch (LigandBindingSiteDataset layout): its first Ls columns.  Raises
    ValueError when a mask is not a prefix of ones or a ligand / receptor is longer than Ls, since the structure model cannot see it.
    Returns (ligand lengths [P], dict of the four cut tensors)."""
    lig_len = _prefix_lengths(batch["ligand_attn_mask"], "ligand_attn_mask")
    rec_len = _prefix_lengths(batch["receptor_attn_mask"], "receptor_attn_mask")
    if int(lig_len.max()) > Ls or int(rec_len.max()) > Ls:
        raise ValueError(f"a ligand ({int(lig_len.max())}) or receptor ({int(rec_len.max())}) is longer than the structure model's "
                         f"{Ls} positions")
    return lig_len, {k: batch[k][:, :Ls] for k in STRUCT_KEYS}


def _check_counts(num_backbones, num_sequences):
    try:
        return check_num_samples(num_backbones), check_num_samples(num_sequences)
    except ValueError as e:
        raise ValueError(f"num_backbones / num_sequences: {e}") from None


def start_noise(n: int, L: int, feature_size: int) -> torch.Tensor:
    """default structure start state: N(0,1) angles wrapped to [-pi, pi) (the reference datasets' sample_noise)"""
    return SM.modulo_with_wrapped_range(torch.randn(n, L, feature_size))


def sequence_schedule(timesteps=None, noise_schedule=None, transition=None):
    """(T, noise schedule, transition) of the design's sequence sampler: CONFIG["timesteps"] steps of the cosine schedule and
    DiscreteUniformTransition(20) unless given"""
    T_q = CONFIG["timesteps"] if timesteps is None else timesteps
    if noise_schedule is None:
        noise_schedule = PredefinedNoiseScheduleDiscrete(CONFIG["noise_schedule"], T_q)
    if transition is None:
        transition = DiscreteUniformTransition(20)  # as the reference's structure -> sequence script (sample_by_generated_angles.py:253)
    return T_q, noise_schedule, transition


def structure_schedule(struct_betas=None, struct_timesteps=None):
    """(T, betas) of the design's structure sampler: the cosine schedule of structure_model.CONFIG["timesteps"] steps unless given"""
    if struct_betas is None:
        T_s = SM.CONFIG["timesteps"] if struct_timesteps is None else int(struct_timesteps)
        struct_betas = SM.cosine_beta_schedule(T_s)
    T_s = len(struct_betas) if struct_timesteps is None else int(struct_timesteps)
    return T_s, struct_betas


def score_design_backbones(struct_model, batch, K: int, backbone_angles, packed: bool = True, seed=None, struct_betas=None,
                           struct_timesteps=None):
    """backbone_loss [P*K] of design()'s backbones of one batch: backbone j of pocket p (angles trimmed to the ligand length, zero-padded
    back to the structure model's length) scored under its pocket with the design's structure schedule (structure_model.score_backbones).
    Philox graph ids continue the process-wide stream."""
    Ls = struct_model.encoder_config.max_position_embeddings
    _, st = structure_inputs(batch, Ls)
    n, Ll_s = len(backbone_angles), st["ligand_attn_mask"].shape[1]
    x0 = torch.zeros((n, Ll_s, struct_model.feature_size), dtype=torch.float32)
    for i, a in enumerate(backbone_angles):
        a = torch.as_tensor(a, dtype=torch.float32)
        x0[i, :a.shape[0]] = a
    T_s, betas = structure_schedule(struct_betas, struct_timesteps)
    loss, _ = SM.score_backbones(struct_model, st["ligand_attn_mask"], x0, st["receptor_seq"], st["receptor_attn_mask"], st["receptor_angles"],
                                 T_s, betas, seed=seed, packed=packed, num_samples=K)
    return loss.tolist()


def score_designs(seq_model, batch, K: int, backbone_angles, pred_sequences, packed: bool = True, seed=None, timesteps=None, noise_schedule=None,
                  transition=None):
    """(nll_per_residue, perplexity) of design()'s rows of one batch: each predicted sequence scored under its pocket and its own generated
    backbone (the swapped batch of the sequence sampler: backbone angles zero-padded to the batch length, one entry per row), with the
    design's sequence schedule, transition and T.  Philox graph ids continue the process-wide stream."""
    P, Lq, _ = batch["ligand_seq"].shape
    n = P * K
    angles = torch.zeros((n, Lq, 8), dtype=torch.float32)
    seqs = torch.zeros((n, Lq, 20), dtype=torch.float32)
    for i in range(n):
        a = torch.as_tensor(backbone_angles[i], dtype=torch.float32)
        angles[i, :a.shape[0]] = a
        idx = torch.tensor([AA_VOCAB.index(c) for c in pred_sequences[i]], dtype=torch.long)
        seqs[i, :idx.numel()] = F.one_hot(idx, 20).float()
    swapped = dict(batch)
    swapped["ligand_angles"] = angles
    T_q, noise_schedule, transition = sequence_schedule(timesteps, noise_schedule, transition)
    _, _, nll, ppl, _ = score(swapped, seq_model, noise_schedule, transition, sequences=seqs, timesteps=T_q, seed=seed, packed=packed,
                              num_samples=K)
    return nll, ppl


@torch.no_grad()
def design_tensors(struct_model, seq_model, batch, num_backbones: int = 1, num_sequences: int = 1, *, packed: bool = True,
                   struct_betas: Optional[torch.Tensor] = None, struct_timesteps: Optional[int] = None, noise_schedule=None,
                   transition=None, diverse: bool = True, timesteps: Optional[int] = None, x_T: Optional[torch.Tensor] = None,
                   seq_x_T: Optional[torch.Tensor] = None, seed: Optional[int] = None, graph_id0: Optional[int] = None,
                   seq_graph_id0: Optional[int] = None):
    """The device part of `design`: returns (backbones [P*K1, Lq, F], final [P*K1*K2, Lq, 20]), each on its model's device.
    backbones = the structure sampler's final angles, 0 at and beyond each ligand length; final = the sequence sampler's result
    (raw logits of the last step, as denoise_tensors)."""
    K1, K2 = _check_counts(num_backbones, num_sequences)
    P, Lq, _ = batch["ligand_seq"].shape
    Ls = struct_model.encoder_config.max_position_embeddings
    lig_len, st = structure_inputs(batch, Ls)
    Ll_s = st["ligand_attn_mask"].shape[1]
    Fs = struct_model.feature_size
    T_s, struct_betas = structure_schedule(struct_betas, struct_timesteps)
    if x_T is None:
        x_T = start_noise(P * K1, Ll_s, Fs)
    if graph_id0 is None:
        graph_id0 = _cabi.GRAPH_IDS.take(P * K1)
    if seq_graph_id0 is None:
        seq_graph_id0 = _cabi.GRAPH_IDS.take(P * K1 * K2)
    _, angles = SM.p_sample_loop_tensors(struct_model, st["ligand_attn_mask"], x_T, st["receptor_seq"], st["receptor_attn_mask"],
                                         st["receptor_angles"], T_s, struct_betas, graph_id0=graph_id0, seed=seed, keep_history=False,
                                         packed=packed, num_samples=K1)
    # hand-off: sample()'s trim + load_generated_angles' zero pad, then Ls -> Lq and one copy per sequence
    valid = (torch.arange(Ll_s)[None, :] < lig_len.repeat_interleave(K1)[:, None]).to(angles.device)
    backbones = F.pad(torch.where(valid[..., None], angles, torch.zeros((), device=angles.device)), (0, 0, 0, Lq - Ll_s))
    swapped = dict(batch)
    swapped["ligand_angles"] = backbones.repeat_interleave(K2, dim=0)
    T_q, noise_schedule, transition = sequence_schedule(timesteps, noise_schedule, transition)
    final = denoise_tensors(swapped, seq_model, noise_schedule, transition, diverse, timesteps=T_q, x_T=seq_x_T, graph_id0=seq_graph_id0,
                            seed=seed, packed=packed, num_samples=K1 * K2)
    return backbones, final


@torch.no_grad()
def design(struct_model, seq_model, batch, num_backbones: int = 1, num_sequences: int = 1, **kw):
    """P pockets x K1 = num_backbones backbones x K2 = num_sequences sequences in one call.  `batch` is a sequence-model batch
    (LigandBindingSiteDataset layout); the structure model reads its first Ls = max_position_embeddings columns.  Keywords (see
    design_tensors): packed (default True; ragged packing in both samplers), struct_betas / struct_timesteps (structure schedule,
    default the cosine schedule of structure_model.CONFIG["timesteps"] steps), noise_schedule / transition / diverse / timesteps (sequence
    sampler, default transition DiscreteUniformTransition(20)), x_T [P*K1, Ls, F] (structure start; default wrapped torch.randn --
    pass the dataset's own sample_noise here), seq_x_T [P*K1*K2, Lq, 20], seed, graph_id0 / seq_graph_id0 (Philox bases of the two
    samplers; None continues the process-wide stream).
    Returns (structure_ids, backbone, backbone_angles, true_sequences, pred_sequences, recovery_rates), P*K1*K2 entries each in
    (pocket, backbone, sequence) order: backbone = j, backbone_angles = the backbone's angles trimmed to the ligand length
    (numpy [len, F], the array structure_model.sample() returns as its last step)."""
    K1, K2 = _check_counts(num_backbones, num_sequences)
    backbones, final = design_tensors(struct_model, seq_model, batch, K1, K2, **kw)
    ids, true_seqs, pred_seqs, rates = decode_batch(final, batch, K1 * K2)
    lig_len = batch["ligand_attn_mask"].detach().float().cpu().sum(dim=1).long()
    host = backbones.cpu()
    trimmed = [host[b, :int(lig_len[b // K1])].numpy() for b in range(host.shape[0])]
    n = len(ids)
    return ids, [(i // K2) % K1 for i in range(n)], [trimmed[i // K2] for i in range(n)], true_seqs, pred_seqs, rates


def design_dataset(dataloader, struct_model, seq_model, num_backbones: int = 1, num_sequences: int = 1, output_path=None, design_fn=None,
                   score: bool = False, score_backbones: bool = False, **kw):
    """Every batch of `dataloader` through `design`; returns sample_dataset's DataFrame (structure_ids / true_sequence /
    predict_sequence / recovery_rate) plus a `backbone` column, pickled to `output_path` like sample_dataset when given.
    score=True adds `nll_per_residue` and `perplexity`: each predicted sequence scored under its pocket and its own backbone
    (score_designs), the candidates' model score where no native peptide exists.
    score_backbones=True adds `backbone_loss`: each backbone scored once under its pocket by the structure model's training objective
    averaged over the timesteps (score_design_backbones, with the design's struct_betas / struct_timesteps, seed and packing), repeated
    over the backbone's num_sequences rows; lower = more native-like to the structure model."""
    import pandas as pd
    K1, K2 = _check_counts(num_backbones, num_sequences)
    fn = design if design_fn is None else design_fn
    skw = {k: kw[k] for k in ("packed", "seed", "timesteps", "noise_schedule", "transition") if k in kw}
    bkw = {k: kw[k] for k in ("packed", "seed", "struct_betas", "struct_timesteps") if k in kw}
    rows = []
    for idx, batch in enumerate(dataloader):
        print(f"Generating Batch {idx}")
        ids, backbone, angles, true_seqs, pred_seqs, rates = fn(struct_model, seq_model, batch, K1, K2, **kw)
        cols = [ids, true_seqs, pred_seqs, rates, backbone]
        if score:
            cols.extend(score_designs(seq_model, batch, K1 * K2, angles, pred_seqs, **skw))
        if score_backbones:
            loss = score_design_backbones(struct_model, batch, K1, angles[::K2], **bkw)
            cols.append([loss[i // K2] for i in range(len(ids))])
        rows.extend(zip(*cols))
    columns = ["structure_ids", "true_sequence", "predict_sequence", "recovery_rate", "backbone"]
    res = pd.DataFrame(rows, columns=columns + (["nll_per_residue", "perplexity"] if score else []) + (["backbone_loss"] if score_backbones else []))
    if output_path is not None:
        res.to_pickle(output_path)
    return res
