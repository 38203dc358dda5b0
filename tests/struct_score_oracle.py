"""Plain-torch restatement of the backbone score (seqdiff_struct_score_multi / structure_model.score_backbones_tensors) on top of
oracle/structdiff_oracle.py -- the reference for tests/test_struct_score*.py and the PyTorch arm of scripts/struct_score_bench.py.

For backbone angles x0 [B, L, F] and T steps, step k = T-1 .. 0 draws x_k = wrap(sqrt_ac[k] * x0 + sqrt_1m_ac[k] * eps_k) in fp32 (the
NoisedAnglesDataset / training q-sample, each operation rounded in this order), runs the denoiser at timestep k (the raw step index, as
the sampler passes it) and adds h(wrap(eps_k - pred)) per valid position and feature into float64 sums, h being the training loss's
smooth-L1 with beta = pi / 10 (struct_train_oracle.angle_loss).  per_feature[b, f] = sum_l terms[b, l, f] / (T * n_b), loss = mean_f."""
from __future__ import annotations

import math

import torch

from oracle import structdiff_oracle as S

BETA = math.pi / 10


def q_sample(x0, qs_k, eps):
    """wrap(sqrt_ac * x0 + sqrt_1m_ac * eps) in fp32; qs_k = (sqrt_ac, sqrt_1m_ac) of the step as fp32 scalars"""
    return S.modulo_with_wrapped_range(qs_k[0] * x0.float() + qs_k[1] * eps.float())


def smooth_l1_terms(eps, pred):
    """h(wrap(eps - pred)) per element: the difference and its wrap in fp32, h as angle_loss computes it"""
    d = S.modulo_with_wrapped_range(eps.float() - pred.float(), -math.pi, math.pi)
    ad = d.abs()
    return torch.where(ad < BETA, 0.5 * d * d / BETA, ad - 0.5 * BETA)


def qs_table(betas):
    ab = S.compute_alphas(betas.float())
    return torch.stack([ab["sqrt_alphas_cumprod"], ab["sqrt_one_minus_alphas_cumprod"]], dim=1)


def score_loop(sd, cfg, x0, ligand_mask, receptor_seq, receptor_angles, receptor_mask, betas, noise_steps, forward=None):
    """terms [B, L, F] float64 as score_backbones_tensors returns them (K = 1: one pocket per backbone); noise_steps [T, B, L, F] (entry k
    at step k).  forward(k, x_k) -> pred replaces the oracle's denoiser (CPU tests with a stand-in model)."""
    T = noise_steps.shape[0]
    qs = qs_table(betas)
    valid = (ligand_mask != 0)[..., None]
    terms = torch.zeros(x0.shape, dtype=torch.float64)
    enc = None if forward is not None else S.struct_encode(sd, cfg, receptor_seq, receptor_angles, receptor_mask)
    for k in reversed(range(T)):
        x_k = q_sample(x0, qs[k], noise_steps[k])
        if forward is None:
            t = torch.full((x0.shape[0],), k, dtype=torch.long)
            pred = S.struct_forward(sd, cfg, t, x_k, ligand_mask, receptor_seq, receptor_angles, receptor_mask, encoder_outputs=enc)
        else:
            pred = forward(k, x_k)
        terms += torch.where(valid, smooth_l1_terms(noise_steps[k], pred).double(), torch.zeros((), dtype=torch.float64))
    return terms


def backbone_loss(terms, ligand_mask, T):
    """(loss [B], per_feature [B, F]) float64"""
    n = (ligand_mask != 0).sum(dim=1).double()
    per_feature = terms.sum(dim=1) / (T * n[:, None])
    return per_feature.mean(dim=-1), per_feature
