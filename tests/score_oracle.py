"""CPU restatement of the sequence score (seqdiff_score_multi / sample.score_tensors) on top of oracle/seqdiff_oracle.py -- test
infrastructure only.  Plain torch, the denoiser in fp32 as the oracle runs it, every sum of the bound in float64.

For native sequence x0 (class a at a valid position) and T steps, step k = T-1 .. 0 uses the sampling loop's tables (t = (k+1)/T,
s = k/T): x_t ~ q(x_t | x0) with prob[i] = Qtb_k[i, a] and the exponential race on E_k; z = denoiser_forward at timestep k (the raw
step index); p = the reverse step's normalised prob (reverse_step_probs), q = the same with one-hot(a) in place of softmax(z);
kl_k = sum_{q_j > 0} q_j (log q_j - log max(p_j, 1e-30)) for k >= 1, the reconstruction term -log softmax(z)_a for k = 0;
ce_k = -log softmax(z)_a at every k.  prior(a) = KL(Qtb_{T-1}[:, a] normalised || uniform over the 20 classes)."""
from __future__ import annotations

import torch
import torch.nn.functional as F

from helpers import O  # (puts the repository root on sys.path for the oracle package)


def step_tables(k: int, T: int, B: int, noise_schedule, transition):
    """(t, s, Qt, Qsb, Qtb) of step k for B graphs, normalised times formed in fp32 like the sampling loop"""
    s_arr = k * torch.ones((B, 1))
    t, s = (s_arr + 1) / T, s_arr / T
    return (t, s) + tuple(O.step_matrices(t, s, noise_schedule, transition))


def q_sample(x0, Qtb, E):
    """x_t ~ q(x_t | x0) at the step's Qtb [B,20,20]: prob[n, i] = Qtb[b, i, x0[n]], exponential race with E [B*L, 20]"""
    B, L, C = x0.shape
    batch = torch.arange(B).repeat_interleave(L)
    prob = (Qtb[batch] @ x0.reshape(B * L, C).unsqueeze(2)).squeeze(-1)
    return F.one_hot(O.sample_indices(prob, True, E).reshape(B, L), C).float()


def posterior_probs(pred, x_t, Qt, Qsb, Qtb):
    """sample.py:162-168 for given class probabilities pred [N, 20] (not logits): the normalised posterior prob [N, 20]"""
    B, L, C = x_t.shape
    batch = torch.arange(B).repeat_interleave(L)
    post = O.posterior_over0(x_t.reshape(B * L, C), Qt, Qsb, Qtb, batch)
    un = (pred.unsqueeze(-1) * post).sum(dim=1)
    un[torch.sum(un, dim=-1) == 0] = 1e-5
    return un / torch.sum(un, dim=-1, keepdim=True)


def kl_terms(q, p):
    """float64 sum_{q_j > 0} q_j (log q_j - log max(p_j, 1e-30)) per row of fp32 q, p [N, 20]"""
    q, p = q.double(), p.double().clamp_min(1e-30)
    return torch.where(q > 0, q * (torch.log(q.clamp_min(1e-300)) - torch.log(p)), torch.zeros((), dtype=torch.float64)).sum(-1)


def prior_terms(Qtb_last):
    """[20] float64: prior(a) = KL(r_a || uniform), r_a = column a of the last step's Qtb [20, 20], normalised"""
    r = Qtb_last.double()
    r = r / r.sum(dim=0, keepdim=True)
    return torch.where(r > 0, r * torch.log(r * r.shape[0]), torch.zeros((), dtype=torch.float64)).sum(dim=0)


def step_terms(k, logits, x0, x_t, Qt, Qsb, Qtb, t, s, noise_schedule, transition):
    """(bound term, ce) [B*L] float64 of step k from the step's logits [B, L, 20]"""
    B, L, C = x0.shape
    a = x0.reshape(B * L, C).argmax(-1)
    ce = -F.log_softmax(logits.reshape(B * L, C).double(), dim=-1).gather(1, a[:, None]).squeeze(1)
    if k == 0:
        return ce, ce
    p = O.reverse_step_probs(t, s, x_t, logits, noise_schedule, transition)
    q = posterior_probs(F.one_hot(a, C).float(), x_t, Qt, Qsb, Qtb)
    return kl_terms(q, p), ce


def score_loop(sd, cfg, batch, x0, noise_schedule, transition, T, noise_E_steps, forward=None):
    """(terms [B, L, 2] float64, prior [B] float64) as score_tensors returns them; noise_E_steps [T, B*L, 20] (entry k at step k).
    forward(k, x_t) -> logits replaces the oracle's denoiser (CPU tests with a stand-in model)."""
    B, L, C = x0.shape
    valid = batch["ligand_attn_mask"] != 0
    terms = torch.zeros((B * L, 2), dtype=torch.float64)
    for k in reversed(range(T)):
        t, s, Qt, Qsb, Qtb = step_tables(k, T, B, noise_schedule, transition)
        x_t = q_sample(x0, Qtb, noise_E_steps[k])
        if forward is None:
            logits = O.denoiser_forward(sd, cfg, k * torch.ones((B, 1)), x_t, batch["ligand_angles"], batch["ligand_attn_mask"],
                                        batch["receptor_seq"], batch["receptor_angles"], batch["receptor_attn_mask"])
        else:
            logits = forward(k, x_t)
        kl, ce = step_terms(k, logits, x0, x_t, Qt, Qsb, Qtb, t, s, noise_schedule, transition)
        terms[:, 0] += kl
        terms[:, 1] += ce
    terms = terms.reshape(B, L, 2) * valid[..., None]
    Qtb_last = step_tables(T - 1, T, 1, noise_schedule, transition)[4][0]
    prior = (prior_terms(Qtb_last)[x0.argmax(-1)] * valid).sum(dim=1)
    return terms, prior


def per_residue(terms, prior, mask, T):
    """(nll_per_residue, perplexity, ce_per_residue) [B] float64"""
    n = (mask != 0).sum(dim=1).double()
    nll = (prior + terms[..., 0].sum(dim=1)) / n
    return nll, torch.exp(nll), terms[..., 1].sum(dim=1) / (T * n)
