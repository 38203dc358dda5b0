"""Plain-torch restatement of the structure model's training objective and of what autograd leaves behind for it: the reference
for tests/test_struct_train.py and the PyTorch arm of scripts/struct_train_bench.py.

The objective is the one the reference inherits from FoldingDiff (structure_model/model.py _get_loss_terms / training_step): for
every angle feature i, d = modulo_with_wrapped_range(known_noise - pred, -pi, pi), l_i = mean over the valid ligand positions of
smooth_l1(d) with beta = pi / 10; loss = mean_i l_i.
"""
import math
from typing import Dict

import torch

from oracle import structdiff_oracle as S

Tensor = torch.Tensor


def angle_loss(pred: Tensor, known_noise: Tensor, mask: Tensor, beta: float = math.pi / 10):
    """(mean_i l_i, [l_i]) for pred, known_noise [B, L, F] and mask [B, L] (valid where != 0)."""
    valid = mask != 0
    d = S.modulo_with_wrapped_range(known_noise - pred, -math.pi, math.pi)[valid]  # [n_valid, F]
    ad = d.abs()
    h = torch.where(ad < beta, 0.5 * d * d / beta, ad - 0.5 * beta)
    per_feature = h.mean(dim=0)
    return per_feature.mean(), per_feature


def training_grads(sd: Dict[str, Tensor], cfg: S.OracleConfig, batch):
    """What `loss = training_step(batch); loss.backward()` leaves behind with dropout off (eval-mode arithmetic): (loss, per-feature
    losses, {state_dict key: gradient or None}, pred).  torch autograd on S.struct_forward; `timestep_projector.W` is a buffer -> None.
    `batch`: corrupted, t, known_noise, ligand_attn_mask, receptor_seq, receptor_angles, receptor_attn_mask."""
    leaf = {k: v.detach().clone().requires_grad_(k != "timestep_projector.W") for k, v in sd.items()}
    pred = S.struct_forward(leaf, cfg, batch["t"], batch["corrupted"], batch["ligand_attn_mask"], batch["receptor_seq"], batch["receptor_angles"],
                            batch["receptor_attn_mask"])
    loss, per_feature = angle_loss(pred, batch["known_noise"], batch["ligand_attn_mask"])
    loss.backward()
    return loss.detach(), per_feature.detach(), {k: (v.grad.detach() if v.grad is not None else None) for k, v in leaf.items()}, pred.detach()
