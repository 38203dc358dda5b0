"""Drop-in for the reference's `structure_model/{model,sample,utils}.py` inference path (SURVEY.md section 8(f) row 3):
the angle denoiser `ConditionalBertForDiffusionBase` (12 + 12 BERT layers, two adaLN SELayers, MLM-style head) and the
Gaussian reverse-diffusion sampler `p_sample` / `p_sample_loop` with the angle wrap -- same names, signatures, state_dict
keys and return values, computed by the hand-written sm_100a kernels of libseqdiff_b200.so (include/seqdiff_b200.h:
seqdiff_struct_*).  As in `model.py`, the nn.Module tree is a parameter container; there is no PyTorch / CPU fallback.

Host-side tables (`cosine_beta_schedule`, `compute_alphas`) use the reference's own torch ops so they are bit-identical.
"""
from __future__ import annotations

import ctypes
import math
from typing import Dict, Optional

import torch
from torch import nn
from torch.nn import functional as F

from . import _cabi
from .sample import check_num_samples
from .model import (BertEmbeddings, BertEncoder, ConditionalBertForDiffusionBase as _SeqBase, GaussianFourierProjection, SELayer,
                    _Container, _BertLayer, BertAttention, _FlatTraining, _Intermediate, _SelfOutput)

SEED = 0          # Philox seed of the in-kernel N(0,1) stream (explicit `noise` tensors override it)
STEP = 1          # structure_model/sample.py:14; only the reference default is implemented
CONFIG = {"batch_size": 64, "timesteps": 1000, "max_seq_len": 64, "pocket_ext": 0}  # the keys sample() reads (sample.py:19-41)


# ---- structure_model/utils.py --------------------------------------------------------------------------------------
def cosine_beta_schedule(timesteps: int, s: float = 8e-3) -> torch.Tensor:
    """reference structure_model/utils.py:8-18."""
    steps = timesteps + 1
    x = torch.linspace(0, timesteps, steps)
    alphas_cumprod = torch.cos(((x / timesteps) + s) / (1 + s) * torch.pi * 0.5) ** 2
    alphas_cumprod = alphas_cumprod / alphas_cumprod[0]
    betas = 1 - (alphas_cumprod[1:] / alphas_cumprod[:-1])
    return torch.clip(betas, 0.0001, 0.9999)


def compute_alphas(betas: torch.Tensor) -> Dict[str, torch.Tensor]:
    """reference structure_model/utils.py:42-58."""
    alphas = 1.0 - betas
    alphas_cumprod = torch.cumprod(alphas, dim=0)
    alphas_cumprod_prev = F.pad(alphas_cumprod[:-1], (1, 0), value=1.0)
    posterior_variance = betas * (1.0 - alphas_cumprod_prev) / (1.0 - alphas_cumprod)
    return {
        "betas": betas,
        "alphas": alphas,
        "alphas_cumprod": alphas_cumprod,
        "sqrt_alphas_cumprod": torch.sqrt(alphas_cumprod),
        "sqrt_one_minus_alphas_cumprod": torch.sqrt(1.0 - alphas_cumprod),
        "posterior_variance": posterior_variance,
    }


def modulo_with_wrapped_range(vals, range_min: float = -math.pi, range_max: float = math.pi):
    """reference structure_model/utils.py:20-40 (host helper; the sampler applies the same wrap inside its kernel)."""
    assert range_min <= 0.0
    assert range_min < range_max
    top_end = range_max - range_min
    return (vals - range_min) % top_end + range_min


def step_coefficients(betas: torch.Tensor) -> torch.Tensor:
    """[T,4] fp32 table the kernels index by step: (1/sqrt(alpha), beta, sqrt(1-alphabar), sqrt(posterior_variance)), each
    derived exactly as p_sample does (structure_model/sample.py:72-85,97)."""
    ab = compute_alphas(betas.detach().float().cpu())
    return torch.stack([1.0 / torch.sqrt(ab["alphas"]), ab["betas"], ab["sqrt_one_minus_alphas_cumprod"],
                        torch.sqrt(ab["posterior_variance"])], dim=1).contiguous()


# ---- structure_model/model.py --------------------------------------------------------------------------------------
class _EncoderLayer(_Container):  # HF BertLayer without cross-attention
    def __init__(self, cfg, relative: bool):
        super().__init__()
        self.attention = BertAttention(cfg, relative)
        self.intermediate = _Intermediate(cfg)
        self.output = _SelfOutput(cfg, cfg.intermediate_size)


class _SelfOnlyEncoder(_Container):
    def __init__(self, cfg, relative: bool):
        super().__init__()
        self.layer = nn.ModuleList([_EncoderLayer(cfg, relative) for _ in range(cfg.num_hidden_layers)])


class AnglesPredictor(_Container):
    """reference structure_model/model.py:119-153."""

    def __init__(self, d_model: int, d_out: int = 4, activation="gelu", eps: float = 1e-12) -> None:
        super().__init__()
        if activation != "gelu":
            raise ValueError("only the reference's default 'gelu' head is implemented in CUDA")
        self.d_model, self.d_out = d_model, d_out
        self.dense1 = nn.Linear(d_model, d_model)
        self.layer_norm = nn.LayerNorm(d_model, eps=eps)
        self.dense2 = nn.Linear(d_model, d_out)


class ConditionalBertForDiffusionBase(_SeqBase):
    """reference structure_model/model.py:155-230.  Reuses the handle management of the sequence-model container
    (`_sync_handle`, `release`, `precision`); only the module tree, the C constructor and `forward` differ."""

    _create_symbol = "seqdiff_struct_model_create"

    def __init__(self, encoder_config, decoder_config, feature_size: int) -> None:
        nn.Module.__init__(self)
        for name in ("hidden_size", "num_attention_heads", "intermediate_size", "num_hidden_layers", "max_position_embeddings"):
            if getattr(encoder_config, name) != getattr(decoder_config, name):
                raise ValueError(f"encoder and decoder configs must agree on {name} (structure_model/sample.py:151-173)")
        self.encoder_config = encoder_config
        self.decoder_config = decoder_config
        self.feature_size = feature_size
        self.precision = "bf16"
        relative = getattr(decoder_config, "position_embedding_type", "absolute") == "relative_key"
        self.receptor_seq_emb = BertEmbeddings(20, encoder_config)
        self.receptor_angle_emb = BertEmbeddings(feature_size, encoder_config)
        self.receptor_emb = SELayer(encoder_config)
        self.encoder = _SelfOnlyEncoder(encoder_config, relative)
        self.ligand_angle_emb = BertEmbeddings(feature_size, decoder_config)
        self.timestep_projector = GaussianFourierProjection(decoder_config.hidden_size)
        self.timestep_emb = SELayer(decoder_config)
        self.decoder = BertEncoder(decoder_config, relative)
        self.angles_predictor = AnglesPredictor(decoder_config.hidden_size, feature_size)
        self._handle = None
        self._handle_sig = None
        self._handle_dev = None
        self._handle_tensors = None

    def initialize_weights(self):  # the structure model keeps torch's default init (no initialize_weights in the reference)
        return None

    def _inputs(self, noised_ligand_angles, ligand_attention_masks, receptor_seq, receptor_angles, receptor_attention_masks, K: int = 1):
        """K > 1: the receptor tensors hold B / K pockets (sampling loop, sample j of pocket p = ligand graph p*K + j)."""
        dev = self._handle_dev
        B, Ll, Fs = noised_ligand_angles.shape
        Lr = receptor_seq.shape[1]
        if Fs != self.feature_size:
            raise ValueError(f"expected {self.feature_size} angle features, got {Fs}")
        if B % K:
            raise ValueError(f"{B} ligand graphs are not {K} samples for each pocket")
        P = B // K

        def prep(x, shape):
            x = x.to(device=dev, dtype=torch.float32).contiguous()
            if tuple(x.shape) != shape:
                raise ValueError(f"expected shape {shape}, got {tuple(x.shape)}")
            return x

        return (B, Ll, Lr, prep(noised_ligand_angles, (B, Ll, Fs)), prep(ligand_attention_masks, (B, Ll)), prep(receptor_seq, (P, Lr, 20)),
                prep(receptor_angles, (P, Lr, Fs)), prep(receptor_attention_masks, (P, Lr)))

    def forward(self, timestep, noised_ligand_angles, ligand_attention_masks, receptor_seq, receptor_angles, receptor_attention_masks,
                ligand_pos_ids=None, receptor_pos_ids=None):
        """reference structure_model/model.py:180-215; `timestep` [B] long (sample.py:136) or float, pos ids ignored."""
        if self.training and (self.decoder_config.hidden_dropout_prob > 0 or self.decoder_config.attention_probs_dropout_prob > 0):
            raise RuntimeError("the CUDA forward implements eval-mode (dropout-free) inference; call model.eval()")
        h = self._sync_handle()
        dev = self._handle_dev
        B, Ll, Lr, x, lm, rs, ra, rm = self._inputs(noised_ligand_angles, ligand_attention_masks, receptor_seq, receptor_angles,
                                                    receptor_attention_masks)
        t = timestep.to(device=dev, dtype=torch.float32).reshape(-1).contiguous()
        if t.numel() != B:
            raise ValueError("timestep must hold one value per batch row")
        out = torch.empty((B, Ll, self.feature_size), device=dev, dtype=torch.float32)
        with torch.cuda.device(dev):
            stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            _cabi.check(_cabi.lib().seqdiff_struct_forward(h, self._precision_code(), B, Ll, Lr, _cabi.ptr(t), _cabi.ptr(x), _cabi.ptr(lm),
                                                           _cabi.ptr(rs), _cabi.ptr(ra), _cabi.ptr(rm), _cabi.ptr(out), stream))
        return out


def _check_valid_ligand(mask):
    if not bool((mask != 0).any()):
        raise ValueError("the batch has no valid ligand position (ligand_attn_mask is all zero): its loss is undefined")


def angle_loss_terms(pred, known_noise, ligand_mask):
    """The F+1 fp64 reduction terms of the structure model's objective (include/seqdiff_b200.h: seqdiff_struct_loss_terms) as a device
    tensor: per-feature sums of the wrapped smooth-L1 over the valid ligand positions, then their count."""
    dev = pred.device
    if dev.type != "cuda":
        raise RuntimeError("angle_loss_terms runs only on a CUDA device (no CPU fallback)")
    Fs = pred.shape[-1]
    pr = pred.to(dtype=torch.float32).reshape(-1, Fs).contiguous()
    kn = known_noise.to(device=dev, dtype=torch.float32).reshape(-1, Fs).contiguous()
    m = ligand_mask.to(device=dev, dtype=torch.float32).reshape(-1).contiguous()
    if not (pr.shape[0] == kn.shape[0] == m.shape[0]):
        raise ValueError("pred, known_noise and ligand_mask must cover the same positions")
    out = torch.empty(Fs + 1, device=dev, dtype=torch.float64)
    with torch.cuda.device(dev):
        stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        _cabi.check(_cabi.lib().seqdiff_struct_loss_terms(pr.shape[0], Fs, _cabi.ptr(pr), _cabi.ptr(kn), _cabi.ptr(m), _cabi.ptr(out), stream))
    return out


class ConditionalBertForDiffusion(_FlatTraining, ConditionalBertForDiffusionBase):
    """reference structure_model/model.py:232-403 without the Lightning base class: the angle denoiser plus its training step.
    `training_step` runs forward (dropout active in train() mode) + the wrapped smooth-L1 loss + the full hand-written backward
    (csrc/train.cu) in one C call; `configure_optimizers` returns the fused clip + AdamW step over the handle's flat parameter space
    (train.py), so `train.fit` trains this model as it trains PeptideDiff.  Only loss="smooth_l1" is implemented."""

    def __init__(self, encoder_config, decoder_config, feature_size: int, *, loss: str = "smooth_l1", learning_rate: float = 5e-5,
                 l2_lambda: float = 0.0, lr_scheduler=None, max_epochs: int = 1, gradient_clip: float = 1.0) -> None:
        if loss != "smooth_l1":
            raise ValueError(f"only the 'smooth_l1' objective is implemented in CUDA, got {loss!r}")
        ConditionalBertForDiffusionBase.__init__(self, encoder_config, decoder_config, feature_size)
        self.loss = loss
        self.lr = learning_rate
        self.l2_lambda = l2_lambda
        self.lr_scheduler = lr_scheduler
        self.max_epochs = max_epochs
        self.gradient_clip = gradient_clip
        self._noise_seed = 0

    def training_step(self, batch, batch_idx):
        """One optimizer step's forward + loss + backward on a NoisedAnglesDataset batch (corrupted, t, known_noise and the keys
        sample() reads).  The gradients land in the flat buffer `self._flat.grads`, ready for `configure_optimizers()["optimizer"].step()`.
        Returns the loss (device scalar); the per-feature losses are kept in `self.last_log`."""
        from . import train as _train
        _check_valid_ligand(batch["ligand_attn_mask"])
        flat = self._flat_params()
        self._train_steps = getattr(self, "_train_steps", 0) + 1
        opt = getattr(self, "_optimizer", None)
        if opt is not None and opt.flat is flat:
            opt.arm_overlap()
        terms, _ = _train.struct_train_step_tensors(self, flat, batch, seed=self._noise_seed, step=self._train_steps)
        if opt is not None and opt.flat is flat:
            opt.launch_overlapped_all_reduce()  # bucket k's all-reduce starts when the backward pass has finished bucket k
        loss, per_feature = _train.angle_loss_from_terms(terms)
        self.last_log = {"train_loss": loss, "train_loss_per_feature": per_feature}
        return loss

    @torch.no_grad()
    def validation_step(self, batch, batch_idx):
        """The same objective on the eval-mode (dropout-free) forward; returns the loss (device scalar), per-feature losses in `last_log`."""
        from . import train as _train
        _check_valid_ligand(batch["ligand_attn_mask"])
        was_training = self.training
        self.eval()
        try:
            pred = self.forward(batch["t"], batch["corrupted"], batch["ligand_attn_mask"], batch["receptor_seq"], batch["receptor_angles"],
                                batch["receptor_attn_mask"])
        finally:
            self.train(was_training)
        loss, per_feature = _train.angle_loss_from_terms(angle_loss_terms(pred, batch["known_noise"], batch["ligand_attn_mask"]))
        self.last_log = {"val_loss": loss, "val_loss_per_feature": per_feature}
        return loss


# ---- structure_model/sample.py -------------------------------------------------------------------------------------
def _p_sample(model, ligand_mask, ligand_angle_noise, receptor_seq, receptor_mask, receptor_angle, timestep, betas, noise, graph_id0, seed,
              wrap: bool):
    t_unique = torch.unique(timestep)
    assert len(t_unique) == 1, f"Got multiple values for t: {t_unique}"
    t_index = int(t_unique.item())
    out = model(timestep, ligand_angle_noise, ligand_mask, receptor_seq, receptor_angle, receptor_mask)
    dev = out.device
    B, L, Fs = out.shape
    if graph_id0 is None:
        graph_id0 = _cabi.GRAPH_IDS.take(B)
    x = ligand_angle_noise.to(device=dev, dtype=torch.float32).contiguous()
    coef = step_coefficients(betas).to(dev)
    z = None if noise is None else noise.to(device=dev, dtype=torch.float32).contiguous()
    res = torch.empty_like(x)
    with torch.cuda.device(dev):
        stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        _cabi.check(_cabi.lib().seqdiff_struct_p_sample(_cabi.ptr(coef), coef.shape[0], t_index, B, L, Fs, _cabi.ptr(x), _cabi.ptr(out),
                                                        _cabi.ptr(z), SEED if seed is None else seed, graph_id0, int(wrap), _cabi.ptr(res),
                                                        stream))
    return res


@torch.no_grad()
def p_sample(model, ligand_mask, ligand_angle_noise, receptor_seq, receptor_mask, receptor_angle, timestep, betas,
             noise: Optional[torch.Tensor] = None, graph_id0: Optional[int] = None, seed: Optional[int] = None) -> torch.Tensor:
    """reference structure_model/sample.py:55-102 (un-wrapped; p_sample_loop applies the wrap).  Extra keywords: `noise`, the
    N(0,1) tensor `torch.randn_like` would have drawn (same-noise parity runs); otherwise counter-based Philox in the kernel,
    keyed by (seed, graph_id0 + b, element, step); graph_id0 = None continues the process-wide noise stream."""
    return _p_sample(model, ligand_mask, ligand_angle_noise, receptor_seq, receptor_mask, receptor_angle, timestep, betas, noise, graph_id0,
                     seed, False)


@torch.no_grad()
def p_sample_wrapped(model, ligand_mask, ligand_angle_noise, receptor_seq, receptor_mask, receptor_angle, timestep, betas,
                     noise: Optional[torch.Tensor] = None, graph_id0: Optional[int] = None, seed: Optional[int] = None) -> torch.Tensor:
    """One iteration of the reference loop body (sample.py:125-141): forward + p_sample + modulo_with_wrapped_range, the update
    and the wrap in ONE kernel."""
    return _p_sample(model, ligand_mask, ligand_angle_noise, receptor_seq, receptor_mask, receptor_angle, timestep, betas, noise, graph_id0,
                     seed, True)


@torch.no_grad()
def p_sample_loop_tensors(model, ligand_mask, ligand_angle_noise, receptor_seq, receptor_mask, receptor_angle, total_timesteps: int, betas,
                          noise_steps: Optional[torch.Tensor] = None, graph_id0: Optional[int] = None, seed: Optional[int] = None,
                          keep_history: bool = True, packed: bool = False, num_samples: int = 1):
    """`p_sample_loop` without the copy to the host: returns (history [T,B,L,F] or None when keep_history=False, final [B,L,F]), both
    on the model's device."""
    K = check_num_samples(num_samples)
    h = model._sync_handle()
    dev = model._handle_dev
    T = int(total_timesteps)
    n_pockets = receptor_seq.shape[0]
    if K > 1 and ligand_mask.shape[0] == n_pockets:
        ligand_mask = ligand_mask.repeat_interleave(K, dim=0)
    if ligand_angle_noise.shape[0] != n_pockets * K:
        raise ValueError(f"ligand_angle_noise must hold P*K = {n_pockets * K} graphs, got {ligand_angle_noise.shape[0]}")
    B, Ll, Lr, x, lm, rs, ra, rm = model._inputs(ligand_angle_noise, ligand_mask, receptor_seq, receptor_angle, receptor_mask, K)
    if graph_id0 is None:
        graph_id0 = _cabi.GRAPH_IDS.take(B)
    Fs = model.feature_size
    coef = step_coefficients(betas)
    if coef.shape[0] != T:
        raise ValueError("betas must hold one value per timestep")
    coef = coef.to(dev)
    z = None
    if noise_steps is not None:
        z = noise_steps.to(device=dev, dtype=torch.float32).contiguous()
        if tuple(z.shape) != (T, B, Ll, Fs):
            raise ValueError("noise_steps must be [T, B, L, F]" if K == 1 else "noise_steps must be [T, P*K, L, F]")
    hist = torch.empty((T, B, Ll, Fs), device=dev, dtype=torch.float32) if keep_history else None
    final = torch.empty((B, Ll, Fs), device=dev, dtype=torch.float32)
    with torch.cuda.device(dev):
        stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        _cabi.check(_cabi.lib().seqdiff_struct_sample_multi(h, model._precision_code(), n_pockets, K, Ll, Lr, T, _cabi.ptr(coef), _cabi.ptr(x),
                                                            _cabi.ptr(lm), _cabi.ptr(rs), _cabi.ptr(ra), _cabi.ptr(rm), _cabi.ptr(z),
                                                            SEED if seed is None else seed, graph_id0, 1 if packed else 0, _cabi.ptr(hist),
                                                            _cabi.ptr(final), stream))
    return hist, final


@torch.no_grad()
def p_sample_loop(model, ligand_mask, ligand_angle_noise, receptor_seq, receptor_mask, receptor_angle, total_timesteps: int, betas,
                  disable_pbar: bool = True, noise_steps: Optional[torch.Tensor] = None, graph_id0: Optional[int] = None, seed: Optional[int] = None,
                  keep_history: bool = True, packed: bool = False, num_samples: int = 1) -> torch.Tensor:
    """reference structure_model/sample.py:104-144: returns a CPU tensor [timesteps, B, L, F] (entry k = wrapped angles after
    the k-th reverse step).  The whole loop is ONE C call (`seqdiff_struct_sample_multi`): the receptor branch is evaluated once, every
    step replays a captured CUDA graph (ligand branch + Gaussian step + wrap), and the history is written by the step kernel --
    one device->host copy at the end instead of one per step.  `keep_history=False` returns only the final [1,B,L,F] entry.
    `noise_steps` [T,B,L,F]: entry i = the N(0,1) draw used at step index i (entry 0 unused).  `graph_id0` = None continues the
    process-wide Philox noise stream, so successive batches / calls draw fresh noise like the reference's `torch.randn_like`.
    `packed=True`: ragged packing (SEQDIFF_SAMPLE_PACKED) -- only the valid prefix of every complex is computed; values at valid
    positions are bit-identical to `packed=False`, padded positions come back as 0 (the reference computes values there, which
    `sample()` trims away).  Masks that are not prefixes of ones, or fp32 precision, run the padded loop.
    `num_samples=K > 1`: K backbones per pocket.  The receptor tensors hold P pockets; ligand_angle_noise, noise_steps, the graph ids
    and the result cover B = P*K graphs, sample j of pocket p being graph p*K + j; ligand_mask is [P*K, L], or [P, L] and repeated.
    The receptor branch runs once per pocket; the result equals the K = 1 loop on the batch whose pockets are repeated K times."""
    hist, final = p_sample_loop_tensors(model, ligand_mask, ligand_angle_noise, receptor_seq, receptor_mask, receptor_angle, total_timesteps,
                                        betas, noise_steps=noise_steps, graph_id0=graph_id0, seed=seed, keep_history=keep_history,
                                        packed=packed, num_samples=num_samples)
    return (hist if keep_history else final[None]).cpu()


def qsample_coefficients(betas: torch.Tensor) -> torch.Tensor:
    """[T,2] fp32 table of the training q-sample, indexed by step: (sqrt(alphabar), sqrt(1 - alphabar)) of compute_alphas(betas)"""
    ab = compute_alphas(betas.detach().float().cpu())
    return torch.stack([ab["sqrt_alphas_cumprod"], ab["sqrt_one_minus_alphas_cumprod"]], dim=1).contiguous()


@torch.no_grad()
def score_backbones_tensors(model, ligand_mask, backbones, receptor_seq, receptor_mask, receptor_angle, total_timesteps: int, betas, *,
                            noise_steps: Optional[torch.Tensor] = None, graph_id0: Optional[int] = None, seed: Optional[int] = None,
                            packed: bool = False, num_samples: int = 1) -> torch.Tensor:
    """The structure model's training objective for given backbones in their pockets, at every timestep (seqdiff_struct_score_multi):
    for k = T-1 .. 0, x_k = wrap(sqrt(alphabar_k) x0 + sqrt(1 - alphabar_k) eps_k) (the training q-sample), pred = the denoiser at
    timestep k, terms += h(wrap(eps_k - pred)) with FoldingDiff's smooth-L1 h (beta = pi/10), from one captured CUDA graph per step.
    Arguments in p_sample_loop's order; `backbones` [P*K, L, F] are the scored angles x0, `ligand_mask` [P*K, L] or [P, L] (repeated),
    the receptor tensors hold the P pockets, `betas` [T] is the schedule compute_alphas() turns into the q-sample's coefficients.
    Returns terms [P*K, L, F] fp64 on the model's device: per position and feature, the sum over the T steps, 0 at masked positions
    (score_backbones forms the per-backbone loss).  `noise_steps` [T, P*K, L, F]: explicit eps, entry k at step k; else Philox keyed as
    the sampler's noise, graph_id0 = None continuing the process-wide stream.  `packed` / `num_samples` as in p_sample_loop: packed terms
    equal the padded ones at the valid positions.  ValueError (before any device work) for disagreeing shapes, betas not of length T,
    a complex without a valid ligand position, non-finite backbones (padded rows reach the valid ones through 0 * NaN in attention) or
    a bad num_samples."""
    K = check_num_samples(num_samples)
    T = int(total_timesteps)
    if T < 1:
        raise ValueError(f"total_timesteps must be >= 1, got {total_timesteps}")
    Fs = model.feature_size
    if receptor_seq.dim() != 3 or receptor_seq.shape[2] != 20:
        raise ValueError(f"receptor_seq must be [P, L_rec, 20], got {tuple(receptor_seq.shape)}")
    P, Lr = receptor_seq.shape[0], receptor_seq.shape[1]
    B = P * K
    if backbones.dim() != 3 or tuple(backbones.shape[::2]) != (B, Fs):
        raise ValueError(f"backbones must be [P*K, L, F] = [{B}, L, {Fs}], got {tuple(backbones.shape)}")
    Ll = backbones.shape[1]
    if K > 1 and tuple(ligand_mask.shape) == (P, Ll):
        ligand_mask = ligand_mask.repeat_interleave(K, dim=0)
    for x, name, shape in ((ligand_mask, "ligand_mask", (B, Ll)), (receptor_mask, "receptor_mask", (P, Lr)),
                           (receptor_angle, "receptor_angle", (P, Lr, Fs))):
        if tuple(x.shape) != shape:
            raise ValueError(f"{name} must be {shape}, got {tuple(x.shape)}")
    betas = torch.as_tensor(betas)
    if betas.dim() != 1 or betas.shape[0] != T:
        raise ValueError(f"betas must hold one value per timestep ({T}), got shape {tuple(betas.shape)}")
    if noise_steps is not None and tuple(noise_steps.shape) != (T, B, Ll, Fs):
        raise ValueError(f"noise_steps must be [T, P*K, L, F] = {(T, B, Ll, Fs)}, got {tuple(noise_steps.shape)}")
    if not bool((ligand_mask != 0).any(dim=1).all()):
        raise ValueError("every backbone needs at least one valid ligand position to be scored")
    if not bool(torch.isfinite(backbones).all()):
        raise ValueError("backbones must be finite everywhere, padded positions included")
    qs = qsample_coefficients(betas)

    h = model._sync_handle()
    dev = model._handle_dev
    if graph_id0 is None:
        graph_id0 = _cabi.GRAPH_IDS.take(B)

    def dv(x):
        return x.to(device=dev, dtype=torch.float32).contiguous()

    terms = torch.empty((B, Ll, Fs), device=dev, dtype=torch.float64)
    args = [dv(qs), dv(backbones), dv(ligand_mask), dv(receptor_seq), dv(receptor_angle), dv(receptor_mask)]
    z = None if noise_steps is None else dv(noise_steps)
    with torch.cuda.device(dev):
        stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        _cabi.check(_cabi.lib().seqdiff_struct_score_multi(h, model._precision_code(), P, K, Ll, Lr, T, *map(_cabi.ptr, args), _cabi.ptr(z),
                                                           SEED if seed is None else seed, graph_id0, 1 if packed else 0, _cabi.ptr(terms),
                                                           stream))
    return terms


def backbone_loss(terms: torch.Tensor, ligand_mask: torch.Tensor, total_timesteps: int):
    """(loss [B], per_feature [B, F]) fp64 on the host from score_backbones_tensors' terms: per_feature[b, f] = sum_l terms[b, l, f] /
    (T * n_b) over the n_b valid positions, loss = mean_f per_feature -- the training objective averaged over the T timesteps"""
    t = terms.detach().cpu()
    n = (ligand_mask.detach().cpu() != 0).sum(dim=1).double()
    if n.shape[0] != t.shape[0]:
        n = n.repeat_interleave(t.shape[0] // n.shape[0])
    per_feature = t.sum(dim=1) / (int(total_timesteps) * n[:, None])
    return per_feature.mean(dim=-1), per_feature


@torch.no_grad()
def score_backbones(model, ligand_mask, backbones, receptor_seq, receptor_mask, receptor_angle, total_timesteps: int, betas, **kw):
    """score_backbones_tensors on the host: (loss [P*K], per_feature [P*K, F]) fp64, one entry per backbone in (pocket, backbone) order.
    loss is the structure model's training objective for the backbone in its pocket, averaged over the T timesteps (one noise draw per
    step): lower = more native-like to the model.  It is a ranking score, not a likelihood."""
    terms = score_backbones_tensors(model, ligand_mask, backbones, receptor_seq, receptor_mask, receptor_angle, total_timesteps, betas, **kw)
    return backbone_loss(terms, ligand_mask, total_timesteps)


def sample(model, test_angle_ds, first_batch_only: bool = True, loop_fn=None, num_samples: int = 1, **kw):
    """reference structure_model/sample.py:191-229: chunk the dataset's features into batches of CONFIG["batch_size"], draw the start
    noise with the dataset's own `sample_noise`, run `p_sample_loop`, and trim every complex to its ligand length -> a list of numpy
    arrays [timesteps, len_i, n_ft].  `test_angle_ds` is duck-typed like the reference's NoisedAnglesDataset (`__len__`,
    `__getitem__` -> dict of tensors, `sample_noise`, `timesteps`, `alpha_beta_terms["betas"]`).  The reference stops after the
    first batch (the `break` at sample.py:228); `first_batch_only=False` samples the whole dataset.  Further keywords go to the loop
    function, e.g. `packed=True` (ragged packing, see `p_sample_loop`): the trimmed arrays are the same, bit for bit.
    `num_samples=K > 1`: K backbones per complex (see `p_sample_loop`), the start noise drawn for all P*K of a batch at once; the list
    then holds the arrays in (complex, sample) order."""
    K = check_num_samples(num_samples)
    if K > 1:
        kw["num_samples"] = K
    fn = p_sample_loop if loop_fn is None else loop_fn
    bs = CONFIG["batch_size"]

    def chunkify_features(feature_name):
        feats = [test_angle_ds[i][feature_name] for i in range(len(test_angle_ds))]
        return [torch.stack(feats[i:i + bs]) for i in range(0, len(test_angle_ds), bs)]

    ligand_mask = chunkify_features("ligand_attn_mask")
    receptor_angle = chunkify_features("receptor_angles")
    receptor_seq = chunkify_features("receptor_seq")
    receptor_mask = chunkify_features("receptor_attn_mask")
    pad, feature_size = test_angle_ds[0]["ligand_angles"].shape
    ligand_len = [m.sum(dim=1).int() for m in ligand_mask]
    retval = []
    for idx, this_lengths in enumerate(ligand_len):
        print(f"Generating Batch {idx}/{len(ligand_len)}")
        batch = len(this_lengths)
        noise = test_angle_ds.sample_noise(torch.zeros((batch * K, pad, feature_size), dtype=torch.float32))
        sampled = fn(model=model, ligand_mask=ligand_mask[idx], ligand_angle_noise=noise, receptor_seq=receptor_seq[idx],
                     receptor_mask=receptor_mask[idx], receptor_angle=receptor_angle[idx], total_timesteps=test_angle_ds.timesteps,
                     betas=test_angle_ds.alpha_beta_terms["betas"], disable_pbar=False, **kw)
        retval.extend(sampled[:, i, :int(this_lengths[i // K]), :].numpy() for i in range(batch * K))
        if first_batch_only:
            break
    return retval
