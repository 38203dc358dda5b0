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
                    _Container, _BertLayer, BertAttention, _Intermediate, _SelfOutput)

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


ConditionalBertForDiffusion = ConditionalBertForDiffusionBase  # the Lightning wrapper (model.py:232-403) adds training only


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
