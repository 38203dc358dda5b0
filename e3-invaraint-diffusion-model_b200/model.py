"""Drop-in for `sequence_model/model.py` of the reference: same class names, constructor and forward
signatures, same state_dict keys and shapes (SURVEY.md Appendix B) -- but `forward` runs the
hand-written sm_100a kernels of libseqdiff_b200.so through the C ABI (include/seqdiff_b200.h).

The nn.Module tree below is a PARAMETER CONTAINER: it exists so `load_state_dict(torch.load(path))`
(reference sample.py:106), `.to(device)`, `.parameters()` and checkpoints keep working.  None of its
sub-module forwards are on the product path; there is no PyTorch / CPU fallback -- without the CUDA
library or a CUDA device `forward` raises.
"""
from __future__ import annotations

import ctypes
from dataclasses import dataclass
from typing import List, Optional

import torch
from torch import nn
from torch.nn import functional as F

from . import _cabi
from .utils import BlosumTransition, DiscreteUniformTransition, PredefinedNoiseScheduleDiscrete, step_tables

AA_VOCAB = "ACDEFGHIKLMNPQRSTVWY"


@dataclass
class BertConfig:
    """The subset of transformers.BertConfig the path consumes (reference sample.py:69-92).  A real
    transformers.BertConfig is accepted everywhere one of these is (duck-typed)."""

    max_position_embeddings: int = 512
    num_attention_heads: int = 12
    hidden_size: int = 768
    intermediate_size: int = 3072
    num_hidden_layers: int = 12
    position_embedding_type: str = "absolute"
    hidden_dropout_prob: float = 0.1
    attention_probs_dropout_prob: float = 0.1
    layer_norm_eps: float = 1e-12
    hidden_act: str = "gelu"
    use_cache: bool = True
    is_decoder: bool = False
    add_cross_attention: bool = False


# ------------------------------------------------------------------------------------------------
# parameter containers (names = reference attribute names => identical state_dict keys)
# ------------------------------------------------------------------------------------------------
class _Container(nn.Module):
    def forward(self, *a, **k):  # pragma: no cover
        raise RuntimeError("parameter container: the computation runs inside ConditionalBertForDiffusionBase.forward "
                           "(CUDA, libseqdiff_b200.so)")


class _SelfAttention(_Container):  # HF BertSelfAttention, transformers 4.38.2 layout
    def __init__(self, cfg, relative: bool):
        super().__init__()
        H = cfg.hidden_size
        self.query, self.key, self.value = nn.Linear(H, H), nn.Linear(H, H), nn.Linear(H, H)
        if relative:
            self.distance_embedding = nn.Embedding(2 * cfg.max_position_embeddings - 1, H // cfg.num_attention_heads)


class _SelfOutput(_Container):  # HF BertSelfOutput / BertOutput
    def __init__(self, cfg, fan_in=None):
        super().__init__()
        self.dense = nn.Linear(fan_in or cfg.hidden_size, cfg.hidden_size)
        self.LayerNorm = nn.LayerNorm(cfg.hidden_size, eps=cfg.layer_norm_eps)


class _Intermediate(_Container):
    def __init__(self, cfg):
        super().__init__()
        self.dense = nn.Linear(cfg.hidden_size, cfg.intermediate_size)


class BertAttention(_Container):
    def __init__(self, cfg, relative: bool):
        super().__init__()
        self.self = _SelfAttention(cfg, relative)
        self.output = _SelfOutput(cfg)


class _BertLayer(_Container):
    def __init__(self, cfg, relative: bool):
        super().__init__()
        self.attention = BertAttention(cfg, relative)
        self.crossattention = BertAttention(cfg, False)  # 4.38.2: position_embedding_type="absolute"
        self.intermediate = _Intermediate(cfg)
        self.output = _SelfOutput(cfg, cfg.intermediate_size)


class BertEncoder(_Container):
    def __init__(self, cfg, relative: bool):
        super().__init__()
        self.layer = nn.ModuleList([_BertLayer(cfg, relative) for _ in range(cfg.num_hidden_layers)])


class SELayer(_Container):
    """reference model.py:26-66."""

    def __init__(self, bert_config, mlp_ratio=4.0, **block_kwargs):
        super().__init__()
        H = bert_config.hidden_size
        relative = getattr(bert_config, "position_embedding_type", "absolute") == "relative_key"
        self.adaLN_modulation = nn.Sequential(nn.Linear(H, H, bias=True), nn.SiLU(), nn.Linear(H, 6 * H, bias=True))
        self.attn = BertAttention(bert_config, relative)
        self.mlp = nn.Sequential(nn.Linear(H, int(H * mlp_ratio)), nn.GELU(), nn.Dropout(bert_config.hidden_dropout_prob),
                                 nn.Linear(int(H * mlp_ratio), H), nn.Dropout(bert_config.hidden_dropout_prob))
        nn.init.zeros_(self.adaLN_modulation[0].weight)
        nn.init.zeros_(self.adaLN_modulation[0].bias)


class GaussianFourierProjection(_Container):
    """reference model.py:68-97 (buffer only; sin/cos features are computed in the CUDA forward)."""

    def __init__(self, embed_dim: int = 384, scale: float = 2 * torch.pi):
        super().__init__()
        w = torch.randn(embed_dim // 2) * scale
        self.register_buffer("W", w)


class BertEmbeddings(_Container):
    """reference model.py:99-117."""

    def __init__(self, in_features, bert_config):
        super().__init__()
        self.linear = nn.Linear(in_features, bert_config.hidden_size)
        self.LayerNorm = nn.LayerNorm(bert_config.hidden_size, eps=bert_config.layer_norm_eps)


class AminoAcidPredictor(_Container):
    """reference model.py:119-153."""

    def __init__(self, d_model: int, d_out: int = 4, activation="gelu", eps: float = 1e-12) -> None:
        super().__init__()
        if activation != "gelu":
            raise ValueError("only the reference's default 'gelu' head is implemented in CUDA")
        self.d_model, self.d_out = d_model, d_out
        self.dense1 = nn.Linear(d_model, d_model)
        self.layer_norm = nn.LayerNorm(d_model, eps=eps)
        self.dense2 = nn.Linear(d_model, d_out)


# ------------------------------------------------------------------------------------------------
class ConditionalBertForDiffusionBase(nn.Module):
    """reference model.py:156-253.  `precision` selects the operand format of the GEMM / attention kernels
    (accumulators, residual stream, LayerNorm, softmax and logits are fp32 in every mode):
      "bf16"       bf16 activations x bf16 weights on tcgen05 (the configuration BASELINE.json names)
      "fp16"       fp16 activations x fp16 weights, same kernels and speed, 8x finer operand rounding
      "fp32"       fp32 SIMT kernels -- the 1e-5 parity mode."""

    _create_symbol = "seqdiff_model_create"  # C entry point that builds the handle for this module tree
    _host_only_prefixes = ("discrete_noise_schedule.", "aa_transition_model.")

    def __init__(self, encoder_config, decoder_config, feature_size: int) -> None:
        super().__init__()
        self.encoder_config = encoder_config
        self.decoder_config = decoder_config
        self.feature_size = feature_size
        self.precision = "bf16"
        relative = getattr(decoder_config, "position_embedding_type", "absolute") == "relative_key"
        self.timestep_projector = GaussianFourierProjection(decoder_config.hidden_size)
        self.ligand_seq_embedding = BertEmbeddings(20, encoder_config)
        self.ligand_angle_embedding = BertEmbeddings(8, encoder_config)
        self.ligand_feature_emb = SELayer(encoder_config)
        self.receptor_seq_embedding = BertEmbeddings(20, encoder_config)
        self.receptor_angle_embedding = BertEmbeddings(8, encoder_config)
        self.receptor_feature_emb = SELayer(encoder_config)  # dead weight in the reference too (model.py:221)
        self.decoder = BertEncoder(decoder_config, relative)
        self.decoder_normalize = SELayer(decoder_config)
        self.amino_acid_predictor = AminoAcidPredictor(decoder_config.hidden_size, feature_size)
        self.initialize_weights()
        self._handle = None
        self._handle_sig = None
        self._handle_dev = None
        self._handle_tensors = None

    def _apply(self, fn, recurse=True):
        self._handle_tensors = None  # .to() / .float() / .cuda() may re-seat the tensors
        return super()._apply(fn, recurse)

    def load_state_dict(self, *a, **kw):
        self._handle_tensors = None
        return super().load_state_dict(*a, **kw)

    def initialize_weights(self):
        """reference model.py:183-198."""

        def _basic_init(module):
            if isinstance(module, nn.Linear):
                torch.nn.init.xavier_uniform_(module.weight)
                if module.bias is not None:
                    nn.init.constant_(module.bias, 0)

        self.apply(_basic_init)
        nn.init.constant_(self.decoder_normalize.adaLN_modulation[0].weight, 0)
        nn.init.constant_(self.decoder_normalize.adaLN_modulation[0].bias, 0)

    # ---- C handle management --------------------------------------------------------------------
    def _config_struct(self):
        d = self.decoder_config
        return _cabi.SeqdiffConfig(
            hidden_size=d.hidden_size, num_attention_heads=d.num_attention_heads, intermediate_size=d.intermediate_size,
            num_hidden_layers=d.num_hidden_layers, max_position_embeddings=d.max_position_embeddings,
            feature_size=self.feature_size,
            relative_key=int(getattr(d, "position_embedding_type", "absolute") == "relative_key"),
            layer_norm_eps=float(getattr(d, "layer_norm_eps", 1e-12)))

    def _precision_code(self):
        if self.precision not in _cabi.PRECISIONS:
            raise ValueError(f"precision must be one of {sorted(_cabi.PRECISIONS)}, got {self.precision!r}")
        return _cabi.PRECISIONS[self.precision]

    def _sync_handle(self):
        """(Re)uploads the weights into the C handle when any tensor of the state_dict changed."""
        lib = _cabi.lib()
        # the denoiser's own tensors only: PeptideDiff also registers the noise schedule's `betas` buffer (reference
        # utils.py:216), which is host-side table data, not a weight of the forward.  The (name, tensor) list is cached -- walking
        # state_dict() costs ~0.5 ms per call, a B = 1 forward ~1 ms -- and dropped whenever the module tree is converted (_apply).
        if self._handle_tensors is None:
            self._handle_tensors = [(k, v) for k, v in self.state_dict().items() if not k.startswith(self._host_only_prefixes)]
        sd = dict(self._handle_tensors)
        dev = self._handle_tensors[0][1].device
        if dev.type != "cuda":
            raise RuntimeError("the sequence denoiser runs only on a CUDA device (no CPU fallback): call model.to('cuda')")
        sig = tuple((t.data_ptr(), t._version) for _, t in self._handle_tensors)
        if self._handle is not None and sig == self._handle_sig and dev == self._handle_dev:
            return self._handle
        stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        with torch.cuda.device(dev):
            if self._handle is None or dev != self._handle_dev:
                self.release()
                h = ctypes.c_void_p()
                cfg = self._config_struct()
                _cabi.check(getattr(lib, self._create_symbol)(ctypes.byref(cfg), dev.index or 0, ctypes.byref(h)))
                self._handle, self._handle_dev = h, dev
            keep = []
            for name, t in sd.items():
                t32 = t.detach()
                if t32.dtype != torch.float32 or not t32.is_contiguous():
                    t32 = t32.float().contiguous()
                    keep.append(t32)
                _cabi.check(lib.seqdiff_model_set_tensor(self._handle, name.encode(), _cabi.ptr(t32), t32.numel(), stream))
            _cabi.check(lib.seqdiff_model_finalize(self._handle, stream))
            torch.cuda.current_stream(dev).synchronize()
        self._handle_sig = sig
        return self._handle

    def release(self):
        if getattr(self, "_handle", None) is not None:
            _cabi.lib().seqdiff_model_destroy(self._handle)
            self._handle = None
            self._handle_sig = None

    def __del__(self):
        try:
            self.release()
        except Exception:
            pass

    # ---- forward --------------------------------------------------------------------------------
    def forward(self, timestep, noised_ligand_seq, ligand_angle, ligand_attention_masks, receptor_seq, receptor_angle,
                receptor_attention_masks, ligand_pos_ids=None, receptor_pos_ids=None):
        """reference model.py:200-237.  pos ids are accepted and ignored, as in the reference."""
        if self.training and (self.decoder_config.hidden_dropout_prob > 0 or self.decoder_config.attention_probs_dropout_prob > 0):
            raise RuntimeError("forward() is the eval-mode (dropout-free) inference path: call model.eval(), or use training_step() "
                               "for the training-mode forward + backward")
        h = self._sync_handle()
        dev = self._handle_dev
        B, Ll = noised_ligand_seq.shape[0], noised_ligand_seq.shape[1]
        Lr = receptor_seq.shape[1]

        def prep(x, shape):
            x = x.to(device=dev, dtype=torch.float32).contiguous()
            if tuple(x.shape) != shape:
                raise ValueError(f"expected shape {shape}, got {tuple(x.shape)}")
            return x

        t = timestep.to(device=dev, dtype=torch.float32).reshape(-1).contiguous()
        if t.numel() != B:
            raise ValueError("timestep must hold one value per batch row")
        x = prep(noised_ligand_seq, (B, Ll, 20))
        la = prep(ligand_angle, (B, Ll, 8))
        lm = prep(ligand_attention_masks, (B, Ll))
        rs = prep(receptor_seq, (B, Lr, 20))
        ra = prep(receptor_angle, (B, Lr, 8))
        rm = prep(receptor_attention_masks, (B, Lr))
        out = torch.empty((B, Ll, self.feature_size), device=dev, dtype=torch.float32)
        with torch.cuda.device(dev):
            stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            _cabi.check(_cabi.lib().seqdiff_forward(h, self._precision_code(), B, Ll, Lr, _cabi.ptr(t), _cabi.ptr(x), _cabi.ptr(la),
                                                    _cabi.ptr(lm), _cabi.ptr(rs), _cabi.ptr(ra), _cabi.ptr(rm), _cabi.ptr(out), stream))
        return out

    def _create_pos_ids(self, sequences: torch.Tensor):
        batch_size, seq_length, *_ = sequences.size()
        return torch.arange(seq_length).expand(batch_size, -1)

    def _exetend_attention_mask(self, mask):
        extended = mask[:, None, None, :].type_as(mask)
        return (1.0 - extended) * -10000.0


def loss_terms(logits, x0, x_t, ligand_mask):
    """The ten fp64 reduction terms of get_loss / elbo_loss (include/seqdiff_b200.h: seqdiff_loss_terms) as a device tensor."""
    dev = logits.device
    if dev.type != "cuda":
        raise RuntimeError("loss_terms runs only on a CUDA device (no CPU fallback)")

    def prep(t, last):
        return t.to(device=dev, dtype=torch.float32).reshape(-1, last).contiguous() if last else t.to(device=dev, dtype=torch.float32).reshape(-1).contiguous()

    lg, a, b, m = prep(logits, 20), prep(x0, 20), prep(x_t, 20), prep(ligand_mask, 0)
    if not (lg.shape[0] == a.shape[0] == b.shape[0] == m.shape[0]):
        raise ValueError("logits, x0, x_t and ligand_mask must cover the same rows")
    out = torch.empty(10, device=dev, dtype=torch.float64)
    with torch.cuda.device(dev):
        stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        _cabi.check(_cabi.lib().seqdiff_loss_terms(lg.shape[0], _cabi.ptr(lg), _cabi.ptr(a), _cabi.ptr(b), _cabi.ptr(m), _cabi.ptr(out), stream))
    return out


class _FlatTraining:
    """The optimizer side shared by the trainable models (PeptideDiff, structure_model.ConditionalBertForDiffusion): the handle's flat
    parameter space, the fused clip + AdamW step and the copy of the trained masters back into the module."""

    def _flat_params(self):
        from . import train as _train
        if getattr(self, "_flat", None) is None or self._flat.handle is not self._handle:
            self._sync_handle()
            self._flat = _train.FlatParams(self)
        return self._flat

    def configure_optimizers(self, group=None, grad_comm: str = "fp32"):
        """reference model.py:416-450: AdamW(lr, weight_decay=l2_lambda) over all parameters -- here the fused clip + AdamW kernel
        over the handle's flat parameter space, with the data-parallel gradient all-reduce in front of it.  The LinearWarmup
        schedule (stepped per epoch, as Lightning does with interval="epoch") is applied by train.fit()."""
        from . import train as _train
        if self.lr_scheduler not in (None, "OneCycleLR", "LinearWarmup"):
            raise ValueError(f"Unknown lr scheduler {self.lr_scheduler}")
        if getattr(self, "_optimizer", None) is None or self._optimizer.flat is not self._flat_params():
            self._optimizer = _train.FlatAdamW(self._flat_params(), lr=self.lr, weight_decay=self.l2_lambda,
                                               gradient_clip=getattr(self, "gradient_clip", 1.0), group=group, grad_comm=grad_comm)
        return {"optimizer": self._optimizer}

    def pull_weights(self):
        """copies the trained masters from the C handle back into this module's parameters (state_dict / checkpoints)."""
        from . import train as _train
        _train.pull_weights(self)

    def state_dict(self, *a, **kw):
        if getattr(self, "_weights_dirty", False):
            self.pull_weights()
        return super().state_dict(*a, **kw)


class PeptideDiff(_FlatTraining, ConditionalBertForDiffusionBase):
    """reference model.py:256-450 without the Lightning base class (Trainer is out of scope, SURVEY.md
    section 2).  Inference-side members match the reference; `apply_aa_noise` runs the CUDA q-sample
    kernel; `get_loss` evaluates the reference's loss terms with the CUDA forward and the CUDA reduction
    kernel; `training_step` runs forward + loss + the full hand-written backward (csrc/train.cu) and
    `configure_optimizers` returns the fused clip + AdamW step (train.py)."""

    def __init__(self, encoder_config, decoder_config, feature_names: List[str], loss_func, noise_schedule, timesteps,
                 max_epochs: int = 1, lr_scheduler=None, l2_lambda: float = 0.0, steps_per_epoch: int = 250,
                 learning_rate: float = 5e-5, **kwargs):
        ConditionalBertForDiffusionBase.__init__(self, encoder_config, decoder_config, len(feature_names))
        self.noise_schedule = noise_schedule
        self.timesteps = timesteps
        self.aa_transition_model = BlosumTransition(x_classes=20)
        self.discrete_noise_schedule = PredefinedNoiseScheduleDiscrete(noise_schedule=self.noise_schedule, timesteps=self.timesteps)
        self.loss_function = loss_func
        self.lr = learning_rate
        self.l2_lambda = l2_lambda
        self.lr_scheduler = lr_scheduler
        self.max_epochs = max_epochs
        self.steps_per_epoch = steps_per_epoch
        self.valid_epoch_losses = []
        self.train_epoch_losses = []
        self._noise_seed = 0
        self._noise_calls = 0

    def apply_aa_noise(self, ligand_seq, t_int, noise_E: Optional[torch.Tensor] = None):
        """reference model.py:291-311.  Qbar_t comes from the host tables exactly as in the reference;
        the per-residue categorical draw runs on the GPU (explicit Exp(1) `noise_E` [B*L,20] for parity
        runs, counter-based Philox otherwise)."""
        B, L, _ = ligand_seq.shape
        dev = ligand_seq.device
        if dev.type != "cuda":
            raise RuntimeError("apply_aa_noise runs only on a CUDA device (no CPU fallback)")
        # Qbar_t of EVERY integer step 0..T, built once on the host with the per-step arithmetic of the reference (t_int / T in
        # fp32 -> alpha_bar -> BLOSUM row softmax: elementwise in t, so row k of the table == what the reference computes for
        # t_int == k) and kept on the device; the per-graph gather runs there, so a training step never waits on the host.
        key = (self.timesteps, dev)
        if getattr(self, "_qtb_all_key", None) != key:
            t_all = torch.arange(self.timesteps + 1, dtype=torch.float32).unsqueeze(1) / self.timesteps
            a_all = self.discrete_noise_schedule.get_alpha_bar(t_normalized=t_all)
            self._qtb_all = self.aa_transition_model.get_Qt_bar(a_all, device=torch.device("cpu")).float().contiguous().to(dev)
            self._qtb_all_key = key
        Qtb = self._qtb_all[t_int.to(dev).reshape(-1).long()].contiguous()
        x0 = ligand_seq.to(torch.float32).contiguous()
        out = torch.empty_like(x0)
        E = None if noise_E is None else noise_E.to(device=dev, dtype=torch.float32).contiguous()
        self._noise_calls += 1
        with torch.cuda.device(dev):
            stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
            _cabi.check(_cabi.lib().seqdiff_apply_aa_noise(_cabi.ptr(Qtb), B, L, _cabi.ptr(x0), _cabi.ptr(E), self._noise_seed, 0,
                                                           self._noise_calls, _cabi.ptr(out), None, stream))
        return out

    @torch.no_grad()
    def get_loss(self, batch, t_norm, noised_ligand_seq):
        """reference model.py:313-345 (evaluation only: no autograd graph).  The forward and ALL reductions run in CUDA
        (`seqdiff_loss_terms`: masked counts, the two cross-entropy sums, the entropy and KL sums of `elbo_loss`); the host
        only forms the ratios.  `loss_func` must be the reference's `torch.nn.CrossEntropyLoss()` (train_model.py)."""
        if not isinstance(self.loss_function, nn.CrossEntropyLoss) or self.loss_function.reduction != "mean" or \
                self.loss_function.label_smoothing != 0.0 or self.loss_function.weight is not None:
            raise ValueError("the CUDA loss reduction implements the reference's plain mean CrossEntropyLoss")
        pred_aa = self.forward(t_norm, noised_ligand_seq, batch["ligand_angles"], batch["ligand_attn_mask"], batch["receptor_seq"],
                               batch["receptor_angles"], batch["receptor_attn_mask"])
        terms = loss_terms(pred_aa, batch["ligand_seq"], noised_ligand_seq, batch["ligand_attn_mask"])
        n_mask, n_noised, n_sel, n_same, n_rec, ce_noised, ce_sel, ent, kl = (terms[i] for i in range(9))
        aa_noise_rate = (n_same / n_mask).float()
        aa_recovery_rate = (n_rec / n_mask).float()
        aa_noised_loss = (ce_noised / n_noised).float()     # CrossEntropyLoss(mean) over the noised rows (nan if there are none)
        aa_all_loss = (ce_sel / n_sel).float()
        elbo = (-ent / n_noised + kl / n_noised).float()    # elbo_loss: nll + kl_div(batchmean)
        total_loss = aa_noised_loss + elbo
        return total_loss, elbo, aa_noised_loss, aa_all_loss, aa_recovery_rate, aa_noise_rate

    def validation_step(self, batch, batch_idx):
        """reference model.py:381-404."""
        t_int = torch.randint(0, self.timesteps + 1, size=(batch["ligand_seq"].shape[0], 1), device=batch["ligand_seq"].device).float()
        t_norm = t_int / self.timesteps
        aa = self.apply_aa_noise(batch["ligand_seq"], t_int)
        loss, *_ = self.get_loss(batch, t_norm, aa)
        return torch.mean(loss)

    # ---- training (BASELINE configs[3]) ----------------------------------------------------------
    def training_step(self, batch, batch_idx, t_int=None, noise_E=None):
        """reference model.py:347-367.  Draws t (torch.randint, as the reference), q-samples x_t on the GPU, then runs forward
        (dropout active in train() mode) + get_loss + the FULL backward in one C call: the gradients of the 61.06 M live
        parameters land in the flat buffer `self._flat.grads` (what `loss.backward()` leaves in the .grad fields), ready for
        `configure_optimizers()["optimizer"].step()`.  Returns the loss (device scalar); the logged quantities of the reference's
        `log_dict` are kept in `self.last_log`.  Extra keywords (parity runs): `t_int` [B,1], `noise_E` [B*L,20]."""
        from . import train as _train
        x0 = batch["ligand_seq"]
        dev = self._handle_dev if self._handle_dev is not None else next(self.parameters()).device
        if t_int is None:
            t_int = torch.randint(0, self.timesteps + 1, size=(x0.shape[0], 1), device=dev).float()
        t_norm = t_int / self.timesteps
        aa = self.apply_aa_noise(x0.to(dev), t_int, noise_E=noise_E)
        flat = self._flat_params()
        self._train_steps = getattr(self, "_train_steps", 0) + 1
        opt = getattr(self, "_optimizer", None)
        if opt is not None and opt.flat is flat:
            opt.arm_overlap()
        terms, _ = _train.train_step_tensors(self, flat, batch, t_norm, aa, seed=self._noise_seed, step=self._train_steps)
        if opt is not None and opt.flat is flat:
            opt.launch_overlapped_all_reduce()  # bucket k's all-reduce starts when the backward pass has finished bucket k
        loss, elbo, aa_noised_loss, aa_all_loss, aa_recovery_rate, aa_noise_rate = _train.loss_from_terms(terms)
        self.last_log = {"aa_noise_rate": aa_noise_rate, "aa_recovery_rate": aa_recovery_rate, "avg_timestep": t_int.mean().int(),
                         "train_loss": loss, "train_aa_noised_loss": aa_noised_loss, "train_aa_all_loss": aa_all_loss, "train_elbo_loss": elbo}
        return loss
