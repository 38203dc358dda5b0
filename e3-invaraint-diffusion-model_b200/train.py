"""Training side of the drop-in (BASELINE configs[3]: "sequence_model training step batch 128 graphs with NCCL gradient
allreduce on 8xB200"): what the reference gets from Lightning + autograd + torch.optim.AdamW, here as two C calls per step

    seqdiff_train_step   forward (dropout) + loss + full backward  -> ONE flat fp32 gradient buffer        (csrc/train.cu)
    [all-reduce of that buffer over the data-parallel group: torch.distributed / NCCL over NVLink -- the only collective]
    seqdiff_adamw_step   1/world scaling + clip_grad_norm_(gradient_clip) + AdamW on the fp32 masters      (csrc/train_kernels.cu)

reference: sequence_model/model.py:347-367 (training_step), :313-345 (get_loss), :416-450 (configure_optimizers),
train_model.py:30-33 (lr 5e-5, l2_norm 0.1, gradient_clip 1.0, LinearWarmup), :95 (gradient_clip_val).

Data parallelism.  Every rank holds the full model (61.06 M live parameters), runs its block of the global batch and the ranks
sum their gradients over the flat buffer (244 MB fp32, or 122 MB with `grad_comm="bf16"`).  The flat index space follows the forward
order of the network, so the backward pass finishes it from the end: the library records one CUDA event per gradient bucket
(seqdiff_train_set_bucket_events) and the all-reduce of bucket k runs on a communication stream as soon as event k has fired -- under
the rest of the backward pass; only the last bucket (embeddings + ligand_feature_emb, 18 % of the bytes) is exposed.  The update
needs the GLOBAL gradient norm (clip), so it starts only after the last bucket has arrived.  Lightning DDP semantics: per-rank mean
loss, gradients averaged over ranks.
"""
from __future__ import annotations

import ctypes
from typing import Dict, Optional

import torch

from . import _cabi


class FlatParams:
    """The handle's flat parameter index space: name -> (offset, numel), plus the torch-owned flat buffers (gradient, AdamW
    moments).  torch only provides device memory here; every kernel touching these buffers is the library's."""

    def __init__(self, model):
        self.model = model
        self.handle = model._sync_handle()
        self.device = model._handle_dev
        lib = _cabi.lib()
        self.total = int(lib.seqdiff_train_param_count(self.handle))
        if self.total <= 0:
            raise _cabi.SeqdiffError("seqdiff_train_param_count failed: " + (lib.seqdiff_last_error() or b"").decode())
        n = lib.seqdiff_train_param_table(self.handle, None, 0, None, None, 0)
        stride = 128
        names = ctypes.create_string_buffer(n * stride)
        offs = (ctypes.c_int64 * n)()
        nums = (ctypes.c_int64 * n)()
        if lib.seqdiff_train_param_table(self.handle, names, stride, offs, nums, n) != n:
            raise _cabi.SeqdiffError("seqdiff_train_param_table failed")
        self.table: Dict[str, tuple] = {}
        for i in range(n):
            self.table[names.raw[i * stride:(i + 1) * stride].split(b"\0")[0].decode()] = (int(offs[i]), int(nums[i]))
        self.grads = torch.zeros(self.total, device=self.device, dtype=torch.float32)
        self.live_numel = sum(v[1] for v in self.table.values())
        nb = int(lib.seqdiff_train_grad_buckets(self.handle, None, 0))
        bounds = (ctypes.c_int64 * (nb + 1))()
        if nb <= 0 or lib.seqdiff_train_grad_buckets(self.handle, bounds, nb + 1) != nb:
            raise _cabi.SeqdiffError("seqdiff_train_grad_buckets failed")
        self.bucket_bounds = [int(b) for b in bounds]   # bucket k = grads[bounds[k]:bounds[k+1]]; the backward finishes k = nb-1 first

    def grad(self, name: str, shape=None) -> torch.Tensor:
        off, n = self.table[name]
        g = self.grads[off:off + n]
        return g if shape is None else g.view(shape)

    def named_grads(self, model=None) -> Dict[str, Optional[torch.Tensor]]:
        """{state_dict key: gradient with the parameter's shape}; tensors without a gradient (the dead receptor_feature_emb block,
        quirk Q1 -- torch leaves their .grad None as well) map to None."""
        m = self.model if model is None else model
        out = {}
        for k, p in m.named_parameters():
            out[k] = self.grad(k, tuple(p.shape)) if k in self.table else None
        return out


class FlatAdamW:
    """torch.optim.AdamW semantics (decoupled weight decay, bias correction, eps outside the sqrt) on the handle's masters, preceded by
    the data-parallel gradient average and torch.nn.utils.clip_grad_norm_(max_norm=gradient_clip).  One fused kernel pass."""

    def __init__(self, flat: FlatParams, lr=5e-5, weight_decay=0.1, betas=(0.9, 0.999), eps=1e-8, gradient_clip=1.0, group=None,
                 grad_comm: str = "fp32", overlap: bool = True):
        self.flat = flat
        self.lr, self.weight_decay, self.betas, self.eps, self.gradient_clip = lr, weight_decay, betas, eps, gradient_clip
        self.exp_avg = torch.zeros_like(flat.grads)
        self.exp_avg_sq = torch.zeros_like(flat.grads)
        self.step_count = 0
        self.group = group
        if grad_comm not in ("fp32", "bf16"):
            raise ValueError("grad_comm must be 'fp32' or 'bf16'")
        self.grad_comm = grad_comm
        self.overlap = bool(overlap)
        self._events = None
        self._comm_stream = None
        self._pending = False
        self.grad_norm = torch.zeros(1, device=flat.device, dtype=torch.float32)
        self.last_allreduce_bytes = 0
        self.param_groups = [{"lr": lr, "weight_decay": weight_decay}]  # what an lr scheduler touches

    def world(self) -> int:
        import torch.distributed as dist
        return dist.get_world_size(self.group) if (dist.is_available() and dist.is_initialized()) else 1

    def _reduce_chunk(self, chunk):
        import torch.distributed as dist
        if self.grad_comm == "bf16":
            c16 = chunk.to(torch.bfloat16)
            dist.all_reduce(c16, group=self.group)
            chunk.copy_(c16)
            self.last_allreduce_bytes += c16.numel() * 2
        else:
            dist.all_reduce(chunk, group=self.group)
            self.last_allreduce_bytes += chunk.numel() * 4

    def arm_overlap(self):
        """Registers one CUDA event per gradient bucket with the handle (once).  From then on every seqdiff_train_step records
        event k when bucket k is final; `launch_overlapped_all_reduce` (called right after training_step) consumes them."""
        if self._events is not None or not self.overlap or self.world() == 1:
            return
        f = self.flat
        nb = len(f.bucket_bounds) - 1
        with torch.cuda.device(f.device):
            self._comm_stream = torch.cuda.Stream(device=f.device)
            self._events = [torch.cuda.Event(enable_timing=False, blocking=False) for _ in range(nb)]
            for e in self._events:
                e.record()  # materialises the cudaEvent_t behind the (lazily created) torch event
            arr = (ctypes.c_void_p * nb)(*[ctypes.c_void_p(e.cuda_event) for e in self._events])
            _cabi.check(_cabi.lib().seqdiff_train_set_bucket_events(f.handle, arr, nb))

    def launch_overlapped_all_reduce(self):
        """Enqueues the per-bucket all-reduces on the communication stream, each behind its bucket's event (tail bucket first: the
        order in which the backward pass finishes them).  Host-side this returns at once; `step()` joins the stream."""
        if self._events is None or not self.overlap:
            return
        f = self.flat
        self.last_allreduce_bytes = 0
        with torch.cuda.stream(self._comm_stream):
            for k in range(len(self._events) - 1, -1, -1):
                self._comm_stream.wait_event(self._events[k])
                self._reduce_chunk(f.grads[f.bucket_bounds[k]:f.bucket_bounds[k + 1]])
        self._pending = True

    def all_reduce_grads(self):
        """sum over the data-parallel ranks, in place on the flat buffer (the averaging 1/world is folded into the update kernel).
        Blocking form (no overlap): the same buckets, on the current stream, after the backward pass."""
        world = self.world()
        self.last_allreduce_bytes = 0
        if world == 1:
            return
        f = self.flat
        for k in range(len(f.bucket_bounds) - 2, -1, -1):
            self._reduce_chunk(f.grads[f.bucket_bounds[k]:f.bucket_bounds[k + 1]])

    def step(self, closure=None, skip_all_reduce: bool = False):
        if self._pending:  # the bucketed all-reduce was launched behind the backward pass: join it
            torch.cuda.current_stream(self.flat.device).wait_stream(self._comm_stream)
            self._pending = False
        elif not skip_all_reduce:
            self.all_reduce_grads()
        self.step_count += 1
        lr = self.param_groups[0]["lr"]
        f = self.flat
        with torch.cuda.device(f.device):
            stream = ctypes.c_void_p(torch.cuda.current_stream(f.device).cuda_stream)
            p = _cabi.ptr
            _cabi.check(_cabi.lib().seqdiff_adamw_step(f.handle, p(f.grads), p(self.exp_avg), p(self.exp_avg_sq), 1.0 / self.world(),
                                                       float(self.gradient_clip or 0.0), float(lr), float(self.betas[0]), float(self.betas[1]),
                                                       float(self.eps), float(self.param_groups[0]["weight_decay"]), self.step_count,
                                                       p(self.grad_norm), stream))
        f.model._weights_dirty = True

    def zero_grad(self, set_to_none: bool = False):
        pass  # seqdiff_train_step overwrites the flat gradient buffer

    def state_dict(self):
        """optimizer checkpoint: step count, the flat AdamW moments (handle index space, see FlatParams.table) and the lr / wd group"""
        return {"step": self.step_count, "exp_avg": self.exp_avg, "exp_avg_sq": self.exp_avg_sq, "param_groups": self.param_groups,
                "table": dict(self.flat.table)}

    def load_state_dict(self, state):
        """resume: restores what state_dict() saved (moments are copied into this optimizer's flat buffers; a checkpoint written for a
        different parameter layout -- other layer count / hidden size -- is rejected)."""
        if "table" in state and dict(state["table"]) != dict(self.flat.table):
            raise ValueError("optimizer state was saved for a different parameter layout")
        for k in ("exp_avg", "exp_avg_sq"):
            src = state[k]
            if src.numel() != getattr(self, k).numel():
                raise ValueError(f"optimizer state '{k}' has {src.numel()} elements, expected {getattr(self, k).numel()}")
            getattr(self, k).copy_(src.to(device=self.flat.device, dtype=torch.float32))
        self.step_count = int(state["step"])
        if state.get("param_groups"):
            self.param_groups[0].update({k: state["param_groups"][0][k] for k in ("lr", "weight_decay") if k in state["param_groups"][0]})


def linear_warmup_factor(epoch: int, warmup: int, total: int) -> float:
    """transformers.get_linear_schedule_with_warmup's lambda (reference model.py:434-446: stepped once per EPOCH)."""
    if epoch < warmup:
        return float(epoch) / float(max(1, warmup))
    return max(0.0, float(total - epoch) / float(max(1, total - warmup)))


def train_step_tensors(model, flat: FlatParams, batch, t_norm, noised_ligand_seq, p_hidden=None, p_attn=None, seed=0, step=0, want_logits=False):
    """forward + loss + backward of one (local) batch: fills flat.grads, returns (terms [10] f64 device tensor, logits or None)."""
    dev = flat.device
    cfg = model.decoder_config
    p_h = float(getattr(cfg, "hidden_dropout_prob", 0.0)) if p_hidden is None else float(p_hidden)
    p_a = float(getattr(cfg, "attention_probs_dropout_prob", 0.0)) if p_attn is None else float(p_attn)
    if not model.training:
        p_h = p_a = 0.0

    def dv(x):
        return x.to(device=dev, dtype=torch.float32).contiguous()

    x0, x_t = dv(batch["ligand_seq"]), dv(noised_ligand_seq)
    B, Ll, _ = x0.shape
    la, lm = dv(batch["ligand_angles"]), dv(batch["ligand_attn_mask"])
    rs, ra, rm = dv(batch["receptor_seq"]), dv(batch["receptor_angles"]), dv(batch["receptor_attn_mask"])
    Lr = rs.shape[1]
    t = dv(t_norm).reshape(-1)
    if t.numel() != B:
        raise ValueError("t_norm must hold one value per graph")
    terms = torch.empty(10, device=dev, dtype=torch.float64)
    logits = torch.empty((B, Ll, 20), device=dev, dtype=torch.float32) if want_logits else None
    h = model._sync_handle()
    with torch.cuda.device(dev):
        stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        p = _cabi.ptr
        _cabi.check(_cabi.lib().seqdiff_train_step(h, model._precision_code(), B, Ll, Lr, p(t), p(x_t), p(x0), p(la), p(lm), p(rs), p(ra), p(rm),
                                                   p_h, p_a, int(seed), int(step) & 0xFFFFFFFF, p(flat.grads), p(terms), p(logits), stream))
    return terms, logits


def struct_train_step_tensors(model, flat: FlatParams, batch, p_hidden=None, p_attn=None, seed=0, step=0, want_pred=False):
    """forward + wrapped smooth-L1 loss + backward of one (local) batch of the structure model (structure_model.ConditionalBertForDiffusion):
    fills flat.grads, returns (terms [F+1] f64 device tensor: per-feature loss sums, then the number of valid ligand positions; the
    prediction [B,L,F] or None).  `batch`: the NoisedAnglesDataset dict (corrupted, t, known_noise, ligand_attn_mask, receptor_seq,
    receptor_angles, receptor_attn_mask); t is the integer step, unnormalised."""
    dev = flat.device
    cfg = model.decoder_config
    p_h = float(getattr(cfg, "hidden_dropout_prob", 0.0)) if p_hidden is None else float(p_hidden)
    p_a = float(getattr(cfg, "attention_probs_dropout_prob", 0.0)) if p_attn is None else float(p_attn)
    if not model.training:
        p_h = p_a = 0.0
    h = model._sync_handle()
    B, Ll, Lr, x, lm, rs, ra, rm = model._inputs(batch["corrupted"], batch["ligand_attn_mask"], batch["receptor_seq"], batch["receptor_angles"],
                                                batch["receptor_attn_mask"])
    Fs = model.feature_size
    noise = batch["known_noise"].to(device=dev, dtype=torch.float32).contiguous()
    if tuple(noise.shape) != (B, Ll, Fs):
        raise ValueError(f"known_noise must be {(B, Ll, Fs)}, got {tuple(noise.shape)}")
    t = batch["t"].to(device=dev, dtype=torch.float32).reshape(-1).contiguous()
    if t.numel() != B:
        raise ValueError("t must hold one step per graph")
    terms = torch.empty(Fs + 1, device=dev, dtype=torch.float64)
    pred = torch.empty((B, Ll, Fs), device=dev, dtype=torch.float32) if want_pred else None
    with torch.cuda.device(dev):
        stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        p = _cabi.ptr
        _cabi.check(_cabi.lib().seqdiff_struct_train_step(h, model._precision_code(), B, Ll, Lr, p(t), p(x), p(noise), p(lm), p(rs), p(ra), p(rm),
                                                          p_h, p_a, int(seed), int(step) & 0xFFFFFFFF, p(flat.grads), p(terms), p(pred), stream))
    return terms, pred


def angle_loss_from_terms(terms):
    """(total loss, per-feature losses) of the structure model's objective from its F+1 reduction terms (device tensors, fp32)."""
    per_feature = (terms[:-1] / terms[-1]).float()
    return per_feature.mean(), per_feature


def loss_from_terms(terms):
    """the 6-tuple of PeptideDiff.get_loss (model.py:345) from the ten reduction terms."""
    n_mask, n_noised, n_sel, n_same, n_rec, ce_noised, ce_sel, ent, kl = (terms[i] for i in range(9))
    aa_noised_loss = (ce_noised / n_noised).float()
    elbo = (-ent / n_noised + kl / n_noised).float()
    return (aa_noised_loss + elbo, elbo, aa_noised_loss, (ce_sel / n_sel).float(), (n_rec / n_mask).float(), (n_same / n_mask).float())


def pull_weights(model):
    """handle masters -> the module's torch parameters (after optimizer steps; before state_dict() / checkpoints)."""
    lib = _cabi.lib()
    h = model._handle
    if h is None:
        return
    dev = model._handle_dev
    with torch.cuda.device(dev):
        stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        names = set(model._flat.table) if getattr(model, "_flat", None) is not None else None
        with torch.no_grad():
            for k, prm in model.named_parameters():
                if names is not None and k not in names:
                    continue
                buf = prm.data if (prm.dtype == torch.float32 and prm.is_contiguous() and prm.device == dev) else torch.empty(prm.shape, device=dev)
                _cabi.check(lib.seqdiff_model_get_tensor(h, k.encode(), _cabi.ptr(buf), buf.numel(), stream))
                if buf is not prm.data:
                    prm.data.copy_(buf)
        torch.cuda.current_stream(dev).synchronize()
    # the torch tensors now EQUAL the handle's masters: refresh the signature so the next forward does not re-upload them
    model._handle_sig = tuple((t.data_ptr(), t._version) for _, t in (model._handle_tensors or []))
    model._weights_dirty = False


def fit(model, train_batches, max_epochs: int = 1, min_epochs: int = 0, log_every_n_steps: int = 30, group=None, log=print, grad_comm="fp32"):
    """The inner loop Lightning's Trainer.fit runs for the reference (train_model.py:92-110): for every epoch, for every batch:
    training_step -> optimizer step (all-reduce + clip + AdamW); LinearWarmup stepped per epoch.  `train_batches`: an iterable of
    batch dicts (re-iterated every epoch).  Returns the list of per-epoch mean training losses."""
    opt = model.configure_optimizers(group=group, grad_comm=grad_comm)["optimizer"]
    base_lr = opt.param_groups[0]["lr"]
    warm = int(max_epochs * 0.1)
    history = []
    model.train()
    for epoch in range(max_epochs):
        if model.lr_scheduler == "LinearWarmup":
            opt.param_groups[0]["lr"] = base_lr * linear_warmup_factor(epoch, warm, max_epochs)
        losses = []
        for i, batch in enumerate(train_batches):
            loss = model.training_step(batch, i)
            opt.step()
            losses.append(loss)
            if log and log_every_n_steps and (i + 1) % log_every_n_steps == 0:
                log(f"epoch {epoch} step {i + 1}: train_loss {float(loss):.4f} grad_norm {float(opt.grad_norm):.3f}")
        mean = float(torch.stack([l.detach().float() for l in losses]).mean()) if losses else float("nan")
        history.append(mean)
        if log:
            log(f"Traning Loss:{mean}")  # (sic) the reference's epoch log line, model.py:375-377
    pull_weights(model)
    return history
