"""Drop-in for `sequence_model/sample.py` of the reference: same module-level CONFIG vocabulary and
the same free functions / signatures, with the arithmetic on the GPU:

  * `sample_p_zs_given_zt_discrete`  -> one launch of the CUDA reverse-step kernel (instead of three
    [N,20,20] temporaries plus a Python loop of N multinomial calls with a D2H sync each);
  * `denoise`                        -> ONE C call (`seqdiff_sample`) that replays a captured CUDA graph
    (denoiser forward + reverse step) T times; no host round trip inside the loop.

Randomness.  The reference draws from torch's global CPU generator (`randint`, then `multinomial`
= argmax(prob / Exp(1))).  Here x_T uses the same `torch.randint` call, and the per-step race noise is
either handed in explicitly (`noise_E`, parity runs) or generated in-kernel by Philox4x32-10 keyed by
(SEED, global graph id, residue, step) so results do not depend on how a batch is sharded over GPUs.
"""
from __future__ import annotations

import ctypes

import torch
from torch.nn import functional as F

from . import _cabi
from .model import AA_VOCAB, BertConfig, PeptideDiff
from .utils import BlosumTransition, DiscreteUniformTransition, PredefinedNoiseScheduleDiscrete, loop_tables, step_tables

GPU_ID = 0
DEVICE = torch.device(f"cuda:{GPU_ID}")
THREAD_NUM = 16
SEED = 0          # Philox key for the in-kernel sampling noise
_CALLS = [0]      # stream offset: every stochastic call consumes one "step" id

# same keys as the reference CONFIG (sample.py:28-50)
CONFIG = {
    "pocket_ext": 0,
    "timesteps": 50,
    "max_seq_len": 64,
    "noise_schedule": "cosine",
    "num_heads": 12,
    "dropout_p": 0.1,
    "hidden_size": 768,
    "num_hidden_layers": 6,
    "intermediate_size": 1024,
    "position_embedding_type": "relative_key",
    "lr": 5e-5,
    "l2_norm": 0.1,
    "loss": "smooth_l1",
    "gradient_clip": 1.0,
    "lr_scheduler": "LinearWarmup",
    "min_epochs": 100,
    "max_epochs": 150,
    "batch_size": 64,
}


def get_model(steps_per_epoch=1, state_dict=None) -> PeptideDiff:
    """reference sample.py:68-110; `state_dict` replaces torch.load(MODEL_PATH) (weights are unreachable)."""
    common = dict(
        max_position_embeddings=CONFIG["max_seq_len"], num_attention_heads=CONFIG["num_heads"], hidden_size=CONFIG["hidden_size"],
        intermediate_size=CONFIG["intermediate_size"], num_hidden_layers=CONFIG["num_hidden_layers"],
        position_embedding_type=CONFIG["position_embedding_type"], hidden_dropout_prob=CONFIG["dropout_p"],
        attention_probs_dropout_prob=CONFIG["dropout_p"], use_cache=False)
    encoder_config = BertConfig(**common)
    decoder_config = BertConfig(**common, is_decoder=True, add_cross_attention=True)
    model = PeptideDiff(encoder_config=encoder_config, decoder_config=decoder_config, feature_names=list(AA_VOCAB),
                        max_epochs=CONFIG["max_epochs"], lr_scheduler=CONFIG["lr_scheduler"], l2_lambda=CONFIG["l2_norm"],
                        steps_per_epoch=steps_per_epoch, learning_rate=CONFIG["lr"], loss_func=torch.nn.CrossEntropyLoss(),
                        noise_schedule=CONFIG["noise_schedule"], timesteps=CONFIG["timesteps"])
    if state_dict is not None:
        model.load_state_dict(state_dict)
    return model.eval().to(DEVICE)


def generate_discrete_noise(batch_size, length, num_classes=20, device=None):
    """reference sample.py:112-116: x_T = one-hot of uniform class indices drawn from torch's global CPU generator (the same
    `torch.randint` call, hence the same x_T under the same `torch.manual_seed`)."""
    classes = torch.randint(0, num_classes, (batch_size, length))
    return F.one_hot(classes, num_classes).to(dtype=torch.float32, device=DEVICE if device is None else device)


def sample_p_zs_given_zt_discrete(t, s, noised_data, pred_noise, noise_schedule, transition, diverse, is_last_step,
                                  noise_E=None, graph_id0=0):
    """reference sample.py:141-179: sample zs ~ p(zs | zt).  Extra keyword `noise_E` [B*L,20] = the Exp(1)
    race noise (what torch.multinomial draws internally) for same-noise parity runs."""
    if is_last_step:
        return pred_noise
    batch_size, seq_len, num_class = noised_data.shape
    if num_class != 20:
        raise ValueError("the CUDA reverse step is specialised for 20 classes")
    dev = pred_noise.device if pred_noise.device.type == "cuda" else DEVICE
    tables = step_tables(t, s, noise_schedule, transition).to(dev)  # [B,3,20,20], host-built like sample.py:156-160
    x = noised_data.to(device=dev, dtype=torch.float32).contiguous()
    logits = pred_noise.to(device=dev, dtype=torch.float32).contiguous()
    E = None if noise_E is None else noise_E.to(device=dev, dtype=torch.float32).contiguous()
    out = torch.empty_like(x)
    _CALLS[0] += 1
    with torch.cuda.device(dev):
        stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        _cabi.check(_cabi.lib().seqdiff_reverse_step(_cabi.ptr(tables), tables.shape[0], batch_size, seq_len, _cabi.ptr(x),
                                                     _cabi.ptr(logits), int(bool(diverse)), _cabi.ptr(E), SEED, graph_id0,
                                                     _CALLS[0] & 0x0FFFFFFF, _cabi.ptr(out), None, stream))
    return out


def check_num_samples(num_samples) -> int:
    """The number of sequences sampled per pocket: a positive int (ValueError otherwise)."""
    if isinstance(num_samples, bool) or not isinstance(num_samples, int) or num_samples < 1:
        raise ValueError(f"num_samples must be a positive int, got {num_samples!r}")
    return num_samples


@torch.no_grad()
def denoise_tensors(batch, model, noise_schedule, transition, diverse, timesteps=None, x_T=None, noise_E_steps=None,
                    graph_id0=None, seed=None, packed=False, num_samples=1):
    """The T-step loop of reference denoise() (sample.py:184-207) as one C call.  Returns the final
    [B,L,20] tensor (raw logits of the last step, quirk Q4) on the model's device.
    `graph_id0` = global id of the batch's first graph in the Philox noise stream; None (default) continues the process-wide
    stream (`_cabi.GRAPH_IDS`), so consecutive batches and repeated calls never share noise.
    `packed=True`: ragged packing (seqdiff_sample_ex, SEQDIFF_SAMPLE_PACKED) -- only the valid prefix of every graph is computed;
    the result is bit-identical at the valid positions (all that denoise() reads) and 0 at the padded ones.
    `num_samples=K > 1`: K sequences per pocket of the batch (seqdiff_sample_multi).  The batch holds P pockets; the result, x_T and
    the graph ids cover B = P*K graphs, sample j of pocket p being graph p*K + j, and noise_E_steps is [T, P*K*L, 20].  Each pocket's
    receptor rows are computed once per step for its K samples; the result equals the K = 1 call on the batch whose entries are
    repeated K times per pocket."""
    K = check_num_samples(num_samples)
    T = CONFIG["timesteps"] if timesteps is None else timesteps
    h = model._sync_handle()
    dev = model._handle_dev  # the handle's device owns the stream, the workspace and every tensor of this call
    n_pockets, max_len, num_class = batch["ligand_seq"].shape
    batch_size = n_pockets * K
    if graph_id0 is None:
        graph_id0 = _cabi.GRAPH_IDS.take(batch_size)
    if x_T is None:
        x_T = generate_discrete_noise(batch_size, max_len, num_class, device=dev)

    def dv(x):
        return x.to(device=dev, dtype=torch.float32, non_blocking=True).contiguous()

    x_T = dv(x_T)
    ligand_mask, ligand_angles = dv(batch["ligand_attn_mask"]), dv(batch["ligand_angles"])
    if K > 1:
        if tuple(x_T.shape) != (batch_size, max_len, num_class):
            raise ValueError(f"x_T must be [P*K, L, {num_class}] = {(batch_size, max_len, num_class)}, got {tuple(x_T.shape)}")
        ligand_mask, ligand_angles = ligand_mask.repeat_interleave(K, dim=0), ligand_angles.repeat_interleave(K, dim=0)
    receptor_seq, receptor_angles = dv(batch["receptor_seq"]), dv(batch["receptor_angles"])
    receptor_attn_mask = dv(batch["receptor_attn_mask"])
    Lr = receptor_seq.shape[1]
    tables = loop_tables(T, noise_schedule, transition)
    if tables.shape[0] != T or tables.shape[1:] != (3, 20, 20):
        raise ValueError("transition tables must be [T,3,20,20] (per-step scalar schedule)")
    tables = tables.to(dev)
    E = None if noise_E_steps is None else dv(noise_E_steps)
    if E is not None and tuple(E.shape) != (T, batch_size * max_len, 20):
        raise ValueError("noise_E_steps must be [T, B*L, 20]" if K == 1 else "noise_E_steps must be [T, P*K*L, 20]")
    out = torch.empty((batch_size, max_len, num_class), device=dev, dtype=torch.float32)
    with torch.cuda.device(dev):
        stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        if K > 1:
            _cabi.check(_cabi.lib().seqdiff_sample_multi(h, model._precision_code(), n_pockets, K, max_len, Lr, T, _cabi.ptr(tables),
                                                         _cabi.ptr(x_T), _cabi.ptr(ligand_angles), _cabi.ptr(ligand_mask),
                                                         _cabi.ptr(receptor_seq), _cabi.ptr(receptor_angles), _cabi.ptr(receptor_attn_mask),
                                                         int(bool(diverse)), _cabi.ptr(E), SEED if seed is None else seed, graph_id0,
                                                         1 if packed else 0, _cabi.ptr(out), stream))
            return out
        _cabi.check(_cabi.lib().seqdiff_sample_ex(h, model._precision_code(), batch_size, max_len, Lr, T, _cabi.ptr(tables), _cabi.ptr(x_T),
                                                  _cabi.ptr(ligand_angles), _cabi.ptr(ligand_mask), _cabi.ptr(receptor_seq),
                                                  _cabi.ptr(receptor_angles), _cabi.ptr(receptor_attn_mask), int(bool(diverse)),
                                                  _cabi.ptr(E), SEED if seed is None else seed, graph_id0, 1 if packed else 0,
                                                  _cabi.ptr(out), stream))
    return out


def decode_tensors(final, ligand_seq, ligand_mask):
    """reference sample.py:208-216 on the device: (pred_idx [B,L] u8, true_idx [B,L] u8, counts [B,2] i64 = matches, valid)."""
    dev = final.device
    if dev.type != "cuda":
        raise RuntimeError("decode runs only on a CUDA device (no CPU fallback)")
    B, L, _ = final.shape
    f = final.to(torch.float32).contiguous()
    t = ligand_seq.to(device=dev, dtype=torch.float32).contiguous()
    m = ligand_mask.to(device=dev, dtype=torch.float32).contiguous()
    pred = torch.empty((B, L), device=dev, dtype=torch.uint8)
    true = torch.empty((B, L), device=dev, dtype=torch.uint8)
    counts = torch.empty((B, 2), device=dev, dtype=torch.int32)
    with torch.cuda.device(dev):
        stream = ctypes.c_void_p(torch.cuda.current_stream(dev).cuda_stream)
        _cabi.check(_cabi.lib().seqdiff_decode(B, L, _cabi.ptr(f), _cabi.ptr(t), _cabi.ptr(m), _cabi.ptr(pred), _cabi.ptr(true),
                                               _cabi.ptr(counts), stream))
    return pred, true, counts.long()


@torch.no_grad()
def denoise(batch, model: PeptideDiff, noise_schedule, transition, diverse, num_samples=1, **kw):
    """reference sample.py:181-229: returns (structure_ids, true_sequences, pred_sequences, recovery_rates).
    `num_samples=K`: K sequences per pocket of the batch (denoise_tensors); the lists then hold P*K entries in (pocket, sample)
    order, with each pocket's structure id and true sequence repeated for its samples."""
    K = check_num_samples(num_samples)
    batch_size = batch["ligand_seq"].shape[0] * K
    final = denoise_tensors(batch, model, noise_schedule, transition, diverse, num_samples=K, **kw)
    ligand_seq, ligand_mask = batch["ligand_seq"], batch["ligand_attn_mask"]
    if K > 1:
        ligand_seq, ligand_mask = ligand_seq.repeat_interleave(K, dim=0), ligand_mask.repeat_interleave(K, dim=0)
    # sample.py:208-224 in one kernel: argmax decode of both sequences + per-graph (matches, valid) counts; the host gets
    # 2 x [B,L] bytes + [B,2] ints in one synchronising copy (the reference syncs once per graph) and only joins letters
    pred_idx, true_idx, counts = decode_tensors(final, ligand_seq, ligand_mask)
    pred_idx, true_idx, counts = pred_idx.cpu(), true_idx.cpu(), counts.cpu()
    n_valid = counts[:, 1].tolist()
    rates = (counts[:, 0] / counts[:, 1]).tolist()  # int64 / int64 -> float32 true division, as recovery_rate.sum()/mask.sum()
    masks = ligand_mask.bool().cpu()
    recovery_rates, pred_sequences, true_sequences, structure_ids = [], [], [], []
    for i in range(batch_size):
        mask = masks[i]
        if int(mask.sum()) != n_valid[i]:
            raise RuntimeError("decode kernel and host disagree on the mask population")
        pred_seq, true_seq = pred_idx[i][mask].tolist(), true_idx[i][mask].tolist()
        recovery_rates.append(rates[i])
        pred_sequences.append("".join(AA_VOCAB[j] for j in pred_seq))
        true_sequences.append("".join(AA_VOCAB[j] for j in true_seq))
        ids = batch.get("structure_ids")
        structure_ids.append(f'{ids["pdb_id"][i // K]}_{ids["ligand_chain"][i // K]}' if ids is not None else str(i // K))
    print(sum(recovery_rates) / len(recovery_rates))
    return structure_ids, true_sequences, pred_sequences, recovery_rates


def load_generated_angles(angles, max_seq_len=None, batch_size=None):
    """reference sample_by_generated_angles.py:54-66: per-complex angle arrays [len_i, 8] (a pickle path, or the list itself --
    e.g. the last step of structure_model.sample()'s outputs) zero-padded to max_seq_len and chunked by batch_size."""
    import pickle

    import numpy as np
    if isinstance(angles, (str, bytes)):
        with open(angles, "rb") as f:
            angles = pickle.load(f)
    L = CONFIG["max_seq_len"] if max_seq_len is None else max_seq_len
    bs = CONFIG["batch_size"] if batch_size is None else batch_size
    padded = torch.Tensor(np.array([np.pad(np.asarray(a, dtype=np.float32), ((0, L - np.asarray(a).shape[0]), (0, 0)), mode="constant",
                                           constant_values=0) for a in angles]))
    return [padded[i:i + bs] for i in range(0, len(padded), bs)]


def denoise_with_generated_angles(batch, generated_angles, model, noise_schedule, transition, diverse, denoise_fn=None, **kw):
    """reference sample_by_generated_angles.py:197-245: `denoise` with the ligand angles replaced by the structure model's output
    (line 202); the caller passes `DiscreteUniformTransition(20)` as the reference's main block does (line 253)."""
    if tuple(generated_angles.shape) != tuple(batch["ligand_angles"].shape):
        raise ValueError(f"generated angles {tuple(generated_angles.shape)} do not match the batch {tuple(batch['ligand_angles'].shape)}")
    swapped = dict(batch)
    swapped["ligand_angles"] = generated_angles
    return (denoise if denoise_fn is None else denoise_fn)(swapped, model, noise_schedule, transition, diverse, **kw)


def sample_dataset(dataloader, model, noise_schedule=None, transition=None, diverse=True, output_path=None, denoise_fn=None,
                   generated_angles=None, num_samples=1, **kw):
    """The `__main__` block of the reference (sample.py:231-257): every batch of `dataloader` through `denoise`, results
    collected in the reference's DataFrame (columns structure_ids / true_sequence / predict_sequence / recovery_rate) and, when
    `output_path` is given, pickled exactly like `res.to_pickle(OUTPUT_PATH)`.  Returns the DataFrame.  `generated_angles` (chunks
    from `load_generated_angles`) turns it into the main block of sample_by_generated_angles.py:247-278.  `num_samples=K > 1`:
    K sequences per pocket, rows in (pocket, sample) order."""
    import pandas as pd
    if check_num_samples(num_samples) > 1:
        kw["num_samples"] = num_samples
    if noise_schedule is None:
        noise_schedule = PredefinedNoiseScheduleDiscrete(CONFIG["noise_schedule"], CONFIG["timesteps"])
    if transition is None:
        transition = BlosumTransition(x_classes=20)
    fn = denoise if denoise_fn is None else denoise_fn
    structure_ids, true_sequences, pred_sequences, recovery_rates = [], [], [], []
    for idx, batch in enumerate(dataloader):
        print(f"Generating Batch {idx}")
        if generated_angles is not None:  # sample_by_generated_angles.py:260-265
            ids, true_seq, pred_seq, rec_rates = denoise_with_generated_angles(batch, generated_angles[idx], model, noise_schedule, transition,
                                                                               diverse, denoise_fn=fn, **kw)
        else:
            ids, true_seq, pred_seq, rec_rates = fn(batch, model, noise_schedule, transition, diverse, **kw)
        structure_ids.extend(ids)
        recovery_rates.extend(rec_rates)
        pred_sequences.extend(pred_seq)
        true_sequences.extend(true_seq)
    res = pd.DataFrame(zip(structure_ids, true_sequences, pred_sequences, recovery_rates),
                       columns=["structure_ids", "true_sequence", "predict_sequence", "recovery_rate"])
    if output_path is not None:
        res.to_pickle(output_path)
    return res
