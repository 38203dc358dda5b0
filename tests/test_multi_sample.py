"""K samples per pocket (seqdiff_sample_multi through denoise_tensors(num_samples=K)): the receptor rows of every step are computed
once per pocket and the K samples' cross-attention reads that pocket's K|V.  A receptor row's value depends on the pocket and the
step only (no split-K GEMM, so a row's result does not depend on M; attention items are per (graph, head)), so the final logits
must equal, bit for bit, the K = 1 sampling of the batch whose entries are repeated K times per pocket -- with the same x_T, noise,
seed and graph ids.  Packed mode: at the valid positions, padded ones 0."""
import pytest
import torch

from helpers import O, make_model, sd_pkg

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

_MODEL = {}


def _model(precision):
    if not _MODEL:
        # variant "B": decoder_normalize is not the identity the reference init makes it
        cfg = O.OracleConfig(max_position_embeddings=128, relative_key=True)
        _MODEL["m"] = make_model(sd_pkg(), cfg, O.init_state_dict(cfg, 1, "B"), precision)
    m = _MODEL["m"]
    m.precision = precision
    return m


def _pockets(case, P, seed):
    if case == "Ll==Lr":
        return O.synthetic_batch(P, 64, (5, 40), (16, 64), seed)
    batch = O.synthetic_batch(P, 48, (1, 48), (1, 48), seed)
    rec = O.synthetic_batch(P, 112, (1, 112), (16, 112), seed + 1)
    for k in ("receptor_seq", "receptor_angles", "receptor_attn_mask"):
        batch[k] = rec[k]
    return batch


def _replicated(batch, K):
    return {k: v.repeat_interleave(K, dim=0) for k, v in batch.items()}


def _check(final, want, batch, K, packed):
    assert final.shape == want.shape
    if not packed:
        assert torch.equal(final, want)
        return
    valid = batch["ligand_attn_mask"].repeat_interleave(K, dim=0).bool().to(DEV)
    assert torch.equal(final[valid], want[valid])
    assert (final[~valid] == 0).all()


@pytest.mark.parametrize("noise", ["exp1", "philox"])
@pytest.mark.parametrize("K", [1, 3])
@pytest.mark.parametrize("case", ["Ll==Lr", "Ll!=Lr"])
@pytest.mark.parametrize("precision,packed", [("bf16", False), ("bf16", True), ("fp16", False), ("fp16", True), ("fp32", False)])
def test_shared_pocket_equals_replicated_batch(precision, packed, case, K, noise):
    sd = sd_pkg()
    m = _model(precision)
    sd.sample.DEVICE = torch.device(DEV)
    T, P = 5, 3
    batch = _pockets(case, P, 71)
    Ll = batch["ligand_seq"].shape[1]
    g = torch.Generator().manual_seed(5)
    x_T = O.generate_discrete_noise(P * K, Ll, generator=g)
    E = torch.empty(T, P * K * Ll, 20).exponential_(1, generator=g) if noise == "exp1" else None
    sched, tr = sd.PredefinedNoiseScheduleDiscrete("cosine", T), sd.BlosumTransition(x_classes=20)
    kw = dict(timesteps=T, x_T=x_T, noise_E_steps=E, seed=11, graph_id0=1000, packed=packed)
    final = sd.denoise_tensors(batch, m, sched, tr, True, num_samples=K, **kw).clone()
    want = sd.denoise_tensors(_replicated(batch, K), m, sched, tr, True, **kw)
    _check(final, want, batch, K, packed)
    if noise == "philox" and K > 1:
        for p in range(P):  # per-graph Philox streams: the samples of one pocket differ
            assert not all(torch.equal(final[p * K], final[p * K + j]) for j in range(1, K)), p


@pytest.mark.parametrize("packed", [False, True])
def test_cached_graph_across_sample_counts(packed):
    """B = 8 graphs as 4 pockets x 2, 2 pockets x 4, then 4 x 2 twice: K is part of the step graph's key, so every change of K
    captures a fresh graph (same B, other receptor row count), and the repeated call replays the cached one.  Each call equals
    its own replicated reference."""
    sd = sd_pkg()
    m = _model("bf16")
    sd.sample.DEVICE = torch.device(DEV)
    T = 4
    sched, tr = sd.PredefinedNoiseScheduleDiscrete("cosine", T), sd.BlosumTransition(x_classes=20)
    g = torch.Generator().manual_seed(6)
    runs, results = [], []
    for i, (P, K) in enumerate(((4, 2), (2, 4), (4, 2), (4, 2))):
        batch = _pockets("Ll==Lr", P, 80 + min(i, 2))  # call 3 repeats call 2's shapes (packed mode keys its graph on the lengths)
        x_T = O.generate_discrete_noise(P * K, batch["ligand_seq"].shape[1], generator=g)
        kw = dict(timesteps=T, x_T=x_T, seed=20 + i, graph_id0=50 * i, packed=packed)
        torch.cuda.synchronize()
        n0 = sd.lib().seqdiff_launch_count()
        final = sd.denoise_tensors(batch, m, sched, tr, True, num_samples=K, **kw).clone()
        torch.cuda.synchronize()
        runs.append(sd.lib().seqdiff_launch_count() - n0)
        results.append((final, batch, K, kw))
    # references only after the four calls: they would replace the cached graph
    for final, batch, K, kw in results:
        _check(final, sd.denoise_tensors(_replicated(batch, K), m, sched, tr, True, **kw), batch, K, packed)
    # a capture adds the dry-run forward's launches: call 2 captures (the previous call had another K), call 3 replays its graph
    assert runs[3] < runs[2], runs
