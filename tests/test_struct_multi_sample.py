"""K backbones per pocket in the structure sampler (p_sample_loop(num_samples=K), seqdiff_struct_sample_multi): the receptor branch
(embeddings, receptor_emb, the encoder and every decoder layer's cross K|V) runs once over the P pockets, and the K samples'
cross-attention reads their pocket's K|V.  A receptor row's value depends on its pocket only (no inference GEMM splits K, attention
items are per (graph, head)), so the whole history and the final angles must equal, bit for bit, the K = 1 loop on the batch whose
pockets are repeated K times -- with the same start state, noise, seed and graph ids."""
import math

import pytest
import torch

from oracle import seqdiff_oracle as O
from oracle import structdiff_oracle as S

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
FS = 8

_MODELS = {}


def _model(L, precision):
    if L not in _MODELS:
        import seqdiff_b200 as sd
        cfg = S.OracleConfig(max_position_embeddings=L, num_hidden_layers=2, feature_size=FS, relative_key=True)
        common = dict(max_position_embeddings=L, num_attention_heads=cfg.num_attention_heads, hidden_size=cfg.hidden_size,
                      intermediate_size=cfg.intermediate_size, num_hidden_layers=2, position_embedding_type="relative_key")
        m = sd.structure_model.ConditionalBertForDiffusionBase(sd.BertConfig(**common),
                                                               sd.BertConfig(**common, is_decoder=True, add_cross_attention=True), FS)
        m.load_state_dict(S.init_struct_state_dict(cfg, 61), strict=True)
        _MODELS[L] = m.eval().to(DEV)
    m = _MODELS[L]
    m.precision = precision
    return m


def _masks(lens, L):
    return (torch.arange(L)[None, :] < torch.tensor(lens)[:, None]).float()


def _pockets(case, P, K, seed):
    """(model length, ligand mask [P*K, Ll] -- every sample its own length --, receptor seq / angles / mask of the P pockets)"""
    g = torch.Generator().manual_seed(seed)
    if case == "Ll==Lr":
        L, Ll, Lr = 64, 64, 64
        lm = O.synthetic_batch(P * K, Ll, (5, 64), (16, 64), seed)["ligand_attn_mask"]
        rm = O.synthetic_batch(P, Lr, (5, 64), (16, 64), seed + 1)["receptor_attn_mask"]
    elif case == "len1":  # a length-1 ligand next to full-length ones
        L, Ll, Lr = 64, 64, 64
        lm = _masks([1, 64, 30][:P * K] + [7] * max(0, P * K - 3), Ll)
        rm = _masks([64, 20, 48][:P] + [33] * max(0, P - 3), Lr)
    else:  # Ll != Lr
        L, Ll, Lr = 96, 40, 96
        lm = O.synthetic_batch(P * K, Ll, (1, 40), (1, 40), seed)["ligand_attn_mask"]
        rm = O.synthetic_batch(P, Lr, (1, 96), (16, 96), seed + 1)["receptor_attn_mask"]
    rseq = torch.nn.functional.one_hot(torch.randint(0, 20, (P, Lr), generator=g), 20).float() * rm[..., None]
    rang = ((torch.rand(P, Lr, FS, generator=g) * 2 - 1) * math.pi) * rm[..., None]
    x_T = (torch.rand(P * K, Ll, FS, generator=g) * 2 - 1) * math.pi
    return L, lm, rseq, rang, rm, x_T


def _run(m, lm, rseq, rang, rm, x_T, T, K, **kw):
    import seqdiff_b200 as sd
    SM = sd.structure_model
    return SM.p_sample_loop(m, lm.to(DEV), x_T.to(DEV), rseq.to(DEV), rm.to(DEV), rang.to(DEV), T, SM.cosine_beta_schedule(T),
                            num_samples=K, **kw)


def _replicated(m, lm, rseq, rang, rm, x_T, T, K, **kw):
    """the K = 1 loop on the batch with every pocket repeated K times"""
    r = lambda t: t.repeat_interleave(K, dim=0)  # noqa: E731
    return _run(m, lm, r(rseq), r(rang), r(rm), x_T, T, 1, **kw)


@pytest.mark.parametrize("noise", ["philox", "explicit"])
@pytest.mark.parametrize("K", [1, 3])
@pytest.mark.parametrize("case", ["Ll==Lr", "Ll!=Lr", "len1"])
@pytest.mark.parametrize("precision,packed", [("bf16", False), ("bf16", True), ("fp16", False), ("fp16", True), ("fp32", False)])
def test_shared_pocket_equals_replicated_batch(precision, packed, case, K, noise):
    P, T = 3, 5
    L, lm, rseq, rang, rm, x_T = _pockets(case, P, K, 31)
    m = _model(L, precision)
    kw = dict(seed=7, graph_id0=500, packed=packed)
    if noise == "explicit":
        kw["noise_steps"] = torch.randn(T, *x_T.shape, generator=torch.Generator().manual_seed(32))
    got = _run(m, lm, rseq, rang, rm, x_T, T, K, **kw)
    want = _replicated(m, lm, rseq, rang, rm, x_T, T, K, **kw)
    assert got.shape == want.shape == (T, P * K, x_T.shape[1], FS)
    assert torch.equal(got, want), (got - want).abs().max()
    final = _run(m, lm, rseq, rang, rm, x_T, T, K, keep_history=False, **kw)
    assert torch.equal(final[0], want[-1])
    if K > 1 and noise == "philox":
        for p in range(P):  # per-graph Philox streams: the backbones of one pocket differ
            assert not all(torch.equal(got[-1, p * K], got[-1, p * K + j]) for j in range(1, K)), p


@pytest.mark.parametrize("packed", [False, True])
def test_per_pocket_ligand_mask_is_repeated(packed):
    """a [P, L] ligand mask stands for its K samples"""
    P, K, T = 2, 3, 4
    L, lm, rseq, rang, rm, x_T = _pockets("Ll==Lr", P, 1, 33)
    x_T = x_T.repeat_interleave(K, dim=0)
    m = _model(L, "bf16")
    kw = dict(seed=4, graph_id0=90, packed=packed)
    assert torch.equal(_run(m, lm, rseq, rang, rm, x_T, T, K, **kw), _run(m, lm.repeat_interleave(K, dim=0), rseq, rang, rm, x_T, T, K, **kw))


@pytest.mark.parametrize("packed", [False, True])
def test_cached_graph_across_sample_counts(packed):
    """B = 8 graphs as 4 pockets x 2, 2 x 4, then 4 x 2 twice: K is part of the step graph's key (same B, another receptor row count),
    so every change of K captures a fresh graph and the repeated call replays the cached one.  Each call equals its own replicated
    reference."""
    import seqdiff_b200 as sd
    T = 4
    m = _model(64, "bf16")
    runs, results = [], []
    for i, (P, K) in enumerate(((4, 2), (2, 4), (4, 2), (4, 2))):
        inputs = _pockets("Ll==Lr", P, K, 40 + min(i, 2))  # call 3 repeats call 2's inputs (packed mode keys its graph on the lengths)
        kw = dict(seed=20 + i, graph_id0=50 * i, packed=packed)
        torch.cuda.synchronize()
        n0 = sd.lib().seqdiff_launch_count()
        got = _run(m, *inputs[1:], T, K, **kw)
        torch.cuda.synchronize()
        runs.append(sd.lib().seqdiff_launch_count() - n0)
        results.append((got, inputs, K, kw))
    # references only after the four calls: they would replace the cached graph
    for got, inputs, K, kw in results:
        assert torch.equal(got, _replicated(m, *inputs[1:], T, K, **kw))
    assert runs[3] < runs[2], runs  # call 2 captures (the previous call had another K), call 3 replays its graph


def test_sample_driver_num_samples():
    """structure_model.sample(num_samples=K): P*K trimmed arrays in (complex, sample) order, equal to sample() on the dataset whose
    complexes are repeated K times (the start noise is drawn for P*K graphs either way)"""
    import seqdiff_b200 as sd
    SM = sd.structure_model
    m = _model(64, "bf16")
    T, n, K = 4, 3, 2
    b = O.synthetic_batch(n, 64, (1, 64), (16, 64), 34)

    class DS:
        timesteps = T
        alpha_beta_terms = {"betas": SM.cosine_beta_schedule(T)}

        def __init__(self, rep):
            self.rep = rep

        def __len__(self):
            return n * self.rep

        def __getitem__(self, i):
            return {k: b[k][i // self.rep] for k in ("ligand_attn_mask", "ligand_angles", "receptor_angles", "receptor_seq",
                                                     "receptor_attn_mask")}

        def sample_noise(self, v):
            return SM.modulo_with_wrapped_range(torch.randn(v.shape, generator=torch.Generator().manual_seed(35)))

    got = SM.sample(m, DS(1), seed=2, graph_id0=0, packed=True, num_samples=K)
    want = SM.sample(m, DS(K), seed=2, graph_id0=0, packed=True)
    assert len(got) == len(want) == n * K
    for i, (g_, w_) in enumerate(zip(got, want)):
        assert g_.shape == (T, int(b["ligand_attn_mask"][i // K].sum()), FS) and g_.tobytes() == w_.tobytes()
