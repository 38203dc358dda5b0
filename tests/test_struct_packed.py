"""Ragged packing of the structure sampler (p_sample_loop(packed=True), seqdiff_struct_sample_ex with SEQDIFF_SAMPLE_PACKED): only the
valid prefix of every complex goes through the two BERT stacks and the Gaussian step.  A padded key's probability underflows to
exactly 0, every other operator is row-local, no inference GEMM splits K, and a valid element draws the Philox value of its group
inside the padded graph -- so every valid position of the history and of the final angles must equal the padded loop bit for bit,
and the padded positions are 0."""
import math

import pytest
import torch

from oracle import seqdiff_oracle as O
from oracle import structdiff_oracle as S

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
FS = 8

_MODELS = {}


def _model(L, layers, rel, precision):
    key = (L, layers, rel)
    if key not in _MODELS:
        import seqdiff_b200 as sd
        cfg = S.OracleConfig(max_position_embeddings=L, num_hidden_layers=layers, feature_size=FS, relative_key=rel)
        pos = "relative_key" if rel else "absolute"
        common = dict(max_position_embeddings=L, num_attention_heads=cfg.num_attention_heads, hidden_size=cfg.hidden_size,
                      intermediate_size=cfg.intermediate_size, num_hidden_layers=layers, position_embedding_type=pos)
        m = sd.structure_model.ConditionalBertForDiffusionBase(sd.BertConfig(**common),
                                                               sd.BertConfig(**common, is_decoder=True, add_cross_attention=True), FS)
        m.load_state_dict(S.init_struct_state_dict(cfg, 61), strict=True)
        _MODELS[key] = m.eval().to(DEV)
    m = _MODELS[key]
    m.precision = precision
    return m


def _masks(lens, L):
    return (torch.arange(L)[None, :] < torch.tensor(lens)[:, None]).float()


def _inputs(case):
    """(model key, ligand mask, receptor seq / angles / mask, x_T) of one test case"""
    g = torch.Generator().manual_seed(17)
    if case == "struct_bench":  # scripts/struct_bench.py: L = 64, 12 + 12 layers, ligand U(5..64), receptor U(16..64)
        key, B, Ll, Lr = (64, 12, True), 16, 64, 64
        b = O.synthetic_batch(B, Ll, (5, 64), (16, 64), 18)
        lm, rm = b["ligand_attn_mask"], b["receptor_attn_mask"]
    elif case == "len1":  # a length-1 ligand next to a full-length one
        key, B, Ll, Lr = (64, 2, True), 3, 64, 64
        lm, rm = _masks([1, 64, 30], Ll), _masks([64, 20, 64], Lr)
    elif case == "Ll!=Lr":
        key, B, Ll, Lr = (96, 2, True), 5, 48, 96
        lm = O.synthetic_batch(B, Ll, (1, 48), (1, 48), 19)["ligand_attn_mask"]
        rm = O.synthetic_batch(B, Lr, (1, 96), (16, 96), 20)["receptor_attn_mask"]
    else:  # "absolute": no relative-position term in any attention
        key, B, Ll, Lr = (64, 2, False), 6, 64, 64
        b = O.synthetic_batch(B, Ll, (3, 64), (10, 64), 21)
        lm, rm = b["ligand_attn_mask"], b["receptor_attn_mask"]
    rseq = torch.nn.functional.one_hot(torch.randint(0, 20, (B, Lr), generator=g), 20).float() * rm[..., None]
    rang = ((torch.rand(B, Lr, FS, generator=g) * 2 - 1) * math.pi) * rm[..., None]
    x_T = ((torch.rand(B, Ll, FS, generator=g) * 2 - 1) * math.pi)
    return key, lm, rseq, rang, rm, x_T


def _args(m, lm, rseq, rang, rm, x_T, T):
    import seqdiff_b200 as sd
    return dict(model=m, ligand_mask=lm.to(DEV), ligand_angle_noise=x_T.to(DEV), receptor_seq=rseq.to(DEV), receptor_mask=rm.to(DEV),
                receptor_angle=rang.to(DEV), total_timesteps=T, betas=sd.structure_model.cosine_beta_schedule(T))


def _check_packed(got, want, lm):
    """got / want [T or 1, B, L, F]: equal at the valid positions, got 0 at the padded ones"""
    assert got.shape == want.shape
    valid = lm.bool()[None, :, :, None].expand_as(got)
    assert torch.equal(got[valid], want[valid]), (got[valid] - want[valid]).abs().max()
    assert (got[~valid] == 0).all()


@pytest.mark.parametrize("noise", ["philox", "explicit"])
@pytest.mark.parametrize("case", ["struct_bench", "len1", "Ll!=Lr", "absolute"])
@pytest.mark.parametrize("precision", ["bf16", "fp16"])
def test_packed_loop_equals_padded_at_valid_positions(precision, case, noise):
    import seqdiff_b200 as sd
    SM = sd.structure_model
    key, lm, rseq, rang, rm, x_T = _inputs(case)
    m = _model(*key, precision)
    T = 6
    args = _args(m, lm, rseq, rang, rm, x_T, T)
    kw = dict(seed=7, graph_id0=300)
    if noise == "explicit":
        kw["noise_steps"] = torch.randn(T, *x_T.shape, generator=torch.Generator().manual_seed(22))
    want = SM.p_sample_loop(**args, **kw)
    got = SM.p_sample_loop(**args, **kw, packed=True)
    _check_packed(got, want, lm)
    final = SM.p_sample_loop(**args, **kw, packed=True, keep_history=False)  # the final tensor alone; a second packed call, same ids
    assert torch.equal(final[0], got[-1])
    assert torch.equal(SM.p_sample_loop(**args, **kw, packed=True), got)


@pytest.mark.parametrize("why", ["mask with a hole", "fp32"])
def test_unusable_packing_runs_the_padded_loop(why):
    """a mask that is not a prefix of ones, or fp32 mode: packed=True is the padded loop, padded positions included"""
    import seqdiff_b200 as sd
    SM = sd.structure_model
    key, lm, rseq, rang, rm, x_T = _inputs("len1")
    precision = "fp32" if why == "fp32" else "bf16"
    if why == "mask with a hole":
        lm = lm.clone()
        lm[2, 10] = 0.0
    m = _model(*key, precision)
    args = _args(m, lm, rseq, rang, rm, x_T, 5)
    want = SM.p_sample_loop(**args, seed=3, graph_id0=0)
    got = SM.p_sample_loop(**args, seed=3, graph_id0=0, packed=True)
    assert torch.equal(got, want)
    assert (want[:, ~lm.bool()] != 0).any()  # the padded loop does compute the padded positions


def test_graph_cache_across_length_compositions():
    """Compositions A, B (same B and L), then A again: the lengths are part of the step graph's key, so each change re-captures and
    the return to A gives A's result.  A padded call after the packed ones equals a fresh padded call."""
    import seqdiff_b200 as sd
    SM = sd.structure_model
    key, lm_a, rseq, rang, rm, x_T = _inputs("absolute")
    lm_b = O.synthetic_batch(lm_a.shape[0], lm_a.shape[1], (3, 64), (10, 64), 23)["ligand_attn_mask"]
    assert not torch.equal(lm_a, lm_b)
    m = _model(*key, "bf16")
    kw = dict(seed=9, graph_id0=40)
    a_args, b_args = _args(m, lm_a, rseq, rang, rm, x_T, 5), _args(m, lm_b, rseq, rang, rm, x_T, 5)
    pad_a = SM.p_sample_loop(**a_args, **kw)
    pad_b = SM.p_sample_loop(**b_args, **kw)
    pk_a = SM.p_sample_loop(**a_args, **kw, packed=True)
    pk_b = SM.p_sample_loop(**b_args, **kw, packed=True)
    pk_a2 = SM.p_sample_loop(**a_args, **kw, packed=True)
    _check_packed(pk_a, pad_a, lm_a)
    _check_packed(pk_b, pad_b, lm_b)
    assert torch.equal(pk_a2, pk_a)
    assert torch.equal(SM.p_sample_loop(**a_args, **kw), pad_a)


def test_packed_noise_stream():
    """graph_id0 = None continues the process-wide Philox stream (fresh noise per call); an explicit (seed, graph_id0) reproduces"""
    import seqdiff_b200 as sd
    SM = sd.structure_model
    key, lm, rseq, rang, rm, x_T = _inputs("len1")
    m = _model(*key, "bf16")
    args = _args(m, lm, rseq, rang, rm, x_T, 4)
    valid = lm.bool()
    e1 = SM.p_sample_loop(**args, seed=5, packed=True, keep_history=False)[0]
    e2 = SM.p_sample_loop(**args, seed=5, packed=True, keep_history=False)[0]
    assert not torch.equal(e1[valid], e2[valid])
    r1 = SM.p_sample_loop(**args, seed=5, graph_id0=77, packed=True, keep_history=False)
    r2 = SM.p_sample_loop(**args, seed=5, graph_id0=77, packed=True, keep_history=False)
    assert torch.equal(r1, r2)
    assert not torch.equal(SM.p_sample_loop(**args, seed=6, graph_id0=77, packed=True, keep_history=False), r1)


def test_sample_driver_packed_returns_the_padded_arrays():
    """structure_model.sample(..., packed=True): the same list of per-complex arrays, trimmed to the ligand length, bit for bit"""
    import seqdiff_b200 as sd
    SM = sd.structure_model
    key = (64, 2, True)
    m = _model(*key, "bf16")
    T, n = 4, 7
    b = O.synthetic_batch(n, 64, (1, 64), (16, 64), 24)

    class DS:
        timesteps = T
        alpha_beta_terms = {"betas": SM.cosine_beta_schedule(T)}

        def __len__(self):
            return n

        def __getitem__(self, i):
            return {"ligand_attn_mask": b["ligand_attn_mask"][i], "ligand_angles": b["ligand_angles"][i],
                    "receptor_angles": b["receptor_angles"][i], "receptor_seq": b["receptor_seq"][i],
                    "receptor_attn_mask": b["receptor_attn_mask"][i]}

        def sample_noise(self, v):
            return SM.modulo_with_wrapped_range(torch.randn(v.shape, generator=torch.Generator().manual_seed(25)))

    old = SM.CONFIG["batch_size"]
    SM.CONFIG["batch_size"] = 3
    try:
        want = SM.sample(m, DS(), first_batch_only=False, seed=2, graph_id0=0)
        got = SM.sample(m, DS(), first_batch_only=False, seed=2, graph_id0=0, packed=True)
    finally:
        SM.CONFIG["batch_size"] = old
    assert len(got) == len(want) == n
    for g_, w_ in zip(got, want):
        assert g_.shape == w_.shape and g_.tobytes() == w_.tobytes()
