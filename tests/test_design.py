"""design(): P pockets x K1 backbones (structure sampler) x K2 sequences per backbone (sequence sampler), handed over on the device.
It must equal, bit for bit, the host composition it replaces: p_sample_loop on the batch with every pocket repeated K1 times, the
trim of structure_model.sample(), load_generated_angles' zero pad, then denoise on the batch with every (pocket, backbone) repeated
K2 times -- with the same start states, seeds and graph ids."""
import pytest
import torch

from helpers import O, make_model, sd_pkg
from oracle import structdiff_oracle as S

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
LS, LQ = 64, 96  # structure model positions; sequence batch length (the hand-off pads Ls -> Lq)

_M = {}


def _models(precision):
    sd = sd_pkg()
    if not _M:
        cfg = S.OracleConfig(max_position_embeddings=LS, num_hidden_layers=2, feature_size=8, relative_key=True)
        common = dict(max_position_embeddings=LS, num_attention_heads=cfg.num_attention_heads, hidden_size=cfg.hidden_size,
                      intermediate_size=cfg.intermediate_size, num_hidden_layers=2, position_embedding_type="relative_key")
        st = sd.structure_model.ConditionalBertForDiffusionBase(sd.BertConfig(**common),
                                                                sd.BertConfig(**common, is_decoder=True, add_cross_attention=True), 8)
        st.load_state_dict(S.init_struct_state_dict(cfg, 61), strict=True)
        _M["struct"] = st.eval().to(DEV)
        qcfg = O.OracleConfig(max_position_embeddings=128, relative_key=True)
        _M["seq"] = make_model(sd, qcfg, O.init_state_dict(qcfg, 1, "B"), precision)
    _M["struct"].precision = _M["seq"].precision = precision
    return _M["struct"], _M["seq"]


def _batch(P, seed):
    b = O.synthetic_batch(P, LQ, (1, LS), (16, LS), seed)
    b["structure_ids"] = {"pdb_id": [f"{i}abc" for i in range(P)], "ligand_chain": ["A"] * P}
    return b


def _rep(batch, K):
    out = {k: v.repeat_interleave(K, dim=0) for k, v in batch.items() if torch.is_tensor(v)}
    out["structure_ids"] = {k: [x for x in v for _ in range(K)] for k, v in batch["structure_ids"].items()}
    return out


def _setup(P, K1, K2, T, seed):
    sd = sd_pkg()
    SM = sd.structure_model
    batch = _batch(P, seed)
    g = torch.Generator().manual_seed(seed + 1)
    x_T = SM.modulo_with_wrapped_range(torch.randn(P * K1, LS, 8, generator=g))
    seq_x_T = O.generate_discrete_noise(P * K1 * K2, LQ, generator=g)
    kw = dict(struct_betas=SM.cosine_beta_schedule(T), noise_schedule=sd.PredefinedNoiseScheduleDiscrete("cosine", T),
              transition=sd.DiscreteUniformTransition(20), timesteps=T, x_T=x_T, seq_x_T=seq_x_T, seed=9, graph_id0=300,
              seq_graph_id0=7000)
    return batch, kw


@pytest.mark.parametrize("precision,packed", [("bf16", True), ("bf16", False), ("fp16", True), ("fp32", False)])
def test_design_equals_host_composition(precision, packed):
    sd = sd_pkg()
    SM = sd.structure_model
    st, sq = _models(precision)
    sd.sample.DEVICE = torch.device(DEV)
    P, K1, K2, T = 3, 2, 3, 4
    batch, kw = _setup(P, K1, K2, T, 51)
    backbones, final = sd.design.design_tensors(st, sq, batch, K1, K2, packed=packed, **kw)
    ids, bb, bb_angles, true_seqs, pred_seqs, rates = sd.design.design(st, sq, batch, K1, K2, packed=packed, **kw)

    # the host composition: structure sampling of the replicated batch, sample()'s trim, load_generated_angles, denoise
    sb = _rep(batch, K1)
    hist = SM.p_sample_loop(st, sb["ligand_attn_mask"][:, :LS], kw["x_T"], sb["receptor_seq"][:, :LS], sb["receptor_attn_mask"][:, :LS],
                            sb["receptor_angles"][:, :LS], T, kw["struct_betas"], seed=9, graph_id0=300, packed=packed)
    lens = sb["ligand_attn_mask"].sum(dim=1).int()
    trimmed = [hist[-1, i, :int(l)].numpy() for i, l in enumerate(lens)]
    generated = sd.load_generated_angles(trimmed, max_seq_len=LQ, batch_size=P * K1)[0]
    qb = _rep(batch, K1 * K2)
    qb["ligand_angles"] = generated.repeat_interleave(K2, dim=0)
    dkw = dict(timesteps=T, x_T=kw["seq_x_T"], seed=9, graph_id0=7000, packed=packed)
    want_final = sd.denoise_tensors(qb, sq, kw["noise_schedule"], kw["transition"], True, **dkw)
    want = sd.denoise(qb, sq, kw["noise_schedule"], kw["transition"], True, **dkw)

    assert torch.equal(backbones.cpu(), generated)
    assert torch.equal(final, want_final)
    assert (ids, true_seqs, pred_seqs, rates) == tuple(want)
    n = P * K1 * K2
    assert len(ids) == n and bb == [(i // K2) % K1 for i in range(n)]
    assert all(a.tobytes() == trimmed[i // K2].tobytes() for i, a in enumerate(bb_angles))
    assert ids[0] == "0abc_A" and ids[-1] == f"{P - 1}abc_A"


def test_packed_and_padded_design_give_the_same_sequences():
    sd = sd_pkg()
    st, sq = _models("bf16")
    batch, kw = _setup(4, 2, 2, 4, 52)
    packed = sd.design.design(st, sq, batch, 2, 2, packed=True, **kw)
    padded = sd.design.design(st, sq, batch, 2, 2, packed=False, **kw)
    assert packed[4] == padded[4] and packed[5] == padded[5]
    assert all(a.tobytes() == b.tobytes() for a, b in zip(packed[2], padded[2]))


def test_single_pocket_and_default_noise():
    """P = 1 with the default start states and graph ids (drawn from the process-wide stream): the shapes and the order hold, and two
    calls draw different backbones"""
    sd = sd_pkg()
    st, sq = _models("bf16")
    batch = _batch(1, 53)
    kw = dict(struct_timesteps=4, timesteps=4)
    b1, f1 = sd.design.design_tensors(st, sq, batch, 3, 2, **kw)
    b2, _ = sd.design.design_tensors(st, sq, batch, 3, 2, **kw)
    assert b1.shape == (3, LQ, 8) and f1.shape == (6, LQ, 20)
    assert not torch.equal(b1, b2)
    L = int(batch["ligand_attn_mask"].sum())
    assert (b1[:, L:] == 0).all()
    ids, bb, angles, _, pred, _ = sd.design.design(st, sq, batch, 3, 2, **kw)
    assert ids == ["0abc_A"] * 6 and bb == [0, 0, 1, 1, 2, 2] and all(len(p) == L for p in pred) and angles[0].shape == (L, 8)
