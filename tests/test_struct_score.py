"""The backbone score on the GPU (seqdiff_struct_score_multi through structure_model.score_backbones_tensors / score_backbones /
design_dataset(score_backbones=True)): fp32 parity with the oracle loop (tests/struct_score_oracle.py), the 16-bit modes against fp32,
the tie to the training path at T = 1, Philox reproducibility and shard invariance, K backbones per pocket and packing (bit for bit
against the replicated / padded batch, as for the sampler), isolation of the score's cached CUDA graph from the sampler's, and the
design column."""
import ctypes
import math

import pytest
import torch

import struct_score_oracle as SSO
from helpers import make_model
from oracle import seqdiff_oracle as O
from oracle import structdiff_oracle as S

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
FS = 8

_MODELS = {}


def _sd():
    import seqdiff_b200 as sd
    return sd


def _new_model(L):
    """(model with a handle of its own, oracle config, state dict): 2 + 2 layers, the structure tests' weights"""
    sd = _sd()
    cfg = S.OracleConfig(max_position_embeddings=L, num_hidden_layers=2, feature_size=FS, relative_key=True)
    common = dict(max_position_embeddings=L, num_attention_heads=cfg.num_attention_heads, hidden_size=cfg.hidden_size,
                  intermediate_size=cfg.intermediate_size, num_hidden_layers=2, position_embedding_type="relative_key")
    m = sd.structure_model.ConditionalBertForDiffusionBase(sd.BertConfig(**common),
                                                           sd.BertConfig(**common, is_decoder=True, add_cross_attention=True), FS)
    state = S.init_struct_state_dict(cfg, 61)
    m.load_state_dict(state, strict=True)
    return m.eval().to(DEV), cfg, state


def _model(L, precision):
    if L not in _MODELS:
        _MODELS[L] = _new_model(L)
    m = _MODELS[L][0]
    m.precision = precision
    return m


def _complexes(case, P, K, seed):
    """(model length, x0 [P*K, Ll, F], ligand mask [P*K, Ll], receptor seq / angles / mask of the P pockets)"""
    g = torch.Generator().manual_seed(seed)
    if case == "Ll==Lr":
        L, Ll, Lr = 64, 64, 64
        lm = O.synthetic_batch(P * K, Ll, (5, 64), (16, 64), seed)["ligand_attn_mask"]
        rm = O.synthetic_batch(P, Lr, (5, 64), (16, 64), seed + 1)["receptor_attn_mask"]
    else:
        L, Ll, Lr = 96, 40, 96
        lm = O.synthetic_batch(P * K, Ll, (1, 40), (1, 40), seed)["ligand_attn_mask"]
        rm = O.synthetic_batch(P, Lr, (1, 96), (16, 96), seed + 1)["receptor_attn_mask"]
    rseq = torch.nn.functional.one_hot(torch.randint(0, 20, (P, Lr), generator=g), 20).float() * rm[..., None]
    rang = ((torch.rand(P, Lr, FS, generator=g) * 2 - 1) * math.pi) * rm[..., None]
    x0 = (torch.rand(P * K, Ll, FS, generator=g) * 2 - 1) * math.pi
    return L, x0, lm, rseq, rang, rm


def _score(m, x0, lm, rseq, rang, rm, T, K=1, tensors=True, **kw):
    SM = _sd().structure_model
    fn = SM.score_backbones_tensors if tensors else SM.score_backbones
    return fn(m, lm.to(DEV), x0.to(DEV), rseq.to(DEV), rm.to(DEV), rang.to(DEV), T, SM.cosine_beta_schedule(T), num_samples=K, **kw)


def _noise(T, x0, seed):
    return torch.randn(T, *x0.shape, generator=torch.Generator().manual_seed(seed))


@pytest.mark.parametrize("T,case", [(5, "Ll==Lr"), (5, "Ll!=Lr"), (50, "Ll==Lr")])
def test_fp32_terms_match_the_oracle(T, case):
    B = 2
    L, x0, lm, rseq, rang, rm = _complexes(case, B, 1, 70 + T)
    m = _model(L, "fp32")
    _, cfg, state = _MODELS[L]
    eps = _noise(T, x0, 3)
    got = _score(m, x0, lm, rseq, rang, rm, T, noise_steps=eps, seed=1, graph_id0=0).cpu()
    with torch.no_grad():
        want = SSO.score_loop(state, cfg, x0, lm, rseq, rang, rm, S.cosine_beta_schedule(T), eps)
    d = (got - want).abs().max().item()
    loss, _ = SSO.backbone_loss(got, lm, T)
    want_loss, _ = SSO.backbone_loss(want, lm, T)
    print(f"struct score parity T={T} {case}: max |d terms| {d:.3e} (terms up to {want.abs().max().item():.2f}), "
          f"max |d loss| {(loss - want_loss).abs().max().item():.3e}")
    assert d < T * 5e-6  # h is 1-Lipschitz, so T x the forward's error bounds it; measured on a B200: 2.6e-6 x T at T = 5, 1.2e-6 x T at T = 50
    assert (got[lm == 0] == 0).all()


@pytest.mark.parametrize("precision,tol", [("bf16", 2e-3), ("fp16", 5e-4)])  # measured on a B200: 6.6e-4 / 1.2e-4
def test_16bit_loss_against_fp32(precision, tol):
    T, P = 50, 8
    L, x0, lm, rseq, rang, rm = _complexes("Ll==Lr", P, 1, 41)
    eps = _noise(T, x0, 4)
    kw = dict(noise_steps=eps, seed=2, graph_id0=0, tensors=False)
    ref, _ = _score(_model(L, "fp32"), x0, lm, rseq, rang, rm, T, **kw)
    worst = 0.0
    for packed in (False, True):
        got, _ = _score(_model(L, precision), x0, lm, rseq, rang, rm, T, packed=packed, **kw)
        worst = max(worst, ((got - ref).abs() / ref.abs()).max().item())
    print(f"struct score {precision}: worst relative backbone-loss deviation from fp32 {worst:.3e} "
          f"(loss {ref.min().item():.4f} .. {ref.max().item():.4f})")
    assert worst < tol


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_one_step_equals_the_training_loss_terms(precision):
    """T = 1 under explicit noise: the in-loop q-sample and forward are the training path's -- per feature, the summed terms equal
    angle_loss_terms(model.forward(0, host q-sample, ...)) to 1e-12 relative"""
    sd = _sd()
    SM = sd.structure_model
    B = 4
    L, x0, lm, rseq, rang, rm = _complexes("Ll==Lr", B, 1, 43)
    m = _model(L, precision)
    eps = _noise(1, x0, 5)
    terms = _score(m, x0, lm, rseq, rang, rm, 1, noise_steps=eps, seed=0, graph_id0=0)
    x_0 = SSO.q_sample(x0, SM.qsample_coefficients(SM.cosine_beta_schedule(1))[0], eps[0])
    with torch.no_grad():
        pred = m(torch.zeros(B, dtype=torch.long, device=DEV), x_0.to(DEV), lm.to(DEV), rseq.to(DEV), rang.to(DEV), rm.to(DEV))
    ref = SM.angle_loss_terms(pred, eps[0].to(DEV), lm.to(DEV)).cpu()
    got = terms.sum(dim=(0, 1)).cpu()
    rel = ((got - ref[:FS]).abs() / ref[:FS].abs()).max().item()
    print(f"struct score T=1 {precision}: max relative deviation from angle_loss_terms {rel:.3e}")
    assert rel < 1e-12 and ref[FS].item() == float((lm != 0).sum())


def test_philox_reproducible_shard_invariant_and_fresh_by_default():
    T, P = 8, 6
    L, x0, lm, rseq, rang, rm = _complexes("Ll==Lr", P, 1, 45)
    m = _model(L, "bf16")
    kw = dict(seed=77, packed=True)
    a = _score(m, x0, lm, rseq, rang, rm, T, graph_id0=500, **kw).clone()
    assert torch.equal(a, _score(m, x0, lm, rseq, rang, rm, T, graph_id0=500, **kw))
    assert not torch.equal(a, _score(m, x0, lm, rseq, rang, rm, T, graph_id0=501, **kw))
    halves = [_score(m, x0[lo:hi], lm[lo:hi], rseq[lo:hi], rang[lo:hi], rm[lo:hi], T, graph_id0=500 + lo, **kw).clone()
              for lo, hi in ((0, 2), (2, 6))]
    assert torch.equal(torch.cat(halves), a)
    c = _score(m, x0, lm, rseq, rang, rm, T, graph_id0=None, **kw).clone()
    d = _score(m, x0, lm, rseq, rang, rm, T, graph_id0=None, **kw).clone()
    assert not torch.equal(c, d)  # fresh draws from the process-wide graph-id stream


@pytest.mark.parametrize("precision,packed", [("bf16", False), ("bf16", True), ("fp16", False), ("fp16", True), ("fp32", False)])
def test_backbones_per_pocket_equal_the_replicated_batch(precision, packed):
    T, P, K = 5, 3, 3
    L, x0, lm, rseq, rang, rm = _complexes("Ll!=Lr", P, K, 47)
    m = _model(L, precision)
    r = lambda t: t.repeat_interleave(K, dim=0)  # noqa: E731
    for eps in (None, _noise(T, x0, 7)):
        kw = dict(noise_steps=eps, seed=5, graph_id0=900, packed=packed)
        got = _score(m, x0, lm, rseq, rang, rm, T, K=K, **kw).clone()
        want = _score(m, x0, lm, r(rseq), r(rang), r(rm), T, **kw)
        assert torch.equal(got, want)


@pytest.mark.parametrize("precision", ["bf16", "fp16"])
def test_packed_equals_padded(precision):
    T, P = 6, 5
    L, x0, lm, rseq, rang, rm = _complexes("Ll==Lr", P, 1, 49)
    m = _model(L, precision)
    valid = (lm != 0).to(DEV)
    for eps in (None, _noise(T, x0, 8)):
        kw = dict(noise_steps=eps, seed=3, graph_id0=40)
        packed = _score(m, x0, lm, rseq, rang, rm, T, packed=True, **kw).clone()
        padded = _score(m, x0, lm, rseq, rang, rm, T, packed=False, **kw)
        assert torch.equal(packed[valid], padded[valid])
        assert (packed[~valid] == 0).all() and (padded[~valid] == 0).all()


def test_score_and_sample_keep_their_own_graphs():
    """sample -> score -> sample -> score -> sample on one handle with explicit ids: every call reproduces the first call of its kind bit
    for bit, and after the first call of each kind neither re-captures (the step graphs are cached side by side)"""
    sd = _sd()
    SM = sd.structure_model
    T, P = 6, 4
    L, x0, lm, rseq, rang, rm = _complexes("Ll==Lr", P, 1, 51)
    m = _model(L, "bf16")
    lib = sd.lib()

    def run(kind):
        torch.cuda.synchronize()
        n0 = lib.seqdiff_launch_count()
        if kind == "sample":
            out = SM.p_sample_loop_tensors(m, lm.to(DEV), x0.to(DEV), rseq.to(DEV), rm.to(DEV), rang.to(DEV), T, SM.cosine_beta_schedule(T),
                                           seed=4, graph_id0=60, keep_history=False, packed=True)[1].clone()
        else:
            out = _score(m, x0, lm, rseq, rang, rm, T, seed=4, graph_id0=60, packed=True).clone()
        torch.cuda.synchronize()
        return out, lib.seqdiff_launch_count() - n0

    seq = ["sample", "score", "sample", "score", "sample"]
    res = [run(k) for k in seq]
    for i, k in enumerate(seq):
        assert torch.equal(res[i][0], res[seq.index(k)][0]), (i, k)
    # a capture adds the un-captured ligand-branch dry run; a replay launches the arm kernel, the receptor branch and T x the graph's nodes
    assert res[2][1] < res[0][1] and res[4][1] == res[2][1], [r[1] for r in res]
    assert res[3][1] < res[1][1], [r[1] for r in res]
    print(f"struct score / sample launches per call (capture, replay): score {res[1][1]}, {res[3][1]}; sample {res[0][1]}, {res[2][1]}")


@pytest.mark.parametrize("packed", [False, True])
def test_cached_graph_serves_every_timestep_count(packed):
    """one batch scored at T = 10, 50, 10, 50 on one handle under Philox noise (no per-call pointer in the graph key): the q-sample table
    follows the fp64 sums in the score's block, so the cached step graph is valid for any T.  Every call equals the first call of its T
    on that handle and the first call on a fresh handle, bit for bit"""
    P = 4
    L, x0, lm, rseq, rang, rm = _complexes("Ll==Lr", P, 1, 57)
    m = _model(L, "bf16")
    kw = dict(seed=11, graph_id0=70, packed=packed)
    got = [_score(m, x0, lm, rseq, rang, rm, T, **kw).clone() for T in (10, 50, 10, 50)]
    for T, i in ((10, 0), (50, 1)):
        fresh, _, _ = _new_model(L)
        fresh.precision = "bf16"
        want = _score(fresh, x0, lm, rseq, rang, rm, T, **kw)
        fresh.release()
        assert torch.equal(got[i], want) and torch.equal(got[i + 2], want), T
    assert not torch.equal(got[0], got[1])


def test_sequence_handle_is_rejected():
    sd = _sd()
    cfg = O.OracleConfig(max_position_embeddings=32, num_hidden_layers=1)
    seq = make_model(sd, cfg, O.init_state_dict(cfg, 1, "B"), "bf16")
    h = seq._sync_handle()
    buf = torch.zeros(4096, device=DEV)
    p = ctypes.c_void_p(buf.data_ptr())
    rc = sd.lib().seqdiff_struct_score_multi(h, 1, 1, 1, 8, 8, 2, p, p, p, p, p, p, None, 0, 0, 0, p, None)
    assert rc == 1 and b"sequence model" in sd.lib().seqdiff_last_error()


def test_design_column_equals_score_backbones():
    sd = _sd()
    SM = sd.structure_model
    LS, LQ = 64, 96
    st = _model(LS, "bf16")
    cfg = O.OracleConfig(max_position_embeddings=128, relative_key=True)
    sq = make_model(sd, cfg, O.init_state_dict(cfg, 1, "B"), "bf16")
    P, K1, K2, T = 2, 2, 2, 4
    batch = O.synthetic_batch(P, LQ, (1, LS), (16, LS), 55)
    batch["structure_ids"] = {"pdb_id": [f"{i}abc" for i in range(P)], "ligand_chain": ["A"] * P}
    g = torch.Generator().manual_seed(56)
    betas = SM.cosine_beta_schedule(T)
    kw = dict(struct_betas=betas, timesteps=T, x_T=SM.modulo_with_wrapped_range(torch.randn(P * K1, LS, FS, generator=g)),
              seq_x_T=O.generate_discrete_noise(P * K1 * K2, LQ, generator=g), seed=9, graph_id0=300, seq_graph_id0=7000)
    plain = sd.design_dataset([batch], st, sq, K1, K2, **kw)
    sd._cabi.GRAPH_IDS.reset(123456)
    df = sd.design_dataset([batch], st, sq, K1, K2, score_backbones=True, **kw)
    assert list(df.columns) == list(plain.columns) + ["backbone_loss"]
    assert df[list(plain.columns)].equals(plain)
    # host composition: the design's own backbones (0 beyond each ligand length) scored under their pockets
    backbones, _ = sd.design.design_tensors(st, sq, batch, K1, K2, **kw)
    _, inputs = sd.design.structure_inputs(batch, LS)
    loss, _ = SM.score_backbones(st, inputs["ligand_attn_mask"], backbones[:, :LS].cpu(), inputs["receptor_seq"], inputs["receptor_attn_mask"],
                                 inputs["receptor_angles"], T, betas, seed=9, graph_id0=123456, packed=True, num_samples=K1)
    assert list(df["backbone_loss"]) == [float(loss[i // K2]) for i in range(P * K1 * K2)]
    order = sorted(range(P * K1), key=lambda b: float(loss[b]))
    print(f"design backbone_loss: {[round(float(v), 4) for v in loss]} (ranking {order})")
