"""CPU tests of the backbone score: the oracle's definition (tests/struct_score_oracle.py), the argument checks of
structure_model.score_backbones_tensors -- all made before any device work, there is no CPU path to fall back to --, the C ABI's own
checks and the design_dataset(score_backbones=True) columns."""
import ctypes
import math
import os

import pytest
import torch

import struct_score_oracle as SSO
import struct_train_oracle as STO
from helpers import O, ROOT
from oracle import structdiff_oracle as S

FS = 8


def _complexes(B, L, seed):
    b = O.synthetic_batch(B, L, (3, L), (4, L), seed)
    g = torch.Generator().manual_seed(seed + 1)
    x0 = S.modulo_with_wrapped_range(torch.randn(B, L, FS, generator=g) * 2)
    return x0, b["ligand_attn_mask"], b["receptor_seq"], b["receptor_angles"], b["receptor_attn_mask"], g


def test_perfect_denoiser_scores_zero():
    T, B, L = 12, 3, 16
    x0, lm, rs, ra, rm, g = _complexes(B, L, 3)
    noise = torch.randn(T, B, L, FS, generator=g)
    terms = SSO.score_loop(None, None, x0, lm, rs, ra, rm, S.cosine_beta_schedule(T), noise, forward=lambda k, x_k: noise[k])
    assert torch.equal(terms, torch.zeros_like(terms))
    # and a wrong prediction scores > 0 at the valid positions only
    terms = SSO.score_loop(None, None, x0, lm, rs, ra, rm, S.cosine_beta_schedule(T), noise, forward=lambda k, x_k: x_k)
    valid = (lm != 0)[..., None].expand_as(terms)
    assert (terms[valid] > 0).all() and (terms[~valid] == 0).all()


def test_one_step_equals_the_training_loss_on_the_q_sampled_batch():
    """T = 1: the score of each backbone is angle_loss (the training objective) of the prediction on x_0 = the training q-sample at t = 0"""
    B, L = 4, 20
    x0, lm, rs, ra, rm, g = _complexes(B, L, 5)
    eps = torch.randn(1, B, L, FS, generator=g)
    pred = torch.randn(B, L, FS, generator=g)
    seen = {}

    def fwd(k, x_k):
        seen[k] = x_k
        return pred
    betas = S.cosine_beta_schedule(1)
    terms = SSO.score_loop(None, None, x0, lm, rs, ra, rm, betas, eps, forward=fwd)
    loss, per_feature = SSO.backbone_loss(terms, lm, 1)
    ab = S.compute_alphas(betas)
    t = torch.zeros(B, dtype=torch.long)
    corrupted = S.modulo_with_wrapped_range(ab["sqrt_alphas_cumprod"][t][:, None, None] * x0 + ab["sqrt_one_minus_alphas_cumprod"][t][:, None, None] * eps[0])
    assert torch.equal(seen[0], corrupted)
    for b in range(B):
        want, want_pf = STO.angle_loss(pred[b:b + 1].double(), eps[0, b:b + 1].double(), lm[b:b + 1])
        assert torch.allclose(per_feature[b], want_pf, rtol=1e-6, atol=0) and abs(loss[b].item() - want.item()) < 1e-6 * want.item()


@pytest.mark.parametrize("k", [0, 1, 24, 49])
def test_in_loop_q_sample_is_the_training_q_sample(k):
    T, B, L = 50, 3, 12
    x0, *_, g = _complexes(B, L, 9)
    eps = torch.randn(B, L, FS, generator=g)
    ab = S.compute_alphas(S.cosine_beta_schedule(T))
    t = torch.full((B,), k, dtype=torch.long)
    want = S.modulo_with_wrapped_range(ab["sqrt_alphas_cumprod"][t][:, None, None] * x0 + ab["sqrt_one_minus_alphas_cumprod"][t][:, None, None] * eps)
    assert torch.equal(SSO.q_sample(x0, SSO.qs_table(S.cosine_beta_schedule(T))[k], eps), want)


def test_host_table_is_the_oracle_table():
    import seqdiff_b200 as sd
    betas = S.cosine_beta_schedule(37)
    assert torch.equal(sd.structure_model.qsample_coefficients(betas), SSO.qs_table(betas))


class _StubModel:
    """a structure model whose every use beyond feature_size means the checks let the call through to the device"""
    feature_size = FS

    def __getattr__(self, name):
        raise AssertionError(f"model.{name} used before the arguments were checked")


def _args(P=2, K=1, L=10, T=4):
    x0, lm, rs, ra, rm, _ = _complexes(P * K, L, 17)
    return dict(model=_StubModel(), ligand_mask=lm, backbones=x0, receptor_seq=rs[:P], receptor_mask=rm[:P], receptor_angle=ra[:P],
                total_timesteps=T, betas=S.cosine_beta_schedule(T))


@pytest.mark.parametrize("why", ["backbone shape", "feature count", "ligand mask shape", "receptor shape", "receptor angle shape",
                                 "receptor mask shape", "betas length", "betas 2-d", "noise shape", "no valid position", "nan at padding",
                                 "inf", "zero steps", "sample count"])
def test_bad_inputs_raise_before_any_c_call(why, monkeypatch):
    import seqdiff_b200 as sd
    SM = sd.structure_model

    def no_lib():
        raise AssertionError("the C library was reached")
    monkeypatch.setattr(sd._cabi, "lib", no_lib)
    a, kw = _args(), {}
    if why == "backbone shape":
        a["backbones"] = a["backbones"][:, :5]
    elif why == "feature count":
        a["backbones"] = a["backbones"][..., :4]
    elif why == "ligand mask shape":
        a["ligand_mask"] = a["ligand_mask"][:1]
    elif why == "receptor shape":
        a["receptor_seq"] = a["receptor_seq"][:1]
    elif why == "receptor angle shape":
        a["receptor_angle"] = a["receptor_angle"][..., :4]
    elif why == "receptor mask shape":
        a["receptor_mask"] = a["receptor_mask"][:, :3]
    elif why == "betas length":
        a["betas"] = S.cosine_beta_schedule(5)
    elif why == "betas 2-d":
        a["betas"] = S.cosine_beta_schedule(4)[None]
    elif why == "noise shape":
        kw["noise_steps"] = torch.zeros(4, 2, 10, 4)
    elif why == "no valid position":
        a["ligand_mask"] = a["ligand_mask"].clone()
        a["ligand_mask"][1] = 0
    elif why == "nan at padding":
        a["backbones"] = a["backbones"].clone()
        b, l = (a["ligand_mask"] == 0).nonzero()[0].tolist()
        a["backbones"][b, l, 0] = float("nan")
    elif why == "inf":
        a["backbones"] = a["backbones"].clone()
        a["backbones"][1, 0, 3] = float("inf")
    elif why == "zero steps":
        a["total_timesteps"], a["betas"] = 0, S.cosine_beta_schedule(4)[:0]
    else:
        kw["num_samples"] = 2  # backbones hold P, not P*K, graphs
    with pytest.raises(ValueError):
        SM.score_backbones_tensors(**a, **kw)
    with pytest.raises(ValueError):
        SM.score_backbones(**a, **kw)


@pytest.mark.parametrize("k", [0, -1, 1.5, True])
def test_bad_sample_counts_raise(k):
    import seqdiff_b200 as sd
    with pytest.raises(ValueError, match="num_samples"):
        sd.structure_model.score_backbones_tensors(**_args(), num_samples=k)


def test_per_pocket_ligand_mask_is_accepted_by_the_checks(monkeypatch):
    """[P, L] ligand mask with K = 2: the checks pass and the call proceeds to the handle"""
    import seqdiff_b200 as sd
    a = _args(P=2, K=2)
    a["ligand_mask"] = a["ligand_mask"][:2]
    with pytest.raises(AssertionError, match="_sync_handle"):
        sd.structure_model.score_backbones_tensors(**a, num_samples=2)


def test_abi_symbol_is_declared():
    import seqdiff_b200 as sd
    with open(os.path.join(ROOT, "include", "seqdiff_b200.h")) as f:
        header = f.read()
    assert "SEQDIFF_API int seqdiff_struct_score_multi(" in header and "not a likelihood" in header
    assert "seqdiff_struct_score_multi" in sd._cabi.PROTOTYPES


def test_c_abi_rejects_bad_sizes_and_flags():
    """seqdiff_struct_score_multi checks its sizes and flags before it touches the handle (a stand-in pointer is never dereferenced)"""
    import seqdiff_b200 as sd
    lib = sd.lib()
    buf = ctypes.create_string_buffer(64)
    p = ctypes.cast(buf, ctypes.c_void_p)
    for P, K, Ll, Lr, T, flags in ((0, 1, 8, 8, 5, 0), (1, 0, 8, 8, 5, 0), (2, 2, 0, 8, 5, 0), (2, 2, 8, 8, 0, 0), (1 << 16, 1 << 10, 64, 128, 5, 0),
                                   (2, 3, 8, 8, 5, 2), (2, 3, 8, 8, 5, -1), (1 << 16, 1, 8, 8, 5, 0), (256, 256, 8, 8, 5, 0)):
        rc = lib.seqdiff_struct_score_multi(p, 1, P, K, Ll, Lr, T, p, p, p, p, p, p, None, 0, 0, flags, p, None)
        assert rc == 1, (P, K, Ll, T, flags)  # SEQDIFF_ERR_INVALID
        assert lib.seqdiff_last_error()


def _fake_design(struct_model, seq_model, batch, K1, K2, **kw):
    P = batch["ligand_seq"].shape[0]
    n = P * K1 * K2
    ids = [batch["structure_ids"]["pdb_id"][i // (K1 * K2)] for i in range(n)]
    angles = [f"b{i // K2}" for i in range(n)]  # one object per backbone, repeated over its sequences
    return ids, [(i // K2) % K1 for i in range(n)], angles, ["T"] * n, [f"s{i}" for i in range(n)], [0.5] * n


def test_design_dataset_backbone_column(monkeypatch):
    import seqdiff_b200 as sd
    P, K1, K2 = 2, 3, 2
    batch = O.synthetic_batch(P, 8, (2, 8), (2, 8), 1)
    batch["structure_ids"] = {"pdb_id": [f"p{i}" for i in range(P)], "ligand_chain": ["A"] * P}
    calls = []

    def fake_scorer(struct_model, batch_, K, backbone_angles, **kw):
        calls.append((K, list(backbone_angles), kw))
        return [100.0 + int(a[1:]) for a in backbone_angles]

    def fake_seq_scorer(seq_model, batch_, K, angles, pred_seqs, **kw):
        return [1.0] * len(pred_seqs), [2.0] * len(pred_seqs)
    monkeypatch.setattr(sd.design, "score_design_backbones", fake_scorer)
    monkeypatch.setattr(sd.design, "score_designs", fake_seq_scorer)
    betas = S.cosine_beta_schedule(7)
    plain = sd.design_dataset([batch], None, None, K1, K2, design_fn=_fake_design)
    assert list(plain.columns) == ["structure_ids", "true_sequence", "predict_sequence", "recovery_rate", "backbone"] and not calls
    df = sd.design_dataset([batch], None, None, K1, K2, design_fn=_fake_design, score_backbones=True, struct_betas=betas, seed=4, packed=False,
                           timesteps=9)
    assert list(df.columns) == list(plain.columns) + ["backbone_loss"]
    assert df[list(plain.columns)].equals(plain)
    assert list(df["backbone_loss"]) == [100.0 + i // K2 for i in range(P * K1 * K2)]
    assert len(calls) == 1 and calls[0][0] == K1 and calls[0][1] == [f"b{j}" for j in range(P * K1)]
    assert set(calls[0][2]) == {"struct_betas", "seed", "packed"} and calls[0][2]["struct_betas"] is betas
    both = sd.design_dataset([batch], None, None, K1, K2, design_fn=_fake_design, score=True, score_backbones=True)
    assert list(both.columns) == list(plain.columns) + ["nll_per_residue", "perplexity", "backbone_loss"]
    assert list(both["backbone_loss"]) == list(df["backbone_loss"])


def test_wrap_and_smooth_l1_have_one_device_definition():
    """wrap_angle and the smooth-L1 h live in common.cuh only, used by the sampler, the training loss and the backbone score"""
    src = os.path.join(ROOT, "e3-invaraint-diffusion-model_b200", "csrc")
    texts = {n: open(os.path.join(src, n)).read() for n in os.listdir(src) if n.endswith((".cu", ".cuh"))}
    defs = [n for n, t in texts.items() if "float wrap_angle(" in t or "float angle_smooth_l1(" in t or "kMin = -3.14159274" in t]
    assert defs == ["common.cuh"]
    assert "wrap_angle(" in texts["gauss_step.cu"] and "angle_smooth_l1(wrap_angle(" in texts["decode_loss.cu"]
    assert math.isclose(SSO.BETA, math.pi / 10)
