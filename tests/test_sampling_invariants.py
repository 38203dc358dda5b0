"""The sampling loop (seqdiff_sample) computes the work that gives the same result at every step once per sampling, before the
replayed step graph: the receptor embedding, the receptor half of ligand_feature_emb's attention sublayer, the timestep features of
steps 0..T-1 and decoder_normalize's modulation table.  The stand-alone forward() still computes everything.  Every hoisted value
comes from the same kernels and the same inputs (no split-K GEMM, attention items per (graph, head)), so the loop's final logits --
and with them every sampled index before them -- must be bit-identical to the same steps issued one by one through forward() and
the single reverse step."""
import pytest
import torch

from helpers import O, make_model, sd_pkg

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

_MODEL = {}


def _model(precision):
    if not _MODEL:
        # variant "B": decoder_normalize is not the identity the reference init makes it, so a wrong modulation row shows
        cfg = O.OracleConfig(max_position_embeddings=128, relative_key=True)
        _MODEL["m"] = make_model(sd_pkg(), cfg, O.init_state_dict(cfg, 1, "B"), precision)
    m = _MODEL["m"]
    m.precision = precision
    return m


def _batch(case, seed):
    if case == "Ll==Lr":  # the stand-alone forward runs ligand_feature_emb's attention as one stacked segment of 2B graphs
        return O.synthetic_batch(4, 64, (5, 40), (16, 64), seed)
    B = 3
    batch = O.synthetic_batch(B, 48, (1, 48), (1, 48), seed)
    rec = O.synthetic_batch(B, 112, (1, 112), (16, 112), seed + 1)
    for k in ("receptor_seq", "receptor_angles", "receptor_attn_mask"):
        batch[k] = rec[k]
    return batch


def _stepwise(sd, m, batch, x_T, E, T, sched, tr):
    """the loop's steps one by one: stand-alone forward() (t as a [B, 1] tensor) + the single reverse step with the same noise"""
    B = x_T.shape[0]
    dv = {k: v.to(DEV) for k, v in batch.items()}
    x = x_T.to(DEV)
    for s_int in reversed(range(T)):
        s = s_int * torch.ones((B, 1))
        with torch.no_grad():
            lg = m(s.to(DEV), x, dv["ligand_angles"], dv["ligand_attn_mask"], dv["receptor_seq"], dv["receptor_angles"], dv["receptor_attn_mask"])
        x = sd.sample_p_zs_given_zt_discrete((s + 1) / T, s / T, x, lg, sched, tr, True, s_int == 0, noise_E=E[s_int])
    return x


def _check(final, want, batch, packed):
    if not packed:
        assert torch.equal(final, want)
        return
    valid = batch["ligand_attn_mask"].bool().to(DEV)
    assert torch.equal(final[valid], want[valid])
    assert (final[~valid] == 0).all()


@pytest.mark.parametrize("case", ["Ll==Lr", "Ll!=Lr"])
@pytest.mark.parametrize("precision,packed", [("bf16", False), ("bf16", True), ("fp16", False), ("fp16", True), ("fp32", False)])
def test_loop_with_hoisted_invariants_equals_stepwise_forward(case, precision, packed):
    sd = sd_pkg()
    m = _model(precision)
    sd.sample.DEVICE = torch.device(DEV)
    T = 5
    batch = _batch(case, 51)
    B, Ll = batch["ligand_seq"].shape[:2]
    g = torch.Generator().manual_seed(3)
    x_T = O.generate_discrete_noise(B, Ll, generator=g)
    E = torch.empty(T, B * Ll, 20).exponential_(1, generator=g)
    sched, tr = sd.PredefinedNoiseScheduleDiscrete("cosine", T), sd.BlosumTransition(x_classes=20)
    final = sd.denoise_tensors(batch, m, sched, tr, True, timesteps=T, x_T=x_T, noise_E_steps=E, packed=packed)
    want = _stepwise(sd, m, batch, x_T, E, T, sched, tr)
    _check(final, want, batch, packed)


@pytest.mark.parametrize("packed", [False, True])
def test_cached_graph_with_new_receptor_and_fewer_steps(packed):
    """Two samplings with the same shapes but other receptor inputs and another T: the second replays the graph the first
    captured (the invariants are recomputed by every call, outside the graph), and each equals its own stepwise reference."""
    sd = sd_pkg()
    m = _model("bf16")
    sd.sample.DEVICE = torch.device(DEV)
    tr = sd.BlosumTransition(x_classes=20)
    first, other = _batch("Ll==Lr", 61), _batch("Ll==Lr", 62)
    # new receptor residues and angles; same masks (packed mode keys its graph on the lengths)
    second = dict(first, receptor_seq=other["receptor_seq"], receptor_angles=other["receptor_angles"])
    B, Ll = first["ligand_seq"].shape[:2]
    g = torch.Generator().manual_seed(4)
    x_T = O.generate_discrete_noise(B, Ll, generator=g)
    # the noise tensor's address is part of the graph key: every call takes a prefix of one device buffer, refilled per call
    E_dev = torch.empty(6, B * Ll, 20, device=DEV)
    runs = []
    for batch, T in ((first, 6), (second, 4), (second, 4)):
        E_dev.copy_(torch.empty(6, B * Ll, 20).exponential_(1, generator=g))
        E = E_dev[:T]
        sched = sd.PredefinedNoiseScheduleDiscrete("cosine", T)
        n0 = sd.lib().seqdiff_launch_count()
        final = sd.denoise_tensors(batch, m, sched, tr, True, timesteps=T, x_T=x_T, noise_E_steps=E, packed=packed)
        torch.cuda.synchronize()
        runs.append(sd.lib().seqdiff_launch_count() - n0)
        _check(final, _stepwise(sd, m, batch, x_T, E, T, sched, tr), batch, packed)
    # a re-capture would add the dry-run forward's launches: the second call counts what the third, surely cached, one does
    assert runs[1] == runs[2], runs
