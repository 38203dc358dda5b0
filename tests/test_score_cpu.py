"""CPU tests of the sequence score: the oracle's definition (tests/score_oracle.py) and the argument checks of score_tensors, which
all happen before any device work -- there is no CPU path to fall back to."""
import pytest
import torch
import torch.nn.functional as F

import score_oracle as SO
from helpers import O


def _tables(T, uniform):
    return O.NoiseScheduleDiscrete("cosine", T), (O.DiscreteUniformTransition(20) if uniform else O.BlosumTransition())


@pytest.mark.parametrize("uniform", [False, True])
@pytest.mark.parametrize("k", [1, 7, 19])
def test_kl_is_nonnegative_and_vanishes_for_a_perfect_denoiser(uniform, k):
    T, B, L = 20, 3, 16
    sched, tr = _tables(T, uniform)
    g = torch.Generator().manual_seed(k)
    x0 = F.one_hot(torch.randint(0, 20, (B, L), generator=g), 20).float()
    t, s, Qt, Qsb, Qtb = SO.step_tables(k, T, B, sched, tr)
    x_t = SO.q_sample(x0, Qtb, torch.empty(B * L, 20).exponential_(1, generator=g))
    rand = torch.randn(B, L, 20, generator=g) * 3
    kl, ce = SO.step_terms(k, rand, x0, x_t, Qt, Qsb, Qtb, t, s, sched, tr)
    assert (kl >= 0).all() and (ce > 0).all()
    kl, ce = SO.step_terms(k, 50 * x0, x0, x_t, Qt, Qsb, Qtb, t, s, sched, tr)
    assert kl.abs().max().item() < 1e-9 and ce.max().item() < 1e-9


def test_prior_matches_the_closed_form_for_the_uniform_transition():
    T = 50
    sched, tr = _tables(T, True)
    Qtb = SO.step_tables(T - 1, T, 1, sched, tr)[4][0]
    a = float(sched.get_alpha_bar(t_int=torch.tensor([T])).double())  # the last step's Qtb is Qbar at t_int = T
    stay, other = a + (1 - a) / 20, (1 - a) / 20
    want = stay * torch.log(torch.tensor(20 * stay, dtype=torch.float64)) + 19 * other * torch.log(torch.tensor(20 * other, dtype=torch.float64))
    got = SO.prior_terms(Qtb)
    assert torch.allclose(got, want.expand(20), rtol=0, atol=1e-6), (got, want)


def test_one_step_bound_is_prior_plus_reconstruction():
    B, L = 2, 12
    sched, tr = _tables(1, False)
    g = torch.Generator().manual_seed(3)
    batch = O.synthetic_batch(B, L, (4, 12), (4, 12), 5)
    x0 = batch["ligand_seq"]
    z = torch.randn(B, L, 20, generator=g)
    terms, prior = SO.score_loop(None, None, batch, x0, sched, tr, 1, torch.empty(1, B * L, 20).exponential_(1, generator=g),
                                 forward=lambda k, x_t: z)
    valid = batch["ligand_attn_mask"] != 0
    recon = -(F.log_softmax(z.double(), -1) * x0.double()).sum(-1) * valid
    assert torch.equal(terms[..., 0], terms[..., 1]) and torch.allclose(terms[..., 0], recon, rtol=0, atol=1e-12)
    nll, _, ce = SO.per_residue(terms, prior, batch["ligand_attn_mask"], 1)
    n = valid.sum(1).double()
    assert torch.allclose(nll, (prior + recon.sum(1)) / n, rtol=0, atol=1e-12) and torch.allclose(ce, recon.sum(1) / n, rtol=0, atol=1e-12)


@pytest.mark.parametrize("uniform", [False, True])
def test_in_loop_q_sample_is_the_training_q_sample_at_the_next_step(uniform):
    T, B, L = 50, 3, 20
    sched, tr = _tables(T, uniform)
    g = torch.Generator().manual_seed(9)
    x0 = F.one_hot(torch.randint(0, 20, (B, L), generator=g), 20).float()
    for k in (0, 1, 24, 49):
        E = torch.empty(B * L, 20).exponential_(1, generator=g)
        Qtb = SO.step_tables(k, T, B, sched, tr)[4]
        want = O.apply_aa_noise(x0, torch.full((B, 1), float(k + 1)), T, sched, tr, E)
        assert torch.equal(SO.q_sample(x0, Qtb, E), want), k


class _NoModel:
    """any use of the model means the checks let the call through to the device"""
    def __getattr__(self, name):
        raise AssertionError(f"model.{name} used before the arguments were checked")


def _batch(P=2, L=10):
    return O.synthetic_batch(P, L, (3, L), (4, L), 17)


def _sched():
    import seqdiff_b200 as sd
    return sd.PredefinedNoiseScheduleDiscrete("cosine", 4), sd.DiscreteUniformTransition(20)


@pytest.mark.parametrize("why", ["not one-hot", "two hot", "fractional", "empty row", "no valid position", "sequence shape",
                                 "sample count", "receptor shape", "angles shape", "noise shape"])
def test_bad_inputs_raise_before_any_device_work(why):
    import seqdiff_b200 as sd
    batch, seqs, kw = _batch(), None, {}
    if why == "not one-hot":
        seqs = batch["ligand_seq"].clone()
        seqs[1, 0] = 0.5 * seqs[1, 0]
    elif why == "two hot":
        seqs = batch["ligand_seq"].clone()
        seqs[0, 1, :2] = 1
    elif why == "fractional":
        seqs = batch["ligand_seq"].clone()
        seqs[0, 0] = seqs[0, 0] * 0.5 + 0.025
    elif why == "empty row":
        seqs = batch["ligand_seq"].clone()
        seqs[1, 0] = 0
    elif why == "no valid position":
        batch["ligand_attn_mask"][1] = 0
    elif why == "sequence shape":
        seqs = batch["ligand_seq"][:, :5]
    elif why == "sample count":
        seqs = batch["ligand_seq"].repeat(3, 1, 1)
        kw["num_samples"] = 2
    elif why == "receptor shape":
        batch["receptor_seq"] = batch["receptor_seq"][:1]
    elif why == "angles shape":
        batch["ligand_angles"] = batch["ligand_angles"][..., :4]
    else:
        kw["noise_E_steps"] = torch.ones(4, 19, 20)
    sched, tr = _sched()
    with pytest.raises(ValueError):
        sd.score_tensors(batch, _NoModel(), sched, tr, sequences=seqs, timesteps=4, **kw)
    with pytest.raises(ValueError):
        sd.score(batch, _NoModel(), sched, tr, sequences=seqs, timesteps=4, **kw)


@pytest.mark.parametrize("k", [0, -1, 1.5, True])
def test_bad_sample_counts_raise(k):
    import seqdiff_b200 as sd
    sched, tr = _sched()
    with pytest.raises(ValueError, match="num_samples"):
        sd.score_tensors(_batch(), _NoModel(), sched, tr, timesteps=4, num_samples=k)


def test_valid_inputs_reach_the_device_and_there_is_no_cpu_fallback():
    """with a CPU model, the checks pass and the call fails at the handle instead of computing on the host"""
    import seqdiff_b200 as sd
    from helpers import make_model
    cfg = O.OracleConfig(hidden_size=256, num_attention_heads=4, intermediate_size=256, num_hidden_layers=1, max_position_embeddings=16)
    m = make_model(sd, cfg, O.init_state_dict(cfg, 0, "B"), device="cpu")
    sched, tr = _sched()
    with pytest.raises((RuntimeError, sd.SeqdiffError)):
        sd.score_tensors(_batch(), m, sched, tr, timesteps=4)


def test_c_abi_rejects_bad_sizes_and_flags():
    """seqdiff_score_multi checks its sizes and flags before it touches the handle (a stand-in pointer is never dereferenced)"""
    import ctypes

    import seqdiff_b200 as sd
    lib = sd.lib()
    buf = ctypes.create_string_buffer(64)
    p = ctypes.cast(buf, ctypes.c_void_p)
    for P, K, Ll, Lr, T, flags in ((0, 1, 8, 8, 5, 0), (1, 0, 8, 8, 5, 0), (2, 2, 0, 8, 5, 0), (2, 2, 8, 8, 0, 0), (1 << 16, 1 << 10, 64, 128, 5, 0),
                                   (2, 3, 8, 8, 5, 2), (2, 3, 8, 8, 5, -1)):
        rc = lib.seqdiff_score_multi(p, 1, P, K, Ll, Lr, T, p, p, p, p, p, p, p, None, 0, 0, flags, p, None)
        assert rc == 1, (P, K, Ll, T, flags)  # SEQDIFF_ERR_INVALID
        assert lib.seqdiff_last_error()
