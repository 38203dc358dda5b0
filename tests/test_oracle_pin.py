"""CPU tests: the oracle against the golden vectors produced from the unmodified reference
(oracle/make_golden.py)."""
import glob
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from helpers import GOLDEN, O


def _load(name):
    return torch.load(os.path.join(GOLDEN, name), weights_only=False)


def test_blosum_tables_fixture():
    z = np.load(os.path.join(GOLDEN, "blosum_tables.npz"))
    assert z["original_score"].shape == (20, 20) and z["Qtb_temperature"].shape == (500,)
    assert str(z["source_sha256"]).startswith("b24cde8e")  # SURVEY.md section 2
    s = z["original_score"]
    assert np.array_equal(s, s.T) and s.min() >= 0 and s.max() == 15


@pytest.mark.parametrize("T", [50, 500])
def test_schedule_and_transitions(T):
    g = _load(f"schedule_T{T}.pt")
    sched = O.NoiseScheduleDiscrete("cosine", T)
    assert torch.equal(sched.betas, g["betas"]) and torch.equal(sched.alphas_bar, g["alphas_bar"])
    a = sched.get_alpha_bar(t_normalized=g["probe_t"])
    assert torch.equal(a, g["alpha_bar_probe"])
    tr = O.BlosumTransition()
    assert torch.equal(tr.temperature_list, g["temperature_list"]) and torch.equal(tr.Qt_temperature, g["Qt_temperature"])
    assert torch.equal(tr.get_Qt_bar(a), g["Qtb_probe"])
    assert torch.equal(tr.get_Qt(a), g["Qt_probe"])
    assert torch.equal(O.DiscreteUniformTransition(20).get_Qt_bar(a), g["uniform_Qtb_probe"])


def test_product_host_tables_match_oracle():
    """The product's host-side schedule/transition mirror (utils.py of the package) builds the same
    per-step (Qt,Qsb,Qtb) tables as the oracle, bit for bit."""
    import seqdiff_b200 as sd
    for T in (50, 500):
        tabs = sd.utils.loop_tables(T, sd.PredefinedNoiseScheduleDiscrete("cosine", T), sd.BlosumTransition(x_classes=20))
        o_s, o_t = O.NoiseScheduleDiscrete("cosine", T), O.BlosumTransition()
        for s_int in (0, 1, T // 2, T - 1):
            s = torch.full((1, 1), float(s_int))
            Qt, Qsb, Qtb = O.step_matrices((s + 1) / T, s / T, o_s, o_t)
            assert torch.equal(tabs[s_int, 0], Qt[0]) and torch.equal(tabs[s_int, 1], Qsb[0]) and torch.equal(tabs[s_int, 2], Qtb[0])
    u = sd.utils.loop_tables(50, sd.PredefinedNoiseScheduleDiscrete("cosine", 50), sd.DiscreteUniformTransition(20))
    assert u.shape == (50, 3, 20, 20)


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLDEN, "reverse_step_*.pt"))), ids=os.path.basename)
def test_reverse_step_golden(path):
    g = torch.load(path, weights_only=False)
    T, s_int = g["T"], g["s_int"]
    sched = O.NoiseScheduleDiscrete("cosine", T)
    tr = O.BlosumTransition() if g["kind"] == "blosum" else O.DiscreteUniformTransition(20)
    x = F.one_hot(g["x_t_idx"].long(), 20).float()
    B = x.shape[0]
    s = s_int * torch.ones((B, 1))
    out = O.reverse_step((s + 1) / T, s / T, x, g["logits"], sched, tr, g["diverse"], s_int == 0, g["E"])
    if s_int == 0:
        assert torch.equal(out, g["out"])
    else:
        assert torch.equal(out.argmax(-1).to(torch.uint8), g["out"])
        assert torch.equal(O.reverse_step_probs((s + 1) / T, s / T, x, g["logits"], sched, tr), g["prob"])


def test_apply_aa_noise_golden():
    g = _load("apply_aa_noise.pt")
    x0 = F.one_hot(g["x0_idx"].long(), 20).float() * g["x0_valid"].float()[..., None]
    out = O.apply_aa_noise(x0, g["t_int"], g["T"], O.NoiseScheduleDiscrete("cosine", g["T"]), O.BlosumTransition(), g["E"])
    assert torch.equal(out.argmax(-1).to(torch.uint8), g["out_idx"])


@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLDEN, "forward_*rel_*.pt"))), ids=os.path.basename)
def test_forward_golden(path):
    g = torch.load(path, weights_only=False)
    if g["B"] > 1 and "cfg1" not in g["name"] and g["relative_key"] is False:
        pytest.skip("covered by the relative_key variant; keeps the CPU suite short")
    cfg = O.OracleConfig(max_position_embeddings=g["L"], relative_key=g["relative_key"])
    sd = O.init_state_dict(cfg, g["weight_seed"], g["variant"])
    batch = O.synthetic_batch(g["B"], g["L"], g["n_lig"], g["n_rec"], g["input_seed"])
    x_t = F.one_hot(g["x_t_idx"].long(), 20).float()
    t = torch.full((g["B"], 1), g["timestep"])
    with torch.no_grad():
        y = O.denoiser_forward(sd, cfg, t, x_t, batch["ligand_angles"], batch["ligand_attn_mask"], batch["receptor_seq"],
                               batch["receptor_angles"], batch["receptor_attn_mask"])
    # bit-exact where generated; a different BLAS thread count on another host may reorder sums
    assert (y - g["logits"]).abs().max().item() <= 2e-5 * g["logits"].abs().max().item()


def test_relative_key_term_matches_naive_einsum():
    """pin (ii) of SURVEY.md section 8c: the restated Rel term against an explicit triple loop."""
    torch.manual_seed(0)
    cfg = O.OracleConfig(hidden_size=128, num_attention_heads=2, max_position_embeddings=16)
    B, L = 2, 11
    q, k, v = torch.randn(B, L, 128), torch.randn(B, L, 128), torch.randn(B, L, 128)
    E = torch.randn(31, 64)
    mask = torch.zeros(B, 1, 1, L)
    got = O.attention_core(cfg, q, k, v, mask, E)
    qh = q.view(B, L, 2, 64).permute(0, 2, 1, 3)
    kh = k.view(B, L, 2, 64).permute(0, 2, 1, 3)
    vh = v.view(B, L, 2, 64).permute(0, 2, 1, 3)
    s = torch.zeros(B, 2, L, L)
    for l in range(L):
        for r in range(L):
            s[:, :, l, r] = ((qh[:, :, l] * kh[:, :, r]).sum(-1) + (qh[:, :, l] * E[l - r + 15]).sum(-1)) / 8.0
    want = (torch.softmax(s, -1) @ vh).permute(0, 2, 1, 3).reshape(B, L, 128)
    assert torch.allclose(got, want, atol=1e-5)


def test_identity_at_init_trap():
    """weight variant A reproduces the reference init where decoder_normalize is the identity
    (SURVEY.md section 7) -- the reason every parity test also runs variant B."""
    cfg = O.OracleConfig(max_position_embeddings=32)
    sd = O.init_state_dict(cfg, 0, "A")
    assert sd["decoder_normalize.adaLN_modulation.0.weight"].abs().max() == 0
    x = torch.randn(1, 32, 768)
    te = torch.randn(1, 1, 768)
    out = O.se_layer(sd, cfg, "decoder_normalize", x, te, torch.zeros(1, 1, 1, 32))
    assert torch.equal(out, x)


def test_reference_live_pin():
    """The reference forward as installed (no relative_key term) on two graphs of L = 64, weight variant B: its stored logits
    (forward_norel_L64_B.pt, the case test_forward_golden skips) against the oracle."""
    g = _load("forward_norel_L64_B.pt")
    assert (g["L"], g["B"], g["variant"], g["relative_key"]) == (64, 2, "B", False)
    cfg = O.OracleConfig(max_position_embeddings=64, relative_key=False)
    sd = O.init_state_dict(cfg, g["weight_seed"], "B")
    b = O.synthetic_batch(2, 64, g["n_lig"], g["n_rec"], g["input_seed"])
    x_t = F.one_hot(g["x_t_idx"].long(), 20).float()
    t = torch.full((2, 1), g["timestep"])
    with torch.no_grad():
        yo = O.denoiser_forward(sd, cfg, t, x_t, b["ligand_angles"], b["ligand_attn_mask"], b["receptor_seq"], b["receptor_angles"],
                                b["receptor_attn_mask"])
    assert (g["logits"] - yo).abs().max().item() < 1e-5


def test_dataset_item_golden():
    """dataset.py:97-129 restatement against values produced by the reference class (ext 0/1/3, wrap-around quirk Q9)."""
    g = _load("dataset_items.pt")
    recs = O.synthetic_records(g["n_complex"], g["seed"])
    for (ext, max_len), want in g["cases"].items():
        items = [O.dataset_item(r, max_len, ext) for r in recs]
        assert torch.equal(torch.tensor([int(i["ligand_length"]) for i in items]), want["ligand_length"])
        assert torch.equal(torch.tensor([int(i["receptor_length"]) for i in items]), want["receptor_length"])
        assert torch.equal(torch.stack([i["receptor_seq"].argmax(-1).to(torch.uint8) for i in items]), want["receptor_seq_idx"])
        assert torch.equal(torch.stack([i["receptor_angles"].double().sum(-1) for i in items]), want["receptor_angle_sum"])
        assert torch.equal(torch.stack([i["ligand_seq"].argmax(-1).to(torch.uint8) for i in items]), want["ligand_seq_idx"])
    # ext > 0 really dilates, and only by exactly +-ext
    assert (g["cases"][(1, 128)]["receptor_length"] >= g["cases"][(0, 128)]["receptor_length"]).all()
    with pytest.raises(RuntimeError, match="Length exceed"):
        O.dataset_item(recs[0], 4, 0)


def test_structure_feed_cfg5_fixture_and_oracle():
    """BASELINE configs[4]: angles generated by the reference structure_model denoiser (12 + 12 layers, feature_size 8;
    oracle/make_golden.py::golden_structure_feed) have the shape / dtype / range the sequence model takes as `ligand_angle`
    (sample_by_generated_angles.py:202), and the oracle's sequence forward accepts them."""
    g = _load("structure_feed_cfg5.pt")
    B, L = g["B"], g["L"]
    ang = g["angles"]
    assert ang.shape == (B, L, 8) and ang.dtype == torch.float32 and torch.isfinite(ang).all()
    assert ang.min() >= -np.pi and ang.max() < np.pi
    cfg = O.OracleConfig(max_position_embeddings=L, num_hidden_layers=1)
    state = O.init_state_dict(cfg, 1, "B")
    batch = O.synthetic_batch(2, L, g["n_lig"], g["n_rec"], g["batch_seed"])
    x_t = O.generate_discrete_noise(2, L, generator=torch.Generator().manual_seed(3))
    with torch.no_grad():
        y = O.denoiser_forward(state, cfg, torch.full((2, 1), 9.0), x_t, ang[:2] * batch["ligand_attn_mask"][..., None],
                               batch["ligand_attn_mask"], batch["receptor_seq"], batch["receptor_angles"], batch["receptor_attn_mask"])
    assert y.shape == (2, L, 20) and torch.isfinite(y).all()


def test_structure_model_reference_shape_live():
    """Same check on what the reference structure model itself returned for 128-residue graphs (its stored outputs, with and
    without the relative_key term): [B, L, 8] fp32, the shape and dtype the sequence model takes as `ligand_angle`."""
    for name in ("struct_forward_norel_L128_l12.pt", "struct_forward_rel_L128_l12.pt"):
        g = _load(name)
        out = g["out"]
        assert out.shape == (g["B"], g["L"], 8) and g["L"] == 128 and out.dtype == torch.float32 and torch.isfinite(out).all()
