"""structure_model path (SURVEY.md section 8(f) row 3): oracle pins on CPU, CUDA parity on the GPU.

CPU (`-m "not gpu"`): the oracle restatement (oracle/structdiff_oracle.py) against the golden vectors the UNMODIFIED reference
produced in the build container (oracle/make_golden.py::golden_structure_model), schedule tables, the wrap, the mirror's
state_dict schema and signatures.  GPU (`-m gpu`): the CUDA forward / Gaussian step / sampling loop through the C ABI
against the oracle and the same golden vectors.
"""
import glob
import inspect
import math
import os

import pytest
import torch

from helpers import GOLDEN, O, rel_err, l2_rel
from oracle import structdiff_oracle as S

gpu = pytest.mark.gpu


def _cfg(L, layers, rel=True):
    return S.OracleConfig(max_position_embeddings=L, num_hidden_layers=layers, feature_size=8, relative_key=rel)


def _case_inputs(g):
    batch = O.synthetic_batch(g["B"], g["L"], tuple(g["n_lig"]), tuple(g["n_rec"]), g["input_seed"])
    return batch, g["noised"], g["timestep"]


def _make_model(cfg, state, precision, device="cuda:0"):
    import seqdiff_b200 as sd
    pos = "relative_key" if cfg.relative_key else "absolute"
    common = dict(max_position_embeddings=cfg.max_position_embeddings, num_attention_heads=cfg.num_attention_heads, hidden_size=cfg.hidden_size,
                  intermediate_size=cfg.intermediate_size, num_hidden_layers=cfg.num_hidden_layers, position_embedding_type=pos)
    m = sd.structure_model.ConditionalBertForDiffusionBase(sd.BertConfig(**common), sd.BertConfig(**common, is_decoder=True, add_cross_attention=True),
                                                           cfg.feature_size)
    m.load_state_dict(state, strict=True)
    m = m.eval().to(device)
    m.precision = precision
    return m


# ------------------------------------------------------------------------------------------------------------------
# CPU: oracle pins + host mirror
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLDEN, "struct_forward_*_L64_l2.pt"))) +
                         sorted(glob.glob(os.path.join(GOLDEN, "struct_forward_rel_L128_l12.pt"))), ids=os.path.basename)
def test_struct_forward_oracle_matches_reference_golden(path):
    g = torch.load(path)
    cfg = _cfg(g["L"], g["layers"], g["relative_key"])
    sd = S.init_struct_state_dict(cfg, g["weight_seed"])
    batch, noised, t = _case_inputs(g)
    torch.set_num_threads(8)
    with torch.no_grad():
        y = S.struct_forward(sd, cfg, t, noised, batch["ligand_attn_mask"], batch["receptor_seq"], batch["receptor_angles"], batch["receptor_attn_mask"])
    assert y.shape == g["out"].shape
    assert rel_err(y, g["out"]) < 2e-6  # reference == oracle was 0.0 when the fixture was written (thread count may reorder sums)


def test_struct_schedule_and_wrap_golden():
    for T in (50, 1000):
        g = torch.load(os.path.join(GOLDEN, f"struct_schedule_T{T}.pt"))
        b = S.cosine_beta_schedule(T)
        assert torch.equal(b, g["betas"])
        assert torch.equal(S.step_coefficients(b), g["coef"])
    # reference doctest (utils.py:27-28): modulo_with_wrapped_range(3, -2, 2) == -1
    assert S.modulo_with_wrapped_range(3, -2, 2) == -1
    v = torch.tensor([-7.0, -math.pi, 0.0, 3.0, math.pi, 9.5])
    w = S.modulo_with_wrapped_range(v)
    assert (w >= -math.pi - 1e-6).all() and (w < math.pi + 1e-6).all()
    assert torch.allclose(torch.sin(w), torch.sin(v), atol=1e-5) and torch.allclose(torch.cos(w), torch.cos(v), atol=1e-5)


def test_struct_p_sample_loop_oracle_matches_reference_golden():
    g = torch.load(os.path.join(GOLDEN, "struct_p_sample_loop_T4.pt"))
    cfg = _cfg(g["L"], g["layers"])
    sd = S.init_struct_state_dict(cfg, g["weight_seed"])
    batch = O.synthetic_batch(g["B"], g["L"], tuple(g["n_lig"]), tuple(g["n_rec"]), g["batch_seed"])
    with torch.no_grad():
        got = S.p_sample_loop(sd, cfg, batch["ligand_attn_mask"], g["x_T"], batch["receptor_seq"], batch["receptor_attn_mask"],
                              batch["receptor_angles"], g["T"], S.cosine_beta_schedule(g["T"]), lambda i: g["noise"][i])
        # caching the receptor branch (what the CUDA loop does) changes nothing
        again = S.p_sample_loop(sd, cfg, batch["ligand_attn_mask"], g["x_T"], batch["receptor_seq"], batch["receptor_attn_mask"],
                                batch["receptor_angles"], g["T"], S.cosine_beta_schedule(g["T"]), lambda i: g["noise"][i], cache_encoder=False)
    assert got.shape == g["steps"].shape == (g["T"], g["B"], g["L"], 8)
    assert (got - g["steps"]).abs().max() < 1e-5
    assert torch.equal(got, again)


def test_struct_mirror_schema_and_signatures():
    import seqdiff_b200 as sd
    SM = sd.structure_model
    for L, layers, rel in ((64, 12, True), (128, 2, False)):
        cfg = _cfg(L, layers, rel)
        pos = "relative_key" if rel else "absolute"
        common = dict(max_position_embeddings=L, intermediate_size=1024, num_hidden_layers=layers, position_embedding_type=pos)
        m = SM.ConditionalBertForDiffusionBase(sd.BertConfig(**common), sd.BertConfig(**common, is_decoder=True, add_cross_attention=True), 8)
        want = S.struct_state_dict_schema(cfg)
        got = {k: tuple(v.shape) for k, v in m.state_dict().items()}
        assert got == {k: tuple(v) for k, v in want.items()}
    f = inspect.signature(SM.ConditionalBertForDiffusionBase.forward)
    assert list(f.parameters)[1:] == ["timestep", "noised_ligand_angles", "ligand_attention_masks", "receptor_seq", "receptor_angles",
                                      "receptor_attention_masks", "ligand_pos_ids", "receptor_pos_ids"]  # model.py:180-183
    p = inspect.signature(SM.p_sample)
    assert list(p.parameters)[:8] == ["model", "ligand_mask", "ligand_angle_noise", "receptor_seq", "receptor_mask", "receptor_angle",
                                      "timestep", "betas"]  # sample.py:56-67
    l = inspect.signature(SM.p_sample_loop)
    assert list(l.parameters)[:9] == ["model", "ligand_mask", "ligand_angle_noise", "receptor_seq", "receptor_mask", "receptor_angle",
                                      "total_timesteps", "betas", "disable_pbar"]  # sample.py:105-117
    # host tables are the reference's
    assert torch.equal(SM.cosine_beta_schedule(50), S.cosine_beta_schedule(50))
    assert torch.equal(SM.step_coefficients(SM.cosine_beta_schedule(50)), S.step_coefficients(S.cosine_beta_schedule(50)))
    # no CPU fallback
    z = torch.zeros
    with pytest.raises(RuntimeError, match="CUDA"):
        m.eval()(z(1), z(1, 128, 8), torch.ones(1, 128), z(1, 128, 20), z(1, 128, 8), torch.ones(1, 128))


def test_struct_reference_live_pin():
    """The first reverse step of the UNMODIFIED structure_model's own p_sample_loop (struct_p_sample_loop_T4.pt: relative_key
    term restored, the N(0,1) draw it made stored) against one oracle forward + p_sample_update + wrap from the same x_T."""
    g = torch.load(os.path.join(GOLDEN, "struct_p_sample_loop_T4.pt"))
    cfg = _cfg(g["L"], g["layers"], True)
    state = S.init_struct_state_dict(cfg, g["weight_seed"])
    batch = O.synthetic_batch(g["B"], g["L"], tuple(g["n_lig"]), tuple(g["n_rec"]), g["batch_seed"])
    T, i = g["T"], g["T"] - 1
    t = torch.full((g["B"],), i, dtype=torch.long)
    with torch.no_grad():
        out = S.struct_forward(state, cfg, t, g["x_T"], batch["ligand_attn_mask"], batch["receptor_seq"], batch["receptor_angles"],
                               batch["receptor_attn_mask"])
    got = S.p_sample_update(g["x_T"], out, S.step_coefficients(S.cosine_beta_schedule(T)), i, g["noise"][i])
    assert (S.modulo_with_wrapped_range(got, -math.pi, math.pi) - g["steps"][0]).abs().max().item() < 1e-5


def test_struct_sample_driver_trims_and_batches():
    """reference structure_model/sample.py:191-229 with an injected loop (no GPU): batches of CONFIG["batch_size"], the dataset's own
    start noise, per-complex trimming to the ligand length, and the reference's stop-after-first-batch quirk."""
    import seqdiff_b200 as sd
    SM = sd.structure_model

    class DS:
        timesteps = 3
        alpha_beta_terms = {"betas": SM.cosine_beta_schedule(3)}

        def __len__(self):
            return 5

        def __getitem__(self, i):
            n = 2 + i
            m = (torch.arange(8) < n).float()
            return {"ligand_attn_mask": m, "ligand_angles": torch.zeros(8, 4), "receptor_angles": torch.zeros(8, 4), "receptor_seq": torch.zeros(8, 20),
                    "receptor_attn_mask": torch.ones(8)}

        def sample_noise(self, v):
            return torch.full_like(v, 0.5)

    calls = []

    def fake_loop(model, ligand_mask, ligand_angle_noise, total_timesteps, **kw):
        calls.append(ligand_angle_noise.shape[0])
        return ligand_angle_noise[None].repeat(total_timesteps, 1, 1, 1) + torch.arange(total_timesteps).float()[:, None, None, None]

    old = SM.CONFIG["batch_size"]
    SM.CONFIG["batch_size"] = 2
    try:
        first = SM.sample(None, DS(), loop_fn=fake_loop)
        assert calls == [2] and [a.shape for a in first] == [(3, 2, 4), (3, 3, 4)]   # reference quirk: first batch only
        calls.clear()
        every = SM.sample(None, DS(), first_batch_only=False, loop_fn=fake_loop)
        assert calls == [2, 2, 1] and [a.shape[1] for a in every] == [2, 3, 4, 5, 6]
        assert float(every[4][2, 0, 0]) == 2.5
    finally:
        SM.CONFIG["batch_size"] = old


# ------------------------------------------------------------------------------------------------------------------
# GPU: CUDA parity through the C ABI
# ------------------------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLDEN, "struct_forward_*.pt"))), ids=os.path.basename)
def test_struct_forward_cuda_matches_reference_golden(path):
    g = torch.load(path)
    cfg = _cfg(g["L"], g["layers"], g["relative_key"])
    state = S.init_struct_state_dict(cfg, g["weight_seed"])
    batch, noised, t = _case_inputs(g)
    args = (t, noised, batch["ligand_attn_mask"], batch["receptor_seq"], batch["receptor_angles"], batch["receptor_attn_mask"])
    m = _make_model(cfg, state, "fp32")
    with torch.no_grad():
        y = m(*[a.cuda() for a in args]).cpu()
        assert rel_err(y, g["out"]) < 1e-5, rel_err(y, g["out"])  # north_star fp32 tolerance
        m.precision = "fp16"
        y16 = m(*[a.cuda() for a in args]).cpu()
        assert rel_err(y16, g["out"]) < 1e-2, rel_err(y16, g["out"])
        m.precision = "bf16"
        yb = m(*[a.cuda() for a in args]).cpu()
        # bf16 operands: norm-wise gate; deeper stack (12 + 12 layers) than the sequence model, same per-layer budget (DESIGN.md section 6)
        assert l2_rel(yb, g["out"]) < (1e-2 if g["layers"] <= 2 else 3e-2), l2_rel(yb, g["out"])
    m.release()


@gpu
def test_struct_forward_ragged_lengths_and_float_timestep():
    """L_lig != L_rec, float timesteps of shape [B,1] (the sequence model's convention) and B = 1."""
    cfg = _cfg(96, 2)
    state = S.init_struct_state_dict(cfg, 41)
    B, Ll, Lr = 3, 48, 96
    lig = O.synthetic_batch(B, Ll, (5, 48), (5, 48), 42)
    rec = O.synthetic_batch(B, Lr, (5, 48), (16, 96), 43)
    g = torch.Generator().manual_seed(44)
    noised = (torch.rand(B, Ll, 8, generator=g) * 2 - 1) * math.pi
    t = torch.tensor([[3.0], [250.0], [999.0]])
    with torch.no_grad():
        want = S.struct_forward(state, cfg, t, noised, lig["ligand_attn_mask"], rec["receptor_seq"], rec["receptor_angles"], rec["receptor_attn_mask"])
    m = _make_model(cfg, state, "fp32")
    with torch.no_grad():
        got = m(t.cuda(), noised.cuda(), lig["ligand_attn_mask"].cuda(), rec["receptor_seq"].cuda(), rec["receptor_angles"].cuda(),
                rec["receptor_attn_mask"].cuda()).cpu()
        got1 = m(t[:1].cuda(), noised[:1].cuda(), lig["ligand_attn_mask"][:1].cuda(), rec["receptor_seq"][:1].cuda(),
                 rec["receptor_angles"][:1].cuda(), rec["receptor_attn_mask"][:1].cuda()).cpu()
    assert rel_err(got, want) < 1e-5
    assert rel_err(got1, want[:1]) < 1e-5
    with pytest.raises(Exception, match="Length exceed"):
        m(t.cuda(), torch.zeros(B, 128, 8).cuda(), torch.ones(B, 128).cuda(), rec["receptor_seq"].cuda(), rec["receptor_angles"].cuda(),
          rec["receptor_attn_mask"].cuda())
    m.release()


@gpu
def test_gauss_step_kernel_bit_exact_vs_oracle():
    """seqdiff_struct_p_sample with explicit noise == the reference arithmetic (p_sample + wrap), bit for bit: every operator
    is a separately rounded fp32 op on both sides and fmod is exact."""
    import seqdiff_b200 as sd
    import ctypes
    lib = sd.lib()
    T = 1000
    coef = S.step_coefficients(S.cosine_beta_schedule(T))
    g = torch.Generator().manual_seed(7)
    for (B, L, Fs) in ((3, 64, 8), (2, 37, 3)):  # second: L*F not a multiple of 4 -> scalar path
        x = (torch.rand(B, L, Fs, generator=g) * 2 - 1) * math.pi
        out = torch.randn(B, L, Fs, generator=g) * 3
        z = torch.randn(B, L, Fs, generator=g)
        for step in (999, 500, 1, 0):
            for wrap in (1, 0):
                want = S.p_sample_update(x, out, coef, step, z)
                if wrap:
                    want = S.modulo_with_wrapped_range(want, -math.pi, math.pi)
                res = torch.empty(B, L, Fs, device="cuda")
                xc, oc, zc, cc = x.cuda(), out.cuda(), z.cuda(), coef.cuda()
                rc = lib.seqdiff_struct_p_sample(sd._cabi.ptr(cc), T, step, B, L, Fs, sd._cabi.ptr(xc), sd._cabi.ptr(oc), sd._cabi.ptr(zc), 0, 0, wrap,
                                                 sd._cabi.ptr(res), ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
                assert rc == 0
                assert torch.equal(res.cpu(), want), (B, L, Fs, step, wrap, (res.cpu() - want).abs().max())


@gpu
def test_gauss_step_philox_noise_statistics_and_shard_invariance():
    import seqdiff_b200 as sd
    import ctypes
    lib = sd.lib()
    T, B, L, Fs = 10, 64, 128, 8
    # coef = (1, 0, 1, 1): x' = x + z, no wrap -> the raw N(0,1) stream
    coef = torch.tensor([[1.0, 0.0, 1.0, 1.0]] * T).cuda()
    x = torch.zeros(B, L, Fs, device="cuda")
    st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def draw(b0, nb, step, seed=11):
        res = torch.empty(nb, L, Fs, device="cuda")
        assert lib.seqdiff_struct_p_sample(sd._cabi.ptr(coef), T, step, nb, L, Fs, sd._cabi.ptr(x), sd._cabi.ptr(x), None, seed, b0, 0,
                                           sd._cabi.ptr(res), st) == 0
        return res.cpu()

    z = draw(0, B, 5)
    n = z.numel()
    assert abs(z.mean().item()) < 4 / math.sqrt(n)
    assert abs(z.var().item() - 1) < 0.02
    assert abs((z ** 3).mean().item()) < 0.05 and abs((z ** 4).mean().item() - 3) < 0.1
    assert torch.equal(draw(0, B, 5), z)                        # counter-based: same call, same stream
    assert not torch.equal(draw(0, B, 6), z) and not torch.equal(draw(0, B, 5, seed=12), z)
    assert torch.equal(draw(16, 8, 5), z[16:24])                # keyed by the global graph id: independent of the sharding
    assert torch.equal(draw(0, B, 0), torch.zeros(B, L, Fs))   # step 0 adds no noise (sample.py:95-96)


@gpu
def test_struct_sample_loop_matches_reference_golden_and_stepwise_calls():
    import seqdiff_b200 as sd
    SM = sd.structure_model
    g = torch.load(os.path.join(GOLDEN, "struct_p_sample_loop_T4.pt"))
    cfg = _cfg(g["L"], g["layers"])
    state = S.init_struct_state_dict(cfg, g["weight_seed"])
    batch = O.synthetic_batch(g["B"], g["L"], tuple(g["n_lig"]), tuple(g["n_rec"]), g["batch_seed"])
    T = g["T"]
    betas = SM.cosine_beta_schedule(T)
    m = _make_model(cfg, state, "fp32")
    args = dict(model=m, ligand_mask=batch["ligand_attn_mask"], ligand_angle_noise=g["x_T"], receptor_seq=batch["receptor_seq"],
                receptor_mask=batch["receptor_attn_mask"], receptor_angle=batch["receptor_angles"], total_timesteps=T, betas=betas)
    hist = SM.p_sample_loop(**args, noise_steps=g["noise"])
    assert hist.shape == g["steps"].shape and hist.device.type == "cpu"
    # Against the reference's own p_sample_loop output, step by step from the reference's state (teacher forcing): the update
    # multiplies the model error by a_t * b_t / c_t (= 100 at t = T-1 of this tiny schedule, where beta is clipped to 0.9999), so the
    # fp32 forward tolerance (1e-5 relative, north_star) is scaled by that factor.  Angles live on a circle: compare modulo 2 pi.
    coef = SM.step_coefficients(betas)
    prev = g["x_T"]
    for k, i in enumerate(reversed(range(T))):
        t = torch.full((g["B"],), i, dtype=torch.long)
        got = SM.p_sample_wrapped(m, batch["ligand_attn_mask"], prev, batch["receptor_seq"], batch["receptor_attn_mask"], batch["receptor_angles"], t,
                                  betas, noise=g["noise"][i]).cpu()
        d = (got - g["steps"][k]).abs()
        d = torch.minimum(d, (2 * math.pi - d).abs())
        amp = (coef[i, 0] * coef[i, 1] / coef[i, 2]).item()
        assert d.max() < 1e-5 * 5.0 * max(amp, 1.0) + 1e-5, (i, d.max(), amp)  # 5.0 >= max |model output| of this case
        prev = g["steps"][k]
    # the one-call loop == T separate forward + p_sample(+wrap) calls, bit for bit (same kernels, cached receptor branch)
    x = g["x_T"].cuda()
    for k, i in enumerate(reversed(range(T))):
        t = torch.full((g["B"],), i, dtype=torch.long)
        x = SM.p_sample_wrapped(m, batch["ligand_attn_mask"], x, batch["receptor_seq"], batch["receptor_attn_mask"], batch["receptor_angles"], t, betas,
                                noise=g["noise"][i])
        assert torch.equal(x.cpu(), hist[k]), (k, (x.cpu() - hist[k]).abs().max())
    # un-wrapped p_sample (the reference function itself) wraps to the same thing
    t = torch.full((g["B"],), T - 1, dtype=torch.long)
    raw = SM.p_sample(m, batch["ligand_attn_mask"], g["x_T"], batch["receptor_seq"], batch["receptor_attn_mask"], batch["receptor_angles"], t, betas,
                      noise=g["noise"][T - 1]).cpu()
    assert torch.equal(SM.modulo_with_wrapped_range(raw), hist[0])
    # product mode (bf16, in-kernel Philox): deterministic, sharding-invariant, final entry only
    m.precision = "bf16"
    a = SM.p_sample_loop(**args, seed=5, graph_id0=0, keep_history=False)
    b = SM.p_sample_loop(**args, seed=5, graph_id0=0)
    assert a.shape == (1, g["B"], g["L"], 8) and torch.equal(a[0], b[-1])
    # without explicit graph ids successive calls continue the process-wide noise stream: fresh noise (ADVICE r1)
    e1 = SM.p_sample_loop(**args, seed=5, keep_history=False)
    e2 = SM.p_sample_loop(**args, seed=5, keep_history=False)
    assert not torch.equal(e1, e2)
    args1 = dict(args, ligand_mask=batch["ligand_attn_mask"][1:], ligand_angle_noise=g["x_T"][1:], receptor_seq=batch["receptor_seq"][1:],
                 receptor_mask=batch["receptor_attn_mask"][1:], receptor_angle=batch["receptor_angles"][1:])
    c = SM.p_sample_loop(**args1, seed=5, graph_id0=1)
    valid = batch["ligand_attn_mask"][1].bool()
    d = (c[-1][0][valid] - b[-1][1][valid]).abs()
    d = torch.minimum(d, (2 * math.pi - d).abs())
    assert d.max() < 5e-2  # same noise stream for graph 1 whether it is sampled alone or in a batch (bf16 GEMM tiles may differ)
    assert torch.isfinite(b).all() and (b >= -math.pi - 1e-5).all() and (b <= math.pi + 1e-5).all()
    m.release()


@gpu
def test_structure_to_sequence_pipeline_feed():
    """sample_by_generated_angles.py:202: the structure model's generated angles are accepted as `ligand_angle` by the sequence
    denoiser (BASELINE configs[4])."""
    import seqdiff_b200 as sd
    from helpers import make_model
    SM = sd.structure_model
    L, B, T = 64, 2, 3
    scfg = _cfg(L, 2)
    m = _make_model(scfg, S.init_struct_state_dict(scfg, 51), "bf16")
    batch = O.synthetic_batch(B, L, (5, 40), (16, 64), 52)
    x_T = SM.modulo_with_wrapped_range(torch.randn(B, L, 8, generator=torch.Generator().manual_seed(53)))
    angles = SM.p_sample_loop(m, batch["ligand_attn_mask"], x_T, batch["receptor_seq"], batch["receptor_attn_mask"], batch["receptor_angles"], T,
                              SM.cosine_beta_schedule(T), seed=3)[-1]
    assert angles.shape == (B, L, 8) and angles.dtype == torch.float32
    qcfg = O.OracleConfig(max_position_embeddings=L)
    q = make_model(sd, qcfg, O.init_state_dict(qcfg, 1, "B"), "bf16")
    x_t = O.generate_discrete_noise(B, L, generator=torch.Generator().manual_seed(54))
    with torch.no_grad():
        logits = q(torch.full((B, 1), 9.0).cuda(), x_t.cuda(), angles.cuda(), batch["ligand_attn_mask"].cuda(), batch["receptor_seq"].cuda(),
                   batch["receptor_angles"].cuda(), batch["receptor_attn_mask"].cuda())
    assert logits.shape == (B, L, 20) and torch.isfinite(logits).all()
    m.release()
    q.release()
