"""Training step of the structure (angle) model: the wrapped smooth-L1 objective and its gradient, the hand-written backward against
torch autograd on the oracle (tests/struct_train_oracle.py: training_grads), the parameter table, fit / checkpoint / validation.

CPU (`-m "not gpu"`): the closed-form loss gradient against autograd, the Python surface and the ABI declarations, no CPU fallback.
GPU: fp32 mode with dropout off -- every gradient tensor within 1e-5 (max-norm relative) of the oracle's, the prediction within 1e-5 and
the loss within 2e-5; 16-bit modes -- flat L2 relative error (bf16 < 3e-2, fp16 < 5e-3) and per-tensor cosines; dropout on -- the
16-bit step against the fp32 step under the same Philox masks."""
import inspect
import math
import os

import pytest
import torch

from helpers import O, sd_pkg
from oracle import structdiff_oracle as S
import struct_train_oracle as T

gpu = pytest.mark.gpu
DEV = "cuda:0"
T_STEPS = 1000
SMALL_COS = {"bf16": 0.995, "fp16": 0.9999}  # the sequence step's bounds for the small gradient tensors (tests/test_train.py)


def _cfg(L, layers, rel=True):
    return S.OracleConfig(max_position_embeddings=L, num_hidden_layers=layers, feature_size=8, relative_key=rel)


def _noised_batch(B, Ll, Lr, n_lig, n_rec, seed):
    """A batch the way FoldingDiff's NoisedAnglesDataset builds one: t ~ U{0..T-1}, known_noise ~ N(0,1), corrupted =
    wrap(sqrt(alphabar_t) x0 + sqrt(1 - alphabar_t) known_noise), on top of the padded dataset tensors."""
    batch = O.synthetic_batch(B, Ll, n_lig, n_rec, seed)
    if Lr != Ll:
        rec = O.synthetic_batch(B, Lr, n_lig, n_rec, seed + 1)
        for k in ("receptor_seq", "receptor_angles", "receptor_attn_mask"):
            batch[k] = rec[k]
    g = torch.Generator().manual_seed(seed + 2)
    ab = S.compute_alphas(S.cosine_beta_schedule(T_STEPS))
    t = torch.randint(0, T_STEPS, (B,), generator=g)
    noise = torch.randn(B, Ll, 8, generator=g)
    x0 = batch["ligand_angles"]
    corrupted = S.modulo_with_wrapped_range(ab["sqrt_alphas_cumprod"][t][:, None, None] * x0 +
                                            ab["sqrt_one_minus_alphas_cumprod"][t][:, None, None] * noise)
    return {"corrupted": corrupted, "t": t, "known_noise": noise, "ligand_attn_mask": batch["ligand_attn_mask"],
            "receptor_seq": batch["receptor_seq"], "receptor_angles": batch["receptor_angles"], "receptor_attn_mask": batch["receptor_attn_mask"]}


def _wrap_margin(diff, mask):
    """smallest distance of known_noise - pred from an odd multiple of pi over the valid positions (the wrap's discontinuity)"""
    r = torch.remainder(diff.double() + math.pi, 2 * math.pi)
    return float(torch.minimum(r, 2 * math.pi - r)[mask != 0].min())


def _make(sd, cfg, state, precision, **kw):
    pos = "relative_key" if cfg.relative_key else "absolute"
    common = dict(max_position_embeddings=cfg.max_position_embeddings, num_attention_heads=cfg.num_attention_heads, hidden_size=cfg.hidden_size,
                  intermediate_size=cfg.intermediate_size, num_hidden_layers=cfg.num_hidden_layers, position_embedding_type=pos)
    m = sd.structure_model.ConditionalBertForDiffusion(sd.BertConfig(**common), sd.BertConfig(**common, is_decoder=True, add_cross_attention=True),
                                                       cfg.feature_size, **kw)
    if state is not None:
        m.load_state_dict(state, strict=True)
    m = m.eval().to(DEV)
    m.precision = precision
    return m


# ---------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------
def test_angle_loss_gradient_formula_matches_autograd():
    """dL/dpred = -h'(d) / (F * n_valid) at valid positions (h' = d / beta inside beta, sign(d) outside; the wrap has derivative 1), fp64,
    with elements on both sides of beta and differences wrapped across +-pi."""
    g = torch.Generator().manual_seed(0)
    B, L, Fs = 3, 16, 8
    beta = math.pi / 10
    noise = torch.randn(B, L, Fs, generator=g, dtype=torch.float64)
    d0 = torch.cat([torch.rand(B, L, 3, generator=g, dtype=torch.float64) * 0.6 - 0.3,          # |d| < beta (mostly)
                    torch.rand(B, L, 3, generator=g, dtype=torch.float64) * 4 - 2,              # beyond beta
                    torch.rand(B, L, 2, generator=g, dtype=torch.float64) * 2 + 3.3], dim=-1)    # |d| > pi: wrapped
    pred = (noise - d0).requires_grad_(True)
    mask = (torch.arange(L)[None, :] < torch.tensor([16, 9, 4])[:, None]).double()
    loss, per_feature = T.angle_loss(pred, noise, mask, beta)
    loss.backward()
    d = S.modulo_with_wrapped_range(noise - pred.detach())
    assert (d0.abs() < beta).any() and (d0.abs() > beta).any() and (d0.abs() > math.pi).any()
    assert (d >= -math.pi).all() and (d < math.pi).all()
    hp = torch.where(d.abs() < beta, d / beta, torch.sign(d))
    want = -hp / (Fs * mask.sum()) * mask[..., None]
    assert torch.allclose(pred.grad, want, atol=1e-15, rtol=1e-12), (pred.grad - want).abs().max()
    # the value: per-feature means of smooth_l1 over the valid positions, then their mean (torch's own smooth_l1_loss per feature)
    ref = torch.stack([torch.nn.functional.smooth_l1_loss(d[..., i][mask != 0], torch.zeros(int(mask.sum()), dtype=torch.float64), beta=beta)
                       for i in range(Fs)])
    assert torch.allclose(per_feature.detach(), ref, rtol=1e-12) and float(loss.detach()) == pytest.approx(float(ref.mean()), rel=1e-12)


def test_struct_training_surface_and_no_cpu_fallback():
    sd = sd_pkg()
    SM = sd.structure_model
    assert issubclass(SM.ConditionalBertForDiffusion, SM.ConditionalBertForDiffusionBase)
    sig = inspect.signature(SM.ConditionalBertForDiffusion.__init__)
    assert list(sig.parameters)[1:4] == ["encoder_config", "decoder_config", "feature_size"]
    kw = {k: p.default for k, p in sig.parameters.items() if p.kind == p.KEYWORD_ONLY}
    assert kw == {"loss": "smooth_l1", "learning_rate": 5e-5, "l2_lambda": 0.0, "lr_scheduler": None, "max_epochs": 1, "gradient_clip": 1.0}
    for name in ("training_step", "validation_step", "configure_optimizers", "pull_weights", "state_dict"):
        assert callable(getattr(SM.ConditionalBertForDiffusion, name)), name
    assert list(inspect.signature(SM.ConditionalBertForDiffusion.training_step).parameters)[1:] == ["batch", "batch_idx"]
    assert list(inspect.signature(SM.ConditionalBertForDiffusion.configure_optimizers).parameters)[1:] == ["group", "grad_comm"]
    assert callable(sd.train.struct_train_step_tensors)
    # the ABI symbols: declared in the header and bound in _cabi.py
    header = open(os.path.join(os.path.dirname(__file__), "..", "include", "seqdiff_b200.h")).read()
    for sym in ("seqdiff_struct_train_step", "seqdiff_struct_loss_terms"):
        assert f"SEQDIFF_API int {sym}(" in header and sym in sd._cabi.PROTOTYPES, sym
    assert len(sd._cabi.PROTOTYPES["seqdiff_struct_train_step"][1]) == 20 and len(sd._cabi.PROTOTYPES["seqdiff_struct_loss_terms"][1]) == 7
    common = dict(max_position_embeddings=32, intermediate_size=1024, num_hidden_layers=1)
    cfgs = (sd.BertConfig(**common), sd.BertConfig(**common, is_decoder=True, add_cross_attention=True))
    with pytest.raises(ValueError, match="smooth_l1"):
        SM.ConditionalBertForDiffusion(*cfgs, 8, loss="l1")
    m = SM.ConditionalBertForDiffusion(*cfgs, 8)
    batch = _noised_batch(1, 8, 8, 8, 8, 0)
    for call in (lambda: m.training_step(batch, 0), lambda: m.validation_step(batch, 0),
                 lambda: SM.angle_loss_terms(batch["known_noise"], batch["known_noise"], batch["ligand_attn_mask"])):
        with pytest.raises(RuntimeError):
            call()
    with pytest.raises(ValueError, match="no valid ligand"):
        m.training_step({**batch, "ligand_attn_mask": torch.zeros(1, 8)}, 0)


# ---------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------
def _step(sd, m, batch, **kw):
    flat = sd.train.FlatParams(m)
    terms, pred = sd.train.struct_train_step_tensors(m, flat, batch, want_pred=True, **kw)
    torch.cuda.synchronize()
    return flat, terms, pred


def _compare_grads(flat, m, grads_ref, tol_rel, what):
    worst = (0.0, "")
    got_all, ref_all = [], []
    gmax = max(float(v.abs().max()) for v in grads_ref.values() if v is not None)
    for k, prm in m.named_parameters():
        ref = grads_ref.get(k)
        assert ref is not None and k in flat.table, k
        got = flat.grad(k, tuple(prm.shape)).cpu()
        got_all.append(got.reshape(-1))
        ref_all.append(ref.reshape(-1))
        err = float((got - ref).abs().max()) / max(float(ref.abs().max()), 1e-3 * gmax)
        if err > worst[0]:
            worst = (err, k)
    assert "timestep_projector.W" not in flat.table and grads_ref["timestep_projector.W"] is None
    got_all, ref_all = torch.cat(got_all), torch.cat(ref_all)
    l2 = float((got_all - ref_all).norm() / ref_all.norm())
    print(f"{what}: worst per-tensor max-norm rel err {worst[0]:.3e} ({worst[1]}); flat-vector L2 rel err {l2:.3e}; {got_all.numel()} elements")
    if tol_rel is not None:
        assert worst[0] < tol_rel, worst
    return worst[0], l2


def _worst_small_tensor_cosine(flat, m, grads_ref):
    gmax = max(float(v.norm()) for v in grads_ref.values() if v is not None)
    worst = (1.0, "")
    for k, prm in m.named_parameters():
        if k not in flat.table or prm.numel() >= 768 * 768:
            continue
        a, b = flat.grad(k).cpu().double(), grads_ref[k].reshape(-1).double()
        if float(b.norm()) < 1e-4 * gmax:
            continue
        cos = float(torch.dot(a, b) / (a.norm() * b.norm()))
        if cos < worst[0]:
            worst = (cos, k)
    return worst


# (Ll, Lr, B, layers, relative_key, n_lig, n_rec, seed).  The seeds are chosen so that no valid known_noise - pred lies within 1e-4 of
# an odd multiple of pi, where the wrap jumps and the fp32 comparison would depend on rounding; each case asserts it.
CASES = {"rel-2+2-L64-ragged": (64, 64, 2, 2, True, (10, 64), (20, 64), 1),
         "abs-Ll!=Lr": (24, 40, 2, 2, False, (5, 24), (12, 40), 2),
         "rel-12+12-L64": (64, 64, 2, 12, True, (30, 64), (40, 64), 3)}


def _oracle_case(case):
    Ll, Lr, B, NL, rel, n_lig, n_rec, seed = CASES[case]
    cfg = _cfg(max(Ll, Lr), NL, rel)
    state = S.init_struct_state_dict(cfg, seed)
    batch = _noised_batch(B, Ll, Lr, n_lig, n_rec, seed + 10)
    return cfg, state, batch


@gpu
@pytest.mark.parametrize("case", list(CASES), ids=list(CASES))
def test_struct_gradient_parity_fp32(case):
    sd = sd_pkg()
    cfg, state, batch = _oracle_case(case)
    torch.set_num_threads(8)
    loss_ref, per_ref, grads_ref, pred_ref = T.training_grads(state, cfg, batch)
    assert _wrap_margin(batch["known_noise"] - pred_ref, batch["ligand_attn_mask"]) > 1e-4
    m = _make(sd, cfg, state, "fp32")
    flat, terms, pred = _step(sd, m, batch)
    assert float((pred.cpu() - pred_ref).abs().max() / pred_ref.abs().max()) < 1e-5
    loss, per = sd.train.angle_loss_from_terms(terms)
    assert float(terms[-1]) == float(batch["ligand_attn_mask"].sum())
    assert float(loss) == pytest.approx(float(loss_ref), rel=2e-5)
    assert torch.allclose(per.cpu(), per_ref, rtol=2e-5, atol=1e-7)
    _compare_grads(flat, m, grads_ref, 1e-5, f"fp32 {case}")
    assert flat.live_numel == sum(v.numel() for v in grads_ref.values() if v is not None)
    m.release()


@gpu
@pytest.mark.parametrize("precision,l2_tol", [("bf16", 3e-2), ("fp16", 5e-3)])
def test_struct_gradient_parity_16bit(precision, l2_tol):
    sd = sd_pkg()
    cfg, state, batch = _oracle_case("rel-2+2-L64-ragged")
    _, _, grads_ref, _ = T.training_grads(state, cfg, batch)
    m = _make(sd, cfg, state, precision)
    flat, _, _ = _step(sd, m, batch)
    _, l2 = _compare_grads(flat, m, grads_ref, None, f"{precision} rel-2+2-L64")
    assert l2 < l2_tol, l2
    for k, prm in m.named_parameters():
        if k in flat.table and prm.numel() >= 768 * 768:
            a, b = flat.grad(k).cpu(), grads_ref[k].reshape(-1)
            cos = float(torch.dot(a, b) / (a.norm() * b.norm()))
            assert cos > 0.999, (k, cos)
    worst = _worst_small_tensor_cosine(flat, m, grads_ref)
    print(f"{precision}: worst cosine over the small gradient tensors {worst[0]:.5f} ({worst[1]})")
    assert worst[0] > SMALL_COS[precision], worst
    m.release()


@gpu
@pytest.mark.parametrize("precision,l2_tol", [("bf16", 3e-2), ("fp16", 5e-3)])
def test_struct_gradient_16bit_with_dropout_matches_fp32_step(precision, l2_tol):
    """p = 0.1 in the 16-bit modes against the fp32 CUDA step with the same seed and step, hence the same Philox masks."""
    sd = sd_pkg()
    cfg, state, batch = _oracle_case("rel-2+2-L64-ragged")
    kw = dict(p_hidden=0.1, p_attn=0.1, seed=23, step=4)
    m32 = _make(sd, cfg, state, "fp32").train()
    flat32, terms32, _ = _step(sd, m32, batch, **kw)
    ref = {k: flat32.grad(k, tuple(prm.shape)).cpu().clone() for k, prm in m32.named_parameters() if k in flat32.table}
    loss32 = float(sd.train.angle_loss_from_terms(terms32)[0])
    m32.release()
    m = _make(sd, cfg, state, precision).train()
    flat, terms, _ = _step(sd, m, batch, **kw)
    assert float(sd.train.angle_loss_from_terms(terms)[0]) == pytest.approx(loss32, rel=2e-2)
    got_all = torch.cat([flat.grad(k).cpu() for k in ref])
    ref_all = torch.cat([v.reshape(-1) for v in ref.values()])
    l2 = float((got_all - ref_all).norm() / ref_all.norm())
    worst = _worst_small_tensor_cosine(flat, m, ref)
    print(f"{precision}, dropout 0.1, vs fp32 step with the same masks: flat L2 rel err {l2:.3e}; worst small-tensor cosine {worst[0]:.5f} ({worst[1]})")
    assert l2 < l2_tol, l2
    assert worst[0] > SMALL_COS[precision], worst
    # dropout is on: the gradient differs from the dropout-off step
    m.eval()
    flat0, _, _ = _step(sd, m, batch)
    assert float((flat0.grads - flat.grads).norm() / flat.grads.norm()) > 0.05
    m.release()


@gpu
def test_struct_parameter_table_and_buckets():
    sd = sd_pkg()
    cfg = _cfg(64, 4, True)
    state = S.init_struct_state_dict(cfg, 5)
    m = _make(sd, cfg, state, "bf16")
    flat = sd.train.FlatParams(m)
    names = list(flat.table)
    assert len(names) == len(set(names))
    assert set(names) == set(state) - {"timestep_projector.W"}
    assert flat.live_numel == sum(v.numel() for k, v in state.items() if k != "timestep_projector.W")
    spans = sorted(flat.table.values())
    assert all(o + n <= o2 for (o, n), (o2, _) in zip(spans, spans[1:])) and spans[-1][0] + spans[-1][1] <= flat.total
    b = flat.bucket_bounds
    assert b[0] == 0 and b[-1] == flat.total and all(x < y for x, y in zip(b, b[1:])) and len(b) == 5
    off = lambda k: flat.table[k][0]  # noqa: E731
    # forward order; the fused projections' parts are contiguous
    assert off("receptor_seq_emb.linear.weight") == 0
    assert off("receptor_emb.mlp.3.bias") < off("encoder.layer.0.attention.self.query.weight") < off("decoder.layer.0.crossattention.self.key.weight")
    assert off("decoder.layer.0.crossattention.self.key.weight") < off("ligand_angle_emb.linear.weight") < off("timestep_emb.mlp.0.weight")
    assert off("timestep_emb.mlp.3.bias") < off("decoder.layer.0.attention.self.query.weight") < off("angles_predictor.dense1.weight")
    H = cfg.hidden_size
    assert off("decoder.layer.0.crossattention.self.value.weight") == off("decoder.layer.0.crossattention.self.key.weight") + H * H
    assert off("encoder.layer.1.attention.self.key.weight") == off("encoder.layer.1.attention.self.query.weight") + H * H
    # buckets: [.., encoder 2) [encoder 2, cross K|V) [cross K|V, decoder 2) [decoder 2, end)
    assert b[1] == off("encoder.layer.2.attention.self.query.weight")
    assert b[2] == off("decoder.layer.0.crossattention.self.key.weight")
    assert b[3] == off("decoder.layer.2.attention.self.query.weight")
    # the bucket events are recorded by the structure step too
    nb = len(b) - 1
    ev = [torch.cuda.Event() for _ in range(nb)]
    for e in ev:
        e.record()
    import ctypes
    arr = (ctypes.c_void_p * nb)(*[ctypes.c_void_p(e.cuda_event) for e in ev])
    sd._cabi.check(sd._cabi.lib().seqdiff_train_set_bucket_events(flat.handle, arr, nb))
    batch = _noised_batch(2, 64, 64, (10, 64), (20, 64), 7)
    sd.train.struct_train_step_tensors(m, flat, batch)
    for e in ev:
        e.synchronize()
    sd._cabi.check(sd._cabi.lib().seqdiff_train_set_bucket_events(flat.handle, None, 0))
    m.release()


@gpu
def test_struct_fit_checkpoint_resume_and_sampling():
    """train.fit lowers the loss on a few synthetic batches; FlatAdamW checkpoint / resume is exact (2 + 2 steps == 4); after
    pull_weights the trained model samples."""
    sd = sd_pkg()
    cfg = _cfg(64, 2, True)
    state = S.init_struct_state_dict(cfg, 11)
    batches = [_noised_batch(4, 64, 64, (20, 64), (30, 64), 100 + i) for i in range(3)]

    def fresh(st=state, precision="bf16"):
        m = _make(sd, cfg, st, precision, learning_rate=2e-4)
        return m.train()

    model = fresh()
    hist = sd.train.fit(model, batches, max_epochs=5, log=None)
    print("epoch losses:", [round(h, 4) for h in hist])
    assert all(math.isfinite(h) for h in hist) and hist[-1] < hist[0]
    trained = model.state_dict()
    assert any(not torch.equal(trained[k].cpu(), state[k]) for k in state if k.startswith("encoder.layer.0"))
    assert torch.equal(trained["timestep_projector.W"].cpu(), state["timestep_projector.W"])
    # validation_step on the trained model == the oracle objective on the model's own eval forward
    b = batches[0]
    v = float(model.validation_step(b, 0))
    assert model.training
    model.eval()
    with torch.no_grad():
        pred = model(b["t"], b["corrupted"], b["ligand_attn_mask"], b["receptor_seq"], b["receptor_angles"], b["receptor_attn_mask"]).cpu()
    want, _ = T.angle_loss(pred.double(), b["known_noise"].double(), b["ligand_attn_mask"])
    assert v == pytest.approx(float(want), rel=1e-5)
    # sampling on the trained handle
    model.pull_weights()
    betas = S.cosine_beta_schedule(4)
    x_T = torch.randn(4, 64, 8, generator=torch.Generator().manual_seed(1))
    out = sd.structure_model.p_sample_loop(model, b["ligand_attn_mask"], x_T, b["receptor_seq"], b["receptor_attn_mask"], b["receptor_angles"], 4, betas)
    assert out.shape == (4, 4, 64, 8) and torch.isfinite(out).all()
    model.release()

    def steps(m, opt, first, n):
        for i in range(first, first + n):
            m._train_steps = i  # the dropout step counter of training_step (it increments before use)
            m.training_step(batches[i % 3], i)
            opt.step()

    # fp16 operands, as the sequence model's resume test: the gradients are summed with floating-point atomics (split-K, column sums), so
    # two runs agree to rounding, not bit for bit, and AdamW turns rounding noise on ~0 gradients into updates of up to lr.  The distance is
    # therefore measured against the size of the 4-step update; a resume without the optimizer state is the negative control.
    a = fresh(precision="fp16")
    oa = a.configure_optimizers()["optimizer"]
    steps(a, oa, 0, 4)
    want_sd = {k: v.detach().cpu().clone() for k, v in a.state_dict().items()}
    bm = fresh(precision="fp16")
    ob = bm.configure_optimizers()["optimizer"]
    steps(bm, ob, 0, 2)
    ck_model = {k: v.detach().cpu().clone() for k, v in bm.state_dict().items()}
    ck_opt = {k: (v.detach().cpu().clone() if torch.is_tensor(v) else v) for k, v in ob.state_dict().items()}

    def resumed(load_opt):
        c = fresh(ck_model, precision="fp16")
        oc = c.configure_optimizers()["optimizer"]
        if load_opt:
            oc.load_state_dict(ck_opt)
        steps(c, oc, 2, 2)
        got = {k: v.detach().cpu().clone() for k, v in c.state_dict().items()}
        c.release()
        return got

    def dist(got):
        num = sum(float((want_sd[k].double() - got[k].double()).pow(2).sum()) for k in want_sd)
        upd = sum(float((want_sd[k].double() - state[k].double()).pow(2).sum()) for k in want_sd)
        return math.sqrt(num / upd)

    good, lost = dist(resumed(True)), dist(resumed(False))
    print(f"resume vs 4 steps, relative to the 4-step update: with the optimizer state {good:.3e}, without it {lost:.3e}")
    assert good < 5e-2 and lost > 4 * good, (good, lost)
    for m in (a, bm):
        m.release()
