"""The padded sampling loop of the 16-bit modes (seqdiff_sample / _ex without packing / _multi) computes only the valid receptor
rows: a receptor row is read by nothing but the decoder's cross-attention, as a key and a value, and a padded key's probability
underflows to exactly 0 there whenever its pocket has a valid key.  Every other operator on receptor rows is row-local.  So the
loop's final logits, padded ligand positions included, must stay bit-identical to T stand-alone forward() calls (which compute
every row) chained through the single reverse step -- and must not depend on what the padded receptor positions hold.
Receptor masks with a hole, a pocket without a valid receptor token and the fp32 mode keep the fully padded path."""
import ctypes

import pytest
import torch

from helpers import O, make_model, sd_pkg

pytestmark = pytest.mark.gpu
DEV = "cuda:0"

_MODEL = {}


def _model(precision):
    if not _MODEL:
        # variant "B": decoder_normalize is not the identity the reference init makes it
        cfg = O.OracleConfig(max_position_embeddings=128, relative_key=True)
        _MODEL["m"] = make_model(sd_pkg(), cfg, O.init_state_dict(cfg, 1, "B"), precision)
    m = _MODEL["m"]
    m.precision = precision
    return m


def _pockets(case, P, seed):
    """P pockets; ligand masks are arbitrary prefixes (the ligand rows stay padded either way)"""
    if case == "Ll==Lr":
        return O.synthetic_batch(P, 64, (5, 40), (16, 64), seed)
    if case == "Ll!=Lr":
        batch = O.synthetic_batch(P, 48, (1, 48), (1, 48), seed)
        rec = O.synthetic_batch(P, 112, (1, 112), (16, 112), seed + 1)
        for k in ("receptor_seq", "receptor_angles", "receptor_attn_mask"):
            batch[k] = rec[k]
        return batch
    assert case == "length-1-pocket"  # a pocket of one residue next to a full one
    batch = O.synthetic_batch(P, 128, (10, 90), (1, 1), seed)
    full = O.synthetic_batch(P, 128, (10, 90), (128, 128), seed + 1)
    for k in ("receptor_seq", "receptor_angles", "receptor_attn_mask"):
        batch[k][1] = full[k][1]
    return batch


def _replicated(batch, K):
    return {k: v.repeat_interleave(K, dim=0) for k, v in batch.items()}


def _stepwise(sd, m, batch, x_T, T, sched, tr, E=None, seed=None, gid0=None):
    """the loop's steps one by one: stand-alone forward() (every receptor row computed) + the single reverse step, with the
    explicit Exp(1) noise E or with the loop's Philox key (seed, global graph ids from gid0, step index)"""
    sd_lib, p = sd.lib(), sd._cabi.ptr
    B, L = x_T.shape[:2]
    dv = {k: v.to(DEV) for k, v in batch.items()}
    tables = sd.utils.loop_tables(T, sched, tr).to(DEV)
    x = x_T.to(DEV)
    for s_int in reversed(range(T)):
        s = s_int * torch.ones((B, 1))
        with torch.no_grad():
            lg = m(s.to(DEV), x, dv["ligand_angles"], dv["ligand_attn_mask"], dv["receptor_seq"], dv["receptor_angles"], dv["receptor_attn_mask"])
        if E is not None:
            x = sd.sample_p_zs_given_zt_discrete((s + 1) / T, s / T, x, lg, sched, tr, True, s_int == 0, noise_E=E[s_int])
        elif s_int == 0:
            x = lg
        else:
            nxt = torch.empty_like(x)
            stream = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
            assert sd_lib.seqdiff_reverse_step(p(tables[s_int:s_int + 1].contiguous()), 1, B, L, p(x), p(lg), 1, None, seed, gid0, s_int,
                                               p(nxt), None, stream) == 0
            x = nxt
    torch.cuda.synchronize()
    return x


def _sample(sd, m, batch, K, x_T, T, sched, tr, E=None, seed=None, gid0=None):
    """the loop, counting the library's launches of the call (a captured step graph adds the dry run's and the capture's)"""
    torch.cuda.synchronize()
    n0 = sd.lib().seqdiff_launch_count()
    out = sd.denoise_tensors(batch, m, sched, tr, True, timesteps=T, x_T=x_T, noise_E_steps=E, seed=seed, graph_id0=gid0,
                             num_samples=K).clone()
    torch.cuda.synchronize()
    return out, sd.lib().seqdiff_launch_count() - n0


@pytest.mark.parametrize("noise", ["exp1", "philox"])
@pytest.mark.parametrize("K", [1, 3])
@pytest.mark.parametrize("case", ["Ll==Lr", "Ll!=Lr", "length-1-pocket"])
@pytest.mark.parametrize("precision", ["bf16", "fp16"])
def test_padded_loop_equals_stepwise_forward(precision, case, K, noise):
    """K = 1 through seqdiff_sample_ex, K = 3 through seqdiff_sample_multi (against the stepwise run of the batch whose pockets
    are repeated K times: same graph ids, same noise)"""
    sd = sd_pkg()
    m = _model(precision)
    sd.sample.DEVICE = torch.device(DEV)
    T, P = 4, 3
    batch = _pockets(case, P, 91)
    Ll = batch["ligand_seq"].shape[1]
    g = torch.Generator().manual_seed(5)
    x_T = O.generate_discrete_noise(P * K, Ll, generator=g)
    E = torch.empty(T, P * K * Ll, 20).exponential_(1, generator=g) if noise == "exp1" else None
    sched, tr = sd.PredefinedNoiseScheduleDiscrete("cosine", T), sd.BlosumTransition(x_classes=20)
    final, _ = _sample(sd, m, batch, K, x_T, T, sched, tr, E=E, seed=17, gid0=300)
    want = _stepwise(sd, m, _replicated(batch, K), x_T, T, sched, tr, E=E, seed=17, gid0=300)
    assert torch.equal(final, want)


@pytest.mark.parametrize("K", [1, 3])
@pytest.mark.parametrize("precision", ["bf16", "fp16"])
def test_padded_receptor_positions_are_never_read(precision, K):
    """random finite values at the padded receptor positions of receptor_seq and receptor_angles: the loop's output, padded
    ligand positions included, is the zero-padded run's"""
    sd = sd_pkg()
    m = _model(precision)
    sd.sample.DEVICE = torch.device(DEV)
    T, P = 4, 4
    batch = _pockets("Ll!=Lr", P, 101)
    Ll = batch["ligand_seq"].shape[1]
    pad = batch["receptor_attn_mask"] == 0
    assert pad.any()
    g = torch.Generator().manual_seed(8)
    noisy = dict(batch)
    noisy["receptor_seq"] = torch.where(pad[..., None], torch.randn(batch["receptor_seq"].shape, generator=g) * 3, batch["receptor_seq"])
    noisy["receptor_angles"] = torch.where(pad[..., None], torch.randn(batch["receptor_angles"].shape, generator=g) * 3, batch["receptor_angles"])
    x_T = O.generate_discrete_noise(P * K, Ll, generator=g)
    sched, tr = sd.PredefinedNoiseScheduleDiscrete("cosine", T), sd.BlosumTransition(x_classes=20)
    clean, _ = _sample(sd, m, batch, K, x_T, T, sched, tr, seed=23, gid0=40)
    dirty, _ = _sample(sd, m, noisy, K, x_T, T, sched, tr, seed=23, gid0=40)
    assert torch.equal(clean, dirty)


def test_cached_graph_across_receptor_compositions():
    """the receptor lengths are part of the step graph's key: composition A captures, B captures, A again captures (one graph is
    cached), A once more replays.  Every call equals its own stepwise reference.  (A capture adds the dry-run forward's launches,
    and the first call of a new GEMM shape the tuner's, so the capturing calls differ among themselves.)"""
    sd = sd_pkg()
    m = _model("bf16")
    sd.sample.DEVICE = torch.device(DEV)
    T, P = 4, 4
    a, b = _pockets("Ll==Lr", P, 111), _pockets("Ll==Lr", P, 112)
    assert not torch.equal(a["receptor_attn_mask"], b["receptor_attn_mask"])
    sched, tr = sd.PredefinedNoiseScheduleDiscrete("cosine", T), sd.BlosumTransition(x_classes=20)
    g = torch.Generator().manual_seed(9)
    runs, results = [], []
    for i, batch in enumerate((a, b, a, a)):
        x_T = O.generate_discrete_noise(P, batch["ligand_seq"].shape[1], generator=g)
        final, n = _sample(sd, m, batch, 1, x_T, T, sched, tr, seed=30 + i, gid0=10 * i)
        runs.append(n)
        results.append((final, batch, x_T, 30 + i, 10 * i))
    for final, batch, x_T, seed, gid0 in results:
        assert torch.equal(final, _stepwise(sd, m, batch, x_T, T, sched, tr, seed=seed, gid0=gid0))
    assert min(runs[1], runs[2]) > runs[3], runs


@pytest.mark.parametrize("kind", ["hole", "empty-pocket", "fp32"])
def test_fallbacks_keep_the_padded_path(kind):
    """a receptor mask with a hole, a pocket with no valid receptor token, and the fp32 mode compute every receptor row: two calls
    whose receptor masks differ replay one graph (its key has no receptor lengths), and each equals its stepwise reference"""
    sd = sd_pkg()
    precision = "fp32" if kind == "fp32" else "bf16"
    m = _model(precision)
    sd.sample.DEVICE = torch.device(DEV)
    T, P = 4, 3
    sched, tr = sd.PredefinedNoiseScheduleDiscrete("cosine", T), sd.BlosumTransition(x_classes=20)
    g = torch.Generator().manual_seed(12)
    runs, results = [], []
    for i, seed in enumerate((121, 122, 122)):
        batch = _pockets("Ll==Lr", P, seed)
        if kind == "hole":
            batch["receptor_attn_mask"][1, 3] = 0.0
        elif kind == "empty-pocket":
            batch["receptor_attn_mask"][2] = 0.0
        x_T = O.generate_discrete_noise(P, batch["ligand_seq"].shape[1], generator=g)
        final, n = _sample(sd, m, batch, 1, x_T, T, sched, tr, seed=50 + i, gid0=7 * i)
        runs.append(n)
        results.append((final, batch, x_T, 50 + i, 7 * i))
    assert runs[1] == runs[2], runs
    for final, batch, x_T, seed, gid0 in results:
        assert torch.equal(final, _stepwise(sd, m, batch, x_T, T, sched, tr, seed=seed, gid0=gid0))
