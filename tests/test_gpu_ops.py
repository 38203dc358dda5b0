"""GPU parity tests of the individual kernels, called through the C ABI (ctypes) and checked against the
oracle / a plain torch fp32 restatement of the same op."""
import ctypes
import glob
import math
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from helpers import BF16, FP16, FP32, GOLDEN, O, assert_indices_match, rel_err, sd_pkg, stream_ptr

pytestmark = pytest.mark.gpu
DEV = "cuda:0"


def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _check(rc):
    if rc != 0:
        raise RuntimeError(sd_pkg().lib().seqdiff_last_error().decode())


# ---------------------------------------------------------------------------------------------------
def _gemm_ref(A, W, bias, resid, epi):
    y = A.float() @ W.float().t() + bias
    if epi == 1:
        y = F.gelu(y)
    elif epi == 2:
        y = F.silu(y)
    if resid is not None:
        y = y + resid.float()
    return y


GEMM_SHAPES = [
    # M, N, K  (the denoiser's own shapes at small / ragged / full token counts)
    (128, 768, 768), (64, 768, 768), (200, 2304, 768), (8192, 768, 768), (300, 4608, 768), (256, 3072, 768),
    (256, 768, 3072), (384, 1024, 768), (130, 768, 1024), (512, 9216, 768), (1, 768, 768), (8192, 1024, 768),
]


_TDT = {BF16: (torch.bfloat16, torch.bfloat16), FP16: (torch.float16, torch.float16)}


@pytest.mark.parametrize("M,N,K", GEMM_SHAPES)
@pytest.mark.parametrize("bn", [0, 128, 192, 256])
@pytest.mark.parametrize("cg2", [0, 1])
@pytest.mark.parametrize("mode", [BF16, FP16])
def test_gemm_tcgen05(M, N, K, bn, cg2, mode):
    """tcgen05/TMA GEMM: 16-bit operands in each format mix; epilogues none/GELU/SiLU -> 16-bit out;
    fp32 residual add -> fp32 out (the LayerNorm-input variant)."""
    if mode != BF16 and (bn != 0 or M > 1024):
        pytest.skip("format variants share the tile code; checked at the auto tile width on the small shapes")
    if cg2 and bn == 0:
        pytest.skip("auto selection is exercised by the cg2=0 / bn=0 case; cg2=1 forces the CTA-pair kernel per tile width")
    if bn and N % bn:
        pytest.skip("tile width does not divide N")
    lib = sd_pkg().lib()
    adt, wdt = _TDT[mode]
    g = torch.Generator(device="cpu").manual_seed(M * 7 + N + K + bn)
    A = (torch.randn(M, K, generator=g)).to(DEV).to(adt)
    W = (torch.randn(N, K, generator=g) / math.sqrt(K)).to(DEV).to(wdt)
    bias = torch.randn(N, generator=g).to(DEV)
    resid = torch.randn(M, N, generator=g).to(DEV)
    for epi, r in ((0, None), (1, None), (2, None), (0, resid)):
        C = torch.full((M, N), float("nan"), device=DEV, dtype=torch.float32 if r is not None else adt)
        _check(lib.seqdiff_op_gemm(mode | (bn << 8) | (cg2 << 20), M, N, K, _p(A), _p(W), _p(bias), _p(r), epi, _p(C), stream_ptr()))
        torch.cuda.synchronize()
        ref = _gemm_ref(A, W, bias, r, epi)
        err = (C.float() - ref).abs().max().item()
        scale = ref.abs().max().item()
        assert torch.isfinite(C.float()).all(), f"non-finite output epi={epi}"
        tol = 2e-5 if r is not None else (1.0 / 128 if adt == torch.bfloat16 else 1.0 / 1024)
        assert err <= tol * scale + 1e-3 * (r is None), f"M{M} N{N} K{K} bn{bn} cg2{cg2} mode{mode} epi{epi} resid{r is not None}: err {err} scale {scale}"


@pytest.mark.parametrize("M,N,K", [(768, 768, 8192), (2304, 768, 1000), (768, 1024, 16), (4608, 768, 4096), (1024, 768, 333), (768, 3072, 2048), (128, 128, 64)])
@pytest.mark.parametrize("split", [1, -1, 5])
@pytest.mark.parametrize("mode", [BF16, FP16])
def test_gemm_tn_wgrad(M, N, K, split, mode):
    """C[M,N] = At^T Bt with At [K,M], Bt [K,N] row-major (both operands MN-major for tcgen05): the weight-gradient product of the
    training step read in place -- against an fp32 matmul of the same 16-bit values.  Ragged token counts K (TMA zero fill), split-K
    (atomic accumulation into a zeroed C) and one k-block cases."""
    if mode != BF16 and K > 2048:
        pytest.skip("format variants share the tile code")
    lib = sd_pkg().lib()
    dt = _TDT[mode][0]
    g = torch.Generator(device="cpu").manual_seed(M + 3 * N + 7 * K)
    At = torch.randn(K, M, generator=g).to(DEV).to(dt)
    Bt = (torch.randn(K, N, generator=g) / math.sqrt(K)).to(DEV).to(dt)
    C = torch.zeros(M, N, device=DEV)
    _check(lib.seqdiff_op_gemm_tn(mode, M, N, K, _p(At), _p(Bt), _p(C), split, stream_ptr()))
    torch.cuda.synchronize()
    ref = At.float().t() @ Bt.float()
    err = (C - ref).abs().max().item()
    assert torch.isfinite(C).all() and err <= 2e-5 * ref.abs().max().item() + 1e-5 * math.sqrt(K), f"M{M} N{N} K{K} split{split}: err {err} scale {ref.abs().max().item()}"


@pytest.mark.parametrize("M,N,K", [(128, 768, 768), (77, 2304, 768), (33, 20, 768), (64, 768, 3072)])
def test_gemm_fp32(M, N, K):
    lib = sd_pkg().lib()
    g = torch.Generator().manual_seed(M + N + K)
    A = torch.randn(M, K, generator=g).to(DEV)
    W = (torch.randn(N, K, generator=g) / math.sqrt(K)).to(DEV)
    bias = torch.randn(N, generator=g).to(DEV)
    resid = torch.randn(M, N, generator=g).to(DEV)
    for epi, r in ((0, None), (1, None), (2, None), (0, resid)):
        C = torch.empty(M, N, device=DEV)
        _check(lib.seqdiff_op_gemm(FP32, M, N, K, _p(A), _p(W), _p(bias), _p(r), epi, _p(C), stream_ptr()))
        ref = _gemm_ref(A.double(), W.double(), bias.double(), None if r is None else r.double(), epi) if False else None
        ref = (A.double() @ W.double().t() + bias.double())
        ref = F.gelu(ref) if epi == 1 else F.silu(ref) if epi == 2 else ref
        if r is not None:
            ref = ref + r.double()
        assert rel_err(C, ref.float()) < 2e-6


# ---------------------------------------------------------------------------------------------------
ATTN_CASES = [
    # B, heads, Lq, Lk, P, rel
    (2, 12, 128, 128, 128, True), (3, 12, 64, 64, 64, True), (2, 12, 128, 128, 128, False), (2, 12, 64, 128, 128, False),
    (2, 4, 100, 100, 128, True), (1, 12, 512, 512, 512, True), (2, 12, 48, 464, 512, False), (2, 2, 17, 17, 32, True),
    # more work items than SMs: several items per persistent CTA (pipelined kernel), one and several key blocks
    (40, 12, 128, 128, 128, True), (40, 12, 128, 128, 128, False), (5, 12, 300, 300, 512, True), (7, 12, 200, 464, 512, False),
]


def test_attention_small_grid_subprocess():
    """the persistent kernel with only 3 CTAs: every CTA walks a long item list."""
    import subprocess, sys
    env = dict(os.environ, SEQDIFF_ATTN_GRID="3")
    r = subprocess.run([sys.executable, "-m", "pytest", __file__, "-q", "-m", "gpu", "-k", "test_attention and not subprocess", "-p",
                        "no:cacheprovider"], env=env, capture_output=True, text=True)
    assert r.returncode == 0, "SEQDIFF_ATTN_GRID=3:\n" + r.stdout[-2000:]


@pytest.mark.parametrize("B,heads,Lq,Lk,P,rel", ATTN_CASES)
@pytest.mark.parametrize("prec", [FP32, BF16, FP16])
def test_attention(B, heads, Lq, Lk, P, rel, prec):
    lib = sd_pkg().lib()
    H = heads * 64
    g = torch.Generator().manual_seed(B + heads + Lq + Lk)
    dt = {FP32: torch.float32, BF16: torch.bfloat16, FP16: torch.float16}[prec]
    # q,k,v packed like the fused QKV GEMM output: [B, L, 3H] with row stride 3H (self) or separate (cross)
    q = torch.randn(B, Lq, H, generator=g).to(DEV).to(dt)
    k = torch.randn(B, Lk, H, generator=g).to(DEV).to(dt)
    v = torch.randn(B, Lk, H, generator=g).to(DEV).to(dt)
    E = (torch.randn(2 * P - 1, 64, generator=g) * 0.5).to(DEV).to(dt) if rel else None
    nk = torch.randint(1, Lk + 1, (B,), generator=g)
    mask = (torch.arange(Lk)[None, :] < nk[:, None]).float().to(DEV)
    out = torch.full((B, Lq, H), float("nan"), device=DEV, dtype=dt)
    _check(lib.seqdiff_op_attention(prec, B, heads, Lq, Lk, _p(q), H, _p(k), H, _p(v), H, _p(E), P, _p(mask), _p(out), stream_ptr()))
    torch.cuda.synchronize()
    cfg = O.OracleConfig(hidden_size=H, num_attention_heads=heads, max_position_embeddings=P)
    ref = O.attention_core(cfg, q.float().cpu(), k.float().cpu(), v.float().cpu(), O.extend_mask(mask.cpu()),
                           None if E is None else E.float().cpu())
    assert torch.isfinite(out.float()).all()
    tol = {FP32: 2e-5, BF16: 2e-2, FP16: 3e-3}[prec]
    assert rel_err(out, ref) < tol, rel_err(out, ref)


@pytest.mark.parametrize("rel", [True, False])
@pytest.mark.parametrize("L", [128, 300])
def test_attention_mask_patterns(rel, L):
    """Key masks that are not a prefix: the kernel skips 32-key chunks without an unmasked key (their probabilities underflow
    to exactly 0 under the reference's additive -10000), so chunk boundaries, holes, a masked first chunk and whole masked
    key blocks must all still match the oracle."""
    lib = sd_pkg().lib()
    heads, P = 4, 512
    H = heads * 64
    pats = []
    ar = torch.arange(L)
    pats.append(ar >= L - 5)                      # only the last keys (first chunks / blocks fully masked)
    pats.append(ar % 2 == 0)                      # holes everywhere
    pats.append((ar >= 40) & (ar < 50))           # one island inside chunk 1
    pats.append(ar < 32)                          # exactly one chunk
    pats.append(ar < 33)                          # one key into the second chunk
    pats.append((ar >= 32) & (ar < 64))           # chunk 0 masked, chunk 1 live
    pats.append(ar == min(L - 1, 129))            # a single key (second key block when L > 128)
    pats.append(torch.ones(L, dtype=torch.bool))
    B = len(pats)
    mask = torch.stack(pats).float().to(DEV)
    g = torch.Generator().manual_seed(L + int(rel))
    q = torch.randn(B, L, H, generator=g).to(DEV).bfloat16()
    k = torch.randn(B, L, H, generator=g).to(DEV).bfloat16()
    v = torch.randn(B, L, H, generator=g).to(DEV).bfloat16()
    E = (torch.randn(2 * P - 1, 64, generator=g) * 0.5).to(DEV).bfloat16() if rel else None
    out = torch.full((B, L, H), float("nan"), device=DEV, dtype=torch.bfloat16)
    _check(lib.seqdiff_op_attention(BF16, B, heads, L, L, _p(q), H, _p(k), H, _p(v), H, _p(E), P, _p(mask), _p(out), stream_ptr()))
    torch.cuda.synchronize()
    cfg = O.OracleConfig(hidden_size=H, num_attention_heads=heads, max_position_embeddings=P)
    ref = O.attention_core(cfg, q.float().cpu(), k.float().cpu(), v.float().cpu(), O.extend_mask(mask.cpu()), None if E is None else E.float().cpu())
    assert torch.isfinite(out.float()).all()
    for b in range(B):
        assert rel_err(out[b], ref[b]) < 2e-2, (b, rel_err(out[b], ref[b]))


@pytest.mark.parametrize("rel", [True, False])
@pytest.mark.parametrize("prec", [BF16, FP16])
def test_attention_pipelined_repeatable(rel, prec):
    """The pipelined kernel hands buffers between roles through mbarriers; a missing edge shows up as a timing-dependent
    difference.  Same inputs, 40 launches under varying cache state / co-running work: every output must be bit-identical."""
    lib = sd_pkg().lib()
    B, heads, L, P = 37, 12, 128, 128
    H = heads * 64
    g = torch.Generator().manual_seed(11 + int(rel))
    dt = {BF16: torch.bfloat16, FP16: torch.float16}[prec]
    qkv = torch.randn(B * L, 3 * H, generator=g).to(DEV).to(dt)
    E = (torch.randn(2 * P - 1, 64, generator=g) * 0.5).to(DEV).to(dt) if rel else None
    nk = torch.randint(1, L + 1, (B,), generator=g)
    mask = (torch.arange(L)[None, :] < nk[:, None]).float().to(DEV)
    junk = torch.empty(64 << 20, dtype=torch.uint8, device=DEV)
    first = None
    for i in range(40):
        out = torch.full((B, L, H), float("nan"), device=DEV, dtype=dt)
        if i % 3 == 1:
            junk.zero_()  # cold L2
        _check(lib.seqdiff_op_attention(prec, B, heads, L, L, _p(qkv), 3 * H, _p(qkv[:, H:]), 3 * H, _p(qkv[:, 2 * H:]), 3 * H, _p(E), P,
                                        _p(mask), _p(out), stream_ptr()))
        if i % 3 == 2:
            junk.zero_()  # memory traffic right behind the launch
        torch.cuda.synchronize()
        if first is None:
            first = out
            q, k, v = (qkv[:, j * H:(j + 1) * H].float().cpu().view(B, L, H) for j in range(3))
            cfg = O.OracleConfig(hidden_size=H, num_attention_heads=heads, max_position_embeddings=P)
            ref = O.attention_core(cfg, q, k, v, O.extend_mask(mask.cpu()), None if E is None else E.float().cpu())
            assert rel_err(out, ref) < {BF16: 2e-2, FP16: 3e-3}[prec]
        else:
            assert torch.equal(out, first), f"launch {i} differs from launch 0"


# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("path", sorted(glob.glob(os.path.join(GOLDEN, "reverse_step_*.pt"))), ids=os.path.basename)
def test_reverse_step_golden(path):
    """Teacher-forced step against the golden vectors of the reference's own function."""
    sd = sd_pkg()
    g = torch.load(path, weights_only=False)
    if g["s_int"] == 0:
        out = sd.sample_p_zs_given_zt_discrete(None, None, None, g["logits"].to(DEV), None, None, True, True)
        assert torch.equal(out.cpu(), g["out"])  # last step: raw logits (quirk Q4)
        return
    T, s_int = g["T"], g["s_int"]
    sched = sd.PredefinedNoiseScheduleDiscrete("cosine", T)
    tr = sd.BlosumTransition(x_classes=20) if g["kind"] == "blosum" else sd.DiscreteUniformTransition(20)
    x = F.one_hot(g["x_t_idx"].long(), 20).float()
    B = x.shape[0]
    s = s_int * torch.ones((B, 1))
    out = sd.sample_p_zs_given_zt_discrete((s + 1) / T, s / T, x.to(DEV), g["logits"].to(DEV), sched, tr, g["diverse"], False,
                                           noise_E=g["E"])
    assert out.shape == x.shape and torch.equal(out.sum(-1).cpu(), torch.ones(B, x.shape[1]))
    score = g["prob"] / g["E"] if g["diverse"] else g["prob"]
    assert_indices_match(out.argmax(-1), g["out"], score, os.path.basename(path))


def test_reverse_step_bulk_vs_oracle():
    """cfg-2-sized step (B=64, L=128, 8192 residues) + per-graph tables + non-one-hot rows."""
    sd = sd_pkg()
    T = 500
    B, L = 64, 128
    g = torch.Generator().manual_seed(11)
    x = F.one_hot(torch.randint(0, 20, (B, L), generator=g), 20).float()
    logits = torch.randn(B, L, 20, generator=g) * 4
    E = torch.empty(B * L, 20).exponential_(1, generator=g)
    s = torch.randint(1, T, (B, 1), generator=g).float()  # a different step per graph
    o_s, o_t = O.NoiseScheduleDiscrete("cosine", T), O.BlosumTransition()
    want = O.reverse_step((s + 1) / T, s / T, x, logits, o_s, o_t, True, False, E)
    prob = O.reverse_step_probs((s + 1) / T, s / T, x, logits, o_s, o_t)
    got = sd.sample_p_zs_given_zt_discrete((s + 1) / T, s / T, x.to(DEV), logits.to(DEV), sd.PredefinedNoiseScheduleDiscrete("cosine", T),
                                           sd.BlosumTransition(x_classes=20), True, False, noise_E=E)
    assert_indices_match(got.argmax(-1), want.argmax(-1), prob / E, "bulk")
    # general (soft) x_t rows follow the dot-product formula of sample.py:129-138
    xs = torch.softmax(torch.randn(2, 16, 20, generator=g), -1)
    lg = torch.randn(2, 16, 20, generator=g)
    s2 = torch.tensor([[7.0], [300.0]])
    want2 = O.reverse_step((s2 + 1) / T, s2 / T, xs, lg, o_s, o_t, False, False)
    got2 = sd.sample_p_zs_given_zt_discrete((s2 + 1) / T, s2 / T, xs.to(DEV), lg.to(DEV), sd.PredefinedNoiseScheduleDiscrete("cosine", T),
                                            sd.BlosumTransition(x_classes=20), False, False)
    assert_indices_match(got2.argmax(-1), want2.argmax(-1), O.reverse_step_probs((s2 + 1) / T, s2 / T, xs, lg, o_s, o_t), "soft", 1e-4)


def _philox_ref(seed, graph, residue, step, call):
    M0, M1, W0, W1 = 0xD2511F53, 0xCD9E8D57, 0x9E3779B9, 0xBB67AE85
    c = [residue, (step * 8 + call) & 0xFFFFFFFF, graph & 0xFFFFFFFF, graph >> 32]
    k0, k1 = seed & 0xFFFFFFFF, seed >> 32
    for _ in range(10):
        p0, p1 = M0 * c[0], M1 * c[2]
        c = [((p1 >> 32) ^ c[1] ^ k0) & 0xFFFFFFFF, p1 & 0xFFFFFFFF, ((p0 >> 32) ^ c[3] ^ k1) & 0xFFFFFFFF, p0 & 0xFFFFFFFF]
        k0, k1 = (k0 + W0) & 0xFFFFFFFF, (k1 + W1) & 0xFFFFFFFF
    return c


def test_philox_stream_is_counter_based_and_shard_invariant():
    lib = sd_pkg().lib()
    seed, B, L, step = 0x1234_5678_9ABC_DEF0, 4, 33, 17
    out = torch.zeros(B * L * 20, dtype=torch.int32, device=DEV)
    _check(lib.seqdiff_op_philox_u32(seed, 100, step, B, L, _p(out), stream_ptr()))
    w = out.cpu().numpy().astype(np.uint32).reshape(B, L, 20)
    # Philox4x32-10 known-answer test (Random123 kat_vectors: ctr=key=0 -> 6627e8d5 e169c58d bc57ac4c 9b00dbd8)
    assert _philox_ref(0, 0, 0, 0, 0) == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]
    for b, l, call in ((0, 0, 0), (3, 32, 4), (1, 7, 2)):
        assert list(w[b, l, call * 4:call * 4 + 4]) == _philox_ref(seed, 100 + b, l, step, call)
    # the same graphs drawn as a different shard (graph_id0 = 102, B = 2) give the same words
    out2 = torch.zeros(2 * L * 20, dtype=torch.int32, device=DEV)
    _check(lib.seqdiff_op_philox_u32(seed, 102, step, 2, L, _p(out2), stream_ptr()))
    assert np.array_equal(out2.cpu().numpy().astype(np.uint32).reshape(2, L, 20), w[2:4])


def test_reverse_step_philox_statistics():
    """In-kernel noise: sampled class frequencies follow the posterior (chi-square-ish bound)."""
    sd = sd_pkg()
    T, B, L = 50, 64, 512
    x = F.one_hot(torch.full((B, L), 3), 20).float()
    logits = torch.zeros(B, L, 20)
    logits[..., 5] = 2.0
    s = torch.full((B, 1), 20.0)
    prob = O.reverse_step_probs((s + 1) / T, s / T, x, logits, O.NoiseScheduleDiscrete("cosine", T), O.BlosumTransition())[0]
    got = sd.sample_p_zs_given_zt_discrete((s + 1) / T, s / T, x.to(DEV), logits.to(DEV), sd.PredefinedNoiseScheduleDiscrete("cosine", T),
                                           sd.BlosumTransition(x_classes=20), True, False)
    freq = got.reshape(-1, 20).mean(0).cpu()
    n = B * L
    assert ((freq - prob).abs() < 5 * torch.sqrt(prob * (1 - prob) / n) + 1e-4).all(), (freq, prob)


def _exp1_from_words(w_u32):
    """Host restatement of how the kernels turn a Philox word into the Exp(1) race noise: u = ((w >> 9) + 0.5) * 2^-23, E = -ln u
    (float64 here; the exact-mode kernel uses fp32 logf, the production kernel lg2.approx / a series near u = 1)."""
    u = ((w_u32.astype(np.uint64) >> np.uint64(9)).astype(np.float64) + 0.5) * 2.0 ** -23
    return -np.log(u)


@pytest.mark.parametrize("B,L,T,per_graph", [(64, 128, 500, False), (64, 128, 500, True), (256, 512, 50, False)], ids=["cfg2", "cfg2-per-graph-t", "cfg3"])
def test_reverse_step_philox_pinned_to_oracle(B, L, T, per_graph):
    """The PRODUCTION variant of the reverse step -- reverse_step_kernel<FAST = true>: in-kernel Philox noise, FMA-contracted
    posterior, ex2 / lg2 / rcp.approx, normalisations skipped -- pinned to the oracle (sample.py:141-179): the Philox words the
    kernel consumes are pulled through seqdiff_op_philox_u32, turned into E ~ Exp(1) on the host, handed to the oracle as its
    multinomial noise, and the sampled indices must agree bit for bit except at near-ties of the reference's own race scores
    (top-2 margin < 1e-5 relative).  cfg-2- and cfg-3-sized batches; shared and per-graph step tables."""
    sd = sd_pkg()
    lib = sd.lib()
    seed, gid0 = 0xC0FFEE1234, 7_000_000_123
    g = torch.Generator().manual_seed(B + L + T)
    x = F.one_hot(torch.randint(0, 20, (B, L), generator=g), 20).float()
    logits = torch.randn(B, L, 20, generator=g) * 3
    s = torch.randint(1, T, (B, 1), generator=g).float() if per_graph else torch.full((B, 1), float(T // 3))
    sched, tr = sd.PredefinedNoiseScheduleDiscrete("cosine", T), sd.BlosumTransition(x_classes=20)
    sd.sample.DEVICE = torch.device(DEV)
    old_seed, old_calls = sd.sample.SEED, sd.sample._CALLS[0]
    try:
        sd.sample.SEED = seed
        got = sd.sample_p_zs_given_zt_discrete((s + 1) / T, s / T, x.to(DEV), logits.to(DEV), sched, tr, True, False, graph_id0=gid0)
        step = sd.sample._CALLS[0] & 0x0FFFFFFF
    finally:
        sd.sample.SEED = old_seed
    assert step == old_calls + 1
    words = torch.zeros(B * L * 20, dtype=torch.int32, device=DEV)
    _check(lib.seqdiff_op_philox_u32(seed, gid0, step, B, L, _p(words), stream_ptr()))
    E = torch.from_numpy(_exp1_from_words(words.cpu().numpy().view(np.uint32))).float().reshape(B * L, 20)
    o_s, o_t = O.NoiseScheduleDiscrete("cosine", T), O.BlosumTransition()
    want = O.reverse_step((s + 1) / T, s / T, x, logits, o_s, o_t, True, False, E)
    prob = O.reverse_step_probs((s + 1) / T, s / T, x, logits, o_s, o_t)
    n_flip = assert_indices_match(got.argmax(-1), want.argmax(-1), prob / E, f"philox {B}x{L}")
    print(f"philox-mode reverse step {B}x{L}: {n_flip} near-tie flips of {B * L}")
    assert torch.equal(got.sum(-1).cpu(), torch.ones(B, L))


def test_inv_exp1_near_one_is_finite_and_accurate():
    """ADVICE r1: lg2.approx has 2^-22 absolute error, so -log2(u) for u -> 1 could come out 0 / negative (inf / NaN race scores).
    Drive the production kernel with posteriors where EVERY class has the same probability, so the winner is decided by the noise
    alone, over enough residues that words with u > 1 - 2^-20 occur (~2.6e6 draws): it must match the oracle's argmin of E."""
    sd = sd_pkg()
    lib = sd.lib()
    T, B, L = 50, 256, 512
    seed, gid0, = 99, 0
    x = F.one_hot(torch.zeros(B, L, dtype=torch.long), 20).float()
    logits = torch.zeros(B, L, 20)
    s = torch.full((B, 1), 2.0)
    sched, tr = sd.PredefinedNoiseScheduleDiscrete("cosine", T), sd.BlosumTransition(x_classes=20)
    sd.sample.DEVICE = torch.device(DEV)
    old = sd.sample.SEED
    try:
        sd.sample.SEED = seed
        got = sd.sample_p_zs_given_zt_discrete((s + 1) / T, s / T, x.to(DEV), logits.to(DEV), sched, tr, True, False, graph_id0=gid0)
        step = sd.sample._CALLS[0] & 0x0FFFFFFF
    finally:
        sd.sample.SEED = old
    words = torch.zeros(B * L * 20, dtype=torch.int32, device=DEV)
    _check(lib.seqdiff_op_philox_u32(seed, gid0, step, B, L, _p(words), stream_ptr()))
    w = words.cpu().numpy().view(np.uint32)
    assert ((w >> 9) >= (1 << 23) - 8).sum() > 0, "no word close to u = 1 in this sample: enlarge it"
    E = torch.from_numpy(_exp1_from_words(w)).float().reshape(B * L, 20)
    o_s, o_t = O.NoiseScheduleDiscrete("cosine", T), O.BlosumTransition()
    prob = O.reverse_step_probs((s + 1) / T, s / T, x, logits, o_s, o_t)
    want = O.reverse_step((s + 1) / T, s / T, x, logits, o_s, o_t, True, False, E)
    assert_indices_match(got.argmax(-1), want.argmax(-1), prob / E, "near-one noise")


def test_apply_aa_noise_golden():
    sd = sd_pkg()
    g = torch.load(os.path.join(GOLDEN, "apply_aa_noise.pt"), weights_only=False)
    x0 = (F.one_hot(g["x0_idx"].long(), 20).float() * g["x0_valid"].float()[..., None]).to(DEV)
    p = sd.PeptideDiff(sd.BertConfig(max_position_embeddings=32, intermediate_size=1024, num_hidden_layers=1),
                       sd.BertConfig(max_position_embeddings=32, intermediate_size=1024, num_hidden_layers=1), list(sd.AA_VOCAB),
                       torch.nn.CrossEntropyLoss(), "cosine", g["T"])
    out = p.apply_aa_noise(x0, g["t_int"], noise_E=g["E"])
    probs = O.apply_aa_noise_probs(x0.cpu(), g["t_int"], g["T"], O.NoiseScheduleDiscrete("cosine", g["T"]), O.BlosumTransition())
    assert_indices_match(out.argmax(-1), g["out_idx"], probs / g["E"], "apply_aa_noise")
    pad = g["x0_valid"] == 0
    assert (out.argmax(-1).cpu()[pad] == 0).all()  # padded rows -> class 0 (model.py:307-308)


@pytest.mark.parametrize("ext,max_len", [(0, 128), (1, 128), (3, 160), (7, 512)])
def test_collate_matches_reference_dataset(ext, max_len):
    """seqdiff_collate == LigandBindingSiteDataset.__getitem__ (dataset.py:97-129), bit for bit: the golden values produced
    by the reference class itself, and the oracle restatement on every item of a wider set (tiny and >256-residue complexes)."""
    sd = sd_pkg()
    recs = O.synthetic_records(6, 41)
    g = torch.load(os.path.join(GOLDEN, "dataset_items.pt"), weights_only=False)
    if (ext, max_len) in g["cases"]:
        got = sd.collate_complexes(recs, max_len, ext, DEV)
        want = g["cases"][(ext, max_len)]
        assert torch.equal(got["receptor_seq"].argmax(-1).to(torch.uint8).cpu(), want["receptor_seq_idx"])
        assert torch.equal(got["ligand_seq"].argmax(-1).to(torch.uint8).cpu(), want["ligand_seq_idx"])
        assert torch.equal(got["receptor_angles"].double().sum(-1).cpu(), want["receptor_angle_sum"])
        assert torch.equal(got["receptor_length"].long(), want["receptor_length"]) and torch.equal(got["ligand_length"].long(), want["ligand_length"])
        assert got["structure_ids"]["pdb_id"][:2] == ["c000", "c001"]
    recs = recs + O.synthetic_records(9, 5, n_lo=3, n_hi=700)
    big = 512  # roomy enough for 700 residues x 15 % pocket x 3 (dilation)
    got = sd.collate_complexes(recs, big, ext, DEV)
    for i, r in enumerate(recs):
        want = O.dataset_item(r, big, ext)
        for k in ("ligand_angles", "ligand_seq", "ligand_attn_mask", "receptor_angles", "receptor_seq", "receptor_attn_mask"):
            assert torch.equal(got[k][i].cpu(), want[k]), (i, k)
        assert int(got["ligand_length"][i]) == int(want["ligand_length"]) and int(got["receptor_length"][i]) == int(want["receptor_length"])
    with pytest.raises(RuntimeError, match="Length exceed"):  # dataset.py:42-43
        sd.collate_complexes(recs, 8, ext, DEV)


def test_reverse_step_cfg3_size_properties():
    """BASELINE cfg 3 size (256 graphs x 512 residues): one-hot output, determinism, agreement with the oracle on a slice."""
    sd = sd_pkg()
    T, B, L = 50, 256, 512
    g = torch.Generator().manual_seed(2)
    x = F.one_hot(torch.randint(0, 20, (B, L), generator=g), 20).float().to(DEV)
    logits = (torch.randn(B, L, 20, generator=g) * 3).to(DEV)
    E = torch.empty(B * L, 20).exponential_(1, generator=g).to(DEV)
    s = torch.full((B, 1), 31.0)
    sched, tr = sd.PredefinedNoiseScheduleDiscrete("cosine", T), sd.BlosumTransition(x_classes=20)
    a = sd.sample_p_zs_given_zt_discrete((s + 1) / T, s / T, x, logits, sched, tr, True, False, noise_E=E)
    b = sd.sample_p_zs_given_zt_discrete((s + 1) / T, s / T, x, logits, sched, tr, True, False, noise_E=E)
    assert torch.equal(a, b) and torch.equal(a.sum(-1), torch.ones(B, L, device=DEV)) and ((a == 0) | (a == 1)).all()
    sl = slice(100, 104)
    want = O.reverse_step((s[sl] + 1) / T, s[sl] / T, x[sl].cpu(), logits[sl].cpu(), O.NoiseScheduleDiscrete("cosine", T), O.BlosumTransition(),
                          True, False, E.view(B, L, 20)[sl].reshape(-1, 20).cpu())
    prob = O.reverse_step_probs((s[sl] + 1) / T, s[sl] / T, x[sl].cpu(), logits[sl].cpu(), O.NoiseScheduleDiscrete("cosine", T), O.BlosumTransition())
    assert_indices_match(a[sl].argmax(-1), want.argmax(-1), prob / E.view(B, L, 20)[sl].reshape(-1, 20).cpu(), "cfg3 slice")


@pytest.mark.parametrize("M,H", [(1, 768), (77, 768), (8192, 768), (300, 256), (129, 1024)])
def test_layernorm_op(M, H):
    """seqdiff_op_layernorm == F.layer_norm (fp32 exactly to rounding; 16-bit outputs to one operand ulp); statistics = (mean, rstd)."""
    sd = sd_pkg()
    lib = sd.lib()
    g = torch.Generator().manual_seed(M + H)
    x = (torch.randn(M, H, generator=g) * 3 + 0.5).to(DEV)
    w = (1 + 0.1 * torch.randn(H, generator=g)).to(DEV)
    b = (0.1 * torch.randn(H, generator=g)).to(DEV)
    ref = F.layer_norm(x, (H,), w, b, 1e-12)
    y32 = torch.empty(M, H, device=DEV)
    st = torch.empty(M, 2, device=DEV)
    _check(lib.seqdiff_op_layernorm(FP32, M, H, _p(x), _p(w), _p(b), 1e-12, _p(y32), None, _p(st), stream_ptr()))
    assert (y32 - ref).abs().max().item() < 2e-5
    assert torch.allclose(st[:, 0], x.mean(1), atol=1e-5) and torch.allclose(st[:, 1], 1 / torch.sqrt(x.var(1, unbiased=False) + 1e-12), rtol=1e-4)
    for prec, dt, tol in ((BF16, torch.bfloat16, 2 ** -8), (FP16, torch.float16, 2 ** -11)):
        y16 = torch.empty(M, H, device=DEV, dtype=dt)
        _check(lib.seqdiff_op_layernorm(prec, M, H, _p(x), _p(w), _p(b), 1e-12, None, _p(y16), None, stream_ptr()))
        assert ((y16.float() - ref).abs() <= tol * ref.abs() + 1e-5).all()
