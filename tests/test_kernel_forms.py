"""Operator-level parity tests of the kernel forms the model reaches only through its own loops: the GEMM whose residual is a LayerNorm
rebuilt in the epilogue (RESID = 2), the split-K fp32 GEMM of the weight gradients, and the packed / shared-key attention -- through
seqdiff_op_gemm_ex and seqdiff_op_attention_packed.  References are float64 on the host, computed from the same 16-bit values the
kernels read.  Every output buffer carries PAD extra rows of NaN that must still be NaN afterwards.  Two exactness claims the packed,
multi-sample and receptor-rows loops rest on are asserted with torch.equal: a GEMM row does not depend on M or on the tile
configuration, and packed attention equals the padded kernel at every valid row."""
import ctypes
import math
import os
import subprocess
import sys

import pytest
import torch

from helpers import BF16, FP16, FP32, O, rel_err, sd_pkg, stream_ptr

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
PAD = 16
DT = {BF16: torch.bfloat16, FP16: torch.float16, FP32: torch.float32}
TILES = [(0, 0), (128, 0), (192, 0), (256, 0), (128, 1), (192, 1), (256, 1)]  # (bn, cg2); (0, 0) = the tuner / cost model


def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _check(rc):
    if rc != 0:
        raise RuntimeError(sd_pkg().lib().seqdiff_last_error().decode())


def _nan(rows, cols, dtype):
    return torch.full((rows + PAD, cols), float("nan"), device=DEV, dtype=dtype)


def _assert_pad_untouched(C, rows):
    assert torch.isnan(C[rows:].float()).all(), "a row past the output was written"


def _gemm_ex(mode, bn, cg2, M, N, K, A, W, bias, C, resid=None, ln=None, epi=0, out_f32=False, split=1):
    st, g, b = ln if ln is not None else (None, None, None)
    _check(sd_pkg().lib().seqdiff_op_gemm_ex(mode | (bn << 8) | (cg2 << 20), M, N, K, _p(A), _p(W), _p(bias), _p(resid), _p(st), _p(g),
                                             _p(b), epi, int(out_f32), split, _p(C), stream_ptr()))


# ---------------------------------------------------------------------------------------------------
# GEMM operands, shared by every M and tile of a (mode, N, K): row i of A, o and the LayerNorm stats is the same at every M, so the
# float64 product is computed once at the largest M and sliced (four sets, ~100 MB of host float64 each)
MAXM = 8192
_CACHE = {}


def _operands(mode, N, K):
    key = (mode, N, K)
    if key not in _CACHE:
        g = torch.Generator().manual_seed(1000 * mode + N + K)
        A = torch.randn(MAXM, K, generator=g).to(DT[mode])
        W = (torch.randn(N, K, generator=g) / math.sqrt(K)).to(DT[mode])
        bias = torch.randn(N, generator=g)
        o = torch.randn(MAXM, N, generator=g) * 3 + 0.5      # the fp32 residual stream before its LayerNorm
        gamma = 1 + 0.1 * torch.randn(N, generator=g)         # distinct per column: a chunk / column mix-up shows
        beta = 0.1 * torch.randn(N, generator=g)
        d = dict(A=A.to(DEV), W=W.to(DEV), bias=bias.to(DEV), o=o.to(DEV), gamma=gamma.to(DEV), beta=beta.to(DEV),
                 prod=A.double() @ W.double().t() + bias.double())
        st = torch.empty(MAXM, 2, device=DEV)
        ln32 = torch.empty(MAXM, N, device=DEV)
        _check(sd_pkg().lib().seqdiff_op_layernorm(FP32, MAXM, N, _p(d["o"]), _p(d["gamma"]), _p(d["beta"]), 1e-12, _p(ln32), None, _p(st),
                                                   stream_ptr()))
        torch.cuda.synchronize()
        d.update(stats=st, ln32=ln32)
        # LayerNorm(o) in float64 with the kernel's own (mean, rstd)
        s64 = st.double().cpu()
        d["ln64"] = (o.double() - s64[:, :1]) * s64[:, 1:] * gamma.double() + beta.double()
        _CACHE[key] = d
    return _CACHE[key]


def _skip_tile(N, bn):
    if bn and N % bn:
        pytest.skip("tile width does not divide N")


@pytest.mark.parametrize("bn,cg2", TILES)
@pytest.mark.parametrize("M", [1, 31, 33, 127, 129, 257, 1000, 8192])
@pytest.mark.parametrize("N,K", [(768, 768), (768, 3072)])
@pytest.mark.parametrize("mode", [BF16, FP16])
def test_gemm_lnresid(bn, cg2, mode, M, N, K):
    """RESID = 2: C = A W^T + bias + LayerNorm(o), the LayerNorm rebuilt in the epilogue from seqdiff_op_layernorm's (mean, rstd) and the
    affine.  (i) against float64 within the fp32-residual bound; (ii) bit-identical to the RESID = 1 GEMM whose residual is the LayerNorm
    kernel's own fp32 output (same fp32 formula and operation order)."""
    _skip_tile(N, bn)
    d = _operands(mode, N, K)
    A, st, o = d["A"][:M], d["stats"][:M], d["o"][:M]
    C2 = _nan(M, N, torch.float32)
    _gemm_ex(mode, bn, cg2, M, N, K, A, d["W"], d["bias"], C2, resid=o, ln=(st, d["gamma"], d["beta"]), out_f32=True)
    C1 = _nan(M, N, torch.float32)
    _gemm_ex(mode, bn, cg2, M, N, K, A, d["W"], d["bias"], C1, resid=d["ln32"][:M], out_f32=True)
    torch.cuda.synchronize()
    _assert_pad_untouched(C2, M)
    _assert_pad_untouched(C1, M)
    ref = d["prod"][:M] + d["ln64"][:M]
    err = (C2[:M].double().cpu() - ref).abs().max().item()
    scale = ref.abs().max().item()
    assert err <= 2e-5 * scale, f"LayerNorm residual: err {err} scale {scale}"
    assert torch.equal(C2[:M], C1[:M]), f"RESID=2 differs from RESID=1 on LayerNorm's fp32 output: max |d| {(C2[:M] - C1[:M]).abs().max().item()}"


# (epilogue, output) forms of the model: 16-bit out with identity / GELU / SiLU, fp32 residual, LayerNorm residual
FORMS = ["identity", "gelu", "silu", "resid", "lnresid"]


@pytest.mark.parametrize("form", FORMS)
@pytest.mark.parametrize("mode", [BF16, FP16])
def test_gemm_rows_independent_of_M_and_tile(form, mode):
    """One fixed set of A rows through every legal tile configuration and the tuner at M = 8192, and at M = 1000 and 129 on prefixes of
    those rows: every shared row must be bit-identical.  The packed and receptor-rows loops compute the same rows at another M, where
    the tuner may pick other tiles."""
    N, K = 768, 768
    d = _operands(mode, N, K)
    epi = {"gelu": 1, "silu": 2}.get(form, 0)
    f32 = form in ("resid", "lnresid")
    first, first_cfg, differ = None, None, []
    for M in (MAXM, 1000, 129):
        for bn, cg2 in TILES:
            if bn and N % bn:
                continue
            C = _nan(M, N, torch.float32 if f32 else DT[mode])
            resid = d["o"][:M] if f32 else None
            ln = (d["stats"][:M], d["gamma"], d["beta"]) if form == "lnresid" else None
            _gemm_ex(mode, bn, cg2, M, N, K, d["A"][:M], d["W"], d["bias"], C, resid=resid, ln=ln, epi=epi, out_f32=f32)
            torch.cuda.synchronize()
            _assert_pad_untouched(C, M)
            if first is None:
                first, first_cfg = C[:M].clone(), (M, bn, cg2)
                assert torch.isfinite(first.float()).all()
            elif not torch.equal(C[:M], first[:M]):
                differ.append(((M, bn, cg2), (C[:M].float() - first[:M].float()).abs().max().item()))
    assert not differ, f"{form}: rows differ from those of (M, bn, cg2) = {first_cfg} at (config, max |d|) {differ}"


# ---------------------------------------------------------------------------------------------------
def _num_sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _k_ranges(M, N, K, bn, cg2, split):
    """How many k-ranges gemm_16 runs (csrc/gemm.cu): the cost-model tile (pick_cfg) when none is forced, the auto split (one scheduled
    tile per CTA slot, >= 4 k-blocks per range), clamped to the k-blocks.  More than one: the partial products are added into C."""
    sms = _num_sms()
    if bn == 0:
        if M <= 64:
            bn, cg2 = 128, 0
        elif N % 256 == 0 and M * N * K >= 2.5e10:
            bn, cg2 = 256, 1
        else:
            best, best_cost = 0, 0.0
            for w in (256, 192, 128):
                if N % w:
                    continue
                cost = -(-(-(-M // 128) * (N // w)) // sms) * w * (1.0 + 48.0 / w)
                if not best or cost < best_cost * 0.97:
                    best, best_cost = w, cost
            bn, cg2 = best, 0
    nkb = -(-K // 64)
    s = split
    if s < 0:
        tiles = -(-M // (256 if cg2 else 128)) * (N // bn)
        s = min((sms // 2 if cg2 else sms) // tiles, nkb // 4)
    return max(1, min(s, nkb))


_SPLIT_REF = {}


@pytest.mark.parametrize("bn,cg2", [(0, 0), (128, 0), (192, 0), (256, 0), (256, 1)])
@pytest.mark.parametrize("split", [1, 2, 5, -1, 10000])
@pytest.mark.parametrize("M,N,K", [(768, 768, 8192), (3072, 768, 16384), (2304, 768, 1000), (768, 3072, 2048), (768, 1024, 16), (128, 128, 64)])
@pytest.mark.parametrize("mode", [BF16, FP16])
def test_gemm_split_k_f32(bn, cg2, mode, split, M, N, K):
    """Split-K NT GEMM with fp32 C (the training step's weight-gradient form): C prefilled with X, nonzero bias.  With more than one
    k-range every range adds into C and the bias is added once: C = X + A W^T + bias; with one (split_k = 1, or clamped to one k-block)
    C = A W^T + bias.  split_k = 10000 is clamped to the number of k-blocks."""
    _skip_tile(N, bn)
    if mode != BF16 and K > 2048:
        pytest.skip("format variants share the tile code")
    key = (mode, M, N, K)
    if key not in _SPLIT_REF:
        g = torch.Generator().manual_seed(M + 3 * N + 7 * K + mode)
        A = torch.randn(M, K, generator=g).to(DT[mode])
        W = (torch.randn(N, K, generator=g) / math.sqrt(K)).to(DT[mode])
        bias = torch.randn(N, generator=g)
        X = torch.randn(M, N, generator=g)
        _SPLIT_REF.clear()
        _SPLIT_REF[key] = (A.to(DEV), W.to(DEV), bias.to(DEV), X, A.double() @ W.double().t() + bias.double())
    A, W, bias, X, prod = _SPLIT_REF[key]
    C = _nan(M, N, torch.float32)
    C[:M] = X.to(DEV)
    _gemm_ex(mode, bn, cg2, M, N, K, A, W, bias, C, out_f32=True, split=split)
    torch.cuda.synchronize()
    _assert_pad_untouched(C, M)
    ks = _k_ranges(M, N, K, bn, cg2, split)
    ref = prod + X.double() if ks > 1 else prod
    err = (C[:M].double().cpu() - ref).abs().max().item()
    scale = ref.abs().max().item()
    assert err <= 2e-5 * scale + 1e-5 * math.sqrt(K), f"{ks} k-ranges: err {err} scale {scale}"


# ---------------------------------------------------------------------------------------------------
# attention
def _attn(prec, B, heads, Lq, Lk, q, ldq, k, ldk, v, ldv, E, P, mask, Lk_mask, out, pack=None, kv_div=1):
    q_off, k_off, q_len, q_rows, k_rows = pack if pack is not None else (None, None, None, 0, 0)
    _check(sd_pkg().lib().seqdiff_op_attention_packed(prec, B, heads, Lq, Lk, _p(q), ldq, _p(k), ldk, _p(v), ldv, _p(E), P, _p(mask), Lk_mask,
                                                      _p(q_off), _p(k_off), _p(q_len), q_rows, k_rows, kv_div, _p(out), stream_ptr()))


def _offsets(lens):
    off = [0]
    for n in lens[:-1]:
        off.append(off[-1] + n)
    return off


def _ref(heads, P, q, k, v, E):
    """float64 attention core of one graph: q [Lq, H], k / v [Lk, H], every key valid"""
    cfg = O.OracleConfig(hidden_size=q.shape[1], num_attention_heads=heads, max_position_embeddings=P)
    zero = torch.zeros(1, 1, 1, k.shape[0], dtype=torch.float64)
    return O.attention_core(cfg, q[None].double(), k[None].double(), v[None].double(), zero, None if E is None else E.double())[0]


def _prefix_mask(lens, width):
    return (torch.arange(width)[None, :] < torch.tensor(lens)[:, None]).float()


def _run_packed_case(prec, heads, q_lens, k_lens, kv_div, self_attn, rel, seed, Lq_pad=None):
    """Runs one packed case and checks it: (i) per graph against float64, (ii) bit-identical to the padded kernel at every valid row,
    (iii) no row past q_rows written.  q_lens: per query graph (B); k_lens: per key graph (B / kv_div).  self_attn: q / k / v are slices
    of one [rows, 3H] matrix; else q is its own [rows, H] matrix and k / v are column slices of a [rows, 6 * 2H] kv_all block.
    Lq_pad: padded queries (q_off = b * Lq_pad, q_len = Lq_pad)."""
    H = heads * 64
    P = 512
    dt = DT[prec]
    B = len(q_lens)
    g = torch.Generator().manual_seed(seed)
    q_off, k_off = _offsets(q_lens), _offsets(k_lens)
    q_rows, k_rows = sum(q_lens), sum(k_lens)
    Lq, Lk = max(q_lens), max(k_lens)
    Lk_mask = P if self_attn else Lk + 56  # cross: the receptor mask keeps its padded pitch, longer than the longest key graph
    E = (torch.randn(2 * P - 1, 64, generator=g) * 0.5).to(dt) if rel else None
    if self_attn:
        qkv = torch.randn(q_rows, 3 * H, generator=g).to(dt)
        q, k, v = qkv[:, :H], qkv[:, H:2 * H], qkv[:, 2 * H:]
        dev = qkv.to(DEV)
        qd, kd, vd, ldq, ldk = dev[:, :H], dev[:, H:2 * H], dev[:, 2 * H:], 3 * H, 3 * H
    else:
        layer = 3
        qm = torch.randn(q_rows, H, generator=g).to(dt)
        kv_all = torch.randn(k_rows, 12 * H, generator=g).to(dt)
        q, k, v = qm, kv_all[:, 2 * H * layer:2 * H * layer + H], kv_all[:, 2 * H * layer + H:2 * H * (layer + 1)]
        qd, kvd = qm.to(DEV), kv_all.to(DEV)
        kd, vd, ldq, ldk = kvd[:, 2 * H * layer:2 * H * layer + H], kvd[:, 2 * H * layer + H:2 * H * (layer + 1)], H, 12 * H
    mask = _prefix_mask(k_lens, Lk_mask).to(DEV)
    ints = lambda a: torch.tensor(a, dtype=torch.int32, device=DEV)
    out = _nan(q_rows, H, dt)
    _attn(prec, B, heads, Lq, Lk, qd, ldq, kd, ldk, vd, ldk, None if E is None else E.to(DEV), P, mask, Lk_mask, out,
          pack=(ints(q_off), ints(k_off), ints(q_lens), q_rows, k_rows), kv_div=kv_div)
    torch.cuda.synchronize()
    # (iii)
    _assert_pad_untouched(out, q_rows)
    got = out[:q_rows].cpu()
    assert torch.isfinite(got.float()).all()
    # (i) per graph: a length-1 graph's error does not hide under a large graph's maximum
    tol = {BF16: 2e-2, FP16: 3e-3}[prec]
    for b in range(B):
        kg = b // kv_div
        qs, ks_ = slice(q_off[b], q_off[b] + q_lens[b]), slice(k_off[kg], k_off[kg] + k_lens[kg])
        ref = _ref(heads, P, q[qs], k[ks_], v[ks_], E)
        e = rel_err(got[qs], ref)
        assert e < tol, f"graph {b} (q_len {q_lens[b]}, key graph {kg} of length {k_lens[kg]}): rel err {e}"
    # (ii) the same graphs scattered into the padded layout (finite junk in the padded rows, prefix key masks), padded kernel, same kv_div
    Lqp = Lq if Lq_pad is None else Lq_pad
    qp = torch.randn(B, Lqp, H, generator=g).to(dt)
    kp = torch.randn(B // kv_div, Lk, H, generator=g).to(dt)
    vp = torch.randn(B // kv_div, Lk, H, generator=g).to(dt)
    for b in range(B):
        qp[b, :q_lens[b]] = q[q_off[b]:q_off[b] + q_lens[b]]
    for kg in range(B // kv_div):
        kp[kg, :k_lens[kg]] = k[k_off[kg]:k_off[kg] + k_lens[kg]]
        vp[kg, :k_lens[kg]] = v[k_off[kg]:k_off[kg] + k_lens[kg]]
    outp = _nan(B * Lqp, H, dt)
    _attn(prec, B, heads, Lqp, Lk, qp.to(DEV), H, kp.to(DEV), H, vp.to(DEV), H, None if E is None else E.to(DEV), P,
          _prefix_mask(k_lens, Lk).to(DEV), Lk, outp, kv_div=kv_div)
    torch.cuda.synchronize()
    _assert_pad_untouched(outp, B * Lqp)
    outp = outp[:B * Lqp].view(B, Lqp, H).cpu()
    for b in range(B):
        a, p_ = got[q_off[b]:q_off[b] + q_lens[b]], outp[b, :q_lens[b]]
        assert torch.equal(a, p_), f"graph {b}: packed differs from padded at valid rows, max |d| {(a.float() - p_.float()).abs().max().item()}"


SELF_LENS = [128, 1, 129, 512, 127, 45, 300]  # offsets not multiples of 128; the last graph's blocks run past q_rows / k_rows


@pytest.mark.parametrize("rel", [True, False])
@pytest.mark.parametrize("heads", [2, 12])
@pytest.mark.parametrize("prec", [BF16, FP16])
def test_packed_self_attention(prec, heads, rel):
    """self-attention of a packed batch: q / k / v slices of one [rows, 3H] matrix, several query and key blocks per graph"""
    _run_packed_case(prec, heads, SELF_LENS, SELF_LENS, 1, True, rel, seed=heads + int(rel))


@pytest.mark.parametrize("kv_div", [1, 3])
@pytest.mark.parametrize("heads", [2, 12])
@pytest.mark.parametrize("prec", [BF16, FP16])
def test_packed_cross_attention_padded_queries(prec, heads, kv_div):
    """padded queries (q_off = b Lq, q_len = Lq) against packed keys, K / V column slices of a kv_all block, Lk < Lk_mask; kv_div query
    graphs per key graph"""
    k_lens = [200, 37, 129]
    Lq = 100
    B = len(k_lens) * kv_div
    _run_packed_case(prec, heads, [Lq] * B, k_lens, kv_div, False, False, seed=7 * heads + kv_div, Lq_pad=Lq)


@pytest.mark.parametrize("heads", [2, 12])
@pytest.mark.parametrize("prec", [BF16, FP16])
def test_packed_cross_attention_packed_queries_shared_keys(prec, heads):
    """packed queries against packed keys, three query graphs per key graph (the packed multi-sample and design form)"""
    q_lens = [1, 1, 1, 130, 130, 130, 64, 64, 64]
    k_lens = [200, 37, 129]
    _run_packed_case(prec, heads, q_lens, k_lens, 3, False, False, seed=11 + heads)


@pytest.mark.parametrize("rel", [True, False])
@pytest.mark.parametrize("heads", [2, 12])
@pytest.mark.parametrize("prec", [BF16, FP16])
def test_packed_attention_many_items(prec, heads, rel):
    """40 packed graphs: more work items than CTAs, every persistent CTA walks several items of different graphs"""
    g = torch.Generator().manual_seed(40 + heads)
    lens = torch.randint(1, 301, (40,), generator=g).tolist()
    _run_packed_case(prec, heads, lens, lens, 1, True, rel, seed=41 + heads + int(rel))


def test_packed_attention_small_grid_subprocess():
    """the packed attention cases with only 3 CTAs (SEQDIFF_ATTN_GRID=3): every CTA walks a long item list across graphs"""
    env = dict(os.environ, SEQDIFF_ATTN_GRID="3")
    r = subprocess.run([sys.executable, "-m", "pytest", __file__, "-q", "-m", "gpu", "-k", "test_packed and not subprocess", "-p",
                        "no:cacheprovider"], env=env, capture_output=True, text=True)
    assert r.returncode == 0, "SEQDIFF_ATTN_GRID=3:\n" + r.stdout[-2000:]


@pytest.mark.parametrize("kv_div", [2, 3])
@pytest.mark.parametrize("Lq,Lk", [(100, 200), (33, 17)])
def test_attention_f32_shared_keys(kv_div, Lq, Lk):
    """fp32 attention kernel, padded form with kv_div query graphs per key graph, against float64"""
    heads, P = 4, 256
    H = heads * 64
    nkg = 2
    B = nkg * kv_div
    g = torch.Generator().manual_seed(kv_div + Lq + Lk)
    q = torch.randn(B, Lq, H, generator=g)
    k = torch.randn(nkg, Lk, H, generator=g)
    v = torch.randn(nkg, Lk, H, generator=g)
    k_lens = [Lk, max(1, Lk // 3)]
    mask = _prefix_mask(k_lens, Lk)
    out = _nan(B * Lq, H, torch.float32)
    _attn(FP32, B, heads, Lq, Lk, q.to(DEV), H, k.to(DEV), H, v.to(DEV), H, None, P, mask.to(DEV), Lk, out, kv_div=kv_div)
    torch.cuda.synchronize()
    _assert_pad_untouched(out, B * Lq)
    got = out[:B * Lq].view(B, Lq, H).cpu()
    for b in range(B):
        kg = b // kv_div
        ref = _ref(heads, P, q[b], k[kg, :k_lens[kg]], v[kg, :k_lens[kg]], None)
        assert rel_err(got[b], ref) < 2e-5, (b, rel_err(got[b], ref))
