"""Operator-level parity tests of the training step's rowwise and elementwise kernels (csrc/train_kernels.cu, angle_loss_bwd in
csrc/decode_loss.cu) through their seqdiff_op_* entries, at the row counts training runs at and at every hidden size the kernels are
instantiated for.

Every kernel is compared with a float64 torch restatement of the same operation computed from the same (16-bit-rounded) inputs; for the
backward kernels the reference is autograd of the float64 forward.  Row counts are derived from the SM count so that each kernel's
grid-stride loop makes a second pass and its last pass is ragged: embed_bwd / predictor_tail_bwd run one CTA per SM (8 rows per CTA pass),
layernorm_bwd and ln_modulate_bwd two (times the rows per warp of per-graph ln_modulate_bwd), the 16-bit layernorm_bwd_cast one wave of
resident CTAs (16 384 rows wrap at any occupancy), the elementwise kernels 2048 CTAs of 256 x 8 elements.

Gates: per-row outputs per row, relative to that row's reference maximum; 16-bit outputs within one ulp of the rounded float64 value (plus
a few fp32 ulps of the row's scale where the kernel's fp32 value comes out of a cancellation); sums over rows per column, relative to the sum
of |terms| of that column (and the prefill).  Each sum check also shows that its gate would notice a dropped row (the last row, the first
row of the last CTA pass).  Accumulating outputs are prefilled, placed once 16 B aligned and once one float off (the two flush branches),
between guard elements that must not change; row-shaped outputs carry NaN rows past M that must stay NaN.  Dropout masks are checked bit
for bit against a numpy restatement of Philox4x32-10 (philox.cuh: drop_scales8)."""
import ctypes
import functools
import math
import zlib

import numpy as np
import pytest
import torch
import torch.nn.functional as F

from helpers import BF16, FP16, FP32, O, sd_pkg, stream_ptr

gpu = pytest.mark.gpu
DEV = "cuda:0"
PAD = 16
GUARD = -777.5
SEED = 0x9E37_79B9_7F4A_7C15  # above 2^32: both key words matter
DT = {FP32: torch.float32, BF16: torch.bfloat16, FP16: torch.float16}
PREC_ID = {FP32: "fp32", BF16: "bf16", FP16: "fp16"}
HS = [256, 512, 768, 1024]
EPS = 1e-12  # BertLayerNorm eps of the model
M32 = np.uint64(0xFFFFFFFF)


def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _check(rc):
    if rc != 0:
        raise RuntimeError(sd_pkg().lib().seqdiff_last_error().decode())


def _lib():
    return sd_pkg().lib()


# ---------------------------------------------------------------------------------------------------
# Philox4x32-10 and the dropout mask, restated on the host
# ---------------------------------------------------------------------------------------------------
def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 on numpy arrays of counters (broadcast), key (k0, k1); returns the four uint32 output words"""
    c = [a.astype(np.uint64) for a in np.broadcast_arrays(*[np.asarray(x, dtype=np.uint64) for x in (c0, c1, c2, c3)])]
    k0, k1 = np.uint64(k0), np.uint64(k1)
    s32 = np.uint64(32)
    for _ in range(10):
        p0, p1 = np.uint64(0xD2511F53) * c[0], np.uint64(0xCD9E8D57) * c[2]
        c = [(p1 >> s32) ^ c[1] ^ k0, p1 & M32, (p0 >> s32) ^ c[3] ^ k1, p0 & M32]
        k0, k1 = (k0 + np.uint64(0x9E3779B9)) & M32, (k1 + np.uint64(0xBB67AE85)) & M32
    return [x.astype(np.uint32) for x in c]


N_MASK = 16389 * 1024  # the largest flat element count a dropout case here uses


@functools.lru_cache(maxsize=4)
def _keep_np(p, site, step):
    """keep flags of flat elements 0 .. N_MASK - 1 as drop_scales8 draws them: word e % 4 of the Philox call with counter
    (e / 4 low, e / 4 high, site, step) and key = seed, kept when word >= uint32(double(float(p)) * 2^32)"""
    q = np.arange(N_MASK // 4, dtype=np.uint64)
    w = philox4x32_10(q & M32, q >> np.uint64(32), site, step, SEED & 0xFFFFFFFF, SEED >> 32)
    thr = np.uint32(int(float(np.float32(p)) * 4294967296.0))
    return np.stack(w, axis=1).reshape(-1) >= thr


def _keep(p, site, step, n):
    """float64 keep-scale of flat elements 0 .. n - 1 on the device (the fp32 scale 1 / (1 - p) the kernels use)"""
    if p == 0:
        return torch.ones(n, dtype=torch.float64, device=DEV)
    sc = float(np.float32(1) / (np.float32(1) - np.float32(p)))
    return torch.from_numpy(_keep_np(p, site, step)[:n]).to(DEV).double() * sc


def test_philox_rounds_match_the_sampler_reference():
    """the vectorised rounds against test_gpu_ops._philox_ref (Random123 known answer, the sampler's counter layout)"""
    from test_gpu_ops import _philox_ref
    assert [int(v) for v in philox4x32_10(0, 0, 0, 0, 0, 0)] == [0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8]
    seed, graph, step = 0x1234_5678_9ABC_DEF0, 7_000_000_123, 17
    res = np.arange(0, 300, 7)
    for call in (0, 3):
        w = philox4x32_10(res, (step * 8 + call) & 0xFFFFFFFF, graph & 0xFFFFFFFF, graph >> 32, seed & 0xFFFFFFFF, seed >> 32)
        for i, r in enumerate(res):
            assert [int(x[i]) for x in w] == _philox_ref(seed, graph, int(r), step, call)


# ---------------------------------------------------------------------------------------------------
# shapes, buffers, gates
# ---------------------------------------------------------------------------------------------------
def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _rows(tag, rpw=1):
    """symbolic row counts: w8 = one CTA per SM x 8 warps (embed_bwd, predictor_tail_bwd), w16 = two CTAs per SM (layernorm_bwd,
    ln_modulate_bwd; x rpw rows per warp), +-1 row"""
    S = _sms()
    for w, base in (("w16", 16 * S * rpw), ("w8", 8 * S)):
        if tag.startswith(w):
            return base + int(tag[len(w):])
    return int(tag)


def _cdiv(a, b):
    return -(-a // b)


def _last_pass_first_row(M, rows_per_pass):
    return (M - 1) // rows_per_pass * rows_per_pass


def _nan(rows, cols, dtype=torch.float32):
    return torch.full((rows + PAD, cols), float("nan"), device=DEV, dtype=dtype)


def _assert_nan_pad(t, rows, what):
    assert torch.isnan(t[rows:].float()).all(), f"{what}: a row past the output was written"


def _prefill(n, salt):
    return (((torch.arange(n, device=DEV) * 7 + salt) % 13) - 6).float() * 0.125


class Acc:
    """an accumulating fp32 output of `shape`, prefilled with known values, as a slice of a larger buffer at float offset `off`
    (4: 16 B aligned, 5: one float past) with guard elements on both sides"""

    def __init__(self, shape, off, salt=0):
        n = math.prod(shape)
        self.off, self.n = off, n
        self.big = torch.full((n + 12,), GUARD, device=DEV)
        self.pre = _prefill(n, salt).view(shape)
        self.big[off:off + n] = self.pre.reshape(-1)
        self.t = self.big[off:off + n].view(shape)

    def check_guards(self, what):
        g = torch.cat([self.big[:self.off], self.big[self.off + self.n:]])
        assert (g == GUARD).all(), f"{what}: a guard element next to the output changed"


WORST = {}


def _note(key, v):
    WORST[key] = max(WORST.get(key, 0.0), float(v))


def _assert_rows(got, ref, rtol, what):
    """per row: max |got - ref| <= rtol * max |ref| of that row"""
    got, ref = got.double(), ref.double()
    err, scale = (got - ref).abs().amax(1), ref.abs().amax(1)
    bad = ~(err <= rtol * scale)
    if bad.any():
        r = int(bad.nonzero()[0])
        raise AssertionError(f"{what}: {int(bad.sum())} rows beyond {rtol:g} of their row max; row {r}: err {float(err[r]):.3e} "
                             f"scale {float(scale[r]):.3e}")
    live = scale > 0
    if live.any():
        _note(what.split(" ")[0], (err[live] / scale[live]).max())


MANT = {BF16: 7, FP16: 10}
MIN_ULP = {BF16: 2.0 ** -133, FP16: 2.0 ** -24}


def _ulp(x, prec):
    e = torch.frexp(x.abs().clamp_min(1e-300))[1]
    return torch.ldexp(torch.ones_like(x), e - 1 - MANT[prec]).clamp_min(MIN_ULP[prec])


def _assert_16bit(got, ref, prec, what, slack=0.0):
    """16-bit output within one ulp of T(ref) (+ slack: the fp32 rounding noise of the kernel's value before its 16-bit rounding)"""
    r = ref.double().to(DT[prec]).double()
    err = (got.double() - r).abs()
    bad = ~(err <= _ulp(r, prec) + slack)
    if bad.any():
        i = bad.nonzero()[0].tolist()
        raise AssertionError(f"{what}: {int(bad.sum())} elements more than one ulp from the rounded float64 value; at {i}: got "
                             f"{float(got[tuple(i)]):.6e} want {float(ref[tuple(i)]):.6e}")


def _row_slack(ref):
    """a few fp32 ulps of each row's scale, broadcast over the row"""
    return 2.0 ** -21 * ref.double().abs().amax(-1, keepdim=True)


def _row_abs(t):
    """sum over rows of each row's largest |term|: the scale of the fp32 rounding a term computed with cancellation carries"""
    return t.abs().amax(-1).sum()


def _assert_sum(acc, got_sum, absum, rtol, what, drop_terms=(), row_abs=0.0):
    """acc.t == prefill + got_sum per column within rtol * (sum of |terms| + |prefill|), plus 2^-20 (8 fp32 ulps) of row_abs where the
    terms come out of a cancellation (a LayerNorm backward): their error scales with their row, not with themselves.  Each entry of
    drop_terms (label, term of one row, same shape) must lie outside that gate: a kernel that lost the row would fail"""
    ref = acc.pre.double() + got_sum
    tol = rtol * (absum + acc.pre.double().abs()) + 2.0 ** -20 * row_abs
    err = (acc.t.double() - ref).abs()
    bad = ~(err <= tol)
    if bad.any():
        i = bad.nonzero()[0].tolist()
        raise AssertionError(f"{what}: {int(bad.sum())} of {bad.numel()} sums beyond {rtol:g} of their sum of |terms|; at {i}: got "
                             f"{float(acc.t[tuple(i)]):.7e} want {float(ref[tuple(i)]):.7e} (sum |terms| {float(absum[tuple(i)]):.3e})")
    if (tol > 0).any():
        _note(what.split(" ")[0] + " (share of its gate)", (err[tol > 0] / tol[tol > 0]).max())
    for label, term in drop_terms:
        assert (term.double().abs() > tol).any(), f"{what}: the gate cannot see a missing {label}"
    acc.check_guards(what)


def _drop_rows(M, rows_per_pass):
    out = {"last row": M - 1}
    first = _last_pass_first_row(M, rows_per_pass)
    if first != M - 1:
        out["first row of the last CTA pass"] = first
    return out


def _gen(*key):
    return torch.Generator(device=DEV).manual_seed(zlib.crc32(repr(key).encode()))


def _randn(g, *shape, scale=1.0, shift=0.0):
    return torch.randn(*shape, generator=g, device=DEV) * scale + shift


def _ln64(x, eps):
    mean = x.mean(-1, keepdim=True)
    return (x - mean) / torch.sqrt(x.var(-1, unbiased=False, keepdim=True) + eps)


# ---------------------------------------------------------------------------------------------------
# dropout_add_layernorm
# ---------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("Mtag", ["1", "9", "w8+1", "16389"])
@pytest.mark.parametrize("H", HS)
@pytest.mark.parametrize("prec", [FP32, BF16, FP16], ids=PREC_ID.get)
def test_dropout_add_layernorm(prec, H, Mtag):
    M = _rows(Mtag)
    p, site, step = 0.1, 5, 9
    g = _gen("dal", prec, H, M)
    d0, resid = _randn(g, M, H, scale=2.0), _randn(g, M, H)
    w, b = _randn(g, H, scale=0.1, shift=1.0), _randn(g, H, scale=0.1)
    d = _nan(M, H)
    d[:M] = d0
    out32 = _nan(M, H)
    out16 = None if prec == FP32 else _nan(M, H, DT[prec])
    keep_bits = torch.full((M + PAD, H // 8), 0xA5, dtype=torch.uint8, device=DEV)
    _check(_lib().seqdiff_op_dropout_add_layernorm(prec, M, H, _p(d), _p(resid), _p(w), _p(b), EPS, p, SEED, site, step, _p(out32),
                                                   _p(out16), _p(keep_bits), stream_ptr()))
    torch.cuda.synchronize()
    keep = _keep(p, site, step, M * H).view(M, H)
    o = d0.double() * keep + resid.double()
    h = _ln64(o, EPS) * w.double() + b.double()
    _assert_rows(d[:M], o, 1e-6, "dropout_add_layernorm.o")
    _assert_rows(out32[:M], h, 1e-5, "dropout_add_layernorm.out32")
    for t, what in ((d, "o"), (out32, "out32")):
        _assert_nan_pad(t, M, what)
    if out16 is not None:
        _assert_16bit(out16[:M], h, prec, "dropout_add_layernorm.out16", _row_slack(h))
        _assert_nan_pad(out16, M, "out16")
    want_bits = np.packbits(keep.cpu().numpy() != 0, axis=1, bitorder="little")
    assert np.array_equal(keep_bits[:M].cpu().numpy(), want_bits), "keep bits differ from the host Philox mask"
    assert (keep_bits[M:] == 0xA5).all(), "keep bits written past M"


# ---------------------------------------------------------------------------------------------------
# layernorm_bwd (fp32) and layernorm_bwd_cast (16-bit dY + bias gradient, keep bits or Philox)
# ---------------------------------------------------------------------------------------------------
LN_MODES = {"fp32": (FP32, 0.0), "bf16": (BF16, 0.0), "bf16-drop": (BF16, 0.1), "fp16-drop": (FP16, 0.1)}
LN_ROWS = ["1", "7", "w16-1", "w16+1", "16384", "16389"]


@gpu
@pytest.mark.parametrize("Mtag", LN_ROWS)
@pytest.mark.parametrize("H", HS)
@pytest.mark.parametrize("mode", list(LN_MODES))
def test_layernorm_bwd(mode, H, Mtag):
    prec, p = LN_MODES[mode]
    site, step = 13, 3
    M = _rows(Mtag)
    off = 4 if LN_ROWS.index(Mtag) % 2 == 0 else 5
    g = _gen("lnb", mode, H, M)
    o, dh = _randn(g, M, H, scale=3.0, shift=0.5), _randn(g, M, H)
    gamma = _randn(g, H, scale=0.1, shift=1.0)
    # float64 reference: autograd of h = LN(o) * gamma + beta
    x = o.double().requires_grad_(True)
    gm = gamma.double().requires_grad_(True)
    bt = torch.zeros(H, dtype=torch.float64, device=DEV, requires_grad=True)
    F.layer_norm(x, (H,), gm, bt, EPS).backward(dh.double())
    d_o_ref = x.grad
    xhat = _ln64(o.double(), EPS)
    keep = _keep(p, site, step, M * H).view(M, H)
    kb = None
    if p > 0:
        kb = torch.from_numpy(np.packbits(keep.cpu().numpy() != 0, axis=1, bitorder="little")).to(DEV)
    S = _sms()
    rows_per_pass = [2 * S * 8] if prec == FP32 else [occ * S * 8 for occ in range(1, 9)]
    drops = {f"{k} ({rpp} rows per pass)": r for rpp in rows_per_pass for k, r in _drop_rows(M, rpp).items()}
    runs = []
    for use_bits in ([True, False] if p > 0 else [False]):
        d_o = _nan(M, H)
        g16 = None if prec == FP32 else _nan(M, H, DT[prec])
        dgamma, dbeta, dbias = Acc((H,), off, 1), Acc((H,), off, 2), Acc((H,), off, 3)
        _check(_lib().seqdiff_op_layernorm_bwd(prec, M, H, _p(dh), _p(o), _p(gamma), EPS, _p(d_o), _p(dgamma.t), _p(dbeta.t), p, SEED, site,
                                               step, _p(kb if use_bits else None), _p(g16), None if prec == FP32 else _p(dbias.t),
                                               stream_ptr()))
        torch.cuda.synchronize()
        form = f"{mode} {'keep bits' if use_bits else 'Philox'}"
        _assert_rows(d_o[:M], d_o_ref, 1e-5, f"layernorm_bwd.d_o ({form})")
        _assert_nan_pad(d_o, M, "d_o")
        tg, tb = dh.double() * xhat, dh.double()
        _assert_sum(dgamma, gm.grad, tg.abs().sum(0), 1e-5, f"layernorm_bwd.dgamma ({form})", [(k, tg[r]) for k, r in drops.items()],
                    _row_abs(tg))
        _assert_sum(dbeta, bt.grad, tb.abs().sum(0), 1e-5, f"layernorm_bwd.dbeta ({form})", [(k, tb[r]) for k, r in drops.items()])
        if prec != FP32:
            gref = d_o_ref * keep
            _assert_16bit(g16[:M], gref, prec, f"layernorm_bwd_cast.gT ({form})", _row_slack(gref))
            _assert_nan_pad(g16, M, "gT")
            if p > 0:
                assert (g16[:M][keep == 0] == 0).all() and (g16[:M][(keep != 0) & (gref.abs() > 1e-3)] != 0).all(), \
                    f"{form}: zero pattern of gT is not the mask"
            # the bias gradient is the column sum of the 16-bit values the weight-gradient GEMM reads, not of their fp32 originals
            t16 = g16[:M].double()
            _assert_sum(dbias, t16.sum(0), t16.abs().sum(0), 1e-5, f"layernorm_bwd_cast.dbias ({form})",
                        [(k, t16[r]) for k, r in drops.items()])
        runs.append((d_o[:M].clone(), None if g16 is None else g16[:M].clone()))
    if len(runs) == 2:
        assert torch.equal(runs[0][0], runs[1][0]) and torch.equal(runs[0][1], runs[1][1]), "keep bits and Philox give different outputs"


# ---------------------------------------------------------------------------------------------------
# ln_modulate_bwd
# ---------------------------------------------------------------------------------------------------
# (mod_div, affine_first, chunk0, sum_out, precision); mod_div 1 = per-token dmodT rows, else per-graph dmod32 with rows per warp
# 16 / 8 / 4 / 2 / 1 (128, 24, 100, 50, 33 rows per graph)
LNM_FORMS = {
    "token-aff-c0-sum-bf16": (1, True, 0, True, BF16),
    "token-c3-fp16": (1, False, 3, False, FP16),
    "token-aff-c3-fp32": (1, True, 3, False, FP32),
    "graph128-aff-c0-sum-bf16": (128, True, 0, True, BF16),
    "graph24-c3-fp32": (24, False, 3, False, FP32),
    "graph100-aff-c3-fp16": (100, True, 3, False, FP16),
    "graph50-c0-sum-bf16": (50, False, 0, True, BF16),
    "graph33-aff-c3-sum-fp32": (33, True, 3, True, FP32),
}
LNM_ROWS = ["1", "9", "w16-1", "w16+1", "16389"]


def _rpw(mod_div, per_graph):
    if per_graph:
        for c in (16, 8, 4, 2):
            if mod_div % c == 0:
                return c
    return 1


@gpu
@pytest.mark.parametrize("Mtag", LNM_ROWS)
@pytest.mark.parametrize("H", HS)
@pytest.mark.parametrize("form", list(LNM_FORMS))
def test_ln_modulate_bwd(form, H, Mtag):
    mod_div, aff, chunk0, want_sum, prec = LNM_FORMS[form]
    per_graph = form.startswith("graph")
    rpw = _rpw(mod_div, per_graph)
    M = _rows(Mtag, rpw)
    off = 4 if LNM_ROWS.index(Mtag) % 2 == 0 else 5
    G = _cdiv(M, mod_div)
    g = _gen("lnm", form, H, M)
    inp, dout = _randn(g, M, H, scale=2.0, shift=0.3), _randn(g, M, H)
    lnw, lnb = _randn(g, H, scale=0.1, shift=1.0), _randn(g, H, scale=0.1)
    mod = _randn(g, G, 6 * H, scale=0.5).to(DT[prec])
    din, sum_out = _nan(M, H), _nan(M, H) if want_sum else None
    dmodT = None if per_graph else _nan(M, 6 * H, DT[prec])
    dmod32 = Acc((G, 6 * H), off, 4) if per_graph else None
    dgamma, dbeta = Acc((H,), off, 5), Acc((H,), off, 6)
    _check(_lib().seqdiff_op_ln_modulate_bwd(prec, M, H, _p(dout), _p(inp), int(aff), _p(lnw), _p(lnb), EPS, _p(mod), mod_div, chunk0,
                                             _p(din), _p(sum_out), _p(dmodT), None if dmod32 is None else _p(dmod32.t),
                                             _p(dgamma.t) if aff else None, _p(dbeta.t) if aff else None, stream_ptr()))
    torch.cuda.synchronize()
    # float64 reference: autograd of out = gate * (LN0(y) * (1 + scale) + shift), y = LN(in; lnw, lnb) or in
    x = inp.double().requires_grad_(True)
    w64, b64 = lnw.double().requires_grad_(True), lnb.double().requires_grad_(True)
    m3 = mod.double()[:, chunk0 * H:(chunk0 + 3) * H].clone().requires_grad_(True)
    y = F.layer_norm(x, (H,), w64, b64, EPS) if aff else x
    if aff:
        y.retain_grad()
    n = F.layer_norm(y, (H,), eps=1e-5)
    rm = m3[torch.arange(M, device=DEV) // mod_div]
    sh, sc, gt = rm[:, :H], rm[:, H:2 * H], rm[:, 2 * H:]
    (gt * (n * (1 + sc) + sh)).backward(dout.double())
    _assert_rows(din[:M], x.grad, 2e-5, f"ln_modulate_bwd.din ({form})")
    _assert_nan_pad(din, M, "din")
    if want_sum:
        _assert_rows(sum_out[:M], x.grad + dout.double(), 2e-5, f"ln_modulate_bwd.sum_out ({form})")
        _assert_nan_pad(sum_out, M, "sum_out")
    grid = min(_cdiv(_cdiv(M, rpw), 8), 2 * _sms())
    drops = _drop_rows(M, grid * 8 * rpw)
    with torch.no_grad():
        nd, go = n.detach(), dout.double()
        terms = torch.cat([go * gt, go * gt * nd, go * (nd * (1 + sc) + sh)], 1)  # d(shift, scale, gate) of each row
    cols = slice(chunk0 * H, (chunk0 + 3) * H)
    if per_graph:
        absum = torch.zeros(G, 3 * H, dtype=torch.float64, device=DEV).index_add_(0, torch.arange(M, device=DEV) // mod_div, terms.abs())
        full_sum, full_abs, full_row = (torch.zeros(G, 6 * H, dtype=torch.float64, device=DEV) for _ in range(3))
        full_sum[:, cols], full_abs[:, cols] = m3.grad, absum
        full_row[:, cols] = torch.zeros(G, dtype=torch.float64, device=DEV).index_add_(0, torch.arange(M, device=DEV) // mod_div,
                                                                                         terms.abs().amax(1))[:, None]
        dt = []
        for k, r in drops.items():
            t = torch.zeros(G, 6 * H, dtype=torch.float64, device=DEV)
            t[r // mod_div, cols] = terms[r]
            dt.append((k, t))
        _assert_sum(dmod32, full_sum, full_abs, 1e-5, f"ln_modulate_bwd.dmod32 ({form})", dt, full_row)
    else:
        got = dmodT[:M, cols]
        if prec == FP32:
            _assert_rows(got, m3.grad, 1e-5, f"ln_modulate_bwd.dmodT ({form})")
        else:
            _assert_16bit(got, m3.grad, prec, f"ln_modulate_bwd.dmodT ({form})", _row_slack(m3.grad))
        rest = torch.cat([dmodT[:M, :cols.start], dmodT[:M, cols.stop:]], 1)
        assert torch.isnan(rest.float()).all(), "dmodT: a chunk outside (shift, scale, gate) was written"
        _assert_nan_pad(dmodT, M, "dmodT")
    if aff:
        with torch.no_grad():
            gy, xh1 = y.grad, _ln64(inp.double(), EPS)
            tg = gy * xh1
        _assert_sum(dgamma, w64.grad, tg.abs().sum(0), 1e-5, f"ln_modulate_bwd.dgamma ({form})", [(k, tg[r]) for k, r in drops.items()],
                    _row_abs(tg))
        _assert_sum(dbeta, b64.grad, gy.abs().sum(0), 1e-5, f"ln_modulate_bwd.dbeta ({form})", [(k, gy[r]) for k, r in drops.items()],
                    _row_abs(gy))
    else:
        assert torch.equal(dgamma.t, dgamma.pre) and torch.equal(dbeta.t, dbeta.pre)


# ---------------------------------------------------------------------------------------------------
# embed_bwd
# ---------------------------------------------------------------------------------------------------
# fin <= 8: DENSE form (thread-owned dW columns; fin = 8 takes the 4-wide flush, 1 and 5 the scalar one); above: shared atomics, 4-wide
# flush when fin % 4 == 0; fin = 32 at H = 1024 uses all 140 KB of shared memory the launcher allows
EMB_FORMS = {"1": (1, False), "5": (5, False), "8": (8, False), "12": (12, False), "20-onehot": (20, True), "20-dense": (20, False),
             "32": (32, False)}
EMB_ROWS = ["7", "w8-1", "w8+1", "16389"]


def _embed_inputs(g, M, fin, onehot, H):
    if onehot:
        x = F.one_hot(torch.randint(0, fin, (M,), generator=g, device=DEV), fin).float()
        x[::11] = 0  # padding rows: every input feature zero
    else:
        x = _randn(g, M, fin)
    Wt = _randn(g, fin, H, scale=1.0 / math.sqrt(fin))
    b, gamma = _randn(g, H, scale=0.1), _randn(g, H, scale=0.1, shift=1.0)
    return x, Wt, b, gamma


def _embed_ref(x, Wt, b, gamma, dout, keep):
    Wt64, b64 = Wt.double().requires_grad_(True), b.double().requires_grad_(True)
    gm, bt = gamma.double().requires_grad_(True), torch.zeros_like(b, dtype=torch.float64).requires_grad_(True)
    lin = x.double() @ Wt64 + b64
    lin.retain_grad()
    ln = _ln64(lin, EPS)
    ((ln * gm + bt) * keep).backward(dout.double())
    return Wt64.grad.t(), b64.grad, gm.grad, bt.grad, lin.grad, ln.detach()


@gpu
@pytest.mark.parametrize("Mtag", EMB_ROWS)
@pytest.mark.parametrize("H", HS)
@pytest.mark.parametrize("form", list(EMB_FORMS))
def test_embed_bwd(form, H, Mtag):
    fin, onehot = EMB_FORMS[form]
    M = _rows(Mtag)
    off = 4 if EMB_ROWS.index(Mtag) % 2 == 0 else 5
    p = 0.1 if (list(EMB_FORMS).index(form) + H // 256) % 2 else 0.0
    site, step = 2, 7
    g = _gen("emb", form, H, M)
    x, Wt, b, gamma = _embed_inputs(g, M, fin, onehot, H)
    dout = _randn(g, M, H)
    dW, db, dgamma, dbeta = Acc((H, fin), off, 7), Acc((H,), off, 8), Acc((H,), off, 9), Acc((H,), off, 10)
    _check(_lib().seqdiff_op_embed_bwd(M, fin, H, _p(dout), _p(x), _p(Wt), _p(b), _p(gamma), EPS, p, SEED, site, step, _p(dW.t), _p(db.t),
                                       _p(dgamma.t), _p(dbeta.t), stream_ptr()))
    torch.cuda.synchronize()
    keep = _keep(p, site, step, M * H).view(M, H)
    rW, rb, rg, rbt, glin, ln = _embed_ref(x, Wt, b, gamma, dout, keep)
    go = dout.double() * keep
    x64 = x.double()
    drops = _drop_rows(M, min(_cdiv(M, 8), _sms()) * 8)
    what = f"(fin {form}, p {p})"
    _assert_sum(dW, rW, glin.abs().t() @ x64.abs(), 1e-5, f"embed_bwd.dW {what}",
                [(k, torch.outer(glin[r], x64[r])) for k, r in drops.items() if x64[r].abs().sum() > 0],
                (glin.abs().amax(1) * x64.abs().amax(1)).sum())
    _assert_sum(db, rb, glin.abs().sum(0), 1e-5, f"embed_bwd.db {what}", [(k, glin[r]) for k, r in drops.items()], _row_abs(glin))
    tg = go * ln
    _assert_sum(dgamma, rg, tg.abs().sum(0), 1e-5, f"embed_bwd.dgamma {what}", [(k, tg[r]) for k, r in drops.items()], _row_abs(tg))
    _assert_sum(dbeta, rbt, go.abs().sum(0), 1e-5, f"embed_bwd.dbeta {what}", [(k, go[r]) for k, r in drops.items()])


@gpu
@pytest.mark.parametrize("fin", [8, 20])
def test_embed_bwd_dropout_mask(fin):
    """only the last row of 16 389 carries a gradient: dbeta is that row's dout where the mask keeps it and exactly 0 where it drops"""
    H, M, p, site, step = 768, 16389, 0.1, 4, 6
    g = _gen("embmask", fin)
    x, Wt, b, gamma = _embed_inputs(g, M, fin, False, H)
    dout = torch.zeros(M, H, device=DEV)
    dout[-1] = _randn(g, H)
    dW, db, dgamma, dbeta = (torch.zeros(n, device=DEV) for n in (H * fin, H, H, H))
    _check(_lib().seqdiff_op_embed_bwd(M, fin, H, _p(dout), _p(x), _p(Wt), _p(b), _p(gamma), EPS, p, SEED, site, step, _p(dW), _p(db),
                                       _p(dgamma), _p(dbeta), stream_ptr()))
    torch.cuda.synchronize()
    keep = _keep(p, site, step, M * H).view(M, H)[-1]
    assert torch.equal(dbeta == 0, keep == 0), "zero pattern of the embedding gradient is not the dropout mask"
    assert torch.equal(dbeta, dout[-1] * keep.float())  # go = dout * keep in fp32, added to zeros


# ---------------------------------------------------------------------------------------------------
# predictor_tail_bwd
# ---------------------------------------------------------------------------------------------------
PTB_ROWS = ["7", "w8-1", "w8+1", "16389"]


@gpu
@pytest.mark.parametrize("Mtag", PTB_ROWS)
@pytest.mark.parametrize("H", HS)
@pytest.mark.parametrize("prec", [FP32, BF16, FP16], ids=PREC_ID.get)
@pytest.mark.parametrize("Fo", [8, 20])
def test_predictor_tail_bwd(Fo, prec, H, Mtag):
    M = _rows(Mtag)
    off = 4 if PTB_ROWS.index(Mtag) % 2 == 0 else 5
    g = _gen("ptb", Fo, prec, H, M)
    y = _randn(g, M, H, scale=1.5, shift=0.2).to(DT[prec])
    gamma, beta = _randn(g, H, scale=0.1, shift=1.0), _randn(g, H, scale=0.1)
    W2 = _randn(g, Fo, H, scale=1.0 / math.sqrt(H))
    dl = _randn(g, M, Fo, scale=0.05)
    r = torch.arange(M, device=DEV)
    dl[r % 5 == 2] = 0                       # rows outside the noised set: all-zero gradient
    dl[(r % 7 == 3)[:, None] & (torch.arange(Fo, device=DEV) < Fo // 2)[None, :]] = 0  # only some outputs non-zero (output 0 zero)
    pass_rows = min(_cdiv(M, 8), _sms()) * 8
    if M > pass_rows:
        dl[pass_rows:2 * pass_rows] = 0      # a whole CTA pass of zero rows right after a live one
    dy = _nan(M, H)
    dW2, db2, dgamma, dbeta = Acc((Fo, H), off, 11), Acc((Fo,), off, 12), Acc((H,), off, 13), Acc((H,), off, 14)
    _check(_lib().seqdiff_op_predictor_tail_bwd(prec, M, H, Fo, _p(dl), _p(y), _p(gamma), _p(beta), EPS, _p(W2), _p(dy), _p(dW2.t), _p(db2.t),
                                                _p(dgamma.t), _p(dbeta.t), stream_ptr()))
    torch.cuda.synchronize()
    y64 = y.double().requires_grad_(True)
    gm, bt, W64 = gamma.double().requires_grad_(True), beta.double().requires_grad_(True), W2.double().requires_grad_(True)
    b2 = torch.zeros(Fo, dtype=torch.float64, device=DEV, requires_grad=True)
    ln = F.layer_norm(y64, (H,), gm, bt, EPS)
    ln.retain_grad()
    (ln @ W64.t() + b2).backward(dl.double())
    what = f"(F {Fo}, {PREC_ID[prec]})"
    _assert_rows(dy[:M], y64.grad, 1e-5, f"predictor_tail_bwd.dy {what}")
    assert (dy[:M][(dl == 0).all(1)] == 0).all(), "dy of a zero-gradient row is not zero"
    _assert_nan_pad(dy, M, "dy")
    drops = _drop_rows(M, pass_rows)
    with torch.no_grad():
        lnd, d64, gln = ln.detach(), dl.double(), ln.grad  # gln = dL/d(LN(y)) = dlogits W2: the dbeta terms
        tg = gln * _ln64(y.double(), EPS)                  # the dgamma terms
    live = {k: r for k, r in drops.items() if (d64[r] != 0).any()}
    _assert_sum(dW2, W64.grad, d64.abs().t() @ lnd.abs(), 1e-5, f"predictor_tail_bwd.dW2 {what}",
                [(k, torch.outer(d64[r], lnd[r])) for k, r in live.items()], (d64.abs().amax(1) * lnd.abs().amax(1)).sum())
    _assert_sum(db2, b2.grad, d64.abs().sum(0), 1e-5, f"predictor_tail_bwd.db2 {what}", [(k, d64[r]) for k, r in live.items()])
    _assert_sum(dgamma, gm.grad, tg.abs().sum(0), 1e-5, f"predictor_tail_bwd.dgamma {what}", [(k, tg[r]) for k, r in live.items()],
                _row_abs(tg))
    _assert_sum(dbeta, bt.grad, gln.abs().sum(0), 1e-5, f"predictor_tail_bwd.dbeta {what}", [(k, gln[r]) for k, r in live.items()],
                _row_abs(gln))


# ---------------------------------------------------------------------------------------------------
# elementwise: act_fwd, act_bwd (T or fp32 gradient), grad_cast, dropout_add
# ---------------------------------------------------------------------------------------------------
ONE_PASS = 2048 * 256 * 8
EW_N = {"small": 2056, "past-cap": 2 * ONE_PASS + 8 * 257}
EW_CASES = {f"act_fwd-{'gelu' if k == 1 else 'silu'}-{PREC_ID[pr]}": (0, k, pr) for k in (1, 2) for pr in (FP32, BF16, FP16)}
EW_CASES.update({f"act_bwd-{'gelu' if k == 1 else 'silu'}-{PREC_ID[pr]}": (1, k, pr) for k in (1, 2) for pr in (FP32, BF16, FP16)})
EW_CASES.update({f"act_bwd_f32grad-{'gelu' if k == 1 else 'silu'}-{PREC_ID[pr]}": (2, k, pr) for k in (1, 2) for pr in (BF16, FP16)})
EW_CASES.update({f"grad_cast-{PREC_ID[pr]}": (3, 0, pr) for pr in (FP32, BF16, FP16)})
EW_CASES.update({"dropout_add-resid": (4, 0, FP32), "dropout_add-noresid": (4, -1, FP32)})


def _act64(z, kind):
    return 0.5 * z * (1 + torch.erf(z / math.sqrt(2))) if kind == 1 else z * torch.sigmoid(z)


def _act_grad64(z, kind):
    if kind == 1:
        return 0.5 * (1 + torch.erf(z / math.sqrt(2))) + z * torch.exp(-0.5 * z * z) / math.sqrt(2 * math.pi)
    s = torch.sigmoid(z)
    return s * (1 + z * (1 - s))


@gpu
@pytest.mark.parametrize("nt", list(EW_N))
@pytest.mark.parametrize("case", list(EW_CASES))
def test_elementwise(case, nt):
    op, kind, prec = EW_CASES[case]
    n = EW_N[nt]
    p, site, step = 0.1, 21, 2
    T = DT[prec]
    g = _gen("ew", case, n)
    keep = _keep(p, site, step, n)
    a = _randn(g, n)
    a = torch.where(a.abs() < 0.05, torch.full_like(a, 0.5), a).clamp(-4, 4)  # non-zero, GELU / SiLU do not underflow in fp16
    b = _randn(g, n)
    out = torch.full((n + 8 * PAD,), float("nan"), device=DEV, dtype=T if op != 4 else torch.float32)
    if op == 0:
        z = a.to(T)
        _check(_lib().seqdiff_op_train_elementwise(0, prec, n, kind, _p(z), None, p, SEED, site, step, _p(out), stream_ptr()))
        ref, slack = _act64(z.double(), kind) * keep, 4e-7 * z.double().abs() * keep
        zero_is_mask = True
    elif op in (1, 2):
        z, da = a.to(T), (b.to(T) if op == 1 else b)
        _check(_lib().seqdiff_op_train_elementwise(op, prec, n, kind, _p(da), _p(z), p, SEED, site, step, _p(out), stream_ptr()))
        ref, slack = da.double() * keep * _act_grad64(z.double(), kind), 4e-7 * da.double().abs() * keep
        zero_is_mask = False
    elif op == 3:
        _check(_lib().seqdiff_op_train_elementwise(3, prec, n, 0, _p(a), None, p, SEED, site, step, _p(out), stream_ptr()))
        ref, slack = a.double() * keep, 0.0
        zero_is_mask = True
        # without dropout the cast is exact
        out0 = torch.empty(n, device=DEV, dtype=T)
        _check(_lib().seqdiff_op_train_elementwise(3, prec, n, 0, _p(a), None, 0.0, SEED, site, step, _p(out0), stream_ptr()))
        torch.cuda.synchronize()
        assert torch.equal(out0, a.to(T))
    else:
        resid = None if kind < 0 else b
        out[:n] = a
        _check(_lib().seqdiff_op_train_elementwise(4, FP32, n, 0, _p(resid), None, p, SEED, site, step, _p(out), stream_ptr()))
        ref = a.double() * keep + (0 if resid is None else resid.double())
        slack, zero_is_mask = 0.0, resid is None
    torch.cuda.synchronize()
    got = out[:n]
    assert torch.isnan(out[n:].float()).all(), "an element past n was written"
    if prec == FP32:
        err = (got.double() - ref).abs()
        bad = ~(err <= 2.0 ** -23 * ref.abs() + (1e-6 * ref.abs() + slack if op < 3 else 0.0))
        assert not bad.any(), f"{case}: {int(bad.sum())} elements off; worst {float(err.max()):.3e}"
    else:
        _assert_16bit(got, ref, prec, case, slack)
    if zero_is_mask:
        assert torch.equal(got == 0, keep == 0), f"{case}: zero pattern is not the dropout mask"


# ---------------------------------------------------------------------------------------------------
# transpose_colsum and colsum_add: small-integer inputs, exact results
# ---------------------------------------------------------------------------------------------------
def _ints(g, rows, cols, T):
    v = torch.randint(1, 9, (rows, cols), generator=g, device=DEV) * (torch.randint(0, 2, (rows, cols), generator=g, device=DEV) * 2 - 1)
    return v.to(T)


TC_SHAPES = [(1, 64, 8), (63, 100, 64), (100, 768, 104), (1037, 1024, 1040), (4097, 3072, 4104), (1000, 200, 0)]


@gpu
@pytest.mark.parametrize("rows,cols,pitch", TC_SHAPES)
@pytest.mark.parametrize("prec", [FP32, BF16, FP16], ids=PREC_ID.get)
def test_transpose_colsum(prec, rows, cols, pitch):
    i = TC_SHAPES.index((rows, cols, pitch))
    off = 4 if i % 2 == 0 else 5
    T = DT[prec]
    x = _ints(_gen("tc", prec, rows, cols), rows, cols, T)
    P = pitch or rows
    out = _nan(cols, P, T)
    cs = Acc((cols,), off, 15)
    _check(_lib().seqdiff_op_transpose_colsum(prec, rows, cols, _p(x), _p(out), pitch, _p(cs.t), stream_ptr()))
    torch.cuda.synchronize()
    assert torch.equal(out[:cols, :rows], x.t()), "transpose"
    assert (out[:cols, rows:P] == 0).all(), "pitch padding is not zero"
    _assert_nan_pad(out, cols, "transpose out")
    x64 = x.double()
    assert torch.equal(cs.t.double(), cs.pre.double() + x64.sum(0)), "column sums"
    _assert_sum(cs, x64.sum(0), x64.abs().sum(0), 0.0, "transpose_colsum.colsum",
                [(k, x64[r]) for k, r in _drop_rows(rows, 64).items()])
    # colsum only (out NULL)
    cs2 = Acc((cols,), 9 - off, 16)
    _check(_lib().seqdiff_op_transpose_colsum(prec, rows, cols, _p(x), None, pitch, _p(cs2.t), stream_ptr()))
    torch.cuda.synchronize()
    assert torch.equal(cs2.t.double(), cs2.pre.double() + x64.sum(0)), "column sums without the transpose"
    cs2.check_guards("colsum only")


@gpu
@pytest.mark.parametrize("off", [4, 5], ids=["aligned", "one-float-off"])
@pytest.mark.parametrize("rows,cols", [(1, 8), (63, 264), (1000, 768), (4097, 3072), (16389, 1024)])
@pytest.mark.parametrize("prec", [BF16, FP16], ids=PREC_ID.get)
def test_colsum_add(prec, rows, cols, off):
    x = _ints(_gen("cs", prec, rows, cols), rows, cols, DT[prec])
    cs = Acc((cols,), off, 17)
    _check(_lib().seqdiff_op_colsum_add(prec, rows, cols, _p(x), _p(cs.t), stream_ptr()))
    torch.cuda.synchronize()
    x64 = x.double()
    assert torch.equal(cs.t.double(), cs.pre.double() + x64.sum(0)), "column sums"
    _assert_sum(cs, x64.sum(0), x64.abs().sum(0), 0.0, "colsum_add", [(k, x64[r]) for k, r in _drop_rows(rows, 64).items()])


# ---------------------------------------------------------------------------------------------------
# loss gradients
# ---------------------------------------------------------------------------------------------------
@gpu
@pytest.mark.parametrize("case", ["mixed", "none-noised"])
@pytest.mark.parametrize("N", [1, 7, 4099, 16389])
def test_loss_bwd(N, case):
    """d(CE_mean + elbo over the noised rows)/d(logits): rows with x_t = x0 get 0, logits of +-80 on some rows; a batch without a noised
    row gets a zero gradient"""
    C = 20
    g = _gen("loss", N, case)
    logits = _randn(g, N, C, scale=3.0)
    r = torch.arange(N, device=DEV)
    big = (r % 5 == 1)
    logits[big] = torch.where(torch.rand(int(big.sum()), C, generator=g, device=DEV) < 0.5, -80.0, 80.0)
    x0 = F.one_hot(torch.randint(0, C, (N,), generator=g, device=DEV), C).float()
    xt = F.one_hot(torch.randint(0, C, (N,), generator=g, device=DEV), C).float()
    keep_clean = (r % 3 == 0) if case == "mixed" else torch.ones(N, dtype=torch.bool, device=DEV)
    xt[keep_clean] = x0[keep_clean]
    noised = xt.argmax(1) != x0.argmax(1)
    terms = torch.zeros(10, dtype=torch.float64, device=DEV)
    terms[1] = float(noised.sum())
    dl = _nan(N, C)
    _check(_lib().seqdiff_op_loss_bwd(N, _p(logits), _p(x0), _p(xt), _p(terms), _p(dl), stream_ptr()))
    torch.cuda.synchronize()
    z = logits.double().requires_grad_(True)
    if noised.any():
        zn = z[noised]
        (F.cross_entropy(zn, x0[noised].argmax(1)) + O.elbo_loss(zn, x0[noised].double())).backward()
        ref = z.grad
    else:
        ref = torch.zeros_like(z)
    _assert_rows(dl[:N], ref, 1e-5, f"loss_bwd ({case})")
    assert (dl[:N][~noised] == 0).all()
    _assert_nan_pad(dl, N, "dlogits")


@gpu
@pytest.mark.parametrize("valid", ["some", "none"])
@pytest.mark.parametrize("N", [1, 7, 16389])
@pytest.mark.parametrize("Fo", [8, 20])
def test_angle_loss_bwd(Fo, N, valid):
    """dL/dpred of the wrapped smooth-L1 angle loss at values next to the kink (|d| = pi / 10), next to +-pi (kept 1e-4 clear of the
    wrap's jump) and wrapped from beyond +-pi"""
    beta = math.pi / 10
    g = _gen("angle", Fo, N, valid)
    u = torch.rand(N, Fo, generator=g, device=DEV)
    sgn = torch.where(torch.rand(N, Fo, generator=g, device=DEV) < 0.5, -1.0, 1.0)
    kind = torch.randint(0, 4, (N, Fo), generator=g, device=DEV)
    d0 = torch.where(kind == 0, sgn * beta * (1 + (u - 0.5) * 2e-3),                     # at the kink
         torch.where(kind == 1, sgn * (math.pi - 1e-3 - u * 1e-2),                        # next to +-pi
         torch.where(kind == 2, sgn * (math.pi + 0.2 + u * 2.5), (u - 0.5) * 2.0)))      # wrapped; anywhere
    noise = _randn(g, N, Fo)
    pred = noise - d0
    diff = (noise - pred).double()  # the fp32 difference the kernel wraps
    rem = torch.remainder(diff + math.pi, 2 * math.pi)
    assert float(torch.minimum(rem, 2 * math.pi - rem).min()) > 1e-4, "a difference sits on the wrap's jump"
    mask = (torch.arange(N, device=DEV) % 4 != 3).float() if valid == "some" else torch.zeros(N, device=DEV)
    n_valid = float(mask.sum())
    terms = torch.zeros(Fo + 1, dtype=torch.float64, device=DEV)
    terms[Fo] = n_valid
    dp = _nan(N, Fo)
    _check(_lib().seqdiff_op_angle_loss_bwd(N, Fo, _p(pred), _p(noise), _p(mask), _p(terms), _p(dp), stream_ptr()))
    torch.cuda.synchronize()
    d = rem - math.pi
    hp = torch.where(d.abs() < beta, d / beta, torch.sign(d))
    ref = -hp / (Fo * n_valid) * mask.double()[:, None] if n_valid else torch.zeros_like(d)
    _assert_rows(dp[:N], ref, 1e-5, f"angle_loss_bwd (F {Fo})")
    assert (dp[:N][mask == 0] == 0).all()
    _assert_nan_pad(dp, N, "dpred")


@pytest.fixture(scope="module", autouse=True)
def _report_worst_errors():
    """after the module (pytest -s): the worst error of each output over the tests that ran -- per-row outputs relative to their row max,
    sums as a share of their gate"""
    yield
    for k in sorted(WORST):
        print(f"worst {k}: {WORST[k]:.3e}")
