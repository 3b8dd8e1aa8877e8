"""vf_gemm_bf16 / vf_gemm_bf16_ln across the whole contract of include/vf_b200.h (GPU box): K tails (the partial last
k-block and K < 64, TMA zero fill), N tails with the row statistics of partly empty tiles, ragged row counts on the
single-CTA kernel and on CTA pairs whose peer CTA has 0, 1 or 127 live rows, strided operands and outputs, element
offsets past 2^31, batch invariance of every epilogue form, the debug SIMT path against float64 (a child process: the
library reads VF_GEMM_DEBUG_SIMT once per process), and contract violations that must return an error without a launch.

The reference is float64 on the same bf16-rounded operands.  Per-element bound of an fp32 output:
    C_F32 * 2^-23 * (|A| @ |W|^T + |bias| + |resid|)
(bf16 outputs add one bf16 ulp of the value; GELU / GeGLU propagate it through the activation).  LayerNorm-folded
outputs are held to the relative bound of test_layernorm_fold_on_adversarial_streams.  Every output sits in a buffer
with sentinel rows above and below and sentinel columns right of its last column, which must come back bit-unchanged,
and every case checks that a reference wrong in one small way is rejected by the same bound."""
import math
import os
import subprocess
import sys

import pytest
import torch

pytestmark = pytest.mark.gpu

from variantformer_b200 import _lib, ops  # noqa: E402
from variantformer_b200._lib import (EPI_BIAS_BF16, EPI_BIAS_F32, EPI_BIAS_GEGLU_BF16, EPI_BIAS_GELU_BF16,  # noqa: E402
                                     EPI_BIAS_RESID_F32)

DEV = "cuda"
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PAD = 96                    # sentinel rows above and below every output
COLPAD = 40                 # sentinel columns right of every output (row stride = columns + COLPAD: a multiple of 8)
C_F32 = 16                  # fp32 bound: C_F32 ulps of the magnitude sum
LN_REL = 6e-3               # LayerNorm fold: max |err| / max |want| (test_gpu_kernels.py: adversarial streams)
GELU_ABS = 1e-5             # the epilogues' erf approximations (vf_common.cuh: |gelu error| <= 9.3e-6)
EPS = 1e-5
U = 2.0 ** -23
BF16 = {EPI_BIAS_BF16, EPI_BIAS_GELU_BF16, EPI_BIAS_GEGLU_BF16}


def _describe_mismatch(got, want, tol):
    if got.dim() == 1:
        got, want = got[:, None], want[:, None]
        tol = tol[:, None] if torch.is_tensor(tol) and tol.dim() == 1 else tol
    err = (got - want).abs()
    bad = err > tol
    rows = bad.any(1).nonzero().flatten().tolist()
    cols = bad.any(0).nonzero().flatten().tolist()
    return (f"max err {err.max().item():.4g} (max err / bound {(err / tol).max().item():.3g}), {int(bad.sum())} bad of "
            f"{bad.numel()}; bad rows[:16]={rows[:16]} (n={len(rows)}) bad cols[:16]={cols[:16]} (n={len(cols)})")


def _assert_within(got, want, tol, what=""):
    got = got.double()
    assert bool(((got - want).abs() <= tol).all()), f"{what}: " + _describe_mismatch(got, want, tol)


def _assert_rejected(got, wrong, tol, what):
    """The control: a reference that is wrong in one small way must fall outside the bound (the case has teeth)."""
    assert not bool(((got.double() - wrong).abs() <= tol).all()), f"{what}: the perturbed reference passes too"


# ---- operands, fenced outputs, the call --------------------------------------------------------------------------------
def _gen(seed):
    return torch.Generator(device="cpu").manual_seed(seed)


def _bf16(shape, g, scale=1.0, ld=None):
    """bf16 [rows, cols] on the device; ld > cols: a column view of a wider buffer (the rest is garbage)."""
    rows, cols = shape
    t = (torch.randn(rows, cols, generator=g) * scale).to(DEV).bfloat16()
    if ld is None or ld == cols:
        return t
    buf = torch.full((rows, ld), 3.0e4, dtype=torch.bfloat16, device=DEV)   # huge values where a K tail must not read
    buf[:, :cols] = t
    return buf[:, :cols]


def _fenced(M, cols, dtype, fill, ld=None):
    buf = torch.full((M + 2 * PAD, cols + COLPAD if ld is None else ld), fill, dtype=dtype, device=DEV)
    return buf, buf[PAD:PAD + M, :cols]


def _fence_intact(buf, M, cols):
    fill = buf.flatten()[0].item()
    assert bool((buf[:PAD] == fill).all()) and bool((buf[PAD + M:] == fill).all()), "sentinel rows overwritten"
    if buf.dim() == 2:
        assert bool((buf[PAD:PAD + M, cols:] == fill).all()), "sentinel columns overwritten"


class Run:
    """One GEMM through ops.gemm into fenced buffers: .out, .out2, .stats (views) after the call."""

    def __init__(self, a, w, epi, bias=None, resid=None, ln=None, mirror=False, stats=False, mirror_only=False,
                 inplace=False, ldo=None, ldo2=None):
        M, N = a.shape[0], w.shape[0]
        n_out = N // 2 if epi == EPI_BIAS_GEGLU_BF16 else N
        self.M, self.N, self.bufs = M, N, []
        self.out = self.out2 = self.stats = None
        f32 = epi in (EPI_BIAS_F32, EPI_BIAS_RESID_F32)
        if not mirror_only:
            b, self.out = _fenced(M, n_out, torch.float32 if f32 else torch.bfloat16, -777.0, ldo)
            self.bufs.append((b, n_out))
            if inplace:                                    # the FFN2 form: out is the fp32 residual stream
                self.out.copy_(resid)
                resid = self.out
        if mirror or mirror_only:
            b, self.out2 = _fenced(M, N, torch.bfloat16, -555.0, ldo2)
            self.bufs.append((b, N))
            if mirror_only and resid is not None and resid.dtype == torch.bfloat16:
                self.out2.copy_(resid)                     # the out_proj form: in place on the bf16 temporary
                resid = self.out2
        if stats:
            b = torch.full((M + 2 * PAD, ops.stats_parts(N), 2), 7.0, device=DEV)
            self.stats = b[PAD:PAD + M]
            self.bufs.append((b, None))
        ops.gemm(a, w, epi, bias=bias, resid=resid, out=None if mirror_only else self.out, out2=self.out2, ln=ln,
                 stats_out=self.stats, mirror_only=mirror_only)

    def fences(self):
        for b, cols in self.bufs:
            _fence_intact(b, self.M, cols)

    def outputs(self):
        return [t for t in (self.out, self.out2, self.stats) if t is not None]


# ---- the float64 reference ----------------------------------------------------------------------------------------------
def _gelu64(x):
    return 0.5 * x * (1.0 + torch.erf(x / math.sqrt(2.0)))


def _ln_of(x):
    """(mean, rstd) in float64 of the fp32 rows a bf16 mirror stands for."""
    x = x.double()
    return x.mean(1), 1.0 / torch.sqrt(x.var(1, unbiased=False) + EPS)


def _ref(a, w, epi, bias=None, resid=None, ln=None, drop_k=0, zero_last_row=False, bias_shift=False):
    """-> (want, bound) float64 [M, n_out].  ln = (mean, rstd, colsum): out = rstd (A W^T - mean colsum) + bias (the
    header's fold).  drop_k / zero_last_row / bias_shift build the wrong references of the controls."""
    A, W = a.double(), w.double()
    if zero_last_row:
        A = A.clone(); A[-1] = 0
    if drop_k:
        A, W = A[:, :A.shape[1] - drop_k], W[:, :W.shape[1] - drop_k]
    y = A @ W.t()
    mag = A.abs() @ W.abs().t()
    if ln is not None:
        mean, rstd, cs = ln
        cs = cs.double()
        y = rstd[:, None] * (y - mean[:, None] * cs[None])
        mag = rstd[:, None] * (mag + mean.abs()[:, None] * cs.abs()[None])
    if bias is not None:
        b = bias.double().clone()
        if bias_shift:
            b[-1] += 1.0
        y = y + b
        mag = mag + b.abs()
    if resid is not None:
        y = y + resid.double()
        mag = mag + resid.double().abs()
    e = C_F32 * U * mag
    if epi == EPI_BIAS_GEGLU_BF16:
        j = torch.arange(w.shape[0] // 2, device=DEV)
        iu = (j // 128) * 256 + j % 128
        u, g, eu, eg = y[:, iu], y[:, iu + 128], e[:, iu], e[:, iu + 128]
        y = u * _gelu64(g)
        e = _gelu64(g).abs() * eu + (u.abs() + eu) * (1.2 * eg + GELU_ABS)
    elif epi == EPI_BIAS_GELU_BF16:
        y = _gelu64(y)
        e = 1.2 * e + GELU_ABS
    if epi in BF16:
        e = e + 2.0 ** -8 * y.abs()
    if ln is not None:
        e = torch.full_like(y, LN_REL * float(y.abs().max()))
    return y, e


def _check_stats(st, vals, what, slack=None):
    """Partials [M, P, 2] of a row add up to the row's sum and sum of squares of the fp32 values vals (float64 [M, N]);
    slack [M, N]: how far the fp32 values the kernel summed may be from vals (0 when vals are its own fp32 outputs).
    Bound: n * 2^-23 times the sum of magnitudes, twice the first-order error of ANY order of n fp32 additions (and of
    the products of the squares); the control: the sums without the last column must be rejected."""
    tot = st.double().sum(1)
    n = vals.shape[1]
    sq = vals * vals
    e1, e2 = n * U * vals.abs().sum(1), n * U * sq.sum(1)
    if slack is not None:
        e1 = e1 + slack.sum(1)
        e2 = e2 + (2 * vals.abs() * slack + slack * slack).sum(1)
    _assert_within(tot[:, 0], vals.sum(1), e1, f"{what}: row sums")
    _assert_within(tot[:, 1], sq.sum(1), e2, f"{what}: row sums of squares")
    _assert_rejected(tot[:, 0], vals[:, :-1].sum(1), e1, f"{what}: row sums without the last column")
    _assert_rejected(tot[:, 1], sq[:, :-1].sum(1), e2, f"{what}: row sums of squares without the last column")


def _empty_halves(N):
    """Partial indices of the 128-column halves (epilogue warp halves: 32-column slabs of one parity) that hold no
    column < N."""
    return [2 * t + h for t in range((N + 255) // 256) for h in (0, 1) if t * 256 + h * 32 >= N]


# Forms of the contract: (name, epilogue, extra keyword arguments of Run, residual kind)
FORMS = [
    ("bias", EPI_BIAS_BF16, {}, None),
    ("gelu", EPI_BIAS_GELU_BF16, {}, None),
    ("geglu", EPI_BIAS_GEGLU_BF16, {}, None),
    ("f32+mirror+stats", EPI_BIAS_F32, dict(mirror=True, stats=True), None),
    ("resid32+out+mirror+stats", EPI_BIAS_RESID_F32, dict(mirror=True, stats=True), "f32"),
    ("ffn2 in place+mirror+stats", EPI_BIAS_RESID_F32, dict(mirror=True, stats=True, inplace=True), "f32"),
    ("resid16 mirror-only+stats", EPI_BIAS_RESID_F32, dict(mirror_only=True, stats=True), "bf16"),
]


def _operands(M, N, K, seed, lda=None, ldw=None):
    g = _gen(seed)
    a = _bf16((M, K), g, 0.5, lda)
    w = _bf16((N, K), g, 1 / math.sqrt(K), ldw)
    bias = torch.randn(N, generator=g).to(DEV)
    resid = (torch.randn(M, N, generator=g) * 2).to(DEV)
    return a, w, bias, resid


def _check_form(r, a, w, epi, bias, resid, kw, control, what, ln=None):
    """Values (out, mirror) against the float64 reference, statistics, fences, and the control."""
    want, tol = _ref(a, w, epi, bias, resid, ln)
    main = r.out2 if kw.get("mirror_only") else r.out
    _assert_within(main, want, tol + (2.0 ** -8 * want.abs() if kw.get("mirror_only") else 0), what)
    if r.out2 is not None and not kw.get("mirror_only"):
        assert torch.equal(r.out2, r.out.bfloat16()), f"{what}: mirror != bf16(out)"
    if r.stats is not None:
        if r.out is not None:
            _check_stats(r.stats, r.out.double(), what)
        else:                                              # mirror only: the fp32 values are within tol of want
            _check_stats(r.stats, want, what, slack=tol)
        for p in _empty_halves(r.N):
            assert bool((r.stats[:, p] == 0).all()), f"{what}: partial {p} of an empty half tile is not 0"
    r.fences()
    wrong, _ = _ref(a, w, epi, bias, resid, ln, **control)
    _assert_rejected(main, wrong, tol + (2.0 ** -8 * want.abs() if kw.get("mirror_only") else 0), f"{what}: control {control}")


def _resid_for(kind, resid):
    return None if kind is None else resid if kind == "f32" else resid.bfloat16()


# ---------------------------------------------------------------------------------------------------------------------
# a. K tails: the partial last k-block (TMA zero fill) and K < 64, every epilogue, with and without the LayerNorm fold
def _ln_inputs(M, K, N, g, source):
    """A = bf16 mirror of an fp32 stream x [M, K] with its row statistics, from vf_center_rows or from a producing fp32
    GEMM's stats_out; gamma-folded weight (random), its fp32 column sums.  -> (a, w, cs, stats, (mean, rstd, cs))."""
    if source == "center_rows":
        x = (torch.randn(M, K, generator=g) * 1.5 + 4.0).to(DEV)
        xb = torch.empty(M, K, dtype=torch.bfloat16, device=DEV)
        _, st = ops.center_rows(x, out_bf16=xb)
    else:
        K0 = 64
        a0 = _bf16((M, K0), g, 0.5); w0 = _bf16((K, K0), g, 1 / math.sqrt(K0))
        b0 = torch.randn(K, generator=g).to(DEV)
        x = torch.empty(M, K, device=DEV); xb = torch.empty(M, K, dtype=torch.bfloat16, device=DEV)
        st = torch.empty(M, ops.stats_parts(K), 2, device=DEV)
        ops.gemm(a0, w0, EPI_BIAS_F32, bias=b0, out=x, out2=xb, stats_out=st)
    w = _bf16((N, K), g, 1 / math.sqrt(K))
    cs = w.float().sum(1).contiguous()
    mean, rstd = _ln_of(x)
    return xb, w, cs, st, (mean, rstd, cs)


@pytest.mark.parametrize("M", [300, 1100])
@pytest.mark.parametrize("K", [8, 24, 40, 72, 200, 520, 1544])
def test_k_tails(K, M):
    seed = 11 * K + M
    for name, epi, kw, rk in FORMS:
        N = 512
        a, w, bias, resid = _operands(M, N, K, seed)
        r = Run(a, w, epi, bias=bias, resid=_resid_for(rk, resid), **kw)
        torch.cuda.synchronize()
        _check_form(r, a, w, epi, bias, _resid_for(rk, resid), kw, dict(drop_k=8), f"{name} K={K} M={M}")
    for epi in (EPI_BIAS_BF16, EPI_BIAS_GELU_BF16, EPI_BIAS_GEGLU_BF16):
        for source in ("center_rows", "stats_out"):
            g = _gen(seed + epi)
            a, w, cs, st, ln_ref = _ln_inputs(M, K, 512, g, source)
            bias = torch.randn(512, generator=g).to(DEV)
            r = Run(a, w, epi, bias=bias, ln=(st, cs, K, EPS))
            torch.cuda.synchronize()
            _check_form(r, a, w, epi, bias, None, {}, dict(drop_k=8), f"ln {source} epi={epi} K={K} M={M}", ln=ln_ref)


# ---------------------------------------------------------------------------------------------------------------------
# b. N tails and the row statistics of partly empty tiles; the LayerNorm-folded consumer of those statistics
@pytest.mark.parametrize("M,K", [(300, 192), (1100, 512)])
@pytest.mark.parametrize("N", [8, 24, 40, 264, 328, 520, 776])
def test_n_tails_and_row_statistics(N, M, K):
    seed = 7 * N + M
    for name, epi, kw, rk in FORMS:
        n = (256 if N < 512 else 768) if epi == EPI_BIAS_GEGLU_BF16 else N
        a, w, bias, resid = _operands(M, n, K, seed)
        r = Run(a, w, epi, bias=bias, resid=_resid_for(rk, resid), **kw)
        torch.cuda.synchronize()
        _check_form(r, a, w, epi, bias, _resid_for(rk, resid), kw, dict(bias_shift=True), f"{name} N={n} M={M}")
    # consumer: Linear(LayerNorm(x)) on the mirror and statistics of an fp32 producer with N output columns
    g = _gen(seed + 1)
    a, w, bias, _ = _operands(M, N, K, seed + 2)
    p = Run(a, w, EPI_BIAS_F32, bias=bias, mirror=True, stats=True)
    N2 = 264
    gamma = (1 + 0.2 * torch.randn(N, generator=g)).to(DEV); beta = (0.1 * torch.randn(N, generator=g)).to(DEV)
    w2 = (torch.randn(N2, N, generator=g) / math.sqrt(N)).to(DEV); b2 = torch.randn(N2, generator=g).to(DEV)
    wf = (w2 * gamma[None, :]).bfloat16().contiguous(); cs = wf.float().sum(1).contiguous(); bf = (b2 + w2 @ beta).contiguous()
    c = Run(p.out2, wf, EPI_BIAS_BF16, bias=bf, ln=(p.stats, cs, N, EPS))
    torch.cuda.synchronize()
    x = p.out.double()
    want = torch.nn.functional.linear(torch.nn.functional.layer_norm(x, (N,), gamma.double(), beta.double(), EPS),
                                      w2.double(), b2.double())
    tol = LN_REL * float(want.abs().max())
    _assert_within(c.out, want, tol, f"Linear(LayerNorm(x)) N={N}")
    wrong = want.clone(); wrong[:, -1] += 1.0
    _assert_rejected(c.out, wrong, tol, "consumer bias of the last column + 1")
    c.fences()


# ---------------------------------------------------------------------------------------------------------------------
# c. Ragged M on both kernels: single CTA below 1024 rows, CTA pairs above (K >= 512) whose last pair tile leaves the
#    peer CTA 0, 1 or 127 live rows
@pytest.mark.parametrize("M", [1, 2, 31, 33, 127, 129, 1024, 1025, 1151, 1152, 1153, 1279, 1281])
def test_ragged_rows_on_both_kernels(M):
    K, N = 512, 512
    for name, epi, kw, rk in FORMS:
        a, w, bias, resid = _operands(M, N, K, M + epi)
        r = Run(a, w, epi, bias=bias, resid=_resid_for(rk, resid), **kw)
        torch.cuda.synchronize()
        _check_form(r, a, w, epi, bias, _resid_for(rk, resid), kw, dict(zero_last_row=True), f"{name} M={M}")


# ---------------------------------------------------------------------------------------------------------------------
# d. Strides: A and W column views of wider buffers (as the engine's qkv slices), outputs with ldo > n_out and
#    n_out % 32 != 0 (the TMA store clipped at the N edge), a residual with ldr != ldo
@pytest.mark.parametrize("M", [300, 1100])
def test_strided_operands_and_outputs(M):
    K = 520
    for name, epi, kw, rk in FORMS:
        N = 512 if epi == EPI_BIAS_GEGLU_BF16 else 328
        n_out = N // 2 if epi == EPI_BIAS_GEGLU_BF16 else N
        a, w, bias, resid = _operands(M, N, K, M + 3 * epi, lda=K + 64, ldw=K + 64)
        assert a.stride(0) == K + 64 and w.stride(0) == K + 64
        res = _resid_for(rk, resid)
        if res is not None and not kw.get("inplace") and not kw.get("mirror_only"):
            rbuf = torch.full((M, N + 72), 1e6, dtype=res.dtype, device=DEV)   # ldr = N + 72 != ldo
            rbuf[:, :N] = res
            res = rbuf[:, :N]
        r = Run(a, w, epi, bias=bias, resid=res, ldo=512, ldo2=512, **kw)
        torch.cuda.synchronize()
        if r.out is not None:
            assert r.out.stride(0) == 512 and n_out % 32 != 0 or epi == EPI_BIAS_GEGLU_BF16
        _check_form(r, a, w, epi, bias, res, kw, dict(drop_k=8), f"{name} strided M={M}")


# ---------------------------------------------------------------------------------------------------------------------
# e. Element offsets past 2^31 (checked on sampled row blocks: the first 256 rows, the 256 rows that straddle element
#    2^31 of the output, the last 256 rows)
def _sample_rows(M, ld):
    r = (2 ** 31) // ld
    assert M * ld > 2 ** 31 and 128 <= r < M - 128
    return torch.cat([torch.arange(0, 256), torch.arange(r - 128, r + 128), torch.arange(M - 256, M)]).to(DEV)


def test_element_offsets_past_2_31():
    g = torch.Generator(device=DEV).manual_seed(31)
    # LayerNorm-folded Wqkv at its production form
    M, N, K = 470_000, 4608, 512
    x = torch.randn(M, K, generator=g, device=DEV) * 1.5 + 2.0
    xb = torch.empty(M, K, dtype=torch.bfloat16, device=DEV)
    _, st = ops.center_rows(x, out_bf16=xb)
    w = (torch.randn(N, K, generator=g, device=DEV) / math.sqrt(K)).bfloat16()
    cs = w.float().sum(1).contiguous(); bias = torch.randn(N, generator=g, device=DEV)
    r = Run(xb, w, EPI_BIAS_BF16, bias=bias, ln=(st, cs, K, EPS))
    torch.cuda.synchronize()
    rows = _sample_rows(M, r.out.stride(0))
    mean, rstd = _ln_of(x[rows])
    want, tol = _ref(xb[rows], w, EPI_BIAS_BF16, bias, ln=(mean, rstd, cs))
    _assert_within(r.out[rows], want, tol, "LN-folded Wqkv past 2^31")
    wrong, _ = _ref(xb[rows], w, EPI_BIAS_BF16, bias, ln=(mean, rstd, cs), drop_k=8)
    _assert_rejected(r.out[rows], wrong, tol, "LN-folded Wqkv past 2^31: K - 8")
    r.fences()
    del r, x, xb, st, w
    torch.cuda.empty_cache()
    # fp32 output with mirror and statistics
    M, N, K = 1_400_000, 1536, 512
    a = (torch.randn(M, K, generator=g, device=DEV) * 0.5).bfloat16()
    w = (torch.randn(N, K, generator=g, device=DEV) / math.sqrt(K)).bfloat16()
    bias = torch.randn(N, generator=g, device=DEV)
    r = Run(a, w, EPI_BIAS_F32, bias=bias, mirror=True, stats=True)
    torch.cuda.synchronize()
    rows = _sample_rows(M, r.out.stride(0))
    want, tol = _ref(a[rows], w, EPI_BIAS_F32, bias)
    _assert_within(r.out[rows], want, tol, "fp32 past 2^31")
    assert torch.equal(r.out2[rows], r.out[rows].bfloat16())
    _check_stats(r.stats[rows], r.out[rows].double(), "fp32 past 2^31")
    wrong, _ = _ref(a[rows], w, EPI_BIAS_F32, bias, drop_k=8)
    _assert_rejected(r.out[rows], wrong, tol, "fp32 past 2^31: K - 8")
    r.fences()
    del r, a, w
    torch.cuda.empty_cache()


# ---------------------------------------------------------------------------------------------------------------------
# f. Batch invariance: rows [0, 640) of an M = 2304 call (CTA pairs) are bit-identical to an M = 640 call (single CTA)
#    and to an M = 1025 call, in every form (values, mirror, statistics): DESIGN section 7's gather check rests on it
INV_FORMS = [
    ("bias", EPI_BIAS_BF16, {}, None, False), ("bias+ln", EPI_BIAS_BF16, {}, None, True),
    ("gelu", EPI_BIAS_GELU_BF16, {}, None, False), ("gelu+ln", EPI_BIAS_GELU_BF16, {}, None, True),
    ("geglu", EPI_BIAS_GEGLU_BF16, {}, None, False), ("geglu+ln", EPI_BIAS_GEGLU_BF16, {}, None, True),
    ("f32+mirror+stats", EPI_BIAS_F32, dict(mirror=True, stats=True), None, False),
    ("resid32+out+mirror+stats", EPI_BIAS_RESID_F32, dict(mirror=True, stats=True), "f32", False),
    ("resid16 mirror-only+stats", EPI_BIAS_RESID_F32, dict(mirror_only=True, stats=True), "bf16", False),
]


def _inv_inputs(M, N, K, seed, epi, ln):
    g = _gen(seed)
    if ln:
        x = (torch.randn(M, K, generator=g) + 3.0).to(DEV)
        a = torch.empty(M, K, dtype=torch.bfloat16, device=DEV)
        _, st = ops.center_rows(x, out_bf16=a)
    else:
        a, st = _bf16((M, K), g, 0.5), None
    w = _bf16((N, K), g, 1 / math.sqrt(K))
    bias = torch.randn(N, generator=g).to(DEV)
    resid = (torch.randn(M, N, generator=g) * 2).to(DEV)
    return a, w, bias, resid, st


def _run_rows(rows, a, w, epi, bias, resid, st, kw, rk):
    res = _resid_for(rk, resid)
    ln = (st[:rows].contiguous(), w.float().sum(1).contiguous(), a.shape[1], EPS) if st is not None else None
    r = Run(a[:rows].contiguous(), w, epi, bias=bias, resid=None if res is None else res[:rows].contiguous(), ln=ln, **kw)
    return r


@pytest.mark.parametrize("N", [768, 1536, 1288])
@pytest.mark.parametrize("K", [512, 1536])
def test_rows_do_not_depend_on_how_many_rows_are_batched(K, N):
    for name, epi, kw, rk, ln in INV_FORMS:
        if epi == EPI_BIAS_GEGLU_BF16 and N % 256:
            continue
        a, w, bias, resid, st = _inv_inputs(2304, N, K, K + N + epi, epi, ln)
        big = _run_rows(2304, a, w, epi, bias, resid, st, kw, rk)
        for rows in (640, 1025):
            small = _run_rows(rows, a, w, epi, bias, resid, st, kw, rk)
            torch.cuda.synchronize()
            for b, s in zip(big.outputs(), small.outputs()):
                assert torch.equal(b[:640], s[:640]), f"{name} K={K} N={N}: rows of M=2304 != rows of M={rows}"
            small.fences()
        big.fences()


# ---------------------------------------------------------------------------------------------------------------------
# g. The debug SIMT path (read once per process: it runs in a child process) agrees with float64
def _ab_cases():
    """name -> (a, w, epi, bias, resid, ln, Run keywords): each form of (f), the out_proj and FFN2 residual forms at
    M >= 1024, a K-tail case and an N-tail case."""
    cases = {}
    for name, epi, kw, rk, ln in INV_FORMS:
        for N in ((768, 1288) if epi != EPI_BIAS_GEGLU_BF16 else (768,)):
            a, w, bias, resid, st = _inv_inputs(1100, N, 512, N + epi + 100 * ln, epi, ln)
            lnarg = (st, w.float().sum(1).contiguous(), 512, EPS) if ln else None
            cases[f"{name} N={N}"] = (a, w, epi, bias, _resid_for(rk, resid), lnarg, kw)
    a, w, bias, resid = _operands(1300, 768, 512, 5)
    cases["out_proj"] = (a, w, EPI_BIAS_RESID_F32, bias, resid.bfloat16(), None, dict(mirror_only=True, stats=True))
    cases["ffn2"] = (a, w, EPI_BIAS_RESID_F32, bias, resid, None, dict(mirror=True, stats=True, inplace=True))
    a, w, bias, resid = _operands(1100, 512, 520, 6)
    cases["k tail"] = (a, w, EPI_BIAS_RESID_F32, bias, resid, None, dict(mirror=True, stats=True))
    a, w, bias, resid = _operands(1100, 328, 512, 7)
    cases["n tail"] = (a, w, EPI_BIAS_F32, bias, None, None, dict(mirror=True, stats=True))
    # M >= 1024 with K < 512 (one to seven k-blocks, K < 64 included)
    a, w, bias, resid = _operands(1100, 512, 200, 8)
    cases["k tail K=200"] = (a, w, EPI_BIAS_RESID_F32, bias, resid, None, dict(mirror=True, stats=True))
    a, w, bias, resid = _operands(1100, 512, 40, 9)
    cases["geglu K=40"] = (a, w, EPI_BIAS_GEGLU_BF16, bias, None, None, {})
    a, w, bias, resid = _operands(1300, 768, 72, 10)
    cases["ffn2 K=72"] = (a, w, EPI_BIAS_RESID_F32, bias, resid, None, dict(mirror=True, stats=True, inplace=True))
    cases["out_proj K=72"] = (a, w, EPI_BIAS_RESID_F32, bias, resid.bfloat16(), None, dict(mirror_only=True, stats=True))
    a, w, bias, resid, st = _inv_inputs(1300, 768, 192, 11, EPI_BIAS_BF16, True)
    cases["bias+ln K=192"] = (a, w, EPI_BIAS_BF16, bias, None, (st, w.float().sum(1).contiguous(), 192, EPS), {})
    assert sum(a.shape[0] >= 1024 and a.shape[1] < 512 for a, *_ in cases.values()) == 5
    return cases


def _ab_child(out_path):
    """Runs every _ab_cases() GEMM under this process's VF_GEMM_DEBUG_SIMT setting and saves the outputs (CPU tensors)."""
    torch.cuda.set_device(0)
    res = {}
    for name, (a, w, epi, bias, resid, ln, kw) in _ab_cases().items():
        r = Run(a, w, epi, bias=bias, resid=resid, ln=ln, **kw)
        torch.cuda.synchronize()
        r.fences()
        res[name] = [t.cpu() for t in r.outputs()]
    torch.save(res, out_path)


def _child(tmp_path, tag, switch):
    env = {k: v for k, v in os.environ.items() if not k.startswith("VF_GEMM_")}
    env.update(switch)
    path = str(tmp_path / f"{tag}.pt")
    code = ("import sys; from tests.test_gpu_gemm_contract import _ab_child; _ab_child(sys.argv[1])")
    p = subprocess.run([sys.executable, "-c", code, path], cwd=ROOT, env=env, timeout=600, capture_output=True, text=True)
    assert p.returncode == 0, f"{switch}: child failed ({p.returncode})\n{p.stdout[-2000:]}\n{p.stderr[-4000:]}"
    return torch.load(path)


def test_debug_simt_path_agrees_with_float64(tmp_path):
    got = _child(tmp_path, "simt", {"VF_GEMM_DEBUG_SIMT": "1"})
    for name, (a, w, epi, bias, resid, ln, kw) in _ab_cases().items():
        lnref = None
        if ln is not None:
            st = ln[0].double().sum(1)                    # the stream is row-centred: the mirror's own statistics
            mean = st[:, 0] / ln[2]
            lnref = (mean, 1.0 / torch.sqrt(st[:, 1] / ln[2] - mean * mean + EPS), ln[1])
        want, tol = _ref(a, w, epi, bias, resid, lnref)
        outs = [t.to(DEV) for t in got[name]]
        main = outs[0]
        _assert_within(main, want, tol + (2.0 ** -8 * want.abs() if kw.get("mirror_only") else 0), f"SIMT {name}")
        if kw.get("mirror") and not kw.get("mirror_only"):
            assert torch.equal(outs[1], main.bfloat16()), f"SIMT {name}: mirror != bf16(out)"
        if kw.get("stats"):
            if kw.get("mirror_only"):
                _check_stats(outs[-1], want, f"SIMT {name}", slack=tol)
            else:
                _check_stats(outs[-1], main.double(), f"SIMT {name}")


# ---------------------------------------------------------------------------------------------------------------------
# h. Contract violations return an error, name it, and launch nothing
def _raw(A=None, lda=64, W=None, ldw=64, M=128, N=256, K=64, epi=EPI_BIAS_BF16, bias=None, resid=None, resid16=0, ldr=0,
         out=None, ldo=256, out2=None, ldo2=0, ln_stats=None, ln_parts=0, ln_colsum=None, ln_dim=0, stats_out=None):
    L = _lib.lib()
    return L.vf_gemm_bf16_ln(A, lda, W, ldw, M, N, K, epi, bias, resid, resid16, ldr, out, ldo, out2, ldo2, ln_stats,
                             ln_parts, ln_colsum, ln_dim, EPS, stats_out, _lib.stream())


def _expect_error(what, needle, **kw):
    n0 = ops.launch_count()
    rc = _raw(**kw)
    msg = _lib.load().vf_last_error().decode()
    assert rc < 0, f"{what}: returned {rc}"
    assert needle in msg, f"{what}: error message {msg!r} does not mention {needle!r}"
    assert ops.launch_count() == n0, f"{what}: launched a kernel"


def test_contract_violations_return_errors_without_launching():
    M, N, K = 128, 256, 64
    buf = torch.zeros(1 << 22, dtype=torch.uint8, device=DEV)    # one allocation, carved by hand (256-byte aligned)
    base = buf.data_ptr()
    A, W, O, O2, R, S, LS, CS, B = (base + i * (1 << 18) for i in range(9))
    ok = dict(A=A, W=W, out=O, bias=B)
    torch.cuda.synchronize()
    _expect_error("N % 8", "multiples of 8", **dict(ok, N=260, ldo=264))
    _expect_error("K % 8", "multiples of 8", **dict(ok, K=60))
    _expect_error("GeGLU N % 256", "GeGLU", **dict(ok, epi=EPI_BIAS_GEGLU_BF16, N=264, ldo=136))
    _expect_error("stats_out with a bf16 epilogue", "row statistics", **dict(ok, stats_out=S))
    _expect_error("LN fold with an fp32 epilogue", "LayerNorm fold",
                  **dict(ok, epi=EPI_BIAS_F32, ln_stats=LS, ln_parts=1, ln_colsum=CS, ln_dim=K))
    _expect_error("ldo < n_out", "output stride", **dict(ok, ldo=248))
    _expect_error("no output", "no output", **dict(ok, out=None))
    _expect_error("A 8 bytes off", "16-byte aligned", **dict(ok, A=A + 8))
    _expect_error("W 8 bytes off", "16-byte aligned", **dict(ok, W=W + 8))
    n0 = ops.launch_count()
    assert _raw(**dict(ok, M=0)) == 0 and ops.launch_count() == n0, "M == 0 must return 0 without a launch"
    # The operands the epilogue writes: probe first with M = 0 (no launch whatever the library does); only a library
    # that rejects the probe may see the M > 0 calls below.
    n0 = ops.launch_count()
    probe = _raw(**dict(ok, M=0, out=O + 8))
    assert ops.launch_count() == n0
    if probe >= 0:
        pytest.fail("vf_gemm_bf16_ln accepts a misaligned output at M == 0: this library does not validate the operands "
                    "its epilogue writes, so the misaligned M > 0 cases are not run")
    f32 = dict(ok, epi=EPI_BIAS_F32)
    _expect_error("bf16 out 8 bytes off", "output must be 16-byte aligned", **dict(ok, out=O + 8))
    _expect_error("fp32 out 4 bytes off", "output must be 16-byte aligned", **dict(f32, out=O + 4))
    _expect_error("mirror 8 bytes off", "mirror", **dict(f32, out2=O2 + 8, ldo2=N))
    _expect_error("mirror stride", "mirror", **dict(f32, out2=O2, ldo2=N + 4))
    rs = dict(f32, epi=EPI_BIAS_RESID_F32)
    _expect_error("fp32 residual 8 bytes off", "residual", **dict(rs, resid=R + 8, ldr=N))
    _expect_error("fp32 residual stride", "residual", **dict(rs, resid=R, ldr=N + 2))
    _expect_error("bf16 residual 8 bytes off", "residual", **dict(rs, out=None, out2=O2, ldo2=N, resid=R + 8, resid16=1, ldr=N))
    _expect_error("bf16 residual stride", "residual", **dict(rs, out=None, out2=O2, ldo2=N, resid=R, resid16=1, ldr=N + 4))
    _expect_error("stats_out 4 bytes off", "stats_out", **dict(f32, stats_out=S + 4))
    _expect_error("ln_stats 4 bytes off", "ln_stats", **dict(ok, ln_stats=LS + 4, ln_parts=1, ln_colsum=CS, ln_dim=K))
    _expect_error("ln_stats 8 bytes off, even parts", "ln_stats",
                  **dict(ok, ln_stats=LS + 8, ln_parts=2, ln_colsum=CS, ln_dim=K))
    for what, kw in (("out", dict(ok, out=O + 8)), ("stats_out", dict(f32, stats_out=S + 4))):
        n0 = ops.launch_count()
        assert _raw(**dict(kw, M=0)) < 0 and ops.launch_count() == n0, f"misaligned {what} at M == 0"
    torch.cuda.synchronize()
    del buf
