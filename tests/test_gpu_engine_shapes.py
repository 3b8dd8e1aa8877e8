"""Kernel parity at the launch shapes only the engine makes (GPU box): the last gene layer's explicit attention tables
(SlotMap.from_units: one-row ALiBi tiles at arbitrary positions, runs of one gene's rows against its CREs), stacked
cross-attention at production tile counts, the in-place FFN2 residual epilogue at ragged row counts with and without
its mirror and statistics, label attention over every head group, and stage-1 batches of more windows than one
launch's grid.y holds.  References are plain fp32 restatements of each operation (TF32 off, the torch default); every
case also checks that a slightly wrong reference is rejected, so the tolerance cannot hide an off-by-one."""
import math

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import stage1 as O  # noqa: E402  (checker only)
from variantformer_b200 import ops  # noqa: E402
from variantformer_b200._lib import EPI_BIAS_RESID_F32  # noqa: E402
from variantformer_b200.stage1 import Genome, SampleVariants, WindowTokenizer, cre_window  # noqa: E402
from variantformer_b200.utils import synth  # noqa: E402

DEV = "cuda"


def _describe_mismatch(got, want, tol):
    err = (got - want).abs()
    bad = err > tol
    rows = bad.any(1).nonzero().flatten().tolist()
    cols = bad.any(0).nonzero().flatten().tolist()
    return (f"max err {err.max().item():.4g} (tol {tol:.3g}), {int(bad.sum())} bad of {bad.numel()}; "
            f"bad rows[:16]={rows[:16]} (n={len(rows)}) bad cols[:16]={cols[:16]} (n={len(cols)}); "
            f"got[0,:4]={got[0, :4].tolist()} want[0,:4]={want[0, :4].tolist()}")


def _assert_close(got, want, tol):
    assert torch.allclose(got.float(), want, atol=tol, rtol=tol), _describe_mismatch(got.float(), want, tol)


def _assert_rejected(got, wrong, tol, what):
    """The control: a reference that is wrong in one small way must fall outside the tolerance (the case has teeth)."""
    assert not torch.allclose(got.float(), wrong, atol=tol, rtol=tol), f"{what}: the perturbed reference passes too"


def _slopes(H):
    return torch.tensor([2 ** (-8 * (h + 1) / H) for h in range(H)], device=DEV)


def _ref_units(q, k, v, units, H, hd, slopes):
    """The slot record of include/vf_b200.h restated in fp32: for each unit {q0, n, k0, Sk, pos0}, rows q0 .. q0+n
    attend over keys k0 .. k0+Sk with the ALiBi bias -slope_h * |pos0 + i - j|; a unit without keys gives zero rows."""
    out = torch.zeros(q.shape[0], H * hd, device=q.device)
    for q0, n, k0, sk, pos0 in np.asarray(units, np.int64).reshape(-1, 5).tolist():
        if n == 0 or sk == 0:
            continue
        kk = k[k0:k0 + sk].float().view(sk, H, hd); vv = v[k0:k0 + sk].float().view(sk, H, hd)
        for r0 in range(0, n, 2048):                             # row chunks keep the score tensor small
            r1 = min(n, r0 + 2048)
            qq = q[q0 + r0:q0 + r1].float().view(r1 - r0, H, hd)
            s = torch.einsum("thd,shd->hts", qq, kk) / math.sqrt(hd)
            if slopes is not None:
                i = torch.arange(r0, r1, device=q.device)[:, None]; j = torch.arange(sk, device=q.device)[None, :]
                s = s - slopes[:, None, None] * (pos0 + i - j).abs()[None]
            out[q0 + r0:q0 + r1] = torch.einsum("hts,shd->thd", s.softmax(-1), vv).reshape(r1 - r0, H * hd)
    return out


def _shift_pos(units):
    u = np.array(units, np.int64); u[:, 4] += 1
    return u


def _drop_last_key(units):
    u = np.array(units, np.int64); u[:, 3] = np.maximum(u[:, 3] - 1, 0)
    return u


def _run_units(monkeypatch, pair, q, k, v, units, H, hd, slopes, fill=7.0):
    """attention_mc on the table SlotMap.from_units builds with PAIR_UNRELATED_TILES = pair (read at call time);
    the output buffer starts as `fill` so that rows the kernel skips show up."""
    monkeypatch.setattr(ops, "PAIR_UNRELATED_TILES", pair)
    slots = ops.SlotMap.from_units(units, DEV)
    out = torch.full((q.shape[0], H * hd), fill, dtype=torch.bfloat16, device=DEV)
    ops.attention_mc(q, k, v, slots, H, hd, slopes, out=out)
    torch.cuda.synchronize()
    return out, slots


# ---------------------------------------------------------------------------------------------------------------------
# A. Last-layer self-attention: one-row query tiles at arbitrary ALiBi positions (engine.py, _prepare_seq2gene)
SEQ_LENS = [1, 2, 63, 64, 65, 127, 128, 129, 201, 301]


def _needed_rows(R, rng):
    """(sequence, offset) of R needed rows: every sequence at offsets 0, len-1, 63, 64, 127, 128 (where they exist),
    then random offsets; R = 1 / 2 pick rows whose tiles straddle the 64-key blocks."""
    if R == 1:
        return [(9, 128)]
    if R == 2:
        return [(0, 0), (7, 64)]
    need = []
    for s, n in enumerate(SEQ_LENS):
        need += [(s, o) for o in sorted({0, n - 1, 63, 64, 127, 128}) if o < n]
    while len(need) < R:
        s = int(rng.integers(0, len(SEQ_LENS)))
        need.append((s, int(rng.integers(0, SEQ_LENS[s]))))
    need = need[:R]
    need.sort()              # rows of one sequence next to each other: without pairing they share one K/V stream
    return need


@pytest.mark.parametrize("R", [1, 2, 37, 601])
def test_last_layer_self_attention_on_unit_tables(R, monkeypatch):
    H, hd = 32, 48
    D = H * hd
    rng = np.random.default_rng(R)
    seq_lens = np.asarray(SEQ_LENS, np.int64)
    reg_rows = np.cumsum(seq_lens) - seq_lens                      # first row of every sequence in the stream
    M = int(seq_lens.sum())
    g = torch.Generator(device="cpu").manual_seed(100 + R)
    qkv = torch.randn(M, 3 * D, generator=g).to(DEV).bfloat16()   # K | V of every row, as the engine's qkv buffer
    k, v = qkv[:, D:2 * D], qkv[:, 2 * D:]
    need = _needed_rows(R, rng)
    assert len(need) == R
    need_seq = np.asarray([s for s, _ in need], np.int64); need_off = np.asarray([o for _, o in need], np.int64)
    q = torch.randn(R, D, generator=g).to(DEV).bfloat16()          # the R needed query rows
    kk = np.arange(R)
    units = np.stack([kk, np.ones_like(kk), reg_rows[need_seq], seq_lens[need_seq], need_off], 1)   # engine.py
    slopes = _slopes(H)

    got, slots = _run_units(monkeypatch, True, q, k, v, units, H, hd, slopes)
    if R > 2:                # consecutive units paired whatever their keys: split-key items
        tab = slots.table.cpu().numpy()
        both = (tab[:, 0, 1] > 0) & (tab[:, 1, 1] > 0)
        assert np.any(tab[both, 0, 2] != tab[both, 1, 2])
    want = _ref_units(q, k, v, units, H, hd, slopes)
    _assert_close(got, want, 2e-2)
    _assert_rejected(got, _ref_units(q, k, v, _shift_pos(units), H, hd, slopes), 2e-2, "ALiBi position + 1")

    # a row's output must not depend on how the units are paired into items ...
    alone, slots = _run_units(monkeypatch, False, q, k, v, units, H, hd, slopes)
    assert torch.equal(got, alone)
    if R > 2:                # the unpaired table still pairs rows of one sequence (one shared K/V stream)
        tab = slots.table.cpu().numpy()
        assert np.any(tab[:, 1, 1] > 0) and np.any(tab[:, 1, 1] == 0)
    # ... nor on its neighbours in the q tensor (the dead rows of its one-row tile) or its place in the table
    perm = rng.permutation(R)
    up = units[perm].copy(); up[:, 0] = kk
    for pair in (True, False):
        gp, _ = _run_units(monkeypatch, pair, q[torch.from_numpy(perm).to(DEV)].contiguous(), k, v, up, H, hd, slopes)
        assert torch.equal(gp, got[torch.from_numpy(perm).to(DEV)])


# ---------------------------------------------------------------------------------------------------------------------
# B. Last-layer cross tables (runs of <= 128 rows of one gene against its CREs) and stacked cross-attention at
#    production tile counts
CROSS_C = [0, 1, 37, 64, 65, 1024, 1500]
CROSS_ROWS = [63, 3, 129, 1, 300, 126, 64]                           # needed rows of each gene


@pytest.mark.parametrize("H,hd", [(32, 48), (8, 64)])
def test_last_layer_cross_attention_on_unit_tables(H, hd, monkeypatch):
    D = H * hd
    C = np.asarray(CROSS_C, np.int64); n_rows = np.asarray(CROSS_ROWS, np.int64)
    R = int(n_rows.sum())
    g = torch.Generator(device="cpu").manual_seed(hd)
    q = torch.randn(R, D, generator=g).to(DEV).bfloat16()
    kv = torch.randn(int(C.sum()), 2 * D, generator=g).to(DEV).bfloat16()
    k, v = kv[:, :D], kv[:, D:]
    gene_of = np.repeat(np.arange(len(C)), n_rows)
    cu_cre = np.concatenate([[0], np.cumsum(C)])
    units, start = [], 0
    for i in range(1, R + 1):                                        # engine.py: runs of one gene, <= 128 rows
        if i == R or gene_of[i] != gene_of[start] or i - start == 128:
            units.append([start, i - start, cu_cre[gene_of[start]], C[gene_of[start]], 0])
            start = i
    units = np.asarray(units, np.int64)
    assert units[:, 1].max() == 128 and (units[:, 3] == 0).any()

    got, slots = _run_units(monkeypatch, True, q, k, v, units, H, hd, None)
    want = _ref_units(q, k, v, units, H, hd, None)                   # (rows of the gene without CREs: zeros)
    _assert_close(got, want, 2e-2)
    assert bool((got[:CROSS_ROWS[0]] == 0).all())
    _assert_rejected(got, _ref_units(q, k, v, _drop_last_key(units), H, hd, None), 2e-2, "last key dropped")
    alone, _ = _run_units(monkeypatch, False, q, k, v, units, H, hd, None)
    assert torch.equal(got, alone)


@pytest.mark.parametrize("H,hd", [(32, 48), (8, 64)])
def test_stacked_cross_attention_at_production_tile_counts(H, hd):
    """Per gene, every tissue copy of its gene stream queries the gene's CREs (plan_gcross): T = 63 tissues x (G = 300
    chunks + registry) = 18 963 query rows, 149 tiles of one sequence, next to a small gene and a gene without CREs."""
    D = H * hd
    q_lens = np.asarray([63 * 301, 5 * 4, 63 * 3], np.int64)
    k_lens = np.asarray([1024, 37, 0], np.int64)
    assert (q_lens[0] + 127) // 128 == 149
    g = torch.Generator(device="cpu").manual_seed(7 + hd)
    q = torch.randn(int(q_lens.sum()), D, generator=g).to(DEV).bfloat16()
    kv = torch.randn(int(k_lens.sum()), 2 * D, generator=g).to(DEV).bfloat16()
    k, v = kv[:, :D], kv[:, D:]
    out = torch.full((q.shape[0], D), 7.0, dtype=torch.bfloat16, device=DEV)
    ops.attention_mc(q, k, v, ops.SlotMap(q_lens, DEV, k_lens=k_lens), H, hd, None, out=out)
    torch.cuda.synchronize()
    cu_q = np.concatenate([[0], np.cumsum(q_lens)]); cu_k = np.concatenate([[0], np.cumsum(k_lens)])
    units = np.stack([cu_q[:-1], q_lens, cu_k[:-1], k_lens, k_lens - q_lens], 1)
    want = _ref_units(q, k, v, units, H, hd, None)
    _assert_close(out, want, 2e-2)
    assert bool((out[cu_q[2]:] == 0).all())
    big = slice(0, int(q_lens[0]))                                   # the control on the 149-tile sequence alone
    _assert_rejected(out[big], _ref_units(q, k, v, _drop_last_key(units), H, hd, None)[big], 2e-2, "last key dropped")


# ---------------------------------------------------------------------------------------------------------------------
# C. The in-place FFN2 residual epilogue (x = x + f W2^T + b2 on the fp32 stream), with and without mirror / statistics
FORMS = {"mirror+stats": (True, True), "stats": (False, True), "mirror": (True, False), "neither": (False, False)}
PAD = 96                                                             # sentinel rows on each side of every output


def _ffn2(a, w, bias, x0, mirror, stats):
    """In place on a copy of x0 that sits between sentinel rows; -> (x, mirror or None, stats or None, [sentinel
    blocks of every output])."""
    M, N = x0.shape
    xbuf = torch.full((M + 2 * PAD, N), -777.0, device=DEV)
    x = xbuf[PAD:PAD + M]
    x.copy_(x0)
    mbuf = torch.full((M + 2 * PAD, N), -555.0, dtype=torch.bfloat16, device=DEV) if mirror else None
    sbuf = torch.full((M + 2 * PAD, ops.stats_parts(N), 2), 7.0, device=DEV) if stats else None
    xb = mbuf[PAD:PAD + M] if mirror else None
    st = sbuf[PAD:PAD + M] if stats else None
    ops.gemm(a, w, EPI_BIAS_RESID_F32, bias=bias, resid=x, out=x, out2=xb, stats_out=st)
    fences = [(b[:PAD], b[PAD + M:]) for b in (xbuf, mbuf, sbuf) if b is not None]
    return x, xb, st, fences


@pytest.mark.parametrize("K", [512, 1024])
@pytest.mark.parametrize("N", [512, 1536])
@pytest.mark.parametrize("M", [1023, 1024, 1025, 1100, 1279, 2049, 4097])
def test_ffn2_inplace_epilogue_ragged_rows(M, N, K):
    """M >= 1024 with K >= 512 runs on CTA pairs with the TMA-staged in-place epilogue (the last gene layer's final GEMM
    takes it with neither mirror nor statistics and a ragged row count); rows [0, 640) must be bit-identical to the
    single-CTA kernel's, in every form, and a partial last row block must not touch the rows around the output."""
    g = torch.Generator(device="cpu").manual_seed(M * 5 + N + K)
    a = (torch.randn(M, K, generator=g) * 0.5).to(DEV).bfloat16()
    w = (torch.randn(N, K, generator=g) / math.sqrt(K)).to(DEV).bfloat16()
    bias = torch.randn(N, generator=g).to(DEV)
    x0 = (torch.randn(M, N, generator=g) * 3).to(DEV)
    want = a.float() @ w.float().t() + bias + x0
    # the control: one 16-wide K step missing from the product
    short = a[:, :K - 16].float() @ w[:, :K - 16].float().t() + bias + x0
    for form, (mirror, stats) in FORMS.items():
        x, xb, st, fences = _ffn2(a, w, bias, x0, mirror, stats)
        x6, xb6, st6, _ = _ffn2(a[:640].contiguous(), w, bias, x0[:640], mirror, stats)     # single-CTA kernel
        torch.cuda.synchronize()
        assert torch.allclose(x, want, atol=2e-3, rtol=2e-3), f"{form}: " + _describe_mismatch(x, want, 2e-3)
        _assert_rejected(x, short, 2e-3, f"{form}: K - 16")
        assert torch.equal(x[:640], x6), form
        if mirror:
            assert torch.equal(xb, x.bfloat16()), form
            assert torch.equal(xb[:640], xb6), form
        if stats:
            tot = st.sum(1)
            assert torch.allclose(tot[:, 0], x.sum(1), atol=2e-2, rtol=1e-4), (form, tot[:4, 0], x.sum(1)[:4])
            assert torch.allclose(tot[:, 1], (x * x).sum(1), atol=2e-2, rtol=1e-4), form
            assert torch.equal(st[:640], st6), form
        for i, (lo, hi) in enumerate(fences):
            assert bool((lo == lo.flatten()[0]).all()) and bool((hi == lo.flatten()[0]).all()), (form, "output", i)


# ---------------------------------------------------------------------------------------------------------------------
# D. Label attention: every head group, the engine's strided q, and the unaligned fallback kernel
@pytest.mark.parametrize("hd", [48, 64])
def test_label_attention_all_head_groups(hd):
    H = 32
    D = H * hd
    C = [1, 700, 37, 900, 512, 64]                                   # the last gene's CREs are all one class
    n = sum(C)
    g = torch.Generator(device="cpu").manual_seed(hd)
    qkv = torch.randn(n, 3 * D, generator=g).to(DEV).bfloat16()
    kv9 = torch.randn(9, 2 * D, generator=g).to(DEV)
    labels = [torch.randint(0, 9, (c,), generator=g) for c in C]
    labels[-1][:] = 3
    counts = torch.stack([torch.bincount(l, minlength=9) for l in labels]).float()
    assert int((counts[-1] == 0).sum()) == 8
    logc = counts.log().to(DEV)
    row_seq = torch.repeat_interleave(torch.arange(len(C)), torch.tensor(C)).int().to(DEV)
    got = ops.label_attention(qkv[:, :D], kv9, logc, row_seq, H, hd)          # q with ldq = 3D, as the engine calls it
    # the same values through a q view 8 bytes off a 16-byte boundary: the warp-per-(row, head) kernel
    buf = torch.zeros(n, 3 * D + 8, dtype=torch.bfloat16, device=DEV)
    buf[:, 4:4 + 3 * D] = qkv
    qf = buf[:, 4:4 + D]
    assert qf.data_ptr() % 16 == 8 and qf.stride(0) % 8 == 0
    fb = ops.label_attention(qf, kv9, logc, row_seq, H, hd)
    # reference: full attention of every CRE over its gene's materialised label keys / values
    kfull = torch.cat([kv9[l.to(DEV)] for l in labels])
    cu = np.concatenate([[0], np.cumsum(C)])
    units = np.stack([cu[:-1], C, cu[:-1], C, np.zeros(len(C), np.int64)], 1)
    want = _ref_units(qkv[:, :D], kfull[:, :D], kfull[:, D:], units, H, hd, None)
    torch.cuda.synchronize()
    assert n >= 2000 and (n + 31) // 32 > 1
    _assert_close(got, want, 1e-2)
    _assert_close(fb, want, 1e-2)
    _assert_close(fb, got.float(), 1e-2)
    # controls: one CRE less per gene; heads past the first group of 8 reading the first group's keys and values
    _assert_rejected(got, _ref_units(qkv[:, :D], kfull[:, :D], kfull[:, D:], _drop_last_key(units), H, hd, None), 1e-2,
                     "last CRE dropped")
    kgrp = kfull.view(n, 2, H, hd).clone()
    kgrp[:, :, 8:] = kgrp[:, :, :8].repeat(1, 1, H // 8 - 1, 1)
    kgrp = kgrp.view(n, 2 * D)
    _assert_rejected(got, _ref_units(qkv[:, :D], kgrp[:, :D], kgrp[:, D:], units, H, hd, None), 1e-2, "head group 0 only")


# ---------------------------------------------------------------------------------------------------------------------
# E. Stage 1: more windows in one call than one launch's grid.y holds
def test_encode_windows_past_the_grid_y_limit():
    n_win = 65_600
    rng = np.random.default_rng(65)
    chroms = {"chr1": synth.make_chromosome(rng, 800_000), "chr2": synth.make_chromosome(rng, 500_000)}
    var = {c: synth.make_variants(rng, s) for c, s in chroms.items()}
    genome = Genome.from_arrays(chroms, DEV)
    sv = SampleVariants(var, DEV)
    tk = WindowTokenizer(DEV)
    names = np.where(rng.random(n_win) < 0.6, "chr1", "chr2")
    a = np.asarray([int(rng.integers(0, len(chroms[c]) - 400)) for c in names])
    span = rng.integers(150, 351, n_win)
    w0, w1 = zip(*[cre_window(s, s + l, 50) for s, l in zip(a, span)])
    rc = rng.integers(0, 2, n_win)
    out, out_len, err = tk.sequences(genome, list(names), list(w0), list(w1), rc, sv)
    out_len = out_len.cpu().numpy()
    assert int(err.item()) == 0
    check = np.unique(np.concatenate([rng.choice(n_win, 300, replace=False), np.arange(65_530, 65_540),
                                      np.arange(n_win - 10, n_win)]))
    rows = out[torch.from_numpy(check).to(DEV)].cpu().numpy()
    alts = {c: (np.array([len(x) for x in v["alt"]], np.int32), np.frombuffer(b"".join(v["alt"]), np.uint8))
            for c, v in var.items()}
    for r, i in zip(rows, check):
        c = names[i]
        v = var[c]
        lens, pool = alts[c]
        want = O.apply_variants(chroms[c], w0[i], w1[i], v["pos"], v["ref_len"], np.cumsum(lens) - lens, lens, v["gt"],
                                pool)
        if rc[i]:
            want = O.reverse_complement(want)
        assert r[:out_len[i]].tobytes() == want, f"window {i} {c}:{w0[i]}-{w1[i]} rc={rc[i]}"
