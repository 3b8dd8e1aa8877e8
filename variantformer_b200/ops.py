"""Tensor-level wrappers over the C ABI (one Python function per exported kernel).

torch is used only for device memory and streams; every computation happens in
libvf_b200.so.  `LAUNCHES` counts kernel launches issued through this module
(bench.py reports it as `gpu_launches`).
"""
import os

import numpy as np
import torch

from . import _lib
from ._lib import (EPI_BIAS_BF16, EPI_BIAS_F32, EPI_BIAS_GEGLU_BF16, EPI_BIAS_GELU_BF16, EPI_BIAS_RESID_F32, check,
                   ptr, stream)

LAUNCHES = 0
PROFILER = None          # set to an EventProfiler to time every launch with CUDA events on the launching stream


class EventProfiler:
    """Per-launch CUDA-event timing grouped by kernel kind (bench.py's roofline numerator/denominator)."""

    def __init__(self):
        self.items = []

    def begin(self):
        e = torch.cuda.Event(enable_timing=True)
        e.record()
        return e

    def end(self, e0, kind, flops=0.0, detail=None, nbytes=0.0):
        e1 = torch.cuda.Event(enable_timing=True)
        e1.record()
        self.items.append((kind, float(flops), e0, e1, detail, float(nbytes)))

    def summarize(self):
        """kind -> {ms, flops, bytes (algorithmic operand + result bytes of the launches), n}."""
        torch.cuda.synchronize()
        out = {}
        for kind, flops, e0, e1, _, nbytes in self.items:
            d = out.setdefault(kind, {"ms": 0.0, "flops": 0.0, "bytes": 0.0, "n": 0})
            d["ms"] += e0.elapsed_time(e1); d["flops"] += flops; d["bytes"] += nbytes; d["n"] += 1
        return out

    def summarize_detail(self):
        """Same, keyed by the launch's shape string (GEMM: "N x K epilogue flags"; attention: heads x head_dim, bias)."""
        torch.cuda.synchronize()
        out = {}
        for kind, flops, e0, e1, detail, nbytes in self.items:
            if detail is None:
                continue
            d = out.setdefault(f"{kind} {detail}", {"ms": 0.0, "flops": 0.0, "bytes": 0.0, "n": 0})
            d["ms"] += e0.elapsed_time(e1); d["flops"] += flops; d["bytes"] += nbytes; d["n"] += 1
        return out


class _timed:
    __slots__ = ("kind", "flops", "e0", "detail", "nbytes")

    def __init__(self, kind, flops=0.0, detail=None, nbytes=0.0):
        self.kind, self.flops, self.e0, self.detail, self.nbytes = kind, flops, None, detail, nbytes

    def __enter__(self):
        if PROFILER is not None:
            self.e0 = PROFILER.begin()

    def __exit__(self, *a):
        global LAUNCHES
        LAUNCHES += 1
        if self.e0 is not None and PROFILER is not None:
            PROFILER.end(self.e0, self.kind, self.flops, self.detail() if callable(self.detail) else self.detail,
                         self.nbytes)
        return False


_EPI_NAME = {EPI_BIAS_BF16: "bias", EPI_BIAS_GEGLU_BF16: "geglu", EPI_BIAS_GELU_BF16: "gelu", EPI_BIAS_RESID_F32: "resid",
             EPI_BIAS_F32: "f32"}
_OUT_DTYPE = {EPI_BIAS_BF16: torch.bfloat16, EPI_BIAS_GEGLU_BF16: torch.bfloat16, EPI_BIAS_GELU_BF16: torch.bfloat16,
              EPI_BIAS_RESID_F32: torch.float32, EPI_BIAS_F32: torch.float32}


def _chk_bf16(t):
    assert t.is_cuda and t.dtype == torch.bfloat16 and t.stride(-1) == 1, "expected a row-major CUDA bf16 tensor"


def gemm(a, w, epilogue, bias=None, resid=None, out=None, out2=None, ln=None, stats_out=None, mirror_only=False):
    """out = epilogue(a[M,K] @ w[N,K]^T).  a, w bf16; bias fp32 [N]; resid fp32 [M,N].
    ln = (stats fp32 [M,P,2], colsum fp32 [N], width, eps): LayerNorm of the rows `a` mirrors, folded into the epilogue
    (w, bias must be the gamma/beta-folded ones); stats_out fp32 [M, stats_parts(N), 2]: partial row (sum, sum of
    squares) of an fp32 output.  resid may be bf16 (residual epilogue); mirror_only: an fp32 epilogue writes only its
    bf16 mirror out2 (and the statistics), no fp32 output."""
    _chk_bf16(a); _chk_bf16(w)
    M, K = a.shape
    N = w.shape[0]
    assert w.shape[1] == K
    n_out = N // 2 if epilogue == EPI_BIAS_GEGLU_BF16 else N
    if mirror_only:
        assert out is None and out2 is not None and _OUT_DTYPE[epilogue] == torch.float32
    else:
        if out is None:
            out = torch.empty((M, n_out), dtype=_OUT_DTYPE[epilogue], device=a.device)
        assert out.dtype == _OUT_DTYPE[epilogue] and out.shape == (M, n_out) and out.stride(1) == 1
    if resid is not None:
        assert resid.dtype in (torch.float32, torch.bfloat16) and resid.shape == (M, N) and resid.stride(1) == 1
    if bias is not None:
        assert bias.dtype == torch.float32 and bias.numel() == N and bias.is_contiguous()
    if out2 is not None:
        assert out2.dtype == torch.bfloat16 and out2.shape == (M, N) and out2.stride(1) == 1
    ln_stats = ln_colsum = None
    ln_dim, ln_eps, ln_parts = 0, 0.0, 0
    if ln is not None:
        ln_stats, ln_colsum, ln_dim, ln_eps = ln
        assert ln_stats.dtype == torch.float32 and ln_stats.dim() == 3 and ln_stats.shape[0] == M and \
            ln_stats.shape[2] == 2 and ln_stats.is_contiguous()
        ln_parts = ln_stats.shape[1]
        assert ln_colsum.dtype == torch.float32 and ln_colsum.numel() == N and ln_colsum.is_contiguous()
    if stats_out is not None:
        assert stats_out.dtype == torch.float32 and stats_out.shape == (M, stats_parts(N), 2) and stats_out.is_contiguous()
    with _timed("gemm", 2.0 * M * N * K, lambda: (
            f"N={N} K={K} {_EPI_NAME[epilogue]}" + (" ln" if ln is not None else "") +
            ("" if resid is None else " resid16" if resid.dtype == torch.bfloat16 else " resid32") +
            (" out32" if out is not None and out.dtype == torch.float32 else "") + (" mirror" if out2 is not None else "") +
            (" stats" if stats_out is not None else "") + (" M>=64k" if M >= 65536 else " M<64k")),
            nbytes=2.0 * M * K + 2.0 * N * K + 4.0 * N + (0 if resid is None else M * N * resid.element_size()) +
            (0 if out is None else M * n_out * out.element_size()) + (0 if out2 is None else 2.0 * M * N) +
            (0 if ln is None else 8.0 * M * ln_parts) + (0 if stats_out is None else 8.0 * M * stats_parts(N))):
        check(_lib.lib().vf_gemm_bf16_ln(ptr(a), a.stride(0), ptr(w), w.stride(0), M, N, K, epilogue, ptr(bias),
                                         ptr(resid), int(resid is not None and resid.dtype == torch.bfloat16),
                                         resid.stride(0) if resid is not None else 0, ptr(out),
                                         out.stride(0) if out is not None else 0, ptr(out2),
                                         out2.stride(0) if out2 is not None else 0,
                                         ptr(ln_stats), ln_parts, ptr(ln_colsum), int(ln_dim), float(ln_eps),
                                         ptr(stats_out), stream()))
    return out2 if mirror_only else out


def stats_parts(n):
    """Partials per row that an fp32 GEMM epilogue with N = n output columns writes into `stats_out`."""
    return 2 * ((n + 255) // 256)


def rowstats(x, stats=None, out_bf16=None):
    """Per-row (sum, sum of squares) of fp32 x [M,d] -> stats [M,1,2]; optional bf16 mirror of x."""
    assert x.dtype == torch.float32 and x.stride(1) == 1
    M, d = x.shape
    if stats is None:
        stats = torch.empty((M, 1, 2), dtype=torch.float32, device=x.device)
    assert stats.shape == (M, 1, 2) and stats.is_contiguous()
    if out_bf16 is not None:
        assert out_bf16.dtype == torch.bfloat16 and out_bf16.shape == (M, d) and out_bf16.stride(1) == 1
    with _timed("misc"):
        check(_lib.lib().vf_rowstats(ptr(x), x.stride(0), M, d, ptr(stats), ptr(out_bf16),
                                     out_bf16.stride(0) if out_bf16 is not None else 0, stream()))
    return stats


def launch_count():
    """Kernels launched by libvf_b200.so since it was loaded (counted inside the library)."""
    return int(_lib.load().vf_launch_count())


def seq2reg_forward(table, tokens_i32, pad_mask_u8, cu, n_tok, slots, workspace, d):
    """Whole window encoder in one call (vf_seq2reg_forward): -> bf16 [n_win, d]."""
    import ctypes as C
    n_win, L = tokens_i32.shape
    out = torch.empty((n_win, d), dtype=torch.bfloat16, device=tokens_i32.device)
    with _timed("seq2reg_forward"):
        check(_lib.lib().vf_seq2reg_forward(C.addressof(table), ptr(tokens_i32), ptr(pad_mask_u8), ptr(cu), n_win, L,
                                            int(n_tok), ptr(slots.table), slots.n_items, ptr(workspace),
                                            workspace.numel(), ptr(out), stream()))
    return out


def seq2gene_forward(table, slab, cre_pooled, gene_pooled, workspace, n_reg, n_tok_rows, D, want_cre_tok):
    """Whole seq2gene forward of one slab in one call (vf_seq2gene_forward).
    -> (pred fp32 [n_reg], emb fp32 [n_reg, D], gene token embeddings or None, CRE token embeddings or None)."""
    import ctypes as C
    dev = cre_pooled.device
    pred = torch.empty(n_reg, dtype=torch.float32, device=dev)
    emb = torch.empty((n_reg, D), dtype=torch.float32, device=dev)
    gtok = torch.empty((n_tok_rows, D), dtype=torch.float32, device=dev) if n_tok_rows else None
    ctok = torch.empty((n_reg, D), dtype=torch.float32, device=dev) if want_cre_tok else None
    with _timed("seq2gene_forward"):
        check(_lib.lib().vf_seq2gene_forward(C.addressof(table), C.addressof(slab), ptr(cre_pooled), ptr(gene_pooled),
                                             ptr(workspace), workspace.numel(), ptr(pred), ptr(emb), ptr(gtok), ptr(ctok),
                                             stream()))
    return pred, emb, gtok, ctok


def cu_seqlens(lens, device):
    cu = np.zeros(len(lens) + 1, np.int32)
    np.cumsum(np.asarray(lens, np.int64), out=cu[1:])
    return torch.from_numpy(cu).to(device, non_blocking=True)


# Left-over query tiles (sequences of <= 128 rows, the odd last tile of longer ones) are paired into one work item even
# though they read DIFFERENT key ranges ("split" items: each slot streams its own K/V through the shared rings).  Round 1
# had to switch this off: an MMA issuer waits by parity on a ring stage whose previous use belonged to the other slot, and
# one launch in 12 000 went wrong.  The kernel now orders those waits behind the producer's issue counters
# (vf_attention_mc.cu: lds_acquire), so pairing is on again; VF_PAIR_TILES=0 restores the one-tile-per-item tables for
# A/B runs.  profiles/r02_stress_attention.log holds the determinism stress this rests on.
PAIR_UNRELATED_TILES = os.environ.get("VF_PAIR_TILES", "1") != "0"


class SlotMap:
    """Work items of vf_attention_mc_varlen for a batch of variable-length sequences (host-built, device-resident).

    Every sequence is cut into 128-row query tiles; consecutive tiles of a sequence are paired into one item (they
    share the sequence's K/V stream); the odd tiles left over (all of them when sequences have <= 128 rows) get an
    item of their own (see PAIR_UNRELATED_TILES).  Record layout: include/vf_b200.h."""

    def __init__(self, q_lens, device, k_lens=None):
        q_lens = np.asarray(q_lens, np.int64)
        k_lens = q_lens if k_lens is None else np.asarray(k_lens, np.int64)
        self.qk_pairs = float((q_lens * k_lens).sum())
        n = len(q_lens)
        cu_q = np.concatenate([[0], np.cumsum(q_lens)]); cu_k = np.concatenate([[0], np.cumsum(k_lens)])
        nt = (q_lens + 127) // 128
        seq = np.repeat(np.arange(n), nt)
        t = np.arange(int(nt.sum())) - np.repeat(np.cumsum(nt) - nt, nt)
        rec = np.zeros((len(seq), 8), np.int32)
        rec[:, 0] = cu_q[seq] + 128 * t
        rec[:, 1] = np.minimum(128, q_lens[seq] - 128 * t)
        rec[:, 2] = cu_k[seq]
        rec[:, 3] = k_lens[seq]
        rec[:, 4] = 128 * t + k_lens[seq] - q_lens[seq]
        # a sequence without keys gets no work item; attention_mc() zero-fills its output rows (what flash_attn
        # returns for an empty key range) so that a reused buffer never leaks a previous slab's values
        self.keyless = [(int(cu_q[i]), int(cu_q[i + 1])) for i in np.nonzero((k_lens == 0) & (q_lens > 0))[0]]
        rec = rec[rec[:, 3] > 0]
        odd = (t == nt[seq] - 1) & (nt[seq] % 2 == 1)
        odd = odd[(k_lens[seq] > 0)]
        pairs, singles = rec[~odd], rec[odd]
        if PAIR_UNRELATED_TILES:
            if len(singles) % 2:
                singles = np.concatenate([singles, np.zeros((1, 8), np.int32)])
            singles = singles.reshape(-1, 2, 8)
        else:                                                             # each left-over tile alone, slot 1 empty
            singles = np.stack([singles, np.zeros_like(singles)], axis=1)
        items = np.concatenate([pairs.reshape(-1, 2, 8), singles])
        self.n_items = int(items.shape[0])
        self.table = torch.from_numpy(np.ascontiguousarray(items)).to(device, non_blocking=True)

    @classmethod
    def from_units(cls, units, device):
        """units: int array [n, 5] of explicit slot records {q row, valid rows, first key row, keys, ALiBi position of
        row 0}; consecutive units are paired into items (units with the same key range share their K/V stream)."""
        self = cls.__new__(cls)
        units = np.asarray(units, np.int64).reshape(-1, 5)
        self.keyless = [(int(u[0]), int(u[0] + u[1])) for u in units if u[3] == 0 and u[1] > 0]
        units = units[units[:, 3] > 0]
        self.qk_pairs = float((units[:, 1] * units[:, 3]).sum())
        n = len(units)
        if PAIR_UNRELATED_TILES:
            first = np.arange(0, n, 2)
            paired = first + 1 < n
        else:
            # greedy left to right: unit i opens an item; unit i+1 joins it only if it reads the same key range
            same_next = np.zeros(n, bool)
            if n > 1:
                same_next[:-1] = (units[:-1, 2] == units[1:, 2]) & (units[:-1, 3] == units[1:, 3])
            first, paired, i = [], [], 0
            while i < n:
                first.append(i); paired.append(bool(same_next[i])); i += 2 if same_next[i] else 1
            first = np.asarray(first, np.int64); paired = np.asarray(paired, bool)
        rec = np.zeros((len(first), 2, 8), np.int32)
        rec[:, 0, :5] = units[first]
        rec[paired, 1, :5] = units[first[paired] + 1]
        self.n_items = int(rec.shape[0])
        self.table = torch.from_numpy(np.ascontiguousarray(rec)).to(device, non_blocking=True)
        return self


def attention_mc(q, k, v, slots: SlotMap, heads, head_dim, slopes=None, out=None):
    """Varlen attention on the two-CTAs-per-SM tcgen05 kernel (vf_attention_mc_varlen)."""
    for t in (q, k, v):
        assert t.is_cuda and t.dtype == torch.bfloat16 and t.stride(1) == 1
    if out is None:
        out = torch.empty((q.shape[0], heads * head_dim), dtype=torch.bfloat16, device=q.device)
    for r0, r1 in slots.keyless:
        out[r0:r1].zero_()
    with _timed("attention", 4.0 * slots.qk_pairs * heads * head_dim,
                lambda: f"h={heads} hd={head_dim}{' alibi' if slopes is not None else ''} rows={q.shape[0]} keys={k.shape[0]}",
                nbytes=2.0 * heads * head_dim * (2 * q.shape[0] + 2 * k.shape[0])):
        check(_lib.lib().vf_attention_mc_varlen(ptr(q), q.stride(0), ptr(k), k.stride(0), ptr(v), v.stride(0),
                                                ptr(out), out.stride(0), q.shape[0], k.shape[0], ptr(slots.table),
                                                slots.n_items, heads, head_dim, ptr(slopes), stream()))
    return out


def label_attention(q, kv9, logc, row_seq, heads, head_dim, out=None):
    assert q.dtype == torch.bfloat16 and kv9.dtype == torch.float32 and logc.dtype == torch.float32
    assert row_seq.dtype == torch.int32 and kv9.is_contiguous() and logc.is_contiguous()
    if out is None:
        out = torch.empty((q.shape[0], heads * head_dim), dtype=torch.bfloat16, device=q.device)
    with _timed("label_attention"):
        check(_lib.lib().vf_label_attention(ptr(q), q.stride(0), ptr(kv9), ptr(logc), ptr(row_seq), q.shape[0], heads,
                                            head_dim, ptr(out), out.stride(0), stream()))
    return out


def layernorm(x, gamma, beta, eps=1e-5, gelu=False, out=None):
    assert x.dtype == torch.float32 and x.stride(1) == 1
    M, d = x.shape
    if out is None:
        out = torch.empty((M, d), dtype=torch.bfloat16, device=x.device)
    with _timed("layernorm"):
        check(_lib.lib().vf_layernorm(ptr(x), x.stride(0), ptr(gamma), ptr(beta), M, d, eps, ptr(out), out.stride(0),
                                      int(gelu), stream()))
    return out


def window_lengths(pad_mask_u8):
    n, L = pad_mask_u8.shape
    lens = torch.empty(n, dtype=torch.int32, device=pad_mask_u8.device)
    with _timed("misc"):
        check(_lib.lib().vf_window_lengths(ptr(pad_mask_u8), n, L, ptr(lens), stream()))
    return lens


def compact_tokens(tokens_i32, pad_mask_u8, cu, n_tok):
    n, L = tokens_i32.shape
    ids = torch.empty(n_tok, dtype=torch.int32, device=tokens_i32.device)
    pos = torch.empty(n_tok, dtype=torch.int32, device=tokens_i32.device)
    with _timed("misc"):
        check(_lib.lib().vf_compact_tokens(ptr(tokens_i32), ptr(pad_mask_u8), ptr(cu), n, L, ptr(ids), ptr(pos), stream()))
    return ids, pos


def embed_tokens(ids, pos, emb, pe):
    n, d = ids.numel(), emb.shape[1]
    out = torch.empty((n, d), dtype=torch.float32, device=ids.device)
    with _timed("misc"):
        check(_lib.lib().vf_embed_tokens(ptr(ids), ptr(pos), ptr(emb), ptr(pe), n, d, ptr(out), stream()))
    return out


def center_rows(x, pivot=None, stats=None, out_bf16=None):
    """x <- x - mean_r in place (fp32 [M,d]); -> (pivot fp32 [M], stats fp32 [M,1,2] of the shifted rows); optional
    bf16 mirror.  The row-centred form of a residual stream (include/vf_b200.h: vf_center_rows)."""
    assert x.dtype == torch.float32 and x.stride(1) == 1
    M, d = x.shape
    if pivot is None:
        pivot = torch.empty(M, dtype=torch.float32, device=x.device)
    if stats is None:
        stats = torch.empty((M, 1, 2), dtype=torch.float32, device=x.device)
    assert pivot.shape == (M,) and pivot.is_contiguous() and stats.shape == (M, 1, 2) and stats.is_contiguous()
    if out_bf16 is not None:
        assert out_bf16.dtype == torch.bfloat16 and out_bf16.shape == (M, d) and out_bf16.stride(1) == 1
    with _timed("misc"):
        check(_lib.lib().vf_center_rows(ptr(x), x.stride(0), M, d, ptr(pivot), ptr(stats), ptr(out_bf16),
                                        out_bf16.stride(0) if out_bf16 is not None else 0, stream()))
    return pivot, stats


def uncenter_rows(x, pivot, idx=None, want_f32=True, want_bf16=False, out_bf16=None):
    """out[r] = x[r] + pivot[idx[r] if idx is given else r]  ->  (fp32 or None, bf16 or None)."""
    assert x.dtype == torch.float32 and x.stride(1) == 1 and pivot.dtype == torch.float32 and pivot.is_contiguous()
    M, d = x.shape
    assert idx is None or (idx.dtype == torch.int32 and idx.numel() == M)
    of = torch.empty((M, d), dtype=torch.float32, device=x.device) if want_f32 else None
    ob = out_bf16 if out_bf16 is not None else \
        (torch.empty((M, d), dtype=torch.bfloat16, device=x.device) if want_bf16 else None)
    if ob is not None:
        assert ob.dtype == torch.bfloat16 and ob.shape == (M, d) and ob.is_contiguous()
    with _timed("misc"):
        check(_lib.lib().vf_uncenter_rows(ptr(x), x.stride(0), ptr(pivot), ptr(idx), M, d, ptr(of), ptr(ob), d, stream()))
    return of, ob


def masked_meanpool(x, cu, n_win, want_f32=False, pivot=None):
    d = x.shape[1]
    ob = torch.empty((n_win, d), dtype=torch.bfloat16, device=x.device)
    of = torch.empty((n_win, d), dtype=torch.float32, device=x.device) if want_f32 else None
    with _timed("misc"):
        check(_lib.lib().vf_masked_meanpool(ptr(x), x.stride(0), ptr(cu), n_win, d, ptr(pivot), ptr(ob), ptr(of), d,
                                            stream()))
    return (ob, of) if want_f32 else ob


def gather_rows(table_a, table_b, idx, want_f32=True, want_bf16=False):
    n, d = idx.numel(), table_a.shape[1]
    of = torch.empty((n, d), dtype=torch.float32, device=idx.device) if want_f32 else None
    ob = torch.empty((n, d), dtype=torch.bfloat16, device=idx.device) if want_bf16 else None
    with _timed("misc"):
        check(_lib.lib().vf_gather_rows(ptr(table_a), table_a.stride(0), ptr(table_b),
                                        table_b.stride(0) if table_b is not None else 0, ptr(idx), n, d, ptr(of), ptr(ob),
                                        d, stream()))
    return of, ob


def head_out(h_bf16, w, b, softplus=True):
    n, d = h_bf16.shape
    out = torch.empty(n, dtype=torch.float32, device=h_bf16.device)
    with _timed("misc"):
        check(_lib.lib().vf_head_out(ptr(h_bf16), h_bf16.stride(0), ptr(w), ptr(b), n, d, int(softplus), ptr(out), stream()))
    return out


def cast_bf16(x):
    assert x.dtype == torch.float32 and x.is_contiguous()
    y = torch.empty(x.shape, dtype=torch.bfloat16, device=x.device)
    with _timed("misc"):
        check(_lib.lib().vf_cast_f32_to_bf16(ptr(x), ptr(y), x.numel(), stream()))
    return y


def forest_predict(x, row_forest, forest, out=None):
    """P(class 1) of every row of x fp32 [n, d] under its gradient-boosted forest (vf_forest_predict).
    forest: dict of device tensors tree_off, base, tree_root, feat, thr, left, right, value (+ op_lt int)."""
    assert x.dtype == torch.float32 and x.stride(1) == 1 and row_forest.dtype == torch.int32
    n, d = x.shape
    if out is None:
        out = torch.empty(n, dtype=torch.float32, device=x.device)
    f = forest
    with _timed("forest"):
        check(_lib.lib().vf_forest_predict(ptr(x), x.stride(0), n, d, ptr(row_forest), ptr(f["tree_off"]), ptr(f["base"]),
                                           ptr(f["tree_root"]), ptr(f["feat"]), ptr(f["thr"]), ptr(f["left"]),
                                           ptr(f["right"]), ptr(f["value"]), int(f.get("op_lt", 0)), ptr(out), stream()))
    return out


# ---- stage 1 -------------------------------------------------------------------------------
def encode_windows(genome, win_base, w0, w1, var_lo, var_hi, flags, variants, max_window, pitch):
    """variants: dict of device tensors pos/ref_len/alt_off/alt_len (int32), gt (uint8), alt_pool (uint8)."""
    n = w0.numel()
    out = torch.empty((n, pitch), dtype=torch.uint8, device=genome.device)
    out_len = torch.empty(n, dtype=torch.int32, device=genome.device)
    err = torch.zeros(1, dtype=torch.int32, device=genome.device)
    v = variants
    with _timed("stage1_encode", nbytes=float(n) * max_window * 2):       # window bytes read + written (upper bound)
        check(_lib.lib().vf_encode_windows(ptr(genome), ptr(win_base), ptr(w0), ptr(w1), ptr(var_lo), ptr(var_hi),
                                           ptr(flags), ptr(v["pos"]), ptr(v["ref_len"]), ptr(v["alt_off"]),
                                           ptr(v["alt_len"]), ptr(v["gt"]), ptr(v["alt_pool"]), n, int(max_window),
                                           ptr(out), int(pitch), ptr(out_len), ptr(err), stream()))
    return out, out_len, err


def mutate_windows(src, src_len, row_src, row_off, row_base, flags, err=None):
    """Single-base substitutions of encoded windows (vf_mutate_windows): row r = src[row_src[r]] with the base at
    forward-strand offset row_off[r] replaced by row_base[r] (complemented on reverse-complemented rows, flags bit 0).
    src uint8 [n_src, pitch] and src_len int32 [n_src] as encode_windows returns them; row_src / row_off int32,
    row_base / flags uint8 [n_rows] device tensors.  -> (out uint8 [n_rows, pitch], out_len int32 [n_rows], err)."""
    n, pitch = row_src.numel(), src.shape[1]
    dev = src.device
    assert src.dtype == torch.uint8 and src.is_contiguous() and src_len.dtype == torch.int32
    assert row_src.dtype == torch.int32 and row_off.dtype == torch.int32 and row_off.numel() == n
    assert row_base.dtype == torch.uint8 and flags.dtype == torch.uint8 and row_base.numel() == n and flags.numel() == n
    out = torch.empty((n, pitch), dtype=torch.uint8, device=dev)
    out_len = torch.empty(n, dtype=torch.int32, device=dev)
    if err is None:
        err = torch.zeros(1, dtype=torch.int32, device=dev)
    for r0 in range(0, n, 65535):                                       # grid.y limit of one launch
        r1 = min(n, r0 + 65535)
        with _timed("stage1_mutate", nbytes=2.0 * (r1 - r0) * pitch):  # row bytes read + written (upper bound)
            check(_lib.lib().vf_mutate_windows(ptr(src), pitch, ptr(src_len), ptr(row_src[r0:r1]), ptr(row_off[r0:r1]),
                                               ptr(row_base[r0:r1]), ptr(flags[r0:r1]), r1 - r0, ptr(out[r0:r1]), pitch,
                                               ptr(out_len[r0:r1]), ptr(err), stream()))
    return out, out_len, err


def bpe_tokenize(seq, lens, max_len, merges, out_pitch, out_cap, want_starts=False, typical_len=None):
    """seq uint8 [n, pitch]; lens int32 [n]; merges = (a, b, new[, batch]) uint16 device tensors (viewed as int16
    storage); `batch` = per-rank batch ids (stage1.merge_batches) or absent."""
    n, pitch = seq.shape
    dev = seq.device
    out = torch.empty((n, out_pitch), dtype=torch.int32, device=dev)
    cnt = torch.empty(n, dtype=torch.int32, device=dev)
    scratch = None                      # long windows run on the cluster kernel, which keeps symbols in shared memory
    t = max_len if typical_len is None else typical_len
    # short windows are latency bound: small CTAs, many windows in flight per SM (vf_encode.cu: bpe_tokenize)
    threads = 64 if t <= 1024 else (256 if t <= 2048 else (512 if t <= 4096 else 1024))
    starts = torch.empty((n, max_len), dtype=torch.int32, device=dev) if want_starts else None
    a, b, c = merges[:3]
    batch = merges[3] if len(merges) > 3 else None         # rank batches (stage1.merge_batches), optional
    # algorithmic bytes: every sequence byte read once (typical length) + int32 tokens of the kept prefix written
    with _timed("stage1_bpe_cluster" if max_len > 8192 else "stage1_bpe", nbytes=float(n) * (t + 4.0 * out_cap)):
        check(_lib.lib().vf_bpe_tokenize(ptr(seq), pitch, ptr(lens), n, int(max_len), ptr(a), ptr(b), ptr(c), ptr(batch),
                                         a.numel(),
                                         ptr(scratch), int(max_len) if scratch is not None else 0, ptr(out), out_pitch,
                                         out_cap, ptr(cnt), ptr(starts), int(max_len) if want_starts else 0, threads,
                                         stream()))
    return (out, cnt, starts) if want_starts else (out, cnt)
