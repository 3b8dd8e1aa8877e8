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


def seq2gene_forward(table, slab, cre_pooled, gene_pooled, workspace, n_reg, n_tok_rows, D, want_cre_tok, attn=None):
    """Whole seq2gene forward of one slab in one call (vf_seq2gene_forward; with attn, an _abi.CreAttention table,
    vf_seq2gene_forward_attn, which also writes the gene -> CRE cross-attention maps).
    -> (pred fp32 [n_reg], emb fp32 [n_reg, D], gene token embeddings or None, CRE token embeddings or None)."""
    import ctypes as C
    dev = cre_pooled.device
    pred = torch.empty(n_reg, dtype=torch.float32, device=dev)
    emb = torch.empty((n_reg, D), dtype=torch.float32, device=dev)
    gtok = torch.empty((n_tok_rows, D), dtype=torch.float32, device=dev) if n_tok_rows else None
    ctok = torch.empty((n_reg, D), dtype=torch.float32, device=dev) if want_cre_tok else None
    args = (C.addressof(table), C.addressof(slab), ptr(cre_pooled), ptr(gene_pooled), ptr(workspace), workspace.numel(),
            ptr(pred), ptr(emb), ptr(gtok), ptr(ctok))
    with _timed("seq2gene_forward"):
        if attn is None:
            check(_lib.lib().vf_seq2gene_forward(*args, stream()))
        else:
            check(_lib.lib().vf_seq2gene_forward_attn(*args, C.addressof(attn), stream()))
    return pred, emb, gtok, ctok


def seq2gene_cre_rows(table, slab, workspace, rows, D):
    """Rows of the final CRE stream of the seq2gene_forward call that just ran on this stream with the same slab and
    workspace (vf_seq2gene_cre_rows).  rows int32 [n] device tensor -> fp32 [n, D] (un-centred)."""
    import ctypes as C
    out = torch.empty((rows.numel(), D), dtype=torch.float32, device=rows.device)
    if rows.numel():
        check(_lib.lib().vf_seq2gene_cre_rows(C.addressof(table), C.addressof(slab), ptr(workspace), workspace.numel(),
                                              ptr(rows), rows.numel(), ptr(out), stream()))
    return out


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


def cross_attention_probs(q, k, q_rows, group_q, group_k, heads, head_dim, out, out_off, layer):
    """Softmax probabilities of the cross-attention of selected query rows (vf_cross_attention_probs): q / k bf16 row
    views (k = the K half of a packed KV buffer); q_rows int32 (None: query index = row); group_q / group_k int32
    [n_groups, 2] = (first query index, count) / (first key row, count); out fp32 flat, out_off int64 [n_queries] = start
    of each query's [n_layers, heads, keys] block; writes the block of `layer`."""
    for t in (q, k):
        assert t.is_cuda and t.dtype == torch.bfloat16 and t.stride(1) == 1
    assert group_q.dtype == torch.int32 and group_k.dtype == torch.int32 and out_off.dtype == torch.int64
    assert out.dtype == torch.float32 and (q_rows is None or q_rows.dtype == torch.int32)
    n_groups = group_q.shape[0]
    with _timed("attention_probs"):
        check(_lib.lib().vf_cross_attention_probs(ptr(q), q.stride(0), ptr(q_rows), ptr(group_q), n_groups, ptr(k),
                                                  k.stride(0), ptr(group_k), heads, head_dim, ptr(out), ptr(out_off),
                                                  layer, stream()))
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


def encode_windows_edit(genome, win_base, w0, w1, var_lo, var_hi, flags, variants, e_pos, e_ref_len, e_alt_off,
                        e_alt_len, e_alt_pool, max_window, pitch, err=None):
    """encode_windows with one extra hom-alt record per row (vf_encode_windows_edit): row w encodes as encode_windows
    does on the table with {e_pos[w], e_ref_len[w], e_alt_pool[e_alt_off[w], + e_alt_len[w])} inserted after every
    record of pos <= e_pos[w].  e_* int32 [n], e_alt_pool uint8 device tensors.
    -> (out uint8 [n, pitch], out_len int32 [n], applied uint8 [n] (1: the row's extra record was applied), err)."""
    n = w0.numel()
    dev = genome.device
    for t in (w0, w1, var_lo, var_hi, e_pos, e_ref_len, e_alt_off, e_alt_len):
        assert t.dtype == torch.int32 and t.numel() == n and t.is_contiguous()
    assert win_base.dtype == torch.int64 and flags.dtype == torch.uint8 and e_alt_pool.dtype == torch.uint8
    out = torch.empty((n, pitch), dtype=torch.uint8, device=dev)
    out_len = torch.empty(n, dtype=torch.int32, device=dev)
    applied = torch.empty(n, dtype=torch.uint8, device=dev)
    if err is None:
        err = torch.zeros(1, dtype=torch.int32, device=dev)
    v = variants
    with _timed("stage1_encode_edit", nbytes=float(n) * max_window * 2):  # window bytes read + written (upper bound)
        check(_lib.lib().vf_encode_windows_edit(ptr(genome), ptr(win_base), ptr(w0), ptr(w1), ptr(var_lo), ptr(var_hi),
                                                ptr(flags), ptr(v["pos"]), ptr(v["ref_len"]), ptr(v["alt_off"]),
                                                ptr(v["alt_len"]), ptr(v["gt"]), ptr(v["alt_pool"]), ptr(e_pos),
                                                ptr(e_ref_len), ptr(e_alt_off), ptr(e_alt_len), ptr(e_alt_pool), n,
                                                int(max_window), ptr(out), int(pitch), ptr(out_len), ptr(applied),
                                                ptr(err), stream()))
    return out, out_len, applied, err


def _edit_records(n, dev, e_off, e_pos, e_ref_len, e_alt_off, e_alt_len, e_gt, e_alt_pool):
    """encode_windows_edits' host checks of the CSR extra records of n rows -> (device arrays with non-NULL stand-ins for
    empty ones, number of records)."""
    off = e_off.cpu().numpy()
    if e_off.dtype != torch.int32 or off.shape != (n + 1,) or off[0] != 0 or (np.diff(off) < 0).any():
        raise ValueError(f"e_off must be int32 [{n + 1}] offsets from 0, nondecreasing (got {e_off.dtype} "
                         f"{tuple(off.shape)})")
    m = int(off[-1])
    for t, dt in ((e_pos, torch.int32), (e_ref_len, torch.int32), (e_alt_off, torch.int32), (e_alt_len, torch.int32),
                  (e_gt, torch.uint8)):
        if t.dtype != dt or t.numel() != m or not t.is_contiguous():
            raise ValueError(f"extra-record arrays must be contiguous {dt} [{m}] (e_off[-1]), got {t.dtype} "
                             f"[{t.numel()}]")
    if e_alt_pool.dtype != torch.uint8:
        raise ValueError(f"e_alt_pool must be uint8, got {e_alt_pool.dtype}")
    # kernels need non-NULL arrays; the tensors stay referenced by the caller until the launch is enqueued
    return [e_off.to(dev)] + [t if t.numel() else torch.zeros(1, dtype=t.dtype, device=dev)
                              for t in (e_pos, e_ref_len, e_alt_off, e_alt_len, e_gt, e_alt_pool)], m


def encode_windows_edits(genome, win_base, w0, w1, var_lo, var_hi, flags, variants, e_off, e_pos, e_ref_len, e_alt_off,
                         e_alt_len, e_gt, e_alt_pool, max_window, pitch, err=None):
    """encode_windows with a list of extra records per row (vf_encode_windows_edits): row w owns the records
    [e_off[w], e_off[w + 1]) (CSR, sorted by pos within the row) and encodes as encode_windows does on the table with
    each record inserted after every record of pos <= its own.  e_off int32 [n + 1]; e_pos / e_ref_len / e_alt_off /
    e_alt_len int32 and e_gt uint8 (0 skip, 1 het, 2 hom) [e_off[-1]]; e_alt_pool uint8; device tensors.
    -> (out uint8 [n, pitch], out_len int32 [n], applied uint8 [e_off[-1]] (1: that record was applied), err)."""
    n = w0.numel()
    dev = genome.device
    for t in (w0, w1, var_lo, var_hi):
        assert t.dtype == torch.int32 and t.numel() == n and t.is_contiguous()
    assert win_base.dtype == torch.int64 and flags.dtype == torch.uint8 and e_alt_pool.dtype == torch.uint8
    e, m = _edit_records(n, dev, e_off, e_pos, e_ref_len, e_alt_off, e_alt_len, e_gt, e_alt_pool)
    out = torch.empty((n, pitch), dtype=torch.uint8, device=dev)
    out_len = torch.empty(n, dtype=torch.int32, device=dev)
    applied = torch.empty(max(m, 1), dtype=torch.uint8, device=dev)
    if err is None:
        err = torch.zeros(1, dtype=torch.int32, device=dev)
    v = variants
    with _timed("stage1_encode_edit", nbytes=float(n) * max_window * 2):  # window bytes read + written (upper bound)
        check(_lib.lib().vf_encode_windows_edits(ptr(genome), ptr(win_base), ptr(w0), ptr(w1), ptr(var_lo), ptr(var_hi),
                                                 ptr(flags), ptr(v["pos"]), ptr(v["ref_len"]), ptr(v["alt_off"]),
                                                 ptr(v["alt_len"]), ptr(v["gt"]), ptr(v["alt_pool"]),
                                                 *[ptr(t) for t in e], n, int(max_window), ptr(out), int(pitch),
                                                 ptr(out_len), ptr(applied), ptr(err), stream()))
    return out, out_len, applied[:m], err


def encode_windows_overrides(genome, win_base, w0, w1, var_lo, var_hi, flags, variants, o_off, o_idx, o_gt, max_window,
                             pitch, err=None):
    """encode_windows with a list of genotype overrides per row (vf_encode_windows_overrides): row w owns the overrides
    [o_off[w], o_off[w + 1]) (CSR), each a record index o_idx into the variant table (strictly increasing within the row,
    inside [var_lo[w], var_hi[w])) and its new gt o_gt (0 removed, 1 het, 2 hom-alt), and encodes as encode_windows does
    on the table with those gts replaced.  o_off int32 [n + 1]; o_idx int32 and o_gt uint8 [o_off[-1]]; device tensors.
    -> (out uint8 [n, pitch], out_len int32 [n], err); err 8 (length 0, that row only) for a malformed row."""
    n = w0.numel()
    dev = genome.device
    for t in (w0, w1, var_lo, var_hi):
        assert t.dtype == torch.int32 and t.numel() == n and t.is_contiguous()
    assert win_base.dtype == torch.int64 and flags.dtype == torch.uint8
    off = o_off.cpu().numpy()
    if o_off.dtype != torch.int32 or off.shape != (n + 1,) or off[0] != 0 or (np.diff(off) < 0).any():
        raise ValueError(f"o_off must be int32 [{n + 1}] offsets from 0, nondecreasing (got {o_off.dtype} "
                         f"{tuple(off.shape)})")
    m = int(off[-1])
    for t, dt in ((o_idx, torch.int32), (o_gt, torch.uint8)):
        if t.dtype != dt or t.numel() != m or not t.is_contiguous():
            raise ValueError(f"override arrays must be contiguous {dt} [{m}] (o_off[-1]), got {t.dtype} [{t.numel()}]")
    if m and int(o_gt.max()) > 2:
        raise ValueError(f"o_gt must be 0, 1 or 2 (got {int(o_gt.max())})")
    # kernels need non-NULL arrays; the tensors stay referenced by the caller until the launch is enqueued
    o = [o_off.to(dev)] + [t if t.numel() else torch.zeros(1, dtype=t.dtype, device=dev) for t in (o_idx, o_gt)]
    out = torch.empty((n, pitch), dtype=torch.uint8, device=dev)
    out_len = torch.empty(n, dtype=torch.int32, device=dev)
    if err is None:
        err = torch.zeros(1, dtype=torch.int32, device=dev)
    v = variants
    with _timed("stage1_encode_overrides", nbytes=float(n) * max_window * 2):   # window bytes read + written (upper bound)
        check(_lib.lib().vf_encode_windows_overrides(ptr(genome), ptr(win_base), ptr(w0), ptr(w1), ptr(var_lo),
                                                     ptr(var_hi), ptr(flags), ptr(v["pos"]), ptr(v["ref_len"]),
                                                     ptr(v["alt_off"]), ptr(v["alt_len"]), ptr(v["gt"]),
                                                     ptr(v["alt_pool"]), *[ptr(t) for t in o], n, int(max_window),
                                                     ptr(out), int(pitch), ptr(out_len), ptr(err), stream()))
    return out, out_len, err


def _genotype_rows(w0, w1, var_lo, var_hi, flags, variants):
    n = w0.numel()
    for t in (w0, w1, var_lo, var_hi):
        assert t.dtype == torch.int32 and t.numel() == n and t.is_contiguous()
    assert flags.dtype == torch.uint8 and flags.numel() == n
    v = variants
    return n, [ptr(w0), ptr(w1), ptr(var_lo), ptr(var_hi), ptr(flags), ptr(v["pos"]), ptr(v["ref_len"]), ptr(v["alt_off"]),
               ptr(v["alt_len"]), ptr(v["gt"]), ptr(v["alt_pool"]), n]


def window_genotype_keys(w0, w1, var_lo, var_hi, flags, variants, key_bits=128, err=None):
    """Genotype keys of (window, sample) rows (vf_window_genotype_keys): rows as encode_windows takes them, variants
    the dict of device arrays (stage1.SampleVariants.dev / CohortVariants.dev).  -> (keys int64 [n, 2] (the 128-bit key
    as two words, 0 for the reference window), count int32 [n] (applied records; -1 past the 2048-record cap, which
    sets err to 2), lens int32 [n] (the encoded length encode_windows checks against its pitch), err).  key_bits < 128 keeps only the low bits of the key (tests: forces collisions, which
    window_genotype_equal then separates)."""
    n, args = _genotype_rows(w0, w1, var_lo, var_hi, flags, variants)
    dev = w0.device
    keys = torch.empty((n, 2), dtype=torch.int64, device=dev)
    count = torch.empty(n, dtype=torch.int32, device=dev)
    lens = torch.empty(n, dtype=torch.int32, device=dev)
    if err is None:
        err = torch.zeros(1, dtype=torch.int32, device=dev)
    with _timed("stage1_keys"):
        check(_lib.lib().vf_window_genotype_keys(*args, ptr(keys), ptr(count), ptr(lens), ptr(err), stream()))
    if key_bits < 64:
        keys[:, 0] &= (1 << key_bits) - 1
        keys[:, 1] = 0
    elif key_bits < 128:
        keys[:, 1] &= (1 << (key_bits - 64)) - 1
    return keys, count, lens, err


def window_genotype_equal(w0, w1, var_lo, var_hi, flags, variants, rep):
    """1 where row r applies the same record list as row rep[r] (int32 [n] device), element by element
    (vf_window_genotype_equal).  -> int32 [n]."""
    n, args = _genotype_rows(w0, w1, var_lo, var_hi, flags, variants)
    assert rep.dtype == torch.int32 and rep.numel() == n
    equal = torch.empty(n, dtype=torch.int32, device=w0.device)
    with _timed("stage1_keys"):
        check(_lib.lib().vf_window_genotype_equal(*args, ptr(rep), ptr(equal), stream()))
    return equal


def window_genotype_keys_edits(w0, w1, var_lo, var_hi, flags, variants, e_off, e_pos, e_ref_len, e_alt_off, e_alt_len,
                               e_gt, e_alt_pool, key_bits=128, err=None):
    """window_genotype_keys for rows with a list of extra records each, in encode_windows_edits' CSR form
    (vf_window_genotype_keys_edits): a row's key, count and length are those of the list encode_windows_edits applies
    for it (background and extras merged); a row without extras gets window_genotype_keys' outputs.  -> (keys, count,
    lens, applied uint8 [e_off[-1]] (encode_windows_edits' flags for the same rows), err); err 4 (count -1, length 0)
    for a row whose extras are not sorted by pos."""
    n, args = _genotype_rows(w0, w1, var_lo, var_hi, flags, variants)
    dev = w0.device
    e, m = _edit_records(n, dev, e_off, e_pos, e_ref_len, e_alt_off, e_alt_len, e_gt, e_alt_pool)
    keys = torch.empty((n, 2), dtype=torch.int64, device=dev)
    count = torch.empty(n, dtype=torch.int32, device=dev)
    lens = torch.empty(n, dtype=torch.int32, device=dev)
    applied = torch.empty(max(m, 1), dtype=torch.uint8, device=dev)
    if err is None:
        err = torch.zeros(1, dtype=torch.int32, device=dev)
    with _timed("stage1_keys"):
        check(_lib.lib().vf_window_genotype_keys_edits(*args[:-1], *[ptr(t) for t in e], n, ptr(keys), ptr(count),
                                                       ptr(lens), ptr(applied), ptr(err), stream()))
    if key_bits < 64:
        keys[:, 0] &= (1 << key_bits) - 1
        keys[:, 1] = 0
    elif key_bits < 128:
        keys[:, 1] &= (1 << (key_bits - 64)) - 1
    return keys, count, lens, applied[:m], err


def window_genotype_equal_edits(w0, w1, var_lo, var_hi, flags, variants, e_off, e_pos, e_ref_len, e_alt_off, e_alt_len,
                                e_gt, e_alt_pool, rep):
    """1 where row r applies the same record list as row rep[r], element by element, extras merged as in
    window_genotype_keys_edits (vf_window_genotype_equal_edits).  -> int32 [n]."""
    n, args = _genotype_rows(w0, w1, var_lo, var_hi, flags, variants)
    assert rep.dtype == torch.int32 and rep.numel() == n
    e, _ = _edit_records(n, w0.device, e_off, e_pos, e_ref_len, e_alt_off, e_alt_len, e_gt, e_alt_pool)
    equal = torch.empty(n, dtype=torch.int32, device=w0.device)
    with _timed("stage1_keys"):
        check(_lib.lib().vf_window_genotype_equal_edits(*args[:-1], *[ptr(t) for t in e], n, ptr(rep), ptr(equal),
                                                        stream()))
    return equal


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


def splice_windows(src, src_len, row_src, row_off, allele_pool, allele_off, allele_len, flags, out_pitch, err=None):
    """Allele splices of encoded windows (vf_splice_windows): row r = src[row_src[r]] with the ONE base at forward-strand
    offset row_off[r] replaced by allele_pool[allele_off[r], + allele_len[r]) (reverse complement of the allele on
    reverse-complemented rows, flags bit 0); the row grows by allele_len[r] - 1 bytes.  src uint8 [n_src, pitch] and
    src_len int32 [n_src] as encode_windows returns them; row_src / row_off / allele_off / allele_len int32, flags uint8
    [n_rows], allele_pool uint8 device tensors; out_pitch: a multiple of 16 that holds the longest output row.
    -> (out uint8 [n_rows, out_pitch], out_len int32 [n_rows], err)."""
    n = row_src.numel()
    dev = src.device
    assert src.dtype == torch.uint8 and src.is_contiguous() and src_len.dtype == torch.int32 and out_pitch % 16 == 0
    for t in (row_src, row_off, allele_off, allele_len):
        assert t.dtype == torch.int32 and t.numel() == n
    assert allele_pool.dtype == torch.uint8 and flags.dtype == torch.uint8 and flags.numel() == n
    out = torch.empty((n, out_pitch), dtype=torch.uint8, device=dev)
    out_len = torch.empty(n, dtype=torch.int32, device=dev)
    if err is None:
        err = torch.zeros(1, dtype=torch.int32, device=dev)
    if n:
        with _timed("stage1_splice", nbytes=2.0 * n * out_pitch):      # row bytes read + written (upper bound)
            check(_lib.lib().vf_splice_windows(ptr(src), src.shape[1], ptr(src_len), ptr(row_src), ptr(row_off),
                                               ptr(allele_pool), ptr(allele_off), ptr(allele_len), ptr(flags), n,
                                               ptr(out), out_pitch, ptr(out_len), ptr(err), stream()))
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
