"""In-silico saturation mutagenesis (ISM): every single-base substitution of a region, scored in batched passes.

The result for position p (1-based), alternative base a and zygosity z is BY DEFINITION what the per-variant path
(datasets/vepdataset.VEPBatchBuilder + variant_prediction) gives for Variant(chrom, p, ref, a): z = 1 writes
get_iupac_code(ref, a), z = 2 writes a, into every window window_hits() says the variant reaches; a background sample
contributes SNPs only and the query base wins at its position.  What is not recomputed (DESIGN section 11):
  * the reference item is encoded and tokenized once per gene;
  * a mutant re-encodes only its hit CRE windows (vf_mutate_windows + the fixed-row BPE) and its gene window (full BPE
    of the mutated 301 kb word: an incremental re-tokenization is not proven exact);
  * a window's pooled seq2reg vector depends on its tokens alone, so every DISTINCT token row (CRE window or 200-token
    gene chunk) is encoded once over the whole region, and items point into the pooled rows (Engine.prepare_shared).
Positions are skipped (not reported) when the reference or background base is not A/C/G/T, or when the position
touches no window ("No overlap").
"""
from dataclasses import dataclass, field
from typing import Dict, List, Optional

import numpy as np
import torch

from . import ops
from .datasets.vepdataset import cre_windows, get_iupac_code, window_hits
from .engine import AttnPlan
from .stage1 import gene_window

ACGT = "ACGT"
# CRE rows per slab of run_pooled.  The CRE rows of a slab size the per-layer K/V buffers of the gene stack's
# cross-attention (25 layers x rows x 2D bf16 = 150 KB per row at D = 1536), and a slab must hold enough mutants to fill
# the GPU: 16 k rows (16 mutants at C = 1024) keeps those buffers at 2.4 GB and the stacked cross-attention
# (all tissues of a mutant x its CREs) at the row counts of the benchmark slab (8 genes x 1024 CREs).
ROWS_BUDGET = 16384
# distinct windows per seq2reg call (bounds the call's workspace; results do not depend on the split)
POOL_ROWS = 8192
# gene windows mutated and tokenized per stage-1 group (each holds the 301 kB row and its 40 000 int32 tokens)
GENE_GROUP = 256


@dataclass
class Mutant:
    pos: int                    # 1-based
    ref: str                    # reference base (upper case)
    alt: str
    zyg: int                    # 1 het, 2 hom
    base: str                   # the byte written into the windows: alt (hom) or get_iupac_code(ref, alt) (het)
    hits: List[int]             # CRE rows (batch order) that get the base
    gene_hit: bool


@dataclass
class IsmPlan:
    mutants: List[Mutant]
    skipped: Dict[str, List[int]] = field(default_factory=dict)   # reason -> skipped positions
    wins: list = None           # CRE windows [w0, w1) in batch order
    gene_window: tuple = None   # (g0, g1)
    minus: bool = False


def plan_mutants(gene, start: int, end: int, ref_bases: bytes, bg_bases: Optional[bytes] = None, zygosity=(2,),
                 cre_neighbour_hood=50, gene_upstream=1000, gene_downstream=300000) -> IsmPlan:
    """Host planner.  ref_bases / bg_bases: the bytes of [start - 1, end) of the reference genome and of the reference
    item's sequence (genome + background SNPs; None = no background), forward strand.  Every (pos, alt, zyg) with
    alt in ACGT minus the reference base, in that nesting order."""
    zygosity = tuple(sorted(set(int(z) for z in zygosity)))
    if not zygosity or any(z not in (1, 2) for z in zygosity):
        raise ValueError(f"zygosity must be a non-empty subset of (1, 2), got {zygosity}")
    if end < start:
        raise ValueError(f"empty region [{start}, {end}]")
    n = end - start + 1
    bg_bases = ref_bases if bg_bases is None else bg_bases
    if len(ref_bases) != n or len(bg_bases) != n:
        raise ValueError("ref_bases / bg_bases must hold one byte per position of the region")
    minus = gene.strand == "-"
    _, wins = cre_windows(gene, cre_neighbour_hood)
    g0, g1 = gene_window(gene.start, gene.end, gene.strand, gene_upstream, gene_downstream)
    plan = IsmPlan([], {"no_overlap": [], "non_acgt": []}, wins, (g0, g1), minus)
    for i in range(n):
        pos = start + i
        hits, cre_hit, _, gene_hit = window_hits(wins, minus, pos, g0, g1)
        if cre_hit is None and not gene_hit:
            plan.skipped["no_overlap"].append(pos)
            continue
        ref = chr(ref_bases[i]).upper()
        if ref not in ACGT or chr(bg_bases[i]).upper() not in ACGT:      # VEP rejects these (seq.py:93-97)
            plan.skipped["non_acgt"].append(pos)
            continue
        for alt in ACGT:
            if alt == ref:
                continue
            for z in zygosity:
                plan.mutants.append(Mutant(pos, ref, alt, z, alt if z == 2 else get_iupac_code(ref, alt), hits, gene_hit))
    return plan


def slab_partition(n_items: int, rows_per_item: int, rows_budget: int = ROWS_BUDGET):
    """[start, stop) ranges of consecutive items with at most rows_budget CRE rows each (at least one item)."""
    per = max(1, rows_budget // max(1, rows_per_item))
    return [(a, min(n_items, a + per)) for a in range(0, n_items, per)]


def _pool(engine, W, tok):
    """seq2reg over token rows int32 [n, L] (pad = 0), POOL_ROWS windows per call -> bf16 [n, d]."""
    dev = engine.device
    outs = []
    for a in range(0, tok.shape[0], POOL_ROWS):
        t = tok[a:a + POOL_ROWS].contiguous()
        msk = (t == 0).to(torch.uint8)
        lens = ops.window_lengths(msk).cpu().numpy().astype(np.int64)
        outs.append(engine.seq2reg(W, t, msk, lens, ops.cu_seqlens(lens, dev), AttnPlan(lens, dev, W.hd)))
    return torch.cat(outs) if len(outs) > 1 else outs[0]


def _u8(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a, np.uint8)).to(dev)


def _i32(a, dev):
    return torch.from_numpy(np.ascontiguousarray(a, np.int32)).to(dev)


def _raise_on_error(err, what):
    code = int(err.item())
    if code:
        raise RuntimeError(f"stage-1 kernel reported error {code} while {what} (1: pitch overflow, 2: >2048 "
                           "variants/window, 3: substitution outside its window)")


@torch.no_grad()
def build_items(hot, gene, start: int, end: int, zygosity=(2,), variants=None):
    """Stage 1 of an ISM pass: the reference item and every mutant as rows of two tables of DISTINCT token rows.
    -> dict(plan, cre_tokens int32 [n_c, L], gene_tokens int32 [n_g, L] (distinct rows, device), cre_rows / gene_rows
    (per item, reference item first: int64 rows of the item's CRE windows / gene chunks in those tables), labels,
    counters)."""
    tok, dev = hot.tok, hot.engine.device
    L = hot.max_length
    t = hot.tokenize([gene], variants)
    off, chrom_len = hot.genome.offsets[gene.chrom]
    if not (1 <= start <= end <= chrom_len):
        raise ValueError(f"region [{start}, {end}] is outside {gene.chrom} (length {chrom_len})")
    ref_bases = hot.genome.seq[off + start - 1: off + end].cpu().numpy().tobytes()
    bg_bases = None
    if variants is not None:
        rseq, _, rerr = tok.sequences(hot.genome, [gene.chrom], [start - 1], [end], [0], variants)
        _raise_on_error(rerr, "encoding the region")
        bg_bases = rseq[0, :end - start + 1].cpu().numpy().tobytes()
    plan = plan_mutants(gene, start, end, ref_bases, bg_bases, zygosity, hot.nb, hot.up, hot.down)
    muts = plan.mutants
    ref_ctok = t["cre_tok"][0]                                      # int32 [C, L]
    ref_gtok = t["gene_tok"][0]                                     # int32 [G_ref, L]
    C, G_ref = ref_ctok.shape[0], ref_gtok.shape[0]
    g0 = plan.gene_window[0]
    flag = int(plan.minus)
    err = t["err"].clone()
    # ---- CRE windows: one mutated row per (mutant, hit window), fixed 200-token rows ----
    c_src, c_off, c_base, c_owner = [], [], [], []
    for m_i, m in enumerate(muts):
        for k in m.hits:
            c_src.append(k); c_off.append(m.pos - 1 - plan.wins[k][0]); c_base.append(ord(m.base)); c_owner.append(m_i)
    cseq, clen = t["cre_seq"]
    if c_src:
        n = len(c_src)
        mseq, mlen, err = ops.mutate_windows(cseq, clen, _i32(c_src, dev), _i32(c_off, dev), _u8(c_base, dev),
                                             _u8([flag] * n, dev), err)
        mtok, _, _ = tok.tokenize_fixed(mseq, mlen, mseq.shape[1], typical_len=max(b - a for a, b in plan.wins))
        cand_c = torch.cat([ref_ctok, mtok.to(ref_ctok.dtype)])
    else:
        cand_c = ref_ctok
    # ---- gene window: mutate + full BPE, keep the 200-token chunks that differ from the reference item's ----
    gseq, glen = t["gene_seq"]
    cap = L * hot.max_chunks
    ref_pad = torch.zeros((hot.max_chunks, L), dtype=torch.int32, device=dev)
    ref_pad[:G_ref] = ref_gtok
    gene_muts = [i for i, m in enumerate(muts) if m.gene_hit]
    g_count = np.full(len(muts), G_ref, np.int64)                  # chunks of every mutant's gene window
    g_changed = {}                                                  # mutant -> bool [G_m] changed chunks
    changed_rows = []
    for a in range(0, len(gene_muts), GENE_GROUP):
        grp = gene_muts[a:a + GENE_GROUP]
        n = len(grp)
        mseq, mlen, err = ops.mutate_windows(gseq, glen, _i32([0] * n, dev),
                                             _i32([muts[i].pos - 1 - g0 for i in grp], dev),
                                             _u8([ord(muts[i].base) for i in grp], dev), _u8([flag] * n, dev), err)
        gt, gc = ops.bpe_tokenize(mseq, mlen, mseq.shape[1], tok.merges, cap, cap)
        del mseq
        G_m = np.minimum(hot.max_chunks, (gc.cpu().numpy().astype(np.int64) + L - 1) // L)
        rows = gt.view(n, hot.max_chunks, L)
        valid = torch.arange(hot.max_chunks, device=dev)[None, :] < torch.from_numpy(G_m).to(dev)[:, None]
        changed = valid & (rows != ref_pad[None]).any(-1)
        changed_h = changed.cpu().numpy()
        changed_rows.append(rows[changed])
        for j, i in enumerate(grp):
            g_count[i] = G_m[j]
            g_changed[i] = changed_h[j, :G_m[j]]
    cand_g = torch.cat([ref_gtok] + changed_rows) if changed_rows else ref_gtok
    _raise_on_error(err, "building the mutant windows")
    # ---- every distinct token row once ----
    uc, inv_c = torch.unique(cand_c, dim=0, return_inverse=True)
    ug, inv_g = torch.unique(cand_g, dim=0, return_inverse=True)
    inv_c = inv_c.cpu().numpy().astype(np.int64); inv_g = inv_g.cpu().numpy().astype(np.int64)
    # ---- item -> rows of the pooled tables ----
    ref_c, ref_g = inv_c[:C], inv_g[:G_ref]
    cre_rows, gene_rows = [ref_c], [ref_g]
    g_next = G_ref
    c_of = {}                                                          # (mutant, window) -> row of cand_c
    for j, (m_i, k) in enumerate(zip(c_owner, c_src)):
        c_of[(m_i, k)] = C + j
    for m_i, m in enumerate(muts):
        r = ref_c.copy()
        for k in m.hits:
            r[k] = inv_c[c_of[(m_i, k)]]
        cre_rows.append(r)
        if m.gene_hit:
            ch = g_changed[m_i]
            gr = np.empty(len(ch), np.int64)
            n_ch = int(ch.sum())
            gr[ch] = inv_g[g_next:g_next + n_ch]
            keep = np.nonzero(~ch)[0]
            gr[keep] = ref_g[keep]
            g_next += n_ch
            gene_rows.append(gr)
        else:
            gene_rows.append(ref_g)
    # windows the per-variant path encodes for the same items: per variant its reference item, plus every requested
    # zygosity item (it also encodes the zygosity not asked for; not counted)
    per_variant = sum(C + int(g_count[i]) for i in range(len(muts))) + \
        len({(m.pos, m.alt) for m in muts}) * (C + G_ref)
    zyg_n = len(set(int(z) for z in zygosity))
    return dict(plan=plan, cre_tokens=uc.to(torch.int32), gene_tokens=ug.to(torch.int32), cre_rows=cre_rows,
                gene_rows=gene_rows, labels=t["labels"][0],
                counters=dict(windows_encoded=int(uc.shape[0] + ug.shape[0]), cre_windows_encoded=int(uc.shape[0]),
                              gene_chunks_encoded=int(ug.shape[0]), windows_per_variant=int(per_variant),
                              skipped={k: 3 * zyg_n * len(v) for k, v in plan.skipped.items()}))


@torch.no_grad()
def saturation_mutagenesis(hot, gene, start: int, end: int, zygosity=(2,), variants=None, rows_budget=ROWS_BUDGET,
                           timer=None):
    """ISM of [start, end] (1-based, inclusive, on gene.chrom) for one gene on HotPath `hot`.  variants: the background
    sample as stage1.SampleVariants of its SNPs only (or None).  timer: optional callable(phase name) -> context
    manager around the stage-1 / seq2reg / seq2gene phases (tools/bench_ism.py).
    -> dict(plan, pred fp32 [n_mut, T], emb fp32 [n_mut, T, D], ref_pred [T], ref_emb [T, D] (device tensors),
    counters: windows_encoded, windows_per_variant, cre_windows_encoded, gene_chunks_encoded, skipped {reason: n})."""
    import contextlib
    eng, dev = hot.engine, hot.engine.device
    phase = timer or (lambda name: contextlib.nullcontext())
    with phase("stage1"):
        it = build_items(hot, gene, start, end, zygosity, variants)
    with phase("seq2reg"):
        cre_pooled = _pool(eng, eng.cre_tok, it["cre_tokens"])
        gene_pooled = _pool(eng, eng.gene_tok, it["gene_tokens"])
    cre_rows, gene_rows = it["cre_rows"], it["gene_rows"]
    tissues = torch.as_tensor(gene.tissues, dtype=torch.long)
    T = len(gene.tissues)
    preds, embs = [], []
    with phase("seq2gene"):
        for a, b in slab_partition(len(cre_rows), len(cre_rows[0]), rows_budget):
            used, local = np.unique(np.concatenate(gene_rows[a:b]), return_inverse=True)
            splits = np.cumsum([len(r) for r in gene_rows[a:b]])[:-1]
            s = eng.prepare_shared(cre_rows[a:b], np.split(local, splits), len(used), [tissues] * (b - a),
                                   [it["labels"]] * (b - a))
            out = eng.run_pooled(s, cre_pooled, gene_pooled.index_select(0, torch.from_numpy(used).to(dev)))
            preds.append(out["pred"].view(b - a, T)); embs.append(out["emb"].view(b - a, T, -1))
    pred = torch.cat(preds); emb = torch.cat(embs)
    return dict(plan=it["plan"], pred=pred[1:], emb=emb[1:], ref_pred=pred[0], ref_emb=emb[0], counters=it["counters"])
