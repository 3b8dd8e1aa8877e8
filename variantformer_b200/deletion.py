"""In-silico genomic deletions: each gene predicted with a span of the genome deleted.

A deletion is a 1-based inclusive span [a, b] on one chromosome (a >= 2, b <= the chromosome's length).  Its result for a
gene g is BY DEFINITION what HotPath.predict gives for g with a sample equal to the background plus one VCF record
(DESIGN section 16): POS = a - 1 (the anchor), REF = genome[a-1 .. b] (L + 1 bases, L = b - a + 1), ALT = the anchor
base, GT 1/1, placed after every background record with the same POS.  This is the encoder's own rule
(vf_encode_windows_edit runs vf_encode_windows' kernel body with the record merged in), so by construction:
  * a window changes only when it contains the whole REF span, anchor included (0-based [a - 2, b) inside [w0, w1)); a
    window the deletion covers or clips keeps its bytes;
  * a background record that starts earlier and overlaps the anchor wins (the deletion is not applied); background
    records that start inside the span are dropped with it;
  * het and hom write the same bytes for an indel, so zygosity is not a parameter;
  * a deletion that no window applies gives exactly the baseline (reported with changed = False).
What is not recomputed:
  * each gene is tokenized once (HotPath.tokenize): the baseline item;
  * a deletion re-encodes only the windows that contain its REF span (its gene's CRE windows on its chromosome, and the
    gene window) with vf_encode_windows_edit; every other window keeps the baseline's token rows, exactly, since the
    record is not applied there.  Re-encoded CRE windows go through the fixed-row BPE, gene windows through the full
    BPE and 200-token chunking, ism.GENE_GROUP at a time;
  * every distinct token row (CRE window or gene chunk) goes through seq2reg once (ism._pool), and the items (baseline
    + one per deletion, per gene) run through Engine.prepare_shared + run_pooled in slabs of at most ism.ROWS_BUDGET CRE
    rows and passes of about PASS_ROWS token rows (knockout.score_items, cohort.plan_passes).  Results depend on
    neither split.
The planning is variant_sets.plan's: a deletion is its one-record set.
"""
import numpy as np
import pandas as pd
import torch

from . import ism, knockout, ops, variant_sets
from .stage1 import cre_window, gene_window

PASS_ROWS = variant_sets.PASS_ROWS


def record(spans):
    """The VCF record of deletions [a, b] (int64 [n, 2], 1-based inclusive) as the encoder reads it: (pos, ref_len) with
    pos the 0-based anchor a - 2 and ref_len = L + 1 = b - a + 2."""
    spans = np.asarray(spans, np.int64).reshape(-1, 2)
    return spans[:, 0] - 2, spans[:, 1] - spans[:, 0] + 2


def contains(w0, w1, spans):
    """Whether the window [w0, w1) (0-based) holds the whole REF span of each deletion, anchor included: the only
    windows the deletion can change.  -> bool [n]."""
    pos, rl = record(spans)
    return (np.asarray(w0) <= pos) & (pos + rl <= np.asarray(w1))


def check_deletions(genes, deletions, chroms=None, chrom_len=None, gene_names=None):
    """Validate the deletions of `genes` before any device work.  deletions: per gene an int64 array [n, 2] of 1-based
    inclusive spans [a, b]; chroms: per gene None (the gene's chromosome), one name for all its deletions or n names;
    chrom_len: {chromosome: length}.  -> per gene (spans int64 [n, 2], chromosome names [n]).  ValueError for a gene
    without CREs, a malformed array, an unknown chromosome, a < 2, b < a or b past the chromosome's end."""
    name = lambda i: gene_names[i] if gene_names is not None else f"{genes[i].chrom}:{genes[i].start}-{genes[i].end}"
    if len(deletions) != len(genes):
        raise ValueError(f"deletions has {len(deletions)} entries for {len(genes)} genes")
    if chroms is not None and len(chroms) != len(genes):
        raise ValueError(f"chroms has {len(chroms)} entries for {len(genes)} genes")
    out = []
    for i, g in enumerate(genes):
        if len(g.cre_start) == 0:
            raise ValueError(f"gene {name(i)} has no CRE: a prediction needs at least one")
        s = np.asarray(deletions[i])
        if s.size == 0:
            s = s.reshape(0, 2)
        if s.ndim != 2 or s.shape[1] != 2:
            raise ValueError(f"deletions of gene {name(i)} must be an [n, 2] array of spans, got shape {s.shape}")
        if s.size and not np.issubdtype(s.dtype, np.integer):
            raise ValueError(f"deletions of gene {name(i)} hold non-integer coordinates ({s.dtype})")
        s = s.astype(np.int64)
        c = chroms[i] if chroms is not None else None
        c = [g.chrom] * len(s) if c is None else ([c] * len(s) if isinstance(c, str) else [str(x) for x in c])
        if len(c) != len(s):
            raise ValueError(f"gene {name(i)} has {len(s)} deletions and {len(c)} chromosomes")
        for j, ((a, b), ch) in enumerate(zip(s.tolist(), c)):
            what = f"deletion {j} [{a}, {b}] on {ch} of gene {name(i)}"
            if chrom_len is not None and ch not in chrom_len:
                raise ValueError(f"{what}: chromosome {ch} is not in the genome")
            if a < 2:
                raise ValueError(f"{what}: a deletion starts at 2 or later (its anchor base, a - 1, must exist)")
            if b < a:
                raise ValueError(f"{what}: the span is empty (end < start)")
            if chrom_len is not None and b > chrom_len[ch]:
                raise ValueError(f"{what} is outside {ch} (length {chrom_len[ch]})")
        out.append((s, c))
    return out


def gene_hits(g, spans, chroms, nb, up, down):
    """Which windows of gene g each deletion changes: (cre bool [n, C] in batch order, gene bool [n])."""
    order = knockout.batch_order(g)
    w = np.asarray([cre_window(g.cre_start[r], g.cre_end[r], nb) for r in order], np.int64).reshape(-1, 2)
    wc = np.asarray([g.chrom if g.cre_chrom is None else g.cre_chrom[r] for r in order], dtype=object)
    dc = np.asarray(chroms, dtype=object).reshape(-1)
    pos, rl = record(spans)
    cre = (dc[:, None] == wc[None, :]) & (w[None, :, 0] <= pos[:, None]) & (pos[:, None] + rl[:, None] <= w[None, :, 1])
    g0, g1 = gene_window(g.start, g.end, g.strand, up, down)
    gene = (dc == g.chrom) & contains(g0, g1, spans)
    return cre.astype(bool), np.asarray(gene, bool)


def _encode_edits(hot, variants, rows, pitch):
    """vf_encode_windows_edit over rows [(chrom, w0, w1, flags, e_pos, e_ref_len, anchor byte)]."""
    dev = hot.engine.device
    v = variants or hot.tok._no_var
    base = np.asarray([hot.genome.offsets[r[0]][0] for r in rows], np.int64)
    lo_hi = np.asarray([v.window_range(r[0], r[1], r[2]) for r in rows], np.int64).reshape(-1, 2)
    col = lambda k, dt: torch.from_numpy(np.ascontiguousarray([r[k] for r in rows], dt)).to(dev)
    i32 = lambda a: torch.from_numpy(np.ascontiguousarray(a, np.int32)).to(dev)
    n = len(rows)
    return ops.encode_windows_edit(hot.genome.seq, torch.from_numpy(base).to(dev), col(1, np.int32), col(2, np.int32),
                                   i32(lo_hi[:, 0]), i32(lo_hi[:, 1]), col(3, np.uint8), v.dev, col(4, np.int32),
                                   col(5, np.int32), i32(np.arange(n)), i32(np.ones(n)), col(6, np.uint8),
                                   max(r[2] - r[1] for r in rows), pitch)


def _encode_rows(hot, variants, rows, pitch):
    """The planner's rows [(chrom, w0, w1, flags, (record,))] of one-record sets, through _encode_edits."""
    return _encode_edits(hot, variants, [(ch, w0, w1, fl, r[0][1], r[0][2], r[0][3][0]) for ch, w0, w1, fl, r in rows],
                         pitch)


@torch.no_grad()
def deletion_scan(hot, genes, deletions, variants=None, chroms=None, embeddings=False, to_host=True,
                  rows_budget=ism.ROWS_BUDGET, pass_rows=None, timer=None, counters=None, min_gene_len=None,
                  gene_names=None):
    """Every deletion of `genes` (GeneSpec list) on HotPath `hot`, with the sample background `variants`
    (stage1.SampleVariants, or None for the reference genome).  deletions / chroms: see check_deletions.
    -> (pred fp32 [sum T], emb fp32 [sum T, D], del_pred: per gene fp32 [n_g, T_g][, del_emb: per gene fp32 [n_g, T_g,
    D] when `embeddings`], applied: per gene dict(cre=bool [n_g, C_g] (CRE windows in batch order), gene=bool [n_g])),
    numpy (to_host) or device tensors (applied is numpy either way).  pred / emb are bit-identical to
    HotPath.predict(genes, variants), del_pred[g][j] to HotPath.predict on gene g with deletion j's record added to the
    background.  applied: the windows whose bytes the deletion changed.  timer: optional callable(phase) -> context
    manager around the "stage1", "seq2reg" and "seq2gene" phases; counters: optional dict filled with item / window
    counts; min_gene_len: VCFDataset's gene-window length rule, a ValueError for any item, baseline or deletion, whose
    encoded gene window is not longer (gene_names name the genes).
    A deletion is the one-record set of variant_sets' planner: its record (record()) with the anchor base as ALT."""
    names = gene_names if gene_names is not None else [f"{g.chrom}:{g.start}-{g.end}" for g in genes]
    dels = check_deletions(genes, deletions, chroms, {k: v[1] for k, v in hot.genome.offsets.items()}, names)
    dev = hot.engine.device
    sets = []
    for s, ch in dels:
        pos, rl = record(s)
        idx = [hot.genome.offsets[x][0] + int(p) for x, p in zip(ch, pos)]
        anc = (hot.genome.seq[torch.as_tensor(idx, dtype=torch.long, device=dev)].cpu().numpy() if idx
               else np.zeros(0, np.uint8))
        sets.append([((x, int(p), int(r), bytes([int(y)]), 2),) for x, p, r, y in zip(ch, pos, rl, anc)])
    c = counters if counters is not None else {}
    out = variant_sets.plan(hot, genes, sets, variants, embeddings, to_host, rows_budget, pass_rows, timer, c,
                            min_gene_len, names, encode=_encode_rows)
    c["deletions"] = c.pop("sets")
    for ap in out[-1]:
        del ap["records"]
    return out


def tiles(chrom, start, end, width, step):
    """Deletions of `width` bases every `step` bases over [start, end] (1-based, inclusive): spans [s, s + width - 1]
    for s = start, start + step, ... while s + width - 1 <= end.  -> DataFrame (chromosome, start, end), to which a
    gene_id (and a label) column is added for VCFProcessor.deletion_scan."""
    if width < 1 or step < 1:
        raise ValueError(f"tile width {width} and step {step} must be at least 1")
    if end - start + 1 < width:
        raise ValueError(f"region [{start}, {end}] is shorter than one tile of {width} bases")
    s = np.arange(int(start), int(end) - int(width) + 2, int(step), dtype=np.int64)
    return pd.DataFrame({"chromosome": chrom, "start": s, "end": s + int(width) - 1})


def default_spans(manifest):
    """The default scan: every CRE's own bases deleted singly, on its manifest chromosome: 1-based [start_cre + 1,
    end_cre] (the manifest's 0-based half-open coordinates).  -> (spans int64 [C, 2], chromosomes [C])."""
    s = manifest["start_cre"].to_numpy(np.int64)
    return np.stack([s + 1, manifest["end_cre"].to_numpy(np.int64)], 1), [str(x) for x in manifest["chromosome"]]


def user_deletions(df):
    """User deletions from a DataFrame with columns gene_id, chromosome, start, end (1-based inclusive) and optionally
    label.  -> {gene_id: (labels [n], spans int64 [n, 2], chromosomes [n])} in first-appearance order; the default label
    is "chromosome:start-end"."""
    missing = [k for k in ("gene_id", "chromosome", "start", "end") if k not in df.columns]
    if missing:
        raise ValueError(f"deletions must have the columns gene_id, chromosome, start and end (missing: {missing})")
    out = {}
    labels = df["label"] if "label" in df.columns else [None] * len(df)
    for gid, ch, a, b, lab in zip(df["gene_id"], df["chromosome"], df["start"], df["end"], labels):
        for x in (a, b):
            if isinstance(x, (bool, np.bool_)) or not isinstance(x, (int, np.integer)):
                raise ValueError(f"deletion {ch}:{a}-{b} of gene {gid}: {x!r} is not an integer coordinate")
        d = out.setdefault(gid, ([], [], []))
        d[0].append(f"{ch}:{a}-{b}" if lab is None or (not isinstance(lab, str) and pd.isna(lab)) else lab)
        d[1].append((int(a), int(b))); d[2].append(str(ch))
    return {g: (lab, np.asarray(s, np.int64).reshape(-1, 2), ch) for g, (lab, s, ch) in out.items()}


FRAME_COLUMNS = ["gene_id", "tissue", "deletion", "chromosome", "del_start", "del_end", "width", "cre_windows_changed",
                 "gene_window_changed", "changed", "start_cre", "end_cre", "cre_name", "baseline_expression",
                 "predicted_expression", "delta"]


def deletion_frame(gene_id, tissues, labels, spans, chroms, applied, base_pred, del_pred, manifest=None):
    """One query row's deletions in long format: one row per (deletion, tissue), in that order.  labels / spans [n, 2] /
    chroms: the deletions; applied: dict(cre=bool [n, C], gene=bool [n]); base_pred fp32 [T]; del_pred fp32 [n, T];
    manifest: for the default scan the gene's manifest (deletion i = its row i), whose columns start_cre, end_cre and
    cre_name fill the frame's (null otherwise), so it joins with cre_knockout's and cre_attention's frames."""
    T, n = len(tissues), len(labels)
    spans = np.asarray(spans, np.int64).reshape(n, 2)
    base = np.asarray(base_pred, np.float32).reshape(T)
    dp = np.asarray(del_pred, np.float32).reshape(n, T)
    rep = lambda xs: np.repeat(np.asarray(xs), T) if n else np.asarray(xs)
    n_cre = applied["cre"].sum(1).astype(np.int64)
    gene = applied["gene"].astype(bool)
    if manifest is not None:
        m = [manifest[k].tolist() for k in ("start_cre", "end_cre", "cre_name")]
    else:
        m = [[None] * n] * 3
    rep_list = lambda xs: [x for x in xs for _ in range(T)]
    return pd.DataFrame({
        "gene_id": [gene_id] * (n * T), "tissue": list(tissues) * n, "deletion": rep_list(labels),
        "chromosome": pd.Series(rep_list(chroms), dtype=object), "del_start": rep(spans[:, 0]).astype(np.int64),
        "del_end": rep(spans[:, 1]).astype(np.int64), "width": rep(spans[:, 1] - spans[:, 0] + 1).astype(np.int64),
        "cre_windows_changed": rep(n_cre).astype(np.int64), "gene_window_changed": rep(gene).astype(bool),
        "changed": rep((n_cre > 0) | gene).astype(bool),
        "start_cre": pd.array([None if x is None else int(x) for x in rep_list(m[0])], dtype="Int64"),
        "end_cre": pd.array([None if x is None else int(x) for x in rep_list(m[1])], dtype="Int64"),
        "cre_name": pd.Series(rep_list(m[2]), dtype=object),
        "baseline_expression": np.tile(base, n), "predicted_expression": dp.reshape(-1),
        "delta": (dp - base[None, :]).reshape(-1)}, columns=FRAME_COLUMNS)
