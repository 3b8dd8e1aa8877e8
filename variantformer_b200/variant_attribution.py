"""Variant attribution: each gene predicted with some of the sample's own records removed or re-genotyped.

A genotype edit is one record of the sample's variant table (stage1.SampleVariants) with a new GT: 0 (the line removed),
1 (het) or 2 (hom-alt); an edit set is one or more edits of distinct records.  The result of set S for gene g is BY
DEFINITION what HotPath.predict gives for g when the sample's table has each edited record's GT replaced (DESIGN
section 19).  GT 0 is the line deleted, since the encoder skips gt 0 records.  Everything else is the encoder's own rule
(vf_encode_windows_overrides runs vf_encode_windows' kernel body reading each record's gt through the row's override
list): removing a record that blocked a later overlapping record lets that record apply, a het SNP writes its IUPAC code
and a hom SNP its ALT, a het indel writes the bytes of a hom indel (so het <-> hom is a no-op for an indel), and editing a
record a window does not apply (blocked, straddling the window's end) leaves that window unchanged.  A set whose windows
all encode to the baseline's tokens gives exactly the baseline, reported with changed = False.
The reference-genome prediction is the set "every record in the gene's windows removed" (all_removed()), equal to
HotPath.predict(genes, None).
What is not recomputed is variant_sets.plan's: each gene is tokenized once; a set re-encodes only the windows that hold
one of its records' whole REF span (the only windows an edit can change: a record straddling a window is never applied
there, so it never blocks anything), one encode row per distinct (window, the set's edits in it) across a pass; every
distinct token row goes through seq2reg once; items run in bounded slabs and passes.  A window is changed iff its token
row (CRE) or chunk list (gene window) differs from the baseline's: tokens past truncation are invisible to the model.
"""
from typing import NamedTuple

import numpy as np
import pandas as pd
import torch

from . import ism, knockout, ops, variant_sets

SCOPES = ("record", "window")


class Edit(NamedTuple):
    """One record of the sample named as in its VCF line (chromosome, 1-based POS, REF, ALT) and its new GT (0 removed,
    1 het, 2 hom-alt).  REF is matched by its length: the variant table keeps no REF bases."""
    chrom: str
    pos: int
    ref: str
    alt: str
    gt: int = 0


def _host(variants, ch):
    return (variants.host_pos[ch], variants.host_ref_len[ch], variants.host_alt[ch], variants.host_gt[ch],
            variants.ranges[ch][0])


def _record(variants, ch, i, gt):
    """The planner's record of table index i on chromosome ch with new gt: (chrom, pos0, ref_len, alt, gt, index)."""
    pos, rl, alt, _, base = _host(variants, ch)
    k = i - base
    return (ch, int(pos[k]), int(rl[k]), bytes(alt[k]), int(gt), int(i))


def check_edits(genes, sets, variants, gene_names=None):
    """Resolve and validate the edit sets of `genes` against the sample `variants` (stage1.SampleVariants) before any
    kernel runs.  sets: per gene a list of sets, each a list of Edit.  -> per gene a list of sets, each a tuple of
    planner records (chrom, pos0, ref_len, alt bytes, new gt, table index) in table order.  ValueError for a gene
    without CREs, an empty set, a record the sample does not carry (chromosome, POS, REF length and ALT, ALT compared
    case-insensitively), an ambiguous match (two such lines), a GT outside {0, 1, 2} and the same record twice in a set."""
    name = lambda i: gene_names[i] if gene_names is not None else f"{genes[i].chrom}:{genes[i].start}-{genes[i].end}"
    if len(sets) != len(genes):
        raise ValueError(f"sets has {len(sets)} entries for {len(genes)} genes")
    out = []
    for i, g in enumerate(genes):
        if len(g.cre_start) == 0:
            raise ValueError(f"gene {name(i)} has no CRE: a prediction needs at least one")
        gs = []
        for j, s in enumerate(sets[i]):
            if len(s) == 0:
                raise ValueError(f"set {j} of gene {name(i)} is empty")
            recs = []
            for e in s:
                e = Edit(*e)
                what = f"edit {variant_sets._label(e)} of set {j} of gene {name(i)}"
                if isinstance(e.gt, (bool, np.bool_)) or not isinstance(e.gt, (int, np.integer)) or e.gt not in (0, 1, 2):
                    raise ValueError(f"{what}: GT {e.gt!r} must be 0 (removed), 1 (het) or 2 (hom-alt)")
                if isinstance(e.pos, (bool, np.bool_)) or not isinstance(e.pos, (int, np.integer)):
                    raise ValueError(f"{what}: POS {e.pos!r} is not an integer")
                if variants is None or e.chrom not in variants.ranges:
                    raise ValueError(f"{what}: the sample carries no such record")
                pos, rl, alt, _, base = _host(variants, e.chrom)
                a = int(np.searchsorted(pos, int(e.pos) - 1, "left")); b = int(np.searchsorted(pos, int(e.pos) - 1, "right"))
                want = str(e.alt).upper().encode()
                hit = [base + k for k in range(a, b) if rl[k] == len(e.ref) and bytes(alt[k]).upper() == want]
                if not hit:
                    raise ValueError(f"{what}: the sample carries no such record")
                if len(hit) > 1:
                    raise ValueError(f"{what}: ambiguous, the sample has {len(hit)} such lines")
                recs.append(_record(variants, e.chrom, hit[0], e.gt))
            recs.sort(key=lambda r: r[5])
            for x, y in zip(recs, recs[1:]):
                if x[5] == y[5]:
                    raise ValueError(f"set {j} of gene {name(i)} edits the record at {x[0]}:{x[1] + 1} twice")
            gs.append(tuple(recs))
        out.append(gs)
    return out


def window_records(g, variants, nb, up, down):
    """The sample's records whose REF span lies in each window of gene g (CRE windows in batch order, then the gene
    window) and whose GT is not 0: -> per window a list of (chrom, table index), in table order."""
    out = []
    for ch, w0, w1 in variant_sets._windows(g, nb, up, down):
        if variants is None or ch not in variants.ranges:
            out.append([]); continue
        pos, rl, _, gt, base = _host(variants, ch)
        lo, hi = variants.window_range(ch, w0, w1)
        k = np.arange(lo - base, hi - base)
        k = k[(pos[k] + rl[k] <= w1) & (gt[k] != 0)]
        out.append([(ch, int(base + x)) for x in k])
    return out


def all_removed(g, variants, nb, up, down):
    """The reference set of gene g: every record of the sample in its windows removed (planner records), or () when
    there is none."""
    recs = sorted({r for w in window_records(g, variants, nb, up, down) for r in w}, key=lambda r: r[1])
    return tuple(_record(variants, ch, i, 0) for ch, i in recs)


def default_sets(g, variants, nb, up, down, scope="record", genome=None):
    """The default scans of gene g.  scope "record" (leave-one-out): one set per record of the sample whose REF span lies
    in at least one of the gene's windows and whose GT is not 0, removing it, in table order; labels
    "chrom:pos:REF>ALT" (REF read from `genome`, stage1.Genome, or "N"s without one).  scope "window": one set per window
    that holds such records, removing all of them; labels "cre_window:<manifest row>" / "gene_window".
    -> (sets of planner records, labels, sample GT per set (None for a window set))."""
    if scope not in SCOPES:
        raise ValueError(f"scope must be one of {SCOPES}, got {scope!r}")
    per_win = window_records(g, variants, nb, up, down)
    if scope == "window":
        order = knockout.batch_order(g)
        sets, labels = [], []
        for k, w in enumerate(per_win):
            if w:
                sets.append(tuple(_record(variants, ch, i, 0) for ch, i in w))
                labels.append(f"cre_window:{int(order[k])}" if k < len(per_win) - 1 else "gene_window")
        return sets, labels, [None] * len(sets)
    recs = sorted({r for w in per_win for r in w}, key=lambda r: r[1])
    sets = [(_record(variants, ch, i, 0),) for ch, i in recs]
    refs = _ref_bases(genome, [s[0] for s in sets])
    labels = [f"{r[0]}:{r[1] + 1}:{ref}>{r[3].decode(errors='replace')}" for (r,), ref in zip(sets, refs)]
    return sets, labels, [sample_gt(variants, s[0]) for s in sets]


def _ref_bases(genome, recs):
    if genome is None or not recs:
        return ["N" * r[2] for r in recs]
    idx = np.concatenate([genome.offsets[r[0]][0] + r[1] + np.arange(r[2]) for r in recs])
    got = genome.seq[torch.as_tensor(idx, dtype=torch.long, device=genome.seq.device)].cpu().numpy().tobytes()
    out, o = [], 0
    for r in recs:
        out.append(got[o:o + r[2]].decode(errors="replace").upper()); o += r[2]
    return out


def _encode_overrides(hot, variants, rows, pitch):
    """vf_encode_windows_overrides over the planner's rows [(chrom, w0, w1, flags, records)], records (chrom, pos0,
    ref_len, alt, new gt, table index) in table order.  -> (out, out_len, applied (unused: zeros), err)."""
    dev = hot.engine.device
    base = np.asarray([hot.genome.offsets[r[0]][0] for r in rows], np.int64)
    lo_hi = np.asarray([variants.window_range(r[0], r[1], r[2]) for r in rows], np.int64).reshape(-1, 2)
    col = lambda k, dt: torch.from_numpy(np.ascontiguousarray([r[k] for r in rows], dt)).to(dev)
    recs = [x for r in rows for x in r[4]]
    off = np.concatenate([[0], np.cumsum([len(r[4]) for r in rows])]).astype(np.int32)
    out, lens, err = ops.encode_windows_overrides(
        hot.genome.seq, torch.from_numpy(base).to(dev), col(1, np.int32), col(2, np.int32),
        torch.from_numpy(lo_hi[:, 0].astype(np.int32)).to(dev), torch.from_numpy(lo_hi[:, 1].astype(np.int32)).to(dev),
        col(3, np.uint8), variants.dev, torch.from_numpy(off).to(dev),
        torch.from_numpy(np.asarray([x[5] for x in recs], np.int32)).to(dev),
        torch.from_numpy(np.asarray([x[4] for x in recs], np.uint8)).to(dev), max(r[2] - r[1] for r in rows), pitch)
    return out, lens, torch.zeros(len(recs), dtype=torch.uint8, device=dev), err


@torch.no_grad()
def scan(hot, genes, sets, variants, embeddings=False, to_host=True, rows_budget=ism.ROWS_BUDGET, pass_rows=None,
         timer=None, counters=None, min_gene_len=None, gene_names=None):
    """Every edit set of `genes` (GeneSpec list) on HotPath `hot` for the sample `variants` (stage1.SampleVariants).
    sets: per gene a list of sets, each a list of Edit.  -> as variant_sets.scan: (pred fp32 [sum T], emb fp32 [sum T,
    D], set_pred: per gene fp32 [n_g, T_g][, set_emb: per gene fp32 [n_g, T_g, D] when `embeddings`], changed: per gene
    dict(cre=bool [n_g, C_g] (CRE windows in batch order), gene=bool [n_g], records=per set bool [len(set)] (a window
    holding the record changed), in the set's table order)).  pred / emb are bit-identical to HotPath.predict(genes,
    variants), set_pred[g][j] to HotPath.predict on gene g with set j's GTs replaced in the sample's table."""
    names = gene_names if gene_names is not None else [f"{g.chrom}:{g.start}-{g.end}" for g in genes]
    checked = check_edits(genes, sets, variants, names)
    return run(hot, genes, checked, variants, embeddings, to_host, rows_budget, pass_rows, timer, counters,
               min_gene_len, names)


def run(hot, genes, checked, variants, embeddings=False, to_host=True, rows_budget=ism.ROWS_BUDGET, pass_rows=None,
        timer=None, counters=None, min_gene_len=None, gene_names=None):
    """scan() on sets already resolved to planner records (check_edits, default_sets, all_removed; an empty set is the
    baseline)."""
    names = gene_names if gene_names is not None else [f"{g.chrom}:{g.start}-{g.end}" for g in genes]
    return variant_sets.plan(hot, genes, checked, variants, embeddings, to_host, rows_budget, pass_rows, timer,
                             counters, min_gene_len, names, encode=_encode_overrides, changed_by_tokens=True)


def user_edits(df):
    """Edit sets from a DataFrame with columns gene_id, chromosome, pos, ref, alt, gt and optionally set and label.
    Without a set column every row is a set of its own, labelled by its record.  -> {gene_id: [(set label, [Edit],
    [record labels])]} (sets in first-appearance order)."""
    if "gt" not in df.columns:
        raise ValueError("edits must have the columns gene_id, chromosome, pos, ref, alt and gt (missing: ['gt'])")
    if "set" not in df.columns:
        out = variant_sets.user_records(df.assign(set=np.arange(len(df))), sets=True)
        return {g: [(ls[0], [Edit(*r) for r in rs], ls) for _, rs, ls in v] for g, v in out.items()}
    out = variant_sets.user_records(df, sets=True)
    return {g: [(sid, [Edit(*r) for r in rs], ls) for sid, rs, ls in v] for g, v in out.items()}


def sample_gt(variants, rec):
    """The sample's own GT of a planner record."""
    return int(variants.host_gt[rec[0]][rec[5] - variants.ranges[rec[0]][0]])


ATTRIBUTION_COLUMNS = variant_sets.SET_COLUMNS + ["sample_gt", "new_gt", "reference_expression"]


def attribution_frame(gene_id, tissues, labels, sets, sample_gt, changed, base_pred, set_pred, ref_pred):
    """One query row's edit sets in long format: one row per (set, tissue), in that order, columns ATTRIBUTION_COLUMNS.
    sets: planner records per set; sample_gt: the sample's GT per set (single-record sets; None otherwise); changed:
    dict(cre, gene, records) as scan returns it; base_pred / ref_pred fp32 [T] (baseline, all records removed);
    set_pred fp32 [n, T].  delta = predicted - baseline: the contribution of a removed record is -delta."""
    T, n = len(tissues), len(labels)
    f = variant_sets.set_frame(gene_id, tissues, labels, [len(s) for s in sets], changed, base_pred, set_pred)
    one = lambda xs: pd.array([None if x is None else int(x) for x in xs for _ in range(T)], dtype="Int64")
    f["sample_gt"] = one([g if len(s) == 1 else None for g, s in zip(sample_gt, sets)])
    f["new_gt"] = one([s[0][4] if len(s) == 1 else None for s in sets])
    f["reference_expression"] = np.tile(np.asarray(ref_pred, np.float32).reshape(T), n)
    return f[ATTRIBUTION_COLUMNS]
