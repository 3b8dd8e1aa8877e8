"""In-silico variant combinations: each gene predicted with a set of VCF records added to the sample.

A record is a VCF line (chromosome, 1-based POS, REF, ALT, GT 1 = het / 2 = hom-alt); a set is one or more records.
The result of set S for gene g is BY DEFINITION what HotPath.predict gives for g with a sample equal to the background
plus S's records (DESIGN section 17), each placed after every background record with the same POS, the set's records in
(POS, given order).  Everything else is the encoder's own rule (vf_encode_windows_edits runs vf_encode_windows' kernel
body with the records merged in): a window changes only if it contains a record's whole REF span, an earlier
overlapping background record wins, a het SNP writes the IUPAC code, het and hom write the same bytes for an indel, and
a set that no window applies gives exactly the baseline (reported with changed = False).
What is not recomputed:
  * each gene is tokenized once (HotPath.tokenize): the baseline item;
  * a set re-encodes only the windows that contain one of its records' REF span (its gene's CRE windows on the record's
    chromosome, and the gene window), each with the set restricted to that window.  One encode row is formed per
    distinct key (window, restricted records) across the sets of a pass, so a pair scan's cross-window pairs reuse its
    singles' rows and only same-window pairs add rows.  CRE rows go through the fixed-row BPE, gene rows through the full
    BPE and 200-token chunking, ism.GENE_GROUP at a time;
  * every distinct token row goes through seq2reg once (ism._pool), and the items (baseline + one per set, per gene) run
    through Engine.prepare_shared + run_pooled in slabs of at most ism.ROWS_BUDGET CRE rows and passes of about
    PASS_ROWS token rows (knockout.score_items, cohort.plan_passes).  Results depend on neither split.
In-silico deletions (deletion.deletion_scan) are the one-record case of this planner (plan()).
"""
import contextlib
from typing import NamedTuple

import numpy as np
import pandas as pd
import torch

from . import cohort, ism, knockout, ops
from .stage1 import FLAG_REVCOMP, cre_window, gene_window

PASS_ROWS = cohort.PASS_ROWS
# edited CRE windows per encode + BPE call (bounds the rows' buffers; results do not depend on the split)
CRE_EDIT_ROWS = 16384
ALT_BASES = set(b"ACGTNacgtn")


class Record(NamedTuple):
    """One VCF line: chromosome, 1-based POS, REF, ALT and GT (1 = het, 2 = hom-alt)."""
    chrom: str
    pos: int
    ref: str
    alt: str
    gt: int = 2


def _label(r):
    return f"{r.chrom}:{r.pos}:{r.ref}>{r.alt}"


def check_sets(genes, sets, genome, gene_names=None):
    """Validate the record sets of `genes` before any kernel of ours runs.  sets: per gene a list of sets, each a list of
    Record; genome: stage1.Genome (REF is compared with its bases).  -> per gene a list of sets, each a tuple of
    (chrom, pos0, ref_len, alt bytes, gt) in (POS, given order), pos0 = POS - 1.  ValueError for a gene without CREs,
    an empty set, an unknown chromosome, a POS outside it, REF not the genome's bases (case-insensitive), ALT empty, not
    in ACGTN, symbolic, '*' or equal to REF, GT not 1 or 2, and two records of one set whose REF spans overlap."""
    name = lambda i: gene_names[i] if gene_names is not None else f"{genes[i].chrom}:{genes[i].start}-{genes[i].end}"
    if len(sets) != len(genes):
        raise ValueError(f"sets has {len(sets)} entries for {len(genes)} genes")
    recs = []                                                   # (gene, set, record) of every record, checked alone
    for i, g in enumerate(genes):
        if len(g.cre_start) == 0:
            raise ValueError(f"gene {name(i)} has no CRE: a prediction needs at least one")
        for j, s in enumerate(sets[i]):
            if len(s) == 0:
                raise ValueError(f"set {j} of gene {name(i)} is empty")
            for r in s:
                r = Record(*r)
                what = f"record {_label(r)} of set {j} of gene {name(i)}"
                if r.chrom not in genome.offsets:
                    raise ValueError(f"{what}: chromosome {r.chrom} is not in the genome")
                if isinstance(r.pos, (bool, np.bool_)) or not isinstance(r.pos, (int, np.integer)):
                    raise ValueError(f"{what}: POS {r.pos!r} is not an integer")
                ref, alt = str(r.ref), str(r.alt)
                n = genome.offsets[r.chrom][1]
                if r.pos < 1 or r.pos + max(len(ref), 1) - 1 > n:
                    raise ValueError(f"{what} is outside {r.chrom} (length {n})")
                if len(ref) == 0:
                    raise ValueError(f"{what}: REF is empty")
                if len(alt) == 0 or alt == "*" or alt.startswith("<") or not set(alt.encode()) <= ALT_BASES:
                    raise ValueError(f"{what}: ALT {alt!r} must be bases from ACGTN (no symbolic or '*' allele)")
                if alt.upper() == ref.upper():
                    raise ValueError(f"{what}: ALT equals REF")
                if r.gt not in (1, 2) or isinstance(r.gt, (bool, np.bool_)):
                    raise ValueError(f"{what}: GT {r.gt!r} must be 1 (het) or 2 (hom-alt)")
                recs.append((what, r))
    if recs:                                                    # REF against the genome: one gather for all records
        idx = np.concatenate([genome.offsets[r.chrom][0] + r.pos - 1 + np.arange(len(r.ref)) for _, r in recs])
        got = genome.seq[torch.as_tensor(idx, dtype=torch.long, device=genome.seq.device)].cpu().numpy().tobytes()
        o = 0
        for what, r in recs:
            b = got[o:o + len(r.ref)]; o += len(r.ref)
            if b.upper() != str(r.ref).upper().encode():
                raise ValueError(f"{what}: REF {r.ref} is not the genome's {b.decode(errors='replace')}")
    out = []
    for i, g in enumerate(genes):
        gs = []
        for j, s in enumerate(sets[i]):
            t = sorted(((str(r[0]), int(r[1]) - 1, len(r[2]), str(r[3]).encode(), int(Record(*r).gt)) for r in s),
                       key=lambda x: (x[0], x[1]))              # stable: records of one POS keep their order
            for a, b in zip(t, t[1:]):
                if a[0] == b[0] and a[1] + a[2] > b[1]:
                    raise ValueError(f"set {j} of gene {name(i)}: the REF spans of the records at {a[0]}:{a[1] + 1} "
                                     f"and {b[0]}:{b[1] + 1} overlap")
            gs.append(tuple(t))
        out.append(gs)
    return out


def pairs(records):
    """A pair scan of `records` (Record list): -> (sets, singles, pair_idx, overlapping): sets = every single, then every
    unordered pair whose REF spans do not overlap; singles[i] / pair_idx[k] = (i, j) index `sets` (set i is record i,
    set len(records) + k the pair pair_idx[k]); overlapping = the pairs (i, j) left out (two alleles of one site, ...)."""
    recs = [Record(*r) for r in records]
    span = lambda r: (r.chrom, int(r.pos), int(r.pos) + len(r.ref))
    sets, pair_idx, overlapping = [[r] for r in recs], [], []
    for i in range(len(recs)):
        for j in range(i + 1, len(recs)):
            (ca, a0, a1), (cb, b0, b1) = span(recs[i]), span(recs[j])
            if ca == cb and a0 < b1 and b0 < a1:
                overlapping.append((i, j))
            else:
                pair_idx.append((i, j)); sets.append([recs[i], recs[j]])
    return sets, list(range(len(recs))), pair_idx, overlapping


def _windows(g, nb, up, down):
    """Gene g's windows: the CRE windows in batch order, then the gene window, as (chrom, w0, w1)."""
    order = knockout.batch_order(g)
    w = [(g.chrom if g.cre_chrom is None else g.cre_chrom[r],) + tuple(int(x) for x in cre_window(g.cre_start[r],
                                                                                                    g.cre_end[r], nb))
         for r in order]
    return w + [(g.chrom,) + tuple(int(x) for x in gene_window(g.start, g.end, g.strand, up, down))]


def set_windows(g, sets, nb, up, down):
    """Which windows of gene g each set's records fall in: per set a dict {window index: record positions in the set},
    window index k < C a CRE window in batch order, C the gene window.  A window holds a record iff it contains the
    record's whole REF span: the only windows the record can change."""
    win = _windows(g, nb, up, down)
    wc = np.asarray([w[0] for w in win], dtype=object)
    w0 = np.asarray([w[1] for w in win], np.int64); w1 = np.asarray([w[2] for w in win], np.int64)
    uniq = {}
    for s in sets:
        for r in s:
            uniq.setdefault(r[:3], None)
    hits = {}
    for key in uniq:
        ch, p, rl = key
        hits[key] = np.flatnonzero((wc == ch) & (w0 <= p) & (p + rl <= w1)).tolist()
    out = []
    for s in sets:
        d = {}
        for m, r in enumerate(s):
            for k in hits[r[:3]]:
                d.setdefault(k, []).append(m)
        out.append(d)
    return out


def _encode_sets(hot, variants, rows, pitch):
    """vf_encode_windows_edits over rows [(chrom, w0, w1, flags, records)] -> (out, out_len, applied per record, err)."""
    dev = hot.engine.device
    v = variants or hot.tok._no_var
    base = np.asarray([hot.genome.offsets[r[0]][0] for r in rows], np.int64)
    lo_hi = np.asarray([v.window_range(r[0], r[1], r[2]) for r in rows], np.int64).reshape(-1, 2)
    col = lambda k, dt: torch.from_numpy(np.ascontiguousarray([r[k] for r in rows], dt)).to(dev)
    i32 = lambda a: torch.from_numpy(np.ascontiguousarray(a, np.int32)).to(dev)
    recs = [x for r in rows for x in r[4]]
    al = np.asarray([len(x[3]) for x in recs], np.int64)
    pool = np.frombuffer(b"".join(x[3] for x in recs), np.uint8)
    return ops.encode_windows_edits(hot.genome.seq, torch.from_numpy(base).to(dev), col(1, np.int32), col(2, np.int32),
                                    i32(lo_hi[:, 0]), i32(lo_hi[:, 1]), col(3, np.uint8), v.dev,
                                    i32(np.concatenate([[0], np.cumsum([len(r[4]) for r in rows])])),
                                    i32([x[1] for x in recs]), i32([x[2] for x in recs]), i32(np.cumsum(al) - al),
                                    i32(al), torch.from_numpy(np.asarray([x[4] for x in recs], np.uint8)).to(dev),
                                    torch.from_numpy(pool.copy()).to(dev), max(r[2] - r[1] for r in rows), pitch)


def _raise(code, name):
    raise RuntimeError(f"stage-1 kernel reported error {code} for an edited window of gene {name} (1: pitch overflow, "
                       "2: >2048 variants/window)")


@torch.no_grad()
def scan(hot, genes, sets, variants=None, embeddings=False, to_host=True, rows_budget=ism.ROWS_BUDGET, pass_rows=None,
         timer=None, counters=None, min_gene_len=None, gene_names=None):
    """Every record set of `genes` (GeneSpec list) on HotPath `hot`, with the sample background `variants`
    (stage1.SampleVariants, or None for the reference genome).  sets: per gene a list of sets, each a list of Record.
    -> (pred fp32 [sum T], emb fp32 [sum T, D], set_pred: per gene fp32 [n_g, T_g][, set_emb: per gene fp32 [n_g, T_g,
    D] when `embeddings`], applied: per gene dict(cre=bool [n_g, C_g] (CRE windows in batch order), gene=bool [n_g],
    records=per set bool [len(set)] in the set's (POS, given order))), numpy (to_host) or device tensors (applied is
    numpy either way).  pred / emb are bit-identical to HotPath.predict(genes, variants), set_pred[g][j] to
    HotPath.predict on gene g with set j's records added to the background.  applied: the windows whose bytes the set
    changed, and whether each record was applied in at least one window.  timer: optional callable(phase) -> context
    manager around the "stage1", "seq2reg" and "seq2gene" phases; counters: optional dict filled with item / window
    counts; min_gene_len: VCFDataset's gene-window length rule, a ValueError for any item whose encoded gene window is
    not longer (gene_names name the genes)."""
    names = gene_names if gene_names is not None else [f"{g.chrom}:{g.start}-{g.end}" for g in genes]
    checked = check_sets(genes, sets, hot.genome, names)
    return plan(hot, genes, checked, variants, embeddings, to_host, rows_budget, pass_rows, timer, counters,
                min_gene_len, names)


def plan(hot, genes, sets, variants, embeddings, to_host, rows_budget, pass_rows, timer, counters, min_gene_len, names,
         encode=None, changed_by_tokens=False):
    """The edited-window planner behind scan(), deletion.deletion_scan and variant_attribution.scan: sets as check_sets
    returns them (validated; a record is a tuple whose first three fields are (chrom, pos0, ref_len), the rest is the
    encoder's); encode(hot, variants, rows, pitch) -> (out, out_len, applied per record, err) encodes rows [(chrom, w0,
    w1, flags, records)] (default _encode_sets, looked up at call time).  changed_by_tokens: a window counts as changed
    when its token row (CRE) or chunk list (gene) differs from the baseline's, and a record as applied when a window
    holding it changed (the encoder's applied flags are not read); otherwise the encoder's applied flags decide."""
    encode = encode if encode is not None else _encode_sets
    eng, dev = hot.engine, hot.engine.device
    phase = timer or (lambda name: contextlib.nullcontext())
    pass_rows = PASS_ROWS if pass_rows is None else pass_rows
    L, CW = hot.max_length, hot.max_chunks
    hits = [set_windows(g, s, hot.nb, hot.up, hot.down) for g, s in zip(genes, sets)]
    T = np.asarray([len(g.tissues) for g in genes], np.int64)
    t_off = np.concatenate([[0], np.cumsum(T)])
    pred = torch.empty(int(t_off[-1]), dtype=torch.float32, device=dev)
    emb = torch.empty((int(t_off[-1]), eng.w.D), dtype=torch.float32, device=dev)
    set_pred, set_emb = [None] * len(genes), [None] * len(genes)
    applied = [dict(cre=np.zeros((len(s), len(g.cre_start)), bool), gene=np.zeros(len(s), bool),
                    records=[np.zeros(len(x), bool) for x in s]) for g, s in zip(genes, sets)]
    c = counters if counters is not None else {}
    c.update(genes=len(genes), sets=sum(len(s) for s in sets), changed=0, items=0, windows_encoded=0,
             windows_per_item=0, cre_windows_edited=0, gene_windows_edited=0, cre_token_rows=0, gene_token_rows=0,
             passes=0, slabs=0)

    def short(n, i):
        return ValueError(f"Mutated sequence is less than {min_gene_len}bp for gene {names[i]}") if \
            min_gene_len is not None and n <= min_gene_len else None

    def key(gi, j, k):
        g = genes[gi]
        w = win[gi][k]
        return (k == len(g.cre_start),) + w + (FLAG_REVCOMP if g.strand == "-" else 0,
                                               tuple(sets[gi][j][m] for m in hits[gi][j][k]))

    win = [_windows(g, hot.nb, hot.up, hot.down) for g in genes]
    n_keys = []                                                 # distinct edited rows per gene, chunks counted for genes
    for gi, g in enumerate(genes):
        ks = {key(gi, j, k) for j in range(len(sets[gi])) for k in hits[gi][j]}
        n_keys.append(sum(CW if x[0] else 1 for x in ks))
    rows_per_gene = [len(g.cre_start) + CW + n for g, n in zip(genes, n_keys)]
    for a, b, _, _ in cohort.plan_passes(rows_per_gene, pass_rows):
        c["passes"] += 1
        with phase("stage1"):
            # ---- the baseline items: each gene tokenized once ----
            ctoks, gtoks, labels, glens = [], [], [], []
            for k0 in range(a, b, ism.GENE_GROUP):
                k1 = min(b, k0 + ism.GENE_GROUP)
                t = hot.tokenize(genes[k0:k1], variants)
                knockout._check_stage1(hot, genes[k0:k1], t, variants, [[]] * (k1 - k0), None, names[k0:k1])
                glens += t["gene_seq"][1].cpu().numpy().astype(np.int64).tolist()
                ctoks += t["cre_tok"]; gtoks += t["gene_tok"]; labels += t["labels"]
                del t
            for i, gi in enumerate(range(a, b)):
                if (e := short(glens[i], gi)) is not None:
                    raise e
            # ---- one encode row per distinct key (window, the set's records in it) of the pass ----
            keys = {}                                          # key -> (row index, owner genes)
            c_rows, g_rows = [], []
            for gi in range(a, b):
                for j in range(len(sets[gi])):
                    for k in hits[gi][j]:
                        kk = key(gi, j, k)
                        if kk not in keys:
                            rows = g_rows if kk[0] else c_rows
                            keys[kk] = (len(rows), set())
                            rows.append(kk[1:])
                        keys[kk][1].add(gi)
            c_own = [set() for _ in c_rows]; g_own = [set() for _ in g_rows]
            for kk, (r, own) in keys.items():
                (g_own if kk[0] else c_own)[r] |= own
            # CRE windows: the per-item path's pitch is its gene's longest CRE span + 4096 (WindowTokenizer.sequences)
            c_pitch = {gi: knockout._pitch(max(w1 - w0 for _, w0, w1 in win[gi][:-1])) for gi in range(a, b)}
            cand_c, c_len, c_app = [torch.cat(ctoks)], [], []
            for r0 in range(0, len(c_rows), CRE_EDIT_ROWS):
                rows = c_rows[r0:r0 + CRE_EDIT_ROWS]
                pitch = max(c_pitch[gi] for o in c_own[r0:r0 + CRE_EDIT_ROWS] for gi in o)
                seq, lens, app, err = encode(hot, variants, rows, pitch)
                if int(err.item()):
                    _raise(int(err.item()), names[min(c_own[r0])])
                tok, _, _ = hot.tok.tokenize_fixed(seq, lens, seq.shape[1], typical_len=max(r[2] - r[1] for r in rows))
                cand_c.append(tok.to(cand_c[0].dtype))
                c_len.append(lens.cpu().numpy().astype(np.int64)); c_app.append(app.cpu().numpy().astype(bool))
                del seq, tok
            c_len = np.concatenate(c_len) if c_len else np.zeros(0, np.int64)
            c_app = np.concatenate(c_app) if c_app else np.zeros(0, bool)
            # gene windows: full BPE, 200-token chunks
            cand_g, g_chunks, g_len, g_app = [torch.cat(gtoks)], [], [], []
            cap = L * CW
            for r0 in range(0, len(g_rows), ism.GENE_GROUP):
                rows = g_rows[r0:r0 + ism.GENE_GROUP]
                pitch = knockout._pitch(max(r[2] - r[1] for r in rows))
                seq, lens, app, err = encode(hot, variants, rows, pitch)
                if int(err.item()):
                    _raise(int(err.item()), names[min(g_own[r0])])
                tok, cnt = ops.bpe_tokenize(seq, lens, seq.shape[1], hot.tok.merges, cap, cap)
                del seq
                G_m = np.minimum(CW, (cnt.cpu().numpy().astype(np.int64) + L - 1) // L)
                tok = tok.view(len(rows), CW, L)
                for j in range(len(rows)):
                    cand_g.append(tok[j, :G_m[j]])
                g_chunks += G_m.tolist()
                g_len.append(lens.cpu().numpy().astype(np.int64)); g_app.append(app.cpu().numpy().astype(bool))
                del tok
            g_len = np.concatenate(g_len) if g_len else np.zeros(0, np.int64)
            g_app = np.concatenate(g_app) if g_app else np.zeros(0, bool)
            # errors the per-item path raises for an item (the gene alone with the set added)
            for own, n in zip(c_own, c_len):
                for gi in sorted(own):
                    if n > c_pitch[gi]:
                        _raise(1, names[gi])
            for row, own, n in zip(g_rows, g_own, g_len):
                for gi in sorted(own):
                    if n > knockout._pitch(row[2] - row[1]):
                        _raise(1, names[gi])
                    if (e := short(n, gi)) is not None:
                        raise e
            # ---- every distinct token row once ----
            uc, inv_c = torch.unique(torch.cat(cand_c), dim=0, return_inverse=True)
            ug, inv_g = torch.unique(torch.cat(cand_g), dim=0, return_inverse=True)
            del cand_c, cand_g
            inv_c = inv_c.cpu().numpy().astype(np.int64); inv_g = inv_g.cpu().numpy().astype(np.int64)
            n_cb = sum(x.shape[0] for x in ctoks); n_gb = sum(x.shape[0] for x in gtoks)
            g_start = n_gb + np.concatenate([[0], np.cumsum(g_chunks)]).astype(np.int64)
            a_off = {False: np.concatenate([[0], np.cumsum([len(r[4]) for r in c_rows])]).astype(np.int64),
                     True: np.concatenate([[0], np.cumsum([len(r[4]) for r in g_rows])]).astype(np.int64)}
            # ---- items: per gene its baseline, then one per set ----
            items = []
            c0 = g0_ = 0
            for i, gi in enumerate(range(a, b)):
                C, G = ctoks[i].shape[0], gtoks[i].shape[0]
                cr, gr, lab = inv_c[c0:c0 + C], inv_g[g0_:g0_ + G], labels[i].numpy().astype(np.int64)
                c0 += C; g0_ += G
                tis = torch.as_tensor(genes[gi].tissues, dtype=torch.long)
                items.append((cr, gr, tis, lab))
                ap = applied[gi]
                for j in range(len(sets[gi])):
                    r, grow = cr.copy(), gr
                    for k, ms in hits[gi][j].items():
                        kk = key(gi, j, k)
                        row = keys[kk][0]
                        if kk[0]:
                            grow = inv_g[g_start[row]:g_start[row + 1]]
                        else:
                            r[k] = inv_c[n_cb + row]
                        if changed_by_tokens:
                            ch = not np.array_equal(grow, gr) if kk[0] else bool(r[k] != cr[k])
                            flags = np.full(len(ms), ch)
                        else:
                            flags = (g_app if kk[0] else c_app)[a_off[kk[0]][row]:a_off[kk[0]][row + 1]]
                        ap["records"][j][ms] |= flags
                        if kk[0]:
                            ap["gene"][j] = flags.any()
                        else:
                            ap["cre"][j, k] = flags.any()
                    items.append((r, grow, tis, lab))
                n_set = len(sets[gi])
                c["windows_per_item"] += (1 + n_set) * (C + 1)
                c["changed"] += int((ap["cre"].any(1) | ap["gene"]).sum())
            del ctoks, gtoks
            c["items"] += len(items)
            c["cre_windows_edited"] += len(c_rows); c["gene_windows_edited"] += len(g_rows)
            c["windows_encoded"] += sum(len(genes[gi].cre_start) + 1 for gi in range(a, b)) + len(c_rows) + len(g_rows)
            c["cre_token_rows"] += int(uc.shape[0]); c["gene_token_rows"] += int(ug.shape[0])
        with phase("seq2reg"):
            cre_pooled = ism._pool(eng, eng.cre_tok, uc.to(torch.int32))
            gene_pooled = ism._pool(eng, eng.gene_tok, ug.to(torch.int32))
            del uc, ug
        with phase("seq2gene"):
            blocks = knockout.score_items(eng, items, [1 + len(sets[gi]) for gi in range(a, b)], cre_pooled,
                                          gene_pooled, rows_budget, embeddings, c)
            for gi, (p, e) in zip(range(a, b), blocks):
                pred[t_off[gi]:t_off[gi + 1]] = p[0]
                set_pred[gi] = p[1:]
                emb[t_off[gi]:t_off[gi + 1]] = e[0] if embeddings else e
                if embeddings:
                    set_emb[gi] = e[1:]
            del blocks, cre_pooled, gene_pooled
    c["windows_per_item"] = int(c["windows_per_item"])
    out = (pred, emb, set_pred) + ((set_emb,) if embeddings else ())
    if to_host:
        host = lambda x: x.cpu().numpy()
        out = (host(pred), host(emb), [host(x) for x in set_pred]) + (([host(x) for x in set_emb],) if embeddings else ())
    return out + (applied,)


def shared_window(g, sets, nb, up, down):
    """Whether some window of gene g contains the REF spans of two or more of a set's records (sets as check_sets
    returns them): such a set needs a newly encoded window.  -> bool [n]."""
    return np.asarray([any(len(m) > 1 for m in d.values()) for d in set_windows(g, sets, nb, up, down)], bool)


def user_records(df, sets=True):
    """Records from a DataFrame with columns gene_id, chromosome, pos, ref, alt (+ set when `sets`), optionally gt
    (default 2) and label (default "chromosome:pos:ref>alt").  -> {gene_id: [(set label, [Record], [record labels])]}
    (sets in first-appearance order) or, without `sets`, {gene_id: ([Record], [labels])}."""
    need = ["gene_id"] + (["set"] if sets else []) + ["chromosome", "pos", "ref", "alt"]
    missing = [k for k in need if k not in df.columns]
    if missing:
        raise ValueError(f"variants must have the columns {', '.join(need)} (missing: {missing})")
    gts = df["gt"] if "gt" in df.columns else [2] * len(df)
    labels = df["label"] if "label" in df.columns else [None] * len(df)
    sids = df["set"] if sets else [None] * len(df)
    out = {}
    for gid, sid, ch, pos, ref, alt, gt, lab in zip(df["gene_id"], sids, df["chromosome"], df["pos"], df["ref"],
                                                     df["alt"], gts, labels):
        for what, x in (("pos", pos), ("gt", gt)):
            if isinstance(x, (bool, np.bool_)) or not isinstance(x, (int, np.integer)):
                raise ValueError(f"variant {ch}:{pos} of gene {gid}: {what} {x!r} is not an integer")
        r = Record(str(ch), int(pos), str(ref), str(alt), int(gt))
        lab = _label(r) if lab is None or (not isinstance(lab, str) and pd.isna(lab)) else lab
        if sets:
            d = out.setdefault(gid, {})
            s = d.setdefault(sid, ([], []))
            s[0].append(r); s[1].append(lab)
        else:
            d = out.setdefault(gid, ([], []))
            d[0].append(r); d[1].append(lab)
    if sets:
        return {g: [(sid, rs, ls) for sid, (rs, ls) in d.items()] for g, d in out.items()}
    return out


SET_COLUMNS = ["gene_id", "tissue", "set", "n_records", "records_applied", "cre_windows_changed", "gene_window_changed",
               "changed", "baseline_expression", "predicted_expression", "delta"]


def set_frame(gene_id, tissues, labels, n_records, applied, base_pred, set_pred):
    """One query row's sets in long format: one row per (set, tissue), in that order.  labels / n_records: per set;
    applied: dict(cre=bool [n, C], gene=bool [n], records=per set bool arrays); base_pred fp32 [T]; set_pred fp32 [n, T]."""
    T, n = len(tissues), len(labels)
    base = np.asarray(base_pred, np.float32).reshape(T)
    sp = np.asarray(set_pred, np.float32).reshape(n, T)
    rep = lambda xs: np.repeat(np.asarray(xs, np.int64 if not isinstance(xs, np.ndarray) else xs.dtype), T)
    n_cre = applied["cre"].sum(1).astype(np.int64)
    gene = applied["gene"].astype(bool)
    return pd.DataFrame({
        "gene_id": [gene_id] * (n * T), "tissue": list(tissues) * n, "set": [x for x in labels for _ in range(T)],
        "n_records": rep(np.asarray(n_records, np.int64)),
        "records_applied": rep(np.asarray([int(np.sum(r)) for r in applied["records"]], np.int64)),
        "cre_windows_changed": rep(n_cre), "gene_window_changed": rep(gene), "changed": rep((n_cre > 0) | gene),
        "baseline_expression": np.tile(base, n), "predicted_expression": sp.reshape(-1),
        "delta": (sp - base[None, :]).reshape(-1)}, columns=SET_COLUMNS)


SUMMARY_COLUMNS = ["gene_id", "set", "tissue", "n_samples", "n_changed", "mean_delta", "sd_delta", "min_delta",
                   "max_delta"]


def cohort_summary(frame):
    """The background dependence of each set across a cohort: one row per (gene_id, set, tissue) of a frame of
    VCFProcessor.cohort_variant_sets (columns sample + SET_COLUMNS), in first-appearance order.  n_samples, n_changed
    (samples whose windows the set changed), and the mean, standard deviation (ddof 0), minimum and maximum of delta
    over the samples, in float64."""
    keys = ["gene_id", "set", "tissue"]
    d = frame.assign(delta=frame["delta"].astype(np.float64))
    g = d.groupby(keys, sort=False)
    out = pd.DataFrame({"n_samples": g["sample"].size(), "n_changed": g["changed"].sum().astype(np.int64),
                        "mean_delta": g["delta"].mean(), "sd_delta": g["delta"].std(ddof=0),
                        "min_delta": g["delta"].min(), "max_delta": g["delta"].max()}).reset_index()
    return out[SUMMARY_COLUMNS]


INTERACTION_COLUMNS = ["gene_id", "tissue", "variant_a", "variant_b", "same_window", "baseline_expression",
                       "expression_a", "expression_b", "expression_ab", "delta_a", "delta_b", "delta_ab", "interaction",
                       "log2_interaction"]


def interaction_frame(gene_id, tissues, labels, pair_idx, same_window, base_pred, single_pred, pair_pred):
    """One query row's pair scan in long format: one row per (pair, tissue), in that order.  labels: per record;
    pair_idx [(i, j)]; same_window bool per pair; base_pred fp32 [T]; single_pred fp32 [N, T]; pair_pred fp32 [P, T].
    interaction = delta_ab - delta_a - delta_b; log2_interaction = log2((ab + 1e-10)(base + 1e-10) / ((a + 1e-10)
    (b + 1e-10))), the 1e-10 convention of saturation mutagenesis' log2fc."""
    T, P = len(tissues), len(pair_idx)
    base = np.asarray(base_pred, np.float32).reshape(1, T)
    sp = np.asarray(single_pred, np.float32).reshape(-1, T)
    ab = np.asarray(pair_pred, np.float32).reshape(P, T)
    ia = np.asarray([i for i, _ in pair_idx], np.int64); ib = np.asarray([j for _, j in pair_idx], np.int64)
    ea, eb = sp[ia].reshape(P, T), sp[ib].reshape(P, T)
    da, db, dab = ea - base, eb - base, ab - base
    eps = 1e-10
    l2 = (np.log2(ab.astype(np.float64) + eps) + np.log2(base.astype(np.float64) + eps)
          - np.log2(ea.astype(np.float64) + eps) - np.log2(eb.astype(np.float64) + eps))
    rep = lambda xs: [x for x in xs for _ in range(T)]
    return pd.DataFrame({
        "gene_id": [gene_id] * (P * T), "tissue": list(tissues) * P, "variant_a": rep([labels[i] for i in ia]),
        "variant_b": rep([labels[j] for j in ib]), "same_window": np.repeat(np.asarray(same_window, bool).reshape(P), T),
        "baseline_expression": np.tile(base[0], P), "expression_a": ea.reshape(-1), "expression_b": eb.reshape(-1),
        "expression_ab": ab.reshape(-1), "delta_a": da.reshape(-1), "delta_b": db.reshape(-1),
        "delta_ab": dab.reshape(-1), "interaction": (dab - da - db).reshape(-1), "log2_interaction": l2.reshape(-1)},
        columns=INTERACTION_COLUMNS)
