"""Variant sets across a cohort: every sample of a multi-sample VCF predicted with each set of records added.

The result of set j for gene g and sample s is BY DEFINITION what HotPath.variant_sets([g], [[set j]], that sample's
SampleVariants) gives (DESIGN section 18): prediction, embedding and applied flags, with section 17's rules unchanged (a
set's records go after the sample's records of the same POS, and a record the sample's own records block is not
applied).  The baseline of sample s is HotPath.predict_cohort's row s.  What is not recomputed:
  * rows are (window, sample) for the baseline windows (cohort.gene_windows) and (window, sample, a set's records in that
    window) for the edited ones, one per distinct (window, restricted records) key (variant_sets.set_windows) times the
    samples.  Both kinds of a window share one grouping (cohort.group_rows over vf_window_genotype_keys_edits, confirmed
    by vf_window_genotype_equal_edits): rows with equal applied lists are one group, so an edit that is blocked in a
    sample, or that leaves two samples with equal windows, is never encoded again;
  * only group representatives are encoded (vf_encode_windows_edits), every distinct token row goes through seq2reg once
    (ism._pool), and equal items (a sample's baseline or a set, as token rows + tissues + labels) are scored once
    (cohort.dedup_items) in slabs of at most ism.ROWS_BUDGET CRE rows and cohort.plan_passes passes bounded per sample.
Stage-1 errors and the gene-window length rule come from the keys before anything is encoded: the first sample (in
cohort order) with one raises what its own variant_sets call raises, with the sample's name.
"""
import contextlib

import numpy as np
import pandas as pd
import torch

from . import cohort, ism, knockout, ops, variant_sets
from .knockout import _pitch


class _Rows:
    """Genotype keys and groups of one window table: rows (window, sample) then (edit, sample), edits = [(window, the
    records applied on top of the sample: (chrom, pos0, ref_len, alt bytes, gt) sorted by POS)]."""

    def __init__(self, hot, cv, wins, edits, samples, key_bits):
        dev = hot.engine.device
        S, W, E = len(samples), len(wins), len(edits)
        self.S, self.W, self.E = S, W, E
        chrom = np.asarray([w[0] for w in wins], dtype=object)
        self.base = np.asarray([hot.genome.offsets[c][0] for c in chrom], np.int64)
        self.w0 = np.asarray([w[1] for w in wins], np.int64); self.w1 = np.asarray([w[2] for w in wins], np.int64)
        self.flags = np.asarray([w[3] for w in wins], np.uint8)
        self.max_window = int((self.w1 - self.w0).max()) if W else 0
        self.pitch = _pitch(self.max_window)                 # no row gets here past its own (smaller) pitch
        ew = np.asarray([e[0] for e in edits], np.int64)
        self.row_w = np.concatenate([np.repeat(np.arange(W), S), np.repeat(ew, S)]).astype(np.int64)
        row_s = np.concatenate([np.tile(np.arange(S), W), np.tile(np.arange(S), E)]).astype(np.int64)
        row_e = np.concatenate([np.full(W * S, -1), np.repeat(np.arange(E), S)]).astype(np.int64)
        self.lo, self.hi = cv.window_ranges(np.asarray(samples, np.int64)[row_s], chrom[self.row_w],
                                            self.w0[self.row_w], self.w1[self.row_w])
        # the distinct records, once each; a row's extras index them (CSR)
        recs = [r for e in edits for r in e[1]]
        n_rec = np.asarray([len(e[1]) for e in edits], np.int64)
        first = np.concatenate([[0], np.cumsum(n_rec)]).astype(np.int64)
        self.rec_pos = np.asarray([r[1] for r in recs], np.int32)
        self.rec_rl = np.asarray([r[2] for r in recs], np.int32)
        self.rec_al = np.asarray([len(r[3]) for r in recs], np.int32)
        self.rec_gt = np.asarray([r[4] for r in recs], np.uint8)
        self.rec_ao = (np.cumsum(self.rec_al, dtype=np.int64) - self.rec_al).astype(np.int32)
        self.pool = torch.from_numpy(np.frombuffer(b"".join(r[3] for r in recs), np.uint8).copy()).to(dev)
        row_n = np.where(row_e >= 0, n_rec[np.maximum(row_e, 0)] if E else 0, 0)
        self.e_off = np.concatenate([[0], np.cumsum(row_n)]).astype(np.int64)
        owner = np.repeat(np.arange(len(row_n)), row_n)
        self.slot_rec = first[row_e[owner]] + np.arange(int(self.e_off[-1])) - self.e_off[owner]
        self.vdev = cv.dev
        rows = np.arange(len(self.row_w))
        args = self._args(dev, rows)
        keys, count, lens, applied, _ = ops.window_genotype_keys_edits(*args, key_bits=key_bits)
        group, rep = cohort.group_rows(torch.from_numpy(self.row_w), count, keys,
                                       lambda r: ops.window_genotype_equal_edits(*args, r.to(torch.int32)) != 0)
        self.group, self.rep = group.cpu().numpy(), rep.cpu().numpy()
        self.count, self.lens = count.cpu().numpy(), lens.cpu().numpy().astype(np.int64)
        self.applied = applied.cpu().numpy().astype(bool)

    def _args(self, dev, rows):
        """Row and CSR extra-record arguments of vf_window_genotype_keys_edits / vf_encode_windows_edits for `rows`."""
        up = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dt)).to(dev)
        w = self.row_w[rows]
        n = self.e_off[rows + 1] - self.e_off[rows]
        off = np.concatenate([[0], np.cumsum(n)]).astype(np.int64)
        own = np.repeat(np.arange(len(rows)), n)
        rec = self.slot_rec[self.e_off[rows][own] + np.arange(int(off[-1])) - off[own]] if len(own) else \
            np.zeros(0, np.int64)
        return (up(self.w0[w], np.int32), up(self.w1[w], np.int32), up(self.lo[rows], np.int32),
                up(self.hi[rows], np.int32), up(self.flags[w], np.uint8), self.vdev, up(off, np.int32),
                up(self.rec_pos[rec], np.int32), up(self.rec_rl[rec], np.int32), up(self.rec_ao[rec], np.int32),
                up(self.rec_al[rec], np.int32), up(self.rec_gt[rec], np.uint8), self.pool)

    def base_row(self, w, s):
        return w * self.S + s

    def edit_row(self, e, s):
        return (self.W + e) * self.S + s

    def flags_of(self, row):
        """The applied flag of each extra record of `row`."""
        return self.applied[self.e_off[row]:self.e_off[row + 1]]

    def encode(self, hot, groups):
        """Encoded bytes of the representatives of `groups` -> (uint8 [n, pitch], int32 lens) on the device."""
        dev = hot.engine.device
        r = self.rep[groups]
        w = self.row_w[r]
        a = self._args(dev, r)
        out, lens, _, _ = ops.encode_windows_edits(hot.genome.seq, torch.from_numpy(self.base[w]).to(dev), *a[:6],
                                                   *a[6:], max(1, self.max_window), self.pitch)
        return out, lens


def _per_sample_error(hot, genes, sets, wins, ct, gt, edit_of, s, min_gene_len, pass_rows, names):
    """The exception HotPath.variant_sets(genes, sets, sample s) raises, restated from the keys' counts and lengths in
    the order that call meets them (variant_sets.plan: per pass the baselines GENE_GROUP genes at a time, then the
    edited CRE rows in CRE_EDIT_ROWS chunks and gene rows in GENE_GROUP chunks, then each item's own pitch).  None if
    it raises nothing."""
    CW = hot.max_chunks
    span = lambda t, w: int(t.w1[w] - t.w0[w])
    c_pitch = [_pitch(max(span(ct, w) for w in wins.cre_of[gi])) for gi in range(len(genes))]

    def code(t, rows, pitch):
        return max([2 if t.count[r] < 0 else 1 if t.lens[r] > pitch else 0 for r in rows] + [0])

    def edited(c, gi):                                   # variant_sets' own message for an edited window
        try:
            variant_sets._raise(c, names[gi])
        except RuntimeError as e:
            return e

    short = lambda n, gi: ValueError(f"Mutated sequence is less than {min_gene_len}bp for gene {names[gi]}") if \
        min_gene_len is not None and n <= min_gene_len else None
    n_keys = [sum(CW if tab == "g" else 1 for tab, _ in {(tab, e) for j in range(len(sets[gi]))
                                                         for _, tab, e, _ in edit_of[gi][j]}) for gi in range(len(genes))]
    rows_per_gene = [len(g.cre_start) + CW + n for g, n in zip(genes, n_keys)]
    for a, b, _, _ in cohort.plan_passes(rows_per_gene, pass_rows if pass_rows is not None else variant_sets.PASS_ROWS):
        for k0 in range(a, b, ism.GENE_GROUP):
            grp = range(k0, min(b, k0 + ism.GENE_GROUP))
            cw = np.concatenate([wins.cre_of[gi] for gi in grp])
            crow = [ct.base_row(w, s) for w in cw]
            grow = [gt.base_row(wins.gene_of[gi], s) for gi in grp]
            c = max(code(ct, crow, _pitch(max(span(ct, w) for w in cw))),
                    code(gt, grow, _pitch(max(span(gt, wins.gene_of[gi]) for gi in grp))))
            if c:
                return RuntimeError(f"stage-1 kernel reported error {c} (1: pitch overflow, 2: >2048 variants/window)")
            for gi in grp:
                lens = [ct.lens[ct.base_row(w, s)] for w in wins.cre_of[gi]]
                w = wins.gene_of[gi]
                if gt.lens[gt.base_row(w, s)] > _pitch(span(gt, w)) or max(lens) > c_pitch[gi]:
                    return RuntimeError(f"stage-1 kernel reported error 1 for gene {names[gi]} (1: pitch overflow, 2: "
                                        ">2048 variants/window)")
        for gi in range(a, b):
            if (e := short(gt.lens[gt.base_row(wins.gene_of[gi], s)], gi)) is not None:
                return e
        keys = {}                                            # (table, edit) -> owner genes, in the planner's row order
        for gi in range(a, b):
            for j in range(len(sets[gi])):
                for _, tab, e, _ in edit_of[gi][j]:
                    keys.setdefault((tab, e), set()).add(gi)
        c_rows = [(e, own) for (tab, e), own in keys.items() if tab == "c"]
        g_rows = [(e, own) for (tab, e), own in keys.items() if tab == "g"]
        for r0 in range(0, len(c_rows), variant_sets.CRE_EDIT_ROWS):
            chunk = c_rows[r0:r0 + variant_sets.CRE_EDIT_ROWS]
            pitch = max(c_pitch[gi] for _, own in chunk for gi in own)
            if (c := code(ct, [ct.edit_row(e, s) for e, _ in chunk], pitch)):
                return edited(c, min(chunk[0][1]))
        for r0 in range(0, len(g_rows), ism.GENE_GROUP):
            chunk = g_rows[r0:r0 + ism.GENE_GROUP]
            pitch = _pitch(max(span(gt, gt.row_w[gt.edit_row(e, s)]) for e, _ in chunk))
            if (c := code(gt, [gt.edit_row(e, s) for e, _ in chunk], pitch)):
                return edited(c, min(chunk[0][1]))
        for e, own in c_rows:
            for gi in sorted(own):
                if ct.lens[ct.edit_row(e, s)] > c_pitch[gi]:
                    return edited(1, gi)
        for e, own in g_rows:
            r = gt.edit_row(e, s)
            for gi in sorted(own):
                if gt.lens[r] > _pitch(span(gt, gt.row_w[r])):
                    return edited(1, gi)
                if (x := short(gt.lens[r], gi)) is not None:
                    return x
    return None


def _check(hot, genes, sets, wins, ct, gt, edit_of, samples, cv, min_gene_len, pass_rows, names):
    """Raise, before anything is encoded, what the first sample (in cohort order) with a stage-1 error or a short gene
    window raises in its own variant_sets call, with the sample's name."""
    S = len(samples)
    bad = np.zeros(S, bool)
    c_pitch = np.asarray([_pitch(max(ct.w1[w] - ct.w0[w] for w in wins.cre_of[gi])) for gi in range(len(genes))])
    lim_c = np.full(ct.W, np.iinfo(np.int64).max)           # a CRE window's smallest pitch over its genes
    for gi in range(len(genes)):
        np.minimum.at(lim_c, wins.cre_of[gi], c_pitch[gi])
    row_s = lambda t: np.concatenate([np.tile(np.arange(S), t.W), np.tile(np.arange(S), t.E)])
    for t, lim in ((ct, lim_c), (gt, np.asarray([_pitch(x) for x in gt.w1 - gt.w0], np.int64))):
        b = (t.count < 0) | (t.lens > lim[t.row_w])
        if t is gt and min_gene_len is not None:
            b |= t.lens <= min_gene_len
        bad[row_s(t)[b]] = True
    for s in np.flatnonzero(bad):
        e = _per_sample_error(hot, genes, sets, wins, ct, gt, edit_of, int(s), min_gene_len, pass_rows, names)
        if e is not None:
            raise type(e)(f"sample {cv.names[samples[s]]}: {e}")


@torch.no_grad()
def scan(hot, genes, sets, cohort_variants, sample_idx=None, embeddings=False, to_host=True,
         rows_budget=ism.ROWS_BUDGET, pass_rows=None, key_bits=128, timer=None, counters=None, min_gene_len=None,
         gene_names=None):
    """Every record set of `genes` (GeneSpec list) in every sample `sample_idx` (default: all) of `cohort_variants`
    (stage1.CohortVariants) on HotPath `hot`.  sets: per gene a list of sets, each a list of variant_sets.Record.
    -> (pred fp32 [S, sum T], emb fp32 [S, sum T, D]: the baselines, bit-identical to HotPath.predict_cohort;
    set_pred: per gene fp32 [S, n_g, T_g][, set_emb: per gene fp32 [S, n_g, T_g, D] when `embeddings`]; applied: per
    gene dict(cre=bool [S, n_g, C_g] (CRE windows in batch order), gene=bool [S, n_g], records=per set bool [S, len])),
    numpy (to_host) or device tensors (applied is numpy either way).  Sample s's entries are bit-identical to
    HotPath.variant_sets(genes, sets, that sample's SampleVariants).  timer: optional callable(phase) -> context manager
    around the "stage1", "keys", "seq2reg" and "seq2gene" phases; counters: optional dict of sample / set / item /
    window counts; key_bits < 128 truncates the genotype keys (tests: forced collisions); min_gene_len: VCFDataset's
    gene-window length rule (gene_names name the genes); pass_rows also sets the per-sample call whose errors are
    restated."""
    names = gene_names if gene_names is not None else [f"{g.chrom}:{g.start}-{g.end}" for g in genes]
    checked = variant_sets.check_sets(genes, sets, hot.genome, names)
    eng, dev = hot.engine, hot.engine.device
    phase = timer or (lambda name: contextlib.nullcontext())
    samples = list(range(len(cohort_variants.names))) if sample_idx is None else [int(s) for s in sample_idx]
    S, CW = len(samples), hot.max_chunks
    T = np.asarray([len(g.tissues) for g in genes], np.int64)
    t_off = np.concatenate([[0], np.cumsum(T)])
    D = eng.w.D
    pred = torch.empty((S, int(t_off[-1])), dtype=torch.float32, device=dev)
    emb = torch.empty((S, int(t_off[-1]), D), dtype=torch.float32, device=dev)
    set_pred = [torch.empty((S, len(s), len(g.tissues)), dtype=torch.float32, device=dev) for g, s in zip(genes, checked)]
    set_emb = [torch.empty((S, len(s), len(g.tissues), D), dtype=torch.float32, device=dev) if embeddings else None
               for g, s in zip(genes, checked)]
    applied = [dict(cre=np.zeros((S, len(s), len(g.cre_start)), bool), gene=np.zeros((S, len(s)), bool),
                    records=[np.zeros((S, len(x)), bool) for x in s]) for g, s in zip(genes, checked)]
    c = counters if counters is not None else {}
    c.update(samples=S, genes=len(genes), sets=sum(len(s) for s in checked), changed=0, items=0, items_scored=0,
             sample_windows=0, windows_encoded=0, cre_groups=0, gene_groups=0, edited_groups=0, cre_token_rows=0,
             gene_token_rows=0, token_rows=0, passes=0, slabs=0)

    def host():
        h = lambda x: x.cpu().numpy()
        out = (h(pred), h(emb), [h(x) for x in set_pred]) + (([h(x) for x in set_emb],) if embeddings else ())
        return out + (applied,)
    if not genes or not S:
        return host() if to_host else (pred, emb, set_pred) + ((set_emb,) if embeddings else ()) + (applied,)
    wins = cohort.gene_windows(genes, hot.nb, hot.up, hot.down)
    hits = [variant_sets.set_windows(g, s, hot.nb, hot.up, hot.down) for g, s in zip(genes, checked)]
    # one edit per distinct (table window, the set's records in it); edit_of[g][j] = [(k, table, edit, record positions)]
    edits = {"c": {}, "g": {}}
    edit_of = []
    for gi, g in enumerate(genes):
        C = len(g.cre_start)
        per = []
        for j, s in enumerate(checked[gi]):
            lst = []
            for k, ms in hits[gi][j].items():
                tab, w = ("g", int(wins.gene_of[gi])) if k == C else ("c", int(wins.cre_of[gi][k]))
                key = (w, tuple(s[m] for m in ms))
                lst.append((k, tab, edits[tab].setdefault(key, len(edits[tab])), ms))
            per.append(lst)
        edit_of.append(per)
    with phase("stage1"), phase("keys"):
        ct = _Rows(hot, cohort_variants, wins.cre, list(edits["c"]), samples, key_bits)
        gt = _Rows(hot, cohort_variants, wins.gene, list(edits["g"]), samples, key_bits)
    tab = {"c": ct, "g": gt}
    _check(hot, genes, checked, wins, ct, gt, edit_of, samples, cohort_variants, min_gene_len, pass_rows, names)
    # ---- applied flags of every (sample, set), from the keys kernel ----
    for gi, g in enumerate(genes):
        ap = applied[gi]
        for j in range(len(checked[gi])):
            for k, tb, e, ms in edit_of[gi][j]:
                t = tab[tb]
                fl = np.stack([t.flags_of(t.edit_row(e, s)) for s in range(S)])      # [S, len(ms)]
                ap["records"][j][:, ms] |= fl
                if tb == "g":
                    ap["gene"][:, j] = fl.any(1)
                else:
                    ap["cre"][:, j, k] = fl.any(1)
        c["changed"] += int((ap["cre"].any(2) | ap["gene"]).sum())
    c["sample_windows"] = int(S * (sum(len(x) for x in wins.cre_of) + len(genes)))
    # ---- passes: about pass_rows token rows each, a gene too large for one pass split by samples ----
    cg_base = ct.group[:ct.W * S].reshape(ct.W, S); gg_base = gt.group[:gt.W * S].reshape(gt.W, S)
    cg_edit = ct.group[ct.W * S:].reshape(ct.E, S); gg_edit = gt.group[gt.W * S:].reshape(gt.E, S)
    g_edits = [sorted({(tb, e) for j in range(len(checked[gi])) for _, tb, e, _ in edit_of[gi][j]})
               for gi in range(len(genes))]

    def groups_of(gi, s0, s1):
        ce = [e for tb, e in g_edits[gi] if tb == "c"]; ge = [e for tb, e in g_edits[gi] if tb == "g"]
        return (np.concatenate([cg_base[wins.cre_of[gi], s0:s1].ravel(), cg_edit[ce, s0:s1].ravel()]),
                np.concatenate([gg_base[[wins.gene_of[gi]], s0:s1].ravel(), gg_edit[ge, s0:s1].ravel()]))
    rows_per_gene = []
    for gi in range(len(genes)):
        cgs, ggs = groups_of(gi, 0, S)
        rows_per_gene.append(len(np.unique(cgs)) + CW * len(np.unique(ggs)))
    sample_rows = [len(g.cre_start) + CW + sum(CW if tb == "g" else 1 for tb, _ in g_edits[gi])
                   for gi, g in enumerate(genes)]
    pass_rows_ = cohort.PASS_ROWS if pass_rows is None else pass_rows
    for a, b, s0, s1 in cohort.plan_passes(rows_per_gene, pass_rows_, S, sample_rows):
        c["passes"] += 1
        with phase("stage1"):
            parts = [groups_of(gi, s0, s1) for gi in range(a, b)]
            c_groups = np.unique(np.concatenate([p[0] for p in parts]))
            g_groups = np.unique(np.concatenate([p[1] for p in parts]))
            c["cre_groups"] += len(c_groups); c["gene_groups"] += len(g_groups)
            c["windows_encoded"] += len(c_groups) + len(g_groups)
            c["edited_groups"] += int((ct.rep[c_groups] >= ct.W * S).sum() + (gt.rep[g_groups] >= gt.W * S).sum())
            # CRE representatives: fixed 200-token rows, CRE_EDIT_ROWS windows at a time
            ctoks = []
            for k in range(0, len(c_groups), variant_sets.CRE_EDIT_ROWS):
                seq, lens = ct.encode(hot, c_groups[k:k + variant_sets.CRE_EDIT_ROWS])
                ctoks.append(hot.tok.tokenize_fixed(seq, lens, seq.shape[1], typical_len=ct.max_window)[0])
                del seq
            uc, inv_c = torch.unique(torch.cat(ctoks), dim=0, return_inverse=True)
            del ctoks
            row_of_cg = np.full(ct.group.max() + 1, -1, np.int64)
            row_of_cg[c_groups] = inv_c.cpu().numpy()
            # gene representatives: chunked tokens, ism.GENE_GROUP windows at a time
            chunks, n_chunks = [], []
            for k in range(0, len(g_groups), ism.GENE_GROUP):
                seq, lens = gt.encode(hot, g_groups[k:k + ism.GENE_GROUP])
                ch, _ = hot.tok.tokenize_chunked(seq, lens, seq.shape[1])
                del seq
                chunks += [x[0] for x in ch]; n_chunks += [x[0].shape[0] for x in ch]
            ug, inv_g = torch.unique(torch.cat(chunks), dim=0, return_inverse=True)
            inv_g = inv_g.cpu().numpy()
            del chunks
            g_off = np.concatenate([[0], np.cumsum(n_chunks)])
            rows_of_gg = {int(q): inv_g[g_off[k]:g_off[k + 1]] for k, q in enumerate(g_groups)}
            c["cre_token_rows"] += int(uc.shape[0]); c["gene_token_rows"] += int(ug.shape[0])
            c["token_rows"] += int(uc.shape[0] + ug.shape[0])
            # items: per (sample, gene) its baseline, then one per set
            items, where = [], []
            for s in range(s0, s1):
                for gi in range(a, b):
                    tis = tuple(int(t) for t in genes[gi].tissues)
                    cr = row_of_cg[cg_base[wins.cre_of[gi], s]]
                    gr = rows_of_gg[int(gg_base[wins.gene_of[gi], s])]
                    items.append((cr, gr, tis, wins.labels[gi])); where.append((s, gi, -1))
                    for j in range(len(checked[gi])):
                        r, grow = cr.copy(), gr
                        for k, tb, e, _ in edit_of[gi][j]:
                            if tb == "g":
                                grow = rows_of_gg[int(gg_edit[e, s])]
                            else:
                                r[k] = row_of_cg[cg_edit[e, s]]
                        items.append((r, grow, tis, wins.labels[gi])); where.append((s, gi, j))
            uniq, of = cohort.dedup_items(items)
            keep_emb = np.zeros(len(uniq), bool)                # embeddings kept: every item's, or the baselines'
            keep_emb[of[[i for i, w in enumerate(where) if embeddings or w[2] < 0]]] = True
            c["items"] += len(items); c["items_scored"] += len(uniq)
        with phase("seq2reg"):
            cre_pooled = ism._pool(eng, eng.cre_tok, uc)
            gene_pooled = ism._pool(eng, eng.gene_tok, ug)
            del uc, ug
        with phase("seq2gene"):
            u_pred, u_emb = [None] * len(uniq), [None] * len(uniq)
            for x0, x1 in cohort.slab_ranges([len(items[i][0]) for i in uniq], rows_budget):
                c["slabs"] += 1
                sl = [items[i] for i in uniq[x0:x1]]
                used, local = np.unique(np.concatenate([x[1] for x in sl]), return_inverse=True)
                splits = np.cumsum([len(x[1]) for x in sl])[:-1]
                s_ = eng.prepare_shared([x[0] for x in sl], np.split(local, splits), len(used),
                                        [torch.as_tensor(x[2], dtype=torch.long) for x in sl],
                                        [torch.from_numpy(x[3]) for x in sl])
                out = eng.run_pooled(s_, cre_pooled, gene_pooled.index_select(0, torch.from_numpy(used).to(dev)))
                r = 0
                for j, x in zip(range(x0, x1), sl):
                    n = len(x[2])
                    u_pred[j] = out["pred"][r:r + n]
                    if keep_emb[j]:                 # a copy: the slab's other embeddings are freed with `out`
                        u_emb[j] = out["emb"][r:r + n] if embeddings else out["emb"][r:r + n].clone()
                    r += n
                del out
            for i, (s, gi, j) in enumerate(where):
                if j < 0:
                    pred[s, t_off[gi]:t_off[gi + 1]] = u_pred[of[i]].reshape(-1)
                    emb[s, t_off[gi]:t_off[gi + 1]] = u_emb[of[i]]
                else:
                    set_pred[gi][s, j] = u_pred[of[i]].reshape(-1)
                    if embeddings:
                        set_emb[gi][s, j] = u_emb[of[i]]
            del cre_pooled, gene_pooled, u_pred, u_emb
    if to_host:
        return host()
    return (pred, emb, set_pred) + ((set_emb,) if embeddings else ()) + (applied,)

