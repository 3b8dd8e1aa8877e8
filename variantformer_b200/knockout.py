"""In-silico CRE knockout: each gene predicted with one CRE, or a set of CREs, removed from its input.

A knockout of gene g (a GeneSpec, CRE arrays in manifest order) by a set K of manifest rows is BY DEFINITION what
HotPath.predict gives for the same GeneSpec with the rows in K removed (DESIGN section 15): the remaining CREs keep
their batch order (sorted by start, reversed on the minus strand), the 9-class label counts of the CRE-layer
cross-attention lose the removed rows (a class left empty gets logc = -inf), and the gene window is unchanged.  What is
not recomputed:
  * each gene is tokenized once (HotPath.tokenize): a window's bytes and tokens depend on the window alone, so removing
    a CRE changes no other window;
  * every distinct token row (CRE window or 200-token gene chunk) goes through seq2reg once (ism._pool);
  * an item is the gene's list of pooled CRE rows with the knocked-out batch positions left out, its gene chunks, its
    tissues and its labels with the same positions left out.  Items run through Engine.prepare_shared + run_pooled in
    slabs of at most ism.ROWS_BUDGET CRE rows (cohort.slab_ranges; consecutive genes share slabs), in passes of about
    PASS_ROWS token rows (cohort.plan_passes), so device memory stays bounded for any number of genes.  Results depend on
    neither split.
What is left per knockout is one seq2gene forward: removing a row changes every CRE-stack row through self-attention.
"""
import contextlib

import numpy as np
import pandas as pd
import torch

from . import cohort, ism
from .stage1 import cre_window, gene_window

# token rows per pass (CRE windows + max_chunks gene chunks per gene, counted before deduplication)
PASS_ROWS = cohort.PASS_ROWS
# the encoder's room for inserted bases (WindowTokenizer.sequences' max_insert): a window encoded alone, or with any
# other windows, fits its pitch when its encoded length is at most its span plus this
MAX_INSERT = 4096


def batch_order(gene):
    """Manifest row of every batch position (HotPath.tokenize: stable sort by start, reversed on the minus strand)."""
    order = np.argsort(np.asarray(gene.cre_start), kind="stable")
    return order[::-1] if gene.strand == "-" else order


def kept_positions(order, knocked):
    """Batch positions an item keeps when the manifest rows `knocked` are removed, in batch order."""
    pos_of = np.empty(len(order), np.int64)
    pos_of[order] = np.arange(len(order))
    return np.delete(np.arange(len(order)), pos_of[np.asarray(knocked, np.int64)])


def check_knockouts(genes, knockouts=None, gene_names=None, labels=None):
    """Validate the knockout sets of `genes` before any device work.  knockouts: per gene a list of index arrays into its
    CRE arrays (manifest rows), or None for every CRE singly (a gene with one CRE then has no knockout).  gene_names /
    labels (per gene, per set) name them in the messages.
    -> per gene a list of sorted int64 arrays.  ValueError for a gene without CREs, a set that is empty, not integer,
    outside the manifest, repeats an index or removes every CRE, and for a knockouts list of another length."""
    name = lambda i: gene_names[i] if gene_names is not None else f"{genes[i].chrom}:{genes[i].start}-{genes[i].end}"
    if knockouts is not None and len(knockouts) != len(genes):
        raise ValueError(f"knockouts has {len(knockouts)} entries for {len(genes)} genes")
    out = []
    for i, g in enumerate(genes):
        C = len(g.cre_start)
        if C == 0:
            raise ValueError(f"gene {name(i)} has no CRE: a prediction needs at least one")
        if knockouts is None:
            out.append([np.asarray([c], np.int64) for c in range(C)] if C > 1 else [])
            continue
        sets = []
        for j, k in enumerate(knockouts[i]):
            a = np.asarray(k).reshape(-1)
            what = f"knockout {labels[i][j] if labels is not None else j!r} of gene {name(i)}"
            if a.size == 0:
                raise ValueError(f"{what} is empty")
            if not np.issubdtype(a.dtype, np.integer):
                raise ValueError(f"{what} holds non-integer CRE indices ({a.dtype})")
            a = np.sort(a.astype(np.int64))
            if a[0] < 0 or a[-1] >= C:
                raise ValueError(f"{what} holds CRE index {int(a[0] if a[0] < 0 else a[-1])} outside the manifest "
                                 f"(0..{C - 1})")
            if (np.diff(a) == 0).any():
                raise ValueError(f"{what} repeats CRE index {int(a[1:][np.diff(a) == 0][0])}")
            if len(a) == C:
                raise ValueError(f"{what} removes every CRE of the gene")
            sets.append(a)
        out.append(sets)
    return out


def _pitch(span):
    return (int(span) + MAX_INSERT + 15) // 16 * 16


def overflows(spans, lens):
    """Whether the per-item path's encoder overflows its pitch (stage-1 error 1) for a set of windows encoded together:
    spans / lens = reference spans and encoded lengths (numpy)."""
    return len(spans) > 0 and int(np.max(lens)) > _pitch(np.max(spans))


def _check_stage1(hot, genes, t, variants, sets, min_gene_len, names):
    """The errors HotPath.predict raises for each gene's items (the gene alone with its knockout applied), known from
    the encoded lengths of one tokenization of all of them."""
    code = int(t["err"].item())
    if code:                     # a window the encoder could not build with the slab's pitch fails alone as well
        raise RuntimeError(f"stage-1 kernel reported error {code} (1: pitch overflow, 2: >2048 variants/window)")
    clen = t["cre_seq"][1].cpu().numpy().astype(np.int64)
    glen = t["gene_seq"][1].cpu().numpy().astype(np.int64)
    c0 = 0
    for i, g in enumerate(genes):
        order = batch_order(g)
        C = len(order)
        lens = clen[c0:c0 + C]; c0 += C
        g0, g1 = gene_window(g.start, g.end, g.strand, hot.up, hot.down)
        if min_gene_len is not None and glen[i] <= min_gene_len:
            raise AssertionError(f"Mutated sequence is less than {min_gene_len}bp for gene {names[i]}")
        if variants is None:     # reference bytes: every window is exactly its span long
            continue
        spans = np.asarray([w1 - w0 for w0, w1 in (cre_window(g.cre_start[r], g.cre_end[r], hot.nb) for r in order)])
        bad = glen[i] > _pitch(g1 - g0) or overflows(spans, lens)
        if not bad and (lens > spans + MAX_INSERT).any():      # only such a window can pass a smaller item's pitch
            bad = any(overflows(spans[k], lens[k]) for k in (kept_positions(order, s) for s in sets[i]))
        if bad:
            raise RuntimeError(f"stage-1 kernel reported error 1 for gene {names[i]} (1: pitch overflow, 2: >2048 "
                               "variants/window)")


def score_items(eng, items, runs, cre_pooled, gene_pooled, rows_budget, embeddings, counters):
    """Items (pooled CRE rows, gene rows, tissues, labels), gene-major with each gene's run of runs[g] items led by its
    baseline, through Engine.prepare_shared + run_pooled in slabs of at most rows_budget CRE rows (cohort.slab_ranges).
    -> per gene (pred fp32 [runs[g], T], emb fp32 [runs[g], T, D], or without `embeddings` the baseline's [T, D] only),
    device tensors.  counters["slabs"] counts the slabs."""
    dev = gene_pooled.device
    base = np.zeros(len(items), bool)                       # the baseline item of each gene leads its run
    base[np.cumsum([0] + list(runs[:-1]))] = True
    n_rows = np.asarray([len(x[2]) for x in items], np.int64)
    preds, embs = [], []
    for x0, x1 in cohort.slab_ranges([len(x[0]) for x in items], rows_budget):
        counters["slabs"] += 1
        sl = items[x0:x1]
        used, local = np.unique(np.concatenate([x[1] for x in sl]), return_inverse=True)
        splits = np.cumsum([len(x[1]) for x in sl])[:-1]
        s = eng.prepare_shared([x[0] for x in sl], np.split(local, splits), len(used), [x[2] for x in sl],
                               [torch.from_numpy(x[3]) for x in sl])
        out = eng.run_pooled(s, cre_pooled, gene_pooled.index_select(0, torch.from_numpy(used).to(dev)))
        preds.append(out["pred"])
        if embeddings:
            embs.append(out["emb"])
        else:                                               # only the baselines' embeddings are returned
            r0 = np.concatenate([[0], np.cumsum(n_rows[x0:x1])])
            rows = [np.arange(r0[j], r0[j + 1]) for j in range(x1 - x0) if base[x0 + j]]
            if rows:
                embs.append(out["emb"].index_select(0, torch.from_numpy(np.concatenate(rows)).to(dev)))
    P = torch.cat(preds)
    E = torch.cat(embs)
    out, r, e = [], 0, 0
    for k, x in zip(runs, np.flatnonzero(base)):
        Tg = int(n_rows[x])
        if embeddings:
            out.append((P[r:r + k * Tg].view(k, Tg), E[r:r + k * Tg].view(k, Tg, -1)))
        else:
            out.append((P[r:r + k * Tg].view(k, Tg), E[e:e + Tg]))
            e += Tg
        r += k * Tg
    return out


@torch.no_grad()
def cre_knockout(hot, genes, knockouts=None, variants=None, embeddings=False, to_host=True, rows_budget=ism.ROWS_BUDGET,
                 pass_rows=None, timer=None, counters=None, min_gene_len=None, gene_names=None):
    """Every knockout of `genes` (GeneSpec list) on HotPath `hot`, with the sample background `variants`
    (stage1.SampleVariants, or None for the reference genome).  knockouts: see check_knockouts.
    -> (pred fp32 [sum T], emb fp32 [sum T, D], ko_pred: per gene fp32 [K_g, T_g][, ko_emb: per gene fp32 [K_g, T_g, D]
    when `embeddings`]), numpy (to_host) or device tensors.  pred / emb are bit-identical to HotPath.predict(genes,
    variants), ko_pred[g][k] to HotPath.predict on gene g with the rows of its k-th set removed.  timer: optional
    callable(phase) -> context manager around the "stage1", "seq2reg" and "seq2gene" phases; counters: optional dict
    filled with item / window counts; min_gene_len: VCFDataset's gene-window length rule (gene_names name the genes)."""
    names = gene_names if gene_names is not None else [f"{g.chrom}:{g.start}-{g.end}" for g in genes]
    sets = check_knockouts(genes, knockouts, names)
    eng, dev = hot.engine, hot.engine.device
    phase = timer or (lambda name: contextlib.nullcontext())
    pass_rows = PASS_ROWS if pass_rows is None else pass_rows
    T = np.asarray([len(g.tissues) for g in genes], np.int64)
    t_off = np.concatenate([[0], np.cumsum(T)])
    D = eng.w.D
    pred = torch.empty(int(t_off[-1]), dtype=torch.float32, device=dev)
    emb = torch.empty((int(t_off[-1]), D), dtype=torch.float32, device=dev)
    ko_pred, ko_emb = [None] * len(genes), [None] * len(genes)
    c = counters if counters is not None else {}
    c.update(genes=len(genes), knockouts=sum(len(s) for s in sets), items=0, windows_encoded=0, windows_per_item=0,
             cre_token_rows=0, gene_token_rows=0, passes=0, slabs=0)
    for a, b, _, _ in cohort.plan_passes([len(g.cre_start) + hot.max_chunks for g in genes], pass_rows):
        c["passes"] += 1
        with phase("stage1"):
            ctoks, gtoks, labels = [], [], []
            for k0 in range(a, b, ism.GENE_GROUP):
                k1 = min(b, k0 + ism.GENE_GROUP)
                t = hot.tokenize(genes[k0:k1], variants)
                _check_stage1(hot, genes[k0:k1], t, variants, sets[k0:k1], min_gene_len, names[k0:k1])
                ctoks += t["cre_tok"]; gtoks += t["gene_tok"]; labels += t["labels"]
                del t
            uc, inv_c = torch.unique(torch.cat(ctoks), dim=0, return_inverse=True)
            ug, inv_g = torch.unique(torch.cat(gtoks), dim=0, return_inverse=True)
            inv_c = inv_c.cpu().numpy().astype(np.int64); inv_g = inv_g.cpu().numpy().astype(np.int64)
            items = []                                      # (cre rows, gene rows, tissues, labels), gene-major
            c0 = g0 = 0
            for i, gi in enumerate(range(a, b)):
                C, G = ctoks[i].shape[0], gtoks[i].shape[0]
                cr, gr, lab = inv_c[c0:c0 + C], inv_g[g0:g0 + G], labels[i].numpy().astype(np.int64)
                c0 += C; g0 += G
                tis = torch.as_tensor(genes[gi].tissues, dtype=torch.long)
                items.append((cr, gr, tis, lab))
                order = batch_order(genes[gi])
                for s in sets[gi]:
                    keep = kept_positions(order, s)
                    items.append((cr[keep], gr, tis, lab[keep]))
                c["windows_per_item"] += (1 + len(sets[gi])) * (C + G) - sum(len(s) for s in sets[gi])
            del ctoks, gtoks
            c["items"] += len(items)
            c["cre_token_rows"] += int(uc.shape[0]); c["gene_token_rows"] += int(ug.shape[0])
            c["windows_encoded"] += int(uc.shape[0] + ug.shape[0])
        with phase("seq2reg"):
            cre_pooled = ism._pool(eng, eng.cre_tok, uc.to(torch.int32))
            gene_pooled = ism._pool(eng, eng.gene_tok, ug.to(torch.int32))
            del uc, ug
        with phase("seq2gene"):
            blocks = score_items(eng, items, [1 + len(sets[gi]) for gi in range(a, b)], cre_pooled, gene_pooled,
                                 rows_budget, embeddings, c)
            for gi, (p, e) in zip(range(a, b), blocks):
                pred[t_off[gi]:t_off[gi + 1]] = p[0]
                ko_pred[gi] = p[1:]
                emb[t_off[gi]:t_off[gi + 1]] = e[0] if embeddings else e
                if embeddings:
                    ko_emb[gi] = e[1:]
            del blocks, cre_pooled, gene_pooled
    out = (pred, emb, ko_pred) + ((ko_emb,) if embeddings else ())
    if to_host:
        host = lambda x: x.cpu().numpy()
        out = (host(pred), host(emb), [host(x) for x in ko_pred]) + (([host(x) for x in ko_emb],) if embeddings else ())
    return out


def knockout_sets(df):
    """User knockout sets from a DataFrame with columns gene_id, knockout (a label) and cre_index (a manifest row, one
    DataFrame row per member).  -> {gene_id: [(label, int64 [n] manifest rows)]}, sets in first-appearance order."""
    missing = [k for k in ("gene_id", "knockout", "cre_index") if k not in df.columns]
    if missing:
        raise ValueError(f"knockouts must have the columns gene_id, knockout and cre_index (missing: {missing})")
    out, where = {}, {}
    for gid, lab, idx in zip(df["gene_id"], df["knockout"], df["cre_index"]):
        if isinstance(idx, (bool, np.bool_)) or not isinstance(idx, (int, np.integer)):
            raise ValueError(f"knockout {lab!r} of gene {gid}: cre_index {idx!r} is not an integer manifest row")
        key = (gid, lab)
        if key not in where:
            where[key] = len(out.setdefault(gid, []))
            out[gid].append((lab, []))
        out[gid][where[key]][1].append(int(idx))
    return {g: [(lab, np.asarray(ix, np.int64)) for lab, ix in v] for g, v in out.items()}


FRAME_COLUMNS = ["gene_id", "tissue", "knockout", "cre_indices", "chromosome", "start_cre", "end_cre", "cre_name",
                 "baseline_expression", "predicted_expression", "delta"]


def knockout_frame(gene_id, tissues, manifest, sets, base_pred, ko_pred):
    """One query row's knockouts in long format: one row per (knockout, tissue), in that order.  manifest: DataFrame
    (chromosome, start_cre, end_cre, cre_name) in manifest order; sets: [(label, manifest rows)]; base_pred fp32 [T];
    ko_pred fp32 [K, T].  The manifest columns name the CRE of a single-CRE knockout and are null for larger sets."""
    T, K = len(tissues), len(sets)
    base = np.asarray(base_pred, np.float32).reshape(T)
    ko = np.asarray(ko_pred, np.float32).reshape(K, T)
    single = [int(ix[0]) if len(ix) == 1 else None for _, ix in sets]
    col = lambda name: [manifest[name].iloc[r] if r is not None else None for r in single]
    rep = lambda xs: [x for x in xs for _ in range(T)]
    to_int = lambda xs: pd.array([None if x is None else int(x) for x in rep(xs)], dtype="Int64")
    return pd.DataFrame({
        "gene_id": [gene_id] * (K * T), "tissue": list(tissues) * K,
        "knockout": rep([lab for lab, _ in sets]), "cre_indices": rep([tuple(int(i) for i in ix) for _, ix in sets]),
        "chromosome": pd.Series(rep(col("chromosome")), dtype=object), "start_cre": to_int(col("start_cre")),
        "end_cre": to_int(col("end_cre")), "cre_name": pd.Series(rep(col("cre_name")), dtype=object),
        "baseline_expression": np.tile(base, K), "predicted_expression": ko.reshape(-1),
        "delta": (ko - base[None, :]).reshape(-1)}, columns=FRAME_COLUMNS)
