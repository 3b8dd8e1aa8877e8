"""Variant tables scored in shared batched passes: every (variant, gene) pair of VariantProcessor.predict, with the
same results, without re-encoding a window whose tokens did not change.

A pair's result is BY DEFINITION what the per-pair path (datasets/vepdataset.VEPBatchBuilder.build + variant_prediction)
gives; this module restates build literally (DESIGN section 12):
  * pairs are grouped by (gene, tissue list); a group's reference item (gene + background SNPs) is tokenized once;
  * per pair, het writes get_iupac_code(REF, ALT) (one byte, 'N' outside the 16 ACGT pairs) and hom writes the ALT
    string (k bytes in place of ONE base: an insertion, or a deletion of that base when the ALT is empty; a multi-base
    REF is not deleted) into the CRE windows that window_hits reaches on the variant's chromosome, and into the gene
    window iff gene_hit and the chromosomes match;
  * the het / hom samples of the builder carry the background only on the variant's chromosome: their windows on other
    chromosomes (except the unreached ones, which the builder re-encodes with the background) are read from the
    reference genome alone;
  * items are deduplicated per group by (chrom, pos, written bytes): duplicate rows and het 'N' collisions are scored
    once and emitted as often as they appear;
  * cre_token_position = cre_hit; gene_token_position = min(token index // L, context - 1) of the token covering the
    variant base in each item's own strand-oriented window (len(seq) - p - 1 on the minus strand, with the edited
    length), with the builder's ValueError for a non-IUPAC character there;
  * groups are taken in passes of about pass_rows distinct token rows (device memory stays bounded for tables of any
    number of genes); within a pass the items of all groups are packed into slabs of at most rows_budget CRE rows, and
    every distinct CRE window and gene chunk goes through seq2reg once (ism.build_edit_items, Engine.prepare_shared /
    run_pooled).  Results do not depend on either split.
"""
import contextlib
from dataclasses import dataclass, field
from typing import List, Optional

import numpy as np
import torch

from . import ism
from .datasets.vepdataset import cre_windows, get_iupac_code, window_hits
from .stage1 import gene_window

GENE_CHARS = "ACGTRYSWKMBDHV"      # characters BPEEncoder.encode_with_position keeps (seq.py:93-97)
# distinct token rows (CRE windows + gene chunks, 800 B each as int32 tokens, 1 KB pooled) per pass: ~100 genes at
# C = 1024, a few hundred MB of tables
PASS_ROWS = 131072


@dataclass
class PairPlan:
    """One (variant, gene) pair: its group, its het / hom edit items (indices into the group's edits) and the builder's
    overlap outcome."""
    group: int
    variant_type: str
    cre_hit: Optional[int] = None
    gene_hit: bool = False
    edits: tuple = ()                # (het edit, hom edit) indices into Group.edits; () for "No overlap"


@dataclass
class Group:
    gene: object
    tissues: list
    edits: List[ism.Edit] = field(default_factory=list)
    edit_of: dict = field(default_factory=dict)     # (chrom, pos, bytes) -> edit index


def plan_pairs(pairs, nb=50, up=1000, down=300000):
    """Host planner.  pairs: dicts with "variant" (vepdataset.Variant, tissue = tissue ids) and "gene" (GeneSpec), as
    VariantProcessor.initialize builds them.  -> (groups, per-pair PairPlan)."""
    groups, group_of, plans = [], {}, []
    for p in pairs:
        v, gene = p["variant"], p["gene"]
        tissues = list(v.tissue if v.tissue is not None else gene.tissues)
        key = (p.get("gene_id", id(gene)), tuple(int(t) for t in tissues))
        if key not in group_of:
            group_of[key] = len(groups)
            groups.append(Group(gene, tissues))
        gi = group_of[key]
        minus = gene.strand == "-"
        order, wins = cre_windows(gene, nb)
        g0, g1 = gene_window(gene.start, gene.end, gene.strand, up, down)
        hits, cre_hit, unreached, gene_hit = window_hits(wins, minus, v.pos, g0, g1)
        if cre_hit is None and not gene_hit:
            plans.append(PairPlan(gi, "No overlap"))
            continue
        # the builder's het / hom samples hold the record and the background of the variant's chromosome only: windows
        # on other chromosomes get neither (unreached windows are re-encoded with the background-only sample)
        chroms = [gene.chrom if gene.cre_chrom is None else gene.cre_chrom[i] for i in order]
        hits = [k for k in hits if chroms[k] == v.chrom]
        plain_cre = [k for k in range(len(wins)) if chroms[k] != v.chrom and k not in unreached]
        edit_gene = gene_hit and gene.chrom == v.chrom
        g = groups[gi]
        ids = []
        for data in (get_iupac_code(v.ref, v.alt).encode(), v.alt.encode()):
            k = (v.chrom, v.pos, data)
            if k not in g.edit_of:
                g.edit_of[k] = len(g.edits)
                g.edits.append(ism.Edit(v.pos, data, hits, edit_gene, plain_cre, gene.chrom != v.chrom))
            ids.append(g.edit_of[k])
        vt = ("Gene and CRE overlap" if cre_hit is not None and gene_hit else
              "CRE overlap only" if cre_hit is not None else "Gene overlap only")
        plans.append(PairPlan(gi, vt, cre_hit, gene_hit, tuple(ids)))
    return groups, plans


def gene_token_position(seq: bytes, starts: np.ndarray, p: int, max_length=200, context_window=200):
    """VEPBatchBuilder.build's gene_token_position for offset p of a strand-oriented gene window `seq` whose BPE tokens
    start at `starts`: the ValueError for a character the tokenizer drops, else min(token index // L, context - 1)."""
    ch = chr(seq[p]).upper()
    return token_position(ch, p, int((starts <= p).sum()) - 1, max_length, context_window)


def token_position(ch: str, p: int, tok_idx: int, max_length=200, context_window=200):
    if ch not in GENE_CHARS:
        raise ValueError(f"Position {p} points to invalid character '{ch}' which is filtered out during "
                         "normalization.")
    return min(tok_idx // max_length, context_window - 1)


@torch.no_grad()
def score_pairs(hot, pairs, variants=None, rows_budget=ism.ROWS_BUDGET, pass_rows=None, timer=None):
    """Every pair of `pairs` (VariantProcessor.initialize's list) on HotPath `hot`.  variants: the background sample as
    stage1.SampleVariants of its SNPs only (or None).  timer: optional callable(phase name) -> context manager around
    the stage-1 / seq2reg / seq2gene phases (tools/bench_vep.py).  pass_rows: distinct token rows per pass (default
    PASS_ROWS).  A ValueError of the builder is raised for the first pair (in table order) that has one, as the per-pair
    path raises it.
    -> (per pair the dict variant_prediction returns for VEPBatchBuilder.build's batch, counters)."""
    eng, dev = hot.engine, hot.engine.device
    phase = timer or (lambda name: contextlib.nullcontext())
    pass_rows = PASS_ROWS if pass_rows is None else pass_rows
    L, CW = hot.max_length, hot.max_chunks
    groups, plans = plan_pairs(pairs, hot.nb, hot.up, hot.down)
    results = [{"pred_gene_exp": [], "embd": [], "variant_type": "No overlap", "gene_token_embedding": [],
                "cre_token_embedding": []} if not pl.edits else None for pl in plans]
    counters = dict(windows_encoded=0, cre_windows_encoded=0, gene_chunks_encoded=0, windows_per_pair=0,
                    pairs=len(pairs), pairs_no_overlap=sum(1 for pl in plans if not pl.edits), items=0, passes=0)
    pairs_of = {}                                          # group -> its pairs with an overlap, in table order
    for n, pl in enumerate(plans):
        if pl.edits:
            pairs_of.setdefault(pl.group, []).append(n)
    errors = []                                            # (pair, ValueError)

    def token_positions(built, pass_pairs):
        """Token positions of every item the pass's pairs read -> ({(group, item): {CRE row}}, {(group, item): {gene
        position}}, per pair (items, gene positions)); a pair with a bad gene position goes to `errors`."""
        need_c, need_g, pair_pos = {}, {}, {}
        for n in pass_pairs:
            pl, pr = plans[n], pairs[n]
            it, g = built[pl.group], groups[pl.group]
            items = (0, 1 + pl.edits[0], 1 + pl.edits[1])
            gpos = [None] * 3
            if pl.gene_hit:
                g0, _ = gene_window(g.gene.start, g.gene.end, g.gene.strand, hot.up, hot.down)
                try:
                    for j, item in enumerate(items):
                        gp = it["gene_pos"][item - 1] if item else None
                        if gp is None:                     # the reference item's gene window, or the plain genome's
                            e = g.edits[item - 1] if item else None
                            seq, starts = it["plain_gene" if e is not None and e.plain_gene else "ref_gene"]
                            p = pr["variant"].pos - 1 - g0
                            if g.gene.strand == "-":
                                p = len(seq) - p - 1
                            gpos[j] = gene_token_position(seq, starts, p, L, CW)
                        else:
                            gpos[j] = token_position(gp[1].upper(), gp[0], gp[2], L, CW)
                except ValueError as e:
                    errors.append((n, e))
                    continue
                for item, gp in zip(items, gpos):
                    need_g.setdefault((pl.group, item), set()).add(gp)
            if pl.cre_hit is not None:
                for item in items:
                    need_c.setdefault((pl.group, item), set()).add(pl.cre_hit)
            pair_pos[n] = (items, gpos)
        return need_c, need_g, pair_pos

    def run_pass(batch):
        counters["passes"] += 1
        built = dict(batch)
        pass_pairs = sorted(n for gi, _ in batch for n in pairs_of[gi])
        with phase("stage1"):
            need_c, need_g, pair_pos = token_positions(built, pass_pairs)
            if errors:                                     # the table fails: what is left only looks for earlier errors
                return
            uc, inv_c = torch.unique(torch.cat([it["cre_tokens"] for _, it in batch]), dim=0, return_inverse=True)
            ug, inv_g = torch.unique(torch.cat([it["gene_tokens"] for _, it in batch]), dim=0, return_inverse=True)
            inv_c = inv_c.cpu().numpy().astype(np.int64); inv_g = inv_g.cpu().numpy().astype(np.int64)
            items = []                                     # (group, item, cre_rows, gene_rows) in the pass's tables
            c_base = g_base = 0
            for gi, it in batch:
                for j, (cr, gr) in enumerate(zip(it["cre_rows"], it["gene_rows"])):
                    items.append((gi, j, inv_c[c_base + cr], inv_g[g_base + gr]))
                c_base += it["cre_tokens"].shape[0]; g_base += it["gene_tokens"].shape[0]
        with phase("seq2reg"):
            cre_pooled = ism._pool(eng, eng.cre_tok, uc.to(torch.int32))
            gene_pooled = ism._pool(eng, eng.gene_tok, ug.to(torch.int32))
        out_of = {}                                        # (group, item) -> (pred, emb, {row: emb}, {pos: [T, D]})
        with phase("seq2gene"):
            a = 0
            while a < len(items):
                b, rows = a, 0
                while b < len(items) and (b == a or rows + len(items[b][2]) <= rows_budget):
                    rows += len(items[b][2]); b += 1
                sl = items[a:b]
                used, local = np.unique(np.concatenate([x[3] for x in sl]), return_inverse=True)
                splits = np.cumsum([len(x[3]) for x in sl])[:-1]
                c_need = [sorted(need_c.get((gi, j), ())) for gi, j, _, _ in sl]
                g_need = [sorted(need_g.get((gi, j), ())) for gi, j, _, _ in sl]
                tis = [torch.as_tensor(groups[gi].tissues, dtype=torch.long) for gi, _, _, _ in sl]
                s = eng.prepare_shared([x[2] for x in sl], np.split(local, splits), len(used), tis,
                                       [built[gi]["labels"] for gi, _, _, _ in sl], cre_token_rows=c_need,
                                       gene_token_positions=g_need)
                out = eng.run_pooled(s, cre_pooled, gene_pooled.index_select(0, torch.from_numpy(used).to(dev)))
                pred, emb = out["pred"].cpu().numpy(), out["emb"].cpu().numpy()
                gtok, ctok = out["gene_token_embedding"].cpu().numpy(), out["cre_token_embedding"].cpu().numpy()
                r = gt = ct = 0
                for (gi, j, _, _), cn, gn in zip(sl, c_need, g_need):
                    T = len(groups[gi].tissues)
                    crow = {row: ctok[ct + x] for x, row in enumerate(cn)}
                    grow = {pos: gtok[gt + x * T: gt + (x + 1) * T] for x, pos in enumerate(gn)}
                    out_of[gi, j] = (pred[r:r + T, None], emb[r:r + T], crow, grow)
                    r += T; ct += len(cn); gt += T * len(gn)
                a = b
        D = emb.shape[1]
        for n in pass_pairs:
            pl = plans[n]
            its, gpos = pair_pos[n]
            T = len(groups[pl.group].tissues)
            o = [out_of[pl.group, i] for i in its]
            zeros = np.zeros((T, D), np.float32)
            results[n] = {"pred_gene_exp": [x[0] for x in o], "embd": [x[1] for x in o],
                          "variant_type": pl.variant_type,
                          "gene_token_embedding": [x[3][gp] if pl.gene_hit else zeros for x, gp in zip(o, gpos)],
                          "cre_token_embedding": [np.repeat(x[2][pl.cre_hit][None], T, 0) if pl.cre_hit is not None
                                                  else zeros for x in o]}
            it = built[pl.group]
            counters["windows_per_pair"] += 3 * it["C"] + it["G_ref"] + sum(int(it["g_count"][i - 1]) for i in its[1:])
        counters["windows_encoded"] += int(uc.shape[0] + ug.shape[0])
        counters["cre_windows_encoded"] += int(uc.shape[0]); counters["gene_chunks_encoded"] += int(ug.shape[0])
        counters["items"] += len(items)

    batch, rows = [], 0
    for gi in sorted(pairs_of):
        g = groups[gi]
        with phase("stage1"):
            it = ism.build_edit_items(hot, g.gene, g.edits, variants, want_gene_pos=True)
        batch.append((gi, it))
        rows += it["cre_tokens"].shape[0] + it["gene_tokens"].shape[0]
        if rows >= pass_rows:
            run_pass(batch)
            batch, rows = [], 0
    if batch:
        run_pass(batch)
    if errors:
        raise min(errors, key=lambda x: x[0])[1]
    return results, counters
