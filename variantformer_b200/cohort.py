"""Cohort prediction: every (sample, gene) of a multi-sample VCF, with each distinct window encoded once across samples.

A (sample, gene) prediction is BY DEFINITION what HotPath.predict(genes, SampleVariants(that sample)) gives.  What is
not recomputed (DESIGN section 14):
  * a window's encoded bytes depend on its (chrom, w0, w1, flags) and on the list of records the encoder applies for
    the sample (stage1 / vf_encode_windows' rule); rows (window, sample) with equal lists are one group, proposed by a
    128-bit key (vf_window_genotype_keys) and confirmed element by element against the group's representative
    (vf_window_genotype_equal; a mismatching row becomes a group of its own).  Windows shared by two genes count once;
  * only representatives are encoded (with the representative sample's records and the per-sample path's pitch) and
    BPE-tokenized, and every DISTINCT token row (CRE window or 200-token gene chunk) goes through seq2reg once;
  * an item (sample, gene) is its list of token rows plus its tissues: equal items are scored once and emitted for
    each of their samples; the rest run as in ism / vep_batch (Engine.prepare_shared + run_pooled, slabs of at most
    ism.ROWS_BUDGET CRE rows, passes of about PASS_ROWS token rows (plan_passes: a gene too large for one pass is
    split by samples, so a pass does not grow with the cohort).  Results depend on neither split.
Stage-1 errors (1: pitch overflow, 2: more than 2048 applied records in a window) are known from the keys before any
window is encoded, per (sample, gene); the first sample (in cohort order) with one raises, with the code the per-sample
call for that sample would raise.
"""
import contextlib
from dataclasses import dataclass

import numpy as np
import torch

from . import ism, ops
from .stage1 import FLAG_REVCOMP, cre_window, gene_window

# distinct token rows per pass (CRE rows + gene chunks, counted before token deduplication): device memory of a pass
# stays bounded whatever the number of samples and genes
PASS_ROWS = 131072


@dataclass
class Windows:
    """Distinct windows of a gene list: CRE windows and gene windows in two tables (they are tokenized differently),
    each indexed by (chrom, w0, w1, flags); per gene its CRE windows in batch order and its gene window."""
    cre: list                 # [(chrom, w0, w1, flags)]
    gene: list
    cre_of: list              # per gene: int64 [C_g] indices into cre
    gene_of: np.ndarray       # per gene: index into gene
    labels: list              # per gene: int64 [C_g] CRE labels in batch order


def gene_windows(genes, nb=50, up=1000, down=300000):
    """Window tables of `genes` in HotPath.tokenize's batch order (CREs sorted by start, reversed on the minus strand)."""
    cre, gene, index_c, index_g, cre_of, gene_of, labels = [], [], {}, {}, [], [], []
    for g in genes:
        minus = g.strand == "-"
        order = np.argsort(g.cre_start, kind="stable")
        if minus:
            order = order[::-1]
        fl = FLAG_REVCOMP if minus else 0
        ks = []
        for i in order:
            a0, a1 = cre_window(g.cre_start[i], g.cre_end[i], nb)
            k = (g.chrom if g.cre_chrom is None else g.cre_chrom[i], a0, a1, fl)
            if k not in index_c:
                index_c[k] = len(cre); cre.append(k)
            ks.append(index_c[k])
        cre_of.append(np.asarray(ks, np.int64))
        labels.append(np.asarray(g.cre_labels)[order].astype(np.int64))
        k = (g.chrom,) + tuple(gene_window(g.start, g.end, g.strand, up, down)) + (fl,)
        if k not in index_g:
            index_g[k] = len(gene); gene.append(k)
        gene_of.append(index_g[k])
    return Windows(cre, gene, cre_of, np.asarray(gene_of, np.int64), labels)


def group_rows(window, count, keys, equal_fn=None):
    """Groups of rows (window, sample) from their genotype keys.  window int64 [n], count int32 [n], keys int64 [n, 2]
    (torch, any device).  Rows of one window with equal (count, key) are proposed as one group, numbered in the order
    of (window, count, key); the representative of a group is its first row.  equal_fn(rep_of_row) -> bool [n]: the
    exact comparison; every row it rejects becomes a group of its own (numbered after the others, in row order).
    -> (group int64 [n], rep int64 [n_groups]) on the keys' device."""
    n = window.numel()
    dev = keys.device
    if n == 0:
        return torch.zeros(0, dtype=torch.int64, device=dev), torch.zeros(0, dtype=torch.int64, device=dev)
    m = torch.stack([window.to(dev, torch.int64), count.to(dev, torch.int64), keys[:, 0], keys[:, 1]], 1)
    _, group = torch.unique(m, dim=0, return_inverse=True)
    n_g = int(group.max().item()) + 1
    rows = torch.arange(n, device=dev)
    rep = torch.full((n_g,), n, dtype=torch.int64, device=dev).scatter_reduce_(0, group, rows, "amin")
    if equal_fn is not None:
        bad = ~equal_fn(rep[group])
        nb = int(bad.sum().item())
        if nb:
            bad_rows = rows[bad]
            group = group.clone()
            group[bad_rows] = n_g + torch.arange(nb, device=dev)
            rep = torch.cat([rep, bad_rows])
    return group, rep


def plan_passes(rows_per_gene, pass_rows=PASS_ROWS, n_samples=1, sample_rows=None):
    """Passes (a, b, s0, s1) = genes [a, b) x samples [s0, s1), in gene order.  rows_per_gene: token rows of each gene
    over all samples; sample_rows: per gene an upper bound of ONE sample's token rows (default: rows_per_gene).
    Consecutive genes are packed with all samples until a pass reaches pass_rows; a gene whose rows alone exceed
    pass_rows gets passes of its own, its samples cut into runs of max(1, pass_rows // sample_rows) samples.  So no
    pass holds more than max(2 pass_rows, one sample's rows of one gene), whatever the number of samples."""
    sample_rows = rows_per_gene if sample_rows is None else sample_rows
    out, a, rows = [], 0, 0
    for i, r in enumerate(rows_per_gene):
        if r > pass_rows:
            if a < i:
                out.append((a, i, 0, n_samples))
            k = max(1, pass_rows // max(1, int(sample_rows[i])))
            out += [(i, i + 1, s0, min(n_samples, s0 + k)) for s0 in range(0, n_samples, k)]
            a, rows = i + 1, 0
            continue
        rows += int(r)
        if rows >= pass_rows:
            out.append((a, i + 1, 0, n_samples)); a, rows = i + 1, 0
    if a < len(rows_per_gene):
        out.append((a, len(rows_per_gene), 0, n_samples))
    return out


def dedup_items(items):
    """items: per (sample, gene) a tuple (cre_rows int64 [C], gene_rows int64 [G], tissues tuple, CRE labels int64 [C]).
    -> (unique item indices in first-occurrence order, index into them per item)."""
    first, of = {}, np.empty(len(items), np.int64)
    uniq = []
    for i, (c, g, t, lab) in enumerate(items):
        k = (np.asarray(c, np.int64).tobytes(), np.asarray(g, np.int64).tobytes(), tuple(t),
             np.asarray(lab, np.int64).tobytes())
        j = first.get(k)
        if j is None:
            j = first[k] = len(uniq); uniq.append(i)
        of[i] = j
    return np.asarray(uniq, np.int64), of


def slab_ranges(cre_rows_per_item, rows_budget=ism.ROWS_BUDGET):
    """Consecutive [a, b) ranges of items with at most rows_budget CRE rows each (at least one item)."""
    out, a = [], 0
    n = len(cre_rows_per_item)
    while a < n:
        b, rows = a, 0
        while b < n and (b == a or rows + cre_rows_per_item[b] <= rows_budget):
            rows += cre_rows_per_item[b]; b += 1
        out.append((a, b)); a = b
    return out


def _up(a, dt, dev):
    return torch.from_numpy(np.ascontiguousarray(a, dt)).to(dev)


class _Table:
    """Genotype keys and groups of one window table x the samples."""

    def __init__(self, hot, cohort, wins, samples, pitch_extra, key_bits, phase):
        dev = hot.engine.device
        S, W = len(samples), len(wins)
        self.S, self.W = S, W
        self.chrom = [w[0] for w in wins]
        self.base = np.asarray([hot.genome.offsets[c][0] for c in self.chrom], np.int64)
        for c, w in zip(self.chrom, wins):
            assert w[2] <= hot.genome.offsets[c][1], "window runs past the end of the chromosome"
        w0 = np.asarray([w[1] for w in wins], np.int64); w1 = np.asarray([w[2] for w in wins], np.int64)
        self.flags = np.asarray([w[3] for w in wins], np.uint8)
        self.max_window = int((w1 - w0).max()) if W else 0
        self.pitch = ((self.max_window + pitch_extra + 15) // 16) * 16        # WindowTokenizer.sequences' pitch rule
        # rows window-major: row = window * S + sample
        rw0, rw1 = np.repeat(w0, S), np.repeat(w1, S)
        lo, hi = cohort.window_ranges(np.tile(np.asarray(samples, np.int64), W), np.repeat(self.chrom, S), rw0, rw1)
        self.lo, self.hi, self.w0, self.w1 = lo, hi, w0, w1
        args = (_up(rw0, np.int32, dev), _up(rw1, np.int32, dev), _up(lo, np.int32, dev), _up(hi, np.int32, dev),
                _up(np.repeat(self.flags, S), np.uint8, dev), cohort.dev)
        with phase("keys"):
            keys, count, lens, _ = ops.window_genotype_keys(*args, key_bits=key_bits)
            self.group, self.rep = group_rows(torch.arange(W * S, device=dev) // max(S, 1), count, keys,
                                              lambda rep: ops.window_genotype_equal(*args, rep.to(torch.int32)) != 0)
            self.group = self.group.cpu().numpy(); self.rep = self.rep.cpu().numpy()
            count = count.cpu().numpy(); lens = lens.cpu().numpy()
        self.vdev = cohort.dev
        # per row: 2 = past the 2048-record cap, 1 = longer than the pitch (the encoder's codes)
        self.err = np.where(count < 0, 2, np.where(lens > self.pitch, 1, 0)).astype(np.int32)
        self.lens = lens

    def encode(self, hot, groups):
        """Encoded bytes of the representatives of `groups` -> (uint8 [n, pitch], int32 lens) on the device."""
        dev = hot.engine.device
        r = self.rep[groups]
        w = r // self.S
        t = lambda a, dt: _up(a, dt, dev)
        out, lens, _ = ops.encode_windows(hot.genome.seq, t(self.base[w], np.int64), t(self.w0[w], np.int32),
                                          t(self.w1[w], np.int32), t(self.lo[r], np.int32), t(self.hi[r], np.int32),
                                          t(self.flags[w], np.uint8), self.vdev, max(1, self.max_window),
                                          self.pitch)
        return out, lens


@torch.no_grad()
def predict_cohort(hot, genes, cohort, sample_idx=None, to_host=True, rows_budget=ism.ROWS_BUDGET, pass_rows=None,
                   key_bits=128, timer=None, counters=None, min_gene_len=None, gene_names=None):
    """Every (sample, gene) of `genes` (GeneSpec list) for the samples `sample_idx` (default: all) of `cohort`
    (stage1.CohortVariants) on HotPath `hot`.  -> (pred fp32 [S, sum T], emb fp32 [S, sum T, D]) in (sample, gene,
    tissue) order, numpy (to_host) or device tensors.  Bit-identical to HotPath.predict(genes, that sample's
    SampleVariants) for every sample.  timer: optional callable(phase) -> context manager around the "stage1", "keys",
    "seq2reg" and "seq2gene" phases; counters: optional dict filled with rows / windows / token rows / items counts;
    key_bits < 128 truncates the genotype keys (tests: forced collisions).  min_gene_len: raise an AssertionError, before
    any window is encoded, for the first (sample, gene) whose encoded gene window is not longer (VCFDataset's rule;
    gene_names name the genes in its message)."""
    eng, dev = hot.engine, hot.engine.device
    phase = timer or (lambda name: contextlib.nullcontext())
    pass_rows = PASS_ROWS if pass_rows is None else pass_rows
    samples = list(range(len(cohort.names))) if sample_idx is None else [int(s) for s in sample_idx]
    S, CW = len(samples), hot.max_chunks
    wins = gene_windows(genes, hot.nb, hot.up, hot.down)
    T = np.asarray([len(g.tissues) for g in genes], np.int64)
    t_off = np.concatenate([[0], np.cumsum(T)])
    D = eng.w.D
    pred = torch.empty((S, int(t_off[-1])), dtype=torch.float32, device=dev)
    emb = torch.empty((S, int(t_off[-1]), D), dtype=torch.float32, device=dev)
    c = counters if counters is not None else {}
    c.update(samples=S, genes=len(genes), sample_windows=0, windows_encoded=0, cre_groups=0, gene_groups=0,
             token_rows=0, sample_token_rows=0, cre_token_rows=0, gene_token_rows=0, items=S * len(genes), items_scored=0,
             passes=0)
    if not genes or not S:
        return (pred.cpu().numpy(), emb.cpu().numpy()) if to_host else (pred, emb)
    with phase("stage1"):
        ct = _Table(hot, cohort, wins.cre, samples, 4096, key_bits, phase)
        gt = _Table(hot, cohort, wins.gene, samples, 4096, key_bits, phase)
    c["sample_windows"] = int(S * (sum(len(x) for x in wins.cre_of) + len(genes)))
    # ---- stage-1 errors, before any work: per sample the maximum code over its windows of every gene ----
    err_sg = np.zeros((S, len(genes)), np.int32)
    ce = ct.err.reshape(ct.W, S); ge = gt.err.reshape(gt.W, S)
    for gi in range(len(genes)):
        e = ge[wins.gene_of[gi]]
        if len(wins.cre_of[gi]):
            e = np.maximum(e, ce[wins.cre_of[gi]].max(0))
        err_sg[:, gi] = e
    bad = np.nonzero(err_sg.max(1))[0]
    if len(bad):
        s = int(bad[0]); gi = int(np.nonzero(err_sg[s])[0][0])
        g = genes[gi]
        raise RuntimeError(f"stage-1 kernel reported error {int(err_sg[s].max())} for sample {cohort.names[samples[s]]} "
                           f"(first at gene {g.chrom}:{g.start}-{g.end}) (1: pitch overflow, 2: >2048 variants/window)")
    if min_gene_len is not None:
        glen = gt.lens.reshape(gt.W, S)[wins.gene_of]                        # [genes, S] encoded gene-window lengths
        short = np.nonzero((glen <= min_gene_len).T.ravel())[0]             # sample-major, as a per-sample loop meets them
        if len(short):
            gi = int(short[0] % len(genes))
            name = gene_names[gi] if gene_names is not None else f"{genes[gi].chrom}:{genes[gi].start}-{genes[gi].end}"
            raise AssertionError(f"Mutated sequence is less than {min_gene_len}bp for gene {name}")
    # ---- passes: about pass_rows token rows (CRE groups + max_chunks per gene group) each ----
    cg = ct.group.reshape(ct.W, S); gg = gt.group.reshape(gt.W, S)
    rows_per_gene = [len(np.unique(cg[wins.cre_of[gi]])) + CW * len(np.unique(gg[wins.gene_of[gi]]))
                     for gi in range(len(genes))]
    for a, b, s0, s1 in plan_passes(rows_per_gene, pass_rows, S, [len(x) + CW for x in wins.cre_of]):
        c["passes"] += 1
        with phase("stage1"):
            c_groups = np.unique(np.concatenate([cg[wins.cre_of[gi], s0:s1].ravel() for gi in range(a, b)]))
            g_groups = np.unique(np.concatenate([gg[wins.gene_of[gi], s0:s1].ravel() for gi in range(a, b)]))
            c["cre_groups"] += len(c_groups); c["gene_groups"] += len(g_groups)
            c["windows_encoded"] += len(c_groups) + len(g_groups)
            # CRE representatives: fixed 200-token rows
            seq, lens = ct.encode(hot, c_groups)
            ctok, _, _ = hot.tok.tokenize_fixed(seq, lens, seq.shape[1], typical_len=ct.max_window)
            del seq
            uc, inv_c = torch.unique(ctok, dim=0, return_inverse=True)
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
            # items (sample, gene) of the pass, sample-major
            items, where = [], []
            for s in range(s0, s1):
                for gi in range(a, b):
                    items.append((row_of_cg[cg[wins.cre_of[gi], s]], rows_of_gg[int(gg[wins.gene_of[gi], s])],
                                  tuple(int(t) for t in genes[gi].tissues), wins.labels[gi]))
                    where.append((s, gi))
            c["sample_token_rows"] += sum(len(x[0]) + len(x[1]) for x in items)
            uniq, of = dedup_items(items)
            c["items_scored"] += len(uniq)
        with phase("seq2reg"):
            cre_pooled = ism._pool(eng, eng.cre_tok, uc)
            gene_pooled = ism._pool(eng, eng.gene_tok, ug)
        with phase("seq2gene"):
            u_pred, u_emb = [None] * len(uniq), [None] * len(uniq)
            for x0, x1 in slab_ranges([len(items[i][0]) for i in uniq], rows_budget):
                sl = [items[i] for i in uniq[x0:x1]]
                used, local = np.unique(np.concatenate([x[1] for x in sl]), return_inverse=True)
                splits = np.cumsum([len(x[1]) for x in sl])[:-1]
                labels = [torch.from_numpy(x[3]) for x in sl]
                s_ = eng.prepare_shared([x[0] for x in sl], np.split(local, splits), len(used),
                                        [torch.as_tensor(x[2], dtype=torch.long) for x in sl], labels)
                out = eng.run_pooled(s_, cre_pooled, gene_pooled.index_select(0, torch.from_numpy(used).to(dev)))
                r = 0
                for j, x in zip(range(x0, x1), sl):
                    n = len(x[2])
                    u_pred[j] = out["pred"][r:r + n]; u_emb[j] = out["emb"][r:r + n]
                    r += n
            for i, (s, gi) in enumerate(where):
                pred[s, t_off[gi]:t_off[gi + 1]] = u_pred[of[i]].reshape(-1)
                emb[s, t_off[gi]:t_off[gi + 1]] = u_emb[of[i]]
    if to_host:
        return pred.cpu().numpy(), emb.cpu().numpy()
    return pred, emb
