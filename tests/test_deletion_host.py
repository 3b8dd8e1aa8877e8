"""Host logic of in-silico deletions (variantformer_b200.deletion): the window-containment rule at its edges on both
strands, validation, tiles, the default scan's spans, the planner's items against a per-item restatement on a fake
engine and encoder (passes, slabs), and the processor's frame.  CPU only."""
import numpy as np
import pandas as pd
import pytest
import torch

from tests.test_knockout_host import _FakeEngine, _fake_pool
from variantformer_b200 import deletion, ism, knockout
from variantformer_b200.pipeline import GeneSpec
from variantformer_b200.stage1 import cre_window, gene_window
from variantformer_b200.utils.constants import REF_CREs

NB, UP, DOWN, L, CW = 50, 100, 3000, 4, 4


def applied_records(pos, ref_len, alt_len, gt, w0, w1, snp_only=False, extra=None):
    """AppliedScan restated: the indices of the records [0, n) applied in window [w0, w1), with `extra` = (pos, ref_len,
    alt_len) merged after every record of pos <= its own (index -1)."""
    order = list(range(len(pos)))
    if extra is not None:
        order.insert(int(np.searchsorted(pos, extra[0], "right")), -1)
    rec = lambda i: extra if i < 0 else (pos[i], ref_len[i], alt_len[i])
    out, cur = [], w0
    for i in order:
        p, rl, al = rec(i)
        if i >= 0 and gt[i] == 0:
            continue
        if p < w0 or p >= w1 or p < cur or p + rl > w1 or (snp_only and not (rl == 1 and al == 1)):
            continue
        cur = p + rl
        out.append(i)
    return out


def encode(chrom, w0, w1, var, extra=None, rc=False):
    """The window's bytes under the rule above (hom ALTs; reverse complement as the plain character reversal suffices
    for the fake tokenizer) -> (bytes, applied extra)."""
    pos, rl, alt = var["pos"], var["ref_len"], var["alt"]
    idx = applied_records(pos, rl, [len(a) for a in alt], np.full(len(pos), 2), w0, w1,
                          extra=None if extra is None else (extra[0], extra[1], len(extra[2])))
    out, x = bytearray(), w0
    for i in idx:
        p, r, a = (extra[:3] if i < 0 else (pos[i], rl[i], alt[i]))
        out += chrom[x:p]; out += a; x = p + r
    out += chrom[x:w1]
    return (bytes(out[::-1]) if rc else bytes(out)), -1 in idx


def fake_tokens(b, cap):
    """One token per 200 bytes (a hash, never 0), first `cap` kept."""
    t = [sum(b[i:i + 200]) % 89 + 1 + (len(b[i:i + 200]) % 7) for i in range(0, len(b), 200)]
    return t[:cap], len(t)


def _tok_rows(seqs, cap):
    rows = np.zeros((len(seqs), cap), np.int32)
    cnt = np.zeros(len(seqs), np.int32)
    for r, s in enumerate(seqs):
        t, n = fake_tokens(s, cap)
        rows[r, :len(t)] = t; cnt[r] = n
    return torch.from_numpy(rows), torch.from_numpy(cnt)


class _Genome:
    def __init__(self, chroms):
        self.chroms = chroms
        self.offsets, o = {}, 0
        for k, v in chroms.items():
            self.offsets[k] = (o, len(v)); o += len(v)
        self.seq = torch.from_numpy(np.frombuffer(b"".join(chroms.values()), np.uint8).copy())


class _FakeHot:
    """HotPath's attributes, tokenize() contract and the edit encoder, on bytes built by the restated rule."""
    nb, up, down, max_length, max_chunks = NB, UP, DOWN, L, CW
    merges = None

    def __init__(self, chroms):
        self.genome = _Genome(chroms)
        self.engine = _FakeEngine()
        self.tok = self

    def _windows(self, g):
        o = knockout.batch_order(g)
        cw = [(g.chrom if g.cre_chrom is None else g.cre_chrom[i],) + cre_window(g.cre_start[i], g.cre_end[i], NB) for i in o]
        return cw, (g.chrom,) + gene_window(g.start, g.end, g.strand, UP, DOWN)

    def _var(self, variants, ch):
        return (variants or {}).get(ch, dict(pos=np.zeros(0, np.int64), ref_len=np.zeros(0, np.int64), alt=[]))

    def tokenize(self, genes, variants=None, extra=None):
        ct, gt, labels, clen, glen = [], [], [], [], []
        for g in genes:
            cw, gw = self._windows(g)
            rc = g.strand == "-"
            cs = [encode(self.genome.chroms[c], a, b, self._var(variants, c), extra if extra and extra[3] == c else None,
                         rc)[0] for c, a, b in cw]
            gs = encode(self.genome.chroms[gw[0]], gw[1], gw[2], self._var(variants, gw[0]),
                        extra if extra and extra[3] == gw[0] else None, rc)[0]
            ct.append(_tok_rows(cs, L)[0])
            t, n = _tok_rows([gs], L * CW)
            G = min(CW, (int(n[0]) + L - 1) // L)
            gt.append(t[0, :G * L].view(G, L))
            labels.append(torch.from_numpy(np.asarray(g.cre_labels)[knockout.batch_order(g)].copy()))
            clen += [len(s) for s in cs]; glen.append(len(gs))
        return dict(cre_tok=ct, gene_tok=gt, labels=labels, err=torch.zeros((), dtype=torch.int32),
                    cre_seq=(None, torch.tensor(clen)), gene_seq=(None, torch.tensor(glen)))

    def tokenize_fixed(self, seq, lens, max_len, typical_len=None):
        t, cnt = _tok_rows(seq, L)
        return t, t == 0, cnt

    def predict(self, genes, variants=None, extra=None):
        t = self.tokenize(genes, variants, extra)
        out = [_FakeEngine.score(c.double().sum(1).numpy(), g.double().sum(1).numpy(), lab.numpy(), x)
               for c, g, lab, gn in zip(t["cre_tok"], t["gene_tok"], t["labels"], genes) for x in gn.tissues]
        emb = np.asarray(out)
        return emb.sum(1), emb


class _Rows(list):
    """Encoded rows as bytes objects, with the [n, pitch] shape of the device rows."""
    def __init__(self, rows, pitch):
        super().__init__(rows)
        self.shape = (len(rows), pitch)


def _fake_encode_edits(hot, variants, rows, pitch):
    seqs, app = _Rows([], pitch), []
    for ch, w0, w1, fl, p, rl, anc in rows:
        s, a = encode(hot.genome.chroms[ch], w0, w1, hot._var(variants, ch), (p, rl, bytes([anc])), bool(fl & 1))
        seqs.append(s); app.append(a)
    return seqs, torch.tensor([len(s) for s in seqs], dtype=torch.int32), torch.tensor(app, dtype=torch.uint8), \
        torch.zeros(1, dtype=torch.int32)


def _fake_bpe(seq, lens, max_len, merges, out_pitch, out_cap, **kw):
    return _tok_rows(seq, out_cap)


def _world(seed=0):
    rng = np.random.default_rng(seed)
    chroms = {c: rng.choice(np.frombuffer(b"ACGT", np.uint8), n).tobytes() for c, n in (("chr1", 40_000), ("chr2", 20_000))}
    var = {}
    for c, n in (("chr1", 40_000), ("chr2", 20_000)):
        pos = np.unique(rng.integers(0, n - 10, n // 60))
        rl = np.where(rng.random(len(pos)) < 0.2, rng.integers(2, 6, len(pos)), 1)
        alt = [rng.choice(np.frombuffer(b"ACGT", np.uint8), int(rng.integers(1, 4))).tobytes() for _ in pos]
        var[c] = dict(pos=pos, ref_len=rl, alt=alt)
    genes = []
    for k, (strand, start) in enumerate((("+", 10_000), ("-", 22_000), ("+", 30_000))):
        cs = np.sort(rng.integers(start - 2_000, start + 4_000, 6 + k)); ce = cs + rng.integers(100, 400, len(cs))
        genes.append(GeneSpec("chr1", start, start + 2_500, strand, cs, ce, rng.integers(0, 9, len(cs)), [62, 3][:1 + k % 2]))
    genes[1].cre_chrom = ["chr1"] * (len(genes[1].cre_start) - 1) + ["chr2"]       # one CRE on another chromosome
    genes[1].cre_start[-1] = 5_000; genes[1].cre_end[-1] = 5_300
    return chroms, var, genes


@pytest.mark.parametrize("strand", ["+", "-"])
def test_containment_edges(strand):
    g = GeneSpec("chr1", 10_000, 12_000, strand, np.array([1_000, 3_000]), np.array([1_200, 3_300]), np.array([0, 1]),
                 [62], cre_chrom=["chr1", "chr2"])
    w0, w1 = 950, 1_250                                       # CRE 0's window [start - 50, end + 50)
    k = list(knockout.batch_order(g)).index(0)                # its batch position
    # 1-based span [a, b]: REF covers 0-based [a - 2, b) (anchor a - 2)
    cases = [((w0 + 1, w0 + 10), False),                      # anchor at w0 - 1: not contained
             ((w0 + 2, w0 + 10), True),                       # anchor at w0
             ((w1 - 20, w1), True),                           # REF ends at w1
             ((w1 - 20, w1 + 1), False),                      # one past it
             ((w0 - 100, w1 + 100), False),                   # covers the window: clipped, unchanged
             ((w0 + 2, w1), True)]                            # the whole window after the anchor
    spans = np.asarray([s for s, _ in cases], np.int64)
    cre, gene = deletion.gene_hits(g, spans, ["chr1"] * len(spans), NB, UP, DOWN)
    assert cre[:, k].tolist() == [w for _, w in cases] and not gene.any()
    assert not cre[:, 1 - k].any()
    assert deletion.contains(w0, w1, spans).tolist() == [w for _, w in cases]
    # the same coordinates on chr2 reach only the chr2 CRE's window, never the chr1 gene window
    g2 = deletion.gene_hits(g, np.array([[2_952, 3_100]]), ["chr2"], NB, UP, DOWN)
    assert g2[0][0, 1 - k] and not g2[0][0, k] and not g2[1][0]
    g0, g1 = gene_window(g.start, g.end, strand, UP, DOWN)
    _, gene = deletion.gene_hits(g, np.array([[g0 + 2, g0 + 5], [g0 + 1, g0 + 5], [g1 - 3, g1], [g1 - 3, g1 + 1]]),
                                 ["chr1"] * 4, NB, UP, DOWN)
    assert gene.tolist() == [True, False, True, False]


def test_record_and_validation_messages():
    pos, rl = deletion.record(np.array([[5, 5], [10, 19]]))
    assert pos.tolist() == [3, 8] and rl.tolist() == [2, 11]
    g = GeneSpec("chr1", 1_000, 2_000, "+", np.array([100]), np.array([300]), np.array([0]), [62])
    lens = {"chr1": 5_000}
    ok = deletion.check_deletions([g], [np.array([[2, 2], [10, 5_000]])], None, lens)
    assert ok[0][0].tolist() == [[2, 2], [10, 5_000]] and ok[0][1] == ["chr1", "chr1"]
    for spans, ch, msg in (([[1, 5]], None, "starts at 2 or later"), ([[10, 9]], None, "empty"),
                           ([[10, 5_001]], None, "outside chr1"), ([[10, 20]], "chrX", "not in the genome"),
                           ([[1.5, 3]], None, "non-integer"), ([[1, 2, 3]], None, r"\[n, 2\]")):
        with pytest.raises(ValueError, match=msg):
            deletion.check_deletions([g], [np.asarray(spans)], None if ch is None else [ch], lens, ["G"])
    with pytest.raises(ValueError, match="deletion 1 \\[10, 9\\] on chr1 of gene G"):
        deletion.check_deletions([g], [np.array([[2, 3], [10, 9]])], None, lens, ["G"])
    with pytest.raises(ValueError, match="no CRE"):
        deletion.check_deletions([GeneSpec("chr1", 1, 2, "+", np.zeros(0), np.zeros(0), np.zeros(0), [1])],
                                 [np.zeros((0, 2))], None, lens)
    with pytest.raises(ValueError, match="2 deletions and 1 chromosomes"):
        deletion.check_deletions([g], [np.array([[2, 3], [4, 5]])], [["chr1"]], lens)
    with pytest.raises(ValueError, match="2 entries for 1 genes"):
        deletion.check_deletions([g], [np.zeros((0, 2)), np.zeros((0, 2))], None, lens)


def test_tiles_and_default_spans():
    t = deletion.tiles("chr3", 1_001, 1_200, 50, 25)
    assert list(t.columns) == ["chromosome", "start", "end"] and set(t["chromosome"]) == {"chr3"}
    assert t["start"].tolist() == [1_001 + 25 * k for k in range(7)] and (t["end"] - t["start"] == 49).all()
    assert t["end"].max() <= 1_200 and deletion.tiles("chr1", 10, 10, 1, 1)["end"].tolist() == [10]
    for args in ((10, 20, 0, 1), (10, 20, 5, 0), (10, 20, 12, 1)):
        with pytest.raises(ValueError):
            deletion.tiles("chr1", *args)
    m = pd.DataFrame({"chromosome": ["chr2", "chr5"], "start_cre": [100, 40], "end_cre": [250, 90],
                      "cre_name": [REF_CREs[0], REF_CREs[1]]})
    spans, ch = deletion.default_spans(m)
    assert spans.tolist() == [[101, 250], [41, 90]] and ch == ["chr2", "chr5"]
    # the CRE's own bases in 0-based [start_cre, end_cre) are exactly the span: its window [start - 50, end + 50)
    # contains the REF span with its anchor
    assert deletion.contains(*cre_window(100, 250, 50), spans[:1])[0]
    u = deletion.user_deletions(pd.DataFrame({"gene_id": ["A", "B", "A"], "chromosome": ["chr1"] * 3,
                                              "start": [5, 7, np.int64(9)], "end": [6, 8, 12]}))
    assert list(u) == ["A", "B"] and u["A"][0] == ["chr1:5-6", "chr1:9-12"] and u["A"][1].tolist() == [[5, 6], [9, 12]]
    with pytest.raises(ValueError, match="missing"):
        deletion.user_deletions(pd.DataFrame({"gene_id": ["A"], "start": [1], "end": [2]}))
    with pytest.raises(ValueError, match="not an integer"):
        deletion.user_deletions(pd.DataFrame({"gene_id": ["A"], "chromosome": ["chr1"], "start": [1.5], "end": [2]}))


def test_planner_items_equal_the_per_item_restatement(monkeypatch):
    monkeypatch.setattr(deletion.ism, "_pool", _fake_pool)
    monkeypatch.setattr(deletion, "_encode_edits", _fake_encode_edits)
    monkeypatch.setattr(deletion.ops, "bpe_tokenize", _fake_bpe)
    chroms, var, genes = _world()
    hot = _FakeHot(chroms)
    spans, chs = [], []
    for g in genes:
        o = knockout.batch_order(g)
        w = [cre_window(g.cre_start[i], g.cre_end[i], NB) for i in o]
        g0, g1 = gene_window(g.start, g.end, g.strand, UP, DOWN)
        s = [(w[0][0] + 12, w[0][0] + 20),                    # inside one CRE window
             (w[1][1] - 5, w[1][1] + 30),                     # straddling a window edge: no CRE window changes
             (int(g.cre_start[o[2]]) + 1, int(g.cre_end[o[2]])),  # a whole CRE
             (g0 + 700, g0 + 1_100),                          # inside the gene window, shifting the chunking
             (g0 + 2, g1),                                    # the whole gene window after its anchor
             (min(w)[0] - 500, max(x[1] for x in w) + 500),  # covers every CRE window: a no-op there
             (2, 3)]                                          # far away: a no-op
        spans.append(np.asarray(s, np.int64)); chs.append(None)
    spans[1] = np.vstack([spans[1], [[5_010, 5_100]]])        # in the chr2 CRE window
    chs[1] = ["chr1"] * (len(spans[1]) - 1) + ["chr2"]
    for background in (None, var):
        runs = []
        for budget, pass_rows in ((ism.ROWS_BUDGET, None), (1, 1), (30, 40)):
            hot.engine.slab_rows = []
            c = {}
            runs.append(deletion.deletion_scan(hot, genes, spans, background, chs, embeddings=True, rows_budget=budget,
                                               pass_rows=pass_rows, counters=c))
            assert all(sum(r) <= budget or len(r) == 1 for r in hot.engine.slab_rows)
            if budget == 1:
                assert c["passes"] == len(genes) and all(len(r) == 1 for r in hot.engine.slab_rows)
        base_p, base_e = hot.predict(genes, background)
        for pred, emb, dp, de, app in runs:
            assert np.array_equal(pred, base_p) and np.array_equal(emb, base_e)
            for gi, g in enumerate(genes):
                assert dp[gi].shape == (len(spans[gi]), len(g.tissues))
                for j, (a, b) in enumerate(spans[gi].tolist()):
                    ch = g.chrom if chs[gi] is None else chs[gi][j]
                    rec = (a - 2, b - a + 2, chroms[ch][a - 2:a - 1], ch)
                    p, e = hot.predict([g], background, rec)
                    assert np.array_equal(dp[gi][j], p) and np.array_equal(de[gi][j], e), (gi, j)
                    t0 = sum(len(x.tissues) for x in genes[:gi])
                    if not (app[gi]["cre"][j].any() or app[gi]["gene"][j]):      # a no-op is exactly the baseline
                        assert np.array_equal(p, base_p[t0:t0 + len(p)]) and np.array_equal(e, base_e[t0:t0 + len(e)])
                assert not app[gi]["cre"][-1 if gi != 1 else -2].any() and not app[gi]["gene"][-1]   # the no-ops
                assert app[gi]["cre"][0].sum() >= 1 and app[gi]["gene"][3]
        assert c["deletions"] == sum(len(s) for s in spans) and c["items"] == c["deletions"] + len(genes)
        assert c["windows_encoded"] < c["windows_per_item"]
        assert runs[0][4][1]["cre"][-1, -1]                    # the chr2 deletion changed the chr2 CRE window only
        assert not runs[0][4][1]["gene"][-1]
        # without embeddings: the same predictions and baselines
        pred, emb, dp, app = deletion.deletion_scan(hot, genes, spans, background, chs, rows_budget=30)
        assert np.array_equal(pred, base_p) and np.array_equal(emb, base_e)
        assert all(np.array_equal(a, b) for a, b in zip(dp, runs[0][2]))


def test_validation_runs_before_any_stage1(monkeypatch):
    chroms, _, genes = _world()
    hot = _FakeHot(chroms)

    def boom(*a, **k):
        raise AssertionError("stage 1 ran")
    monkeypatch.setattr(hot, "tokenize", boom)
    for bad in ([[1, 4]], [[9, 8]], [[10, 40_001]]):
        with pytest.raises(ValueError):
            deletion.deletion_scan(hot, genes, [np.zeros((0, 2))] * 2 + [np.asarray(bad)])


def test_short_gene_window_is_a_value_error(monkeypatch):
    monkeypatch.setattr(deletion.ism, "_pool", _fake_pool)
    monkeypatch.setattr(deletion, "_encode_edits", _fake_encode_edits)
    monkeypatch.setattr(deletion.ops, "bpe_tokenize", _fake_bpe)
    chroms, _, genes = _world()
    hot = _FakeHot(chroms)
    g = genes[0]
    g0, g1 = gene_window(g.start, g.end, g.strand, UP, DOWN)
    ran = []
    monkeypatch.setattr(hot.engine, "run_pooled", lambda *a, **k: ran.append(1))
    with pytest.raises(ValueError, match="less than 1000bp"):
        deletion.deletion_scan(hot, [g], [np.array([[g0 + 2, g1 - 500]])], min_gene_len=1000)
    assert not ran


def test_frame_columns_changed_flags_and_join():
    m = pd.DataFrame({"chromosome": ["chr2"] * 3, "start_cre": [100, 300, 200], "end_cre": [150, 390, 260],
                      "cre_name": [REF_CREs[i] for i in (0, 1, 2)]})
    spans, ch = deletion.default_spans(m)
    app = dict(cre=np.array([[1, 0, 0, 0], [0, 0, 0, 0], [0, 1, 1, 0]], bool), gene=np.array([False, False, True]))
    base = np.array([1.0, 2.0], np.float32)
    dp = np.array([[1.5, 2.0], [1.0, 2.0], [0.5, -1.0]], np.float32)
    df = deletion.deletion_frame("G1", ["thyroid", "whole blood"], [0, 1, 2], spans, ch, app, base, dp, m)
    assert list(df.columns) == deletion.FRAME_COLUMNS and len(df) == 6
    assert df["deletion"].tolist() == [0, 0, 1, 1, 2, 2] and df["tissue"].tolist() == ["thyroid", "whole blood"] * 3
    assert df["del_start"].tolist()[::2] == [101, 301, 201] and df["width"].tolist()[::2] == [50, 90, 60]
    assert df["cre_windows_changed"].tolist()[::2] == [1, 0, 2] and df["gene_window_changed"].tolist()[::2] == [0, 0, 1]
    assert df["changed"].tolist()[::2] == [True, False, True]
    assert np.array_equal(df["delta"].to_numpy(), (dp - base).reshape(-1))
    assert np.array_equal(df["baseline_expression"].to_numpy(), np.tile(base, 3))
    assert df.loc[df["changed"] == False, "delta"].eq(0).all()                      # noqa: E712
    # joins with cre_knockout's frame on (gene, tissue, CRE)
    ko = knockout.knockout_frame("G1", ["thyroid", "whole blood"], m, [(i, np.array([i])) for i in range(3)], base,
                                 np.zeros((3, 2), np.float32))
    keys = ["gene_id", "tissue", "chromosome", "start_cre", "end_cre", "cre_name"]
    j = df.merge(ko, on=keys, suffixes=("_del", "_ko"))
    assert len(j) == 6 and (j["deletion"] == j["knockout"]).all()
    # user deletions: the manifest columns are null
    u = deletion.deletion_frame("G1", ["thyroid"], ["t0"], np.array([[5, 9]]), ["chr2"],
                                dict(cre=np.zeros((1, 3), bool), gene=np.zeros(1, bool)), base[:1], dp[:1, :1])
    assert u["start_cre"].isna().all() and u["cre_name"].isna().all() and u["width"].tolist() == [5]
    empty = deletion.deletion_frame("G2", ["thyroid"], [], np.zeros((0, 2)), [],
                                    dict(cre=np.zeros((0, 3), bool), gene=np.zeros(0, bool)), base[:1],
                                    np.zeros((0, 1), np.float32))
    assert list(empty.columns) == deletion.FRAME_COLUMNS and len(empty) == 0
