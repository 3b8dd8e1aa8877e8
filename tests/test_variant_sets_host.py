"""Host logic of in-silico variant combinations (variantformer_b200.variant_sets): the planner's items against a
per-item restatement on the fake encoder and engine of the deletion and knockout tests (slab and pass splits, with and
without a background), the exact encode count of a pair scan, records on another chromosome's CRE, validation
messages, pairs() and the frames' arithmetic.  CPU only."""
import numpy as np
import pandas as pd
import pytest
import torch

from tests.test_deletion_host import (NB, UP, DOWN, _FakeHot, _Rows, _fake_bpe, _world, applied_records,
                                      encode)
from tests.test_knockout_host import _fake_pool
from variantformer_b200 import ism, knockout, variant_sets as vs
from variantformer_b200.pipeline import GeneSpec
from variantformer_b200.stage1 import cre_window, gene_window
from variantformer_b200.variant_sets import Record


def _with_records(var, recs):
    """The background dict with records (chrom, pos0, ref_len, alt bytes, gt) inserted after every record of pos <= their
    own, in list order.  -> (per-chromosome dict, {record index: its index in its chromosome's table})."""
    out = {k: dict(pos=list(v["pos"]), ref_len=list(v["ref_len"]), alt=list(v["alt"])) for k, v in (var or {}).items()}
    at = {}
    for n, (ch, p, rl, alt, _) in enumerate(recs):
        d = out.setdefault(ch, dict(pos=[], ref_len=[], alt=[]))
        k = int(np.searchsorted(np.asarray(d["pos"], np.int64), p, "right"))
        d["pos"].insert(k, p); d["ref_len"].insert(k, rl); d["alt"].insert(k, alt)
        at = {m: (i + 1 if i >= k and recs[m][0] == ch else i) for m, i in at.items()}
        at[n] = k
    return {k: dict(pos=np.asarray(v["pos"], np.int64), ref_len=np.asarray(v["ref_len"], np.int64), alt=v["alt"])
            for k, v in out.items()}, at


def _fake_encode_sets(hot, variants, rows, pitch):
    seqs, app = _Rows([], pitch), []
    for ch, w0, w1, fl, recs in rows:
        v, at = _with_records({ch: hot._var(variants, ch)}, list(recs))
        s, _ = encode(hot.genome.chroms[ch], w0, w1, v[ch], None, bool(fl & 1))
        idx = applied_records(v[ch]["pos"], v[ch]["ref_len"], [len(a) for a in v[ch]["alt"]], np.full(len(v[ch]["pos"]), 2),
                              w0, w1)
        seqs.append(s); app += [at[m] in idx for m in range(len(recs))]
    return seqs, torch.tensor([len(s) for s in seqs], dtype=torch.int32), torch.tensor(app, dtype=torch.uint8), \
        torch.zeros(1, dtype=torch.int32)


@pytest.fixture
def fakes(monkeypatch):
    monkeypatch.setattr(vs.ism, "_pool", _fake_pool)
    monkeypatch.setattr(vs, "_encode_sets", _fake_encode_sets)
    monkeypatch.setattr(vs.ops, "bpe_tokenize", _fake_bpe)


def _rec(chroms, ch, pos0, ref_len=1, alt=None, gt=2):
    ref = chroms[ch][pos0:pos0 + ref_len].decode()
    if alt is None:
        alt = "T" if ref[0] != "T" else "G"
    return Record(ch, pos0 + 1, ref, alt, gt)


def _scan_sets(chroms, genes):
    """Per gene: singles, a cross-window pair, a same-window pair, a CRE + gene-window pair, a 3-record haplotype with an
    insertion and a deletion, a set on the chr2 CRE (gene 1) and a set far from every window (a no-op)."""
    out = []
    for gi, g in enumerate(genes):
        o = knockout.batch_order(g)
        w = [cre_window(g.cre_start[i], g.cre_end[i], NB) for i in o]
        g0, g1 = gene_window(g.start, g.end, g.strand, UP, DOWN)
        a = _rec(chroms, "chr1", w[0][0] + 10)
        b = _rec(chroms, "chr1", w[0][0] + 30, 3, "C")                  # same CRE window as a (a deletion)
        c = _rec(chroms, "chr1", w[-1][0] + 15, 1, "ACGT")              # another CRE window (an insertion)
        d = _rec(chroms, "chr1", g0 + 900)                              # the gene window
        e = _rec(chroms, "chr1", g0 + 1_400, 2, "A", gt=1)
        far = _rec(chroms, "chr1", 3)
        sets = [[a], [b], [c], [d], [a, c], [a, b], [c, d], [e, d, a], [far]]
        if gi == 1:
            sets.append([_rec(chroms, "chr2", 5_010), a])
        out.append(sets)
    return out


@pytest.mark.parametrize("background", [False, True])
def test_planner_items_equal_the_per_item_restatement(fakes, background):
    chroms, var, genes = _world()
    var = var if background else None
    hot = _FakeHot(chroms)
    sets = _scan_sets(chroms, genes)
    checked = vs.check_sets(genes, sets, hot.genome)
    runs = []
    for budget, pass_rows in ((ism.ROWS_BUDGET, None), (1, 1), (30, 40)):
        hot.engine.slab_rows = []
        c = {}
        runs.append(vs.scan(hot, genes, sets, var, embeddings=True, rows_budget=budget, pass_rows=pass_rows, counters=c))
        assert all(sum(r) <= budget or len(r) == 1 for r in hot.engine.slab_rows)
        if budget == 1:
            assert c["passes"] == len(genes)
        assert c["items"] == sum(len(s) + 1 for s in sets) and c["windows_encoded"] < c["windows_per_item"]
    base_p, base_e = hot.predict(genes, var)
    for pred, emb, sp, se, app in runs:
        assert np.array_equal(pred, base_p) and np.array_equal(emb, base_e)
        t0 = 0
        for gi, g in enumerate(genes):
            T = len(g.tissues)
            assert sp[gi].shape == (len(sets[gi]), T)
            for j, s in enumerate(checked[gi]):
                p, e = hot.predict([g], _with_records(var, list(s))[0])
                assert np.array_equal(sp[gi][j], p) and np.array_equal(se[gi][j], e), (gi, j)
                changed = app[gi]["cre"][j].any() or app[gi]["gene"][j]
                assert changed == app[gi]["records"][j].any()
                if not changed:
                    assert np.array_equal(p, base_p[t0:t0 + T])
            assert not app[gi]["records"][8].any() and not app[gi]["cre"][8].any()      # the far set: a no-op
            assert app[gi]["gene"][3] and app[gi]["records"][7].all()
            t0 += T
    for r in runs[1:]:
        assert all(np.array_equal(x, y) for x, y in zip(r[2], runs[0][2]))
    # the chr2 record changes the chr2 CRE window only (the last one in gene 1's batch order)
    app = runs[0][4][1]
    assert app["cre"][9, -1] and app["records"][9].all()


def test_pair_scan_encodes_singles_and_same_window_pairs_only(fakes):
    chroms, var, genes = _world()
    hot = _FakeHot(chroms)
    g = genes[0]
    o = knockout.batch_order(g)
    w = [cre_window(g.cre_start[i], g.cre_end[i], NB) for i in o]
    g0, _ = gene_window(g.start, g.end, g.strand, UP, DOWN)
    # 3 records in CRE window 0 (which may overlap others), 1 in the last CRE window, 2 in the gene window
    recs = [_rec(chroms, "chr1", w[0][0] + d) for d in (5, 40, 80)] + [_rec(chroms, "chr1", w[-1][0] + 7)] + \
           [_rec(chroms, "chr1", g0 + d) for d in (600, 1_700)]
    sets, singles, pair_idx, overlapping = vs.pairs(recs)
    assert singles == list(range(6)) and len(pair_idx) == 15 and not overlapping
    c1, c2 = {}, {}
    vs.scan(hot, [g], [sets[:6]], var, counters=c1)
    vs.scan(hot, [g], [sets], var, counters=c2)
    win = vs._windows(g, NB, UP, DOWN)
    inside = lambda r, k: win[k][0] == r.chrom and win[k][1] <= r.pos - 1 and r.pos - 1 + len(r.ref) <= win[k][2]
    same = sum(1 for i, j in pair_idx for k in range(len(win)) if inside(recs[i], k) and inside(recs[j], k))
    assert same >= 3 + 1                                       # the CRE-window pairs and the gene-window pair
    assert c2["windows_encoded"] == c1["windows_encoded"] + same
    assert c2["items"] == 1 + 6 + 15
    assert vs.shared_window(g, vs.check_sets([g], [sets], hot.genome)[0][6:], NB, UP, DOWN).sum() == \
        sum(1 for i, j in pair_idx if any(inside(recs[i], k) and inside(recs[j], k) for k in range(len(win))))


def test_validation_messages():
    chroms, _, genes = _world()
    hot = _FakeHot(chroms)
    g = genes[0]
    ok = _rec(chroms, "chr1", 100)
    low = _rec(chroms, "chr1", 500, 2, "a")                    # REF and ALT in lower case
    assert vs.check_sets([g], [[[ok, low._replace(ref=low.ref.lower())]]], hot.genome)[0][0][1][3] == b"a"
    n = len(chroms["chr1"])
    cases = [([Record("chrX", 5, "A", "C")], "not in the genome"),
             ([Record("chr1", 0, "A", "C")], "outside chr1"),
             ([Record("chr1", n, chroms["chr1"][n - 1:].decode() + "A", "C")], "outside chr1"),
             ([Record("chr1", 100, "N" if chroms["chr1"][99:100] != b"N" else "A", "C")], "not the genome's"),
             ([Record("chr1", ok.pos, ok.ref, "")], "ALT"), ([Record("chr1", ok.pos, ok.ref, "<DEL>")], "ALT"),
             ([Record("chr1", ok.pos, ok.ref, "*")], "ALT"), ([Record("chr1", ok.pos, ok.ref, "AXG")], "ALT"),
             ([Record("chr1", ok.pos, ok.ref, ok.ref.lower())], "equals REF"),
             ([Record("chr1", ok.pos, ok.ref, ok.alt, 0)], "GT"), ([Record("chr1", ok.pos, ok.ref, ok.alt, 3)], "GT"),
             ([], "empty"),
             ([_rec(chroms, "chr1", 200, 5, "A"), _rec(chroms, "chr1", 203)], "overlap"),
             ([ok, Record("chr1", ok.pos, ok.ref, "A" if ok.ref != "A" else "C")], "overlap")]
    for s, msg in cases:
        with pytest.raises(ValueError, match=msg):
            vs.check_sets([g], [[s]], hot.genome, ["G"])
    with pytest.raises(ValueError, match="no CRE"):
        vs.check_sets([GeneSpec("chr1", 1, 2, "+", np.zeros(0), np.zeros(0), np.zeros(0), [1])], [[[ok]]], hot.genome)
    with pytest.raises(ValueError, match="2 entries for 1 genes"):
        vs.check_sets([g], [[], []], hot.genome)
    # validation comes before any stage 1
    hot.tokenize = lambda *a, **k: (_ for _ in ()).throw(AssertionError("stage 1 ran"))
    with pytest.raises(ValueError, match="GT"):
        vs.scan(hot, [g], [[[Record("chr1", ok.pos, ok.ref, ok.alt, 5)]]])
    # records of a set come in (POS, given order)
    c = vs.check_sets([g], [[[_rec(chroms, "chr1", 300), _rec(chroms, "chr1", 100, 2, "A")]]], hot.genome)[0][0]
    assert [r[1] for r in c] == [100, 300] and c[0][2] == 2 and c[0][3] == b"A"


def test_pairs_and_user_records():
    a, b = Record("chr1", 100, "A", "C"), Record("chr1", 100, "A", "G")       # two alleles of one site
    d, e = Record("chr1", 99, "TA", "T"), Record("chr2", 100, "A", "T")       # d's REF covers 99-100
    f = Record("chr1", 101, "C", "T")
    sets, singles, pair_idx, overlapping = vs.pairs([a, b, d, e, f])
    assert singles == [0, 1, 2, 3, 4] and sets[:5] == [[a], [b], [d], [e], [f]]
    assert overlapping == [(0, 1), (0, 2), (1, 2)]
    assert pair_idx == [(0, 3), (0, 4), (1, 3), (1, 4), (2, 3), (2, 4), (3, 4)]
    assert [sets[5 + k] for k in range(len(pair_idx))] == [[[a, b, d, e, f][i], [a, b, d, e, f][j]] for i, j in pair_idx]
    df = pd.DataFrame({"gene_id": ["G", "G", "H"], "set": ["s1", "s1", "s2"], "chromosome": ["chr1"] * 3,
                       "pos": [5, 9, np.int64(7)], "ref": ["A", "C", "G"], "alt": ["T", "G", "A"], "gt": [1, 2, 2]})
    u = vs.user_records(df)
    assert list(u) == ["G", "H"] and u["G"][0][0] == "s1" and u["G"][0][1] == [Record("chr1", 5, "A", "T", 1),
                                                                               Record("chr1", 9, "C", "G", 2)]
    assert u["G"][0][2] == ["chr1:5:A>T", "chr1:9:C>G"]
    u2 = vs.user_records(df.drop(columns=["set", "gt"]).assign(label=["x", None, "z"]), sets=False)
    assert u2["G"][1] == ["x", "chr1:9:C>G"] and u2["G"][0][1].gt == 2
    with pytest.raises(ValueError, match="missing"):
        vs.user_records(df.drop(columns=["set"]))
    with pytest.raises(ValueError, match="not an integer"):
        vs.user_records(df.assign(pos=[1.5, 2.0, 3.0]))


def test_frames_arithmetic():
    base = np.array([1.0, 2.0], np.float32)
    single = np.array([[1.5, 2.0], [0.5, 4.0], [1.0, 1.0]], np.float32)
    pair = np.array([[2.0, 4.0], [1.0, 1.0], [0.25, 0.5]], np.float32)
    df = vs.interaction_frame("G", ["thyroid", "lung"], ["a", "b", "c"], [(0, 1), (0, 2), (1, 2)],
                              [True, False, False], base, single, pair)
    assert list(df.columns) == vs.INTERACTION_COLUMNS and len(df) == 6
    assert df["variant_a"].tolist() == ["a", "a", "a", "a", "b", "b"] and df["same_window"].tolist() == [True] * 2 + [False] * 4
    ea, eb = single[[0, 0, 1]], single[[1, 2, 2]]
    want = (pair - base) - (ea - base) - (eb - base)
    assert np.array_equal(df["interaction"].to_numpy(), want.reshape(-1))
    assert np.array_equal(df["delta_ab"].to_numpy(), (pair - base).reshape(-1))
    f = lambda x: x.astype(np.float64) + 1e-10                 # in float64, as saturation mutagenesis' log2fc
    l2 = np.log2(f(pair) * f(base) / (f(ea) * f(eb)))
    assert np.allclose(df["log2_interaction"].to_numpy(), l2.reshape(-1), rtol=0, atol=1e-12)
    assert df["log2_interaction"].iloc[0] == pytest.approx(np.log2(2.0 * 1.0 / (1.5 * 0.5)))
    app = dict(cre=np.array([[1, 0], [0, 0]], bool), gene=np.array([False, True]),
               records=[np.array([True, False]), np.array([True])])
    sf = vs.set_frame("G", ["thyroid", "lung"], ["s1", "s2"], [2, 1], app, base, pair[:2])
    assert list(sf.columns) == vs.SET_COLUMNS and sf["records_applied"].tolist() == [1, 1, 1, 1]
    assert sf["n_records"].tolist() == [2, 2, 1, 1] and sf["changed"].all()
    assert np.array_equal(sf["delta"].to_numpy(), (pair[:2] - base).reshape(-1))
