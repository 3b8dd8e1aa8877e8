"""Host logic of in-silico CRE knockout (variantformer_b200.knockout): batch positions on both strands, validation, the
planner's items against a per-item restatement on a fake engine (passes, slabs, labels), the pitch rule and the
processor's frame.  CPU only."""
import numpy as np
import pandas as pd
import pytest
import torch

from variantformer_b200 import ism, knockout
from variantformer_b200.pipeline import GeneSpec
from variantformer_b200.utils.constants import REF_CREs

L = 4


def _gene(strand, n=9, seed=0, tissues=(62,)):
    rng = np.random.default_rng(seed)
    start = rng.integers(10_000, 20_000, n)
    if n >= 7:
        start[[1, 4, 6]] = start[2]                                   # tied starts
    return GeneSpec("chr1", 15_000, 40_000, strand, start, start + rng.integers(100, 900, n), rng.integers(0, 9, n),
                    list(tissues))


def _reduced(g, knocked):
    keep = np.setdiff1d(np.arange(len(g.cre_start)), knocked)
    return GeneSpec(g.chrom, g.start, g.end, g.strand, g.cre_start[keep], g.cre_end[keep], g.cre_labels[keep],
                    list(g.tissues))


@pytest.mark.parametrize("strand", ["+", "-"])
def test_kept_positions_are_the_reduced_genes_batch_order(strand):
    g = _gene(strand)
    order = knockout.batch_order(g)
    want = np.argsort(g.cre_start, kind="stable")                     # HotPath.tokenize's rule
    assert np.array_equal(order, want[::-1] if strand == "-" else want)
    rng = np.random.default_rng(1)
    for ko in [[0], [2], [8], [1, 4, 6], [2, 4], list(rng.choice(9, 5, replace=False))]:
        keep = knockout.kept_positions(order, ko)
        r = _reduced(g, ko)
        # the manifest rows at the kept positions, in order, are the reduced gene's batch order (as manifest rows)
        rows_left = np.setdiff1d(np.arange(9), ko)
        assert np.array_equal(order[keep], rows_left[knockout.batch_order(r)])
        assert np.array_equal(np.asarray(g.cre_labels)[order[keep]], np.asarray(r.cre_labels)[knockout.batch_order(r)])


def test_validation_errors():
    g, h = _gene("+"), _gene("-", n=1)
    assert [s.tolist() for s in knockout.check_knockouts([g])[0]] == [[i] for i in range(9)]
    assert knockout.check_knockouts([h]) == [[]]                       # one CRE: nothing to knock out by default
    ok = knockout.check_knockouts([g], [[np.array([5, 1]), [3], np.int32(7)]])[0]
    assert [s.tolist() for s in ok] == [[1, 5], [3], [7]]
    for sets, msg in (([[]], "empty"), ([[9]], "outside the manifest"), ([[-1]], "outside the manifest"),
                      ([[2, 3, 2]], "repeats CRE index 2"), ([list(range(9))], "removes every CRE"),
                      ([[1.0]], "non-integer")):
        with pytest.raises(ValueError, match=msg):
            knockout.check_knockouts([g], [sets])
    with pytest.raises(ValueError, match="knockout 'enh' of gene G"):
        knockout.check_knockouts([g], [[[9]]], ["G"], [["enh"]])
    with pytest.raises(ValueError, match="removes every CRE"):
        knockout.check_knockouts([h], [[[0]]])
    with pytest.raises(ValueError, match="2 entries for 1 genes"):
        knockout.check_knockouts([g], [[], []])
    with pytest.raises(ValueError, match="no CRE"):
        knockout.check_knockouts([_gene("+", n=0)])


def test_pitch_rule():
    # windows encoded together share the pitch of the longest span + 4096, rounded up to 16
    assert not knockout.overflows(np.array([100, 5000]), np.array([4196, 5000]))
    assert knockout.overflows(np.array([100]), np.array([4197 + 15]))
    assert not knockout.overflows(np.array([100]), np.array([4196 + 12]))     # (100 + 4096) rounds up to 4208
    assert not knockout.overflows(np.array([], np.int64), np.array([], np.int64))


class _FakeEngine:
    """Stand-in for the engine's shared-window interface: an item's prediction is an exact, order- and label-sensitive
    function of its pooled CRE rows, its gene chunks and its tissue, so the planner's items can be checked against
    the same function applied to the reduced gene's own windows."""
    device = torch.device("cpu")
    cre_tok = gene_tok = None

    class w:
        D = 3

    def __init__(self):
        self.slab_rows = []

    def prepare_shared(self, cre_rows, gene_rows, n_gene_chunks, tissues, ref_labels):
        self.slab_rows.append([len(r) for r in cre_rows])
        return dict(cre=cre_rows, gene=gene_rows, tis=tissues, lab=ref_labels)

    @staticmethod
    def score(cre_vec, gene_vec, labels, tissue):
        k = np.arange(1, len(cre_vec) + 1, dtype=np.float64)
        counts = np.bincount(labels, minlength=9)
        return np.array([(k * cre_vec).sum(), gene_vec.sum() + tissue, (k * labels).sum() + 0.5 * (counts == 0).sum()])

    def run_pooled(self, s, cre_pooled, gene_pooled):
        out = []
        for c, g, t, lab in zip(s["cre"], s["gene"], s["tis"], s["lab"]):
            for x in t.tolist():
                out.append(self.score(cre_pooled[c].numpy(), gene_pooled[g].numpy(), lab.numpy(), x))
        emb = torch.from_numpy(np.asarray(out))
        return {"pred": emb[:, 0] + emb[:, 1] + emb[:, 2], "emb": emb}


class _FakeHot:
    """HotPath's attributes and tokenize() contract with token rows derived from the windows."""
    nb, up, down, max_chunks = 50, 1000, 300000, 4

    def __init__(self):
        self.engine = _FakeEngine()

    def tokenize(self, genes, variants=None):
        ct, gt, labels, clen, glen = [], [], [], [], []
        for g in genes:
            o = knockout.batch_order(g)
            ct.append(torch.tensor([[int(g.cre_start[i]) % 97 + 1, int(g.cre_end[i]) % 89 + 1, 0, 0] for i in o],
                                   dtype=torch.int32).reshape(-1, L))
            gt.append(torch.tensor([[g.start % 7 + j + 1, 3, 0, 0] for j in range(3)], dtype=torch.int32))
            labels.append(torch.from_numpy(np.asarray(g.cre_labels)[o].copy()))
            clen += [int(g.cre_end[i] - g.cre_start[i]) + 100 for i in o]; glen.append(5000)
        return dict(cre_tok=ct, gene_tok=gt, labels=labels, err=torch.zeros((), dtype=torch.int32),
                    cre_seq=(None, torch.tensor(clen)), gene_seq=(None, torch.tensor(glen)))

    def predict(self, genes):
        """The per-item path restated on the fake engine."""
        t = self.tokenize(genes)
        out = [_FakeEngine.score(c.double().sum(1).numpy(), g.double().sum(1).numpy(), lab.numpy(), x)
               for c, g, lab, gn in zip(t["cre_tok"], t["gene_tok"], t["labels"], genes) for x in gn.tissues]
        emb = np.asarray(out)
        return emb.sum(1), emb


def _fake_pool(engine, W, tok):
    return tok.double().sum(1)


def test_planner_items_equal_the_per_item_restatement(monkeypatch):
    monkeypatch.setattr(knockout.ism, "_pool", _fake_pool)
    hot = _FakeHot()
    genes = [_gene("+", seed=2, tissues=(62,)), _gene("-", n=12, seed=3, tissues=(1, 2)), _gene("+", n=2, seed=4),
             _gene("-", n=5, seed=5, tissues=list(range(7)))]
    sets = [[[i] for i in range(9)], [[0], [11, 3], [1, 4, 6], list(range(1, 12))], [[1]], [[4, 0, 2]]]
    runs = []
    for budget, pass_rows in ((ism.ROWS_BUDGET, None), (1, 1), (20, 30)):
        hot.engine.slab_rows = []
        c = {}
        runs.append(knockout.cre_knockout(hot, genes, sets, embeddings=True, rows_budget=budget, pass_rows=pass_rows,
                                          counters=c))
        # every slab within the budget, or one item alone
        assert all(sum(r) <= budget or len(r) == 1 for r in hot.engine.slab_rows)
        if budget == 1:
            assert c["passes"] == len(genes) and all(len(r) == 1 for r in hot.engine.slab_rows)
    base_p, base_e = hot.predict(genes)
    off = np.concatenate([[0], np.cumsum([len(g.tissues) for g in genes])])
    for pred, emb, ko_pred, ko_emb in runs:
        assert np.array_equal(pred, base_p) and np.array_equal(emb, base_e)
        for gi, g in enumerate(genes):
            assert ko_pred[gi].shape == (len(sets[gi]), len(g.tissues))
            for k, s in enumerate(sets[gi]):
                p, e = hot.predict([_reduced(g, s)])
                assert np.array_equal(ko_pred[gi][k], p) and np.array_equal(ko_emb[gi][k], e), (gi, k)
            assert np.array_equal(emb[off[gi]:off[gi + 1]], base_e[off[gi]:off[gi + 1]])
    assert c["knockouts"] == sum(len(s) for s in sets) and c["items"] == c["knockouts"] + len(genes)
    assert c["windows_encoded"] < c["windows_per_item"]
    # without embeddings: the same predictions and baselines, three elements
    pred, emb, ko_pred = knockout.cre_knockout(hot, genes, sets, rows_budget=20)
    assert np.array_equal(pred, base_p) and np.array_equal(emb, base_e)
    assert all(np.array_equal(a, b) for a, b in zip(ko_pred, runs[0][2]))


def test_validation_runs_before_any_stage1(monkeypatch):
    hot = _FakeHot()

    def boom(*a, **k):
        raise AssertionError("stage 1 ran")
    monkeypatch.setattr(hot, "tokenize", boom)
    g = _gene("+")
    for sets in ([[[]]], [[[9]]], [[[3, 3]]], [[list(range(9))]]):
        with pytest.raises(ValueError):
            knockout.cre_knockout(hot, [g], sets)


def test_knockout_sets_keep_first_appearance_order():
    df = pd.DataFrame({"gene_id": ["A", "B", "A", "A", "B", "A"], "knockout": ["x", "p", "y", "x", "q", "z"],
                       "cre_index": [3, 0, 1, 5, 2, np.int64(4)]})
    s = knockout.knockout_sets(df)
    assert list(s) == ["A", "B"]
    assert [(lab, ix.tolist()) for lab, ix in s["A"]] == [("x", [3, 5]), ("y", [1]), ("z", [4])]
    assert [(lab, ix.tolist()) for lab, ix in s["B"]] == [("p", [0]), ("q", [2])]
    with pytest.raises(ValueError, match="cre_index"):
        knockout.knockout_sets(df.drop(columns="cre_index"))
    with pytest.raises(ValueError, match="not an integer"):
        knockout.knockout_sets(pd.DataFrame({"gene_id": ["A"], "knockout": ["x"], "cre_index": [1.5]}))


def test_frame_order_columns_delta_and_null_sets():
    m = pd.DataFrame({"chromosome": ["chr2"] * 4, "start_cre": [100, 300, 200, 50], "end_cre": [150, 390, 260, 90],
                      "cre_name": [REF_CREs[i] for i in (0, 1, 2, 3)]})
    sets = [(0, np.array([0])), (2, np.array([2])), ("pair", np.array([1, 3]))]
    base = np.array([1.0, 2.0], np.float32)
    ko = np.array([[1.5, 2.0], [0.25, 3.0], [1.0, -1.0]], np.float32)
    df = knockout.knockout_frame("G1", ["thyroid", "whole blood"], m, sets, base, ko)
    assert list(df.columns) == knockout.FRAME_COLUMNS and len(df) == 6
    assert df["knockout"].tolist() == [0, 0, 2, 2, "pair", "pair"]
    assert df["tissue"].tolist() == ["thyroid", "whole blood"] * 3
    assert df["cre_indices"].tolist() == [(0,), (0,), (2,), (2,), (1, 3), (1, 3)]
    assert df["start_cre"].tolist()[:4] == [100, 100, 200, 200] and df["start_cre"].isna().tolist()[4:] == [True, True]
    assert df["cre_name"].tolist()[:4] == [REF_CREs[0]] * 2 + [REF_CREs[2]] * 2 and df["cre_name"].isna().sum() == 2
    assert df["chromosome"].isna().sum() == 2 and df["end_cre"].tolist()[2] == 260
    assert np.array_equal(df["predicted_expression"].to_numpy(), ko.reshape(-1))
    assert np.array_equal(df["baseline_expression"].to_numpy(), np.tile(base, 3))
    assert np.array_equal(df["delta"].to_numpy(), (ko - base).reshape(-1))
    # joins with cre_attention's manifest columns on (gene, tissue, CRE)
    att = pd.DataFrame({"gene_id": "G1", "tissue": "thyroid", "chromosome": m["chromosome"], "start_cre": m["start_cre"],
                        "end_cre": m["end_cre"], "cre_name": m["cre_name"], "attention": [0.1, 0.2, 0.3, 0.4]})
    j = df.merge(att, on=["gene_id", "tissue", "chromosome", "start_cre", "end_cre", "cre_name"])
    assert sorted(j["attention"].tolist()) == [0.1, 0.3]
    empty = knockout.knockout_frame("G2", ["thyroid"], m, [], base[:1], np.zeros((0, 1), np.float32))
    assert list(empty.columns) == knockout.FRAME_COLUMNS and len(empty) == 0
