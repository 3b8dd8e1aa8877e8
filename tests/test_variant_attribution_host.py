"""Host logic of variant attribution (variantformer_b200.variant_attribution): the override walk of
vf_encode_windows_overrides restated against "delete the line or rewrite the GT, then walk the plain rule", record
resolution and its errors, the windows an edit can change and the default / per-window scans, the planner against a
per-item restatement on the fake encoder and engine of the deletion tests (slab and pass splits, a no-op edit sharing the
baseline's rows, the all-removed set equal to the reference genome), and frame assembly.  CPU only."""
import numpy as np
import pandas as pd
import pytest
import torch

import tests.test_deletion_host as dh
from tests.test_deletion_host import NB, UP, DOWN, _FakeHot, _Rows, _fake_bpe, _world, applied_records
from tests.test_knockout_host import _fake_pool
from variantformer_b200 import ism, knockout, variant_attribution as va, variant_sets as vs
from variantformer_b200.pipeline import GeneSpec
from variantformer_b200.stage1 import SampleVariants, cre_window, gene_window
from variantformer_b200.variant_attribution import Edit

IUPAC = {frozenset("AC"): "M", frozenset("AG"): "R", frozenset("AT"): "W", frozenset("CG"): "S", frozenset("CT"): "Y",
         frozenset("GT"): "K"}


def override_walk(pos, ref_len, alt_len, gt, lo, hi, w0, w1, o_idx, o_gt, snp_only=False):
    """OverrideScan restated: records [lo, hi) in index order, each record's gt read through the sorted override list by
    a two-pointer merge.  -> [(index, gt applied with)]."""
    out, cur, k = [], w0, 0
    for i in range(lo, hi):
        g = gt[i]
        if k < len(o_idx) and o_idx[k] == i:
            g = o_gt[k]; k += 1
        p, rl, al = pos[i], ref_len[i], alt_len[i]
        if g == 0 or p < cur or p + rl > w1 or (snp_only and not (rl == 1 and al == 1)):
            continue
        cur = p + rl
        out.append((i, g))
    return out


def encode_gt(chrom, w0, w1, var, extra=None, rc=False):
    """The encoder's bytes of a window with genotypes: het SNP -> IUPAC, hom SNP and any indel -> ALT (the reverse
    complement as a plain reversal suffices for the fake tokenizer).  -> (bytes, False)."""
    pos, rl, alt = var["pos"], var["ref_len"], var["alt"]
    gt = var.get("gt", np.full(len(pos), 2))
    out, x = bytearray(), w0
    for i in applied_records(pos, rl, [len(a) for a in alt], gt, w0, w1):
        a = alt[i]
        if rl[i] == 1 and len(a) == 1 and gt[i] == 1:
            r, b = chr(chrom[pos[i]]).upper(), chr(a[0]).upper()
            a = IUPAC.get(frozenset(r + b), "N").encode() if r in "ACGT" and b in "ACGT" and r != b else b"N"
        out += chrom[x:pos[i]]; out += a; x = pos[i] + rl[i]
    out += chrom[x:w1]
    return (bytes(out[::-1]) if rc else bytes(out)), False


def _table(variants, ch):
    """A SampleVariants chromosome as the fake encoder's dict."""
    return dict(pos=variants.host_pos[ch], ref_len=variants.host_ref_len[ch], alt=list(variants.host_alt[ch]),
                gt=variants.host_gt[ch])


class _AttrHot(_FakeHot):
    def _var(self, variants, ch):
        if isinstance(variants, SampleVariants):
            return _table(variants, ch) if ch in variants.ranges else super()._var(None, ch)
        return super()._var(variants, ch)


def _edited(variants, recs):
    """SampleVariants with the planner records' GTs replaced."""
    d = {ch: dict(pos=variants.host_pos[ch], ref_len=variants.host_ref_len[ch], alt=list(variants.host_alt[ch]),
                  gt=variants.host_gt[ch].copy()) for ch in variants.ranges}
    for r in recs:
        d[r[0]]["gt"][r[5] - variants.ranges[r[0]][0]] = r[4]
    return SampleVariants(d, "cpu")


def _fake_encode_overrides(hot, variants, rows, pitch):
    seqs = _Rows([], pitch)
    for ch, w0, w1, fl, recs in rows:
        t = _table(_edited(variants, recs), ch)
        seqs.append(encode_gt(hot.genome.chroms[ch], w0, w1, t, None, bool(fl & 1))[0])
    n = sum(len(r[4]) for r in rows)
    return seqs, torch.tensor([len(s) for s in seqs], dtype=torch.int32), torch.zeros(n, dtype=torch.uint8), \
        torch.zeros(1, dtype=torch.int32)


@pytest.fixture
def fakes(monkeypatch):
    monkeypatch.setattr(vs.ism, "_pool", _fake_pool)
    monkeypatch.setattr(va, "_encode_overrides", _fake_encode_overrides)
    monkeypatch.setattr(vs.ops, "bpe_tokenize", _fake_bpe)
    monkeypatch.setattr(dh, "encode", encode_gt)


def _sample(chroms, var, seed=1):
    """The deletion tests' background with GTs (0, 1, 2) and a few records sharing a POS."""
    rng = np.random.default_rng(seed)
    d = {}
    for ch, v in var.items():
        pos = np.asarray(v["pos"], np.int64).copy()
        dup = rng.choice(len(pos), len(pos) // 20, replace=False)
        pos = np.sort(np.concatenate([pos, pos[dup]]))
        rl = np.where(rng.random(len(pos)) < 0.2, rng.integers(2, 6, len(pos)), 1)
        alt = [bytes([b"ACGT"[int(rng.integers(0, 4))]]) if rl[k] == 1 and rng.random() < 0.7 else
               rng.choice(np.frombuffer(b"ACGT", np.uint8), int(rng.integers(1, 4))).tobytes() for k in range(len(pos))]
        gt = rng.choice([0, 1, 2], len(pos), p=[0.1, 0.5, 0.4]).astype(np.uint8)
        d[ch] = dict(pos=pos, ref_len=rl, alt=alt, gt=gt)
    return SampleVariants(d, "cpu"), d


def test_override_walk_equals_the_edited_table():
    rng = np.random.default_rng(5)
    for trial in range(300):
        n = int(rng.integers(0, 60))
        pos = np.sort(rng.integers(0, 400, n))
        if n and trial % 3 == 0:
            pos[n // 2:n // 2 + 3] = pos[n // 2]                # records at one POS
            pos = np.sort(pos)
        rl = np.where(rng.random(n) < 0.3, rng.integers(2, 30, n), 1)
        al = np.where(rng.random(n) < 0.3, rng.integers(2, 6, n), 1)
        gt = rng.integers(0, 3, n)
        w0 = int(rng.integers(0, 100)); w1 = w0 + int(rng.integers(50, 350))
        lo, hi = int(np.searchsorted(pos, w0)), int(np.searchsorted(pos, w1))
        k = int(rng.integers(0, min(9, hi - lo) + 1))
        o_idx = np.sort(rng.choice(np.arange(lo, hi), k, replace=False)) if k else np.zeros(0, np.int64)
        o_gt = rng.integers(0, 3, k)
        snp = trial % 5 == 0
        got = override_walk(pos, rl, al, gt, lo, hi, w0, w1, o_idx, o_gt, snp_only=snp)
        # the edited table: GT rewritten, GT-0 lines deleted
        g2 = gt.copy(); g2[o_idx] = o_gt
        keep = np.flatnonzero(g2 != 0)
        want = [(int(keep[i]), int(g2[keep[i]])) for i in
                applied_records(pos[keep], rl[keep], al[keep], g2[keep], w0, w1, snp_only=snp)]
        assert got == want, trial


def test_check_edits_resolves_records_and_raises():
    chroms, var, genes = _world()
    sv, d = _sample(chroms, var)
    g = genes[0]
    c1 = d["chr1"]
    i = int(np.flatnonzero(c1["gt"] != 0)[5])
    e = Edit("chr1", int(c1["pos"][i]) + 1, "N" * int(c1["ref_len"][i]), c1["alt"][i].decode().lower(), 1)
    got = va.check_edits([g], [[[e]]], sv)[0][0]
    assert got == (("chr1", int(c1["pos"][i]), int(c1["ref_len"][i]), c1["alt"][i], 1, i),)
    j = i + 3
    e2 = Edit("chr1", int(c1["pos"][j]) + 1, "N" * int(c1["ref_len"][j]), c1["alt"][j].decode(), 0)
    two = va.check_edits([g], [[[e2, e]]], sv)[0][0]
    assert [r[5] for r in two] == [i, j]                       # table order
    # an ambiguous match: two identical lines at one POS
    amb = {"chr1": dict(pos=[10, 10], ref_len=[1, 1], alt=[b"A", b"A"], gt=[1, 2])}
    sv2 = SampleVariants(amb, "cpu")
    cases = [(sv, [Edit("chr1", e.pos, e.ref, "T" if e.alt.upper() != "T" else "G", 0)], "carries no such record"),
             (sv, [e._replace(ref=e.ref + "N")], "carries no such record"),
             (sv, [e._replace(chrom="chr9")], "carries no such record"),
             (sv, [e._replace(gt=3)], "GT"), (sv, [e._replace(gt=True)], "GT"), (sv, [e._replace(gt=-1)], "GT"),
             (sv, [e, e._replace(gt=2)], "twice"), (sv, [], "empty"),
             (sv2, [Edit("chr1", 11, "N", "A", 0)], "ambiguous"), (None, [e], "carries no such record")]
    for v, s, msg in cases:
        with pytest.raises(ValueError, match=msg):
            va.check_edits([g], [[s]], v, ["G"])
    with pytest.raises(ValueError, match="no CRE"):
        va.check_edits([GeneSpec("chr1", 1, 2, "+", np.zeros(0), np.zeros(0), np.zeros(0), [1])], [[[e]]], sv)
    # validation comes before any stage 1
    hot = _AttrHot(chroms)
    hot.tokenize = lambda *a, **k: (_ for _ in ()).throw(AssertionError("stage 1 ran"))
    with pytest.raises(ValueError, match="GT"):
        va.scan(hot, [g], [[[e._replace(gt=7)]]], sv)


def test_window_records_and_default_scans():
    chroms, var, genes = _world()
    sv, d = _sample(chroms, var)
    for g in genes:
        win = vs._windows(g, NB, UP, DOWN)
        per = va.window_records(g, sv, NB, UP, DOWN)
        assert len(per) == len(win)
        for (ch, w0, w1), recs in zip(win, per):
            t, base = d.get(ch), sv.ranges.get(ch, (0, 0))[0]
            want = [] if t is None else [(ch, base + k) for k in range(len(t["pos"])) if
                                         w0 <= t["pos"][k] and t["pos"][k] + t["ref_len"][k] <= w1 and t["gt"][k] != 0]
            assert recs == want
        sets, labels, gts = va.default_sets(g, sv, NB, UP, DOWN, "record")
        uniq = sorted({r for w in per for r in w}, key=lambda r: r[1])
        assert [s[0][5] for s in sets] == [i for _, i in uniq] and all(len(s) == 1 and s[0][4] == 0 for s in sets)
        assert all(x != 0 for x in gts) and len(labels) == len(sets)
        ref = va.all_removed(g, sv, NB, UP, DOWN)
        assert [r[5] for r in ref] == [s[0][5] for s in sets]
        ws, wl, wg = va.default_sets(g, sv, NB, UP, DOWN, "window")
        order = knockout.batch_order(g)
        assert wl == [f"cre_window:{int(order[k])}" if k < len(win) - 1 else "gene_window"
                      for k, w in enumerate(per) if w]
        assert [[r[5] for r in s] for s in ws] == [[i for _, i in w] for w in per if w] and wg == [None] * len(ws)
    with pytest.raises(ValueError, match="scope"):
        va.default_sets(genes[0], sv, NB, UP, DOWN, "gene")
    assert va.window_records(genes[0], None, NB, UP, DOWN) == [[]] * len(vs._windows(genes[0], NB, UP, DOWN))


def _edit_sets(sv, d, genes):
    """Per gene: leave-one-out of a few records, a window revert, a het <-> hom rewrite of an indel (a no-op), a record
    re-genotyped from 0, a blocker removed and the all-removed set."""
    out = []
    for g in genes:
        loo, _, _ = va.default_sets(g, sv, NB, UP, DOWN, "record")
        ws, _, _ = va.default_sets(g, sv, NB, UP, DOWN, "window")
        sets = loo[::max(1, len(loo) // 6)] + ws[:2]
        ind = [r for s in loo for r in s if r[2] > 1]
        if ind:                                                # het <-> hom of an indel: the same bytes
            r = ind[0]
            sets.append(((*r[:4], 3 - va.sample_gt(sv, r), r[5]),))
        c1, base = d["chr1"], sv.ranges["chr1"][0]
        z = [k for k in np.flatnonzero(c1["gt"] == 0) if any(w[0] == "chr1" and w[1] <= c1["pos"][k] and
                                                               c1["pos"][k] + c1["ref_len"][k] <= w[2]
                                                               for w in vs._windows(g, NB, UP, DOWN))]
        if z:                                                  # a line of GT 0 made hom-alt
            sets.append((va._record(sv, "chr1", base + int(z[0]), 2),))
        sets.append(va.all_removed(g, sv, NB, UP, DOWN))
        out.append(sets)
    return out


def test_planner_equals_the_per_item_restatement(fakes):
    chroms, var, genes = _world()
    sv, d = _sample(chroms, var)
    hot = _AttrHot(chroms)
    sets = _edit_sets(sv, d, genes)
    runs = []
    for budget, pass_rows in ((ism.ROWS_BUDGET, None), (1, 1), (30, 40)):
        hot.engine.slab_rows = []
        c = {}
        runs.append(va.run(hot, genes, sets, sv, embeddings=True, rows_budget=budget, pass_rows=pass_rows, counters=c))
        assert all(sum(r) <= budget or len(r) == 1 for r in hot.engine.slab_rows)
        assert c["items"] == sum(len(s) + 1 for s in sets) and c["windows_encoded"] < c["windows_per_item"]
    base_p, base_e = hot.predict(genes, sv)
    ref_p, ref_e = hot.predict(genes, None)
    n_unchanged = 0
    for pred, emb, sp, se, ch in runs:
        assert np.array_equal(pred, base_p) and np.array_equal(emb, base_e)
        t0 = 0
        for gi, g in enumerate(genes):
            T = len(g.tissues)
            for j, s in enumerate(sets[gi]):
                p, e = hot.predict([g], _edited(sv, s))
                assert np.array_equal(sp[gi][j], p) and np.array_equal(se[gi][j], e), (gi, j)
                changed = ch[gi]["cre"][j].any() or ch[gi]["gene"][j]
                assert changed == ch[gi]["records"][j].any()
                if not changed:                                # shares the baseline's rows: exactly the baseline
                    n_unchanged += 1
                    assert np.array_equal(p, base_p[t0:t0 + T]) and np.array_equal(sp[gi][j], base_p[t0:t0 + T])
            # the all-removed set is the reference genome
            assert np.array_equal(sp[gi][-1], ref_p[t0:t0 + T]) and np.array_equal(se[gi][-1], ref_e[t0:t0 + T])
            t0 += T
    assert n_unchanged > 0                                     # the het <-> hom indel rewrites
    for r in runs[1:]:
        assert all(np.array_equal(x, y) for x, y in zip(r[2], runs[0][2]))
        assert all(np.array_equal(x["cre"], y["cre"]) and np.array_equal(x["gene"], y["gene"])
                   for x, y in zip(r[4], runs[0][4]))


def test_changed_windows_follow_the_tokens(fakes):
    """A removed record changes exactly the windows that hold it and apply it; a blocked record changes nothing until
    its blocker goes."""
    chroms = {"chr1": np.random.default_rng(3).choice(np.frombuffer(b"ACGT", np.uint8), 40_000).tobytes()}
    g = GeneSpec("chr1", 10_000, 12_500, "+", np.array([8_000, 20_000]), np.array([8_300, 20_200]), np.array([1, 2]),
                 [62])
    w = [cre_window(s, e, NB) for s, e in zip(g.cre_start, g.cre_end)]
    p0 = w[0][0] + 40
    # a 10-base deletion, a SNP it blocks, and a SNP in the other CRE window
    sv = SampleVariants({"chr1": dict(pos=[p0, p0 + 5, w[1][0] + 10], ref_len=[10, 1, 1], alt=[b"A", b"T", b"G"],
                                      gt=[2, 2, 1])}, "cpu")
    hot = _AttrHot(chroms)
    base = sv.ranges["chr1"][0]
    rec = lambda i, gt=0: va._record(sv, "chr1", base + i, gt)
    sets = [[(rec(1),), (rec(0),), (rec(2),), (rec(0), rec(1))]]
    pred, emb, sp, ch = va.run(hot, [g], sets, sv)
    k0 = list(knockout.batch_order(g)).index(0)
    assert not ch[0]["cre"][0].any() and not ch[0]["gene"][0]          # the blocked SNP: a no-op
    assert np.array_equal(sp[0][0], pred)
    assert ch[0]["cre"][1, k0] and ch[0]["cre"][1].sum() == 1        # the blocker removed
    assert ch[0]["cre"][2].sum() == 1 and not ch[0]["cre"][2, k0]
    assert ch[0]["records"][3].all()
    g0, g1 = gene_window(g.start, g.end, g.strand, UP, DOWN)
    assert not (g0 <= p0 < g1)


def test_user_edits_and_frame():
    df = pd.DataFrame({"gene_id": ["G", "G", "H"], "chromosome": ["chr1"] * 3, "pos": [5, 9, np.int64(7)],
                       "ref": ["A", "C", "G"], "alt": ["T", "G", "A"], "gt": [0, 1, 2]})
    u = va.user_edits(df)
    assert list(u) == ["G", "H"] and [s[0] for s in u["G"]] == ["chr1:5:A>T", "chr1:9:C>G"]
    assert u["G"][1][1] == [Edit("chr1", 9, "C", "G", 1)]
    u2 = va.user_edits(df.assign(set=["s", "s", "t"], label=["x", None, "z"]))
    assert u2["G"][0][0] == "s" and u2["G"][0][1] == [Edit("chr1", 5, "A", "T", 0), Edit("chr1", 9, "C", "G", 1)]
    with pytest.raises(ValueError, match="gt"):
        va.user_edits(df.drop(columns=["gt"]))
    base = np.array([1.0, 2.0], np.float32)
    sp = np.array([[1.5, 2.0], [0.5, 4.0]], np.float32)
    ref = np.array([0.25, 3.0], np.float32)
    sets = [(("chr1", 4, 1, b"T", 0, 7),), (("chr1", 4, 1, b"T", 0, 7), ("chr1", 8, 1, b"G", 1, 9))]
    ch = dict(cre=np.array([[1, 0], [0, 0]], bool), gene=np.array([False, True]),
              records=[np.array([True]), np.array([False, True])])
    f = va.attribution_frame("G", ["thyroid", "lung"], ["a", "b"], sets, [2, None], ch, base, sp, ref)
    assert list(f.columns) == va.ATTRIBUTION_COLUMNS and len(f) == 4
    assert f["sample_gt"].tolist() == [2, 2, pd.NA, pd.NA] or f["sample_gt"].isna().tolist() == [False, False, True, True]
    assert f["sample_gt"].iloc[0] == 2 and f["new_gt"].iloc[1] == 0 and f["new_gt"].isna().tolist()[2:] == [True, True]
    assert np.array_equal(f["delta"].to_numpy(), (sp - base).reshape(-1))
    assert np.array_equal(f["reference_expression"].to_numpy(), np.tile(ref, 2))
    assert f["n_records"].tolist() == [1, 1, 2, 2] and f["changed"].tolist() == [True] * 4
    assert f["records_applied"].tolist() == [1, 1, 1, 1]
