"""Host logic of variant sets across a cohort (variantformer_b200.cohort_sets): the planner against HotPath.variant_sets
run on each sample alone (on the fake encoder and engine of the deletion and variant-set host tests, with fake genotype
keys that collide) under several slab and pass splits, the exact counters of a small cohort with a blocked record, the
per-sample error restatement, validation before any kernel, and cohort_summary's arithmetic.  CPU only."""
import numpy as np
import pandas as pd
import pytest
import torch

from tests.test_deletion_host import CW, L, _FakeHot, _Rows, _fake_bpe, _tok_rows, _world
from tests.test_knockout_host import _fake_pool
from tests.test_variant_sets_host import _fake_encode_sets, _rec, _scan_sets, _with_records
from variantformer_b200 import cohort_sets, ism, knockout, ops, variant_sets as vs
from variantformer_b200.pipeline import GeneSpec
from variantformer_b200.stage1 import CohortVariants, cre_window, gene_window
from variantformer_b200.variant_sets import Record


def _lists(w0, w1, lo, hi, flags, vdev, e_off, e_pos, e_rl, e_ao, e_al, e_gt, e_pool):
    """The merged rule restated per row: -> [(applied records (pos, ref_len, gt, alt), applied extra indices)]."""
    h = {k: t.numpy() for k, t in vdev.items()}
    pool, epool = h["alt_pool"].tobytes(), e_pool.numpy().tobytes()
    w0, w1, lo, hi, flags = (t.numpy() for t in (w0, w1, lo, hi, flags))
    off, pos, rl, ao, al, gt = (t.numpy() for t in (e_off, e_pos, e_rl, e_ao, e_al, e_gt))
    out = []
    for r in range(len(w0)):
        bg = [(int(h["pos"][i]), int(h["ref_len"][i]), int(h["gt"][i]),
               pool[h["alt_off"][i]:h["alt_off"][i] + h["alt_len"][i]], None) for i in range(lo[r], hi[r])]
        merged, i = [], 0
        for k in range(off[r], off[r + 1]):                 # an extra goes after the background records of pos <= its own
            while i < len(bg) and bg[i][0] <= pos[k]:
                merged.append(bg[i]); i += 1
            merged.append((int(pos[k]), int(rl[k]), int(gt[k]), epool[ao[k]:ao[k] + al[k]], k))
        merged += bg[i:]
        cur, lst, app = w0[r], [], []
        for p, n, g, a, k in merged:
            if g == 0 or p < cur or p + n > w1[r] or (flags[r] & 2 and not (n == 1 and len(a) == 1)):
                continue
            cur = p + n
            lst.append((p, n, g, a))
            if k is not None:
                app.append(k)
        out.append((lst, app))
    return out


def _fake_keys(*a, key_bits=128, err=None):
    rows = _lists(*a)
    ids = {}
    keys = torch.tensor([[ids.setdefault(tuple(x), len(ids)) % 3 if x else 0, 0] for x, _ in rows], dtype=torch.int64)
    applied = torch.zeros(int(a[6][-1]), dtype=torch.uint8)
    for _, app in rows:
        applied[app] = 1
    lens = torch.tensor([int(a[1][r] - a[0][r]) + sum(len(x[3]) - x[1] for x in lst) for r, (lst, _) in enumerate(rows)],
                        dtype=torch.int32)
    return keys, torch.tensor([len(x) for x, _ in rows], dtype=torch.int32), lens, applied, torch.zeros(1, dtype=torch.int32)


def _fake_equal(*a):
    *args, rep = a
    rows = _lists(*args)
    w0, w1, fl = args[0].numpy(), args[1].numpy(), args[4].numpy()
    return torch.tensor([int(rows[r][0] == rows[q][0] and w0[r] == w0[q] and w1[r] == w1[q] and (fl[r] ^ fl[q]) & 3 == 0)
                         for r, q in enumerate(rep.tolist())], dtype=torch.int32)


def _fake_encode(genome, win_base, *a):
    """vf_encode_windows_edits on the merged rule with hom ALTs (the bytes the variant-set host tests' encoder builds)."""
    *args, max_window, pitch = a
    g, base = genome.numpy().tobytes(), win_base.numpy()
    w0, w1, fl = args[0].numpy(), args[1].numpy(), args[4].numpy()
    seqs, applied = _Rows([], pitch), torch.zeros(int(args[6][-1]), dtype=torch.uint8)
    for r, (lst, app) in enumerate(_lists(*args)):
        out, x = bytearray(), int(w0[r])
        for p, n, _, alt in lst:
            out += g[base[r] + x:base[r] + p]; out += alt; x = p + n
        out += g[base[r] + x:base[r] + w1[r]]
        seqs.append(bytes(out[::-1]) if fl[r] & 1 else bytes(out))
        applied[app] = 1
    return seqs, torch.tensor([len(x) for x in seqs], dtype=torch.int32), applied, torch.zeros(1, dtype=torch.int32)


class _CohortHot(_FakeHot):
    def tokenize_chunked(self, seq, lens, max_len):
        out = []
        for s in seq:
            t, n = _tok_rows([s], L * CW)
            G = min(CW, (int(n[0]) + L - 1) // L)
            out.append((t[0, :G * L].view(G, L), None))
        return out, None


@pytest.fixture
def fakes(monkeypatch):
    monkeypatch.setattr(ism, "_pool", _fake_pool)
    monkeypatch.setattr(vs, "_encode_sets", _fake_encode_sets)
    monkeypatch.setattr(ops, "bpe_tokenize", _fake_bpe)
    monkeypatch.setattr(ops, "window_genotype_keys_edits", _fake_keys)
    monkeypatch.setattr(ops, "window_genotype_equal_edits", _fake_equal)
    monkeypatch.setattr(ops, "encode_windows_edits", _fake_encode)


def _sample(d):
    """A per-sample dict as CohortVariants takes it (hom-alt calls)."""
    return {c: dict(pos=np.asarray(v["pos"], np.int64), ref_len=np.asarray(v["ref_len"], np.int32), alt=list(v["alt"]),
                    gt=np.full(len(v["pos"]), 2, np.uint8)) for c, v in d.items()}


def _check(hot, genes, sets, per, got, embeddings=True):
    """Every sample's outputs against HotPath.variant_sets (vs.scan) on that sample alone."""
    pred, emb, sp = got[:3]
    se, app = (got[3], got[4]) if embeddings else (None, got[3])
    for s, d in enumerate(per):
        want = vs.scan(hot, genes, sets, d, embeddings=True)
        assert np.array_equal(pred[s], want[0]) and np.array_equal(emb[s], want[1]), s
        for gi in range(len(genes)):
            assert np.array_equal(sp[gi][s], want[2][gi]), (s, gi)
            if embeddings:
                assert np.array_equal(se[gi][s], want[3][gi]), (s, gi)
            for k in ("cre", "gene"):
                assert np.array_equal(app[gi][k][s], want[4][gi][k]), (s, gi, k)
            for j in range(len(sets[gi])):
                assert np.array_equal(app[gi]["records"][j][s], want[4][gi]["records"][j]), (s, gi, j)


def test_planner_equals_variant_sets_on_each_sample(fakes):
    chroms, var, genes = _world()
    hot = _CohortHot(chroms)
    sets = _scan_sets(chroms, genes)
    checked = vs.check_sets(genes, sets, hot.genome)
    a = checked[0][0][0]                                      # gene 0's first record: sample 3 carries it (blocked)
    rng = np.random.default_rng(9)
    thin = {c: {k: (np.asarray(v[k])[keep] if k != "alt" else [x for x, m in zip(v[k], keep) if m]) for k in v}
            for c, v in var.items() for keep in [rng.random(len(v["pos"])) < 0.5]}
    carrier, _ = _with_records({c: v for c, v in thin.items()}, [a])
    per = [_sample(var), {}, _sample(thin), _sample(carrier), _sample(var)]      # sample 4 repeats sample 0
    cv = CohortVariants([f"S{i}" for i in range(len(per))], per, "cpu")
    runs = []
    for budget, pass_rows in ((ism.ROWS_BUDGET, None), (1, 1), (30, 40)):
        hot.engine.slab_rows = []
        c = {}
        runs.append(cohort_sets.scan(hot, genes, sets, cv, embeddings=True, rows_budget=budget, pass_rows=pass_rows,
                                     counters=c))
        assert all(sum(r) <= budget or len(r) == 1 for r in hot.engine.slab_rows)
        if budget == 1:                                       # pass_rows 1: one (gene, sample) per pass
            assert c["passes"] == len(genes) * len(per)
        assert c["items"] == len(per) * sum(1 + len(s) for s in sets)
        assert c["items_scored"] <= c["items"] - sum(1 + len(s) for s in sets)      # sample 4 scores nothing new
        _check(hot, genes, sets, per, runs[-1])
    for r in runs[1:]:
        for k in (0, 1):
            assert np.array_equal(r[k], runs[0][k])
    # the set made of a record sample 3 carries: not applied there, and its prediction is sample 3's baseline
    app = runs[0][4][0]
    assert not app["records"][0][3].any() and app["records"][0][[0, 1, 2]].all()
    T0 = len(genes[0].tissues)
    assert np.array_equal(runs[0][2][0][3, 0], runs[0][0][3, :T0])
    # the restated per-item path for one sample with records added
    for j, s in enumerate(checked[0][:4]):
        p, _ = hot.predict([genes[0]], _with_records(per[2], list(s))[0])
        assert np.array_equal(runs[0][2][0][2, j], p)
    # without embeddings: the same predictions, only the baselines' embeddings
    lean = cohort_sets.scan(hot, genes, sets, cv)
    assert len(lean) == 4 and np.array_equal(lean[1], runs[0][1])
    assert all(np.array_equal(x, y) for x, y in zip(lean[2], runs[0][2]))


def test_counters_of_a_small_cohort_with_a_blocked_record(fakes):
    rng = np.random.default_rng(4)
    chroms = {"chr1": rng.choice(np.frombuffer(b"ACGT", np.uint8), 40_000).tobytes()}
    hot = _CohortHot(chroms)
    # two CREs far from the gene window [19 900, 25 500)
    g = GeneSpec("chr1", 20_000, 22_500, "+", np.array([5_000, 6_000]), np.array([5_200, 6_300]), np.array([1, 2]), [62])
    a = _rec(chroms, "chr1", 5_000)                           # in CRE window 0
    b = _rec(chroms, "chr1", 21_000)                          # in the gene window
    far = _rec(chroms, "chr1", 30_000)                        # in no window
    rec = lambda r: {"chr1": dict(pos=np.array([r.pos - 1]), ref_len=np.array([len(r.ref)], np.int32),
                                  alt=[r.alt.encode()], gt=np.array([r.gt], np.uint8))}
    per = [{}, rec(a), rec(far)]                              # sample 1 carries a; sample 2 encodes as sample 0
    cv = CohortVariants(["s0", "s1", "s2"], per, "cpu")
    c = {}
    out = cohort_sets.scan(hot, [g], [[[a], [b], [a, b]]], cv, counters=c)
    # CRE window 0: {no record}, {a} (sample 1's baseline and every sample's edit, a blocked in sample 1);
    # CRE window 1: {no record}; gene window: {no record}, {b} (edited rows only)
    assert (c["cre_groups"], c["gene_groups"], c["windows_encoded"], c["edited_groups"]) == (3, 2, 5, 1)
    assert c["sample_windows"] == 9 and c["passes"] == 1
    # items: s0 = base, a, b, ab; s1 = base (== s0's a), a (blocked: == its base), b (== s0's ab), ab (== its b);
    # s2 = s0's
    assert (c["items"], c["items_scored"]) == (12, 4)
    assert c["changed"] == 3 + 2 + 3
    app = out[3][0]
    assert app["records"][0][:, 0].tolist() == [True, False, True]
    assert app["records"][2].tolist() == [[True, True], [False, True], [True, True]]
    assert np.array_equal(out[2][0][1, 0], out[0][1]) and np.array_equal(out[2][0][1, 2], out[2][0][1, 1])
    assert np.array_equal(out[0][1], out[2][0][0, 0]) and np.array_equal(out[2][0][1, 1], out[2][0][0, 2])
    _check(hot, [g], [[[a], [b], [a, b]]], per, out, embeddings=False)


def test_errors_are_the_first_failing_samples_own(fakes):
    chroms, _, genes = _world()
    hot = _CohortHot(chroms)
    g = genes[0]
    g0 = gene_window(g.start, g.end, g.strand, hot.up, hot.down)[0]
    p = g0 + 2_000
    ins = Record("chr1", p + 1, chroms["chr1"][p:p + 1].decode(), chroms["chr1"][p:p + 1].decode() + "A" * 4_500)
    # sample a: a background deletion covering the insertion's POS blocks it; sample b: the edited gene window passes
    # the per-item pitch
    dele = {"chr1": dict(pos=np.array([p - 2]), ref_len=np.array([5], np.int32), alt=[chroms["chr1"][p - 2:p - 1]],
                         gt=np.array([2], np.uint8))}
    per = [dele, {}]
    cv = CohortVariants(["a", "b"], per, "cpu")
    sets = [[[ins]]]
    assert vs.scan(hot, [g], sets, per[0]) is not None
    with pytest.raises(RuntimeError) as want:
        vs.scan(hot, [g], sets, per[1], gene_names=["G"])
    with pytest.raises(RuntimeError) as got:
        cohort_sets.scan(hot, [g], sets, cv, gene_names=["G"])
    assert str(got.value) == f"sample b: {want.value}" and "edited window of gene G" in str(got.value)
    # the gene-window length rule: every sample fails it, the first in cohort order is named
    ok = [[[_rec(chroms, "chr1", p)]]]
    with pytest.raises(ValueError) as want:
        vs.scan(hot, [g], ok, per[0], min_gene_len=10_000, gene_names=["G"])
    with pytest.raises(ValueError) as got:
        cohort_sets.scan(hot, [g], ok, cv, min_gene_len=10_000, gene_names=["G"])
    assert str(got.value) == f"sample a: {want.value}"


def test_validation_comes_before_any_kernel(monkeypatch):
    chroms, _, genes = _world()
    hot = _FakeHot(chroms)
    boom = lambda *a, **k: (_ for _ in ()).throw(AssertionError("a kernel ran"))
    for name in ("window_genotype_keys_edits", "window_genotype_equal_edits", "encode_windows_edits"):
        monkeypatch.setattr(ops, name, boom)
    ref = chroms["chr1"][99:100].decode()
    alt = "T" if ref != "T" else "G"
    cases = [([[Record("chr1", 100, ref, alt, 5)]], "GT"), ([[Record("chrX", 100, "A", "C")]], "not in the genome"),
             ([[]], "empty"), ([[Record("chr1", 100, "N" if ref != "N" else "A", alt)]], "not the genome's")]
    for s, msg in cases:
        with pytest.raises(ValueError, match=msg):
            cohort_sets.scan(hot, genes[:1], [s], cohort_variants=None)
    with pytest.raises(ValueError, match="2 entries for 1 genes"):
        cohort_sets.scan(hot, genes[:1], [[], []], cohort_variants=None)


def test_cohort_summary_arithmetic():
    rows = []
    deltas = {("G", "s1", "lung"): [0.5, -1.0, 2.0], ("G", "s1", "thyroid"): [0.0, 0.0, 0.0],
              ("H", "s2", "lung"): [1.25, 3.0, -0.5]}
    for (gid, sid, t), ds in deltas.items():
        for k, x in enumerate(ds):
            rows.append({"sample": f"S{k}", "gene_id": gid, "tissue": t, "set": sid, "n_records": 1,
                         "records_applied": int(x != 0), "cre_windows_changed": 0, "gene_window_changed": x != 0,
                         "changed": x != 0, "baseline_expression": np.float32(1.0),
                         "predicted_expression": np.float32(1.0 + x), "delta": np.float32(x)})
    frame = pd.DataFrame(rows)[["sample"] + vs.SET_COLUMNS]
    s = vs.cohort_summary(frame)
    assert list(s.columns) == vs.SUMMARY_COLUMNS and len(s) == 3
    assert [tuple(r) for r in s[["gene_id", "set", "tissue"]].to_numpy()] == list(deltas)
    for (_, r), ds in zip(s.iterrows(), deltas.values()):
        x = np.asarray(ds, np.float64)
        assert r["n_samples"] == 3 and r["n_changed"] == int((x != 0).sum())
        assert r["mean_delta"] == x.mean() and r["sd_delta"] == x.std(ddof=0)
        assert r["min_delta"] == x.min() and r["max_delta"] == x.max()
    assert s["mean_delta"].dtype == np.float64 and s["n_changed"].dtype == np.int64
