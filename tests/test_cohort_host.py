"""Host logic of cohort prediction (variantformer_b200.cohort, stage1.CohortVariants) with fake keys: window tables,
grouping, item deduplication, pass and slab partitions.  CPU only."""
import numpy as np
import torch

from variantformer_b200 import cohort
from variantformer_b200.pipeline import GeneSpec
from variantformer_b200.stage1 import CohortVariants, SampleVariants, cre_window, gene_window
from variantformer_b200.utils import synth


def _per_sample(rng, n_samples=17, length=200_000):
    chrom = synth.make_chromosome(rng, length)
    out = []
    for s in range(n_samples):
        d = {}
        if s != 3:                                           # sample 3 carries no variant
            for c in ("chr1", "chr2") if s % 2 else ("chr2",):
                d[c] = synth.make_variants(rng, chrom, rate=1 / 300)
        out.append(d)
    return out


def test_window_ranges_equal_each_samples_ranges():
    rng = np.random.default_rng(3)
    per = _per_sample(rng)
    cv = CohortVariants([f"S{i}" for i in range(len(per))], per, "cpu")
    rows = [(s, c, int(a), int(a) + int(w)) for s in range(len(per)) for c in ("chr1", "chr2", "chr9")
            for a, w in zip(rng.integers(0, 190_000, 40), rng.integers(1, 9_000, 40))]
    lo, hi = cv.window_ranges([r[0] for r in rows], [r[1] for r in rows], [r[2] for r in rows], [r[3] for r in rows])
    pos = cv.dev["pos"].numpy()
    for (s, c, a, b), l, h in zip(rows, lo, hi):
        sv = SampleVariants(per[s], "cpu")
        l1, h1 = sv.window_range(c, a, b)
        assert h - l == h1 - l1, (s, c, a, b)
        if h > l:
            assert np.array_equal(pos[l:h], sv.dev["pos"].numpy()[l1:h1])
            assert np.array_equal(cv.dev["alt_len"].numpy()[l:h], sv.dev["alt_len"].numpy()[l1:h1])
    # the ALT bytes of a record follow its offset in the concatenated pool
    al, ao, pool = cv.dev["alt_len"].numpy(), cv.dev["alt_off"].numpy(), cv.dev["alt_pool"].numpy().tobytes()
    flat = [a for d in per for c in cv.chroms if c in d for a in d[c]["alt"]]
    assert [pool[o:o + k] for o, k in zip(ao, al)] == flat


def test_blocks_respect_the_index_limit():
    rng = np.random.default_rng(4)
    per = _per_sample(rng, n_samples=9)
    names = [f"S{i}" for i in range(9)]
    sizes = [CohortVariants.sizes([d]) for d in per]
    limit = max(max(r, a) for r, a in sizes) * 2 + 1
    blocks = CohortVariants.blocks(per, limit=limit)
    assert [x for a, b in blocks for x in range(a, b)] == list(range(9)) and len(blocks) > 1
    for a, b in blocks:
        r, x = CohortVariants.sizes(per[a:b])
        assert (r <= limit and x <= limit) or b - a == 1
    assert CohortVariants.blocks(per) == [(0, 9)]


def test_gene_windows_count_shared_windows_once():
    rng = np.random.default_rng(5)
    lay = synth.make_gene_layout(rng, 3_000_000, 12, strand="+", body_len=20_000, cre_span=50_000)
    g = GeneSpec("chr1", lay["start"], lay["end"], "+", lay["cre_start"], lay["cre_end"], lay["labels"], [1])
    g2 = GeneSpec("chr1", lay["start"] + 10, lay["end"], "+", lay["cre_start"][::-1].copy(), lay["cre_end"][::-1].copy(),
                  lay["labels"][::-1].copy(), [1, 2])
    gm = GeneSpec("chr1", lay["start"], lay["end"], "-", lay["cre_start"], lay["cre_end"], lay["labels"], [0])
    w = cohort.gene_windows([g, g2, gm])
    assert len(w.cre) == 24 and len(w.gene) == 3                 # the minus strand's windows are other windows
    assert np.array_equal(w.cre_of[0], w.cre_of[1]) and np.array_equal(w.labels[0], w.labels[1])
    order = np.argsort(lay["cre_start"], kind="stable")
    assert [w.cre[k][1:3] for k in w.cre_of[0]] == [cre_window(lay["cre_start"][i], lay["cre_end"][i], 50) for i in order]
    assert [w.cre[k][1:3] for k in w.cre_of[2]] == [cre_window(lay["cre_start"][i], lay["cre_end"][i], 50)
                                                   for i in order[::-1]]
    assert w.gene[w.gene_of[2]] == ("chr1",) + gene_window(g.start, g.end, "-", 1000, 300000) + (1,)


def test_group_rows_with_fake_keys():
    rng = np.random.default_rng(6)
    W, S = 7, 16
    window = torch.arange(W * S) // S
    keys = torch.from_numpy(rng.integers(0, 3, (W * S, 2))).long()
    count = torch.from_numpy(rng.integers(0, 2, W * S)).int()
    keys[count == 0] = 0
    group, rep = cohort.group_rows(window, count, keys)
    g, r = group.numpy(), rep.numpy()
    # one group = one (window, count, key); its representative is its first row; groups never cross windows
    for i in range(W * S):
        j = r[g[i]]
        assert j <= i and window[j] == window[i] and count[j] == count[i] and torch.equal(keys[j], keys[i])
    sig = {(int(window[i]), int(count[i]), int(keys[i, 0]), int(keys[i, 1])) for i in range(W * S)}
    assert len(r) == len(sig) and sorted(set(g.tolist())) == list(range(len(r)))
    # deterministic
    g2, r2 = cohort.group_rows(window, count, keys)
    assert torch.equal(group, g2) and torch.equal(rep, r2)
    # the exact comparison splits: rejected rows become groups of their own, in row order, after the others
    reject = torch.zeros(W * S, dtype=torch.bool)
    reject[[5, 40, 41]] = True
    reject[r[g[5]]] = False                                  # a representative always equals itself
    g3, r3 = cohort.group_rows(window, count, keys, lambda rep_of: ~reject)
    bad = torch.nonzero(reject).ravel().numpy()
    assert g3.numpy()[bad].tolist() == list(range(len(r), len(r) + len(bad)))
    assert r3.numpy()[len(r):].tolist() == bad.tolist()
    keep = ~reject.numpy()
    assert np.array_equal(g3.numpy()[keep], g[keep])


def test_items_passes_and_slabs_cover_everything_once():
    rng = np.random.default_rng(7)
    items = []
    for _ in range(300):
        k = int(rng.integers(0, 6))
        items.append((np.arange(k, k + 5), np.arange(k % 2, k % 2 + 3), (1, 2) if k < 4 else (3,), np.zeros(5, np.int64)))
    uniq, of = cohort.dedup_items(items)
    assert len(uniq) == 6 and sorted(uniq.tolist()) == uniq.tolist()
    for i, it in enumerate(items):
        u = items[uniq[of[i]]]
        assert np.array_equal(u[0], it[0]) and np.array_equal(u[1], it[1]) and u[2] == it[2]
    # labels are part of an item
    lab = [(np.arange(3), np.arange(2), (1,), np.asarray([0, 1, 2])), (np.arange(3), np.arange(2), (1,), np.asarray([0, 1, 3]))]
    assert len(cohort.dedup_items(lab)[0]) == 2
    rows = rng.integers(1, 3000, 97).tolist()
    for budget in (1, 2500, 16384, 1 << 30):
        sl = cohort.slab_ranges(rows, budget)
        assert [x for a, b in sl for x in range(a, b)] == list(range(97))
        assert all(b - a == 1 or sum(rows[a:b]) <= budget for a, b in sl)
    # passes: every (gene, sample) exactly once, in gene order; a pass stays under max(2 pass_rows, one sample's rows
    # of one gene) for any number of samples
    S = 37
    per_sample = rng.integers(1, 400, 97)
    rows = (per_sample * rng.integers(1, S + 1, 97)).tolist()        # a gene's rows grow with the samples that differ
    for pass_rows in (1, 500, 5000, 1 << 30):
        ps = cohort.plan_passes(rows, pass_rows, S, per_sample)
        seen = [(g, s) for a, b, s0, s1 in ps for g in range(a, b) for s in range(s0, s1)]
        assert sorted(seen) == [(g, s) for g in range(97) for s in range(S)] and len(seen) == 97 * S
        assert [a for a, _, _, _ in ps] == sorted(a for a, _, _, _ in ps)
        for a, b, s0, s1 in ps:
            if (s0, s1) != (0, S):                               # a gene split by samples
                assert b - a == 1 and rows[a] > pass_rows and (s1 - s0 == 1 or (s1 - s0) * per_sample[a] <= pass_rows)
            else:
                assert sum(rows[a:b]) < 2 * pass_rows or b - a == 1
    assert cohort.plan_passes([10, 10], 5, 1) == [(0, 1, 0, 1), (1, 2, 0, 1)]
    assert cohort.plan_passes([], 10) == [] and cohort.slab_ranges([], 10) == []
