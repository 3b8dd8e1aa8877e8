"""Variant sets across a cohort on the B200: the genotype-key kernels with extra records against a restatement of the
merged rule and against vf_encode_windows_edits, HotPath.cohort_variant_sets bit for bit against HotPath.variant_sets on
every sample, its errors, and VCFProcessor.cohort_variant_sets against VCFProcessor.variant_sets on single-sample cuts."""
import numpy as np
import pandas as pd
import pytest
import torch

pytestmark = pytest.mark.gpu

from tests.test_gpu_cohort import N_SAMPLES, _applied, _cohort, _genes, _write_cohort_vcf  # noqa: E402
from tests.test_gpu_pipeline import CFG, HP, _write_artifacts  # noqa: E402
from variantformer_b200 import _lib, cohort as cohort_mod, engine as engine_mod, knockout, ops, variant_sets as vs  # noqa: E402
from variantformer_b200.cohort import group_rows  # noqa: E402
from variantformer_b200.engine import Engine  # noqa: E402
from variantformer_b200.pipeline import HotPath  # noqa: E402
from variantformer_b200.stage1 import CohortVariants, Genome, SampleVariants, cre_window, gene_window  # noqa: E402
from variantformer_b200.utils import random_init, synth  # noqa: E402
from variantformer_b200.variant_sets import Record  # noqa: E402

d = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dt)).cuda()


def _merged(v, lo, hi, extras):
    """The background records [lo, hi) of table v with `extras` ((pos, ref_len, gt, alt bytes), sorted by pos) inserted
    after every background record of pos <= their own, as one table (pos, rl, al, gt, off, pool) and each extra's
    index in it."""
    pos, rl, al, gt, off, pool = v
    bg = [(int(pos[i]), int(rl[i]), int(gt[i]), bytes(pool[off[i]:off[i] + al[i]])) for i in range(lo, hi)]
    out, at, i = [], [], 0
    for x in extras:
        while i < len(bg) and bg[i][0] <= x[0]:
            out.append(bg[i]); i += 1
        at.append(len(out)); out.append(x)
    out += bg[i:]
    p = b"".join(r[3] for r in out)
    ln = np.asarray([len(r[3]) for r in out], np.int64)
    return (np.asarray([r[0] for r in out], np.int64), np.asarray([r[1] for r in out], np.int64), ln,
            np.asarray([r[2] for r in out], np.int64), np.cumsum(ln) - ln, p), at


def _rows(rng, cv, chrom, W=240):
    """Windows x samples with 0-8 extras per row: SNVs and short indels, het and hom, at a background POS, inside a
    background deletion, adjacent to a background record, and at random places."""
    S = N_SAMPLES
    h = {k: t.cpu().numpy() for k, t in cv.dev.items()}
    w0 = rng.integers(0, 3_000_000 - 310_000, W)
    w1 = w0 + np.where(rng.random(W) < 0.1, 301_000, rng.integers(60, 6_000, W))
    fl = rng.integers(0, 4, W).astype(np.uint8)
    rs, rw0, rw1, rfl = np.tile(np.arange(S), W), np.repeat(w0, S), np.repeat(w1, S), np.repeat(fl, S)
    lo, hi = cv.window_ranges(rs, ["chr1"] * len(rs), rw0, rw1)
    extras = []
    for r in range(len(rs)):
        n = int(rng.integers(0, 9)) if rng.random() < 0.7 else 0
        cand = []
        for _ in range(n):
            u = rng.random()
            if hi[r] > lo[r] and u < 0.5:                           # at, inside or next to a background record
                i = int(rng.integers(lo[r], hi[r]))
                p = int(h["pos"][i]) + [0, 0, int(h["ref_len"][i]) // 2, int(h["ref_len"][i])][int(rng.integers(0, 4))]
            else:
                p = int(rng.integers(rw0[r], rw1[r]))
            rl = 1 if rng.random() < 0.7 else int(rng.integers(2, 6))
            alt = bytes(rng.choice(list(b"ACGT"), 1 if rng.random() < 0.6 else int(rng.integers(2, 7))).tolist())
            if p + rl > len(chrom):
                continue
            cand.append((p, rl, int(rng.integers(1, 3)), alt))
        extras.append(sorted(cand, key=lambda x: x[0]))
    return (rs, rw0, rw1, rfl, lo, hi), extras


def _csr(extras):
    n = [len(e) for e in extras]
    flat = [x for e in extras for x in e]
    al = np.asarray([len(x[3]) for x in flat], np.int64)
    return (d(np.concatenate([[0], np.cumsum(n)]), np.int32), d([x[0] for x in flat], np.int32),
            d([x[1] for x in flat], np.int32), d(np.cumsum(al) - al, np.int32), d(al, np.int32),
            d([x[2] for x in flat], np.uint8), d(np.frombuffer(b"".join(x[3] for x in flat), np.uint8), np.uint8))


def test_genotype_keys_edits_against_the_merged_rule_and_the_encoder():
    rng = np.random.default_rng(81)
    chrom = synth.make_chromosome(rng, 3_000_000)
    _, per = _cohort(rng, chrom, common_rate=1 / 150, private_rate=1 / 800)
    cv = CohortVariants([f"S{i}" for i in range(N_SAMPLES)], per, "cuda")
    genome = Genome.from_arrays({"chr1": chrom}, "cuda")
    (rs, rw0, rw1, rfl, lo, hi), extras = _rows(rng, cv, chrom)
    base = (d(rw0, np.int32), d(rw1, np.int32), d(lo, np.int32), d(hi, np.int32), d(rfl, np.uint8), cv.dev)
    e = _csr(extras)
    keys, count, lens, applied, err = ops.window_genotype_keys_edits(*base, *e)
    assert int(err.item()) == 0
    keys, count, lens, applied = keys.cpu().numpy(), count.cpu().numpy(), lens.cpu().numpy(), applied.cpu().numpy()
    # an empty list: the plain kernel's key, count and length bit for bit
    k0, c0, l0, _ = ops.window_genotype_keys(*base)
    empty = np.asarray([len(x) == 0 for x in extras])
    assert empty.sum() > 100
    assert np.array_equal(keys[empty], k0.cpu().numpy()[empty]) and np.array_equal(count[empty], c0.cpu().numpy()[empty])
    assert np.array_equal(lens[empty], l0.cpu().numpy()[empty])
    # the restated merged rule: equal lists <-> equal keys, blocked extras key as the row without them
    h = {k: t.cpu().numpy() for k, t in cv.dev.items()}
    v = (h["pos"], h["ref_len"], h["alt_len"], h["gt"], h["alt_off"], h["alt_pool"].tobytes())
    lists, app_want, blocked_rows = [], [], 0
    for r in range(len(rs)):
        m, at = _merged(v, lo[r], hi[r], extras[r])
        a = _applied((m[0], m[1], m[2], m[3], m[4], m[5]), 0, len(m[0]), rw0[r], rw1[r], rfl[r] & 2)
        lists.append(a)
        # which extras were applied: walk the rule once more, tracking indices
        cur, got = rw0[r], set()
        for i in range(len(m[0])):
            if m[3][i] == 0 or m[0][i] < cur or m[0][i] + m[1][i] > rw1[r] or (rfl[r] & 2 and not (m[1][i] == 1 and m[2][i] == 1)):
                continue
            got.add(i); cur = m[0][i] + m[1][i]
        app_want += [i in got for i in at]
        if extras[r] and not any(i in got for i in at):
            blocked_rows += 1
            assert tuple(keys[r]) == tuple(k0.cpu().numpy()[r]) and count[r] == c0.cpu().numpy()[r]
    assert blocked_rows > 20 and np.array_equal(applied.astype(bool), np.asarray(app_want, bool))
    by = {}
    for r, a in enumerate(lists):
        assert count[r] == len(a)
        by.setdefault((r // N_SAMPLES, a), set()).add(tuple(keys[r]))
    assert all(len(x) == 1 for x in by.values())
    assert len({(w, next(iter(k))) for (w, _), k in by.items()}) == len(by)
    # the encoder: same lengths and applied flags; groups (also with 4-bit keys) encode byte-identically
    mw = int((rw1 - rw0).max())
    out, out_len, app_enc, e2 = ops.encode_windows_edits(genome.seq, d(np.zeros(len(rs)), np.int64), *base, *e, mw,
                                                         knockout._pitch(mw))
    assert int(e2.item()) == 0 and np.array_equal(out_len.cpu().numpy(), lens)
    assert np.array_equal(app_enc.cpu().numpy(), applied)
    out = out.cpu().numpy()
    for bits in (128, 4):
        k, cnt, _, _, _ = ops.window_genotype_keys_edits(*base, *e, key_bits=bits)
        group, reps = group_rows(torch.arange(len(rs), device="cuda") // N_SAMPLES, cnt, k,
                                 lambda rp: ops.window_genotype_equal_edits(*base, *e, rp.to(torch.int32)) != 0)
        group, reps = group.cpu().numpy(), reps.cpu().numpy()
        for r in range(len(rs)):
            q = reps[group[r]]
            assert lists[q] == lists[r] and out[q, :lens[q]].tobytes() == out[r, :lens[r]].tobytes()
        assert len(reps) == len(by) if bits == 128 else len(reps) >= len(by)
    # the comparison against a random representative of the window
    rep = (np.arange(len(rs)) // N_SAMPLES) * N_SAMPLES + rng.integers(0, N_SAMPLES, len(rs))
    eq = ops.window_genotype_equal_edits(*base, *e, d(rep, np.int32)).cpu().numpy()
    assert np.array_equal(eq.astype(bool), np.asarray([lists[r] == lists[q] for r, q in enumerate(rep)]))


def test_genotype_keys_edits_errors_and_arguments():
    rng = np.random.default_rng(82)
    chrom = synth.make_chromosome(rng, 300_000)
    per = [{"chr1": dict(pos=np.arange(10_000, 10_000 + 3 * 2040, 3, dtype=np.int64), ref_len=np.ones(2040, np.int32),
                         alt=[b"A"] * 2040, gt=np.full(2040, 2, np.uint8))}, {}]
    cv = CohortVariants(["a", "b"], per, "cuda")
    genome = Genome.from_arrays({"chr1": chrom}, "cuda")
    w0, w1 = np.array([5_000, 5_000, 5_000]), np.array([40_000, 40_000, 40_000])
    s = np.array([0, 0, 1])
    lo, hi = cv.window_ranges(s, ["chr1"] * 3, w0, w1)
    base = (d(w0, np.int32), d(w1, np.int32), d(lo, np.int32), d(hi, np.int32), d(np.zeros(3), np.uint8), cv.dev)
    # row 0: 8 extras after the background (2048 applied: under the cap), row 1: 9 (over), row 2: unsorted
    ex = [[(30_000 + 2 * k, 1, 2, b"C") for k in range(8)], [(30_000 + 2 * k, 1, 2, b"C") for k in range(9)],
          [(20_000, 1, 2, b"C"), (19_000, 1, 1, b"G")]]
    e = _csr(ex)
    keys, count, lens, applied, err = ops.window_genotype_keys_edits(*base, *e)
    assert int(err.item()) == 4 and count.cpu().tolist() == [2048, -1, -1] and int(lens[2].item()) == 0
    _, out_len, app_enc, e2 = ops.encode_windows_edits(genome.seq, d(np.zeros(3), np.int64), *base, *e, 35_000,
                                                       knockout._pitch(35_000))
    assert int(e2.item()) == 4 and np.array_equal(app_enc.cpu().numpy(), applied.cpu().numpy())
    e_two = _csr(ex[:2])
    _, count, _, _, err = ops.window_genotype_keys_edits(*(t[:2] for t in base[:5]), cv.dev, *e_two)
    assert int(err.item()) == 2 and count.cpu().tolist() == [2048, -1]
    eq = ops.window_genotype_equal_edits(*base, *e, d([2, 1, 0], np.int32)).cpu().tolist()
    assert eq == [0, 1, 0]                                      # an unsorted row equals no other row
    # malformed arguments fail before any launch
    with pytest.raises(ValueError, match="e_off"):
        ops.window_genotype_keys_edits(*base, d([0, 1], np.int32), *e[1:])
    with pytest.raises(ValueError, match="extra-record arrays"):
        ops.window_genotype_keys_edits(*base, e[0], e[1][:-1], *e[2:])
    with pytest.raises(_lib.VFError, match="n_rows"):
        _lib.check(_lib.lib().vf_window_genotype_keys_edits(*([None] * 18), -1, None, None, None, None, None, None))
    with pytest.raises(_lib.VFError, match="extra-record array is NULL"):
        _lib.check(_lib.lib().vf_window_genotype_equal_edits(*[ops.ptr(t) for t in base[:5]], *[ops.ptr(cv.dev[k]) for k in
                   ("pos", "ref_len", "alt_off", "alt_len", "gt", "alt_pool")], None, *[ops.ptr(t) for t in e[1:]], 3,
                   ops.ptr(d([0, 1, 2], np.int32)), ops.ptr(d([0, 0, 0], np.int32)), None))


def _sets(rng, chrom, genes, per):
    """Per gene: singles in a CRE window and the gene window (SNVs and indels, het and hom), a cross-window pair, a
    same-window pair, a 3-record haplotype; gene 0 also a record sample 2 already carries (blocked there) and an SNV
    under a deletion given to sample 4."""
    out = []
    rec = lambda p, rl=1, alt=None, gt=2: Record("chr1", int(p) + 1, chrom[p:p + rl].tobytes().decode(),
                                                 alt or ("T" if chrom[p:p + 1].tobytes().upper() != b"T" else "G"), gt)
    for gi, g in enumerate(genes):
        o = knockout.batch_order(g)
        w = [cre_window(g.cre_start[i], g.cre_end[i], 50) for i in o]
        g0, _ = gene_window(g.start, g.end, g.strand, 1000, 300000)
        a, b = rec(w[0][0] + 12), rec(w[0][0] + 40, 3, "C", 1)
        c = rec(w[-1][0] + 20, 1, "ACGT")
        dd, e = rec(g0 + 1500, 1, None, 1), rec(g0 + 2500, 2, "A")
        s = [[a], [b], [c], [dd], [e], [a, c], [a, b], [c, dd], [e, dd, a]]
        if gi == 0:
            r = per[2]["chr1"]                                  # a record sample 2 carries, inside a CRE window
            i = next(i for i in range(len(r["pos"])) for a0, a1 in w[1:]
                     if r["gt"][i] and a0 <= r["pos"][i] and r["pos"][i] + r["ref_len"][i] <= a1)
            p = int(r["pos"][i])
            s.append([Record("chr1", p + 1, chrom[p:p + int(r["ref_len"][i])].tobytes().decode(), r["alt"][i].decode(),
                             int(r["gt"][i]))])
            q = w[2][0] + 30                                    # sample 4: a 20 bp deletion over this SNV
            r4 = per[4].setdefault("chr1", dict(pos=np.zeros(0, np.int64), ref_len=np.zeros(0, np.int32), alt=[],
                                                gt=np.zeros(0, np.uint8)))
            keep = (r4["pos"] + r4["ref_len"] <= q - 10) | (r4["pos"] > q + 12)
            k = int(np.searchsorted(r4["pos"][keep], q - 10))
            per[4]["chr1"] = dict(pos=np.insert(r4["pos"][keep], k, q - 10), ref_len=np.insert(r4["ref_len"][keep], k, 21),
                                  alt=[x for x, m in zip(r4["alt"], keep) if m][:k] + [chrom[q - 10:q - 9].tobytes()] +
                                  [x for x, m in zip(r4["alt"], keep) if m][k:], gt=np.insert(r4["gt"][keep], k, 2))
            s.append([rec(q)])
        out.append(s)
    return out


def _check_against_variant_sets(hot, genes, sets, per, got, idx):
    pred, emb, sp, se, app = got
    for row, s in enumerate(idx):
        want = hot.variant_sets(genes, sets, SampleVariants(per[s], "cuda"), embeddings=True)
        assert np.array_equal(pred[row], want[0]) and np.array_equal(emb[row], want[1]), s
        for gi in range(len(genes)):
            assert np.array_equal(sp[gi][row], want[2][gi]) and np.array_equal(se[gi][row], want[3][gi]), (s, gi)
            for k in ("cre", "gene"):
                assert np.array_equal(app[gi][k][row], want[4][gi][k]), (s, gi, k)
            for j in range(len(sets[gi])):
                assert np.array_equal(app[gi]["records"][j][row], want[4][gi]["records"][j]), (s, gi, j)


def test_cohort_variant_sets_bit_identical_to_variant_sets_per_sample(monkeypatch):
    rng = np.random.default_rng(83)
    chrom = synth.make_chromosome(rng, 3_000_000)
    _, per = _cohort(rng, chrom)
    genes = _genes(rng, len(chrom), n=5)                       # both strands; the last gene repeats gene 1
    genes[2].tissues = list(range(63))
    sets = _sets(rng, chrom, genes, per)
    sd = random_init.make_state_dict(CFG, HP, seed=5)
    hot = HotPath(Engine(sd, CFG, HP), Genome.from_arrays({"chr1": chrom}, "cuda"))
    cv = CohortVariants([f"S{i}" for i in range(N_SAMPLES)], per, "cuda")
    for coarse, stream in ((True, True), (False, True), (True, False)):
        monkeypatch.setattr(engine_mod, "COARSE", coarse)
        monkeypatch.setattr(engine_mod, "CRE_STREAM", stream)
        c = {}
        got = hot.cohort_variant_sets(genes, sets, cv, embeddings=True, counters=c)
        _check_against_variant_sets(hot, genes, sets, per, got, range(N_SAMPLES))
        base = hot.predict_cohort(genes, cv)
        assert np.array_equal(got[0], base[0]) and np.array_equal(got[1], base[1])
        if coarse and stream:
            # one item per slab and one (gene, sample) per pass; two samples per pass; colliding keys: the same bits;
            # and a second run
            seen = []
            plan = cohort_mod.plan_passes
            monkeypatch.setattr(cohort_mod, "plan_passes", lambda *a: seen.append(a) or plan(*a))
            again = [hot.cohort_variant_sets(genes, sets, cv, embeddings=True, rows_budget=1, pass_rows=1, key_bits=4)]
            two = 2 * int(max(seen[-1][3]))                    # twice the largest per-sample row bound
            again.append(hot.cohort_variant_sets(genes, sets, cv, embeddings=True, pass_rows=two))
            passes = plan(*seen[-1])
            assert any(s1 - s0 == 2 for _, _, s0, s1 in passes) and all(s1 - s0 >= 2 or s1 == N_SAMPLES
                                                                         for _, _, s0, s1 in passes)
            monkeypatch.setattr(cohort_mod, "plan_passes", plan)
            again.append(hot.cohort_variant_sets(genes, sets, cv, embeddings=True))
            for r in again:
                assert all(np.array_equal(x, y) for x, y in zip(r[:2], got[:2]))
                assert all(np.array_equal(x, y) for k in (2, 3) for x, y in zip(r[k], got[k]))
            sub = hot.cohort_variant_sets(genes, sets, cv, sample_idx=[5, 2], embeddings=True)
            _check_against_variant_sets(hot, genes, sets, per, sub, [5, 2])
            # the record sample 2 carries is blocked there: its item is the baseline, scored once
            a, carried, under = got[4][0], len(sets[0]) - 2, len(sets[0]) - 1
            assert not a["records"][carried][2].any() and a["records"][carried].any()
            assert np.array_equal(got[2][0][2, carried], got[0][2, :len(genes[0].tissues)])
            assert not a["records"][under][4].any() and a["records"][under].any()   # under sample 4's deletion
            assert c["items_scored"] < c["items"] == N_SAMPLES * sum(1 + len(s) for s in sets)
            c1 = {}
            one = hot.cohort_variant_sets(genes[:1], [[sets[0][carried]]], cv, sample_idx=[2], counters=c1)
            assert (c1["items"], c1["items_scored"]) == (2, 1) and np.array_equal(one[2][0][0, 0], one[0][0])
            assert c["windows_encoded"] < c["sample_windows"] and c["edited_groups"] > 0
            # without embeddings: the same predictions
            lean = hot.cohort_variant_sets(genes, sets, cv)
            assert len(lean) == 4 and all(np.array_equal(x, y) for x, y in zip(lean[2], got[2]))


def test_cohort_variant_sets_errors_name_the_sample_the_per_sample_call_fails_for(monkeypatch):
    rng = np.random.default_rng(84)
    chrom = synth.make_chromosome(rng, 3_000_000)
    _, per = _cohort(rng, chrom, n_samples=4)
    genes = _genes(rng, len(chrom), n=2)[:2]
    g0 = gene_window(genes[0].start, genes[0].end, genes[0].strand, 1000, 300000)[0]
    # sample 2: 2046 SNVs in gene 0's window; a set of 3 more passes the cap only with the set added
    pos = np.arange(g0 + 100, g0 + 100 + 2046 * 3, 3, dtype=np.int64)
    per[2] = {"chr1": dict(pos=pos, ref_len=np.ones(len(pos), np.int32), alt=[b"T"] * len(pos),
                           gt=np.ones(len(pos), np.uint8))}
    sd = random_init.make_state_dict(CFG, HP, seed=5)
    hot = HotPath(Engine(sd, CFG, HP), Genome.from_arrays({"chr1": chrom}, "cuda"))
    cv = CohortVariants(["a", "b", "c", "d"], per, "cuda")
    ins = lambda p, n: Record("chr1", p + 1, chrom[p:p + 1].tobytes().decode(), chrom[p:p + 1].tobytes().decode() + "A" * n)
    cap = [[ins(g0 + 7000 + 10 * k, 1) for k in range(3)]]
    # the cap: only sample c fails; the pitch: every sample fails, and the first in cohort order is named
    long = [[ins(g0 + 9000, 4000), ins(g0 + 20000, 1000)]]
    for sets, s, name in (([cap, []], 2, "c"), ([long, []], 0, "a")):
        with pytest.raises(RuntimeError) as want:
            hot.variant_sets(genes, sets, SampleVariants(per[s], "cuda"))
        with pytest.raises(RuntimeError) as got:
            hot.cohort_variant_sets(genes, sets, cv)
        assert str(got.value) == f"sample {name}: {want.value}"
    # VCFDataset's gene-window length rule
    with pytest.raises(ValueError, match="sample a: Mutated sequence is less than 10000000bp for gene G0"):
        hot.cohort_variant_sets(genes, [cap, []], cv, min_gene_len=10_000_000, gene_names=["G0", "G1"])
    # validation before any launch
    boom = lambda *a, **k: (_ for _ in ()).throw(AssertionError("a kernel ran"))
    monkeypatch.setattr(ops, "window_genotype_keys_edits", boom)
    monkeypatch.setattr(ops, "encode_windows_edits", boom)
    with pytest.raises(ValueError, match="GT"):
        hot.cohort_variant_sets(genes, [[[Record("chr1", 100, chrom[99:100].tobytes().decode(), "A", 7)]], []], cv)


def test_vcfprocessor_cohort_variant_sets_equals_variant_sets_on_single_sample_vcfs(tmp_path, monkeypatch):
    from variantformer_b200.processors.vcfprocessor import VCFProcessor
    from tests.test_gpu_pipeline import _world
    chroms, var, genes = _world(seed=85, n_genes=3, n_cres=20)
    rng = np.random.default_rng(85)
    names = ["NA1", "NA2", "NA3", "NA4"]
    sites = synth.make_variants(rng, chroms["chr1"], rate=1 / 1500)
    g = rng.integers(0, 3, (len(sites["pos"]), len(names))).astype(np.uint8)
    g[:, 3] = 0
    private = [synth.make_variants(rng, chroms["chr1"], rate=1 / 20000) if s != 3 else
               dict(pos=np.zeros(0, np.int64), ref_len=[], alt=[], gt=[]) for s in range(len(names))]
    art, rows = _write_artifacts(tmp_path, chroms, var, genes)
    vcf = str(tmp_path / "cohort.vcf")
    _write_cohort_vcf(vcf, (sites["pos"], sites["ref_len"], sites["alt"], g), private, names, chroms["chr1"])
    vp = VCFProcessor("v4_pcg", base_dir=str(tmp_path), model_overrides=dict(CFG, random_init=5, seq2reg_hyper_parameters=HP))
    query = pd.DataFrame({"gene_id": [r["gene_id"] for r in rows], "tissues": ["whole blood,thyroid", "K562",
                                                                              "thyroid,whole blood,K562"]})
    recs = []
    for gid, gs in zip([r["gene_id"] for r in rows], genes):
        o = knockout.batch_order(gs)
        w0 = cre_window(gs.cre_start[o[0]], gs.cre_end[o[0]], 50)[0]
        gw = gene_window(gs.start, gs.end, gs.strand, 1000, 300000)[0]
        for sid, ps in (("one", [w0 + 10]), ("two", [w0 + 10, gw + 2000])):
            for p in ps:
                ref = bytes(chroms["chr1"][p:p + 1]).decode()
                recs.append((gid, sid, "chr1", p + 1, ref, "T" if ref.upper() != "T" else "G", 1))
    variants = pd.DataFrame(recs, columns=["gene_id", "set", "chromosome", "pos", "ref", "alt", "gt"])
    got = vp.cohort_variant_sets(vcf, query, variants)
    assert list(got.columns) == ["sample"] + vs.SET_COLUMNS
    want = pd.concat([vp.variant_sets(f"{vcf}.{n}.vcf", query, variants).assign(sample=n) for n in names],
                     ignore_index=True)[["sample"] + vs.SET_COLUMNS]
    pd.testing.assert_frame_equal(got, want, check_exact=True)
    pd.testing.assert_frame_equal(vp.cohort_variant_sets(vcf, query, variants, genes_per_slab=2, samples_per_slab=3), got,
                                  check_exact=True)
    summary = vs.cohort_summary(got)
    assert len(summary) == len(got) // len(names) and (summary["n_samples"] == len(names)).all()
    # sub-blocks past a lowered index limit: the same frame
    from variantformer_b200 import ingest, stage1
    _, per = ingest.load_vcf_cohort(vcf)
    limit = max(max(stage1.CohortVariants.sizes([x])) for x in per)
    monkeypatch.setattr(stage1, "INT32_LIMIT", limit)
    assert len(stage1.CohortVariants.blocks(per)) >= 2
    pd.testing.assert_frame_equal(vp.cohort_variant_sets(vcf, query, variants), got, check_exact=True)
    monkeypatch.undo()
    # invalid records raise before the model is loaded
    monkeypatch.setattr(vp, "load_model", lambda: (_ for _ in ()).throw(AssertionError("model loaded")))
    with pytest.raises(ValueError, match="GT"):
        vp.cohort_variant_sets(vcf, query, variants.assign(gt=5))
