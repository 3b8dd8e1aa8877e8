"""Cohort prediction on the B200: the genotype-key kernels against a restatement of the encoder's rule and against the
encoder itself, HotPath.predict_cohort bit for bit against the per-sample path for every sample, and
VCFProcessor.predict_cohort (in memory and resumable on disk) against a loop over single-sample VCFs."""
import os

import numpy as np
import pandas as pd
import pytest
import torch

pytestmark = pytest.mark.gpu

from tests.test_gpu_pipeline import CFG, HP, _write_artifacts  # noqa: E402
from variantformer_b200 import engine as engine_mod, ops  # noqa: E402
from variantformer_b200.engine import Engine  # noqa: E402
from variantformer_b200.pipeline import GeneSpec, HotPath  # noqa: E402
from variantformer_b200.stage1 import CohortVariants, Genome, SampleVariants  # noqa: E402
from variantformer_b200.utils import random_init, synth  # noqa: E402

N_SAMPLES = 17
EMPTY = 5                                                    # the sample without any variant


def _cohort(rng, chrom, n_samples=N_SAMPLES, common_rate=1 / 900, private_rate=1 / 6000):
    """Shared common sites (allele frequencies from a skewed Beta(0.3, 2)) plus private variants per sample; SNVs and
    indels (overlapping and window-straddling records included), het and hom calls.  -> (sites, per-sample dicts) with
    sites = (pos, ref_len, alt, genotypes [n_samples]) of the common sites."""
    c = synth.make_variants(rng, chrom, rate=common_rate, indel_frac=0.2)
    af = rng.beta(0.3, 2.0, len(c["pos"]))
    g = (rng.random((len(c["pos"]), n_samples)) < af[:, None]).astype(np.uint8) + \
        (rng.random((len(c["pos"]), n_samples)) < af[:, None]).astype(np.uint8)
    if EMPTY < n_samples:
        g[:, EMPTY] = 0
    per = []
    for s in range(n_samples):
        keep = np.nonzero(g[:, s])[0]
        pos = list(c["pos"][keep]); rl = list(c["ref_len"][keep]); alt = [c["alt"][i] for i in keep]; gt = list(g[keep, s])
        if s != EMPTY:
            p = synth.make_variants(rng, chrom, rate=private_rate, indel_frac=0.3)
            pos += list(p["pos"]); rl += list(p["ref_len"]); alt += p["alt"]; gt += list(p["gt"])
        o = np.argsort(np.asarray(pos, np.int64), kind="stable")
        per.append({"chr1": dict(pos=np.asarray(pos, np.int64)[o], ref_len=np.asarray(rl, np.int32)[o],
                                 alt=[alt[i] for i in o], gt=np.asarray(gt, np.uint8)[o])} if len(o) else {})
    return (c["pos"], c["ref_len"], c["alt"], g), per


def _applied(v, lo, hi, w0, w1, snp):
    """The encoder's rule restated: the applied records of one row as comparable tuples."""
    out, cur = [], w0
    pos, rl, al, gt, off, pool = v
    for i in range(lo, hi):
        if gt[i] == 0 or pos[i] < cur or pos[i] + rl[i] > w1 or (snp and not (rl[i] == 1 and al[i] == 1)):
            continue
        out.append((int(pos[i]), int(rl[i]), int(gt[i]), bytes(pool[off[i]:off[i] + al[i]])))
        cur = pos[i] + rl[i]
    return tuple(out)


def test_genotype_keys_group_rows_that_encode_identically():
    rng = np.random.default_rng(31)
    chrom = synth.make_chromosome(rng, 400_000)
    _, per = _cohort(rng, chrom, common_rate=1 / 150, private_rate=1 / 800)
    cv = CohortVariants([f"S{i}" for i in range(N_SAMPLES)], per, "cuda")
    genome = Genome.from_arrays({"chr1": chrom}, "cuda")
    W = 300
    w0 = rng.integers(0, 390_000, W)
    cand = cv.dev["pos"].cpu().numpy()
    cand = cand[cand < 390_000]
    w0[:20] = cand[rng.integers(0, len(cand), 20)] + 1                    # windows starting inside a record
    w1 = w0 + rng.integers(50, 6_000, W)
    fl = rng.integers(0, 4, W).astype(np.uint8)                            # both strands, SNP-only or not
    S = N_SAMPLES
    rs, rw0, rw1, rfl = np.tile(np.arange(S), W), np.repeat(w0, S), np.repeat(w1, S), np.repeat(fl, S)
    lo, hi = cv.window_ranges(rs, ["chr1"] * len(rs), rw0, rw1)
    d = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dt)).cuda()
    args = (d(rw0, np.int32), d(rw1, np.int32), d(lo, np.int32), d(hi, np.int32), d(rfl, np.uint8), cv.dev)
    keys, count, lens, err = ops.window_genotype_keys(*args)
    assert int(err.item()) == 0
    keys, count, lens = keys.cpu().numpy(), count.cpu().numpy(), lens.cpu().numpy()
    h = {k: t.cpu().numpy() for k, t in cv.dev.items()}
    v = (h["pos"], h["ref_len"], h["alt_len"], h["gt"], h["alt_off"], h["alt_pool"].tobytes())
    lists = [_applied(v, lo[r], hi[r], rw0[r], rw1[r], rfl[r] & 2) for r in range(len(rs))]
    # equal lists <-> equal keys (128 bits: no collision expected here); the empty list is key 0
    by_list = {}
    for r, a in enumerate(lists):
        assert count[r] == len(a) and (len(a) > 0) == bool(keys[r].any())
        by_list.setdefault((r // S, a), set()).add(tuple(keys[r]))
    assert all(len(k) == 1 for k in by_list.values())
    assert len({(w, next(iter(k))) for (w, _), k in by_list.items()}) == len(by_list)
    n_nonempty = sum(1 for a in lists if a)
    assert n_nonempty > len(rs) // 4 and len(by_list) < len(rs)          # real sharing, real variety
    # every row against every other row of its window as representative: equal iff the lists are equal
    rep = (np.arange(len(rs)) // S) * S + rng.integers(0, S, len(rs))
    eq = ops.window_genotype_equal(*args, d(rep, np.int32)).cpu().numpy()
    assert np.array_equal(eq.astype(bool), np.asarray([lists[r] == lists[q] for r, q in enumerate(rep)]))
    # encode every row: the encoded length is the keys' length, and rows of one group encode byte-identically, also
    # when 4-bit keys force collisions that only the comparison separates
    pitch = ((int((w1 - w0).max()) + 4096 + 15) // 16) * 16
    out, out_len, e2 = ops.encode_windows(genome.seq, d(np.zeros(len(rs)), np.int64), *args[:5], cv.dev,
                                          int((w1 - w0).max()), pitch)
    assert int(e2.item()) == 0 and np.array_equal(out_len.cpu().numpy(), lens)
    out = out.cpu().numpy()
    from variantformer_b200.cohort import group_rows
    for bits in (128, 4):
        k, cnt, _, _ = ops.window_genotype_keys(*args, key_bits=bits)
        group, reps = group_rows(torch.arange(len(rs), device="cuda") // S, cnt, k,
                                 lambda rp: ops.window_genotype_equal(*args, rp.to(torch.int32)) != 0)
        group, reps = group.cpu().numpy(), reps.cpu().numpy()
        for r in range(len(rs)):
            q = reps[group[r]]
            assert lists[q] == lists[r] and out[q, :lens[q]].tobytes() == out[r, :lens[r]].tobytes()
        # 128 bits: one group per distinct list; 4 bits: collisions split, never merged across lists
        assert len(reps) == len(by_list) if bits == 128 else len(reps) >= len(by_list)


def test_genotype_keys_cap_matches_the_encoder():
    rng = np.random.default_rng(32)
    chrom = synth.make_chromosome(rng, 300_000)
    # sample 0: 3000 SNVs in [10 000, 40 000) (over the cap); samples 1..16: 1000 distinct SNVs each in the same span
    # (17 000 cohort records in the window, every sample under the cap)
    per = []
    for s in range(N_SAMPLES):
        n = 3000 if s == 0 else 1000
        pos = np.sort(rng.choice(np.arange(10_000, 40_000), n, replace=False)).astype(np.int64)
        per.append({"chr1": dict(pos=pos, ref_len=np.ones(n, np.int32), alt=[b"A"] * n, gt=np.full(n, 2, np.uint8))})
    cv = CohortVariants([f"S{i}" for i in range(N_SAMPLES)], per, "cuda")
    genome = Genome.from_arrays({"chr1": chrom}, "cuda")
    d = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dt)).cuda()
    for samples in (list(range(N_SAMPLES)), list(range(1, N_SAMPLES))):
        n = len(samples)
        lo, hi = cv.window_ranges(samples, ["chr1"] * n, [5_000] * n, [50_000] * n)
        args = (d([5_000] * n, np.int32), d([50_000] * n, np.int32), d(lo, np.int32), d(hi, np.int32),
                d([0] * n, np.uint8), cv.dev)
        _, count, _, err = ops.window_genotype_keys(*args)
        _, _, e_enc = ops.encode_windows(genome.seq, d([0] * n, np.int64), *args[:5], cv.dev, 45_000, 45_056 + 4096)
        assert int(err.item()) == int(e_enc.item()) == (2 if samples[0] == 0 else 0)
        want = [-1 if s == 0 else 1000 for s in samples]
        assert count.cpu().numpy().tolist() == want
    # malformed arguments fail before any launch
    from variantformer_b200 import _lib
    with pytest.raises(_lib.VFError, match="NULL"):
        _lib.check(_lib.lib().vf_window_genotype_keys(*([None] * 11), 3, None, None, None, None, None))
    with pytest.raises(_lib.VFError, match="n_rows"):
        _lib.check(_lib.lib().vf_window_genotype_equal(*([None] * 11), -1, None, None, None))


def _genes(rng, chrom_len, n=7):
    genes = []
    for g in range(n):
        lay = synth.make_gene_layout(rng, chrom_len, int(rng.integers(12, 40)), strand="+-"[g % 2],
                                     body_len=int(rng.integers(20_000, 60_000)), cre_span=150_000)
        genes.append(GeneSpec("chr1", lay["start"], lay["end"], lay["strand"], lay["cre_start"], lay["cre_end"],
                              lay["labels"], [[62, 3, 14], [5], list(range(10)), [0, 62]][g % 4]))
    genes.append(genes[1])                                   # a gene twice: its windows and items are shared
    return genes


def test_predict_cohort_bit_identical_to_the_per_sample_path(monkeypatch):
    rng = np.random.default_rng(33)
    chrom = synth.make_chromosome(rng, 3_000_000)
    _, per = _cohort(rng, chrom)
    genes = _genes(rng, len(chrom))
    sd = random_init.make_state_dict(CFG, HP, seed=5)
    hot = HotPath(Engine(sd, CFG, HP), Genome.from_arrays({"chr1": chrom}, "cuda"))
    cv = CohortVariants([f"S{i}" for i in range(N_SAMPLES)], per, "cuda")
    for coarse in (True, False):
        monkeypatch.setattr(engine_mod, "COARSE", coarse)
        want = [hot.predict(genes, SampleVariants(per[s], "cuda")) for s in range(N_SAMPLES)]
        c = {}
        runs = [hot.predict_cohort(genes, cv, counters=c), hot.predict_cohort(genes, cv)]
        if coarse:                                           # forced key collisions, one gene per pass, one item per slab
            runs.append(hot.predict_cohort(genes, cv, key_bits=4, pass_rows=1, rows_budget=1))
            runs.append(hot.predict_cohort(genes, cv, sample_idx=[EMPTY, 2]))
        for k, (pred, emb) in enumerate(runs):
            idx = [EMPTY, 2] if k == 3 else range(N_SAMPLES)
            assert pred.shape[0] == len(idx)
            for row, s in enumerate(idx):
                assert np.array_equal(pred[row], want[s][0]) and np.array_equal(emb[row], want[s][1]), (coarse, k, s)
    # windows really are shared across samples
    assert c["windows_encoded"] < c["sample_windows"] and c["token_rows"] < c["sample_token_rows"]
    assert c["items_scored"] < c["items"]


def test_predict_cohort_raises_for_the_sample_the_per_sample_path_raises_for():
    rng = np.random.default_rng(34)
    chrom = synth.make_chromosome(rng, 3_000_000)
    _, per = _cohort(rng, chrom, n_samples=4)
    genes = _genes(rng, len(chrom), n=2)[:2]
    g0, g1 = genes[0].start, genes[0].end
    pos = np.arange(g0, g0 + 2100 * 3, 3, dtype=np.int64)              # 2100 applied SNVs in gene 0's window
    per[2] = {"chr1": dict(pos=pos, ref_len=np.ones(len(pos), np.int32), alt=[b"T"] * len(pos),
                           gt=np.ones(len(pos), np.uint8))}
    sd = random_init.make_state_dict(CFG, HP, seed=5)
    hot = HotPath(Engine(sd, CFG, HP), Genome.from_arrays({"chr1": chrom}, "cuda"))
    with pytest.raises(RuntimeError, match="error 2"):
        hot.predict(genes, SampleVariants(per[2], "cuda"))
    cv = CohortVariants(["a", "b", "c", "d"], per, "cuda")
    with pytest.raises(RuntimeError, match="error 2 for sample c "):
        hot.predict_cohort(genes, cv)
    # VCFDataset's gene-window length rule, checked before any window is encoded
    with pytest.raises(AssertionError, match="less than 10000000bp for gene G0"):
        hot.predict_cohort(genes, cv, sample_idx=[0, 1, 3], min_gene_len=10_000_000, gene_names=["G0", "G1"])
    pred, _ = hot.predict_cohort(genes, cv, sample_idx=[0, 1, 3])
    assert np.array_equal(pred[2], hot.predict(genes, SampleVariants(per[3], "cuda"))[0])


def _write_cohort_vcf(path, sites, per_private, names, chrom):
    """One N-column VCF: the common sites with every sample's genotype, plus each sample's private records."""
    pos, rl, alt, g = sites
    lines = []
    for p, r, a, gg in zip(pos, rl, alt, g):
        ref = chrom[p:p + r].tobytes().decode().upper()
        cols = ["0/0", "0/1", "1|1"]
        lines.append((int(p), f"chr1\t{p + 1}\t.\t{ref}\t{a.decode()}\t.\tPASS\t.\tGT\t" + "\t".join(cols[x] for x in gg)))
    for s, v in enumerate(per_private):
        for p, r, a, gt in zip(v["pos"], v["ref_len"], v["alt"], v["gt"]):
            ref = chrom[p:p + r].tobytes().decode().upper()
            cols = ["0/0"] * len(names)
            cols[s] = "0/1" if gt == 1 else "1/1"
            lines.append((int(p), f"chr1\t{p + 1}\t.\t{ref}\t{a.decode()}\t.\tPASS\t.\tGT\t" + "\t".join(cols)))
    lines.sort(key=lambda x: x[0])
    head = "##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t"
    with open(path, "w") as f:
        f.write(head + "\t".join(names) + "\n" + "".join(l + "\n" for _, l in lines))
    for s, n in enumerate(names):                            # the single-sample cuts of the same file
        with open(f"{path}.{n}.vcf", "w") as f:
            f.write(head + n + "\n")
            for _, l in lines:
                x = l.split("\t")
                f.write("\t".join(x[:9] + [x[9 + s]]) + "\n")


def test_vcfprocessor_predict_cohort_equals_the_single_sample_loop(tmp_path, monkeypatch):
    from variantformer_b200.processors.vcfprocessor import VCFProcessor
    from tests.test_gpu_pipeline import _world
    chroms, var, genes = _world(seed=35, n_genes=3, n_cres=20)
    rng = np.random.default_rng(35)
    names = ["NA1", "NA2", "NA3", "NA4", "NA5"]
    sites = synth.make_variants(rng, chroms["chr1"], rate=1 / 1500)
    g = rng.integers(0, 3, (len(sites["pos"]), len(names))).astype(np.uint8)
    g[:, 3] = 0                                              # NA4: no variant at all
    private = [synth.make_variants(rng, chroms["chr1"], rate=1 / 20000) if s != 3 else
               dict(pos=np.zeros(0, np.int64), ref_len=[], alt=[], gt=[]) for s in range(len(names))]
    art, rows = _write_artifacts(tmp_path, chroms, var, genes)
    vcf = str(tmp_path / "cohort.vcf")
    _write_cohort_vcf(vcf, (sites["pos"], sites["ref_len"], sites["alt"], g), private, names, chroms["chr1"])
    vp = VCFProcessor("v4_pcg", base_dir=str(tmp_path), model_overrides=dict(CFG, random_init=5, seq2reg_hyper_parameters=HP))
    query = pd.DataFrame({"gene_id": [r["gene_id"] for r in rows] + ["ENSG_missing"],
                          "tissues": ["whole blood,thyroid", "K562,not-a-tissue", "thyroid,whole blood,K562", "thyroid"]})
    got = vp.predict_cohort(vcf, query, genes_per_slab=2, samples_per_slab=2)
    assert list(got.columns) == ["sample", "gene_id", "tissue", "predicted_expression", "embeddings"]
    model, ckpt, trainer = vp.load_model()
    want = []
    for n in names:
        ds, dl = vp.create_data(f"{vcf}.{n}.vcf", query, batch_size=2)
        out = vp.predict(model, None, trainer, dl, ds)
        for _, r in out.iterrows():
            for k, t in enumerate(r["tissue_names"]):
                want.append((n, r["gene_id"], t, r["predicted_expression"][k, 0], r["embeddings"][k]))
    assert len(got) == len(want) == 5 * (2 + 1 + 3)
    for (_, x), w in zip(got.iterrows(), want):
        assert (x["sample"], x["gene_id"], x["tissue"]) == w[:3]
        assert x["predicted_expression"] == w[3] and np.array_equal(x["embeddings"], w[4])
    # a subset of the samples
    sub = vp.predict_cohort(vcf, query, samples=["NA4", "NA2"], embeddings=False)
    assert list(sub.columns) == ["sample", "gene_id", "tissue", "predicted_expression"]
    assert sub["sample"].tolist() == ["NA4"] * 6 + ["NA2"] * 6
    assert np.array_equal(sub["predicted_expression"].to_numpy(),
                          got.set_index("sample").loc[["NA4", "NA2"], "predicted_expression"].to_numpy())
    # a sample block whose variant table passes the index limit is computed in sub-blocks, with the same results
    from variantformer_b200 import ingest, stage1
    _, per = ingest.load_vcf_cohort(vcf)
    limit = max(max(stage1.CohortVariants.sizes([d])) for d in per)
    assert len(stage1.CohortVariants.blocks(per, limit=limit)) >= 3
    monkeypatch.setattr(stage1, "INT32_LIMIT", limit)
    split = vp.predict_cohort(vcf, query, samples_per_slab=5)
    monkeypatch.undo()
    assert split[["sample", "gene_id", "tissue"]].equals(got[["sample", "gene_id", "tissue"]])
    assert np.array_equal(split["predicted_expression"].to_numpy(), got["predicted_expression"].to_numpy())
    assert np.array_equal(np.stack(split["embeddings"].to_numpy()), np.stack(got["embeddings"].to_numpy()))
    # on disk: one file per slab; deleting some and rerunning recomputes only those and gives the uninterrupted result
    def read_all(d):
        return pd.concat([pd.read_parquet(os.path.join(d, f)) for f in sorted(os.listdir(d)) if f.endswith(".parquet")],
                         ignore_index=True)
    out_dir = str(tmp_path / "run")
    assert vp.predict_cohort(vcf, query, output_dir=out_dir, genes_per_slab=2, samples_per_slab=2) == out_dir
    files = sorted(f for f in os.listdir(out_dir) if f.endswith(".parquet"))
    assert len(files) == 2 * 3
    full = read_all(out_dir)
    for f in files[1::2]:
        os.remove(os.path.join(out_dir, f))
    stat = lambda f: (os.stat(os.path.join(out_dir, f)).st_ino, os.stat(os.path.join(out_dir, f)).st_mtime_ns)
    kept = {f: stat(f) for f in files[0::2]}
    vp.predict_cohort(vcf, query, output_dir=out_dir, genes_per_slab=2, samples_per_slab=2)
    assert sorted(f for f in os.listdir(out_dir) if f.endswith(".parquet")) == files
    assert {f: stat(f) for f in kept} == kept                 # the slabs on disk were skipped, not rewritten
    again = read_all(out_dir)
    assert len(again) == len(full) == len(got)
    for c in ("slab", "item", "sample", "gene_id", "tissue", "predicted_expression"):
        assert again[c].tolist() == full[c].tolist(), c
    assert np.array_equal(np.stack(again["embeddings"].to_numpy()), np.stack(full["embeddings"].to_numpy()))
    key = lambda df: df.sort_values(["sample", "gene_id", "predicted_expression"])["predicted_expression"].to_numpy()
    assert np.array_equal(key(full), key(got))
