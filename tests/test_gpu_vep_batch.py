"""Variant tables in shared passes on the B200: vf_splice_windows byte for byte, every item's token rows equal to the
VEP builder's, VariantProcessor.predict_batched equal to predict in every column and bit, and the CRE-row gather of
the coarse forward equal to its cre_pos_idx gather."""
import numpy as np
import pandas as pd
import pytest
import torch

pytestmark = pytest.mark.gpu

from tests.test_gpu_pipeline import CFG, HP, _world, _write_artifacts  # noqa: E402
from tests.test_vep_batch_host import splice_np  # noqa: E402
from variantformer_b200 import engine as engine_mod, ism, ops, vep_batch  # noqa: E402
from variantformer_b200.datasets.vepdataset import VEPBatchBuilder, Variant, cre_windows  # noqa: E402
from variantformer_b200.pipeline import HotPath  # noqa: E402
from variantformer_b200.stage1 import Genome, SampleVariants, gene_window  # noqa: E402
from variantformer_b200.utils import random_init  # noqa: E402

d = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dt)).cuda()


def test_splice_windows_matches_numpy():
    rng = np.random.default_rng(12)
    pitch = 33_008
    lens = np.array([1, 15, 16, 17, 8191, 8193, 16_383, 16_384, 16_385, 33_000], np.int32)
    src = np.zeros((len(lens), pitch), np.uint8)
    for i, n in enumerate(lens):
        src[i, :n] = rng.choice(np.frombuffer(b"ACGTacgtNRYKMSW", np.uint8), n)
    pool, rows = bytearray(), []
    for i, n in enumerate(lens):
        n = int(n)
        offs = {0, n - 1, int(rng.integers(0, n))} | {x for x in (15, 16, 31, 16_383, 16_384) if x < n}
        for off in sorted(offs):
            for k in (0, 1, 2, 15, 16, 17, 31, 200):       # k = 0 deletes the base (an empty ALT)
                for rc in (0, 1):
                    a = rng.choice(np.frombuffer(b"ACGTNRYacgt", np.uint8), k).tobytes()
                    rows.append((i, off, len(pool), k, rc)); pool += a
    r_src, r_off, r_aoff, r_alen, r_fl = (np.array([r[j] for r in rows]) for j in range(5))
    out_pitch = pitch + 208                                           # 33 000 + 200 - 1 fits, nothing more
    out, out_len, err = ops.splice_windows(d(src, np.uint8), d(lens, np.int32), d(r_src, np.int32), d(r_off, np.int32),
                                           d(np.frombuffer(bytes(pool), np.uint8), np.uint8), d(r_aoff, np.int32),
                                           d(r_alen, np.int32), d(r_fl, np.uint8), out_pitch)
    out, out_len = out.cpu().numpy(), out_len.cpu().numpy()
    assert int(err.item()) == 0
    for j, (i, off, a0, k, rc) in enumerate(rows):
        n = int(lens[i])
        want = splice_np(src[i, :n].tobytes(), int(off), bytes(pool[a0:a0 + k]), bool(rc))
        assert out_len[j] == n + k - 1 and out[j, :n + k - 1].tobytes() == want, (i, off, k, rc)
    # an exactly fitting out pitch (33 000 + 16 - 1 < 33 024), then one byte too long (error 1), an offset outside the
    # row (error 3): such rows get length 0
    for k, pitch_o, code in ((16, 33_024, 0), (26, 33_024, 1)):
        a = rng.choice(np.frombuffer(b"ACGT", np.uint8), k)
        o, ol, e = ops.splice_windows(d(src, np.uint8), d(lens, np.int32), d([9], np.int32), d([32_999], np.int32),
                                      d(a, np.uint8), d([0], np.int32), d([k], np.int32), d([1], np.uint8), pitch_o)
        assert int(e.item()) == code
        if code == 0:
            assert ol.item() == 33_000 + k - 1
            assert o.cpu().numpy()[0, :ol.item()].tobytes() == splice_np(src[9, :33_000].tobytes(), 32_999, a.tobytes(), True)
        else:
            assert ol.item() == 0
    _, bad_len, err = ops.splice_windows(d(src, np.uint8), d(lens, np.int32), d([1, 2], np.int32), d([15, -1], np.int32),
                                         d(list(b"AC"), np.uint8), d([0, 1], np.int32), d([1, 1], np.int32),
                                         d([0, 1], np.uint8), out_pitch)
    assert int(err.item()) == 3 and bad_len.cpu().numpy().tolist() == [0, 0]


def _model(seed=5):
    sd = random_init.make_state_dict(CFG, HP, seed=seed)
    from variantformer_b200.seq2gene.model_combined_modulator import Seq2GenePredictorCombinedModulator, attach_trainer
    from variantformer_b200.seq2reg.model import Seq2RegPredictor
    model = Seq2GenePredictorCombinedModulator(cre_tokenizer=Seq2RegPredictor(**HP), gene_tokenizer=Seq2RegPredictor(**HP),
                                               **CFG)
    model.load_state_dict(sd); model.eval().to("cuda"); model.vep = True; attach_trainer(model)
    return model


def _alt(r):
    return "ACGT"[("ACGT".index(r) + 1) % 4] if r in "ACGT" else "A"


def _sites(g):
    """(CRE-only position, gene-window position inside a CRE window, gene-window position outside every CRE window)."""
    _, wins = cre_windows(g, 50)
    g0, g1 = gene_window(g.start, g.end, g.strand, 1000, 300000)
    cre_only = next((a + b) // 2 for a, b in wins if b < g0 or a > g1)
    both = next((a + b) // 2 for a, b in wins if g0 + 10 < a and b < g1)
    inside = [(a, b) for a, b in wins]
    gene_only = next(p for p in range(g0 + 100, g1) if not any(a < p <= b for a, b in inside))
    return cre_only, both, gene_only


@pytest.mark.parametrize("strand,with_background", [("+", False), ("-", False), ("+", True), ("-", True)])
def test_item_tokens_equal_the_vep_builder(strand, with_background):
    chroms, var, genes = _world(seed=79, n_genes=2, n_cres=30)
    g = genes[0 if strand == "+" else 1]
    g.tissues = [62, 3]
    genome = Genome.from_arrays(chroms, "cuda")
    hot = HotPath(_model().engine(), genome)
    background = var if with_background else None
    bg = SampleVariants({c: VEPBatchBuilder._snps_only(b) for c, b in var.items()}, "cuda") if with_background else None
    cre_only, both, gene_only = _sites(g)
    seq = chroms["chr1"]
    ref = lambda p: chr(seq[p - 1]).upper()
    vs = [Variant("chr1", cre_only, ref(cre_only), "TTGCA"),            # insertion in a CRE window (het 'N')
          Variant("chr1", cre_only, ref(cre_only) + "C", "G"),          # multi-base REF: one base replaced
          Variant("chr1", both, ref(both), _alt(ref(both))),
          Variant("chr1", gene_only, ref(gene_only), _alt(ref(gene_only))),
          Variant("chr1", both, ref(both), "GATTACA" * 3)]              # insertion in the gene window and a CRE window
    pairs = [dict(variant=Variant(v.chrom, v.pos, v.ref, v.alt, tissue=g.tissues), gene=g, gene_id="g") for v in vs]
    groups, plans = vep_batch.plan_pairs(pairs)
    it = ism.build_edit_items(hot, g, groups[0].edits, bg, want_gene_pos=True)
    ct, gt = it["cre_tokens"].cpu().numpy(), it["gene_tokens"].cpu().numpy()
    builder = VEPBatchBuilder(genome)
    for v, pl in zip(vs, plans):
        items = (0, 1 + pl.edits[0], 1 + pl.edits[1])
        try:
            b = builder.build(g, v, background)
        except ValueError:                                  # het 'N' in the gene window: build the hom sample alone
            assert v.alt == "GATTACA" * 3
            bgd = {c: VEPBatchBuilder._snps_only(x) for c, x in var.items()} if with_background else None
            sv = SampleVariants(VEPBatchBuilder._with_record(bgd, "chr1", v.pos - 1, v.alt.encode()), "cuda")
            g0, g1 = gene_window(g.start, g.end, g.strand, 1000, 300000)
            gseq, glens, _ = builder.tok.sequences(genome, ["chr1"], [g0], [g1], [int(g.strand == "-")], sv)
            tok, cnt = ops.bpe_tokenize(gseq, glens, gseq.shape[1], builder.tok.merges, 40_000, 40_000)
            G = (int(cnt[0]) + 199) // 200
            assert (gt[it["gene_rows"][items[2]]] == tok[0, :G * 200].view(G, 200).cpu().numpy()).all()
            continue
        for k, item in enumerate(items):
            assert (ct[it["cre_rows"][item]] == b["cre_sequences"][k][:, 0].cpu().numpy()).all(), (v, k)
            assert (gt[it["gene_rows"][item]] == b["gene_embeddings"][k][:, 0].cpu().numpy()).all(), (v, k)


def _table(rows, g_ids, genes, chroms):
    """~30 rows over both genes: SNVs and insertions in CRE windows, SNVs in the gene window, duplicates, a multi-base
    REF, a row that touches nothing, one gene on two rows with different tissue lists."""
    seq = chroms["chr1"]
    ref = lambda p: chr(seq[p - 1]).upper()
    out = []
    for gi, g in enumerate(genes):
        cre_only, both, gene_only = _sites(g)
        alt = lambda p: _alt(ref(p))
        for p in (cre_only, cre_only + 1, both, gene_only):
            out.append((p, ref(p), alt(p), "whole blood,thyroid", g_ids[gi]))
        out += [(cre_only, ref(cre_only), "TTGCA", "whole blood,thyroid", g_ids[gi]),
                (cre_only + 2, ref(cre_only + 2), "AC", "thyroid", g_ids[gi]),
                (cre_only, ref(cre_only) + "G", "C", "whole blood", g_ids[gi]),
                (both, ref(both), alt(both), "whole blood,thyroid", g_ids[gi]),       # duplicate row
                (both, ref(both), alt(both), "thyroid", g_ids[gi]),                   # same gene, other tissues
                (gene_only + 7, ref(gene_only + 7), alt(gene_only + 7), "thyroid", g_ids[gi]),
                (cre_only - 3, ref(cre_only - 3), "G" * 20, "whole blood", g_ids[gi]),
                (1, "A", "G", "whole blood", g_ids[gi]),                             # "No overlap"
                (both + 1, ref(both + 1), alt(both + 1), "whole blood,thyroid", g_ids[gi]),
                (cre_only, ref(cre_only), "TTGCA", "whole blood,thyroid", g_ids[gi]),  # duplicate insertion
                (cre_only + 4, ref(cre_only + 4), "", "thyroid", g_ids[gi])]          # empty ALT: a deletion
    return pd.DataFrame(out, columns=["pos", "ref", "alt", "tissue", "gene_id"]).assign(chr="chr1")


def _same(a, b):
    assert list(a.columns) == list(b.columns) and len(a) == len(b)
    for c in a.columns:
        for x, y in zip(a[c], b[c]):
            if isinstance(x, np.ndarray) or isinstance(y, np.ndarray):
                assert isinstance(x, np.ndarray) and isinstance(y, np.ndarray) and x.dtype == y.dtype, c
                assert np.array_equal(x, y), c
            elif x is None or y is None:
                assert x is None and y is None, c
            elif isinstance(x, float) and np.isnan(x):
                assert isinstance(y, float) and np.isnan(y), c
            else:
                assert x == y, c


def test_predict_batched_equals_predict(tmp_path, monkeypatch):
    from variantformer_b200.processors.variantprocessor import VariantProcessor
    chroms, var, genes = _world(seed=81, n_genes=2, n_cres=20)
    art, rows = _write_artifacts(tmp_path, chroms, var, genes)
    vp = VariantProcessor("v4_pcg", base_dir=str(tmp_path), model_overrides=dict(CFG, random_init=5, seq2reg_hyper_parameters=HP))
    df = _table(rows, [r["gene_id"] for r in rows], genes, chroms)
    assert 25 <= len(df) <= 40
    want = vp.predict(df, str(tmp_path / "ref"))
    assert want["variant_type"].nunique() >= 3 and (want["variant_type"] == "No overlap").any()
    with pytest.raises(FileExistsError):
        vp.predict_batched(df, str(tmp_path / "ref"))
    n = 0
    for coarse in (True, False):
        monkeypatch.setattr(engine_mod, "COARSE", coarse)
        for budget in (1, 1 << 30):                        # one item per slab; every item in one slab
            got = vp.predict_batched(df, str(tmp_path / f"b{n}"), rows_budget=budget)
            _same(got, want)
            _same(pd.read_parquet(tmp_path / f"b{n}" / "variants_VF.parquet"), pd.read_parquet(tmp_path / "ref" / "variants_VF.parquet"))
            n += 1
    # one group per pass
    monkeypatch.setattr(engine_mod, "COARSE", True)
    monkeypatch.setattr(vep_batch, "PASS_ROWS", 1)
    _same(vp.predict_batched(df, str(tmp_path / "passes")), want)
    monkeypatch.setattr(vep_batch, "PASS_ROWS", 1 << 30)
    # with a background sample
    vcf = str(tmp_path / "sample.vcf")
    _same(vp.predict_batched(df, str(tmp_path / "bg_b"), vcf_path=vcf, sample_name="S1"),
          vp.predict(df, str(tmp_path / "bg_r"), vcf_path=vcf, sample_name="S1"))


def _two_chromosomes(tmp_path):
    """The _world genes on chr1 plus a chr2 with its own background SNPs; every third CRE row of gene 0 lies on chr2."""
    from variantformer_b200.utils import synth
    chroms, var, genes = _world(seed=83, n_genes=2, n_cres=20)
    rng = np.random.default_rng(84)
    chroms["chr2"] = synth.make_chromosome(rng, len(chroms["chr1"]))
    var["chr2"] = synth.make_variants(rng, chroms["chr2"])
    art, rows = _write_artifacts(tmp_path, {"chr1": chroms["chr1"]}, {"chr1": var["chr1"]}, genes)
    with open(art / "GRCh38_no_alt_analysis_set_GCA_000001405.15.fasta.gz", "ab") as f:
        f.write(b">chr2 synthetic\n")
        s2 = chroms["chr2"].tobytes()
        for i in range(0, len(s2), 60):
            f.write(s2[i:i + 60] + b"\n")
    v = var["chr2"]
    with open(tmp_path / "sample.vcf", "a") as f:
        for p, rl, alt, gt in zip(v["pos"], v["ref_len"], v["alt"], v["gt"]):
            ref = chroms["chr2"][p:p + rl].tobytes().decode().upper()
            f.write(f"chr2\t{p + 1}\t.\t{ref}\t{alt.decode()}\t.\tPASS\t.\tGT\t{'0/1' if gt == 1 else '1|1'}\n")
    man = art / "gene_cre_manifests" / f"{rows[0]['gene_id']}.csv"
    m = pd.read_csv(man)
    m.loc[m.index % 3 == 1, "chromosome"] = "chr2"
    m.to_csv(man, index=False)
    genes[0].cre_chrom = list(m["chromosome"])
    return chroms, genes, rows


def test_predict_batched_equals_predict_across_chromosomes(tmp_path):
    """Windows on another chromosome than the variant's: the builder's het / hom samples encode them without the
    background, its reference sample with it."""
    from variantformer_b200.processors.variantprocessor import VariantProcessor
    chroms, genes, rows = _two_chromosomes(tmp_path)
    vp = VariantProcessor("v4_pcg", base_dir=str(tmp_path), model_overrides=dict(CFG, random_init=5, seq2reg_hyper_parameters=HP))
    order, wins = cre_windows(genes[0], 50)
    on2 = [k for k, i in enumerate(order) if genes[0].cre_chrom[i] == "chr2"]
    on1 = [k for k, i in enumerate(order) if genes[0].cre_chrom[i] == "chr1"]
    ref = lambda c, p: chr(chroms[c][p - 1]).upper()
    p2 = (wins[on2[0]][0] + wins[on2[0]][1]) // 2                      # inside a chr2 CRE row of gene 0
    p1 = (wins[on1[0]][0] + wins[on1[0]][1]) // 2                      # inside a chr1 CRE row of gene 0
    _, both, gene_only = _sites(genes[1])
    table = [("chr2", p2, ref("chr2", p2), _alt(ref("chr2", p2)), rows[0]["gene_id"]),
             ("chr1", p1, ref("chr1", p1), _alt(ref("chr1", p1)), rows[0]["gene_id"]),
             ("chr2", p1, ref("chr2", p1), "TTA", rows[0]["gene_id"]),   # chr2 variant at a chr1 row's coordinates
             ("chr2", both, ref("chr2", both), _alt(ref("chr2", both)), rows[1]["gene_id"]),  # gene window elsewhere
             ("chr2", gene_only, ref("chr2", gene_only), _alt(ref("chr2", gene_only)), rows[1]["gene_id"])]
    df = pd.DataFrame(table, columns=["chr", "pos", "ref", "alt", "gene_id"]).assign(tissue="whole blood,thyroid")
    vcf = str(tmp_path / "sample.vcf")
    want = vp.predict(df, str(tmp_path / "r"), vcf_path=vcf, sample_name="S1")
    assert (want["variant_type"] != "No overlap").all()
    _same(vp.predict_batched(df, str(tmp_path / "b"), vcf_path=vcf, sample_name="S1"), want)
    _same(vp.predict_batched(df, str(tmp_path / "b0")), vp.predict(df, str(tmp_path / "r0")))


def test_gene_hit_on_a_non_iupac_base_raises_like_predict(tmp_path, monkeypatch):
    from variantformer_b200.processors.variantprocessor import VariantProcessor
    chroms, var, genes = _world(seed=81, n_genes=2, n_cres=20)
    art, rows = _write_artifacts(tmp_path, chroms, var, genes)
    vp = VariantProcessor("v4_pcg", base_dir=str(tmp_path), model_overrides=dict(CFG, random_init=5, seq2reg_hyper_parameters=HP))
    _, _, gene_only = _sites(genes[0])
    seq = chroms["chr1"]
    for alt in ("GATTACA", "X"):                           # het 'N' / hom 'X' land on the variant base
        df = pd.DataFrame(dict(chr="chr1", pos=[gene_only], ref=[chr(seq[gene_only - 1]).upper()], alt=[alt],
                               tissue="whole blood", gene_id=rows[0]["gene_id"]))
        with pytest.raises(ValueError) as want:
            vp.predict(df, str(tmp_path / f"r{alt}"))
        with pytest.raises(ValueError) as got:
            vp.predict_batched(df, str(tmp_path / f"b{alt}"))
        assert str(got.value) == str(want.value) and "invalid character" in str(got.value)
    # the first bad pair of the table decides, even when its group is scored in a later pass: gene 0 (group 0, first
    # pass) holds a bad pair after gene 1's (group 1, second pass)
    cre_only0 = _sites(genes[0])[0]
    gene_only1 = _sites(genes[1])[2]
    base = lambda p: chr(seq[p - 1]).upper()
    df = pd.DataFrame(dict(chr="chr1", pos=[cre_only0, gene_only1, gene_only], alt=["G", "TTT", "TTTT"],
                           ref=[base(cre_only0), base(gene_only1), base(gene_only)], tissue="whole blood",
                           gene_id=[rows[0]["gene_id"], rows[1]["gene_id"], rows[0]["gene_id"]]))
    monkeypatch.setattr(vep_batch, "PASS_ROWS", 1)
    with pytest.raises(ValueError) as want:
        vp.predict(df, str(tmp_path / "r_order"))
    with pytest.raises(ValueError) as got:
        vp.predict_batched(df, str(tmp_path / "b_order"))
    assert str(got.value) == str(want.value)


def test_seq2gene_cre_rows_equals_the_cre_pos_gather():
    chroms, var, genes = _world(seed=79, n_genes=2, n_cres=30)
    genome = Genome.from_arrays(chroms, "cuda")
    eng = _model().engine()
    hot = HotPath(eng, genome)
    t = hot.tokenize(genes)
    tissues = [torch.as_tensor(g.tissues, dtype=torch.long) for g in genes]
    cpos = [3, 17]
    s = eng.prepare(t["cre_tok"], t["cre_msk"], t["gene_tok"], t["gene_msk"], tissues, t["labels"], lens=t["lens"],
                    cre_token_position=cpos)
    out = eng.run(s)                                       # coarse: vf_seq2gene_forward's cre_pos_idx gather
    C = [x.shape[0] for x in t["cre_tok"]]
    rows = d([cpos[0], C[0] + cpos[1], 0, C[0] + C[1] - 1], np.int32)
    import ctypes as Cc
    from variantformer_b200 import _lib
    nb = int(_lib.lib().vf_seq2gene_workspace_bytes(Cc.addressof(eng.w.abi()), Cc.addressof(s["_abi_slab"])))
    got = ops.seq2gene_cre_rows(eng.w.abi(), s["_abi_slab"], eng.ws.get("coarse_g", (nb,), torch.uint8), rows, eng.w.D)
    ctok = out["cre_token_embedding"].cpu().numpy()
    g = got.cpu().numpy()
    T0 = len(genes[0].tissues)
    assert np.array_equal(g[0], ctok[0]) and np.array_equal(g[1], ctok[T0])
    assert np.isfinite(g).all() and not np.array_equal(g[2], g[3])


def test_windows_encoded_counter():
    chroms, var, genes = _world(seed=79, n_genes=2, n_cres=30)
    genome = Genome.from_arrays(chroms, "cuda")
    hot = HotPath(_model().engine(), genome)
    seq = chroms["chr1"]
    pairs = []
    for g in genes:
        g.tissues = [62]
        cre_only, both, gene_only = _sites(g)
        for p, alt in ((cre_only, "TTGCA"), (cre_only, "TTGCA"), (both, None), (gene_only, None), (cre_only + 1, None)):
            r = chr(seq[p - 1]).upper()
            alt = alt or _alt(r)
            pairs.append(dict(variant=Variant("chr1", p, r, alt, tissue=[62]), gene=g, gene_id=id(g)))
    res, c = vep_batch.score_pairs(hot, pairs)
    builder = VEPBatchBuilder(genome)
    cre_rows, gene_rows = set(), set()
    for p in pairs:
        b = builder.build(p["gene"], p["variant"])
        for k in range(3):
            cre_rows |= {r.tobytes() for r in b["cre_sequences"][k][:, 0].cpu().numpy().astype(np.int32)}
            gene_rows |= {r.tobytes() for r in b["gene_embeddings"][k][:, 0].cpu().numpy().astype(np.int32)}
    assert c["windows_encoded"] == len(cre_rows) + len(gene_rows)
    assert c["windows_encoded"] < c["windows_per_pair"]
