"""Saturation mutagenesis on the B200: vf_mutate_windows byte for byte, mutant tokens equal to the VEP builder's, and
every mutant's prediction bit-identical to the per-variant path (VEPBatchBuilder.build + variant_prediction)."""
import numpy as np
import pandas as pd
import pytest
import torch

pytestmark = pytest.mark.gpu

from tests.test_gpu_pipeline import CFG, HP, _world, _write_artifacts  # noqa: E402
from tests.test_ism_host import mutate_np  # noqa: E402
from variantformer_b200 import engine as engine_mod, ism, ops  # noqa: E402
from variantformer_b200.datasets.vepdataset import VEPBatchBuilder, Variant, cre_windows  # noqa: E402
from variantformer_b200.pipeline import HotPath  # noqa: E402
from variantformer_b200.stage1 import Genome, SampleVariants, gene_window  # noqa: E402
from variantformer_b200.utils import random_init  # noqa: E402


def test_mutate_windows_matches_numpy():
    rng = np.random.default_rng(11)
    pitch = 40_000
    lens = np.array([1, 16, 17, 200, 8191, 8193, 16_384, 16_385, 33_000, 39_999], np.int32)
    src = np.zeros((len(lens), pitch), np.uint8)
    for i, n in enumerate(lens):
        src[i, :n] = rng.choice(np.frombuffer(b"ACGTacgtNRYKMSW", np.uint8), n)
    rows = []
    for i, n in enumerate(lens):
        for off in sorted({0, int(n) - 1, int(rng.integers(0, n))}):
            for rc in (0, 1):
                rows.append((i, off, rng.choice(list(b"ACGTRYKMSW")), rc))
    r_src, r_off, r_base, r_fl = (np.array([r[k] for r in rows]) for k in range(4))
    d = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dt)).cuda()
    out, out_len, err = ops.mutate_windows(d(src, np.uint8), d(lens, np.int32), d(r_src, np.int32), d(r_off, np.int32),
                                           d(r_base, np.uint8), d(r_fl, np.uint8))
    out, out_len = out.cpu().numpy(), out_len.cpu().numpy()
    assert int(err.item()) == 0
    for j, (i, off, base, rc) in enumerate(rows):
        n = int(lens[i])
        want = mutate_np(src[i, :n].tobytes(), int(off), chr(base), bool(rc))
        assert out_len[j] == n and out[j, :n].tobytes() == want, (i, off, chr(base), rc)
    # an offset outside its row: error flag 3, length 0
    _, bad_len, err = ops.mutate_windows(d(src, np.uint8), d(lens, np.int32), d([1, 2], np.int32), d([16, -1], np.int32),
                                         d(list(b"AC"), np.uint8), d([0, 1], np.uint8))
    assert int(err.item()) == 3 and bad_len.cpu().numpy().tolist() == [0, 0]


def _setup(strand, with_background, seed=5):
    chroms, var, genes = _world(seed=79, n_genes=2, n_cres=30)
    g = genes[0 if strand == "+" else 1]
    g.tissues = [62, 3]
    genome = Genome.from_arrays(chroms, "cuda")
    sd = random_init.make_state_dict(CFG, HP, seed=seed)
    from variantformer_b200.seq2gene.model_combined_modulator import Seq2GenePredictorCombinedModulator, attach_trainer
    from variantformer_b200.seq2reg.model import Seq2RegPredictor
    model = Seq2GenePredictorCombinedModulator(cre_tokenizer=Seq2RegPredictor(**HP), gene_tokenizer=Seq2RegPredictor(**HP),
                                               **CFG)
    model.load_state_dict(sd); model.eval().to("cuda"); model.vep = True; attach_trainer(model)
    hot = HotPath(model.engine(), genome)
    background = var if with_background else None
    bg = SampleVariants({c: VEPBatchBuilder._snps_only(b) for c, b in var.items()}, "cuda") if with_background else None
    # region: straddles the left edge of a CRE window inside the gene window
    _, wins = cre_windows(g, 50)
    g0, g1 = gene_window(g.start, g.end, g.strand, 1000, 300000)
    a0 = next(a for a, b in wins if g0 + 10 < a and b < g1)
    return chroms, g, genome, model, hot, background, bg, (a0 - 2, a0 + 3)


@pytest.mark.parametrize("strand", ["+", "-"])
def test_mutant_tokens_equal_the_vep_builder(strand):
    chroms, g, genome, model, hot, background, bg, (start, end) = _setup(strand, True)
    it = ism.build_items(hot, g, start, end, (1, 2), bg)
    builder = VEPBatchBuilder(genome)
    ct, gt = it["cre_tokens"].cpu().numpy(), it["gene_tokens"].cpu().numpy()
    muts = it["plan"].mutants
    assert muts and any(m.hits for m in muts) and any(not m.hits for m in muts) and all(m.gene_hit for m in muts)
    for i, m in enumerate(muts):
        b = builder.build(g, Variant(g.chrom, m.pos, m.ref, m.alt, tissue=g.tissues), background)
        k = m.zyg
        assert (ct[it["cre_rows"][i + 1]] == b["cre_sequences"][k][:, 0].cpu().numpy()).all(), (m.pos, m.alt, k)
        assert (gt[it["gene_rows"][i + 1]] == b["gene_embeddings"][k][:, 0].cpu().numpy()).all(), (m.pos, m.alt, k)
        if i == 0:
            assert (ct[it["cre_rows"][0]] == b["cre_sequences"][0][:, 0].cpu().numpy()).all()
            assert (gt[it["gene_rows"][0]] == b["gene_embeddings"][0][:, 0].cpu().numpy()).all()


@pytest.mark.parametrize("strand,with_background", [("+", False), ("-", False), ("+", True), ("-", True)])
def test_ism_is_bit_identical_to_variant_prediction(strand, with_background, monkeypatch):
    chroms, g, genome, model, hot, background, bg, (start, end) = _setup(strand, with_background)
    builder = VEPBatchBuilder(genome)
    ref_rows, results = {}, {}
    for coarse in (True, False):
        monkeypatch.setattr(engine_mod, "COARSE", coarse)
        for budget in (len(g.cre_start), ism.ROWS_BUDGET):                # one item per slab, all items in one slab
            results[coarse, budget] = ism.saturation_mutagenesis(hot, g, start, end, (1, 2), bg, rows_budget=budget)
    monkeypatch.setattr(engine_mod, "COARSE", True)
    muts = results[True, ism.ROWS_BUDGET]["plan"].mutants
    cre_rows, gene_rows = set(), set()
    for i, m in enumerate(muts):
        key = (m.pos, m.alt)
        if key not in ref_rows:
            b = builder.build(g, Variant(g.chrom, m.pos, m.ref, m.alt, tissue=g.tissues), background)
            ref_rows[key] = model.variant_prediction(b)
            for k in (0, 1, 2):
                cre_rows |= {r.tobytes() for r in b["cre_sequences"][k][:, 0].cpu().numpy().astype(np.int32)}
                gene_rows |= {r.tobytes() for r in b["gene_embeddings"][k][:, 0].cpu().numpy().astype(np.int32)}
        want = ref_rows[key]
        for r in results.values():
            assert np.array_equal(r["pred"][i].cpu().numpy(), want["pred_gene_exp"][m.zyg][:, 0]), (m, "pred")
            assert np.array_equal(r["emb"][i].cpu().numpy(), want["embd"][m.zyg]), (m, "emb")
    any_ref = next(iter(ref_rows.values()))
    for r in results.values():
        assert np.array_equal(r["ref_pred"].cpu().numpy(), any_ref["pred_gene_exp"][0][:, 0])
        assert np.array_equal(r["ref_emb"].cpu().numpy(), any_ref["embd"][0])
    # every distinct window once: the counter equals the distinct token rows of all items (the per-variant batches
    # hold every item's rows; their tokens are pinned to the oracle by test_vep_triplet_matches_reference_semantics)
    c = results[True, ism.ROWS_BUDGET]["counters"]
    assert c["windows_encoded"] == len(cre_rows) + len(gene_rows)
    assert c["windows_encoded"] < c["windows_per_variant"]


def test_variantprocessor_saturation_mutagenesis(tmp_path):
    from variantformer_b200.processors.variantprocessor import VariantProcessor
    chroms, var, genes = _world(seed=80, n_genes=2, n_cres=20)
    art, rows = _write_artifacts(tmp_path, chroms, var, genes)
    g = genes[0]
    _, wins = cre_windows(g, 50)
    g0, g1 = gene_window(g.start, g.end, g.strand, 1000, 300000)
    a0 = next(a for a, b in wins if g0 + 10 < a and b < g1)
    start, end = a0 - 1, a0 + 2
    vp = VariantProcessor("v4_pcg", base_dir=str(tmp_path), model_overrides=dict(CFG, random_init=5, seq2reg_hyper_parameters=HP))
    tissues = ["whole blood", "thyroid"]
    df = vp.saturation_mutagenesis(rows[0]["gene_id"], tissues, start, end, zygosity=(1, 2))
    assert list(df.columns) == ["chrom", "pos", "ref", "alt", "genes", "tissues", "variant_type", "population",
                                "sample_name", "zygosity", "gene_exp", "ref_gene_exp", "log2fc"]
    seq = chroms["chr1"]
    ok = [p for p in range(start, end + 1) if chr(seq[p - 1]).upper() in "ACGT"]
    assert len(df) == 3 * len(ok) * 2 * len(tissues) and set(df["pos"]) == set(ok)
    assert np.allclose(df["log2fc"], np.log2((df["gene_exp"] + 1e-10) / (df["ref_gene_exp"] + 1e-10)))
    assert set(df["tissues"]) == set(tissues) and set(df["zygosity"]) == {"1", "2"}
    with pytest.raises(ValueError, match="unknown tissue"):
        vp.saturation_mutagenesis(rows[0]["gene_id"], ["not-a-tissue"], start, end)
    # equal to VariantProcessor.predict for two of its variants
    pick = df.drop_duplicates(["pos", "alt"]).iloc[[0, -1]]
    var_df = pd.DataFrame({"chr": pick["chrom"], "pos": pick["pos"], "ref": pick["ref"], "alt": pick["alt"],
                           "tissue": ",".join(tissues), "gene_id": rows[0]["gene_id"]})
    out = vp.predict(var_df, str(tmp_path / "out"))
    for _, r in out[out["zygosity"] != "0"].iterrows():
        hit = df[(df["pos"] == r["pos"]) & (df["alt"] == r["alt"]) & (df["zygosity"] == r["zygosity"]) &
                 (df["tissues"] == r["tissues"])]
        assert len(hit) == 1 and hit["gene_exp"].iloc[0] == r["gene_exp"]
    for _, r in out[out["zygosity"] == "0"].iterrows():
        hit = df[(df["pos"] == r["pos"]) & (df["tissues"] == r["tissues"])]
        assert (hit["ref_gene_exp"] == r["gene_exp"]).all()
