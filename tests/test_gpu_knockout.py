"""In-silico CRE knockout on the B200: every knockout's prediction and embedding bit-identical to HotPath.predict on the
reduced GeneSpec (both strands, T = 1 / 2 / 63, reference genome and a sample background, coarse and fine engine, with
and without the CRE stream), the emptied-label-class path, split invariance, and VCFProcessor.cre_knockout against
create_data + predict on manifests with the rows deleted."""
import numpy as np
import pandas as pd
import pytest

pytestmark = pytest.mark.gpu

from tests.test_gpu_pipeline import CFG, HP, _world, _write_artifacts  # noqa: E402
from variantformer_b200 import engine as engine_mod, knockout  # noqa: E402
from variantformer_b200.engine import Engine  # noqa: E402
from variantformer_b200.pipeline import GeneSpec, HotPath  # noqa: E402
from variantformer_b200.stage1 import Genome, SampleVariants  # noqa: E402
from variantformer_b200.utils import random_init  # noqa: E402
from variantformer_b200.utils.constants import REF_CREs  # noqa: E402


def _reduced(g, knocked):
    keep = np.setdiff1d(np.arange(len(g.cre_start)), knocked)
    return GeneSpec(g.chrom, g.start, g.end, g.strand, g.cre_start[keep], g.cre_end[keep],
                    np.asarray(g.cre_labels)[keep], list(g.tissues))


def _setup():
    chroms, var, genes = _world(seed=91, n_genes=3, n_cres=14)
    for g, t in zip(genes, ([62, 3], list(range(63)), [14])):
        g.tissues = t
        lab = np.asarray(g.cre_labels) % 7
        lab[2] = 8                                           # class 8: one member
        lab[[5, 9]] = 7                                      # class 7: two members
        g.cre_labels = lab
    sd = random_init.make_state_dict(CFG, HP, seed=5)
    hot = HotPath(Engine(sd, CFG, HP), Genome.from_arrays(chroms, "cuda"))
    return hot, genes, SampleVariants(var, "cuda")


@pytest.mark.parametrize("with_background", [False, True])
def test_knockouts_bit_identical_to_predict_on_the_reduced_gene(with_background, monkeypatch):
    hot, genes, sv = _setup()
    variants = sv if with_background else None
    assert [g.strand for g in genes] == ["+", "-", "+"]
    sets = [[[i] for i in range(len(g.cre_start))] + [[5, 9], [0, 13, 6]] for g in genes]
    for coarse, stream in ((True, True), (False, True), (True, False), (False, False)):
        monkeypatch.setattr(engine_mod, "COARSE", coarse)
        monkeypatch.setattr(engine_mod, "CRE_STREAM", stream)
        pred, emb, ko_pred, ko_emb = hot.cre_knockout(genes, sets, variants, embeddings=True)
        p0, e0 = hot.predict(genes, variants)
        assert np.array_equal(pred, p0) and np.array_equal(emb, e0), (coarse, stream, "baseline")
        for gi, g in enumerate(genes):
            assert ko_pred[gi].shape == (len(sets[gi]), len(g.tissues))
            assert ko_emb[gi].shape == (len(sets[gi]), len(g.tissues), CFG["emb_dim"])
            for k, s in enumerate(sets[gi]):
                p, e = hot.predict([_reduced(g, s)], variants)
                assert np.array_equal(ko_pred[gi][k], p) and np.array_equal(ko_emb[gi][k], e), (coarse, stream, gi, s)
            assert np.isfinite(ko_pred[gi]).all()
        if coarse and stream:
            assert all(ko_pred[gi].std() > 0 for gi in range(3))          # the knockouts move the prediction
            # split invariance: one item per slab and one gene per pass; a second run; without embeddings
            c = {}
            runs = [hot.cre_knockout(genes, sets, variants, embeddings=True, rows_budget=1, pass_rows=1, counters=c),
                    hot.cre_knockout(genes, sets, variants, embeddings=True)]
            assert c["passes"] == 3 and c["slabs"] == c["items"] == sum(len(s) + 1 for s in sets)
            assert c["windows_encoded"] < c["windows_per_item"]
            for r in runs:
                assert np.array_equal(r[0], pred) and np.array_equal(r[1], emb)
                assert all(np.array_equal(a, b) for a, b in zip(r[2], ko_pred))
                assert all(np.array_equal(a, b) for a, b in zip(r[3], ko_emb))
            p3, e3, k3 = hot.cre_knockout(genes, sets, variants)
            assert np.array_equal(p3, pred) and np.array_equal(e3, emb)
            assert all(np.array_equal(a, b) for a, b in zip(k3, ko_pred))
            # the default scan: every CRE singly, the same bits as the explicit singles
            _, _, kd = hot.cre_knockout(genes, None, variants)
            assert all(np.array_equal(kd[gi], ko_pred[gi][:len(g.cre_start)]) for gi, g in enumerate(genes))


def test_validation_errors_are_raised_without_a_launch(monkeypatch):
    hot, genes, sv = _setup()

    def boom(*a, **k):
        raise AssertionError("stage 1 ran")
    monkeypatch.setattr(hot, "tokenize", boom)
    monkeypatch.setattr(hot.engine, "run_pooled", boom)
    n = len(genes[0].cre_start)
    for bad, msg in (([[n]], "outside the manifest"), ([[]], "empty"), ([[1, 1]], "repeats"),
                     ([list(range(n))], "removes every CRE")):
        with pytest.raises(ValueError, match=msg):
            hot.cre_knockout(genes, [[[0]], bad, [[0]]], sv)


def test_vcfprocessor_cre_knockout_equals_predict_on_edited_manifests(tmp_path, monkeypatch, capsys):
    from variantformer_b200.datasets.vcfdataset import LocalGeneManifest
    from variantformer_b200.processors.vcfprocessor import VCFProcessor
    chroms, var, genes = _world(seed=92, n_genes=2, n_cres=12)
    single = GeneSpec("chr1", genes[0].start, genes[0].end, "+", genes[0].cre_start[:1], genes[0].cre_end[:1],
                      np.asarray(genes[0].cre_labels)[:1], [62])
    art, rows = _write_artifacts(tmp_path, chroms, var, genes + [single])
    ids = [r["gene_id"] for r in rows]
    vcf = str(tmp_path / "sample.vcf")
    vp = VCFProcessor("v4_pcg", base_dir=str(tmp_path), model_overrides=dict(CFG, random_init=5, seq2reg_hyper_parameters=HP))
    # gene 0 (+ strand) from the sample, gene 1 (- strand) from the reference genome (empty path)
    query = pd.DataFrame({"gene_id": [ids[0], ids[1]], "tissues": ["whole blood,thyroid", "thyroid,not-a-tissue"],
                          "vcf_path": [vcf, ""]})
    C = len(genes[0].cre_start)
    kos = pd.DataFrame({"gene_id": [ids[0]] * 5 + [ids[1]] * 3,
                        "knockout": ["last", "first", "mid", "pair", "pair", "b", "b2", "b2"],
                        "cre_index": [C - 1, 0, C // 2, 1, 3, 2, C - 1, 0]})
    got = vp.cre_knockout(None, query, kos)
    assert list(got.columns) == knockout.FRAME_COLUMNS
    assert got["gene_id"].tolist() == [ids[0]] * 8 + [ids[1]] * 2
    assert got["knockout"].tolist() == ["last", "last", "first", "first", "mid", "mid", "pair", "pair", "b", "b2"]
    assert got["tissue"].tolist() == ["whole blood", "thyroid"] * 4 + ["thyroid"] * 2
    model, _, trainer = vp.load_model()

    def predict(manifest_dir, row):
        p = VCFProcessor("v4_pcg", base_dir=str(tmp_path), gene_cre_manifest=LocalGeneManifest(manifest_dir),
                         model_overrides=dict(CFG, random_init=5, seq2reg_hyper_parameters=HP))
        ds, dl = p.create_data(row["vcf_path"] or None, pd.DataFrame([row]).drop(columns="vcf_path"), batch_size=1)
        return vp.predict(model, None, trainer, dl, ds)["predicted_expression"].iloc[0][:, 0]
    man = art / "gene_cre_manifests"
    for qi, (_, row) in enumerate(query.iterrows()):
        gid = row["gene_id"]
        sub = got[got["gene_id"] == gid]
        T = 2 if qi == 0 else 1
        base = predict(str(man), row)
        assert np.array_equal(sub["baseline_expression"].to_numpy()[:T], base)
        m = pd.read_csv(man / f"{gid}.csv")
        for k in range(0, len(sub), T):
            r = sub.iloc[k]
            d = tmp_path / f"ko_{gid}_{r['knockout']}"
            d.mkdir()
            m.drop(index=list(r["cre_indices"])).to_csv(d / f"{gid}.csv", index=False)
            want = predict(str(d), row)
            assert np.array_equal(sub["predicted_expression"].to_numpy()[k:k + T], want), (gid, r["knockout"])
            assert np.array_equal(sub["delta"].to_numpy()[k:k + T], want - base)
            if len(r["cre_indices"]) == 1:
                i = r["cre_indices"][0]
                assert (r["chromosome"], r["start_cre"], r["end_cre"], r["cre_name"]) == tuple(
                    m[["chromosome", "start_cre", "end_cre", "cre_name"]].iloc[i])
            else:
                assert pd.isna(r["start_cre"]) and pd.isna(r["cre_name"])
    # the default scan: every CRE in manifest order; a single-CRE gene gets no rows and a message
    capsys.readouterr()
    full = vp.cre_knockout(vcf, pd.DataFrame({"gene_id": [ids[1], ids[2]], "tissues": ["thyroid", "thyroid"]}))
    assert "has a single CRE" in capsys.readouterr().out
    assert full["knockout"].tolist() == list(range(len(genes[1].cre_start)))
    assert full["cre_name"].tolist() == pd.read_csv(man / f"{ids[1]}.csv")["cre_name"].tolist()
    assert set(full["cre_name"]) <= set(REF_CREs)
    # invalid sets fail before the model is loaded
    monkeypatch.setattr(vp, "load_model", lambda: (_ for _ in ()).throw(AssertionError("model loaded")))
    for idx, msg in ((C, "outside the manifest"), (-1, "outside the manifest")):
        bad = pd.DataFrame({"gene_id": [ids[0]], "knockout": ["x"], "cre_index": [idx]})
        with pytest.raises(ValueError, match=msg):
            vp.cre_knockout(vcf, query, bad)
    with pytest.raises(ValueError, match="repeats"):
        vp.cre_knockout(vcf, query, pd.DataFrame({"gene_id": [ids[0]] * 2, "knockout": ["x"] * 2, "cre_index": [1, 1]}))
    with pytest.raises(ValueError, match="removes every CRE"):
        vp.cre_knockout(vcf, query, pd.DataFrame({"gene_id": [ids[0]] * C, "knockout": ["x"] * C,
                                                  "cre_index": list(range(C))}))
