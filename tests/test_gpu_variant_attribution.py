"""Variant attribution on the B200: vf_encode_windows_overrides byte for byte against vf_encode_windows on per-row tables
with the records deleted or re-genotyped (random SNP + indel backgrounds, 0-8 overrides per row to GT 0 / 1 / 2, a
removed blocker, records at one POS, straddling records, SNP-only rows, both strands, windows up to 301 kB, the
2048-record cap), empty lists equal to vf_encode_windows, error 8 confined to its row, malformed arguments; every edit
set's prediction and embedding bit-identical to HotPath.predict with the edited table (T = 1 / 2 / 63, coarse and fine
engine, with and without the CRE stream, split invariance) and the all-removed set equal to the reference genome; and
VCFProcessor.variant_attribution against create_data + predict on VCF copies with the line removed or its GT rewritten."""
import numpy as np
import pandas as pd
import pytest
import torch

pytestmark = pytest.mark.gpu

from tests.test_gpu_deletion import _d, _setup, _table  # noqa: E402
from tests.test_gpu_pipeline import CFG, HP, _world, _write_artifacts  # noqa: E402
from variantformer_b200 import _lib, engine as engine_mod, ops, variant_attribution as va  # noqa: E402
from variantformer_b200.stage1 import SampleVariants, gene_window  # noqa: E402
from variantformer_b200.utils import synth  # noqa: E402
from variantformer_b200.variant_attribution import Edit  # noqa: E402


def _override_rows(chrom, var, rows, delete=True):
    """vf_encode_windows_overrides on rows (w0, w1, flags, [(index, gt)]) against vf_encode_windows on per-row tables
    with each record's GT replaced (GT 0 lines deleted when `delete`).  -> (overrides (out, len, err), plain (out, len,
    err))."""
    n = len(rows)
    w0 = np.asarray([r[0] for r in rows]); w1 = np.asarray([r[1] for r in rows])
    fl = np.asarray([r[2] for r in rows], np.uint8)
    genome = _d(chrom, np.uint8)
    mw = int((w1 - w0).max()); pitch = (mw + 4096 + 15) // 16 * 16
    bg = dict(pos=np.asarray(var["pos"]), ref_len=np.asarray(var["ref_len"]), alt=list(var["alt"]),
              gt=np.asarray(var["gt"], np.uint8))
    dev, _ = _table([bg])
    lo = np.searchsorted(bg["pos"], w0, "left"); hi = np.searchsorted(bg["pos"], w1, "left")
    ov = [x for r in rows for x in r[3]]
    got = ops.encode_windows_overrides(
        genome, _d(np.zeros(n), np.int64), _d(w0, np.int32), _d(w1, np.int32), _d(lo, np.int32), _d(hi, np.int32),
        _d(fl, np.uint8), dev, _d(np.concatenate([[0], np.cumsum([len(r[3]) for r in rows])]), np.int32),
        _d([x[0] for x in ov], np.int32), _d([x[1] for x in ov], np.uint8), mw, pitch)
    tabs = []
    for (_, _, _, o), l_, h_ in zip(rows, lo, hi):
        gt = bg["gt"].copy()
        for i, g in o:
            gt[i] = g
        keep = np.arange(l_, h_)
        if delete:
            keep = keep[gt[keep] != 0]
        tabs.append(dict(pos=bg["pos"][keep], ref_len=bg["ref_len"][keep], alt=[bg["alt"][i] for i in keep],
                         gt=gt[keep]))
    dev2, rr = _table(tabs)
    plain = ops.encode_windows(genome, _d(np.zeros(n), np.int64), _d(w0, np.int32), _d(w1, np.int32),
                               _d([r[0] for r in rr], np.int32), _d([r[1] for r in rr], np.int32), _d(fl, np.uint8), dev2,
                               mw, pitch)
    return got, plain


def _same(got, plain, n):
    (out, olen, err), (pout, plen, perr) = got, plain
    assert int(err.item()) == int(perr.item())
    olen, plen = olen.cpu().numpy(), plen.cpu().numpy()
    assert np.array_equal(olen, plen)
    o, po = out.cpu().numpy(), pout.cpu().numpy()
    for r in range(n):
        assert np.array_equal(o[r, :olen[r]], po[r, :plen[r]]), r


def _background(rng, chrom):
    """SNPs and indels at 1 per 300 bp, some at a shared POS, GTs 0 / 1 / 2."""
    v = synth.make_variants(rng, chrom, rate=1 / 300, indel_frac=0.3)
    dup = np.sort(rng.choice(len(v["pos"]), len(v["pos"]) // 15, replace=False))
    order = np.argsort(np.concatenate([v["pos"], v["pos"][dup]]), kind="stable")
    cat = lambda a, b: np.concatenate([a, b])[order]
    alts = list(v["alt"]) + [bytes([b"ACGT"[int(rng.integers(0, 4))]]) for _ in dup]
    alt = [alts[k] for k in order]
    rl = cat(v["ref_len"], np.ones(len(dup), np.int32))
    return dict(pos=cat(v["pos"], v["pos"][dup]), ref_len=rl, alt=alt,
                gt=rng.choice(np.array([0, 1, 1, 2], np.uint8), len(order)))


def test_kernel_bytes_equal_encode_windows_on_the_edited_table():
    rng = np.random.default_rng(21)
    chrom = synth.make_chromosome(rng, 1_000_000)
    var = _background(rng, chrom)
    pos, rl = var["pos"], var["ref_len"]
    rows = []
    for r in range(200):
        span = int(rng.choice([300, 2_000, 20_000, 301_000]))
        w0 = int(rng.integers(10, len(chrom) - span - 10)); w1 = w0 + span
        lo, hi = int(np.searchsorted(pos, w0)), int(np.searchsorted(pos, w1))
        k = min(r % 9, hi - lo)                                # 0 .. 8 overrides (empty rows included)
        idx = np.sort(rng.choice(np.arange(lo, hi), k, replace=False)) if k else []
        if r % 4 == 0 and hi > lo:                             # a blocker removed: a deletion and what it covers
            dl = [i for i in range(lo, hi) if rl[i] > 1]
            if dl:
                idx = np.unique(np.concatenate([np.asarray(idx, np.int64), [dl[0]]]))
        if r % 7 == 0 and hi > lo:                             # the record straddling the window's end
            idx = np.unique(np.concatenate([np.asarray(idx, np.int64), [hi - 1]]))
        ov = [(int(i), int(rng.integers(0, 3))) for i in idx]
        rows.append((w0, w1, int(rng.integers(0, 2)) | (2 if r % 11 == 0 else 0), ov))
    for delete in (True, False):                               # GT 0: the line deleted, or kept with GT 0
        got, plain = _override_rows(chrom, var, rows, delete)
        assert int(got[2].item()) == 0
        _same(got, plain, len(rows))
    # empty override lists are vf_encode_windows, bit for bit
    empty = [(a, b, f, []) for a, b, f, _ in rows]
    got, plain = _override_rows(chrom, var, empty)
    _same(got, plain, len(rows))
    # a removed blocker changes the bytes (the walk is not a no-op)
    dl = int(np.flatnonzero((rl > 1) & (var["gt"] != 0))[3])
    row = [(int(pos[dl]) - 100, int(pos[dl]) + 100, 0, [(dl, 0)]), (int(pos[dl]) - 100, int(pos[dl]) + 100, 0, [])]
    (out, olen, _), _ = _override_rows(chrom, var, row)
    assert int(olen[0]) != int(olen[1])


def test_cap_error_8_and_malformed_arguments():
    rng = np.random.default_rng(22)
    chrom = synth.make_chromosome(rng, 40_000, n_rate=0.0)
    # a deletion blocking two SNPs, then 2047 SNPs: 2048 applied; removing the deletion applies 2049 -> err 2
    p = np.concatenate([[100, 101, 102], np.arange(200, 200 + 4 * 2047, 4)])
    n = len(p)
    var = dict(pos=p, ref_len=np.concatenate([[5], np.ones(n - 1, np.int32)]).astype(np.int32),
               alt=[b"A"] * n, gt=np.full(n, 2, np.uint8))
    for ov, code in (([], 0), ([(0, 0)], 2), ([(0, 0), (1, 0)], 0), ([(0, 1)], 0)):
        got, plain = _override_rows(chrom, var, [(0, 40_000, 0, ov)])
        assert int(got[2].item()) == code and int(plain[2].item()) == code
        if code == 0:
            _same(got, plain, 1)
    # error 8: unsorted, repeated and out-of-range lists; only those rows are affected
    var = dict(pos=np.array([50, 60, 70, 5_000]), ref_len=np.ones(4, np.int32), alt=[b"A", b"C", b"G", b"T"],
               gt=np.array([1, 2, 1, 2], np.uint8))
    good = (0, 1_000, 0, [(0, 0), (2, 2)])
    bad = [(0, 1_000, 0, [(2, 0), (0, 0)]), (0, 1_000, 0, [(1, 0), (1, 2)]), (0, 1_000, 0, [(3, 0)]),
           (100, 1_000, 0, [(0, 0)])]
    for b in bad:
        (out, olen, err), (pout, plen, _) = _override_rows(chrom, var, [good, b, good])
        assert int(err.item()) == 8 and int(olen[1]) == 0
        for r in (0, 2):
            assert int(olen[r]) == int(plen[r]) and torch.equal(out[r, :int(olen[r])], pout[r, :int(plen[r])])
    # the wrapper checks the CSR shape and the GT values on the host
    d = torch.zeros(4, dtype=torch.int32, device="cuda")
    u8 = torch.zeros(4, dtype=torch.uint8, device="cuda")
    base = [u8, torch.zeros(1, dtype=torch.int64, device="cuda")] + [d[:1]] * 4 + [u8[:1], _table([var])[0]]
    for off, idx, gt, msg in ((torch.tensor([1, 1], dtype=torch.int32), d[:0], u8[:0], "o_off"),
                              (torch.tensor([0], dtype=torch.int32), d[:0], u8[:0], "o_off"),
                              (torch.tensor([0, 2], dtype=torch.int32), d[:1], u8[:2], "override arrays"),
                              (torch.tensor([0, 1], dtype=torch.int32), d[:1], u8[:1] + 3, "o_gt")):
        with pytest.raises(ValueError, match=msg):
            ops.encode_windows_overrides(*base, off.cuda(), idx, gt, 1, 16)
    # the C entry: NULL arrays and n_win < 0 fail without a launch
    lib = _lib.lib()
    x = torch.zeros(16, dtype=torch.int32, device="cuda")
    q = x.data_ptr()
    n0 = lib.vf_launch_count()
    good = [q] * 16 + [1, 16, q, 16, q, q, None]
    for args, msg in ((good[:16] + [-1] + good[17:], b"n_win"), (good[:16] + [1, 32] + good[18:], b"pitch"),
                      ([None] + good[1:], b"NULL"), (good[:13] + [None] + good[14:], b"override"),
                      (good[:15] + [None] + good[16:], b"override"), (good[:21] + [None] + good[22:], b"err")):
        assert lib.vf_encode_windows_overrides(*args) != 0
        assert msg in lib.vf_last_error()
    assert lib.vf_encode_windows_overrides(*(good[:16] + [0] + good[17:])) == 0        # nothing to do
    assert lib.vf_launch_count() == n0


def _edited(var, recs):
    """The sample dict with the planner records' GTs replaced (GT 0 lines deleted)."""
    v = var["chr1"]
    gt = np.asarray(v["gt"], np.uint8).copy()
    for r in recs:
        gt[r[5]] = r[4]
    keep = np.flatnonzero(gt != 0)
    return {"chr1": dict(pos=np.asarray(v["pos"])[keep], ref_len=np.asarray(v["ref_len"])[keep],
                         alt=[v["alt"][i] for i in keep], gt=gt[keep])}


def _gene_sets(hot, g, sv):
    """Leave-one-out of a spread of records (CRE windows and the gene window), window reverts, het <-> hom rewrites, a
    multi-record set across windows and the all-removed set (last)."""
    loo, _, gts = va.default_sets(g, sv, hot.nb, hot.up, hot.down, "record")
    ws, _, _ = va.default_sets(g, sv, hot.nb, hot.up, hot.down, "window")
    pick = loo[::max(1, len(loo) // 12)]
    flips = [((*s[0][:4], 3 - gt, s[0][5]),) for s, gt in list(zip(loo, gts))[1::max(1, len(loo) // 6)]]
    multi = tuple(sorted({r for s in pick[:4] for r in s}, key=lambda r: r[5]))
    return pick + ws[:3] + ws[-1:] + flips + [multi, va.all_removed(g, sv, hot.nb, hot.up, hot.down)]


def test_sets_bit_identical_to_predict_on_the_edited_table(monkeypatch):
    hot, chroms, var, genes = _setup()
    g = genes[0]                                             # two overlapping CRE windows
    g.cre_start[6] = g.cre_start[5] + 20; g.cre_end[6] = g.cre_end[5] + 40
    sv = SampleVariants(var, "cuda")
    sets = [_gene_sets(hot, g, sv) for g in genes]
    assert any(gg.strand == "-" for gg in genes)
    ref_p, ref_e = hot.predict(genes, None)
    for coarse, stream in ((True, True), (False, True), (True, False), (False, False)):
        monkeypatch.setattr(engine_mod, "COARSE", coarse)
        monkeypatch.setattr(engine_mod, "CRE_STREAM", stream)
        pred, emb, sp, se, ch = va.run(hot, genes, sets, sv, embeddings=True)
        p0, e0 = hot.predict(genes, sv)
        assert np.array_equal(pred, p0) and np.array_equal(emb, e0), (coarse, stream, "baseline")
        t0 = 0
        for gi, gg in enumerate(genes):
            T = len(gg.tissues)
            for j, s in enumerate(sets[gi]):
                p, e = hot.predict([gg], SampleVariants(_edited(var, s), "cuda"))
                assert np.array_equal(sp[gi][j], p) and np.array_equal(se[gi][j], e), (coarse, stream, gi, j)
                if not (ch[gi]["cre"][j].any() or ch[gi]["gene"][j]):
                    assert np.array_equal(sp[gi][j], p0[t0:t0 + T])
            assert np.array_equal(sp[gi][-1], ref_p[t0:t0 + T]) and np.array_equal(se[gi][-1], ref_e[t0:t0 + T])
            assert ch[gi]["gene"].any() and ch[gi]["cre"].any()
            t0 += T
        if coarse and stream:
            c = {}
            runs = [va.run(hot, genes, sets, sv, embeddings=True, rows_budget=1, pass_rows=1, counters=c),
                    va.run(hot, genes, sets, sv, rows_budget=7, pass_rows=500)]
            assert c["passes"] == 3 and c["windows_encoded"] < c["windows_per_item"]
            for r in runs:
                assert np.array_equal(r[0], pred) and np.array_equal(r[1], emb)
                assert all(np.array_equal(x, y) for x, y in zip(r[2], sp))
            assert all(np.array_equal(x, y) for x, y in zip(runs[0][3], se))
    # the public form: Edit lists resolved against the sample
    v = var["chr1"]
    i = sets[0][0][0][5]
    e = Edit("chr1", int(v["pos"][i]) + 1, "N" * int(v["ref_len"][i]), v["alt"][i].decode(), 0)
    n0 = _lib.lib().vf_launch_count()
    with pytest.raises(ValueError, match="twice"):
        hot.genotype_edits(genes, [[[e, e]], [], []], sv)
    assert _lib.lib().vf_launch_count() == n0
    _, _, sp1, _ = hot.genotype_edits(genes[:1], [[[e]]], sv)
    assert np.array_equal(sp1[0][0], sp[0][0])


def _vcf_edited(tmp_path, name, lines, edits):
    """A copy of the sample VCF with lines (by table index) removed (GT 0) or their GT rewritten."""
    path = tmp_path / name
    with open(path, "w") as f:
        f.write("##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tS1\n")
        for k, x in enumerate(lines):
            if k in edits:
                if edits[k] == 0:
                    continue
                x = x.rsplit("\t", 1)[0] + ("\t0/1\n" if edits[k] == 1 else "\t1/1\n")
            f.write(x)
    return str(path)


def test_vcfprocessor_attribution_equals_predict_on_vcf_copies(tmp_path, monkeypatch):
    from variantformer_b200.processors.vcfprocessor import VCFProcessor
    chroms, var, genes = _world(seed=97, n_genes=2, n_cres=10)
    art, rows = _write_artifacts(tmp_path, chroms, var, genes)
    ids = [r["gene_id"] for r in rows]
    vcf = str(tmp_path / "sample.vcf")
    with open(vcf) as f:
        lines = [x for x in f if not x.startswith("#")]
    over = dict(CFG, random_init=5, seq2reg_hyper_parameters=HP)
    vp = VCFProcessor("v4_pcg", base_dir=str(tmp_path), model_overrides=over)
    model, _, trainer = vp.load_model()

    def predict(path, gid, tissues):
        ds, dl = vp.create_data(path, pd.DataFrame({"gene_id": [gid], "tissues": [tissues]}), batch_size=1)
        return vp.predict(model, None, trainer, dl, ds)["predicted_expression"].iloc[0][:, 0]
    v = var["chr1"]
    key = lambda lab: next(k for k in range(len(v["pos"])) if lab == f"chr1:{v['pos'][k] + 1}:"
                           f"{chroms['chr1'][v['pos'][k]:v['pos'][k] + v['ref_len'][k]].tobytes().decode().upper()}>"
                           f"{v['alt'][k].decode()}")
    query = pd.DataFrame({"gene_id": [ids[0]], "tissues": ["whole blood,thyroid"]})
    got = vp.variant_attribution(vcf, query)
    assert list(got.columns) == va.ATTRIBUTION_COLUMNS and len(got) % 2 == 0
    base = predict(vcf, ids[0], "whole blood,thyroid")
    labels = list(dict.fromkeys(got["set"]))
    assert np.array_equal(got["baseline_expression"].to_numpy()[:2], base)
    ref = predict(_vcf_edited(tmp_path, "ref.vcf", lines, {k: 0 for k in range(len(lines))}), ids[0],
                  "whole blood,thyroid")
    assert np.array_equal(got["reference_expression"].to_numpy()[:2], ref)
    for lab in labels[::max(1, len(labels) // 5)] + labels[-1:]:
        k = key(lab)
        want = predict(_vcf_edited(tmp_path, f"d{k}.vcf", lines, {k: 0}), ids[0], "whole blood,thyroid")
        r = got[got["set"] == lab]
        assert np.array_equal(r["predicted_expression"].to_numpy(), want), lab
        assert r["new_gt"].tolist() == [0, 0] and r["sample_gt"].tolist() == [int(v["gt"][k])] * 2
    # scope "window": each window with records reverted to the reference
    win = vp.variant_attribution(None, query.assign(vcf_path=vcf), scope="window")
    assert win["sample_gt"].isna().all() and win["set"].iloc[-1] == "gene_window"
    g = genes[0]
    g0, g1 = gene_window(g.start, g.end, g.strand, 1000, 300000)
    in_gene = {k for k in range(len(v["pos"])) if g0 <= v["pos"][k] and v["pos"][k] + v["ref_len"][k] <= g1
               and v["gt"][k] != 0}
    want = predict(_vcf_edited(tmp_path, "gw.vcf", lines, {k: 0 for k in in_gene}), ids[0], "whole blood,thyroid")
    assert np.array_equal(win[win["set"] == "gene_window"]["predicted_expression"].to_numpy(), want)
    # explicit edits: a GT rewrite and a two-record set
    k1, k2 = key(labels[0]), key(labels[-1])
    rec = lambda k, gt: dict(gene_id=ids[0], chromosome="chr1", pos=int(v["pos"][k]) + 1,
                             ref=chroms["chr1"][v["pos"][k]:v["pos"][k] + v["ref_len"][k]].tobytes().decode().upper(),
                             alt=v["alt"][k].decode(), gt=gt)
    df = pd.DataFrame([rec(k1, 3 - int(v["gt"][k1])), rec(k1, 0), rec(k2, 0)]).assign(set=["flip", "pair", "pair"])
    ex = vp.variant_attribution(vcf, query, edits=df)
    assert ex["set"].tolist() == ["flip", "flip", "pair", "pair"]
    w1 = predict(_vcf_edited(tmp_path, "flip.vcf", lines, {k1: 3 - int(v["gt"][k1])}), ids[0], "whole blood,thyroid")
    w2 = predict(_vcf_edited(tmp_path, "pair.vcf", lines, {k1: 0, k2: 0}), ids[0], "whole blood,thyroid")
    assert np.array_equal(ex["predicted_expression"].to_numpy(), np.concatenate([w1, w2]))
    # the reference genome has no records: an empty frame; invalid edits fail before the model is loaded
    assert len(vp.variant_attribution(None, query)) == 0
    monkeypatch.setattr(vp, "load_model", lambda: (_ for _ in ()).throw(AssertionError("model loaded")))
    for bad, msg in ((dict(gt=5), "GT"), (dict(alt="<DEL>"), "no such record")):
        with pytest.raises(ValueError, match=msg):
            vp.variant_attribution(vcf, query, edits=df.assign(**bad))
