"""In-silico variant combinations on the B200: vf_encode_windows_edits byte for byte against vf_encode_windows on the
table with the records inserted (random SNP + indel backgrounds, 0-8 extras per row: het and hom SNPs, insertions,
deletions, MNPs, at a background record's POS, overlapped by earlier records, adjacent; SNP-only rows, both strands,
windows up to 301 kB), the applied flags against the host restatement, errors 2 and 4, malformed arguments,
vf_encode_windows_edit as the one-record case; every set's prediction and embedding bit-identical to HotPath.predict
with the records added (T = 1 / 2 / 63, reference genome and a sample background, coarse and fine engine, with and
without the CRE stream, split invariance); and VCFProcessor.variant_sets / variant_interactions against create_data +
predict on VCF copies with the lines added."""
import numpy as np
import pandas as pd
import pytest
import torch

pytestmark = pytest.mark.gpu

from tests.test_deletion_host import applied_records  # noqa: E402
from tests.test_gpu_deletion import _d, _setup, _table  # noqa: E402
from tests.test_gpu_pipeline import CFG, HP, _world, _write_artifacts  # noqa: E402
from variantformer_b200 import _lib, engine as engine_mod, knockout, ops, variant_sets as vs  # noqa: E402
from variantformer_b200.stage1 import SampleVariants, cre_window, gene_window  # noqa: E402
from variantformer_b200.utils import synth  # noqa: E402
from variantformer_b200.variant_sets import Record  # noqa: E402


def _inserted(bg, recs):
    """bg (pos, ref_len, alt, gt) with recs [(pos, ref_len, alt, gt)] inserted, each after every record of pos <= its
    own, in list order.  -> (table dict, index of each inserted record)."""
    t = dict(pos=list(bg["pos"]), ref_len=list(bg["ref_len"]), alt=list(bg["alt"]), gt=list(bg["gt"]))
    at = []
    for p, rl, alt, gt in recs:
        k = int(np.searchsorted(np.asarray(t["pos"], np.int64), p, "right"))
        at = [i + 1 if i >= k else i for i in at] + [k]
        for key, x in zip(("pos", "ref_len", "alt", "gt"), (p, rl, alt, gt)):
            t[key].insert(k, x)
    return dict(pos=np.asarray(t["pos"], np.int64), ref_len=np.asarray(t["ref_len"], np.int32), alt=t["alt"],
                gt=np.asarray(t["gt"], np.uint8)), at


def _edits_rows(chrom, var, rows):
    """vf_encode_windows_edits on rows (w0, w1, flags, [(pos, ref_len, alt, gt)]) against vf_encode_windows on per-row
    tables with the records inserted.  -> (edits (out, len, applied, err), plain (out, len, err), per-row applied want)."""
    n = len(rows)
    w0 = np.asarray([r[0] for r in rows]); w1 = np.asarray([r[1] for r in rows])
    fl = np.asarray([r[2] for r in rows], np.uint8)
    genome = _d(chrom, np.uint8)
    mw = int((w1 - w0).max()); pitch = (mw + 4096 + 15) // 16 * 16
    bg = dict(pos=np.asarray(var["pos"]), ref_len=np.asarray(var["ref_len"]), alt=list(var["alt"]), gt=np.asarray(var["gt"]))
    dev, _ = _table([bg])
    lo = np.searchsorted(bg["pos"], w0, "left"); hi = np.searchsorted(bg["pos"], w1, "left")
    recs = [x for r in rows for x in r[3]]
    al = np.asarray([len(x[2]) for x in recs], np.int32)
    edits = ops.encode_windows_edits(
        genome, _d(np.zeros(n), np.int64), _d(w0, np.int32), _d(w1, np.int32), _d(lo, np.int32), _d(hi, np.int32),
        _d(fl, np.uint8), dev, _d(np.concatenate([[0], np.cumsum([len(r[3]) for r in rows])]), np.int32),
        _d([x[0] for x in recs], np.int32), _d([x[1] for x in recs], np.int32), _d(np.cumsum(al) - al, np.int32),
        _d(al, np.int32), _d([x[3] for x in recs], np.uint8),
        _d(np.frombuffer(b"".join(x[2] for x in recs) or b"\0", np.uint8), np.uint8), mw, pitch)
    tabs, want = [], []
    for (a, b, f, ex), l_, h_ in zip(rows, lo, hi):
        cut = {k: (v[l_:h_] if k != "alt" else v[l_:h_]) for k, v in bg.items()}
        t, at = _inserted(cut, ex)
        keep = (t["pos"] >= a) & (t["pos"] < b)
        idx = np.flatnonzero(keep)
        t = {k: (np.asarray(v)[keep] if k != "alt" else [v[i] for i in idx]) for k, v in t.items()}
        pos_in = {int(i): m for m, i in enumerate(idx)}
        tabs.append(t)
        ap = applied_records(t["pos"], t["ref_len"], [len(x) for x in t["alt"]], t["gt"], a, b, snp_only=bool(f & 2))
        want += [k in pos_in and pos_in[k] in ap for k in at]
    dev2, rr = _table(tabs)
    plain = ops.encode_windows(genome, _d(np.zeros(n), np.int64), _d(w0, np.int32), _d(w1, np.int32),
                               _d([r[0] for r in rr], np.int32), _d([r[1] for r in rr], np.int32), _d(fl, np.uint8), dev2,
                               mw, pitch)
    return edits, plain, np.asarray(want, bool)


def _random_extras(rng, chrom, var, w0, w1, k):
    """k extra records in [w0, w1), of every kind the encoder distinguishes, sorted by pos (equal pos in list order)."""
    pos, rl = var["pos"], var["ref_len"]
    out = []
    for _ in range(k):
        kind = int(rng.integers(0, 8))
        if kind == 0:                                          # at a background record's POS
            i = min(len(pos) - 1, int(np.searchsorted(pos, int(rng.integers(w0, w1))))); p = int(pos[i])
        elif kind == 1:                                        # inside a background deletion (overlapped by it)
            dl = np.flatnonzero(rl > 1)
            i = int(dl[min(len(dl) - 1, int(np.searchsorted(pos[dl], int(rng.integers(w0, w1)))))]); p = int(pos[i]) + 1
        elif kind == 2 and out:                                # adjacent to the previous extra
            p = out[-1][0] + out[-1][1]
        else:
            p = int(rng.integers(w0, w1))
        p = min(max(p, 0), len(chrom) - 10)
        shape = int(rng.integers(0, 4))
        ref = bytes(chrom[p:p + 1]).upper()
        if shape == 0:
            out.append((p, 1, b"ACGT"[int(rng.integers(0, 4))].to_bytes(1, "little"), int(rng.integers(1, 3))))   # SNP
        elif shape == 1:
            out.append((p, 1, ref + rng.choice(np.frombuffer(b"ACGT", np.uint8), int(rng.integers(1, 30))).tobytes(), int(rng.integers(1, 3))))
        elif shape == 2:
            out.append((p, int(rng.integers(2, 400)), ref, int(rng.integers(1, 3))))                           # deletion
        else:
            L = int(rng.integers(2, 5))
            out.append((p, L, rng.choice(np.frombuffer(b"ACGT", np.uint8), L).tobytes(), int(rng.integers(0, 3))))                   # MNP / gt 0
    out.sort(key=lambda x: x[0])
    return out


def test_kernel_bytes_equal_encode_windows_with_the_records_inserted():
    rng = np.random.default_rng(11)
    chrom = synth.make_chromosome(rng, 1_000_000)
    var = synth.make_variants(rng, chrom, rate=1 / 300, indel_frac=0.3)
    rows = []
    for r in range(180):
        span = int(rng.choice([300, 2_000, 20_000, 301_000]))
        w0 = int(rng.integers(10, len(chrom) - span - 10)); w1 = w0 + span
        k = r % 9                                              # 0 .. 8 extras (empty rows included)
        fl = int(rng.integers(0, 2)) | (2 if r % 13 == 0 else 0)
        rows.append((w0, w1, fl, _random_extras(rng, chrom, var, w0 - 5, w1 + 5, k)))
    (out, olen, app, err), (pout, plen, perr), want = _edits_rows(chrom, var, rows)
    assert int(err.item()) == 0 and int(perr.item()) == 0
    olen, plen = olen.cpu().numpy(), plen.cpu().numpy()
    assert np.array_equal(olen, plen)
    o, po = out.cpu().numpy(), pout.cpu().numpy()
    for r in range(len(rows)):
        assert np.array_equal(o[r, :olen[r]], po[r, :plen[r]]), r
    got = app.cpu().numpy().astype(bool)
    assert np.array_equal(got, want)
    assert 50 < got.sum() < len(got) - 50                    # both outcomes are exercised


def test_one_record_entry_point_is_the_list_kernel_with_one_hom_record():
    rng = np.random.default_rng(12)
    chrom = synth.make_chromosome(rng, 400_000)
    var = synth.make_variants(rng, chrom, rate=1 / 200, indel_frac=0.3)
    rows = []
    for r in range(64):
        w0 = int(rng.integers(10, 90_000)); w1 = w0 + int(rng.choice([500, 301_000]))
        p = int(rng.integers(w0, w1 - 20)); L = int(rng.integers(1, 12))
        rows.append((w0, w1, r % 2, [(p, L + 1, bytes(chrom[p:p + 1]), 2)]))
    (out, olen, app, err), _, want = _edits_rows(chrom, var, rows)
    n = len(rows)
    bg = dict(pos=np.asarray(var["pos"]), ref_len=np.asarray(var["ref_len"]), alt=list(var["alt"]), gt=np.asarray(var["gt"]))
    w0 = np.asarray([r[0] for r in rows]); w1 = np.asarray([r[1] for r in rows])
    pitch = out.shape[1]
    one = ops.encode_windows_edit(_d(chrom, np.uint8), _d(np.zeros(n), np.int64), _d(w0, np.int32), _d(w1, np.int32),
                                  _d(np.searchsorted(bg["pos"], w0), np.int32), _d(np.searchsorted(bg["pos"], w1), np.int32),
                                  _d([r[2] for r in rows], np.uint8), _table([bg])[0],
                                  _d([r[3][0][0] for r in rows], np.int32), _d([r[3][0][1] for r in rows], np.int32),
                                  _d(np.arange(n), np.int32), _d(np.ones(n), np.int32),
                                  _d([r[3][0][2][0] for r in rows], np.uint8), int((w1 - w0).max()), pitch)
    assert int(one[3].item()) == 0 and torch.equal(one[1], olen) and torch.equal(one[2], app)
    for r in range(n):
        L = int(olen[r])
        assert torch.equal(one[0][r, :L], out[r, :L]), r
    assert np.array_equal(app.cpu().numpy().astype(bool), want)


def test_errors_2_and_4_and_malformed_arguments():
    rng = np.random.default_rng(13)
    chrom = synth.make_chromosome(rng, 40_000, n_rate=0.0)
    for n_bg, code in ((2047, 2), (2046, 0)):                 # two extras on top: the 2049th applied record is err 2
        p = np.arange(100, 100 + 4 * n_bg, 4)
        var = dict(pos=p, ref_len=np.ones(n_bg, np.int32), alt=[b"A"] * n_bg, gt=np.full(n_bg, 2, np.uint8))
        extras = [(30_000, 3, b"C", 2), (30_010, 1, b"G", 1)]
        (_, olen, app, err), (_, plen, perr), _ = _edits_rows(chrom, var, [(0, 40_000, 0, extras)])
        assert int(err.item()) == code and int(perr.item()) == code
        assert app.cpu().numpy().tolist() == ([1, 1] if code == 0 else [1, 0])
        if code == 0:
            assert int(olen.item()) == int(plen.item()) == 40_000 - 2
    # an unsorted row: err 4, length 0, nothing merged; its sorted neighbour is unaffected
    var = dict(pos=np.array([50]), ref_len=np.ones(1, np.int32), alt=[b"A"], gt=np.full(1, 2, np.uint8))
    rows = [(0, 1_000, 0, [(500, 1, b"C", 2), (400, 1, b"G", 2)]), (0, 1_000, 0, [(400, 1, b"G", 2)])]
    (out, olen, app, err), (pout, plen, _), _ = _edits_rows(chrom, var, rows)
    assert int(err.item()) == 4 and olen.cpu().tolist()[0] == 0 and int(olen[1]) == int(plen[1])
    assert torch.equal(out[1, :int(olen[1])], pout[1, :int(plen[1])])
    # the wrapper checks the CSR shape on the host
    d = torch.zeros(4, dtype=torch.int32, device="cuda")
    u8 = torch.zeros(4, dtype=torch.uint8, device="cuda")
    base = [u8, torch.zeros(1, dtype=torch.int64, device="cuda")] + [d[:1]] * 4 + [u8[:1], _table([var])[0]]
    for off, msg in ((torch.tensor([1, 1], dtype=torch.int32), "e_off"), (torch.tensor([0], dtype=torch.int32), "e_off"),
                     (torch.tensor([0, 2, 1], dtype=torch.int32)[:2], "extra-record"),
                     (torch.tensor([0, -1], dtype=torch.int32), "e_off")):
        with pytest.raises(ValueError, match=msg):
            ops.encode_windows_edits(*base, off, d[:1], d[:1], d[:1], d[:1], u8[:1], u8[:1], 1, 16)
    # the C entry: NULL arrays and n_win < 0 fail without a launch
    lib = _lib.lib()
    x = torch.zeros(16, dtype=torch.int32, device="cuda")
    p = x.data_ptr()
    n0 = lib.vf_launch_count()
    good = [p] * 20 + [1, 16, p, 16, p, p, p, None]
    for args, msg in ((good[:20] + [-1] + good[21:], b"n_win"), (good[:20] + [1, 32] + good[22:], b"pitch"),
                      ([None] + good[1:], b"NULL"), (good[:13] + [None] + good[14:], b"extra-record"),
                      (good[:18] + [None] + good[19:], b"extra-record"), (good[:25] + [None] + good[26:], b"applied")):
        assert lib.vf_encode_windows_edits(*args) != 0
        assert msg in lib.vf_last_error()
    assert lib.vf_encode_windows_edits(*(good[:20] + [0] + good[21:])) == 0        # nothing to do
    assert lib.vf_launch_count() == n0


def _rec(chrom, ch, p0, ref_len=1, alt=None, gt=2):
    ref = bytes(chrom[p0:p0 + ref_len]).decode().upper()
    if alt is None or alt == ref:
        alt = ("T" if ref[0] != "T" else "G") + (alt or "")[1:]
    return Record(ch, p0 + 1, ref, alt, gt)


def _gene_sets(g, chrom):
    """Sets of every kind the planner distinguishes, for gene g."""
    order = knockout.batch_order(g)
    w = [cre_window(g.cre_start[i], g.cre_end[i], 50) for i in order]
    g0, g1 = gene_window(g.start, g.end, g.strand, 1000, 300000)
    outside = [k for k, (a, b) in enumerate(w) if b < g0 or a > g1]
    k1, k2 = outside[0], outside[-1]
    a = _rec(chrom, "chr1", w[k1][0] + 20)
    b = _rec(chrom, "chr1", w[k1][0] + 60, 4, "G")                  # same window as a: a deletion
    c = _rec(chrom, "chr1", w[k2][0] + 25, 1, "TTAGC")             # another CRE window: an insertion
    d = _rec(chrom, "chr1", g0 + 4_000, gt=1)                      # gene window, het SNP
    e = _rec(chrom, "chr1", g0 + 9_000, 2, "CA")                   # gene window, MNP
    hap = [_rec(chrom, "chr1", g0 + 20_000 + 997 * i, gt=1 + i % 2) for i in range(10)]
    far = _rec(chrom, "chr1", 5)
    return [[a], [b], [c], [d], [a, c], [a, b], [d, e], [a, d], hap, [c._replace(alt="TTTTTTTTTTTTTTTTTTTTTTTT")], [far]]


def _predict_with(hot, g, var, recs):
    bg = var["chr1"] if var is not None else dict(pos=np.zeros(0, np.int64), ref_len=np.zeros(0, np.int32), alt=[],
                                                  gt=np.zeros(0, np.uint8))
    t, _ = _inserted(bg, [(r.pos - 1, len(r.ref), r.alt.encode(), r.gt) for r in sorted(recs, key=lambda r: r.pos)])
    return hot.predict([g], SampleVariants({**(var or {}), "chr1": t}, "cuda"))


@pytest.mark.parametrize("with_background", [False, True])
def test_sets_bit_identical_to_predict_with_the_records(with_background, monkeypatch):
    hot, chroms, var, genes = _setup()
    sv = SampleVariants(var, "cuda") if with_background else None
    sets = [_gene_sets(g, chroms["chr1"]) for g in genes]
    for coarse, stream in ((True, True), (False, True), (True, False), (False, False)):
        monkeypatch.setattr(engine_mod, "COARSE", coarse)
        monkeypatch.setattr(engine_mod, "CRE_STREAM", stream)
        pred, emb, sp, se, app = hot.variant_sets(genes, sets, sv, embeddings=True)
        p0, e0 = hot.predict(genes, sv)
        assert np.array_equal(pred, p0) and np.array_equal(emb, e0), (coarse, stream, "baseline")
        t0 = 0
        for gi, g in enumerate(genes):
            T = len(g.tissues)
            assert sp[gi].shape == (len(sets[gi]), T) and se[gi].shape == (len(sets[gi]), T, CFG["emb_dim"])
            for j, s in enumerate(sets[gi]):
                p, e = _predict_with(hot, g, var if with_background else None, s)
                assert np.array_equal(sp[gi][j], p) and np.array_equal(se[gi][j], e), (coarse, stream, gi, j)
            ap = app[gi]
            assert ap["cre"][0].any() and ap["gene"][3] and ap["gene"][8] and ap["records"][4].all()
            assert not ap["cre"][10].any() and not ap["gene"][10] and not ap["records"][10].any()     # a no-op
            assert np.array_equal(sp[gi][10], p0[t0:t0 + T]) and np.array_equal(se[gi][10], e0[t0:t0 + T])
            t0 += T
        if coarse and stream:
            c = {}
            runs = [hot.variant_sets(genes, sets, sv, embeddings=True, rows_budget=1, pass_rows=1, counters=c),
                    hot.variant_sets(genes, sets, sv)]
            assert c["passes"] == 3 and c["slabs"] == c["items"] == sum(len(s) + 1 for s in sets)
            assert c["windows_encoded"] < c["windows_per_item"]
            for r in runs:
                assert np.array_equal(r[0], pred) and np.array_equal(r[1], emb)
                assert all(np.array_equal(x, y) for x, y in zip(r[2], sp))
            assert all(np.array_equal(x, y) for x, y in zip(runs[0][3], se))


def test_validation_raises_without_a_launch(monkeypatch):
    hot, chroms, var, genes = _setup()
    monkeypatch.setattr(hot, "tokenize", lambda *a, **k: (_ for _ in ()).throw(AssertionError("stage 1 ran")))
    ok = _rec(chroms["chr1"], "chr1", 1_000)
    n0 = _lib.lib().vf_launch_count()
    for bad, msg in (([ok._replace(chrom="chr9")], "not in the genome"), ([ok._replace(ref="A" if ok.ref != "A" else "C")], "not the genome's"),
                     ([ok._replace(alt="<DEL>")], "ALT"), ([ok._replace(gt=0)], "GT"), ([ok, ok], "overlap"), ([], "empty")):
        with pytest.raises(ValueError, match=msg):
            hot.variant_sets(genes, [[[ok]], [bad], []], SampleVariants(var, "cuda"))
    assert _lib.lib().vf_launch_count() == n0


def _vcf_with(tmp_path, name, base_lines, recs):
    """A copy of the sample VCF (or an empty one) with the records' lines placed after every line of their POS."""
    add = [(r.pos, f"{r.chrom}\t{r.pos}\t.\t{r.ref}\t{r.alt}\t.\tPASS\t.\tGT\t{'0/1' if r.gt == 1 else '1/1'}\n")
           for r in recs]
    lines = sorted(base_lines + add, key=lambda x: x[0])       # stable: after the lines of the same POS
    path = tmp_path / name
    with open(path, "w") as f:
        f.write("##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tS1\n")
        f.writelines(x[1] for x in lines)
    return str(path)


def test_vcfprocessor_sets_and_interactions_equal_predict_on_vcf_copies(tmp_path, monkeypatch):
    from variantformer_b200.processors.vcfprocessor import VCFProcessor
    chroms, var, genes = _world(seed=95, n_genes=2, n_cres=10)
    art, rows = _write_artifacts(tmp_path, chroms, var, genes)
    ids = [r["gene_id"] for r in rows]
    vcf = str(tmp_path / "sample.vcf")
    with open(vcf) as f:
        base_lines = [(int(x.split("\t")[1]), x) for x in f if not x.startswith("#")]
    over = dict(CFG, random_init=5, seq2reg_hyper_parameters=HP)
    vp = VCFProcessor("v4_pcg", base_dir=str(tmp_path), model_overrides=over)
    model, _, trainer = vp.load_model()

    def predict(path, gid, tissues):
        ds, dl = vp.create_data(path, pd.DataFrame({"gene_id": [gid], "tissues": [tissues]}), batch_size=1)
        return vp.predict(model, None, trainer, dl, ds)["predicted_expression"].iloc[0][:, 0]
    chrom = chroms["chr1"]
    g = genes[0]
    taken = set(int(x) for x in var["chr1"]["pos"])
    free = lambda p: next(q for q in range(p, p + 500) if all(q + d not in taken for d in range(-6, 8))
                          and all(chr(c) in "ACGTacgt" for c in chrom[q:q + 4]))
    k = knockout.batch_order(g)[2]
    g0, _ = gene_window(g.start, g.end, g.strand, 1000, 300000)
    ps = [free(int(g.cre_start[k]) + 10), free(int(g.cre_start[k]) + 80), free(g0 + 5_000)]
    recs = [_rec(chrom, "chr1", ps[0]), _rec(chrom, "chr1", ps[1], 3, "A", gt=1), _rec(chrom, "chr1", ps[2], 1, "CAT")]
    ov = recs[0]._replace(alt="A" if recs[0].ref != "A" else "C")          # a second allele at recs[0]'s site
    df = pd.DataFrame({"gene_id": [ids[0]] * 4, "chromosome": ["chr1"] * 4, "pos": [r.pos for r in recs + [ov]],
                       "ref": [r.ref for r in recs + [ov]], "alt": [r.alt for r in recs + [ov]],
                       "gt": [r.gt for r in recs + [ov]], "label": ["a", "b", "c", "d"]})
    query = pd.DataFrame({"gene_id": [ids[0], ids[1]], "tissues": ["whole blood,thyroid", "thyroid"],
                          "vcf_path": [vcf, ""]})
    got = vp.variant_interactions(None, query, df)
    assert list(got.columns) == vs.INTERACTION_COLUMNS
    pairs = list(zip(got["variant_a"][::2], got["variant_b"][::2]))
    assert ("a", "d") not in pairs and len(pairs) == 6 - 1     # the overlapping pair is skipped
    base = predict(vcf, ids[0], "whole blood,thyroid")
    lab = dict(zip("abcd", recs + [ov]))
    single = {x: predict(_vcf_with(tmp_path, f"s{x}.vcf", base_lines, [lab[x]]), ids[0], "whole blood,thyroid")
              for x in "abcd"}
    for j, (x, y) in enumerate(pairs):
        want = predict(_vcf_with(tmp_path, f"p{j}.vcf", base_lines, [lab[x], lab[y]]), ids[0], "whole blood,thyroid")
        rows_ = got.iloc[2 * j:2 * j + 2]
        assert np.array_equal(rows_["expression_ab"].to_numpy(), want), (x, y)
        assert np.array_equal(rows_["expression_a"].to_numpy(), single[x])
        assert np.array_equal(rows_["expression_b"].to_numpy(), single[y])
        assert np.array_equal(rows_["baseline_expression"].to_numpy(), base)
    # one set through the vcf_path argument
    sdf = df.iloc[[0, 2]].assign(set="s1")
    sets = vp.variant_sets(vcf, pd.DataFrame({"gene_id": [ids[0]], "tissues": ["thyroid"]}), sdf)
    assert list(sets.columns) == vs.SET_COLUMNS and sets["n_records"].tolist() == [2]
    want = predict(_vcf_with(tmp_path, "set.vcf", base_lines, [recs[0], recs[2]]), ids[0], "thyroid")
    assert np.array_equal(sets["predicted_expression"].to_numpy(), want) and sets["changed"].all()
    # invalid records fail before the model is loaded
    monkeypatch.setattr(vp, "load_model", lambda: (_ for _ in ()).throw(AssertionError("model loaded")))
    for bad, msg in ((dict(ref=["A" if r.ref[0] != "A" else "C" for r in (recs[0], recs[2])]), "not the genome's"), (dict(alt="<DEL>"), "ALT"), (dict(gt=3), "GT")):
        with pytest.raises(ValueError, match=msg):
            vp.variant_sets(vcf, query, sdf.assign(**bad))
