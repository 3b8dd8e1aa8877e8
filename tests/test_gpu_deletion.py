"""In-silico deletions on the B200: vf_encode_windows_edit byte for byte against vf_encode_windows on the table with the
record inserted (random backgrounds with SNPs and indels, records overlapping the anchor, inside the span and at equal
POS, both strands, spans 1 bp to 5 kb, windows up to 301 kB, the applied flags against the host restatement, error 2 at
the cap, malformed arguments); every deletion's prediction and embedding bit-identical to HotPath.predict with the record
added (T = 1 / 2 / 63, reference genome and an indel-bearing background, coarse and fine engine, with and without the CRE
stream, split invariance); and VCFProcessor.deletion_scan against create_data + predict on VCF copies with the line."""
import numpy as np
import pandas as pd
import pytest
import torch

pytestmark = pytest.mark.gpu

from tests.test_deletion_host import applied_records  # noqa: E402
from tests.test_gpu_pipeline import CFG, HP, _world, _write_artifacts  # noqa: E402
from variantformer_b200 import _lib, deletion, engine as engine_mod, knockout, ops  # noqa: E402
from variantformer_b200.engine import Engine  # noqa: E402
from variantformer_b200.pipeline import HotPath  # noqa: E402
from variantformer_b200.stage1 import Genome, SampleVariants, cre_window, gene_window  # noqa: E402
from variantformer_b200.utils import random_init, synth  # noqa: E402


def _d(a, dt):
    return torch.from_numpy(np.ascontiguousarray(a, dt)).cuda()


def _insert(v, pos, rl, alt):
    """A per-chromosome record dict with one hom-alt record added after every record of pos <= its own."""
    k = int(np.searchsorted(v["pos"], pos, "right"))
    return dict(pos=np.insert(np.asarray(v["pos"], np.int64), k, pos), ref_len=np.insert(np.asarray(v["ref_len"]), k, rl),
                alt=list(v["alt"][:k]) + [alt] + list(v["alt"][k:]), gt=np.insert(np.asarray(v["gt"], np.uint8), k, 2))


def _table(recs):
    """Records of many rows concatenated into one device table: -> (dev dict, [(lo, hi)])."""
    pos, rl, al, gt, pool, rng_ = [], [], [], [], [], []
    n = 0
    for v in recs:
        pos.append(v["pos"]); rl.append(v["ref_len"]); gt.append(v["gt"]); al += [len(a) for a in v["alt"]]
        pool += list(v["alt"]); rng_.append((n, n + len(v["pos"]))); n += len(v["pos"])
    al = np.asarray(al, np.int32)
    dev = dict(pos=_d(np.concatenate(pos), np.int32), ref_len=_d(np.concatenate(rl), np.int32),
               alt_off=_d(np.cumsum(al) - al, np.int32), alt_len=_d(al, np.int32), gt=_d(np.concatenate(gt), np.uint8),
               alt_pool=_d(np.frombuffer(b"".join(pool) or b"\0", np.uint8), np.uint8))
    return dev, rng_


def _edit_rows(chrom, var, rows):
    """Both encoders on rows (w0, w1, flags, pos, ref_len): -> (edit (out, len, applied, err), plain (out, len, err))."""
    n = len(rows)
    w0 = np.asarray([r[0] for r in rows]); w1 = np.asarray([r[1] for r in rows])
    fl = np.asarray([r[2] for r in rows], np.uint8)
    ep = np.asarray([r[3] for r in rows]); erl = np.asarray([r[4] for r in rows])
    anc = np.asarray([chrom[p] for p in ep], np.uint8)
    genome = _d(chrom, np.uint8)
    mw = int((w1 - w0).max()); pitch = (mw + 4096 + 15) // 16 * 16
    bg = dict(pos=np.asarray(var["pos"]), ref_len=np.asarray(var["ref_len"]), alt=var["alt"], gt=np.asarray(var["gt"]))
    dev, _ = _table([bg])
    lo = np.searchsorted(bg["pos"], w0, "left"); hi = np.searchsorted(bg["pos"], w1, "left")
    edit = ops.encode_windows_edit(genome, _d(np.zeros(n), np.int64), _d(w0, np.int32), _d(w1, np.int32), _d(lo, np.int32),
                                   _d(hi, np.int32), _d(fl, np.uint8), dev, _d(ep, np.int32), _d(erl, np.int32),
                                   _d(np.arange(n), np.int32), _d(np.ones(n), np.int32), _d(anc, np.uint8), mw, pitch)
    recs = [_insert(bg, int(p), int(r), bytes([a])) for p, r, a in zip(ep, erl, anc)]
    cut = lambda x, a, b: {k: x[k][int(np.searchsorted(x["pos"], a)):int(np.searchsorted(x["pos"], b))] for k in x}
    recs = [cut(x, a, b) for x, a, b in zip(recs, w0, w1)]     # each row's candidates [w0, w1), record included
    dev2, rr = _table(recs)
    plain = ops.encode_windows(genome, _d(np.zeros(n), np.int64), _d(w0, np.int32), _d(w1, np.int32),
                               _d([r[0] for r in rr], np.int32), _d([r[1] for r in rr], np.int32), _d(fl, np.uint8), dev2,
                               mw, pitch)
    return edit, plain, recs


def test_kernel_bytes_equal_encode_windows_with_the_record_inserted():
    rng = np.random.default_rng(3)
    chrom = synth.make_chromosome(rng, 1_000_000)
    var = synth.make_variants(rng, chrom, rate=1 / 300, indel_frac=0.3)
    pos = var["pos"]
    rows = []
    for k in range(160):
        span = int(rng.choice([300, 2_000, 20_000, 301_000]))
        w0 = int(rng.integers(10, len(chrom) - span - 10)); w1 = w0 + span
        L = int(rng.choice([1, 2, 7, 50, 400, 5_000]))
        kind = k % 6
        if kind == 0:                                    # anchor on a background record (equal POS)
            i = int(np.searchsorted(pos, w0 + span // 3)); p = int(pos[i])
        elif kind == 1:                                  # a background record that starts earlier and overlaps the anchor
            dl = np.flatnonzero(var["ref_len"] > 1)
            i = int(dl[min(len(dl) - 1, int(np.searchsorted(pos[dl], w0 + span // 4)))])
            p = int(pos[i]) + 1
        elif kind == 2:                                  # records inside the span
            i = int(np.searchsorted(pos, w0 + span // 2)); p = int(pos[i]) - 1
        elif kind == 3:                                  # at the window's edges
            p = w0 + int(rng.integers(-1, 2)); L = min(L, span - 3)
        elif kind == 4:
            p = w1 - L - 1 + int(rng.integers(0, 2))     # REF ending at w1 or one past it
        else:
            p = int(rng.integers(w0, w1))
        rows.append((w0, w1, int(rng.integers(0, 2)) | (2 if k % 17 == 0 else 0), p, L + 1))
    (out, olen, app, err), (pout, plen, perr), recs = _edit_rows(chrom, var, rows)
    assert int(err.item()) == 0 and int(perr.item()) == 0
    olen, plen = olen.cpu().numpy(), plen.cpu().numpy()
    assert np.array_equal(olen, plen)
    o, po = out.cpu().numpy(), pout.cpu().numpy()
    for r in range(len(rows)):
        assert np.array_equal(o[r, :olen[r]], po[r, :plen[r]]), r
    # applied against the host restatement of the rule
    bg_al = np.asarray([len(a) for a in var["alt"]])
    want = []
    for w0, w1, fl, p, rl in rows:
        lo, hi = np.searchsorted(pos, w0), np.searchsorted(pos, w1)
        idx = applied_records(pos[lo:hi], var["ref_len"][lo:hi], bg_al[lo:hi], var["gt"][lo:hi], w0, w1,
                              snp_only=bool(fl & 2), extra=(p, rl, 1))
        want.append(-1 in idx)
    got = app.cpu().numpy().astype(bool)
    assert np.array_equal(got, np.asarray(want))
    assert 20 < got.sum() < len(rows) - 20                   # both outcomes are exercised
    # a deletion the encoder does not apply leaves the row's bytes as they are without it
    base, blen, _ = ops.encode_windows(_d(chrom, np.uint8), _d(np.zeros(len(rows)), np.int64),
                                       _d([r[0] for r in rows], np.int32), _d([r[1] for r in rows], np.int32),
                                       *[_d(np.searchsorted(pos, [r[i] for r in rows]), np.int32) for i in (0, 1)],
                                       _d([r[2] for r in rows], np.uint8), _table([var])[0],
                                       max(r[1] - r[0] for r in rows), out.shape[1])
    blen = blen.cpu().numpy()
    b = base.cpu().numpy()
    for r in np.flatnonzero(~got):
        assert olen[r] == blen[r] and np.array_equal(o[r, :olen[r]], b[r, :blen[r]])


def test_error_2_from_the_extra_record_at_the_cap():
    rng = np.random.default_rng(4)
    chrom = synth.make_chromosome(rng, 40_000, n_rate=0.0)
    for n_bg, code in ((2048, 2), (2047, 0)):
        p = np.arange(100, 100 + 4 * n_bg, 4)
        var = dict(pos=p, ref_len=np.ones(n_bg, np.int32), alt=[b"A"] * n_bg, gt=np.full(n_bg, 2, np.uint8))
        (_, olen, app, err), (_, plen, perr), _ = _edit_rows(chrom, var, [(0, 40_000, 0, 30_000, 11)])
        assert int(err.item()) == code and int(perr.item()) == code
        assert bool(app.item()) == (code == 0)
        if code == 0:
            assert int(olen.item()) == int(plen.item()) == 40_000 - 10


def test_malformed_arguments_fail_without_a_launch():
    lib = _lib.lib()
    x = torch.zeros(16, dtype=torch.int32, device="cuda")
    p = x.data_ptr()
    n0 = lib.vf_launch_count()
    good = [p] * 18 + [1, 16, p, 16, p, p, p, None]
    for args, msg in ((good[:18] + [-1] + good[19:], b"n_win"), (good[:18] + [1, 32] + good[20:], b"pitch"),
                      ([None] + good[1:], b"NULL"), (good[:13] + [None] + good[14:], b"extra-record"),
                      (good[:23] + [None] + good[24:], b"applied")):
        assert lib.vf_encode_windows_edit(*args) != 0
        assert msg in lib.vf_last_error()
    assert lib.vf_encode_windows_edit(*(good[:18] + [0] + good[19:])) == 0        # nothing to do
    assert lib.vf_launch_count() == n0


def _setup():
    chroms, var, genes = _world(seed=93, n_genes=3, n_cres=14)
    for g, t in zip(genes, ([62, 3], list(range(63)), [14])):
        g.tissues = t
        g0, _ = gene_window(g.start, g.end, g.strand, 1000, 300000)
        g.cre_start[[3, 4]] = g0 + 2_000, g0 + 8_000          # two CREs inside the gene window (the gene body)
        g.cre_end[[3, 4]] = g0 + 2_300, g0 + 8_250
    sd = random_init.make_state_dict(CFG, HP, seed=5)
    hot = HotPath(Engine(sd, CFG, HP), Genome.from_arrays(chroms, "cuda"))
    return hot, chroms, var, genes


def _spans(g, chrom_len):
    """Deletions of every kind the planner distinguishes, for gene g."""
    order = knockout.batch_order(g)
    w = [cre_window(g.cre_start[i], g.cre_end[i], 50) for i in order]
    g0, g1 = gene_window(g.start, g.end, g.strand, 1000, 300000)
    inside = [k for k, (a, b) in enumerate(w) if g0 + 10 < a and b < g1 - 6_000]
    outside = [k for k, (a, b) in enumerate(w) if b < g0 or a > g1]
    k_in, k_out = inside[len(inside) // 2], (outside or [0])[0]
    r = order[k_out]
    s = [(w[k_out][0] + 22, w[k_out][0] + 31),               # inside one CRE window
         (w[k_out][1] - 10, w[k_out][1] + 40),               # straddling a CRE window's edge
         (int(g.cre_start[r]) + 1, int(g.cre_end[r])),       # a whole CRE
         (g0 + 5_000, g0 + 5_013),                           # inside the gene window: shifts the chunking
         (w[k_in][0] + 30, w[k_in][0] + 60),                 # in overlapping CRE and gene windows
         (w[k_in][0] - 500, w[k_in][1] + 500),               # longer than a CRE window
         (2, 3 + chrom_len // 1000)]                         # far from every window: a no-op
    return np.asarray(s, np.int64)


def _predict_with(hot, g, var, a, b, chroms):
    chrom = chroms[g.chrom]
    rec = _insert(var[g.chrom] if var is not None else dict(pos=np.zeros(0, np.int64), ref_len=np.zeros(0, np.int32),
                                                            alt=[], gt=np.zeros(0, np.uint8)),
                  a - 2, b - a + 2, bytes([chrom[a - 2]]))
    sv = SampleVariants({**(var or {}), g.chrom: rec}, "cuda")
    return hot.predict([g], sv)


@pytest.mark.parametrize("with_background", [False, True])
def test_deletions_bit_identical_to_predict_with_the_record(with_background, monkeypatch):
    hot, chroms, var, genes = _setup()
    sv = SampleVariants(var, "cuda") if with_background else None
    assert [g.strand for g in genes] == ["+", "-", "+"]
    spans = [_spans(g, len(chroms["chr1"])) for g in genes]
    for coarse, stream in ((True, True), (False, True), (True, False), (False, False)):
        monkeypatch.setattr(engine_mod, "COARSE", coarse)
        monkeypatch.setattr(engine_mod, "CRE_STREAM", stream)
        pred, emb, dp, de, app = hot.deletion_scan(genes, spans, sv, embeddings=True)
        p0, e0 = hot.predict(genes, sv)
        assert np.array_equal(pred, p0) and np.array_equal(emb, e0), (coarse, stream, "baseline")
        t0 = 0
        for gi, g in enumerate(genes):
            T = len(g.tissues)
            assert dp[gi].shape == (len(spans[gi]), T) and de[gi].shape == (len(spans[gi]), T, CFG["emb_dim"])
            for j, (a, b) in enumerate(spans[gi].tolist()):
                p, e = _predict_with(hot, g, var if with_background else None, a, b, chroms)
                assert np.array_equal(dp[gi][j], p) and np.array_equal(de[gi][j], e), (coarse, stream, gi, j)
            c, gw = app[gi]["cre"], app[gi]["gene"]
            assert c[0].sum() >= 1 and not gw[0]             # one CRE window
            assert gw[3] and gw[4] and c[4].any() and gw[5]   # gene window; CRE + gene windows; longer than a CRE window
            assert not c[6].any() and not gw[6]              # the no-op equals the baseline exactly
            assert np.array_equal(dp[gi][6], p0[t0:t0 + T]) and np.array_equal(de[gi][6], e0[t0:t0 + T])
            assert not np.array_equal(dp[gi][3], p0[t0:t0 + T])
            t0 += T
        if coarse and stream:
            c = {}
            runs = [hot.deletion_scan(genes, spans, sv, embeddings=True, rows_budget=1, pass_rows=1, counters=c),
                    hot.deletion_scan(genes, spans, sv, embeddings=True)]
            assert c["passes"] == 3 and c["slabs"] == c["items"] == sum(len(s) + 1 for s in spans)
            assert c["windows_encoded"] < c["windows_per_item"]
            for r in runs:
                assert np.array_equal(r[0], pred) and np.array_equal(r[1], emb)
                assert all(np.array_equal(x, y) for x, y in zip(r[2], dp))
                assert all(np.array_equal(x, y) for x, y in zip(r[3], de))
            p3, e3, d3, _ = hot.deletion_scan(genes, spans, sv)
            assert np.array_equal(p3, pred) and np.array_equal(e3, emb)
            assert all(np.array_equal(x, y) for x, y in zip(d3, dp))


def test_validation_raises_without_a_launch(monkeypatch):
    hot, chroms, var, genes = _setup()

    def boom(*a, **k):
        raise AssertionError("stage 1 ran")
    monkeypatch.setattr(hot, "tokenize", boom)
    n0 = _lib.lib().vf_launch_count()
    for bad, msg in (([[1, 5]], "starts at 2"), ([[10, 9]], "empty"), ([[10, len(chroms["chr1"]) + 1]], "outside chr1")):
        with pytest.raises(ValueError, match=msg):
            hot.deletion_scan(genes, [np.array([[5, 6]]), np.asarray(bad), np.zeros((0, 2))], SampleVariants(var, "cuda"))
    assert _lib.lib().vf_launch_count() == n0


def _vcf_with(tmp_path, name, chrom, base_lines, a, b):
    """A copy of the sample VCF (or an empty one) with the deletion's line placed after every line of its POS."""
    ref = bytes(chrom[a - 2:b]).decode().upper()
    line = (a - 1, f"chr1\t{a - 1}\t.\t{ref}\t{ref[0]}\t.\tPASS\t.\tGT\t1/1\n")
    lines = sorted(base_lines + [line], key=lambda x: x[0])     # stable: after the lines of the same POS
    path = tmp_path / name
    with open(path, "w") as f:
        f.write("##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tS1\n")
        f.writelines(x[1] for x in lines)
    return str(path)


def test_vcfprocessor_deletion_scan_equals_predict_on_vcf_copies(tmp_path, monkeypatch):
    from variantformer_b200.processors.vcfprocessor import VCFProcessor
    chroms, var, genes = _world(seed=94, n_genes=2, n_cres=10)
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
    # gene 0 (+ strand): a tiled region around a CRE from the sample; gene 1 (- strand): the default scan from the
    # reference genome (empty per-row path)
    g = genes[0]
    k = knockout.batch_order(g)[3]
    tl = deletion.tiles("chr1", int(g.cre_start[k]) - 60, int(g.cre_end[k]) + 60, 120, 90)
    tl["gene_id"] = ids[0]
    query = pd.DataFrame({"gene_id": [ids[0], ids[1]], "tissues": ["whole blood,thyroid", "thyroid"], "vcf_path": [vcf, ""]})
    got = vp.deletion_scan(None, query, tl)
    assert list(got.columns) == deletion.FRAME_COLUMNS
    assert got["gene_id"].tolist() == [ids[0]] * (2 * len(tl))           # gene 1 has no user deletion
    assert got["deletion"].tolist()[::2] == [f"chr1:{a}-{b}" for a, b in zip(tl["start"], tl["end"])]
    base = predict(vcf, ids[0], "whole blood,thyroid")
    assert np.array_equal(got["baseline_expression"].to_numpy()[:2], base)
    for j, (a, b) in enumerate(zip(tl["start"], tl["end"])):
        want = predict(_vcf_with(tmp_path, f"t{j}.vcf", chrom, base_lines, int(a), int(b)), ids[0], "whole blood,thyroid")
        assert np.array_equal(got["predicted_expression"].to_numpy()[2 * j:2 * j + 2], want), (a, b)
        assert np.array_equal(got["delta"].to_numpy()[2 * j:2 * j + 2], want - base)
    assert got["changed"].any() and got["start_cre"].isna().all()
    full = vp.deletion_scan(None, pd.DataFrame({"gene_id": [ids[1]], "tissues": ["thyroid"], "vcf_path": [""]}))
    m = pd.read_csv(art / "gene_cre_manifests" / f"{ids[1]}.csv")
    assert full["deletion"].tolist() == list(range(len(m))) and full["cre_name"].tolist() == m["cre_name"].tolist()
    assert (full["del_start"] == m["start_cre"] + 1).all() and (full["del_end"] == m["end_cre"]).all()
    assert (full["cre_windows_changed"] >= 1).all()          # a CRE's own window always contains its bases
    base1 = predict(None, ids[1], "thyroid")
    for j, (a, b) in enumerate(zip(full["del_start"], full["del_end"])):
        want = predict(_vcf_with(tmp_path, f"d{j}.vcf", chrom, [], int(a), int(b)), ids[1], "thyroid")
        assert np.array_equal(full["predicted_expression"].to_numpy()[j:j + 1], want), j
        assert np.array_equal(full["baseline_expression"].to_numpy()[j:j + 1], base1)
    # the frame joins with cre_knockout's on the manifest columns
    ko = vp.cre_knockout(None, pd.DataFrame({"gene_id": [ids[1]], "tissues": ["thyroid"], "vcf_path": [""]}))
    keys = ["gene_id", "tissue", "chromosome", "start_cre", "end_cre", "cre_name"]
    assert len(full.merge(ko, on=keys)) == len(m)
    # invalid spans fail before the model is loaded
    monkeypatch.setattr(vp, "load_model", lambda: (_ for _ in ()).throw(AssertionError("model loaded")))
    for a, b, msg in ((1, 5, "starts at 2"), (50, 40, "empty"), (10, len(chrom) + 1, "outside chr1")):
        with pytest.raises(ValueError, match=msg):
            vp.deletion_scan(vcf, query, pd.DataFrame({"gene_id": [ids[0]], "chromosome": ["chr1"], "start": [a],
                                                       "end": [b]}))
