"""In-silico variant-combination throughput on one GPU (HotPath.variant_sets): a pair scan, with the per-set
HotPath.predict loop (the records added to the sample) as the baseline in the same run, and the rate of
vf_encode_windows_edits next to vf_encode_windows_edit and vf_encode_windows.

    python tools/bench_variant_sets.py [--cres 1024] [--tissues 1,63] [--baseline 16] [--parent-lib PATH] [--out f.json]

Full-size random-init model (utils/random_init), synthetic 6 Mb chromosome and a synthetic sample background (SNPs and
indels, utils/synth), one gene with --cres CREs and a 301 kb gene window.  The pair scan has 48 variants: 32 in CRE
windows outside the gene window (8 windows hold two each, 16 windows one each) and 16 in the gene window: 48 singles
and 1 128 pairs.  Per T one JSON object: items/s; ms per item split into stage 1 / seq2reg / seq2gene (CUDA events);
windows encoded against the windows the per-item path encodes; the per-set predict loop on --baseline sets, each output
checked bit-identical; the speed-up.  Then the encoder rate on 256 gene-window rows, every kernel timed alternately in
the same run (bytes = reference bytes read + row bytes written): vf_encode_windows, vf_encode_windows_edit (one 50 bp
deletion per row) and vf_encode_windows_edits with 0, 1 and 8 records per row; with --parent-lib (a libvf_b200.so
built from the parent commit) its vf_encode_windows_edit too.  The card's name and power limit are read in the same
run.  Prints one JSON line.
"""
import argparse
import ctypes
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from tools.bench_ism import Phases, card  # noqa: E402
from variantformer_b200 import _lib, knockout, ops, variant_sets as vs  # noqa: E402
from variantformer_b200.engine import Engine  # noqa: E402
from variantformer_b200.pipeline import GeneSpec, HotPath  # noqa: E402
from variantformer_b200.stage1 import Genome, SampleVariants, cre_window, gene_window  # noqa: E402
from variantformer_b200.utils import random_init, synth  # noqa: E402


def pick_variants(rng, g, chrom, var, hot):
    """48 SNV / indel records away from the background: 16 CRE windows with one, 8 with two, 16 in the gene window."""
    taken = np.asarray(var["chr1"]["pos"])
    free = lambda p: not (np.abs(taken - p) < 8).any()
    order = knockout.batch_order(g)
    g0, g1 = gene_window(g.start, g.end, g.strand, hot.up, hot.down)
    w = [cre_window(g.cre_start[i], g.cre_end[i], hot.nb) for i in order]
    outside = [k for k, (a, b) in enumerate(w) if b < g0 or a > g1]
    ks = rng.choice(outside, 24, replace=False)
    spots = [(k, d) for n, k in enumerate(ks) for d in ((10, 60) if n < 8 else (30,))]
    pos = [w[k][0] + d for k, d in spots] + list(np.linspace(g0 + 2_000, g1 - 2_000, 16).astype(int))
    recs = []
    for n, p in enumerate(pos):
        p = int(p)
        while not free(p):
            p += 1
        ref = chr(chrom[p]).upper()
        if n % 4 == 3:                                            # an insertion or a deletion every fourth record
            recs.append(vs.Record("chr1", p + 1, ref, ref + "GATTACA") if n % 8 == 3 else
                        vs.Record("chr1", p + 1, bytes(chrom[p:p + 4]).decode().upper(), ref))
        else:
            recs.append(vs.Record("chr1", p + 1, ref, "T" if ref != "T" else "C", 1 + n % 2))
    return recs


def with_records(var, recs):
    v = var["chr1"]
    t = dict(pos=list(v["pos"]), ref_len=list(v["ref_len"]), alt=list(v["alt"]), gt=list(v["gt"]))
    for r in sorted(recs, key=lambda r: r.pos):
        k = int(np.searchsorted(np.asarray(t["pos"]), r.pos - 1, "right"))
        for key, x in zip(("pos", "ref_len", "alt", "gt"), (r.pos - 1, len(r.ref), r.alt.encode(), r.gt)):
            t[key].insert(k, x)
    return SampleVariants({"chr1": {k: (np.asarray(x) if k != "alt" else x) for k, x in t.items()}}, "cuda")


def run(hot, g, recs, var, T, n_base):
    sv = SampleVariants(var, "cuda")
    g.tissues = list(range(T))
    sets, _, pair_idx, overlapping = vs.pairs(recs)
    assert not overlapping and len(sets) == 48 + 1128
    hot.variant_sets([g], [sets[:4] + sets[-4:]], sv)                  # warm-up of the kernels and allocator
    torch.cuda.synchronize()
    ph, cnt = Phases(), {}
    t0 = time.perf_counter()
    _, _, sp, _ = hot.variant_sets([g], [sets], sv, to_host=False, timer=ph, counters=cnt)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    sp = sp[0].cpu().numpy()
    n = len(sets)
    picks = list(np.linspace(0, n - 1, n_base).astype(int))
    svs = [with_records(var, sets[k]) for k in picks]
    hot.predict([g], svs[0], to_host=False)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    outs = [hot.predict([g], s, to_host=False)[0] for s in svs]
    torch.cuda.synchronize()
    bw = time.perf_counter() - t0
    same = all(np.array_equal(o.cpu().numpy(), sp[k]) for o, k in zip(outs, picks))
    assert same, "set output differs from the per-set path"
    return {"tissues": T, "sets": n, "singles": 48, "pairs": len(pair_idx), "items": cnt["items"],
            "changed": cnt["changed"], "items_per_s": round(cnt["items"] / wall, 1),
            "ms_per_item": round(1e3 * wall / cnt["items"], 3),
            "ms_per_item_split": {k: round(v / cnt["items"], 3) for k, v in ph.ms.items()},
            "windows_encoded": cnt["windows_encoded"], "windows_per_item_path": cnt["windows_per_item"],
            "cre_windows_edited": cnt["cre_windows_edited"], "gene_windows_edited": cnt["gene_windows_edited"],
            "cre_token_rows": cnt["cre_token_rows"], "gene_token_rows": cnt["gene_token_rows"],
            "slabs": cnt["slabs"], "passes": cnt["passes"],
            "baseline_per_set_predict": {"sets": len(picks), "sets_per_s": round(len(picks) / bw, 1),
                                         "ms_per_set": round(1e3 * bw / len(picks), 2), "bit_identical": same},
            "speedup": round((bw / len(picks)) / (wall / n), 2)}


def encoder_rate(hot, var, g, parent_lib=None, rows=256, reps=20):
    """The encoders on `rows` copies of g's gene window, alternated in one run."""
    sv = SampleVariants(var, "cuda")
    g0, g1 = gene_window(g.start, g.end, g.strand, hot.up, hot.down)
    d = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dt)).cuda()
    lo, hi = sv.window_range("chr1", g0, g1)
    args = [hot.genome.seq, d(np.zeros(rows), np.int64), d([g0] * rows, np.int32), d([g1] * rows, np.int32),
            d([lo] * rows, np.int32), d([hi] * rows, np.int32), d(np.zeros(rows), np.uint8), sv.dev]
    pos = np.linspace(g0 + 100, g1 - 200, rows).astype(np.int64)
    edit = [d(pos, np.int32), d(np.full(rows, 51), np.int32), d(np.arange(rows), np.int32), d(np.ones(rows), np.int32),
            hot.genome.seq.index_select(0, d(pos, np.int64))]
    span = g1 - g0
    pitch = (span + 4096 + 15) // 16 * 16

    def lists(k):                                                   # k records per row: 50 bp deletions 1 kb apart
        p = (pos[:, None] - 1_000 * np.arange(k)[None, ::-1]).reshape(-1) if k else np.zeros(0, np.int64)
        m = rows * k
        return [d(np.arange(rows + 1) * k, np.int32), d(p, np.int32), d(np.full(m, 51), np.int32),
                d(np.arange(m), np.int32), d(np.ones(m), np.int32), d(np.full(m, 2), np.uint8),
                hot.genome.seq.index_select(0, d(p, np.int64)) if m else d(np.zeros(1), np.uint8)]
    ex = {k: lists(k) for k in (0, 1, 8)}
    fns = {"vf_encode_windows": lambda: ops.encode_windows(*args, span, pitch),
           "vf_encode_windows_edit": lambda: ops.encode_windows_edit(*args, *edit, span, pitch),
           **{f"vf_encode_windows_edits ({k} per row)": (lambda k=k: ops.encode_windows_edits(*args, *ex[k], span, pitch))
              for k in ex}}
    if parent_lib:                                                 # the parent commit's one-record kernel, same arguments
        plib = ctypes.CDLL(parent_lib)
        plib.vf_encode_windows_edit.argtypes, plib.vf_encode_windows_edit.restype = _lib.SIGNATURES["vf_encode_windows_edit"]
        ptr = lambda t: t.data_ptr()
        out = torch.empty((rows, pitch), dtype=torch.uint8, device="cuda")
        olen = torch.empty(rows, dtype=torch.int32, device="cuda"); app = torch.empty(rows, dtype=torch.uint8, device="cuda")
        err = torch.zeros(1, dtype=torch.int32, device="cuda")
        v = sv.dev
        pargs = [ptr(x) for x in args[:7]] + [ptr(v[k]) for k in ("pos", "ref_len", "alt_off", "alt_len", "gt", "alt_pool")] + \
            [ptr(x) for x in edit] + [rows, span, ptr(out), pitch, ptr(olen), ptr(app), ptr(err),
                                      torch.cuda.current_stream().cuda_stream]
        fns["vf_encode_windows_edit (parent commit)"] = lambda: plib.vf_encode_windows_edit(*pargs)
        fns["vf_encode_windows_edit"]()
        mine = ops.encode_windows_edit(*args, *edit, span, pitch)
        fns["vf_encode_windows_edit (parent commit)"]()
        torch.cuda.synchronize()
        assert int(err.item()) == 0 and torch.equal(olen, mine[1]) and torch.equal(app, mine[2])
        assert all(torch.equal(out[r, :int(olen[r])], mine[0][r, :int(olen[r])]) for r in range(rows))
    for f in fns.values():
        f()
    ms = {k: 0.0 for k in fns}
    for _ in range(reps):
        for k, f in fns.items():
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); f(); e1.record(); e1.synchronize()
            ms[k] += e0.elapsed_time(e1)
    nbytes = 2.0 * rows * span
    return {"rows": rows, "row_bytes": span, "reps": reps,
            **{k: {"ms": round(v / reps, 4), "GB_per_s": round(nbytes / (v / reps * 1e-3) / 1e9, 1)} for k, v in ms.items()}}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cres", type=int, default=1024)
    ap.add_argument("--tissues", default="1,63")
    ap.add_argument("--baseline", type=int, default=16)
    ap.add_argument("--seed", type=int, default=11)
    ap.add_argument("--parent-lib", default=None)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    torch.cuda.set_device(0)
    cfg, hp = dict(random_init.V4_PCG_MODEL), dict(random_init.SEQ2REG_HP)
    eng = Engine(random_init.make_state_dict(cfg, hp, seed=a.seed, device="cuda"), cfg, hp)
    rng = np.random.default_rng(a.seed)
    chrom_len = 6_000_000
    chrom = synth.make_chromosome(rng, chrom_len, n_rate=0.0)
    var = {"chr1": synth.make_variants(rng, chrom)}
    hot = HotPath(eng, Genome.from_arrays({"chr1": chrom}, "cuda"))
    lay = synth.make_gene_layout(rng, chrom_len, a.cres, strand="+", body_len=300_000, cre_span=600_000)
    g = GeneSpec("chr1", lay["start"], lay["end"], "+", lay["cre_start"], lay["cre_end"], lay["labels"], [0])
    recs = pick_variants(rng, g, chrom, var, hot)
    res = {"workload": f"pair scan of 48 variants (32 in CRE windows, 16 in the gene window) of one gene, C = {a.cres}, "
                       "301 kb gene window; synthetic sample background (SNPs + indels), full-size random-init model, "
                       "synthetic 6 Mb chromosome", **card(), "runs": []}
    for T in [int(x) for x in a.tissues.split(",")]:
        r = run(hot, g, recs, var, T, a.baseline)
        res["runs"].append(r)
        print(json.dumps(r), file=sys.stderr, flush=True)
    res["encoder"] = encoder_rate(hot, var, g, a.parent_lib)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
