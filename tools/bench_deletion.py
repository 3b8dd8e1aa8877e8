"""In-silico deletion throughput on one GPU (HotPath.deletion_scan), with the per-deletion HotPath.predict loop (the
deletion's record added to the sample) as the baseline in the same run, and the rate of vf_encode_windows_edit next to
vf_encode_windows.

    python tools/bench_deletion.py [--cres 1024] [--genes 4] [--tissues 1,63] [--baseline 16] [--out result.json]

Full-size random-init model (utils/random_init), synthetic 6 Mb chromosome and a synthetic sample background (SNPs and
indels, utils/synth).  Two workloads, at each T:
  * one gene with --cres CREs and a 301 kb gene window, scanned by 50 bp tiles at step 25 over a 20 kb region that
    straddles the gene window's start, so it covers CRE windows inside and outside the gene window;
  * the default CRE scan (every CRE's own bases deleted singly) of --genes config-5-like genes (as tools/bench_knockout).
Per (workload, T) one JSON object: deletions/s; ms per deletion split into stage 1 / seq2reg / seq2gene (CUDA events);
windows encoded against the windows the per-deletion path encodes; the per-deletion predict loop on --baseline
deletions, each output checked bit-identical; the speed-up.  Then the encoder rate on 256 gene-window rows, both
kernels timed alternately in the same run (bytes = reference bytes read + row bytes written), and the card's name and
power limit read in the same run.  Prints one JSON line.
"""
import argparse
import json
import os
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from tools.bench_ism import Phases, card  # noqa: E402
from variantformer_b200 import deletion, ops  # noqa: E402
from variantformer_b200.engine import Engine  # noqa: E402
from variantformer_b200.pipeline import GeneSpec, HotPath  # noqa: E402
from variantformer_b200.stage1 import Genome, SampleVariants, gene_window  # noqa: E402
from variantformer_b200.utils import random_init, synth  # noqa: E402


def with_record(var, chrom, a, b):
    v = var["chr1"]
    k = int(np.searchsorted(v["pos"], a - 2, "right"))
    rec = dict(pos=np.insert(v["pos"], k, a - 2), ref_len=np.insert(v["ref_len"], k, b - a + 2),
               alt=v["alt"][:k] + [bytes([chrom[a - 2]])] + v["alt"][k:], gt=np.insert(v["gt"], k, 2))
    return SampleVariants({"chr1": rec}, "cuda")


def run(hot, genes, spans, var, chrom, T, n_base):
    sv = SampleVariants(var, "cuda")
    for g in genes:
        g.tissues = list(range(T))
    hot.deletion_scan(genes, [s[:2] for s in spans], sv)              # warm-up of the kernels and allocator
    torch.cuda.synchronize()
    ph, cnt = Phases(), {}
    t0 = time.perf_counter()
    _, _, dp, _ = hot.deletion_scan(genes, spans, sv, to_host=False, timer=ph, counters=cnt)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    dp = [p.cpu().numpy() for p in dp]
    n = cnt["deletions"]
    picks = [(gi, int(k)) for gi, s in enumerate(spans)
             for k in np.linspace(0, len(s) - 1, max(1, n_base // len(genes))).astype(int)]
    svs = [with_record(var, chrom, *spans[gi][k]) for gi, k in picks]
    hot.predict([genes[0]], svs[0], to_host=False)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    outs = [hot.predict([genes[gi]], s, to_host=False)[0] for (gi, k), s in zip(picks, svs)]
    torch.cuda.synchronize()
    bw = time.perf_counter() - t0
    same = all(np.array_equal(o.cpu().numpy(), dp[gi][k]) for o, (gi, k) in zip(outs, picks))
    assert same, "deletion output differs from the per-deletion path"
    return {"tissues": T, "deletions": n, "changed": cnt["changed"], "deletions_per_s": round(n / wall, 1),
            "ms_per_deletion": round(1e3 * wall / n, 3),
            "ms_per_deletion_split": {k: round(v / n, 3) for k, v in ph.ms.items()},
            "windows_encoded": cnt["windows_encoded"], "windows_per_item_path": cnt["windows_per_item"],
            "cre_windows_edited": cnt["cre_windows_edited"], "gene_windows_edited": cnt["gene_windows_edited"],
            "cre_token_rows": cnt["cre_token_rows"], "gene_token_rows": cnt["gene_token_rows"],
            "items": cnt["items"], "slabs": cnt["slabs"], "passes": cnt["passes"],
            "baseline_per_deletion_predict": {"deletions": len(picks), "deletions_per_s": round(len(picks) / bw, 1),
                                              "ms_per_deletion": round(1e3 * bw / len(picks), 2),
                                              "bit_identical": same},
            "speedup": round((bw / len(picks)) / (wall / n), 2)}


def encoder_rate(hot, var, g, rows=256, reps=20):
    """vf_encode_windows_edit against vf_encode_windows on `rows` copies of g's gene window, each with its own 50 bp
    deletion (edit) / without it (plain), alternated in one run."""
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
    fns = {"vf_encode_windows": lambda: ops.encode_windows(*args, span, pitch),
           "vf_encode_windows_edit": lambda: ops.encode_windows_edit(*args, *edit, span, pitch)}
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
    ap.add_argument("--genes", type=int, default=4)
    ap.add_argument("--tissues", default="1,63")
    ap.add_argument("--baseline", type=int, default=16)
    ap.add_argument("--seed", type=int, default=11)
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
    big = [GeneSpec("chr1", lay["start"], lay["end"], "+", lay["cre_start"], lay["cre_end"], lay["labels"], [0])]
    g0, _ = gene_window(big[0].start, big[0].end, "+", hot.up, hot.down)
    tl = deletion.tiles("chr1", g0 - 10_000, g0 + 9_999, 50, 25)
    big_spans = [tl[["start", "end"]].to_numpy(np.int64)]
    cfg5 = []
    for _ in range(a.genes):
        C = int(np.clip(rng.lognormal(np.log(600), 0.6), 32, 3000))
        lay = synth.make_gene_layout(rng, chrom_len, C, body_len=int(np.clip(rng.lognormal(np.log(25_000), 1.0), 1_000,
                                                                                 300_000)), cre_span=600_000)
        cfg5.append(GeneSpec("chr1", lay["start"], lay["end"], lay["strand"], lay["cre_start"], lay["cre_end"],
                             lay["labels"], [0]))
    cfg5_spans = [np.stack([g.cre_start + 1, g.cre_end], 1).astype(np.int64) for g in cfg5]
    res = {"workload": "in-silico deletions, synthetic sample background (SNPs + indels), full-size random-init model, "
                       "synthetic 6 Mb chromosome", **card(), "runs": []}
    for name, genes, spans in ((f"one gene, C = {a.cres}, 301 kb gene window, 50 bp tiles at step 25 over 20 kb "
                                "straddling the gene window's start", big, big_spans),
                               (f"default CRE scan of {a.genes} config-5-like genes (C = "
                                f"{[len(g.cre_start) for g in cfg5]})", cfg5, cfg5_spans)):
        for T in [int(x) for x in a.tissues.split(",")]:
            r = {"genes": name, **run(hot, genes, spans, var, chrom, T, a.baseline)}
            res["runs"].append(r)
            print(json.dumps(r), file=sys.stderr, flush=True)
    res["encoder"] = encoder_rate(hot, var, big[0])
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
