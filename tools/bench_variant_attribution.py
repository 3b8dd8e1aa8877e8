"""Variant-attribution throughput on one GPU (variant_attribution.run): the leave-one-out scan of a synthetic sample, with
the per-edit HotPath.predict loop (a SampleVariants built from the edited table) as the baseline, alternated in the same
run, and each of its outputs checked bit-identical to the scan's.

    python tools/bench_variant_attribution.py [--genes 4] [--tissues 1,63] [--baseline 16] [--rounds 2] [--out f.json]

Full-size random-init model (utils/random_init), synthetic 6 Mb chromosome, a sample at 1 record per 700 bp with 10 %
indels (utils/synth), --genes config-5-like genes (C lognormal around 600, as tools/bench_cohort_variant_sets.py).  The
scan is every record of the sample in a gene's windows removed singly, plus the all-removed (reference) set per gene.
Per T: edit sets/s of the scan and of the loop (best of --rounds alternations), the speed-up, ms split into stage 1 /
seq2reg / seq2gene (CUDA events), windows encoded, and how many sets changed a window.  The card's name and power limit
are read in the same run.  Prints one JSON line.
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
from variantformer_b200 import variant_attribution as va  # noqa: E402
from variantformer_b200.engine import Engine  # noqa: E402
from variantformer_b200.pipeline import GeneSpec, HotPath  # noqa: E402
from variantformer_b200.stage1 import Genome, SampleVariants  # noqa: E402
from variantformer_b200.utils import random_init, synth  # noqa: E402


def edited(var, recs):
    """The sample dict with the planner records' GTs replaced (GT 0 lines deleted)."""
    v = var["chr1"]
    gt = np.asarray(v["gt"], np.uint8).copy()
    for r in recs:
        gt[r[5]] = r[4]
    keep = np.flatnonzero(gt != 0)
    return {"chr1": dict(pos=v["pos"][keep], ref_len=v["ref_len"][keep], alt=[v["alt"][i] for i in keep], gt=gt[keep])}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--tissues", default="1,63")
    ap.add_argument("--genes", type=int, default=4)
    ap.add_argument("--baseline", type=int, default=16)
    ap.add_argument("--rounds", type=int, default=2)
    ap.add_argument("--seed", type=int, default=11)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_variant_attribution needs a CUDA GPU")
    torch.cuda.set_device(0)
    cfg, hp = dict(random_init.V4_PCG_MODEL), dict(random_init.SEQ2REG_HP)
    eng = Engine(random_init.make_state_dict(cfg, hp, seed=a.seed, device="cuda"), cfg, hp)
    rng = np.random.default_rng(a.seed)
    chrom_len = 6_000_000
    chrom = synth.make_chromosome(rng, chrom_len, n_rate=0.0)
    var = {"chr1": synth.make_variants(rng, chrom, rate=1 / 700, indel_frac=0.1)}
    sv = SampleVariants(var, "cuda")
    hot = HotPath(eng, Genome.from_arrays({"chr1": chrom}, "cuda"))
    genes = []
    for _ in range(a.genes):
        C = int(np.clip(rng.lognormal(np.log(600), 0.6), 32, 3000))
        lay = synth.make_gene_layout(rng, chrom_len, C, body_len=int(np.clip(rng.lognormal(np.log(25_000), 1.0), 1_000,
                                                                                 300_000)), cre_span=600_000)
        genes.append(GeneSpec("chr1", lay["start"], lay["end"], lay["strand"], lay["cre_start"], lay["cre_end"],
                              lay["labels"], [0]))
    sets = []
    for g in genes:
        s, _, _ = va.default_sets(g, sv, hot.nb, hot.up, hot.down, "record")
        sets.append(s + [va.all_removed(g, sv, hot.nb, hot.up, hot.down)])
    n_sets = sum(len(s) for s in sets)
    # the loop's subset: --baseline edits spread over the genes (gene index, set index)
    flat = [(gi, j) for gi in range(len(genes)) for j in range(len(sets[gi]))]
    sub = [flat[k] for k in np.linspace(0, len(flat) - 1, a.baseline).astype(int)]
    res = {"workload": f"variant attribution, leave-one-out: {a.genes} config-5-like genes (C = "
                       f"{[len(g.cre_start) for g in genes]}), sample at 1 record / 700 bp, 10 % indels "
                       f"({len(var['chr1']['pos'])} records), {n_sets} edit sets incl. one all-removed set per gene, "
                       "synthetic 6 Mb chromosome", **card(), "runs": []}
    for T in [int(x) for x in a.tissues.split(",")]:
        for g in genes:
            g.tissues = list(range(T))
        va.run(hot, genes, [s[:2] for s in sets], sv)                  # warm-up of the shapes
        hot.predict(genes[:1], sv)
        t_scan, t_loop = [], []
        for _ in range(a.rounds):                                      # alternated
            ph, cnt = Phases(), {}
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            got = va.run(hot, genes, sets, sv, to_host=False, timer=ph, counters=cnt)
            torch.cuda.synchronize()
            t_scan.append(time.perf_counter() - t0)
            sp = [x.cpu().numpy() for x in got[2]]
            del got
            outs = []
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            for gi, j in sub:
                outs.append(hot.predict([genes[gi]], SampleVariants(edited(var, sets[gi][j]), "cuda"), to_host=False))
            torch.cuda.synchronize()
            t_loop.append(time.perf_counter() - t0)
            for (gi, j), o in zip(sub, outs):
                assert np.array_equal(o[0].cpu().numpy(), sp[gi][j]), "an edit differs from predict on the edited table"
        ms = ph.ms
        r = {"tissues": T, "sets": n_sets, "scan_sets_per_s": round(n_sets / min(t_scan), 1),
             "loop_sets_per_s": round(len(sub) / min(t_loop), 2),
             "speedup": round((n_sets / min(t_scan)) / (len(sub) / min(t_loop)), 2), "bit_identical_sets": len(sub),
             "scan_s": [round(x, 3) for x in t_scan], "loop_s": [round(x, 3) for x in t_loop],
             "windows_encoded": cnt["windows_encoded"], "windows_per_item": cnt["windows_per_item"],
             "gene_windows_edited": cnt["gene_windows_edited"], "cre_windows_edited": cnt["cre_windows_edited"],
             "changed_sets": cnt["changed"], "passes": cnt["passes"],
             "ms": {k: round(ms.get(k, 0), 1) for k in ("stage1", "seq2reg", "seq2gene")}}
        res["runs"].append(r)
        print(json.dumps(r), file=sys.stderr, flush=True)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
