"""In-silico CRE knockout throughput on one GPU (HotPath.cre_knockout), with the per-knockout HotPath.predict loop as the
baseline in the same run.

    python tools/bench_knockout.py [--cres 1024] [--genes 4] [--tissues 1,63] [--baseline 16] [--out result.json]

Full-size random-init model (utils/random_init), reference genome only (synthetic, utils/synth).  Two workloads, every
single-CRE knockout of every gene, at each T:
  * one gene with --cres CREs and a 301 kb gene window (a 300 kb body), as tools/bench_ism.py;
  * --genes config-5-like genes drawn as in tools/bench_cohort.py (C lognormal around 600, clipped to 32-3000).
Per (workload, T) one JSON object: knockouts/s; ms per knockout split into stage 1 / seq2reg / seq2gene (CUDA events);
distinct windows encoded against the windows the per-knockout path encodes; the per-knockout predict loop on --baseline
knockouts spread over the genes, each output checked bit-identical to the knockout path's; the speed-up; and the card's
name and power limit read in the same run.  Prints one JSON line.
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
from variantformer_b200.engine import Engine  # noqa: E402
from variantformer_b200.pipeline import GeneSpec, HotPath  # noqa: E402
from variantformer_b200.stage1 import Genome  # noqa: E402
from variantformer_b200.utils import random_init, synth  # noqa: E402


def reduced(g, knocked):
    keep = np.setdiff1d(np.arange(len(g.cre_start)), knocked)
    return GeneSpec(g.chrom, g.start, g.end, g.strand, g.cre_start[keep], g.cre_end[keep],
                    np.asarray(g.cre_labels)[keep], list(g.tissues))


def run(hot, genes, T, n_base):
    for g in genes:
        g.tissues = list(range(T))
    warm = [[[0], [len(g.cre_start) - 1]] for g in genes]
    hot.cre_knockout(genes, warm)                                      # warm-up of the kernels and allocator
    hot.predict([reduced(genes[0], [0])])
    torch.cuda.synchronize()
    ph, cnt = Phases(), {}
    t0 = time.perf_counter()
    _, _, ko_pred = hot.cre_knockout(genes, None, to_host=False, timer=ph, counters=cnt)
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    ko_pred = [p.cpu().numpy() for p in ko_pred]
    n = cnt["knockouts"]
    picks = [(gi, int(k)) for gi, g in enumerate(genes)
             for k in np.linspace(0, len(g.cre_start) - 1, max(1, n_base // len(genes))).astype(int)]
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    outs = [hot.predict([reduced(genes[gi], [k])], to_host=False)[0] for gi, k in picks]
    torch.cuda.synchronize()
    bw = time.perf_counter() - t0
    same = all(np.array_equal(o.cpu().numpy(), ko_pred[gi][k]) for o, (gi, k) in zip(outs, picks))
    assert same, "knockout output differs from the per-knockout path"
    return {"tissues": T, "knockouts": n, "knockouts_per_s": round(n / wall, 1),
            "ms_per_knockout": round(1e3 * wall / n, 3),
            "ms_per_knockout_split": {k: round(v / n, 3) for k, v in ph.ms.items()},
            "windows_encoded": cnt["windows_encoded"], "windows_per_item_path": cnt["windows_per_item"],
            "items": cnt["items"], "slabs": cnt["slabs"], "passes": cnt["passes"],
            "baseline_per_knockout_predict": {"knockouts": len(picks), "knockouts_per_s": round(len(picks) / bw, 1),
                                              "ms_per_knockout": round(1e3 * bw / len(picks), 2),
                                              "bit_identical": same},
            "speedup": round((bw / len(picks)) / (wall / n), 2)}


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
    hot = HotPath(eng, Genome.from_arrays({"chr1": chrom}, "cuda"))
    lay = synth.make_gene_layout(rng, chrom_len, a.cres, strand="+", body_len=300_000, cre_span=600_000)
    big = [GeneSpec("chr1", lay["start"], lay["end"], "+", lay["cre_start"], lay["cre_end"], lay["labels"], [0])]
    cfg5 = []
    for _ in range(a.genes):
        C = int(np.clip(rng.lognormal(np.log(600), 0.6), 32, 3000))
        lay = synth.make_gene_layout(rng, chrom_len, C, body_len=int(np.clip(rng.lognormal(np.log(25_000), 1.0), 1_000,
                                                                                 300_000)), cre_span=600_000)
        cfg5.append(GeneSpec("chr1", lay["start"], lay["end"], lay["strand"], lay["cre_start"], lay["cre_end"],
                             lay["labels"], [0]))
    res = {"workload": "every single-CRE knockout, reference genome, full-size random-init model, synthetic 6 Mb "
                       "chromosome", **card(), "runs": []}
    for name, genes in ((f"one gene, C = {a.cres}, 301 kb gene window", big),
                        (f"{a.genes} config-5-like genes (C = {[len(g.cre_start) for g in cfg5]})", cfg5)):
        for T in [int(x) for x in a.tissues.split(",")]:
            r = {"genes": name, **run(hot, genes, T, a.baseline)}
            res["runs"].append(r)
            print(json.dumps(r), file=sys.stderr, flush=True)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
