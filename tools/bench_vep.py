"""Variant-table throughput on one GPU (vep_batch.score_pairs, what VariantProcessor.predict_batched runs), with the
per-pair path as the baseline in the same run.

    python tools/bench_vep.py [--cres 1024] [--baseline 16] [--tissues 1,63] [--out result.json]

Full-size random-init model (utils/random_init), synthetic genome and genes (utils/synth) with --cres CREs each.
Workloads:
  dense   256 variants in one gene: 128 in CRE windows outside the gene window (half SNVs, half 2-20 bp insertion ALTs)
          and 128 SNVs in the gene window (an insertion there writes a het 'N' at the variant base, which the per-pair
          path rejects with a ValueError, so a table cannot hold one);
  sparse  64 genes x 1 variant (even genes: a CRE-window insertion, odd genes: a gene-window SNV): no reference item
          is shared, only slab packing and window dedup remain.
Each at every --tissues count.  Prints one JSON line: pairs/s, ms per pair split into stage 1 / seq2reg / seq2gene (CUDA
events), windows encoded against the per-pair count, vf_splice_windows GB/s, the per-pair baseline (VEPBatchBuilder.build
+ predict_step on --baseline pairs, checked bit-identical in every output), and the card's name and power limit read
in the same run.
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
from variantformer_b200 import ops, vep_batch  # noqa: E402
from variantformer_b200.datasets.vepdataset import VEPBatchBuilder, Variant, cre_windows  # noqa: E402
from variantformer_b200.pipeline import GeneSpec, HotPath  # noqa: E402
from variantformer_b200.stage1 import Genome, gene_window  # noqa: E402
from variantformer_b200.utils import random_init, synth  # noqa: E402


def _sites(gene):
    _, wins = cre_windows(gene, 50)
    g0, g1 = gene_window(gene.start, gene.end, gene.strand, 1000, 300000)
    return [w for w in wins if w[1] <= g0 or w[0] >= g1], (g0, g1)


def _alt(r, rng):
    return str(rng.choice([b for b in "ACGT" if b != r]))


def workloads(rng, chrom, genes):
    seq = lambda p: chr(chrom[p - 1]).upper()
    ins = lambda: "".join(rng.choice(list("ACGT"), int(rng.integers(2, 21))))
    dense, g = [], genes[0]
    outside, (g0, g1) = _sites(g)
    for i in range(256):
        if i < 128:
            a, b = outside[int(rng.integers(0, len(outside)))]
            p = int(rng.integers(a + 1, b + 1))
            alt = _alt(seq(p), rng) if i % 2 else ins()
        else:
            p = int(rng.integers(g0 + 1, g1 + 1))
            alt = _alt(seq(p), rng)
        dense.append(dict(variant=Variant("chr1", p, seq(p), alt, tissue=None), gene=g, gene_id="g0"))
    sparse = []
    for j, g in enumerate(genes[1:65]):
        outside, (g0, g1) = _sites(g)
        if j % 2 == 0 and outside:
            a, b = outside[int(rng.integers(0, len(outside)))]
            p = int(rng.integers(a + 1, b + 1)); alt = ins()
        else:
            p = int(rng.integers(g0 + 1, g1 + 1)); alt = _alt(seq(p), rng)
        sparse.append(dict(variant=Variant("chr1", p, seq(p), alt, tissue=None), gene=g, gene_id=f"g{j + 1}"))
    return {"dense": dense, "sparse": sparse}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cres", type=int, default=1024)
    ap.add_argument("--baseline", type=int, default=16)
    ap.add_argument("--tissues", default="1,63")
    ap.add_argument("--seed", type=int, default=4)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    torch.cuda.set_device(0)
    from variantformer_b200.seq2gene.model_combined_modulator import Seq2GenePredictorCombinedModulator, attach_trainer
    from variantformer_b200.seq2reg.model import Seq2RegPredictor
    cfg, hp = dict(random_init.V4_PCG_MODEL), dict(random_init.SEQ2REG_HP)
    model = Seq2GenePredictorCombinedModulator(cre_tokenizer=Seq2RegPredictor(**hp), gene_tokenizer=Seq2RegPredictor(**hp),
                                               **cfg)
    model.load_state_dict(random_init.make_state_dict(cfg, hp, seed=a.seed, device="cuda"))
    model.eval().to("cuda"); model.vep = True; attach_trainer(model)
    rng = np.random.default_rng(a.seed)
    chrom_len = 8_000_000
    chrom = synth.make_chromosome(rng, chrom_len, n_rate=0.0)
    genome = Genome.from_arrays({"chr1": chrom}, "cuda")
    genes = []
    for i in range(65):
        lay = synth.make_gene_layout(rng, chrom_len, a.cres, strand="+-"[i % 2], body_len=int(rng.integers(20_000, 300_000)),
                                     cre_span=600_000)
        genes.append(GeneSpec("chr1", lay["start"], lay["end"], lay["strand"], lay["cre_start"], lay["cre_end"],
                              lay["labels"], [0]))
    hot = HotPath(model.engine(), genome)
    builder = VEPBatchBuilder(genome)
    res = {"workload": f"variant tables, C={a.cres}: dense = 256 variants x 1 gene (64 CRE SNVs, 64 CRE insertions of "
                       "2-20 bp, 128 gene-window SNVs); sparse = 64 genes x 1 variant", **card()}

    # vf_splice_windows bandwidth: 256 rows of the 301 kB gene window per launch, 10-base insertions
    t = hot.tokenize([genes[0]])
    gseq, glen = t["gene_seq"]
    n, k = 256, 10
    d = lambda x, dt: torch.from_numpy(np.asarray(x, dt)).cuda()
    args = (gseq, glen, d([0] * n, np.int32), d(rng.integers(0, int(glen[0]), n), np.int32),
            d(rng.integers(65, 85, n * k), np.uint8), d(np.arange(n) * k, np.int32), d([k] * n, np.int32),
            d([0] * n, np.uint8), gseq.shape[1] + 16)
    for _ in range(3):
        ops.splice_windows(*args)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 50
    e0.record()
    for _ in range(reps):
        ops.splice_windows(*args)
    e1.record(); e1.synchronize()
    res["splice_windows_GBps"] = round(n * (2.0 * int(glen[0]) + k - 1) * reps / (e0.elapsed_time(e1) * 1e-3) / 1e9, 1)

    for T in [int(x) for x in a.tissues.split(",")]:
        for g in genes:
            g.tissues = list(range(T))
        for name, pairs in workloads(np.random.default_rng(a.seed + 1), chrom, genes).items():
            for p in pairs:
                p["variant"].tissue = list(range(T))
            vep_batch.score_pairs(hot, pairs[:3])                      # warm-up
            torch.cuda.synchronize()
            ph = Phases()
            t0 = time.perf_counter()
            out, c = vep_batch.score_pairs(hot, pairs, timer=ph)
            torch.cuda.synchronize()
            wall = time.perf_counter() - t0
            n_p = len(pairs)
            r = {"pairs": n_p, "items": c["items"], "pairs_per_s": round(n_p / wall, 2),
                 "ms_per_pair": round(1e3 * wall / n_p, 3),
                 "ms_per_pair_split": {k_: round(v / n_p, 3) for k_, v in ph.ms.items()},
                 "windows_encoded": c["windows_encoded"], "windows_per_pair_path": c["windows_per_pair"]}
            # baseline: the per-pair path on a subset, checked bit-identical in every output
            picks = np.linspace(0, n_p - 1, min(a.baseline, n_p)).astype(int)
            model.predict_step(builder.build(pairs[0]["gene"], pairs[0]["variant"]), 0)          # warm-up
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            same = True
            for i in picks:
                want = model.predict_step(builder.build(pairs[i]["gene"], pairs[i]["variant"]), 0)
                for key in ("pred_gene_exp", "embd", "gene_token_embedding", "cre_token_embedding"):
                    same &= all(np.array_equal(x, y) for x, y in zip(want[key], out[i][key]))
                same &= want["variant_type"] == out[i]["variant_type"]
            torch.cuda.synchronize()
            bw = time.perf_counter() - t0
            r["baseline_per_pair"] = {"pairs": len(picks), "pairs_per_s": round(len(picks) / bw, 2),
                                      "ms_per_pair": round(1e3 * bw / len(picks), 1), "bit_identical": bool(same)}
            r["speedup_vs_per_pair"] = round((bw / len(picks)) / (wall / n_p), 2)
            res[f"{name}_T{T}"] = r
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
