"""Cohort throughput on one GPU (HotPath.predict_cohort, what VCFProcessor.predict_cohort runs), with the per-sample
loop as the baseline in the same run.

    python tools/bench_cohort.py [--samples 64,256] [--tissues 1,63] [--genes 4] [--baseline 8] [--out result.json]

Full-size random-init model (utils/random_init), a synthetic 6 Mb chromosome (utils/synth) and --genes genes drawn
like bench.py --config 5 (C lognormal around 600, clipped to 32-3000; lognormal gene bodies), every gene at one tissue
count T.  The cohort: shared sites at one per 250 bp whose allele frequencies follow a skewed Beta(0.3, 2), plus one
private variant per 20 kb per sample (SNVs and 1-5 bp indels), written as one S-column VCF.
For every S and T one JSON object: predictions/s of the cohort path and of the per-sample loop (HotPath.predict with
that sample's SampleVariants) on --baseline samples, every compared prediction and embedding checked bit-identical;
(sample, window) rows against distinct encoded windows, (sample, token row) pairs against distinct token rows; the
stage 1 / keys / seq2reg / seq2gene split (CUDA events; "stage1" excludes the keys); one cohort parse of the VCF against S single-sample parses;
and the card's name and power limit read in the same run.  Prints one JSON line.
"""
import argparse
import json
import os
import sys
import tempfile
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from tools.bench_ism import Phases, card  # noqa: E402
from variantformer_b200 import ingest  # noqa: E402
from variantformer_b200.pipeline import GeneSpec, HotPath  # noqa: E402
from variantformer_b200.stage1 import CohortVariants, Genome, SampleVariants  # noqa: E402
from variantformer_b200.utils import random_init, synth  # noqa: E402


def write_vcf(path, rng, chrom, n_samples, site_rate=1 / 250, private_rate=1 / 20000):
    sites = synth.make_variants(rng, chrom, rate=site_rate)
    af = rng.beta(0.3, 2.0, len(sites["pos"]))
    g = (rng.random((len(af), n_samples)) < af[:, None]).astype(np.int64) + \
        (rng.random((len(af), n_samples)) < af[:, None]).astype(np.int64)
    lines = []
    gts = np.asarray(["0/0", "0/1", "1/1"])
    for i, (p, rl, a) in enumerate(zip(sites["pos"], sites["ref_len"], sites["alt"])):
        ref = chrom[p:p + rl].tobytes().decode().upper()
        lines.append((int(p), f"chr1\t{p + 1}\t.\t{ref}\t{a.decode()}\t.\tPASS\t.\tGT\t" + "\t".join(gts[g[i]])))
    hom_ref = ["0/0"] * n_samples
    for s in range(n_samples):
        v = synth.make_variants(rng, chrom, rate=private_rate, indel_frac=0.2)
        for p, rl, a, gt in zip(v["pos"], v["ref_len"], v["alt"], v["gt"]):
            cols = list(hom_ref); cols[s] = "0/1" if gt == 1 else "1/1"
            ref = chrom[p:p + rl].tobytes().decode().upper()
            lines.append((int(p), f"chr1\t{p + 1}\t.\t{ref}\t{a.decode()}\t.\tPASS\t.\tGT\t" + "\t".join(cols)))
    lines.sort(key=lambda x: x[0])
    names = [f"S{i:04d}" for i in range(n_samples)]
    with open(path, "w") as f:
        f.write("##fileformat=VCFv4.2\n#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t" + "\t".join(names) + "\n")
        for _, l in lines:
            f.write(l + "\n")
    return names


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", default="64,256")
    ap.add_argument("--tissues", default="1,63")
    ap.add_argument("--genes", type=int, default=4)
    ap.add_argument("--baseline", type=int, default=8)
    ap.add_argument("--seed", type=int, default=11)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    torch.cuda.set_device(0)
    cfg, hp = dict(random_init.V4_PCG_MODEL), dict(random_init.SEQ2REG_HP)
    from variantformer_b200.engine import Engine
    eng = Engine(random_init.make_state_dict(cfg, hp, seed=a.seed, device="cuda"), cfg, hp)
    rng = np.random.default_rng(a.seed)
    chrom_len = 6_000_000
    chrom = synth.make_chromosome(rng, chrom_len, n_rate=0.0)
    hot = HotPath(eng, Genome.from_arrays({"chr1": chrom}, "cuda"))
    genes = []
    for _ in range(a.genes):
        C = int(np.clip(rng.lognormal(np.log(600), 0.6), 32, 3000))
        lay = synth.make_gene_layout(rng, chrom_len, C, body_len=int(np.clip(rng.lognormal(np.log(25_000), 1.0), 1_000,
                                                                                 300_000)), cre_span=600_000)
        genes.append(GeneSpec("chr1", lay["start"], lay["end"], lay["strand"], lay["cre_start"], lay["cre_end"],
                              lay["labels"], [0]))
    res = {"workload": f"cohort: {a.genes} config-5-like genes (C = {[len(g.cre_start) for g in genes]}), synthetic "
                       "6 Mb chromosome, shared sites Beta(0.3, 2) + private variants", **card(), "runs": []}
    tmp = tempfile.mkdtemp(prefix="bench_cohort_")
    try:
        for S in [int(x) for x in a.samples.split(",")]:
            vcf = os.path.join(tmp, f"cohort{S}.vcf")
            names = write_vcf(vcf, np.random.default_rng(a.seed + S), chrom, S)
            t0 = time.perf_counter()
            got_names, per = ingest.load_vcf_cohort(vcf)
            t_cohort = time.perf_counter() - t0
            t0 = time.perf_counter()
            singles = [ingest.load_vcf_sample(vcf, sample=n) for n in names]
            t_single = time.perf_counter() - t0
            assert got_names == names
            for d, w in zip(per, singles):
                assert d.keys() == w.keys() and all(np.array_equal(d[c]["pos"], w[c]["pos"]) and d[c]["alt"] == w[c]["alt"]
                                                    for c in d)
            del singles
            cv = CohortVariants(names, per, "cuda")
            base = [SampleVariants(per[s], "cuda") for s in range(a.baseline)]
            for T in [int(x) for x in a.tissues.split(",")]:
                for g in genes:
                    g.tissues = list(range(T))
                n_pred = S * sum(len(g.tissues) for g in genes)
                hot.predict_cohort(genes, cv, sample_idx=range(min(S, 4)))          # warm-up of the shapes
                for v in base[:1]:
                    hot.predict(genes, v)
                torch.cuda.synchronize()
                ph, cnt = Phases(), {}
                t0 = time.perf_counter()
                pred, emb = hot.predict_cohort(genes, cv, to_host=False, timer=ph, counters=cnt)
                torch.cuda.synchronize()
                t_c = time.perf_counter() - t0
                pred_h, emb_h = pred.cpu().numpy(), emb.cpu().numpy()
                t0 = time.perf_counter()
                outs = [hot.predict(genes, v, to_host=False)[:2] for v in base]
                torch.cuda.synchronize()
                t_b = time.perf_counter() - t0
                same = all(np.array_equal(p.cpu().numpy(), pred_h[s]) and np.array_equal(e.cpu().numpy(), emb_h[s])
                           for s, (p, e) in enumerate(outs))
                assert same, "cohort output differs from the per-sample path"
                ms = ph.ms
                r = {"samples": S, "tissues": T, "predictions": n_pred,
                     "cohort_predictions_per_s": round(n_pred / t_c, 1),
                     "per_sample_predictions_per_s": round(a.baseline * n_pred / S / t_b, 1),
                     "speedup": round((n_pred / t_c) / (a.baseline * n_pred / S / t_b), 2),
                     "bit_identical_samples": a.baseline,
                     "sample_window_rows": cnt["sample_windows"], "distinct_windows_encoded": cnt["windows_encoded"],
                     "sample_token_rows": cnt["sample_token_rows"], "distinct_token_rows": cnt["token_rows"],
                     "cre_token_rows": cnt["cre_token_rows"],
                     "gene_token_rows": cnt["gene_token_rows"], "items": cnt["items"],
                     "items_scored": cnt["items_scored"], "passes": cnt["passes"],
                     "ms": {"total": round(1e3 * t_c, 1), "stage1": round(ms.get("stage1", 0) - ms.get("keys", 0), 1),
                            "keys": round(ms.get("keys", 0), 2), "seq2reg": round(ms.get("seq2reg", 0), 1),
                            "seq2gene": round(ms.get("seq2gene", 0), 1)},
                     "parse_s": {"one_cohort_parse": round(t_cohort, 3), "single_sample_parses": round(t_single, 3),
                                 "n": S}}
                res["runs"].append(r)
                print(json.dumps(r), file=sys.stderr, flush=True)
                del pred, emb, outs
            del cv, base
    finally:
        for f in os.listdir(tmp):
            os.remove(os.path.join(tmp, f))
        os.rmdir(tmp)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
