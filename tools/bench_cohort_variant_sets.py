"""Variant sets across a cohort on one GPU (HotPath.cohort_variant_sets, what VCFProcessor.cohort_variant_sets runs),
with the per-sample HotPath.variant_sets loop as the baseline in the same run.

    python tools/bench_cohort_variant_sets.py [--samples 64,256] [--tissues 1,63] [--genes 4] [--singles 16]
                                              [--baseline 8] [--out result.json]

Full-size random-init model and the synthetic cohort of tools/bench_cohort.py (6 Mb chromosome, shared sites with
Beta(0.3, 2) allele frequencies plus private variants, one S-column VCF), --genes config-5-like genes at one tissue count
T.  Per gene --singles single-record sets, half in CRE windows and half in the gene window (SNVs and 1-4 bp indels), plus
every pair of them.  For every S and T one JSON object: (sample, set) items/s of the cohort path and of the per-sample
loop on --baseline samples, every compared output (baseline predictions and embeddings, set predictions, applied window
and record flags) checked bit-identical; windows encoded by the cohort path against the loop's (counted on the baseline
samples and scaled to S), items against items scored; the stage1 / keys / seq2reg / seq2gene split (CUDA events; "stage1" excludes the keys); one cohort parse
against S single-sample parses; and the card's name, power limit and max SM clock read in the same run.  Needs a GPU.
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

from tools.bench_cohort import write_vcf  # noqa: E402
from tools.bench_ism import Phases, card  # noqa: E402
from variantformer_b200 import ingest, knockout, variant_sets as vs  # noqa: E402
from variantformer_b200.pipeline import GeneSpec, HotPath  # noqa: E402
from variantformer_b200.stage1 import CohortVariants, Genome, SampleVariants, cre_window, gene_window  # noqa: E402
from variantformer_b200.utils import random_init, synth  # noqa: E402


def gene_sets(rng, chrom, g, n):
    """n single-record sets of gene g (n // 2 in distinct CRE windows, the rest in the gene window) and every pair."""
    o = knockout.batch_order(g)
    cw = [cre_window(g.cre_start[i], g.cre_end[i], 50) for i in o]
    g0, g1 = gene_window(g.start, g.end, g.strand, 1000, 300000)
    recs, used = [], set()
    picks = [("c", int(k)) for k in rng.choice(len(cw), n // 2, replace=False)] + [("g", 0)] * (n - n // 2)
    for kind, k in picks:
        while True:
            p = int(rng.integers(cw[k][0] + 5, cw[k][1] - 10)) if kind == "c" else int(rng.integers(g0 + 10, g1 - 10))
            if all(abs(p - q) > 8 for q in used):
                break
        used.add(p)
        ref = chrom[p:p + 1].tobytes().decode()
        u = rng.random()
        if u < 0.6:
            recs.append(vs.Record("chr1", p + 1, ref, "T" if ref.upper() != "T" else "G", int(rng.integers(1, 3))))
        elif u < 0.8:
            recs.append(vs.Record("chr1", p + 1, ref, ref + "ACGT"[:int(rng.integers(1, 5))], 2))
        else:
            k = int(rng.integers(2, 6))
            recs.append(vs.Record("chr1", p + 1, chrom[p:p + k].tobytes().decode(), ref, 2))
    sets, _, _, _ = vs.pairs(recs)
    return sets


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--samples", default="64,256")
    ap.add_argument("--tissues", default="1,63")
    ap.add_argument("--genes", type=int, default=4)
    ap.add_argument("--singles", type=int, default=16)
    ap.add_argument("--baseline", type=int, default=8)
    ap.add_argument("--seed", type=int, default=11)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("bench_cohort_variant_sets needs a CUDA GPU")
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
    sets = [gene_sets(rng, chrom, g, a.singles) for g in genes]
    n_sets = sum(len(s) for s in sets)
    res = {"workload": f"cohort variant sets: {a.genes} config-5-like genes (C = {[len(g.cre_start) for g in genes]}), "
                       f"{a.singles} single-record sets per gene + their pairs ({n_sets} sets), synthetic 6 Mb "
                       "chromosome, shared sites Beta(0.3, 2) + private variants", **card(), "runs": []}
    tmp = tempfile.mkdtemp(prefix="bench_cohort_sets_")
    try:
        for S in [int(x) for x in a.samples.split(",")]:
            vcf = os.path.join(tmp, f"cohort{S}.vcf")
            names = write_vcf(vcf, np.random.default_rng(a.seed + S), chrom, S)
            t0 = time.perf_counter()
            _, per = ingest.load_vcf_cohort(vcf)
            t_cohort = time.perf_counter() - t0
            t0 = time.perf_counter()
            for n in names:
                ingest.load_vcf_sample(vcf, sample=n)
            t_single = time.perf_counter() - t0
            cv = CohortVariants(names, per, "cuda")
            base = [SampleVariants(per[s], "cuda") for s in range(a.baseline)]
            for T in [int(x) for x in a.tissues.split(",")]:
                for g in genes:
                    g.tissues = list(range(T))
                items = S * n_sets
                hot.cohort_variant_sets(genes, sets, cv, sample_idx=range(min(S, 2)))      # warm-up of the shapes
                hot.variant_sets(genes, sets, base[0])
                torch.cuda.synchronize()
                ph, cnt = Phases(), {}
                t0 = time.perf_counter()
                got = hot.cohort_variant_sets(genes, sets, cv, to_host=False, timer=ph, counters=cnt)
                torch.cuda.synchronize()
                t_c = time.perf_counter() - t0
                pred, emb, sp, app = got[0].cpu().numpy(), got[1].cpu().numpy(), [x.cpu().numpy() for x in got[2]], got[3]
                loop_cnt, outs = [], []
                t0 = time.perf_counter()
                for v in base:
                    c = {}
                    outs.append(hot.variant_sets(genes, sets, v, to_host=False, counters=c))
                    loop_cnt.append(c)
                torch.cuda.synchronize()
                t_b = time.perf_counter() - t0
                for s, o in enumerate(outs):
                    assert np.array_equal(o[0].cpu().numpy(), pred[s]), "baseline differs from the per-sample path"
                    assert np.array_equal(o[1].cpu().numpy(), emb[s]), "baseline embedding differs"
                    for gi in range(len(genes)):
                        assert np.array_equal(o[2][gi].cpu().numpy(), sp[gi][s]), "set prediction differs"
                        assert np.array_equal(o[3][gi]["cre"], app[gi]["cre"][s]) and \
                            np.array_equal(o[3][gi]["gene"], app[gi]["gene"][s]), "applied flags differ"
                        assert all(np.array_equal(x, y[s]) for x, y in zip(o[3][gi]["records"], app[gi]["records"])), \
                            "applied record flags differ"
                ms = ph.ms
                loop_windows = sum(c["windows_encoded"] for c in loop_cnt) * S / a.baseline
                r = {"samples": S, "tissues": T, "sets": n_sets, "items": items,
                     "cohort_items_per_s": round(items / t_c, 1),
                     "per_sample_items_per_s": round(a.baseline * n_sets / t_b, 1),
                     "speedup": round((items / t_c) / (a.baseline * n_sets / t_b), 2),
                     "bit_identical_samples": a.baseline,
                     "windows_encoded": cnt["windows_encoded"], "loop_windows_encoded_scaled_to_S": int(loop_windows),
                     "edited_groups": cnt["edited_groups"], "items_with_baselines": cnt["items"],
                     "items_scored": cnt["items_scored"], "token_rows": cnt["token_rows"], "passes": cnt["passes"],
                     "changed_sample_sets": cnt["changed"],
                     "ms": {"total": round(1e3 * t_c, 1), "stage1": round(ms.get("stage1", 0) - ms.get("keys", 0), 1),
                            "keys": round(ms.get("keys", 0), 2), "seq2reg": round(ms.get("seq2reg", 0), 1),
                            "seq2gene": round(ms.get("seq2gene", 0), 1)},
                     "parse_s": {"one_cohort_parse": round(t_cohort, 3), "single_sample_parses": round(t_single, 3),
                                 "n": S}}
                res["runs"].append(r)
                print(json.dumps(r), file=sys.stderr, flush=True)
                del got, outs
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
