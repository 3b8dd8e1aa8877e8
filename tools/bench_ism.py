"""Saturation-mutagenesis throughput on one GPU, with the per-variant path as the baseline in the same run.

    python tools/bench_ism.py [--cres 1024] [--region 300] [--baseline 16] [--out result.json]

Full-size random-init model (utils/random_init), synthetic genome and gene (utils/synth) with --cres CREs.  The region
is --region bp in two halves: one inside a CRE window outside the gene window (CRE-only mutants), one inside the gene
window (gene-window mutants: full re-tokenization of the 301 kb word).  Hom mutants (zygosity 2), T = 1 and T = 63.
Prints one JSON line: mutants/s, ms per mutant split into stage 1 / seq2reg / seq2gene (CUDA events), algorithmic FLOPs
per mutant with and without the window dedup (from the token counts of the windows actually encoded),
vf_mutate_windows GB/s, the per-variant baseline (VEPBatchBuilder.build + predict_step on --baseline of the mutants,
checked bit-identical to the ISM rows), and the card's name and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from variantformer_b200 import ism, ops  # noqa: E402
from variantformer_b200.datasets.vepdataset import VEPBatchBuilder, Variant, cre_windows  # noqa: E402
from variantformer_b200.pipeline import GeneSpec, HotPath  # noqa: E402
from variantformer_b200.stage1 import Genome, gene_window  # noqa: E402
from variantformer_b200.utils import random_init, synth  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        name, power, clk = [x.strip() for x in q.stdout.strip().split(",")]
        return {"gpu": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as e:                                       # the numbers still carry the device name
        return {"gpu": torch.cuda.get_device_name(), "power_limit": f"unavailable ({type(e).__name__})"}


def seq2reg_flops(n_tok, hp, ffn=random_init.FFN_HIDDEN):
    """Window encoder, per window of n tokens: the four GEMMs of each layer + attention (QK^T and PV)."""
    d, L = hp["embedding_dim"], hp["num_layers"]
    n = np.asarray(n_tok, np.float64)
    return float(L * (2 * n * (3 * d * d + d * d + d * 2 * ffn + ffn * d) + 4 * n * n * d).sum())


def seq2gene_flops(C, G, T, cfg, ffn=random_init.FFN_HIDDEN):
    """cre_map / gene_map + CRE stack (C rows, label cross-attention ~free) + gene stack (T (G + 1) rows, cross-
    attention to the C CREs, K/V projection of the CRE context shared by the tissues) per item."""
    D, tdim, NL = cfg["emb_dim"], cfg["token_dim"], cfg["num_layers"]
    lin = 2 * (3 * D * D + D * D + D * D + D * D + D * 2 * ffn + ffn * D)     # qkv, out, q, out2, g1, g2 per row
    M = T * (G + 1)
    cre = (NL - 1) * (C * lin + 4 * C * C * D)
    gene = NL * (M * lin + 4 * T * (G + 1) ** 2 * D + 4 * M * C * D + 2 * C * D * 2 * D)
    return float(2 * C * tdim * D + 2 * G * tdim * D + cre + gene)


class Phases:
    def __init__(self):
        self.ms = {}

    def __call__(self, name):
        ph = self

        class _Ctx:
            def __enter__(self):
                self.e0 = torch.cuda.Event(enable_timing=True); self.e0.record()

            def __exit__(self, *a):
                e1 = torch.cuda.Event(enable_timing=True); e1.record(); e1.synchronize()
                ph.ms[name] = ph.ms.get(name, 0.0) + self.e0.elapsed_time(e1)
        return _Ctx()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--cres", type=int, default=1024)
    ap.add_argument("--region", type=int, default=300)
    ap.add_argument("--baseline", type=int, default=16)
    ap.add_argument("--tissues", default="1,63")
    ap.add_argument("--seed", type=int, default=3)
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
    chrom_len = 5_000_000
    chrom = synth.make_chromosome(rng, chrom_len, n_rate=0.0)
    genome = Genome.from_arrays({"chr1": chrom}, "cuda")
    lay = synth.make_gene_layout(rng, chrom_len, a.cres, strand="+", body_len=300_000, cre_span=600_000)
    gene = GeneSpec("chr1", lay["start"], lay["end"], "+", lay["cre_start"], lay["cre_end"], lay["labels"], [0])
    hot = HotPath(model.engine(), genome)
    _, wins = cre_windows(gene, 50)
    g0, g1 = gene_window(gene.start, gene.end, gene.strand, 1000, 300000)
    half = a.region // 2
    w_out = next((w0, w1) for w0, w1 in wins if (w1 <= g0 or w0 >= g1) and w1 - w0 >= half + 2)
    gpos = next(w0 for w0, w1 in wins if g0 + 5000 < w0 and w1 + 5000 < g1) - 3000          # inside the gene window
    regions = [(w_out[0] + 2, w_out[0] + 1 + half), (gpos, gpos + a.region - half - 1)]
    builder = VEPBatchBuilder(genome)
    res = {"workload": f"ISM {a.region} bp (CRE-only {half} + gene window {a.region - half}), C={len(wins)}, hom",
           **card()}

    # vf_mutate_windows bandwidth: 256 mutant rows of the 301 kB gene window per launch
    t = hot.tokenize([gene])
    gseq, glen = t["gene_seq"]
    n = 256
    d = lambda x, dt: torch.from_numpy(np.asarray(x, dt)).cuda()
    args = (gseq, glen, d([0] * n, np.int32), d(rng.integers(0, int(glen[0]), n), np.int32), d([ord("A")] * n, np.uint8),
            d([0] * n, np.uint8))
    for _ in range(3):
        ops.mutate_windows(*args)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    reps = 50
    e0.record()
    for _ in range(reps):
        ops.mutate_windows(*args)
    e1.record(); e1.synchronize()
    res["mutate_windows_GBps"] = round(2.0 * n * int(glen[0]) * reps / (e0.elapsed_time(e1) * 1e-3) / 1e9, 1)

    for T in [int(x) for x in a.tissues.split(",")]:
        gene.tissues = list(range(T))
        for r0, r1 in regions:                                    # warm-up of every shape of the timed pass
            ism.saturation_mutagenesis(hot, gene, r0, r0 + 5, (2,))
        torch.cuda.synchronize()
        ph = Phases()
        outs = []
        t0 = time.perf_counter()
        for r0, r1 in regions:
            outs.append(ism.saturation_mutagenesis(hot, gene, r0, r1, (2,), timer=ph))
        torch.cuda.synchronize()
        wall = time.perf_counter() - t0
        n_mut = sum(len(o["plan"].mutants) for o in outs)
        # FLOPs from the windows actually encoded (the same stage 1 again, untimed)
        f_dedup = f_plain = s2r_unique = s2r_all = 0.0
        for r0, r1 in regions:
            it = ism.build_items(hot, gene, r0, r1, (2,))
            ct = (it["cre_tokens"] != 0).sum(1).cpu().numpy(); gt = (it["gene_tokens"] != 0).sum(1).cpu().numpy()
            uniq = seq2reg_flops(ct, hp) + seq2reg_flops(gt, hp)
            items = [seq2reg_flops(ct[c], hp) + seq2reg_flops(gt[g], hp) for c, g in zip(it["cre_rows"], it["gene_rows"])]
            s2g = [seq2gene_flops(len(c), len(g), T, cfg) for c, g in zip(it["cre_rows"], it["gene_rows"])]
            s2r_unique += uniq; s2r_all += sum(items)
            f_dedup += sum(s2g) + uniq; f_plain += sum(s2g) + sum(items)
        n_items = n_mut + len(regions)
        r = {"mutants": n_mut, "mutants_per_s": round(n_mut / wall, 2), "ms_per_mutant": round(1e3 * wall / n_mut, 3),
             "ms_per_mutant_split": {k: round(v / n_mut, 3) for k, v in ph.ms.items()},
             "tflop_per_mutant_dedup": round(f_dedup / n_items / 1e12, 3),
             "tflop_per_mutant_per_variant_path": round(f_plain / n_items / 1e12, 3),
             "seq2reg_work_removed": round(1 - s2r_unique / s2r_all, 4),
             "windows_encoded": sum(o["counters"]["windows_encoded"] for o in outs),
             "windows_per_variant": sum(o["counters"]["windows_per_variant"] for o in outs),
             "achieved_tflops_dedup": round(f_dedup / wall / 1e12, 1)}
        # baseline: the per-variant path on a subset, checked bit-identical
        picks = []
        for o in outs:
            m = o["plan"].mutants
            for i in np.linspace(0, len(m) - 1, a.baseline // len(outs)).astype(int):
                picks.append((o, int(i)))
        batches = [builder.build(gene, Variant("chr1", o["plan"].mutants[i].pos, o["plan"].mutants[i].ref,
                                               o["plan"].mutants[i].alt, tissue=gene.tissues)) for o, i in picks[:1]]
        model.predict_step(batches[0], 0)                          # warm-up
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        same = True
        for o, i in picks:
            m = o["plan"].mutants[i]
            b = builder.build(gene, Variant("chr1", m.pos, m.ref, m.alt, tissue=gene.tissues))
            p = model.predict_step(b, 0)
            same &= bool(np.array_equal(p["pred_gene_exp"][2][:, 0], o["pred"][i].cpu().numpy()) and
                         np.array_equal(p["embd"][2], o["emb"][i].cpu().numpy()))
        torch.cuda.synchronize()
        bw = time.perf_counter() - t0
        r["baseline_per_variant"] = {"variants": len(picks), "variants_per_s": round(len(picks) / bw, 2),
                                     "ms_per_variant": round(1e3 * bw / len(picks), 1), "bit_identical": same}
        r["speedup_vs_per_variant"] = round((bw / len(picks)) / (wall / n_mut), 2)
        res[f"T{T}"] = r
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
