"""Cost of the gene -> CRE cross-attention maps on one GPU (Engine.run(slab, cre_attention=True)).

    python tools/bench_cre_attention.py [--genes 8] [--cres 1024] [--chunks 200] [--tissues 63] [--reps 10] [--out r.json]

Full-size random-init model (utils/random_init), the benchmark's config-3 slab as synthetic tokens (utils/synth): 8 genes
x C = 1024 CRE windows x G = 200 gene chunks x T = 63 tissues.  Stages 2-4 of the slab run --reps times without and with
the maps, alternating in one process, each timed with CUDA events (median and spread reported).  The kernel alone
(vf_cross_attention_probs on the slab's registry rows, one launch per gene layer, on K of the same shape) is timed over
--reps x n_layers launches; bytes written per second = map bytes / kernel time.  Prints one JSON line with the card's
name and power limit read in the same run.
"""
import argparse
import json
import os
import subprocess
import sys

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from variantformer_b200 import ops  # noqa: E402
from variantformer_b200.engine import Engine, cre_attention_layout  # noqa: E402
from variantformer_b200.utils import random_init, synth  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader",
                            "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30)
        name, power, clk = [x.strip() for x in q.stdout.strip().split(",")]
        return {"gpu": name, "power_limit": power, "sm_max_clock": clk}
    except Exception as e:
        return {"gpu": torch.cuda.get_device_name(), "power_limit": f"unavailable ({type(e).__name__})"}


def timed(fn):
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); r = fn(); e1.record(); e1.synchronize()
    return e0.elapsed_time(e1), r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--genes", type=int, default=8)
    ap.add_argument("--cres", type=int, default=1024)
    ap.add_argument("--chunks", type=int, default=200)
    ap.add_argument("--tissues", type=int, default=63)
    ap.add_argument("--reps", type=int, default=10)
    ap.add_argument("--out", default=None)
    a = ap.parse_args()
    cfg, hp = dict(random_init.V4_PCG_MODEL), dict(random_init.SEQ2REG_HP)
    sd = random_init.make_state_dict(cfg, hp, seed=0, device="cuda")
    eng = Engine(sd, cfg, hp)
    batch = synth.token_batch(7, a.genes, a.cres, a.chunks, a.tissues)
    sq = lambda xs: [x[:, 0, :] for x in xs]
    slab = eng.prepare(sq(batch["cre_sequences"]), sq(batch["cre_attention_masks"]), sq(batch["gene_embeddings"]),
                       sq(batch["gene_attention_masks"]), batch["tissue_context"], batch["ref_cre_labels"])
    L, H, hd, D = eng.w.NL, eng.w.H, eng.w.hd, eng.w.D

    # ---- forward with and without the maps, alternating ----
    plain, maps = [], []
    out0 = eng.run(slab); out1 = eng.run(slab, cre_attention=True)          # warm-up of both
    torch.cuda.synchronize()
    identical = bool(torch.equal(out0["pred"], out1["pred"]) and torch.equal(out0["emb"], out1["emb"]))
    del out0, out1
    for _ in range(a.reps):
        plain.append(timed(lambda: eng.run(slab)["pred"])[0])
        maps.append(timed(lambda: eng.run(slab, cre_attention=True)["pred"])[0])
    p_ms, m_ms = float(np.median(plain)), float(np.median(maps))

    # ---- the kernel alone on the slab's registry rows ----
    gq, gk, off, total = cre_attention_layout(slab["T"], slab["C"], L, H)
    dev = torch.device("cuda")
    g = torch.Generator(device=dev).manual_seed(1)
    q = torch.randn(slab["Mg"], 3 * D, device=dev, generator=g).to(torch.bfloat16)
    kv = torch.randn(int(slab["C"].sum()), 2 * D, device=dev, generator=g).to(torch.bfloat16)
    out = torch.empty(total, dtype=torch.float32, device=dev)
    tabs = [torch.from_numpy(x).to(dev) for x in (gq, gk, off)]

    def kernel_pass():
        for layer in range(L):
            ops.cross_attention_probs(q[:, :D], kv[:, :D], slab["reg_idx"], tabs[0], tabs[1], H, hd, out, tabs[2], layer)
    kernel_pass()
    torch.cuda.synchronize()
    k_ms = [timed(kernel_pass)[0] for _ in range(a.reps)]
    k_med = float(np.median(k_ms))
    n_reg = int(np.sum(slab["T"]))
    res = {
        "workload": {"genes": a.genes, "cres": a.cres, "chunks": a.chunks, "tissues": a.tissues, "n_layers": L,
                     "heads": H, "head_dim": hd, "predictions": n_reg, "map_bytes": 4 * total,
                     "model": "full-size random init"},
        "forward_ms": {"without_maps": p_ms, "with_maps": m_ms,
                       "without_maps_min_max": [float(min(plain)), float(max(plain))],
                       "with_maps_min_max": [float(min(maps)), float(max(maps))]},
        "overhead_pct": 100.0 * (m_ms - p_ms) / p_ms,
        "kernel_ms_per_forward": k_med, "kernel_ms_per_layer": k_med / L,
        "kernel_write_GBps": 4 * total / (k_med * 1e-3) / 1e9,
        # q.k of every (prediction, head, CRE) in both passes
        "kernel_score_TFLOPs": 4.0 * float((slab["C"] * slab["T"]).sum()) * H * hd * L / (k_med * 1e-3) / 1e12,
        "pred_emb_bit_identical": identical,
        "reps": a.reps,
        "card": card(),
    }
    line = json.dumps(res)
    print(line)
    if a.out:
        os.makedirs(os.path.dirname(os.path.abspath(a.out)), exist_ok=True)
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
