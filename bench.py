"""bench.py — gene x tissue predictions/s of the VariantFormer batched-inference hot path on B200.

    python bench.py --gpus N --steps K --warmup W            (N>1: launched by torchrun, one rank per GPU)
    python bench.py --impl reference --gpus N --steps K --warmup W   (CPU arm: the oracle port on the host cores)
    python bench.py --config {1,2,3,4,5} ...                  (3 = default = the driver's line; see CONFIGS below)
    python bench.py ... --dump-outputs DIR                   (+ what the last timed step returned, as DIR/<name>.npy)

One step = one pass of the FULL hot path over one slab of synthetic input per GPU:
  stage 1  genotype application + reverse complement + BPE-500 for B x C CRE windows and B gene windows
           (genome + the sample's variants resident in HBM),
  stage 2  seq2reg encoders over every window (valid tokens only),
  stage 3  seq2gene CombinedModulator, 24 CRE + 25 gene layers, T tissues stacked per gene,
  stage 4  expression head,
at the configuration BASELINE.json's metric is quoted on (config 3: full hierarchical model, C=1024 CRE windows,
G=200 gene chunks, T=63 tissues per gene; B genes per slab).  Weak scaling: every rank owns its own slab; the
only collective is the final gather of expression + embeddings (inside the timed region).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "gene_x_tissue_predictions_per_s"

# The contract is ONE JSON line on stdout.  Libraries write there too (NCCL prints its version banner on the first
# communicator), so file descriptor 1 is pointed at stderr for the whole run and the line goes to the saved descriptor.
_RESULT_OUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)


def emit(obj):
    _RESULT_OUT.write(json.dumps(obj) + "\n")
    _RESULT_OUT.flush()


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir, arrays):
    """Write what the timed path handed its caller in its last step as out_dir/<name>.npy, so that two builds run with
    the same arguments (hence the same seeded inputs) can be compared output for output.  float64 stays float64, every
    other dtype is written as float32.  Above DUMP_LIMIT_BYTES in all, every array keeps the same share of its rows,
    drawn with a fixed seed from its row count alone: arrays with as many rows (pred and emb) keep the same rows."""
    import torch
    host = {}
    for name, a in arrays.items():
        if torch.is_tensor(a):
            a = a.detach().cpu()
            a = a.numpy() if a.dtype == torch.float64 else a.float().numpy()
        a = np.asarray(a)
        host[name] = a.astype(np.float64 if a.dtype == np.float64 else np.float32, copy=False)
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_LIMIT_BYTES:
        share = DUMP_LIMIT_BYTES / total
        for name, a in host.items():
            if a.ndim and a.shape[0] > 1:
                rows = np.random.default_rng(0).choice(a.shape[0], max(1, int(a.shape[0] * share)), replace=False)
                host[name] = a[np.sort(rows)]
    os.makedirs(out_dir, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def load_peaks():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            p = json.load(f)
        return dict(p, source="measured")
    except Exception:
        return {"hbm_gbs": 6650.0, "bf16_tflops": 1590.0, "bf16_tflops_sustained": 1400.0, "source": "fallback"}


# ----------------------------------------------------------------------------------------------------------------
# synthetic workload (SURVEY §8d): seeded genome, one sample's variants, genes with C CREs and a 301 kb window
# ----------------------------------------------------------------------------------------------------------------
def make_workload(seed, n_sets, B, C, T, chrom_len=24_000_000):
    from variantformer_b200.pipeline import GeneSpec
    from variantformer_b200.utils import synth
    rng = np.random.default_rng(seed)
    chrom = synth.make_chromosome(rng, chrom_len)
    var = synth.make_variants(rng, chrom)
    sets = []
    for _ in range(n_sets):
        genes = []
        for _ in range(B):
            lay = synth.make_gene_layout(rng, chrom_len, C, body_len=int(rng.integers(320_000, 900_000)))
            genes.append(GeneSpec("chr1", lay["start"], lay["end"], lay["strand"], lay["cre_start"], lay["cre_end"],
                                  lay["labels"], list(range(T))))
        sets.append(genes)
    return {"chr1": chrom}, {"chr1": var}, sets


class ClockSampler:
    QUERY = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.lines, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits",
                                          "-lms", "100", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=lambda: [self.lines.append(l) for l in self.proc.stdout], daemon=True).start()
        except Exception:
            self.proc = None

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for l in self.lines:
            f = [x.strip() for x in l.split(",")]
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except Exception:
                continue
            for n, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------------------------
# CPU arm: the oracle port (oracle/ is test infrastructure; this is one of the two places allowed to execute it)
# ----------------------------------------------------------------------------------------------------------------
def cpu_sample(sd_cpu, cfg, hp, chroms, var, gene, C, n_tissues, tissues=None):
    """Stage 1 (C oracle) + stages 2-4 (fp32 torch oracle, REFERENCE schedule) for ONE gene x n_tissues on the host
    (tissue ids: the first n_tissues of `tissues`, default 0..n-1).
    -> dict(t_stage1, t_model, pred [T], emb [T, D], cre_tokens [C, 200], gene_tokens [G, 200])."""
    import torch
    from oracle import model_fp32, stage1 as O
    from variantformer_b200.stage1 import cre_window, gene_window
    t0 = time.perf_counter()
    bpe = O.OracleBPE()
    chrom = chroms[gene.chrom]; v = var[gene.chrom]
    lens = np.array([len(a) for a in v["alt"]], np.int32); pool = np.frombuffer(b"".join(v["alt"]), np.uint8)
    aoff = np.cumsum(lens) - lens
    minus = gene.strand == "-"

    def window(a0, a1):
        lo, hi = np.searchsorted(v["pos"], a0), np.searchsorted(v["pos"], a1)
        s = O.apply_variants(chrom, a0, a1, v["pos"][lo:hi], v["ref_len"][lo:hi], aoff[lo:hi], lens[lo:hi],
                             v["gt"][lo:hi], pool)
        return O.reverse_complement(s) if minus else s
    order = np.argsort(gene.cre_start, kind="stable")
    order = order[::-1] if minus else order
    toks, masks = [], []
    for i in order:
        a0, a1 = cre_window(gene.cre_start[i], gene.cre_end[i], 50)
        o, m = O.adjust_length(bpe.encode(window(a0, a1)), 200)
        toks.append(o); masks.append(m)
    a0, a1 = gene_window(gene.start, gene.end, gene.strand, 1000, 300000)
    gt, gm = O.chunkify(bpe.encode(window(a0, a1)), 200, 200)
    t_stage1 = time.perf_counter() - t0
    batch = {"cre_sequences": [torch.from_numpy(np.stack(toks)).long().unsqueeze(1)],
             "cre_attention_masks": [torch.from_numpy(np.stack(masks)).unsqueeze(1)],
             "gene_embeddings": [torch.from_numpy(gt).long().unsqueeze(1)],
             "gene_attention_masks": [torch.from_numpy(gm).unsqueeze(1)],
             "tissue_context": [torch.arange(n_tissues) if tissues is None else
                                torch.as_tensor(list(tissues)[:n_tissues], dtype=torch.long)],
             "ref_cre_labels": [torch.from_numpy(np.asarray(gene.cre_labels)[order].copy())]}
    t0 = time.perf_counter()
    out = model_fp32.predict_step(sd_cpu, cfg, hp, batch, schedule="reference")
    return {"T": n_tissues, "t_stage1": t_stage1, "t_model": time.perf_counter() - t0,
            "pred": np.asarray(out["pred_gene_exp"][0]).ravel(), "emb": np.asarray(out["embeddings"][0]),
            "cre_tokens": np.stack(toks), "gene_tokens": np.asarray(gt)}


CPU_SAMPLE_TISSUES = (1, 2, 4)


def fit_rate(points, stage1_s, T):
    """points: [(n_tissues, seconds)].  The reference schedule repeats the CRE and gene streams once per tissue
    (model_combined_modulator.py:622-649), so cost(T) = base + T * marginal exactly; least squares over the samples
    (three or more tissue counts: a two-point difference was noise-dominated, +-40 % in round 1).
    -> (predictions/s at T tissues, base seconds incl. stage 1, marginal seconds per tissue)."""
    x = np.asarray([p[0] for p in points], np.float64); y = np.asarray([p[1] for p in points], np.float64)
    if len(set(x.tolist())) >= 2:
        marginal, base = np.polyfit(x, y, 1)
    else:
        marginal, base = y.mean() / x.mean(), 0.0
    marginal = max(float(marginal), 1e-9); base = max(float(base), 0.0) + stage1_s
    return T / (base + T * marginal), base, marginal


def cpu_baseline(sd_cpu, cfg, hp, chroms, var, gene, C, T, tissue_counts=CPU_SAMPLE_TISSUES, tissues=None):
    """Bounded sample (~35 s): one gene timed at 1, 2 and 4 tissues; the T-tissue rate of the configured workload is
    T / (base + T * marginal) from a least-squares line.  Also returns the largest sample's outputs (bench parity)."""
    import torch
    torch.set_num_threads(os.cpu_count())
    torch.set_float32_matmul_precision("highest")
    samples = [cpu_sample(sd_cpu, cfg, hp, chroms, var, gene, C, n, tissues) for n in tissue_counts]
    s1 = float(np.mean([x["t_stage1"] for x in samples]))
    value, base, marginal = fit_rate([(x["T"], x["t_model"]) for x in samples], s1, T)
    desc = ", ".join(f"T={x['T']}: {x['t_model']:.1f}s" for x in samples)
    return {"value": value, "unit": "predictions/s", "cores": os.cpu_count(), "kind": "port",
            "sample": (f"oracle port (C stage 1 + torch fp32 reference schedule), 1 gene C={C} G=200 timed at {desc}, "
                       f"stage1 {s1:.2f}s; least-squares line: value = {T}/(base+{T}*marginal), base={base:.1f}s "
                       f"marginal={marginal:.2f}s; bcftools/samtools subprocess cost not timeable (absent)"),
            "samples_s": {str(x["T"]): x["t_model"] for x in samples}, "t_stage1_s": s1}, samples[-1]


def run_reference(args):
    """CPU arm: W warm-up + K timed steps; a step = ONE bounded sample (one gene of the configured workload through
    the oracle port, reference schedule) at 1, 2 or 4 tissues in rotation; the line's value is the least-squares rate at
    the configured tissue count over all timed steps."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch
    from variantformer_b200.utils import random_init
    torch.set_num_threads(os.cpu_count())
    torch.set_float32_matmul_precision("highest")
    cfg, hp = dict(random_init.V4_PCG_MODEL), dict(random_init.SEQ2REG_HP)
    sd = random_init.make_state_dict(cfg, hp, seed=0)
    chroms, var, sets = make_workload(1234, 1, 1, args.cre, args.tissues, chrom_len=8_000_000)
    gene = sets[0][0]
    t_all = time.perf_counter()
    warm = []                                                # warm-up samples at T = 2: a second tissue count for the line
    for _ in range(args.warmup):                             # below when the timed steps cover only one (K = 1)
        r = cpu_sample(sd, cfg, hp, chroms, var, gene, args.cre, 2)
        warm.append((r["T"], r["t_model"]))
    pts, s1, t_timed = [], [], time.perf_counter()
    for i in range(args.steps):
        r = cpu_sample(sd, cfg, hp, chroms, var, gene, args.cre, CPU_SAMPLE_TISSUES[i % len(CPU_SAMPLE_TISSUES)])
        pts.append((r["T"], r["t_model"])); s1.append(r["t_stage1"])
    t_timed = time.perf_counter() - t_timed
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"pred": r["pred"], "emb": r["emb"]})
    fit_pts = list(pts)
    if len({p[0] for p in fit_pts}) < 2:                     # one tissue count cannot separate base from marginal cost
        fit_pts += warm[-1:] if warm else [(lambda r: (r["T"], r["t_model"]))(
            cpu_sample(sd, cfg, hp, chroms, var, gene, args.cre, 2))]
    v, base, marginal = fit_rate(fit_pts, float(np.mean(s1)), args.tissues)
    cb = {"value": v, "unit": "predictions/s", "cores": os.cpu_count(), "kind": "port",
          "sample": (f"oracle port (C stage 1 + torch fp32 reference schedule): {args.steps} samples of 1 gene C={args.cre} "
                     f"G=200 at T in {CPU_SAMPLE_TISSUES} in rotation; least-squares line base={base:.1f}s "
                     f"marginal={marginal:.2f}s/tissue -> {args.tissues}/(base+{args.tissues}*marginal); "
                     "bcftools/samtools subprocess cost not timeable (absent)")}
    emit(({
        "impl": "reference", "metric": METRIC, "value": v, "unit": "predictions/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t_timed / max(args.steps, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": bench_config(args, 1), "cpu_baseline": cb,
        "e2e": {"value": v, "unit": "predictions/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "note": "CPU arm: rank 0 only, host cores", "wall_s": time.perf_counter() - t_all}))


CONFIGS = {
    1: "config1-latency: vcf2exp single sample x 1 gene x 1 tissue (C CRE windows, G=200 gene chunks), full model, one "
       "HotPath.predict call per step",
    2: "config2-seq2reg: CRE window encoder alone, {n} windows of one genome per step (BPE-500 tokens, 6L x 512d x 8h)",
    3: "config3-slab: full hierarchical seq2reg(6L,512d)+seq2gene(25L,1536d,32h) + stage-1 tokenisation, "
       "{B} genes/GPU/step x C={C} CRE windows x G=200 gene chunks x T={T} tissues",
    4: "config4-vep: variant scoring, {P} (variant, gene) pairs per step x 3 zygosities (ref/het/hom) x T={T} tissues, "
       "C={C} CRE windows, token-position gathers on, each triplet one batched pass",
    5: "config5-cohort: {S} synthetic diploid genomes x {Gn} genes (C lognormal 32-3000, T mixed), (sample, gene) items "
       "LPT-sharded over the ranks, padded gather + scatter to query order; fixed sub-grid (strong scaling)",
}
METRICS = {1: (METRIC, "predictions/s"), 2: ("cre_windows_per_s", "windows/s"), 3: (METRIC, "predictions/s"),
           4: ("variant_gene_pairs_per_s", "pairs/s"), 5: (METRIC, "predictions/s")}


def workload_name(args):
    return CONFIGS[args.config].format(n=args.windows, B=args.genes_per_step, C=args.cre, T=args.tissues, P=args.pairs,
                                       S=args.cohort_samples, Gn=args.cohort_genes)


def bench_config(args, world):
    """`config` of the JSON line: identical for the b200 arm and the reference arm of one configuration."""
    return {"workload": workload_name(args), "config_id": args.config,
            "weights": "random-init vf_model.yaml v4_pcg (seed 0)",
            "l2": "per-step working set (>10 GB of activations) far exceeds the 126 MB L2; 3 input sets rotate",
            "parallelism": f"dp{world} (gene x sample sharding, final all_gather only)"}


# tolerance of the parity block (definition and its deviation from SURVEY 8(d): tests/common.py)
REL_ERR_MAX, PEARSON_MIN, REL_ERR_RMS_MAX = 1e-2, 0.9999, 5e-2


def parity_report(got, want):
    got = np.asarray(got, np.float64); want = np.asarray(want, np.float64)
    d = np.abs(got - want).max()
    r = {"rel_err_max_norm": float(d / max(np.abs(want).max(), 1e-30)),
         "rel_err_rms_norm": float(d / max(np.sqrt(np.mean(want * want)), 1e-30)),
         "pearson": float(np.corrcoef(got.ravel(), want.ravel())[0, 1]) if got.size > 1 and want.std() > 0 else 1.0}
    r["ok"] = bool(r["rel_err_max_norm"] <= REL_ERR_MAX and r["pearson"] >= PEARSON_MIN and
                   r["rel_err_rms_norm"] <= REL_ERR_RMS_MAX)
    return r


class Bench:
    """Shared set-up of the b200 arm: process group, full-size random-init model, engine, timing helpers."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        from variantformer_b200 import ops, parallel
        from variantformer_b200.engine import Engine
        from variantformer_b200.utils import random_init
        self.args, self.torch, self.dist, self.ops, self.parallel = args, torch, dist, ops, parallel
        self.rank, self.world, self.local = parallel.init_from_env()
        assert self.world == args.gpus or self.world == 1, f"--gpus {args.gpus} but WORLD_SIZE={self.world}"
        torch.cuda.set_device(self.local)
        self.dev = torch.device("cuda", self.local)
        self.cfg = dict(random_init.V4_PCG_MODEL, num_layers=args.layers); self.hp = dict(random_init.SEQ2REG_HP)
        self.sd = random_init.make_state_dict(self.cfg, self.hp, seed=0, device=self.dev)
        self.engine = Engine(self.sd, self.cfg, self.hp, device=self.dev)
        self.peaks = load_peaks()
        self.last_clocks = None

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        t = self.torch.tensor([x], device=self.dev, dtype=self.torch.float64)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def time_device(self, fn):
        """barrier + synchronize, CUDA events around fn() on the current stream, synchronize + barrier; max over ranks
        -> (milliseconds, fn's result, kernel launches, clocks sampled under load)."""
        torch = self.torch
        sampler = ClockSampler(self.local); sampler.start()
        try:                                              # a failing step must not leave nvidia-smi running
            n0 = self.ops.launch_count()                  # counted inside libvf_b200.so (vf_launch_count)
            self.barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            res = fn()
            e1.record()
            self.barrier()
            ms = self.max_over_ranks(e0.elapsed_time(e1))
        finally:
            self.last_clocks = sampler.stop()
        return ms, res, self.ops.launch_count() - n0, self.last_clocks

    def time_wall(self, fn):
        self.barrier()
        t0 = time.perf_counter()
        res = fn()
        self.torch.cuda.synchronize()
        return self.max_over_ranks(time.perf_counter() - t0), res

    def instrumented(self, fn, steps, timed_ms):
        """The same steps once more with a CUDA-event pair around every launch, on ONE stream (the CRE stack otherwise
        overlaps the gene stack on a second stream and a kernel's event-to-event time would include its neighbour):
        numerator / denominator of the rooflines and the kernel breakdown."""
        from variantformer_b200 import engine as engine_mod
        torch, ops = self.torch, self.ops
        prof = ops.EventProfiler(); ops.PROFILER = prof
        two = engine_mod.CRE_STREAM
        engine_mod.CRE_STREAM = False
        torch.cuda.synchronize()
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record(); fn(); p1.record()
        torch.cuda.synchronize()
        prof_ms = p0.elapsed_time(p1)
        engine_mod.CRE_STREAM = two
        ops.PROFILER = None
        summ = prof.summarize()
        pk = self.peaks
        out = {}

        def tensor_roofline(kind, kernel):
            g = summ.get(kind, {"ms": 0.0, "flops": 0.0, "bytes": 0.0, "n": 0})
            ach = g["flops"] / (g["ms"] / 1e3) / 1e12 if g["ms"] > 0 else 0.0
            peak = pk["bf16_tflops_sustained"]
            return {"bound": "tensor", "kernel": kernel, "achieved": ach, "peak": peak, "unit": "TFLOP/s",
                    "frac": ach / peak, "traffic": None,
                    "algorithmic_bytes_per_launch": g["bytes"] / g["n"] if g["n"] else None,
                    "avg_launch_ms": g["ms"] / g["n"] if g["n"] else None,
                    "peak_source": f"{pk['source']} bf16_tflops_sustained (kernel timed inside a long step)",
                    "launches": g["n"], "share_of_step": g["ms"] / prof_ms if prof_ms else None,
                    "measured_in": "single-stream instrumented pass after the timed region "
                                   f"({prof_ms / steps:.1f} ms/step vs {timed_ms / steps:.1f} timed)"}
        out["roofline"] = tensor_roofline("gemm", "gemm_tcgen05_kernel (all epilogues, 1-CTA and CTA-pair)")
        tr = load_traffic()
        if tr is not None and args_config_matches(tr, self.args):
            out["roofline"]["traffic"] = tr["gemm_dram_bytes_per_launch"]
            out["roofline"]["traffic_source"] = tr["source"]
            out["roofline"]["traffic_over_algorithmic"] = tr["gemm_dram_bytes_per_launch"] / max(
                out["roofline"]["algorithmic_bytes_per_launch"] or 1.0, 1.0)
        others = []
        if "attention" in summ:
            att = tensor_roofline("attention", "attention_mc_kernel (every attention of the path)")
            # second bound of a softmax kernel: one ex2 per score on the MUFU pipe (16 results / clk / SM, measured:
            # tools/ubench/ex2_rate.cu); a score costs 4 * head_dim tensor FLOPs, so at head dim 48 the MUFU ceiling is
            # about half of the tensor peak.  Stated at the SM clock sampled during the timed region.
            import re
            exps = 0.0
            for k, v in prof.summarize_detail().items():
                m = re.search(r"attention .*hd=(\d+)", k)
                if m:
                    exps += v["flops"] / (4.0 * int(m.group(1)))
            mhz = (self.last_clocks or {}).get("sm_mhz") or 0.0
            if exps > 0 and mhz > 0 and summ["attention"]["ms"] > 0:
                sms = torch.cuda.get_device_properties(self.local).multi_processor_count
                t_min_ms = exps / (16.0 * sms * mhz * 1e6) * 1e3
                ceil_tf = summ["attention"]["flops"] / (t_min_ms / 1e3) / 1e12
                att["mufu_ceiling"] = {"tflops": ceil_tf, "frac_of_ceiling": att["achieved"] / ceil_tf, "sm_mhz": mhz,
                                       "note": "one ex2 per score at 16/clk/SM; FLOPs per score = 4 x head_dim"}
            others.append(att)
        s1 = [k for k in ("stage1_encode", "stage1_bpe", "stage1_bpe_cluster") if k in summ]
        if s1:
            ms = sum(summ[k]["ms"] for k in s1); by = sum(summ[k]["bytes"] for k in s1); n = sum(summ[k]["n"] for k in s1)
            ach = by / (ms / 1e3) / 1e9 if ms > 0 else 0.0
            others.append({"bound": "hbm", "kernel": "stage 1: encode_windows_kernel + bpe_tokenize(_cluster)_kernel",
                           "achieved": ach, "peak": pk["hbm_gbs"], "unit": "GB/s", "frac": ach / pk["hbm_gbs"],
                           "traffic": None, "launches": n, "ms_per_step": ms / steps,
                           "note": "latency-bound integer work (rank sweeps with a barrier per applied merge rank): "
                                   "bytes are the window bytes in + int32 token rows out"})
        out["roofline_other"] = others
        out["kernel_breakdown_ms_per_step"] = {k: v["ms"] / steps for k, v in summ.items()}
        det = prof.summarize_detail()
        out["kernel_detail"] = {k: {"ms_per_step": round(v["ms"] / steps, 3), "launches_per_step": v["n"] / steps,
                                    "tflops": round(v["flops"] / (v["ms"] / 1e3) / 1e12, 1) if v["ms"] > 0 else 0.0,
                                    "algorithmic_GBps": round(v["bytes"] / (v["ms"] / 1e3) / 1e9, 1) if v["ms"] > 0 else 0.0}
                                for k, v in sorted(det.items(), key=lambda kv: -kv[1]["ms"])[:24]}
        total_flops = sum(v["flops"] for v in summ.values())
        out["algorithmic_tflop_per_step"] = total_flops / steps / 1e12
        out["achieved_tflops_all_kernels"] = total_flops / (timed_ms / 1e3) / 1e12
        return out

    def line(self, value, ms_per_step, e2e_value, h2d, d2h, launches, clocks, scaling="weak"):
        a = self.args
        metric, unit = METRICS[a.config]
        return {"metric": metric, "value": value, "unit": unit, "n_gpus": self.world, "steps": a.steps,
                "warmup": a.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": scaling,
                "vs_baseline": None, "dtype": "bf16", "data": "synthetic", "config": bench_config(a, self.world),
                "clocks": clocks, "gpu_launches": launches,
                "e2e": {"value": e2e_value, "unit": unit, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h)}}

    def finish(self, out):
        if self.rank == 0:
            emit(out)
        if self.world > 1:
            self.dist.barrier()
            self.dist.destroy_process_group()


def load_traffic():
    """DRAM bytes per GEMM launch from the committed ncu pass over this same command (profiles/r02_gemm_traffic.json,
    written by tools/ncu_traffic.py); None when the file is absent."""
    try:
        with open(os.path.join(ROOT, "profiles", "r02_gemm_traffic.json")) as f:
            return json.load(f)
    except Exception:
        return None


def args_config_matches(tr, args):
    return tr.get("config_id") == args.config and tr.get("genes_per_step") == args.genes_per_step and \
        tr.get("cre") == args.cre and tr.get("tissues") == args.tissues


# ----------------------------------------------------------------------------------------------------------------
# config 3 (default, the driver's line) and config 1 (single gene x 1 tissue latency)
# ----------------------------------------------------------------------------------------------------------------
def run_config3(args):
    import copy
    from variantformer_b200.pipeline import HotPath
    from variantformer_b200.stage1 import Genome, SampleVariants
    b = Bench(args)
    torch, ops, parallel = b.torch, b.ops, b.parallel
    single = args.config == 1
    B, C, T = (1, args.cre, 1) if single else (args.genes_per_step, args.cre, args.tissues)
    n_sets = 3
    chroms, var, sets = make_workload(1234 + b.rank, n_sets, B, C, T)
    if single:
        for genes in sets:
            genes[0].tissues = [62]                         # whole blood (SURVEY 8d config 1)
    hot = HotPath(b.engine, Genome.from_arrays(chroms, b.dev))
    variants = SampleVariants(var, b.dev)
    preds_per_step = B * T
    counts = [preds_per_step] * b.world

    def run_steps(n, to_host, gather=True):
        """n consecutive steps through the pipelined public API (stage 1 of slab i+1 overlaps the model of slab i)."""
        last = None
        for last in hot.predict_pipelined((sets[i % n_sets] for i in range(n)), variants, to_host=to_host):
            if b.world > 1 and not to_host and gather:  # the one collective: final gather of expression + embeddings
                parallel.gather_rows(last[0], counts, b.world, b.rank); parallel.gather_rows(last[1], counts, b.world, b.rank)
        return last

    run_steps(args.warmup, False)
    torch.cuda.synchronize()
    # ---- timed region: device-resident leg (`value`) ----
    elapsed_ms, (pred, emb, err), launches, clocks = b.time_device(lambda: run_steps(args.steps, False))
    assert int(err.item()) == 0, "stage-1 kernel flagged an error"
    assert bool(torch.isfinite(pred).all()) and bool(torch.isfinite(emb).all()), "non-finite outputs"
    if args.dump_outputs and b.rank == 0:
        dump_outputs(args.dump_outputs, {"pred": pred, "emb": emb})
    value = b.world * preds_per_step * args.steps / (elapsed_ms / 1e3)
    # ---- end-to-end leg: host window tables in, numpy results out, every step ----
    e2e_s, (p_np, e_np) = b.time_wall(lambda: run_steps(args.steps, True))
    e2e_value = b.world * preds_per_step * args.steps / e2e_s
    h2d = B * C * (8 + 8 + 4 + 4 + 4 + 1 + 8) + B * 40 + B * T * 8           # window tables, labels, tissue ids
    d2h = p_np.nbytes + e_np.nbytes + 4 * (B * C + B)                        # results + token counts
    out = b.line(value, elapsed_ms / args.steps, e2e_value, h2d, d2h, launches, clocks)
    out["config"]["pipelining"] = ("stage 1 + host bookkeeping of slab i+1 on a side stream while slab i's model runs; "
                                   "CRE stack on its own stream next to the gene stack")
    if single:
        out["latency_ms"] = {"device_resident": elapsed_ms / args.steps, "end_to_end": 1e3 * e2e_s / args.steps}
    if b.rank == 0:
        out.update(b.instrumented(lambda: run_steps(args.steps, False, gather=False), args.steps, elapsed_ms))
        out["config"]["algorithmic_tflop_per_step"] = out.pop("algorithmic_tflop_per_step")
        if b.world == 1 and not args.no_cpu_baseline:
            # ---- CPU leg (bounded sample) + parity of the GPU path against it at the benchmark's own configuration:
            #      gene 0 of input set 0, full depth, the first tissues of its tissue list ----
            sd_cpu = {k: v.float().cpu() for k, v in b.sd.items()}
            gene0 = copy.copy(sets[0][0])
            tis = [1] if single else list(CPU_SAMPLE_TISSUES)
            cb, sample = cpu_baseline(sd_cpu, b.cfg, b.hp, chroms, var, gene0, C, T, tissue_counts=tis,
                                      tissues=gene0.tissues)
            out["cpu_baseline"] = cb
            gene0.tissues = list(gene0.tissues[: sample["T"]])
            tk = hot.tokenize([gene0], variants)
            tok_equal = bool((tk["cre_tok"][0].cpu().numpy() == sample["cre_tokens"]).all() and
                             (tk["gene_tok"][0].cpu().numpy() == sample["gene_tokens"]).all())
            g_pred, g_emb = hot.predict([gene0], variants)
            par = parity_report(g_emb, sample["emb"])
            par["pred_rel_err_max_norm"] = parity_report(g_pred, sample["pred"])["rel_err_max_norm"]
            par["tokens_equal"] = tok_equal
            par["what"] = (f"GPU path vs the fp32 oracle (reference schedule) on gene 0 of the timed input set, full depth "
                           f"({b.cfg['num_layers']} gene layers), C={C}, G=200, {sample['T']} tissues; embeddings "
                           f"[{sample['T']}, {b.cfg['emb_dim']}]; bounds {REL_ERR_MAX} / {REL_ERR_RMS_MAX} / {PEARSON_MIN}")
            par["ok"] = bool(par["ok"] and tok_equal and par["pred_rel_err_max_norm"] <= REL_ERR_MAX)
            out["parity"] = par
            if not par["ok"]:
                sys.stderr.write(f"PARITY FAILURE: {json.dumps(par)}\n")
                raise SystemExit(3)                          # a fast result that differs from the reference is not a result
    b.finish(out)


# ----------------------------------------------------------------------------------------------------------------
# config 2: the seq2reg window encoder alone
# ----------------------------------------------------------------------------------------------------------------
def run_config2(args):
    from variantformer_b200.engine import AttnPlan
    from variantformer_b200.stage1 import Genome, SampleVariants, WindowTokenizer
    from variantformer_b200.utils import synth
    b = Bench(args)
    torch, ops = b.torch, b.ops
    rng = np.random.default_rng(4321 + b.rank)
    chrom_len = 24_000_000
    chrom = synth.make_chromosome(rng, chrom_len)
    var = synth.make_variants(rng, chrom)
    genome = Genome.from_arrays({"chr1": chrom}, b.dev); variants = SampleVariants({"chr1": var}, b.dev)
    tok = WindowTokenizer(b.dev)
    n = args.windows
    sets = []
    for _ in range(3):                                     # cCRE-like windows: 150-350 bp + 2 x 50 bp flank
        s0 = np.sort(rng.integers(1000, chrom_len - 1000, n)); ln = rng.integers(150, 351, n)
        sets.append((np.maximum(0, s0 - 50), s0 + ln + 50))
    W = b.engine.cre_tok

    def tokens_of(i):
        w0, w1 = sets[i % 3]
        seq, lens, err = tok.sequences(genome, ["chr1"] * n, w0, w1, [0] * n, variants)
        t, m, cnt = tok.tokenize_fixed(seq, lens, seq.shape[1], typical_len=tok.last_max_window)
        return t, m.to(torch.uint8), np.minimum(cnt.cpu().numpy(), 200).astype(np.int64), err

    def encode(t, m, lens):
        return b.engine.seq2reg(W, t, m, lens, ops.cu_seqlens(lens, b.dev), AttnPlan(lens, b.dev, W.hd))

    resident = [tokens_of(i) for i in range(3)]
    n_tok = int(np.mean([r[2].sum() for r in resident]))

    def steps_resident(k):
        out = None
        for i in range(k):
            t, m, lens, _ = resident[i % 3]
            out = encode(t, m, lens)
        return out

    def steps_e2e(k):
        out = None
        for i in range(k):
            t, m, lens, err = tokens_of(i)
            out = encode(t, m, lens).cpu()
            assert int(err.item()) == 0
        return out
    steps_resident(args.warmup)
    ms, pooled, launches, clocks = b.time_device(lambda: steps_resident(args.steps))
    assert bool(torch.isfinite(pooled.float()).all())
    if args.dump_outputs and b.rank == 0:
        dump_outputs(args.dump_outputs, {"pooled": pooled})
    value = b.world * n * args.steps / (ms / 1e3)
    e2e_s, pooled_h = b.time_wall(lambda: steps_e2e(args.steps))
    out = b.line(value, ms / args.steps, b.world * n * args.steps / e2e_s, n * 16 + n * 9, pooled_h.numel() * 2 + 4 * n,
                 launches, clocks)
    out["tokens_per_s"] = b.world * n_tok * args.steps / (ms / 1e3)
    out["config"]["tokens_per_step"] = n_tok
    out["config"]["note"] = ("value: tokens resident in HBM; e2e: host window tables -> genotype encoding + BPE on the device "
                             "-> encoder -> pooled embeddings back on the host")
    if b.rank == 0:
        out.update(b.instrumented(lambda: steps_resident(args.steps), args.steps, ms))
        out["config"]["algorithmic_tflop_per_step"] = out.pop("algorithmic_tflop_per_step")
        if b.world == 1 and not args.no_cpu_baseline:
            out["cpu_baseline"] = cpu_seq2reg_sample(b, resident[0])
    b.finish(out)


def cpu_seq2reg_sample(b, resident, n_sample=256):
    """fp32 oracle of the window encoder on the first windows of a resident set: rate + parity of the pooled vectors."""
    import torch
    from oracle import model_fp32
    torch.set_num_threads(os.cpu_count()); torch.set_float32_matmul_precision("highest")
    t, m, lens, _ = resident
    sd_cpu = {k: v.float().cpu() for k, v in b.sd.items() if k.startswith("cre_tokenizer.")}
    tok = t[:n_sample].cpu().long(); msk = m[:n_sample].cpu().bool()
    t0 = time.perf_counter()
    want = model_fp32.seq2reg_embed(sd_cpu, "cre_tokenizer.", b.hp, tok, msk).numpy()
    dt = time.perf_counter() - t0
    from variantformer_b200.engine import AttnPlan
    ln = lens[:n_sample]
    got = b.engine.seq2reg(b.engine.cre_tok, t[:n_sample].contiguous(), m[:n_sample].contiguous(), ln,
                           b.ops.cu_seqlens(ln, b.dev), AttnPlan(ln, b.dev, b.engine.cre_tok.hd)).float().cpu().numpy()
    return {"value": n_sample / dt, "unit": "windows/s", "cores": os.cpu_count(), "kind": "port",
            "sample": f"oracle seq2reg_embed (torch fp32) on {n_sample} windows of the timed set: {dt:.1f}s",
            "parity": parity_report(got, want)}


# ----------------------------------------------------------------------------------------------------------------
# config 4: variant scoring (ref / het / hom triplets)
# ----------------------------------------------------------------------------------------------------------------
def run_config4(args):
    from variantformer_b200.datasets.vepdataset import VEPBatchBuilder, Variant
    from variantformer_b200.seq2gene.model_combined_modulator import Seq2GenePredictorCombinedModulator, attach_trainer
    from variantformer_b200.seq2reg.model import Seq2RegPredictor
    from variantformer_b200.stage1 import Genome
    b = Bench(args)
    torch = b.torch
    P, C, T = args.pairs, args.cre, args.tissues
    chroms, var, sets = make_workload(977 + b.rank, 3, P, C, T)
    genome = Genome.from_arrays(chroms, b.dev)
    builder = VEPBatchBuilder(genome, b.dev)
    model = Seq2GenePredictorCombinedModulator(cre_tokenizer=Seq2RegPredictor(**b.hp), gene_tokenizer=Seq2RegPredictor(**b.hp),
                                               **b.cfg)
    model.load_state_dict(b.sd); model.eval().to(b.dev); model.vep = True; attach_trainer(model)
    model._engine_obj = None
    rng = np.random.default_rng(5 + b.rank)
    chrom = chroms["chr1"]

    def make_pairs(genes):
        """A SNP inside a CRE window of the gene (and, for most genes, inside the gene window as well)."""
        pairs = []
        for g in genes:
            k = int(rng.integers(0, len(g.cre_start)))
            for _ in range(50):
                pos0 = int(rng.integers(g.cre_start[k], g.cre_end[k]))
                ref = chr(chrom[pos0]).upper()
                if ref in "ACGT" and chr(chrom[pos0]) != "N":
                    break
            # SNPs: inside the gene window the reference rejects anything whose het code is not an IUPAC letter
            # (multi-base alleles encode as 'N' -> ValueError in encode_with_position, utils/seq.py:93-97)
            alt = [c for c in "ACGT" if c != ref][int(rng.integers(0, 3))]
            pairs.append((g, Variant("chr1", pos0 + 1, ref, alt, tissue=list(range(T)))))
        return pairs
    pair_sets = [make_pairs(genes) for genes in sets]

    def build(i):
        return [builder.build(g, v) for g, v in pair_sets[i % 3]]

    def score(batches):
        return [model.predict_step(bt, 0) for bt in batches]
    prebuilt = [build(i) for i in range(3)]

    def steps_resident(k):
        out = None
        for i in range(k):
            out = score(prebuilt[i % 3])
        return out

    def steps_e2e(k):
        out = None
        for i in range(k):
            out = score(build(i))
        return out
    steps_resident(min(args.warmup, 3))
    ms, res, launches, clocks = b.time_device(lambda: steps_resident(args.steps))
    assert all(np.isfinite(np.asarray(r["pred_gene_exp"])).all() for r in res)
    if args.dump_outputs and b.rank == 0:                  # per pair: [ref, het, hom] stacked on the first axis
        dump_outputs(args.dump_outputs, {f"pair{i}_{k}": np.stack(r[k]) for i, r in enumerate(res)
                                         for k in ("pred_gene_exp", "embd", "gene_token_embedding", "cre_token_embedding")})
    value = b.world * P * args.steps / (ms / 1e3)
    e2e_s, res = b.time_wall(lambda: steps_e2e(args.steps))
    d2h = sum(np.asarray(r[k]).nbytes for r in res for k in ("pred_gene_exp", "embd", "gene_token_embedding",
                                                               "cre_token_embedding") if k in r)
    out = b.line(value, ms / args.steps, b.world * P * args.steps / e2e_s, P * (C * 24 + 64), d2h, launches, clocks)
    out["predictions_per_s"] = value * 3 * T
    out["config"]["note"] = ("value: triplet batches resident (tokens built), model.predict_step (variant_prediction) only, "
                             "numpy results out; e2e: (gene, variant) in -> VEPBatchBuilder (stage-1 kernels, 3 zygosities) -> "
                             "predict_step -> numpy")
    if b.rank == 0:
        out.update(b.instrumented(lambda: steps_resident(args.steps), args.steps, ms))
        out["config"]["algorithmic_tflop_per_step"] = out.pop("algorithmic_tflop_per_step")
        if b.world == 1 and not args.no_cpu_baseline:
            sd_cpu = {k: v.float().cpu() for k, v in b.sd.items()}
            cb, _ = cpu_baseline(sd_cpu, b.cfg, b.hp, chroms, {"chr1": dict(pos=np.zeros(0, np.int64), ref_len=np.zeros(0, np.int32),
                                                                              alt=[], gt=np.zeros(0, np.uint8))},
                                 pair_sets[0][0][0], C, T, tissue_counts=[1, 2])
            # a pair = 3 forwards (ref, het, hom) of T tissues each in the reference (model_combined_modulator.py:948-968)
            per_pair_s = 3.0 * T / cb["value"]
            cb.update(value=1.0 / per_pair_s, unit="pairs/s",
                      sample=cb["sample"] + f"; a pair = 3 sequential forwards of T={T}: {per_pair_s:.0f}s")
            out["cpu_baseline"] = cb
    b.finish(out)


# ----------------------------------------------------------------------------------------------------------------
# config 5: cohort sub-grid, (sample, gene) items sharded over the ranks — strong scaling with ragged items
# ----------------------------------------------------------------------------------------------------------------
def run_config5(args):
    from variantformer_b200.pipeline import GeneSpec, HotPath
    from variantformer_b200.stage1 import Genome, SampleVariants
    from variantformer_b200.utils import synth
    b = Bench(args)
    torch, parallel = b.torch, b.parallel
    S, Gn = args.cohort_samples, args.cohort_genes
    rng = np.random.default_rng(2330)                      # the SAME grid on every rank
    chrom_len = 24_000_000
    chrom = synth.make_chromosome(rng, chrom_len)
    genes = []
    for _ in range(Gn):
        C = int(np.clip(rng.lognormal(np.log(600), 0.6), 32, 3000))
        lay = synth.make_gene_layout(rng, chrom_len, C, body_len=int(np.clip(rng.lognormal(np.log(25_000), 1.0), 1_000, 900_000)))
        T = 63 if rng.random() < 0.5 else int(rng.integers(1, 63))
        tissues = sorted(rng.choice(63, T, replace=False).tolist())
        genes.append(GeneSpec("chr1", lay["start"], lay["end"], lay["strand"], lay["cre_start"], lay["cre_end"],
                              lay["labels"], tissues))
    sample_vars = [synth.make_variants(np.random.default_rng(9000 + s), chrom) for s in range(S)]
    items = [(s, g) for s in range(S) for g in range(Gn)]
    rows = [len(genes[g].tissues) for _, g in items]
    costs = [parallel.item_cost(97 * len(genes[g].cre_start), 40000, len(genes[g].cre_start), 200, len(genes[g].tissues))
             for _, g in items]
    parts = parallel.shard_items(costs, b.world)
    counts = [sum(rows[i] for i in p) for p in parts]
    hot = HotPath(b.engine, Genome.from_arrays({"chr1": chrom}, b.dev))
    dev_vars = {}

    def variants_of(s):
        if s not in dev_vars:
            dev_vars[s] = SampleVariants({"chr1": sample_vars[s]}, b.dev)
        return dev_vars[s]

    def slabs_of(my_items, cap_rows=8 * 63 * 201, cap_cre=8192):
        """Consecutive items of one sample, bounded by the gene-stream rows and CRE windows a slab may hold."""
        slabs, cur, cur_s, r, c = [], [], None, 0, 0
        for i in my_items:
            s, g = items[i]
            gr, gc = rows[i] * 201, len(genes[g].cre_start)
            if cur and (s != cur_s or r + gr > cap_rows or c + gc > cap_cre):
                slabs.append((cur_s, cur)); cur, r, c = [], 0, 0
            cur.append(i); cur_s = s; r += gr; c += gc
        if cur:
            slabs.append((cur_s, cur))
        return slabs

    def run_items(my_items):
        """-> (pred [rows], emb [rows, D]) of my_items in order (device tensors)."""
        preds, embs = [], []
        for s, idx in slabs_of(my_items):
            p, e, err = hot.predict([genes[items[i][1]] for i in idx], variants_of(s), to_host=False)
            preds.append(p); embs.append(e)
        D = b.cfg["emb_dim"]
        if not preds:
            return torch.zeros(0, device=b.dev), torch.zeros(0, D, device=b.dev)
        return torch.cat(preds), torch.cat(embs)

    def job():
        p, e = run_items(parts[b.rank])
        t_rank = time.perf_counter()
        gp = parallel.scatter_to_query_order(parallel.gather_rows(p, counts, b.world, b.rank), parts, rows)
        ge = parallel.scatter_to_query_order(parallel.gather_rows(e, counts, b.world, b.rank), parts, rows)
        return gp, ge, t_rank
    for _ in range(min(args.warmup, 1)):                   # one warm-up pass over the whole grid (allocations, tables)
        job()
    torch.cuda.synchronize()
    # per-rank busy time (before the gather) for the imbalance figure
    b.barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); run_items(parts[b.rank]); e1.record(); torch.cuda.synchronize()
    mine_ms = e0.elapsed_time(e1)
    t = torch.tensor([mine_ms], device=b.dev, dtype=torch.float64)
    all_ms = [torch.zeros_like(t) for _ in range(b.world)]
    if b.world > 1:
        b.dist.all_gather(all_ms, t)
    else:
        all_ms = [t]
    all_ms = [float(x.item()) for x in all_ms]
    ms, (gp, ge, _), launches, clocks = b.time_device(lambda: [job() for _ in range(args.steps)][-1])
    if args.dump_outputs and b.rank == 0:
        dump_outputs(args.dump_outputs, {"pred": gp, "emb": ge})
    total_preds = sum(rows)
    value = total_preds * args.steps / (ms / 1e3)
    e2e_s, (hp_, he_) = b.time_wall(lambda: [(lambda r: (r[0].cpu().numpy(), r[1].cpu().numpy()))(job())
                                             for _ in range(args.steps)][-1])
    n_win = sum(len(genes[g].cre_start) for _, g in items)
    out = b.line(value, ms / args.steps, total_preds * args.steps / e2e_s, (n_win * 37 + len(items) * 600) / b.world,
                 hp_.nbytes + he_.nbytes, launches, clocks, scaling="strong")
    out["rank_busy_ms"] = {"per_rank": all_ms, "max_over_mean": max(all_ms) / (sum(all_ms) / len(all_ms))}
    out["config"].update(items=len(items), predictions=total_preds,
                         cre_windows_per_item={"min": int(min(len(g.cre_start) for g in genes)),
                                               "max": int(max(len(g.cre_start) for g in genes))},
                         extrapolation=("full cohort = 2,330 genomes x 17,859 genes; at the measured rate and this mix of "
                                        "tissue counts: 2330*17859*mean_T / value seconds"))
    out["full_cohort_hours_at_this_rate"] = 2330 * 17859 * (total_preds / len(items)) / value / 3600.0
    if b.rank == 0 and b.world > 1 and not args.no_gather_check:
        # the N-rank gathered result must equal the 1-rank result bit for bit (every kernel is row / sequence local with
        # a fixed reduction order, so results do not depend on how items are grouped into slabs)
        p1, e1_ = run_items(list(range(len(items))))
        out["gather_check"] = {"ranks": b.world, "bit_identical_to_single_rank": bool(torch.equal(p1, gp) and torch.equal(e1_, ge)),
                               "max_abs_diff_emb": float((e1_ - ge).abs().max())}
        if not out["gather_check"]["bit_identical_to_single_rank"]:
            sys.stderr.write("GATHER CHECK FAILED\n")
    if b.rank == 0:
        out.update(b.instrumented(lambda: run_items(parts[0]), 1, ms / args.steps))
        out["config"]["algorithmic_tflop_per_step"] = out.pop("algorithmic_tflop_per_step")
        out.pop("achieved_tflops_all_kernels", None)          # (rank 0's share only: not a whole-job figure)
    if b.rank == 0 and not args.no_cpu_baseline and b.world == 1:
        sd_cpu = {k: v.float().cpu() for k, v in b.sd.items()}
        g0 = genes[int(np.argmin([abs(len(g.cre_start) - 600) for g in genes]))]
        cb, _ = cpu_baseline(sd_cpu, b.cfg, b.hp, {"chr1": chrom}, {"chr1": sample_vars[0]}, g0, len(g0.cre_start),
                             len(g0.tissues), tissue_counts=[1, 2])
        out["cpu_baseline"] = cb
    b.finish(out)


# ----------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", type=int, default=3, choices=[1, 2, 3, 4, 5],
                    help="BASELINE.json configuration (3 = full hierarchical slab = the driver's line)")
    ap.add_argument("--genes-per-step", type=int, default=8)
    ap.add_argument("--cre", type=int, default=1024)
    ap.add_argument("--tissues", type=int, default=63)
    ap.add_argument("--windows", type=int, default=16384, help="config 2: CRE windows per step")
    ap.add_argument("--pairs", type=int, default=4, help="config 4: (variant, gene) pairs per step")
    ap.add_argument("--cohort-samples", type=int, default=4, help="config 5: genomes of the fixed sub-grid")
    ap.add_argument("--cohort-genes", type=int, default=48, help="config 5: genes of the fixed sub-grid")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-gather-check", action="store_true")
    ap.add_argument("--layers", type=int, default=25, help="debug only: seq2gene depth (25 = the benchmark)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step returned (rank 0) as "
                    "DIR/<name>.npy, float32 / float64, at most 64 MB in all (a fixed, seeded sample of rows beyond)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.impl == "reference":
        return run_reference(args)
    args.warmup = max(args.warmup, 3)
    {1: run_config3, 2: run_config2, 3: run_config3, 4: run_config4, 5: run_config5}[args.config](args)


if __name__ == "__main__":
    main()
