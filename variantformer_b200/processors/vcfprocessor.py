"""VCFProcessor — the vcf2exp API with the reference's method names and return shapes
(processors/vcfprocessor.py:24-61, :217-277), plus a Lightning-free `Trainer` exposing `.predict` / `.precision`."""
import logging
import os

import numpy as np
import pandas as pd
import torch
from torch.utils.data import DataLoader

from ..datasets.vcfdataset import LocalGeneManifest, VCFDataset, collate_fn_batching
from ..utils.config import CONFIG_DIR, PACKAGE_ROOT, VOCAB_DIR, load_yaml
from .model_manager import ModelManager

log = logging.getLogger(__name__)


class Trainer:
    """Stand-in for lightning.pytorch.Trainer(accelerator='gpu', devices=1, precision=...): single process, current
    CUDA stream, `predict(model, dataloader, ckpt_path=None) -> list[dict]`."""

    def __init__(self, accelerator="gpu", devices=1, logger=False, precision="bf16-mixed", enable_checkpointing=False,
                 **_):
        assert devices == 1, "one process drives one GPU; use variantformer_b200.parallel for multi-GPU sharding"
        self.precision = precision

    def predict(self, model, dataloaders, ckpt_path=None):
        if ckpt_path and os.path.exists(ckpt_path):             # Lightning reloads the weights (vcfprocessor.py:262)
            ck = torch.load(ckpt_path, map_location="cpu")
            model.load_state_dict(ck["state_dict"] if "state_dict" in ck else ck)
            model.to("cuda")
        model.trainer = self
        model.eval()
        return [model.predict_step(batch, i) for i, batch in enumerate(dataloaders)]


class VCFProcessor:
    def __init__(self, model_class: str = "v4_pcg", base_dir=None, gene_cre_manifest=None, model_overrides=None):
        """base_dir: where relative artifact paths (`_artifacts/...`) are resolved (reference: the repo root).
        gene_cre_manifest: object with get_file_path(gene_id); default = <base_dir>/_artifacts/gene_cre_manifests/."""
        base_dir = base_dir or PACKAGE_ROOT
        self.config_location = CONFIG_DIR
        self.model_config = load_yaml(os.path.join(CONFIG_DIR, "vf_model.yaml"))[model_class]
        if model_overrides:
            self.model_config.model.update(model_overrides)
        self.tissue_vocab = load_yaml(os.path.join(VOCAB_DIR, "tissue_vocab.yaml"))
        self.vcf_loader_config = load_yaml(os.path.join(CONFIG_DIR, "vcfloader.yaml"))
        self.gene_cre_manifest = gene_cre_manifest or LocalGeneManifest(
            os.path.join(base_dir, "_artifacts", "gene_cre_manifests"))

        def fix(node, key):
            if node.get(key) and not os.path.isabs(node[key]):
                node[key] = os.path.join(base_dir, node[key])
        fix(self.vcf_loader_config, "CRE_BED"); fix(self.vcf_loader_config, "fasta_path")
        fix(self.model_config.dataset, "gencode_v24"); fix(self.model_config.model, "checkpoint_path")
        fix(self.model_config.model.cre_tokenizer, "path"); fix(self.model_config.model.gene_tokenizer, "path")
        assert torch.cuda.is_available(), "GPU is not available"
        self.accelerator = "gpu"

    def get_tissues(self):
        return self.tissue_vocab.keys()

    def get_genes(self):
        return pd.read_csv(self.model_config.dataset.gencode_v24)

    def create_data(self, vcf_path: str, query_df: pd.DataFrame, **kwargs):
        cfg = dict(self.vcf_loader_config.dataloader)
        cfg.update(kwargs)
        # items are produced by CUDA kernels in the main process: no worker processes, no pinning of device tensors
        cfg.update(num_workers=0, pin_memory=False); cfg.pop("prefetch_factor", None)
        ds = self.model_config.dataset
        dataset = VCFDataset(max_length=ds.max_length, max_chunks=ds.max_chunks, cre_neighbour_hood=ds.cre_neighbour_hood,
                             gencode_v24=ds.gencode_v24, gene_cre_manifest=self.gene_cre_manifest,
                             gene_upstream_neighbour_hood=ds.gene_upstream_neighbour_hood,
                             gene_downstream_neighbour_hood=ds.gene_downstream_neighbour_hood, query_df=query_df,
                             fasta_path=self.vcf_loader_config.fasta_path, vcf_path=vcf_path)
        return dataset, DataLoader(dataset, collate_fn=collate_fn_batching, **cfg)

    def load_model(self):
        model, checkpoint_path = ModelManager(self.model_config.model).load_model()
        trainer = Trainer(accelerator=self.accelerator, devices=1, logger=False,
                          precision=self.model_config.model.precision, enable_checkpointing=False)
        return model, checkpoint_path, trainer

    def predict(self, model, checkpoint_path, trainer, dataloader, vcf_dataset):
        predictions = trainer.predict(model, dataloader, ckpt_path=checkpoint_path)
        return self.format_output(vcf_dataset.query_df, predictions)

    def cre_attention(self, vcf_path: str, query_df: pd.DataFrame, **kwargs):
        """Which CREs each prediction reads: the gene -> CRE cross-attention of the registry (tissue) token at every
        gene layer (DESIGN.md section 13), for the query rows of create_data / predict.  Writes no file.
        -> (df, maps): maps[(gene_id, tissue)] = fp32 [num_layers, num_heads, C] in manifest row order; df = one row per
        (gene_id, tissue, layer, CRE) with the CRE's manifest columns, the head-mean `attention` and the prediction's
        `predicted_expression`."""
        dataset, dataloader = self.create_data(vcf_path, query_df, **kwargs)
        model, _, trainer = self.load_model()
        model.trainer = trainer
        frames, maps, i = [], {}, 0
        for batch in dataloader:
            out = model.predict_cre_attention(batch)
            for pred, a in zip(out["pred_gene_exp"], out["cre_attention"]):
                row = dataset.query_df.iloc[i]
                i += 1
                manifest, order = dataset.cre_manifest(row["gene_id"])
                df, m = cre_attention_frame(row["gene_id"], row["tissue_names"], manifest, order, a, pred)
                frames.append(df); maps.update(m)
        return pd.concat(frames, ignore_index=True), maps

    def predict_cohort(self, vcf_path: str, query_df: pd.DataFrame, output_dir=None, samples=None, embeddings=True,
                       genes_per_slab=8, samples_per_slab=256):
        """Every (sample, gene, tissue) of the query for the samples of one multi-sample VCF (samples: names, default
        every sample column), with one region-restricted parse of the VCF and each distinct window encoded once across
        samples (variantformer_b200.cohort, DESIGN.md section 14).  The query is filtered with VCFDataset's rules; each
        prediction equals what create_data + predict give for that sample alone.
        -> output_dir None: a long DataFrame (sample, gene_id, tissue (name), predicted_expression[, embeddings]) in
        (sample, gene, tissue) order.  Else: results go through ResultWriter into output_dir, one Parquet file per slab
        (genes_per_slab query genes x samples_per_slab samples; slab index = gene block x number of sample blocks +
        sample block, a function of the query and the sample list only), slabs already on disk are skipped, and the
        directory is returned.  A sample block whose variant table would pass 2^31 records or ALT bytes is computed in
        sub-blocks (CohortVariants.blocks) and still written as one slab."""
        from .. import ingest
        from ..pipeline import GeneSpec, HotPath
        from ..stage1 import CohortVariants, cre_window, gene_window
        ds = self.model_config.dataset
        dataset = VCFDataset(max_length=ds.max_length, max_chunks=ds.max_chunks, cre_neighbour_hood=ds.cre_neighbour_hood,
                             gencode_v24=ds.gencode_v24, gene_cre_manifest=self.gene_cre_manifest,
                             gene_upstream_neighbour_hood=ds.gene_upstream_neighbour_hood,
                             gene_downstream_neighbour_hood=ds.gene_downstream_neighbour_hood, query_df=query_df,
                             fasta_path=self.vcf_loader_config.fasta_path, vcf_path=None)
        q = dataset.query_df
        genes, gene_ids, tissue_names, regions = [], [], [], []
        nb, up, down = ds.cre_neighbour_hood, ds.gene_upstream_neighbour_hood, ds.gene_downstream_neighbour_hood
        for _, row in q.iterrows():
            info = dataset._get_gene_info(row["gene_id"])
            assert info["chromosome"] in ["chr" + str(i) for i in range(1, 23)], \
                f"Chromosome {info['chromosome']} is not a valid chromosome. Sex chromosomes are not supported"
            m, _ = dataset.cre_manifest(row["gene_id"], info)
            labels = np.asarray([dataset.ref_cre_to_idx[x] for x in m["cre_name"]], np.int64)
            genes.append(GeneSpec(info["chromosome"], int(info["start"]), int(info["end"]), info["strand"],
                                  m["start_cre"].to_numpy(np.int64), m["end_cre"].to_numpy(np.int64), labels,
                                  list(row["tissues"]), cre_chrom=list(m["chromosome"])))
            gene_ids.append(row["gene_id"]); tissue_names.append(list(row["tissue_names"]))
            regions += [(c, *cre_window(s, e, nb)) for c, s, e in zip(m["chromosome"], m["start_cre"], m["end_cre"])]
            regions.append((info["chromosome"], *gene_window(info["start"], info["end"], info["strand"], up, down)))
        names, per_sample = ingest.load_vcf_cohort(vcf_path, samples=samples, regions=regions)
        model, _, _ = self.load_model()
        hot = HotPath(model.engine(), dataset._genome(), max_length=ds.max_length, max_chunks=ds.max_chunks,
                      cre_neighbour_hood=nb, gene_upstream=up, gene_downstream=down)
        g_blocks = [(a, min(len(genes), a + genes_per_slab)) for a in range(0, len(genes), genes_per_slab)]
        s_blocks = [(a, min(len(names), a + samples_per_slab)) for a in range(0, len(names), samples_per_slab)]
        writer = None
        if output_dir is not None:
            from ..writer import ResultWriter
            writer = ResultWriter(output_dir, hot.engine.w.D, embeddings=embeddings,
                                  meta={"cohort": os.path.basename(vcf_path), "samples": names, "genes": gene_ids,
                                        "tissues": [list(map(int, g.tissues)) for g in genes],
                                        "genes_per_slab": genes_per_slab, "samples_per_slab": samples_per_slab})
            done = writer.done()
        frames = {}
        try:
            for sb, (s0, s1) in enumerate(s_blocks):
                todo = [gb for gb in range(len(g_blocks)) if writer is None or gb * len(s_blocks) + sb not in done]
                if not todo:
                    continue
                # sample sub-blocks whose variant tables fit the kernels' int32 indices (one, short of 2^31 records)
                subs = CohortVariants.blocks(per_sample[s0:s1])
                table = lambda a, b: CohortVariants(names[s0 + a:s0 + b], per_sample[s0 + a:s0 + b], hot.engine.device)
                kept = table(*subs[0]) if len(subs) == 1 else None
                for gb in todo:
                    g0, g1 = g_blocks[gb]
                    parts = [hot.predict_cohort(genes[g0:g1], kept if kept is not None else table(a, b),
                                                min_gene_len=1000, gene_names=gene_ids[g0:g1]) for a, b in subs]
                    pred = np.concatenate([p for p, _ in parts]); emb = np.concatenate([e for _, e in parts])
                    del parts
                    rows = [(k, names[s0 + s], gene_ids[g0 + k], int(t), tn)
                            for s in range(s1 - s0) for k in range(g1 - g0)
                            for t, tn in zip(genes[g0 + k].tissues, tissue_names[g0 + k])]
                    pred = pred.reshape(-1); emb = emb.reshape(len(rows), -1)
                    if writer is not None:
                        writer.submit(gb * len(s_blocks) + sb, [r[:4] for r in rows], pred, emb)
                    else:
                        frames[(sb, gb)] = (rows, pred, emb)
        finally:
            if writer is not None:
                writer.close()
        if writer is not None:
            return output_dir
        # (sample, gene, tissue) order: sample blocks outer, then sample, gene block, gene, tissue
        out = []
        for sb, (s0, s1) in enumerate(s_blocks):
            parts = [frames[(sb, gb)] for gb in range(len(g_blocks))]
            per_s = [[] for _ in range(s1 - s0)]
            for (g0, g1), (rows, pred, emb) in zip(g_blocks, parts):
                n = len(rows) // (s1 - s0)
                for s in range(s1 - s0):
                    per_s[s].append((rows[s * n:(s + 1) * n], pred[s * n:(s + 1) * n], emb[s * n:(s + 1) * n]))
            for lst in per_s:
                for rows, pred, emb in lst:
                    d = {"sample": [r[1] for r in rows], "gene_id": [r[2] for r in rows], "tissue": [r[4] for r in rows],
                         "predicted_expression": pred}
                    if embeddings:
                        d["embeddings"] = list(emb)
                    out.append(pd.DataFrame(d))
        return pd.concat(out, ignore_index=True)

    def cre_knockout(self, vcf_path: str, query_df: pd.DataFrame, knockouts: pd.DataFrame = None):
        """In-silico CRE knockout (DESIGN.md section 15): every query row predicted with one CRE, or a set of CREs,
        removed from its gene's manifest, each distinct window encoded once.  A knockout's prediction equals what
        create_data + predict give with those rows deleted from the manifest.  The query is filtered with VCFDataset's
        rules; the sample is `vcf_path` or a per-row vcf_path column (empty or missing: the reference genome).
        knockouts: None = every CRE of every query gene singly (a gene with one CRE gets none), or a DataFrame with
        columns gene_id, knockout (a label) and cre_index (a manifest row; one row per member of the set).  Invalid sets
        raise a ValueError before any device work.  Writes no file.
        -> one row per (query row, knockout, tissue), in that order (default knockouts in manifest order, user sets in
        first-appearance order): gene_id, tissue (name), knockout (label; the manifest row for the default scan),
        cre_indices, the manifest columns of a single-CRE knockout (null for larger sets), baseline_expression,
        predicted_expression and delta = predicted - baseline."""
        from .. import knockout as ko
        from ..pipeline import GeneSpec, HotPath
        ds = self.model_config.dataset
        dataset = VCFDataset(max_length=ds.max_length, max_chunks=ds.max_chunks, cre_neighbour_hood=ds.cre_neighbour_hood,
                             gencode_v24=ds.gencode_v24, gene_cre_manifest=self.gene_cre_manifest,
                             gene_upstream_neighbour_hood=ds.gene_upstream_neighbour_hood,
                             gene_downstream_neighbour_hood=ds.gene_downstream_neighbour_hood, query_df=query_df,
                             fasta_path=self.vcf_loader_config.fasta_path, vcf_path=vcf_path)
        q = dataset.query_df
        user = ko.knockout_sets(knockouts) if knockouts is not None else None
        genes, manifests, sets, paths = [], [], [], []
        for _, row in q.iterrows():
            gid = row["gene_id"]
            info = dataset._get_gene_info(gid)
            assert info["chromosome"] in ["chr" + str(i) for i in range(1, 23)], \
                f"Chromosome {info['chromosome']} is not a valid chromosome. Sex chromosomes are not supported"
            m, _ = dataset.cre_manifest(gid, info)
            labels = np.asarray([dataset.ref_cre_to_idx[x] for x in m["cre_name"]], np.int64)
            genes.append(GeneSpec(info["chromosome"], int(info["start"]), int(info["end"]), info["strand"],
                                  m["start_cre"].to_numpy(np.int64), m["end_cre"].to_numpy(np.int64), labels,
                                  list(row["tissues"]), cre_chrom=list(m["chromosome"])))
            manifests.append(m)
            if user is not None:
                sets.append(user.get(gid, []))
            elif len(m) > 1:
                sets.append([(i, np.asarray([i], np.int64)) for i in range(len(m))])
            else:
                print(f"Gene {gid} has a single CRE so skipping its knockouts")
                sets.append([])
            p = row["vcf_path"] if "vcf_path" in q.columns else vcf_path
            paths.append(None if p is None or (not isinstance(p, str) and pd.isna(p)) or str(p) == "" else str(p))
        if user is not None:
            for gid in user:
                if gid not in set(q["gene_id"]):
                    print(f"Gene {gid} of the knockouts is not in the query so skipping it")
        gene_ids = list(q["gene_id"])
        checked = ko.check_knockouts(genes, [[ix for _, ix in s] for s in sets], gene_ids,
                                     [[lab for lab, _ in s] for s in sets])
        sets = [[(lab, ix) for (lab, _), ix in zip(s, c)] for s, c in zip(sets, checked)]
        model, _, _ = self.load_model()
        hot = HotPath(model.engine(), dataset._genome(), max_length=ds.max_length, max_chunks=ds.max_chunks,
                      cre_neighbour_hood=ds.cre_neighbour_hood, gene_upstream=ds.gene_upstream_neighbour_hood,
                      gene_downstream=ds.gene_downstream_neighbour_hood)
        base, kos = [None] * len(genes), [None] * len(genes)
        for p in dict.fromkeys(paths):                       # one call per sample, in first-appearance order
            rows = [i for i, x in enumerate(paths) if x == p]
            pred, _, ko_pred = hot.cre_knockout([genes[i] for i in rows], [[ix for _, ix in sets[i]] for i in rows],
                                                dataset._variants(p), min_gene_len=1000,
                                                gene_names=[gene_ids[i] for i in rows])
            off = np.concatenate([[0], np.cumsum([len(genes[i].tissues) for i in rows])])
            for k, i in enumerate(rows):
                base[i], kos[i] = pred[off[k]:off[k + 1]], ko_pred[k]
        frames = [ko.knockout_frame(gid, list(q["tissue_names"].iloc[i]), manifests[i], sets[i], base[i], kos[i])
                  for i, gid in enumerate(gene_ids)]
        return pd.concat(frames, ignore_index=True)

    def deletion_scan(self, vcf_path: str, query_df: pd.DataFrame, deletions: pd.DataFrame = None):
        """In-silico genomic deletions (DESIGN.md section 16): every query row predicted with a span of the genome
        deleted, each window the deletion does not change encoded once.  A deletion [start, end] (1-based, inclusive)
        gives what create_data + predict give on the sample's VCF with one more line: POS = start - 1, REF = the
        reference bases start - 1 .. end, ALT = the anchor base, GT 1/1.  The query is filtered with VCFDataset's rules;
        the sample is `vcf_path` or a per-row vcf_path column (empty or missing: the reference genome).
        deletions: None = every CRE's own bases deleted singly, on its manifest chromosome ([start_cre + 1, end_cre]),
        or a DataFrame with columns gene_id, chromosome, start, end and optionally label (deletion.tiles builds tilings).
        Invalid spans raise a ValueError before the model is loaded.  Writes no file.
        -> one row per (query row, deletion, tissue), in that order (default deletions in manifest order, user ones in
        first-appearance order), columns deletion.FRAME_COLUMNS: deletion (label; the manifest row for the default
        scan), chromosome, del_start, del_end, width, cre_windows_changed / gene_window_changed / changed (windows whose
        bytes the deletion changed), the deleted CRE's manifest columns (default scan; null otherwise),
        baseline_expression, predicted_expression and delta = predicted - baseline."""
        from .. import deletion as dl
        from ..pipeline import GeneSpec, HotPath
        ds = self.model_config.dataset
        dataset = VCFDataset(max_length=ds.max_length, max_chunks=ds.max_chunks, cre_neighbour_hood=ds.cre_neighbour_hood,
                             gencode_v24=ds.gencode_v24, gene_cre_manifest=self.gene_cre_manifest,
                             gene_upstream_neighbour_hood=ds.gene_upstream_neighbour_hood,
                             gene_downstream_neighbour_hood=ds.gene_downstream_neighbour_hood, query_df=query_df,
                             fasta_path=self.vcf_loader_config.fasta_path, vcf_path=vcf_path)
        q = dataset.query_df
        user = dl.user_deletions(deletions) if deletions is not None else None
        genes, manifests, dels, paths = [], [], [], []
        for _, row in q.iterrows():
            gid = row["gene_id"]
            info = dataset._get_gene_info(gid)
            assert info["chromosome"] in ["chr" + str(i) for i in range(1, 23)], \
                f"Chromosome {info['chromosome']} is not a valid chromosome. Sex chromosomes are not supported"
            m, _ = dataset.cre_manifest(gid, info)
            labels = np.asarray([dataset.ref_cre_to_idx[x] for x in m["cre_name"]], np.int64)
            genes.append(GeneSpec(info["chromosome"], int(info["start"]), int(info["end"]), info["strand"],
                                  m["start_cre"].to_numpy(np.int64), m["end_cre"].to_numpy(np.int64), labels,
                                  list(row["tissues"]), cre_chrom=list(m["chromosome"])))
            manifests.append(m)
            if user is not None:
                dels.append(user.get(gid, ([], np.zeros((0, 2), np.int64), [])))
            else:
                spans, chroms = dl.default_spans(m)
                dels.append((list(range(len(m))), spans, chroms))
            p = row["vcf_path"] if "vcf_path" in q.columns else vcf_path
            paths.append(None if p is None or (not isinstance(p, str) and pd.isna(p)) or str(p) == "" else str(p))
        if user is not None:
            for gid in user:
                if gid not in set(q["gene_id"]):
                    print(f"Gene {gid} of the deletions is not in the query so skipping it")
        gene_ids = list(q["gene_id"])
        genome = dataset._genome()
        dl.check_deletions(genes, [d[1] for d in dels], [d[2] for d in dels],
                           {k: v[1] for k, v in genome.offsets.items()}, gene_ids)
        model, _, _ = self.load_model()
        hot = HotPath(model.engine(), genome, max_length=ds.max_length, max_chunks=ds.max_chunks,
                      cre_neighbour_hood=ds.cre_neighbour_hood, gene_upstream=ds.gene_upstream_neighbour_hood,
                      gene_downstream=ds.gene_downstream_neighbour_hood)
        base, dpred, applied = [None] * len(genes), [None] * len(genes), [None] * len(genes)
        for p in dict.fromkeys(paths):                       # one call per sample, in first-appearance order
            rows = [i for i, x in enumerate(paths) if x == p]
            pred, _, d_pred, app = hot.deletion_scan([genes[i] for i in rows], [dels[i][1] for i in rows],
                                                     dataset._variants(p), chroms=[dels[i][2] for i in rows],
                                                     min_gene_len=1000, gene_names=[gene_ids[i] for i in rows])
            off = np.concatenate([[0], np.cumsum([len(genes[i].tissues) for i in rows])])
            for k, i in enumerate(rows):
                base[i], dpred[i], applied[i] = pred[off[k]:off[k + 1]], d_pred[k], app[k]
        frames = [dl.deletion_frame(gid, list(q["tissue_names"].iloc[i]), dels[i][0], dels[i][1], dels[i][2],
                                    applied[i], base[i], dpred[i], manifests[i] if user is None else None)
                  for i, gid in enumerate(gene_ids)]
        return pd.concat(frames, ignore_index=True)

    def _edit_query(self, vcf_path, query_df):
        """The query of an in-silico edit with VCFDataset's rules: -> (dataset, filtered query, GeneSpec per row, sample
        path per row (None: the reference genome))."""
        from ..pipeline import GeneSpec
        ds = self.model_config.dataset
        dataset = VCFDataset(max_length=ds.max_length, max_chunks=ds.max_chunks, cre_neighbour_hood=ds.cre_neighbour_hood,
                             gencode_v24=ds.gencode_v24, gene_cre_manifest=self.gene_cre_manifest,
                             gene_upstream_neighbour_hood=ds.gene_upstream_neighbour_hood,
                             gene_downstream_neighbour_hood=ds.gene_downstream_neighbour_hood, query_df=query_df,
                             fasta_path=self.vcf_loader_config.fasta_path, vcf_path=vcf_path)
        q = dataset.query_df
        genes, paths = [], []
        for _, row in q.iterrows():
            gid = row["gene_id"]
            info = dataset._get_gene_info(gid)
            assert info["chromosome"] in ["chr" + str(i) for i in range(1, 23)], \
                f"Chromosome {info['chromosome']} is not a valid chromosome. Sex chromosomes are not supported"
            m, _ = dataset.cre_manifest(gid, info)
            labels = np.asarray([dataset.ref_cre_to_idx[x] for x in m["cre_name"]], np.int64)
            genes.append(GeneSpec(info["chromosome"], int(info["start"]), int(info["end"]), info["strand"],
                                  m["start_cre"].to_numpy(np.int64), m["end_cre"].to_numpy(np.int64), labels,
                                  list(row["tissues"]), cre_chrom=list(m["chromosome"])))
            p = row["vcf_path"] if "vcf_path" in q.columns else vcf_path
            paths.append(None if p is None or (not isinstance(p, str) and pd.isna(p)) or str(p) == "" else str(p))
        return dataset, q, genes, paths

    def _run_sets(self, dataset, genes, sets, paths, gene_ids):
        """variant_sets.scan per sample (one HotPath call per distinct path, in first-appearance order).
        -> per query row (baseline fp32 [T], set predictions [n, T], applied)."""
        from ..pipeline import HotPath
        ds = self.model_config.dataset
        model, _, _ = self.load_model()
        hot = HotPath(model.engine(), dataset._genome(), max_length=ds.max_length, max_chunks=ds.max_chunks,
                      cre_neighbour_hood=ds.cre_neighbour_hood, gene_upstream=ds.gene_upstream_neighbour_hood,
                      gene_downstream=ds.gene_downstream_neighbour_hood)
        out = [None] * len(genes)
        for p in dict.fromkeys(paths):
            rows = [i for i, x in enumerate(paths) if x == p]
            pred, _, s_pred, app = hot.variant_sets([genes[i] for i in rows], [sets[i] for i in rows],
                                                    dataset._variants(p), min_gene_len=1000,
                                                    gene_names=[gene_ids[i] for i in rows])
            off = np.concatenate([[0], np.cumsum([len(genes[i].tissues) for i in rows])])
            for k, i in enumerate(rows):
                out[i] = (pred[off[k]:off[k + 1]], s_pred[k], app[k])
        return out

    def variant_sets(self, vcf_path: str, query_df: pd.DataFrame, variants: pd.DataFrame):
        """In-silico variant combinations (DESIGN.md section 17): every query row predicted with each set of VCF
        records added to its sample, each window no record of the set lies in encoded once.  A set's prediction equals
        what create_data + predict give on the sample's VCF with the set's lines added (each after the lines of its
        POS).  The query is filtered with VCFDataset's rules; the sample is `vcf_path` or a per-row vcf_path column
        (empty or missing: the reference genome).  variants: DataFrame with columns gene_id, set (a label), chromosome,
        pos (1-based), ref, alt, optionally gt (1 het, 2 hom-alt; default 2) and label; one row per record.  Invalid
        records raise a ValueError before the model is loaded.  Writes no file.
        -> one row per (query row, set, tissue), in that order (sets in first-appearance order), columns
        variant_sets.SET_COLUMNS: set, n_records, records_applied (records applied in at least one window),
        cre_windows_changed / gene_window_changed / changed, baseline_expression, predicted_expression and delta."""
        from .. import variant_sets as vs
        user = vs.user_records(variants, sets=True)
        dataset, q, genes, paths = self._edit_query(vcf_path, query_df)
        gene_ids = list(q["gene_id"])
        for gid in user:
            if gid not in set(gene_ids):
                print(f"Gene {gid} of the variant sets is not in the query so skipping it")
        sets = [user.get(gid, []) for gid in gene_ids]
        vs.check_sets(genes, [[rs for _, rs, _ in s] for s in sets], dataset._genome(), gene_ids)
        res = self._run_sets(dataset, genes, [[rs for _, rs, _ in s] for s in sets], paths, gene_ids)
        frames = [vs.set_frame(gid, list(q["tissue_names"].iloc[i]), [sid for sid, _, _ in sets[i]],
                               [len(rs) for _, rs, _ in sets[i]], res[i][2], res[i][0], res[i][1])
                  for i, gid in enumerate(gene_ids)]
        return pd.concat(frames, ignore_index=True)

    def cohort_variant_sets(self, vcf_path: str, query_df: pd.DataFrame, variants: pd.DataFrame, samples=None,
                            genes_per_slab=8, samples_per_slab=256):
        """Variant sets across a cohort (DESIGN.md section 18): every query row predicted, in every sample of one
        multi-sample VCF (samples: names, default every sample column), with each set of records added to that sample.
        The query follows predict_cohort's rules (VCFDataset's filtering, one region-restricted parse of the VCF, sample
        sub-blocks past the kernels' int32 limits); variants as variant_sets (gene_id, set, chromosome, pos, ref, alt,
        optionally gt and label), invalid records raising a ValueError before the model is loaded.  A record the
        sample's own records block is not applied in that sample (records_applied / changed say so per sample).  Each
        row equals what variant_sets gives on that sample's VCF alone.  Computed in slabs of genes_per_slab query genes x
        samples_per_slab samples, so device memory does not grow with the query or the cohort.  Writes no file.
        -> one row per (sample, query row, set, tissue), in that order: sample, then variant_sets.SET_COLUMNS
        (variant_sets.cohort_summary condenses it over the samples)."""
        from .. import ingest
        from .. import variant_sets as vs
        from ..pipeline import HotPath
        from ..stage1 import CohortVariants, cre_window, gene_window
        user = vs.user_records(variants, sets=True)
        dataset, q, genes, _ = self._edit_query(None, query_df)
        gene_ids = list(q["gene_id"])
        for gid in user:
            if gid not in set(gene_ids):
                print(f"Gene {gid} of the variant sets is not in the query so skipping it")
        sets = [user.get(gid, []) for gid in gene_ids]
        recs = [[rs for _, rs, _ in s] for s in sets]
        vs.check_sets(genes, recs, dataset._genome(), gene_ids)
        ds = self.model_config.dataset
        nb, up, down = ds.cre_neighbour_hood, ds.gene_upstream_neighbour_hood, ds.gene_downstream_neighbour_hood
        regions = []
        for g in genes:
            regions += [(c, *cre_window(a, b, nb)) for c, a, b in zip(g.cre_chrom, g.cre_start, g.cre_end)]
            regions.append((g.chrom, *gene_window(g.start, g.end, g.strand, up, down)))
        names, per_sample = ingest.load_vcf_cohort(vcf_path, samples=samples, regions=regions)
        model, _, _ = self.load_model()
        hot = HotPath(model.engine(), dataset._genome(), max_length=ds.max_length, max_chunks=ds.max_chunks,
                      cre_neighbour_hood=nb, gene_upstream=up, gene_downstream=down)
        frames = []
        for s0 in range(0, len(names), samples_per_slab):
            s1 = min(len(names), s0 + samples_per_slab)
            per_s = [[] for _ in range(s1 - s0)]             # frames of each sample of the slab, in query order
            # sample sub-blocks whose variant tables fit the kernels' int32 indices
            for a, b in CohortVariants.blocks(per_sample[s0:s1]):
                cv = CohortVariants(names[s0 + a:s0 + b], per_sample[s0 + a:s0 + b], hot.engine.device)
                for g0 in range(0, len(genes), genes_per_slab):
                    g1 = min(len(genes), g0 + genes_per_slab)
                    pred, _, s_pred, app = hot.cohort_variant_sets(genes[g0:g1], recs[g0:g1], cv, min_gene_len=1000,
                                                                   gene_names=gene_ids[g0:g1])
                    off = np.concatenate([[0], np.cumsum([len(g.tissues) for g in genes[g0:g1]])])
                    for s in range(b - a):
                        for k, i in enumerate(range(g0, g1)):
                            ap = dict(cre=app[k]["cre"][s], gene=app[k]["gene"][s],
                                      records=[r[s] for r in app[k]["records"]])
                            f = vs.set_frame(gene_ids[i], list(q["tissue_names"].iloc[i]), [sid for sid, _, _ in sets[i]],
                                             [len(rs) for rs in recs[i]], ap, pred[s, off[k]:off[k + 1]], s_pred[k][s])
                            f.insert(0, "sample", names[s0 + a + s])
                            per_s[a + s].append(f)
                    del pred, s_pred, app
                del cv
            frames += [f for fs in per_s for f in fs]
        if not frames:
            return pd.DataFrame(columns=["sample"] + vs.SET_COLUMNS)
        return pd.concat(frames, ignore_index=True)

    def variant_attribution(self, vcf_path: str, query_df: pd.DataFrame, edits: pd.DataFrame = None, scope="record"):
        """Variant attribution (DESIGN.md section 19): every query row predicted with some of its sample's own records
        removed or re-genotyped, each window no edit lies in encoded once.  A set's prediction equals what create_data +
        predict give on the sample's VCF with those lines removed (GT 0) or their GT rewritten.  The query is filtered
        with VCFDataset's rules; the sample is `vcf_path` or a per-row vcf_path column.  edits: None = the default scan,
        scope "record" (leave-one-out: each record of the sample whose REF span lies in one of the gene's windows and
        whose GT is not 0, removed singly) or "window" (each window holding such records reverted to the reference); or
        a DataFrame with columns gene_id, chromosome, pos (1-based), ref, alt, gt (the new GT: 0, 1 or 2) and
        optionally set (a label; one set per row without it) and label.  Invalid edits raise a ValueError before the
        model is loaded.  A row whose sample has no record in the gene's windows gives no rows.  Writes no file.
        -> one row per (query row, set, tissue), in that order, columns variant_attribution.ATTRIBUTION_COLUMNS:
        variant_sets.SET_COLUMNS (changed: a window's tokens differ from the baseline's), sample_gt and new_gt
        (single-record sets), reference_expression (every record in the gene's windows removed) and delta =
        predicted - baseline (a removed record contributes -delta)."""
        from .. import variant_attribution as va
        from ..pipeline import HotPath
        if scope not in va.SCOPES:
            raise ValueError(f"scope must be one of {va.SCOPES}, got {scope!r}")
        user = va.user_edits(edits) if edits is not None else None
        dataset, q, genes, paths = self._edit_query(vcf_path, query_df)
        gene_ids = list(q["gene_id"])
        if user is not None:
            for gid in user:
                if gid not in set(gene_ids):
                    print(f"Gene {gid} of the edits is not in the query so skipping it")
        ds = self.model_config.dataset
        nb, up, down = ds.cre_neighbour_hood, ds.gene_upstream_neighbour_hood, ds.gene_downstream_neighbour_hood
        genome = dataset._genome()
        todo = []                                            # (row, sets incl. the all-removed one last, labels, gts)
        for i, (g, gid, p) in enumerate(zip(genes, gene_ids, paths)):
            v = dataset._variants(p)
            ref = va.all_removed(g, v, nb, up, down)
            if user is not None:
                us = user.get(gid, [])
                sets = va.check_edits([g], [[es for _, es, _ in us]], v, [gid])[0]
                labels = [sid for sid, _, _ in us]
                gts = [va.sample_gt(v, s[0]) if len(s) == 1 else None for s in sets]
            else:
                if not ref:
                    continue
                sets, labels, gts = va.default_sets(g, v, nb, up, down, scope, genome)
            if sets:
                todo.append((i, sets + [ref], labels, gts))
        frames = []
        if todo:
            model, _, _ = self.load_model()
            hot = HotPath(model.engine(), genome, max_length=ds.max_length, max_chunks=ds.max_chunks,
                          cre_neighbour_hood=nb, gene_upstream=up, gene_downstream=down)
            res = {}
            for p in dict.fromkeys(paths[t[0]] for t in todo):   # one call per sample, in first-appearance order
                part = [t for t in todo if paths[t[0]] == p]
                pred, _, s_pred, app = va.run(hot, [genes[t[0]] for t in part], [t[1] for t in part],
                                              dataset._variants(p), min_gene_len=1000,
                                              gene_names=[gene_ids[t[0]] for t in part])
                off = np.concatenate([[0], np.cumsum([len(genes[t[0]].tissues) for t in part])])
                for k, t in enumerate(part):
                    res[t[0]] = (pred[off[k]:off[k + 1]], s_pred[k], app[k])
            for i, sets, labels, gts in todo:
                base, sp, ap = res[i]
                n = len(labels)
                ap = dict(cre=ap["cre"][:n], gene=ap["gene"][:n], records=ap["records"][:n])
                frames.append(va.attribution_frame(gene_ids[i], list(q["tissue_names"].iloc[i]), labels, sets[:n], gts,
                                                   ap, base, sp[:n], sp[n]))
        if not frames:
            return pd.DataFrame(columns=va.ATTRIBUTION_COLUMNS)
        return pd.concat(frames, ignore_index=True)

    def variant_interactions(self, vcf_path: str, query_df: pd.DataFrame, variants: pd.DataFrame):
        """Pairwise interaction scan (DESIGN.md section 17): for every query row, each of its gene's variants singly and
        every unordered pair of them added to the sample, all in one planner call per sample.  Query and sample as
        variant_sets; variants: DataFrame with columns gene_id, chromosome, pos (1-based), ref, alt, optionally gt
        (default 2) and label.  Pairs whose REF spans overlap (two alleles of one site) are skipped.  Invalid records
        raise a ValueError before the model is loaded.  Writes no file.
        -> one row per (query row, pair, tissue), columns variant_sets.INTERACTION_COLUMNS: variant_a / variant_b
        (labels), same_window (one window holds both), baseline_expression, expression_a / _b / _ab, delta_a / _b / _ab,
        interaction = delta_ab - delta_a - delta_b and log2_interaction = log2((ab + 1e-10)(base + 1e-10) /
        ((a + 1e-10)(b + 1e-10)))."""
        from .. import variant_sets as vs
        user = vs.user_records(variants, sets=False)
        dataset, q, genes, paths = self._edit_query(vcf_path, query_df)
        gene_ids = list(q["gene_id"])
        for gid in user:
            if gid not in set(gene_ids):
                print(f"Gene {gid} of the variants is not in the query so skipping it")
        scans = []
        for gid in gene_ids:
            recs, labels = user.get(gid, ([], []))
            sets, _, pair_idx, overlapping = vs.pairs(recs)
            for a, b in overlapping:
                print(f"Variants {labels[a]} and {labels[b]} of gene {gid} overlap so skipping their pair")
            scans.append((labels, sets, pair_idx))
        ds = self.model_config.dataset
        checked = vs.check_sets(genes, [s for _, s, _ in scans], dataset._genome(), gene_ids)
        res = self._run_sets(dataset, genes, [s for _, s, _ in scans], paths, gene_ids)
        frames = []
        for i, gid in enumerate(gene_ids):
            labels, sets, pair_idx = scans[i]
            n = len(labels)
            same = vs.shared_window(genes[i], checked[i][n:], ds.cre_neighbour_hood, ds.gene_upstream_neighbour_hood,
                                    ds.gene_downstream_neighbour_hood)
            base, sp, _ = res[i]
            frames.append(vs.interaction_frame(gid, list(q["tissue_names"].iloc[i]), labels, pair_idx, same, base,
                                               sp[:n], sp[n:]))
        return pd.concat(frames, ignore_index=True)

    def format_output(self, df, predictions):
        pred_exp, embd = [], []
        for p in predictions:
            pred_exp.extend(p["pred_gene_exp"]); embd.extend(p["embeddings"])
        assert len(df) == len(pred_exp), "DataFrame and predictions length mismatch"
        df["predicted_expression"] = pd.Series(pred_exp, index=df.index)
        df["embeddings"] = pd.Series(embd, index=df.index)
        return df


def cre_attention_frame(gene_id, tissues, manifest, order, maps_batch, pred):
    """One gene's maps in manifest order and long format.  manifest: DataFrame (chromosome, start_cre, end_cre,
    cre_name); order: manifest row of every CRE in batch order; maps_batch: [T, layers, heads, C] in batch order; pred:
    [T, 1].  -> (df, {(gene_id, tissue): [layers, heads, C]})."""
    maps_batch = np.asarray(maps_batch)
    T, L, H, C = maps_batch.shape
    assert len(manifest) == C and len(order) == C and len(tissues) == T
    m = np.empty_like(maps_batch)
    m[..., np.asarray(order)] = maps_batch                   # batch position k holds manifest row order[k]
    att = m.mean(axis=2)                                    # [T, L, C]
    rep = lambda col: np.tile(manifest[col].to_numpy(), T * L)
    df = pd.DataFrame({"gene_id": gene_id, "tissue": np.repeat(np.asarray(tissues, object), L * C),
                       "layer": np.tile(np.repeat(np.arange(L), C), T), "chromosome": rep("chromosome"),
                       "start_cre": rep("start_cre"), "end_cre": rep("end_cre"), "cre_name": rep("cre_name"),
                       "attention": att.reshape(-1),
                       "predicted_expression": np.repeat(np.asarray(pred, np.float32).reshape(T), L * C)})
    return df, {(gene_id, t): m[k] for k, t in enumerate(tissues)}
