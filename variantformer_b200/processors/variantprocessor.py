"""VariantProcessor — variant-effect scoring with the reference's call shape
(processors/variantprocessor.py:31-123, :499-513: `VariantProcessor(model_class).predict(var_df, output_dir,
vcf_path=None, sample_name=None) -> DataFrame`) and its long-format output columns (:303-445).

In scope here: the hot path — triplet construction on the GPU (datasets/vepdataset.py), one batched
`variant_prediction` per (variant, gene) pair, zygosity-wise expression / embedding rows and the log2 fold change.
Out of scope (SURVEY §2.1 #4, #10, #12): the variant->gene annotation join (`multi_datasets_loader.py`; `var_df`
must carry `gene_id`), the 1000-Genomes population sequence tables on S3 (`population` is always "REF_HG38" or the
given sample) and the AF-weighted aggregate scores.
"""
import logging
import os

import numpy as np
import pandas as pd
import torch

from .. import ingest
from ..datasets.vcfdataset import LocalGeneManifest
from ..datasets.vepdataset import Variant, VEPBatchBuilder
from ..pipeline import GeneSpec
from ..stage1 import Genome
from ..utils.config import CONFIG_DIR, PACKAGE_ROOT, VOCAB_DIR, load_yaml
from ..utils.constants import MAP_REF_CRE_TO_IDX
from .model_manager import ModelManager
from .vcfprocessor import Trainer

log = logging.getLogger(__name__)


class VariantProcessor:
    def __init__(self, model_class: str = "v4_pcg", base_dir=None, gene_cre_manifest=None, model_overrides=None):
        base_dir = base_dir or PACKAGE_ROOT
        self.base_dir = base_dir
        self.model_config = load_yaml(os.path.join(CONFIG_DIR, "vf_model.yaml"))[model_class]
        if model_overrides:
            self.model_config.model.update(model_overrides)
        self.vep_loader_config = load_yaml(os.path.join(CONFIG_DIR, "veploader.yaml"))
        self.tissue_vocab = load_yaml(os.path.join(VOCAB_DIR, "tissue_vocab.yaml"))
        self.tissue_idx_to_name = {v: k for k, v in self.tissue_vocab.items()}
        self.gene_cre_manifest = gene_cre_manifest or LocalGeneManifest(
            os.path.join(base_dir, "_artifacts", "gene_cre_manifests"))

        def fix(node, key):
            if node.get(key) and not os.path.isabs(node[key]):
                node[key] = os.path.join(base_dir, node[key])
        fix(self.vep_loader_config, "fasta_path"); fix(self.vep_loader_config, "af_path")
        fix(self.model_config.dataset, "gencode_v24")
        fix(self.model_config.model, "checkpoint_path")
        fix(self.model_config.model.cre_tokenizer, "path"); fix(self.model_config.model.gene_tokenizer, "path")
        assert torch.cuda.is_available(), "GPU is not available"
        self.model_manager = ModelManager(self.model_config.model)
        self._genome = None

    # ------------------------------------------------------------------------------------------------------------
    def _gene_spec(self, gene_row, tissues):
        m = pd.read_csv(self.gene_cre_manifest.get_file_path(gene_row["gene_id"]))
        return GeneSpec(gene_row["chromosome"], int(gene_row["start"]), int(gene_row["end"]), gene_row["strand"],
                        m["start_cre"].to_numpy(np.int64), m["end_cre"].to_numpy(np.int64),
                        np.asarray([MAP_REF_CRE_TO_IDX.get(c, 0) for c in m["cre_name"]], np.int64), tissues,
                        cre_chrom=list(m["chromosome"]))

    def _load_inputs(self, vcf_path=None, sample_name=None):
        """Genome (loaded once, HBM-resident), the optional background sample and the gene table."""
        genes = pd.read_csv(self.model_config.dataset.gencode_v24).set_index("gene_id", drop=False)
        if self._genome is None:
            self._genome = Genome.from_arrays(ingest.load_fasta(self.vep_loader_config.fasta_path), "cuda")
        self.background = ingest.load_vcf_sample(vcf_path, sample=sample_name) if vcf_path else None
        return genes

    def initialize(self, var_df, output_dir, vcf_path=None, sample_name=None):
        """-> (pairs, model, trainer, checkpoint_path).  One pair per (variant row, gene)."""
        os.makedirs(output_dir, exist_ok=True)
        self.output_file = os.path.join(output_dir, "variants_VF.parquet")
        if os.path.exists(self.output_file):                        # variantprocessor.py:151-154, 284-301
            raise FileExistsError(f"{self.output_file} already exists; refusing to overwrite")
        df = var_df.rename(columns={"chr": "chrom"})
        for col in ("chrom", "pos", "ref", "alt", "tissue", "gene_id"):
            assert col in df.columns, f"var_df must contain a '{col}' column"
        genes = self._load_inputs(vcf_path, sample_name)
        pairs = []
        for _, r in df.iterrows():
            names = [t.strip() for t in str(r["tissue"]).split(",") if t.strip() in self.tissue_vocab]
            if r["gene_id"] not in genes.index or not names:
                log.info(f"skipping {r['chrom']}:{r['pos']} / {r['gene_id']}: unknown gene or tissue")
                continue
            tissues = [self.tissue_vocab[t] for t in names]
            v = Variant(str(r["chrom"]), int(r["pos"]), str(r["ref"]), str(r["alt"]), tissue=tissues,
                        gene_id=[r["gene_id"]])
            pairs.append(dict(variant=v, gene=self._gene_spec(genes.loc[r["gene_id"]], tissues),
                              gene_id=r["gene_id"], population="SAMPLE" if vcf_path else "REF_HG38",
                              sample_name=sample_name or "hg38"))
        model, ckpt = self.model_manager.load_model()
        model.vep = True
        trainer = Trainer(precision=self.model_config.model.precision)
        return pairs, model, trainer, ckpt

    def predict(self, var_df: pd.DataFrame, output_dir: str, vcf_path: str = None, sample_name: str = None):
        pairs, model, trainer, _ = self.initialize(var_df, output_dir, vcf_path, sample_name)
        ds = self.model_config.dataset
        builder = VEPBatchBuilder(self._genome, "cuda", max_length=ds.max_length, context_window=ds.max_chunks,
                                  cre_neighbour_hood=ds.cre_neighbour_hood,
                                  gene_upstream_neighbour_hood=ds.gene_upstream_neighbour_hood,
                                  gene_downstream_neighbour_hood=ds.gene_downstream_neighbour_hood)
        batches = (builder.build(p["gene"], p["variant"], self.background) for p in pairs)
        predictions = trainer.predict(model, batches)
        df = self.compile_predictions(pairs, predictions)
        df.to_parquet(self.output_file)
        return df

    def saturation_mutagenesis(self, gene_id, tissues, start, end, vcf_path=None, sample_name=None, zygosity=(2,)):
        """In-silico saturation mutagenesis of [start, end] (1-based, inclusive, on the gene's chromosome): every
        single-base substitution, scored as `predict` scores Variant(chrom, pos, ref, alt) for this gene, in batched
        passes that encode every distinct window once (variantformer_b200.ism).  tissues: tissue names (or one name);
        zygosity: a subset of {1 (het), 2 (hom)}.  Positions whose reference or background base is not A/C/G/T, and
        positions that touch no window, are skipped.  Writes no file.
        -> long format, one row per (pos, alt, zygosity, tissue): chrom, pos, ref, alt, genes, tissues, variant_type,
        population, sample_name, zygosity, gene_exp, ref_gene_exp, log2fc = log2((gene_exp + 1e-10) /
        (ref_gene_exp + 1e-10)) (the eqtl_scores form)."""
        from .. import ism
        from ..pipeline import HotPath
        from ..stage1 import SampleVariants
        names = [tissues] if isinstance(tissues, str) else [str(t).strip() for t in tissues]
        unknown = [t for t in names if t not in self.tissue_vocab]
        if unknown or not names:
            raise ValueError(f"unknown tissue(s) {unknown}; see tissue_vocab.yaml" if unknown else "no tissue given")
        genes = self._load_inputs(vcf_path, sample_name)
        if gene_id not in genes.index:
            raise KeyError(f"gene {gene_id!r} is not in the gene table")
        tis = [self.tissue_vocab[t] for t in names]
        gene = self._gene_spec(genes.loc[gene_id], tis)
        model, _ = self.model_manager.load_model()
        ds = self.model_config.dataset
        hot = HotPath(model.engine(), self._genome, max_length=ds.max_length, max_chunks=ds.max_chunks,
                      cre_neighbour_hood=ds.cre_neighbour_hood, gene_upstream=ds.gene_upstream_neighbour_hood,
                      gene_downstream=ds.gene_downstream_neighbour_hood)
        bg = None
        if self.background:                                   # the sample contributes SNPs only (variant_type="SNP")
            bg = SampleVariants({c: VEPBatchBuilder._snps_only(b) for c, b in self.background.items()}, "cuda")
        res = ism.saturation_mutagenesis(hot, gene, int(start), int(end), zygosity, bg)
        pred = res["pred"].cpu().numpy(); ref = res["ref_pred"].cpu().numpy()
        muts = res["plan"].mutants
        nt = len(tis)
        rep = lambda xs: np.repeat(np.asarray(xs, dtype=object), nt)
        gene_exp = pred.reshape(-1).astype(np.float64)
        ref_exp = np.tile(ref.astype(np.float64), len(muts))
        vtype = ["Gene and CRE overlap" if m.hits and m.gene_hit else "CRE overlap only" if m.hits else
                 "Gene overlap only" for m in muts]
        return pd.DataFrame({
            "chrom": [gene.chrom] * (nt * len(muts)), "pos": np.repeat([m.pos for m in muts], nt).astype(np.int64),
            "ref": rep([m.ref for m in muts]), "alt": rep([m.alt for m in muts]), "genes": [gene_id] * (nt * len(muts)),
            "tissues": names * len(muts), "variant_type": rep(vtype),
            "population": ["SAMPLE" if vcf_path else "REF_HG38"] * (nt * len(muts)),
            "sample_name": [sample_name or "hg38"] * (nt * len(muts)), "zygosity": rep([str(m.zyg) for m in muts]),
            "gene_exp": gene_exp, "ref_gene_exp": ref_exp,
            "log2fc": np.log2((gene_exp + 1e-10) / (ref_exp + 1e-10))})

    def compile_predictions(self, pairs, predictions):
        """Long format, one row per (pair, zygosity, tissue): the reference's column set (variantprocessor.py:305-320)."""
        cols = ("chrom", "pos", "ref", "alt", "genes", "tissues", "variant_type", "population", "sample_name",
                "zygosity", "gene_exp", "gene_emb", "gene_token_embedding", "cre_token_embedding")
        D = {c: [] for c in cols}
        for p, pred in zip(pairs, predictions):
            v = p["variant"]
            nt = len(v.tissue)
            empty = len(pred["pred_gene_exp"]) == 0
            for zyg, k in (("2", 2), ("1", 1), ("0", 0)):           # hom, het, ref — the reference's order
                for ti in range(nt):
                    D["chrom"].append(v.chrom); D["pos"].append(v.pos); D["ref"].append(v.ref); D["alt"].append(v.alt)
                    D["genes"].append(p["gene_id"]); D["tissues"].append(self.tissue_idx_to_name[v.tissue[ti]])
                    D["variant_type"].append(pred["variant_type"]); D["population"].append(p["population"])
                    D["sample_name"].append(p["sample_name"]); D["zygosity"].append(zyg)
                    D["gene_exp"].append(np.nan if empty else float(pred["pred_gene_exp"][k][ti, 0]))
                    for key, src in (("gene_emb", "embd"), ("gene_token_embedding", "gene_token_embedding"),
                                     ("cre_token_embedding", "cre_token_embedding")):
                        D[key].append(None if empty else pred[src][k][ti])
        return pd.DataFrame(D)

    def format_scores(self, df: pd.DataFrame):
        """Long -> wide (processors/variantprocessor.py:454-497): one row per (variant, gene, tissue) with one expression
        column per `<population>-<zygosity>-exp`; rows without a reference prediction are dropped."""
        df = df.copy()
        df["variant_id"] = df[["chrom", "pos", "ref", "alt"]].astype(str).agg("_".join, axis=1)
        df["gt-exp"] = df["population"] + "-" + df["zygosity"] + "-exp"
        df = df.rename(columns={"chrom": "chr"})
        idx = ["variant_id", "genes", "tissues", "chr", "pos", "ref", "alt", "variant_type"]
        wide = (df[idx + ["gt-exp", "gene_exp"]]
                .drop_duplicates(subset=["variant_id", "genes", "tissues", "variant_type", "gt-exp"], keep="first")
                .pivot(index=idx, columns="gt-exp", values="gene_exp").reset_index())
        wide.columns.name = None
        return wide.dropna(subset=["REF_HG38-0-exp"]).reset_index(drop=True)

    def eqtl_scores(self, df: pd.DataFrame):
        """log2 fold-change scores of the wide table (processors/variantprocessor.py:447-452 -> utils/functions.py:250-301)."""
        from ..utils.functions import generate_log2fc_score
        return generate_log2fc_score(df, self.vep_loader_config.af_path)
