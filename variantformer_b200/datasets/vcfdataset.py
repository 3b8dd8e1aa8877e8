"""VCFDataset — per-gene items (CRE windows + gene window -> tokens/masks/labels) behind the reference's
constructor and item/collate layout (datasets/vcfdataset.py:73-121, :305-336, :18-63), produced by the stage-1
CUDA kernels from a genome and variant set resident in HBM instead of per-window subprocesses."""
import os

import numpy as np
import pandas as pd
import torch
import yaml
from torch.utils.data import Dataset

from .. import ingest
from ..stage1 import Genome, SampleVariants, WindowTokenizer, cre_window, gene_window
from ..utils.config import VOCAB_DIR
from ..utils.constants import MAP_REF_CRE_TO_IDX, PAD_TOKEN_ID

_GENOMES, _SAMPLES = {}, {}          # (path, device) -> device-resident data, shared by datasets


def collate_fn_batching(batch):
    """Same dict as the reference's collate (vcfdataset.py:18-63)."""
    keys = ("cre_sequences", "cre_attention_masks", "tissue_context", "cre_labels", "ref_cre_labels", "strand",
            "gene_embeddings", "gene_attention_masks")
    cols = list(zip(*batch))
    D = {k: list(v) for k, v in zip(keys, cols)}
    D["strand_val"] = torch.cat([s.unsqueeze(0) for s in D.pop("strand")], dim=0)
    return D


class LocalGeneManifest:
    """`get_file_path(gene_id)` over a directory of per-gene CRE manifests (<dir>/<gene_id>.csv with columns
    chromosome,start_cre,end_cre,cre_name) — the offline stand-in for utils/assets.py::GeneManifestLookup (S3)."""

    def __init__(self, directory):
        self.directory = directory

    def get_file_path(self, gene_id):
        return os.path.join(self.directory, f"{gene_id}.csv")


class VCFDataset(Dataset):
    def __init__(self, max_length: int, max_chunks: int, cre_neighbour_hood: int, gencode_v24: str,
                 gene_cre_manifest, gene_upstream_neighbour_hood: int, gene_downstream_neighbour_hood: int,
                 query_df: pd.DataFrame, fasta_path: str, vcf_path: str = None, device="cuda"):
        self.max_length, self.max_chunks = max_length, max_chunks
        self.cre_neighbour_hood = cre_neighbour_hood
        self.gene_upstream_neighbour_hood = gene_upstream_neighbour_hood
        self.gene_downstream_neighbour_hood = gene_downstream_neighbour_hood
        self.query_df = query_df
        self.gene_cre_manifest = gene_cre_manifest
        self.fasta_path, self.vcf_path = fasta_path, vcf_path
        self.device = torch.device(device)
        self.pad_token_id = PAD_TOKEN_ID
        self.ref_cre_to_idx = MAP_REF_CRE_TO_IDX
        self.gencode_v24 = gencode_v24 if isinstance(gencode_v24, pd.DataFrame) else pd.read_csv(gencode_v24)
        with open(os.path.join(VOCAB_DIR, "tissue_vocab.yaml")) as f:
            self.tissue_vocab = yaml.safe_load(f)
        self.tokenizer = WindowTokenizer(self.device, max_length=max_length, max_chunks=max_chunks)
        self._check_filter_query_df()

    # -- query validation: same rules and messages as vcfdataset.py:123-169 --------------------------------------
    def _check_filter_query_df(self):
        assert self.query_df is not None, "Query dataframe is not provided"
        assert "gene_id" in self.query_df.columns, "Query dataframe must contain gene_id column"
        assert "tissues" in self.query_df.columns, "Query dataframe must contain tissues column"
        n0, rows = len(self.query_df), []
        known = set(self.gencode_v24["gene_id"].values)
        for _, row in self.query_df.iterrows():
            gene_id = row["gene_id"]
            if gene_id not in known:
                print(f"Gene {gene_id} not found in the training set so skipping it")
                continue
            T, names = [], []
            for tissue in row["tissues"].split(","):
                if tissue in self.tissue_vocab:
                    T.append(self.tissue_vocab[tissue]); names.append(tissue)
                else:
                    print(f"Tissue {tissue} not found in the tissue vocab so skipping it")
            if not T:
                print(f"No tissues found for gene {gene_id}")
                continue
            rec = {"gene_id": gene_id, "tissues": T, "tissue_names": names}
            if "vcf_path" in self.query_df.columns:
                rec["vcf_path"] = row["vcf_path"]
            rows.append(rec)
        if not rows:
            raise ValueError("No genes found in the query df that are present in the gencode v24 and have at least "
                             "one tissue in the training set of VariantFormer")
        self.query_df = pd.DataFrame(rows)
        print(f"Filtered query df to {len(self.query_df)} genes reducing from {n0}")
        return True

    def __len__(self):
        return len(self.query_df)

    def __getitem__(self, idx):
        return self._load_file(idx)

    # -- device-resident inputs ------------------------------------------------------------------------------------
    def _genome(self) -> Genome:
        key = (self.fasta_path, str(self.device))
        if key not in _GENOMES:
            _GENOMES[key] = Genome.from_arrays(ingest.load_fasta(self.fasta_path), self.device)
        return _GENOMES[key]

    def _variants(self, vcf_path):
        if not vcf_path:
            return None
        key = (vcf_path, str(self.device))
        if key not in _SAMPLES:
            _SAMPLES[key] = SampleVariants(ingest.load_vcf_sample(vcf_path), self.device)
        return _SAMPLES[key]

    def _get_gene_info(self, gene_id: str) -> dict:
        return self.gencode_v24[self.gencode_v24["gene_id"] == gene_id].iloc[0].to_dict()

    def cre_manifest(self, gene_id, gene_info=None):
        """The gene's CRE manifest (chromosome, start_cre, end_cre, cre_name) and its batch order: manifest row of the
        k-th CRE window of the item (sorted by start, reversed for '-' genes)."""
        gene_info = gene_info or self._get_gene_info(gene_id)
        m = pd.read_csv(self.gene_cre_manifest.get_file_path(gene_id))
        w = [cre_window(s, e, self.cre_neighbour_hood) for s, e in zip(m["start_cre"], m["end_cre"])]
        order = np.argsort(np.asarray([x[0] for x in w]), kind="stable")      # process_subject sorts by start_cre
        if gene_info["strand"] == "-":
            order = order[::-1]
        return m, order

    def _get_cres(self, gene_id, gene_info, vcf_path):
        """vcfdataset.py:219-283: CRE windows [start-50, end+50) sorted by start, reversed + reverse-complemented for
        '-' genes, tokenised, padded/truncated to max_length."""
        m, order = self.cre_manifest(gene_id, gene_info)
        m = m.rename(columns={"chromosome": "chrom", "start_cre": "start", "end_cre": "end", "cre_name": "cCRE"})
        w = [cre_window(s, e, self.cre_neighbour_hood) for s, e in zip(m["start"], m["end"])]
        minus = gene_info["strand"] == "-"
        chroms = [m["chrom"].iloc[i] for i in order]
        w0 = [w[i][0] for i in order]; w1 = [w[i][1] for i in order]
        seq, lens, err = self.tokenizer.sequences(self._genome(), chroms, w0, w1, [int(minus)] * len(order),
                                                  self._variants(vcf_path))
        tok, mask, _ = self.tokenizer.tokenize_fixed(seq, lens, seq.shape[1], typical_len=self.tokenizer.last_max_window)
        self._check(err)
        labels = torch.tensor([self.ref_cre_to_idx[m["cCRE"].iloc[i]] for i in order], dtype=torch.long)
        return tok.long().unsqueeze(1), mask.unsqueeze(1), labels, torch.zeros(len(order), dtype=torch.long)

    def _get_gene(self, gene_id, gene_info, vcf_path):
        """vcfdataset.py:285-303 + chunkify_data :338-394."""
        minus = gene_info["strand"] == "-"
        a0, a1 = gene_window(gene_info["start"], gene_info["end"], gene_info["strand"],
                             self.gene_upstream_neighbour_hood, self.gene_downstream_neighbour_hood)
        seq, lens, err = self.tokenizer.sequences(self._genome(), [gene_info["chromosome"]], [a0], [a1], [int(minus)],
                                                  self._variants(vcf_path))
        assert int(lens[0]) > 1000, f"Mutated sequence is less than 1000bp for gene {gene_id}"
        chunks, _ = self.tokenizer.tokenize_chunked(seq, lens, seq.shape[1])
        self._check(err)
        tok, mask = chunks[0]
        return tok.long().unsqueeze(1), mask.unsqueeze(1)

    @staticmethod
    def _check(err):
        code = int(err.item())
        if code:
            raise RuntimeError({1: "encoded window exceeds the output pitch (too many inserted bases)",
                                2: "more than 2048 applied variants in one window"}.get(code, f"stage-1 error {code}"))

    def _load_file(self, idx: int) -> tuple:
        row = self.query_df.iloc[idx]
        vcf_path = row["vcf_path"] if "vcf_path" in self.query_df.columns else self.vcf_path
        gene_info = self._get_gene_info(row["gene_id"])
        assert gene_info["chromosome"] in ["chr" + str(i) for i in range(1, 23)], \
            f"Chromosome {gene_info['chromosome']} is not a valid chromosome. Sex chromosomes are not supported"
        X, mask, ref_labels, labels = self._get_cres(row["gene_id"], gene_info, vcf_path)
        gene_tok, gene_mask = self._get_gene(row["gene_id"], gene_info, vcf_path)
        strand = torch.tensor([0] if gene_info["strand"] == "+" else [1], dtype=torch.long)
        return (X, mask, torch.tensor(row["tissues"], dtype=torch.long), labels, ref_labels, strand, gene_tok, gene_mask)
