"""Variant-effect (VEP) batches: the (ref, het, hom) triplet of one (variant, gene) pair, built by the stage-1 CUDA
kernels from the HBM-resident genome instead of per-item pandas copies and Python string surgery.

Semantics restated from the reference's datasets/vepdataset.py:
  * SequenceProcessor.get_iupac_code / apply_variant (:94-131): het = ONE base replaced by the IUPAC code of
    (ref, alt) — anything outside the 16 ACGT pairs (incl. multi-base alleles) is 'N'; hom = the same single base
    replaced by the ALT string (a multi-base ALT is an insertion, a multi-base REF is NOT deleted).
  * apply_variant_to_data (:347-477): the variant touches the CRE window with start_cre < pos <= end_cre (windows
    include the +-50 bp neighbourhood, pos is 1-based) and the gene window when seq_start < pos <= seq_end;
    cre_token_position = index of that CRE in batch order; gene_token_position = min(token_index // 200, 199) of the
    token covering the variant base in the strand-oriented sequence (check_if_variant_in_gene_context :479-493),
    computed separately for ref / het / hom.
  * create_batch / load_data (:563-637, :765-799): dict keys and the ref+het+hom concatenation; variant_type strings.
A background sample (VCF) contributes SNPs only, like load_gene_data_from_vcf's variant_type="SNP".
"""
from dataclasses import dataclass
from typing import List, Optional

import numpy as np
import torch

from .. import ops
from ..pipeline import GeneSpec
from ..stage1 import Genome, SampleVariants, WindowTokenizer, cre_window, gene_window

_IUPAC = {"AA": "A", "AC": "M", "CA": "M", "AG": "R", "GA": "R", "AT": "W", "TA": "W", "CC": "C", "CG": "S", "GC": "S",
          "CT": "Y", "TC": "Y", "GG": "G", "GT": "K", "TG": "K", "TT": "T"}


@dataclass
class Variant:
    chrom: str
    pos: int                # 1-based
    ref: str
    alt: str
    tissue: object = None
    gene_id: Optional[List[str]] = None
    consequence: Optional[str] = None
    label: Optional[int] = None

    def __post_init__(self):
        if not self.chrom.startswith("chr"):
            self.chrom = "chr" + self.chrom


def collate_fn(batch):
    assert len(batch) == 1, "Batch size must be 1 for VEPDataset collate function"
    return batch[0]


def get_iupac_code(ref: str, alt: str) -> str:
    return _IUPAC.get(ref + alt, "N")


def cre_windows(gene: GeneSpec, nb: int):
    """-> (order, windows): the gene's CRE rows in batch order (by start, descending on the minus strand) and their
    [w0, w1) windows."""
    order = np.argsort(gene.cre_start, kind="stable")
    order = order[::-1] if gene.strand == "-" else order
    return order, [cre_window(gene.cre_start[i], gene.cre_end[i], nb) for i in order]


def window_hits(wins, minus: bool, pos: int, g0: int, g1: int):
    """Which windows a variant at 1-based `pos` changes -> (hits, cre_hit, unreached, gene_hit).

    Overlap tests use 1-based pos against 0-based half-open windows: start < pos <= end.  The reference walks the rows
    in batch order with no break after a hit (vepdataset.py:367-407): EVERY overlapping window it reaches gets the
    variant (`hits`), cre_token_position is the LAST of them (`cre_hit`, None without a hit), and the walk stops early
    at the first row that starts past the variant (+ strand) / ends before it (- strand, rows descending).  Windows
    containing the variant that the early break never reached (`unreached`) keep their background sequence.
    `gene_hit`: g0 < pos <= g1."""
    hits = []
    for k, (a, b) in enumerate(wins):
        if (not minus and a > pos) or (minus and b < pos):
            break
        if a < pos <= b:
            hits.append(k)
    cre_hit = hits[-1] if hits else None
    unreached = [k for k, (a, b) in enumerate(wins) if a < pos <= b and k not in hits]
    return hits, cre_hit, unreached, g0 < pos <= g1


class VEPBatchBuilder:
    def __init__(self, genome: Genome, device="cuda", max_length=200, context_window=200, cre_neighbour_hood=50,
                 gene_upstream_neighbour_hood=1000, gene_downstream_neighbour_hood=300000):
        self.genome = genome
        self.tok = WindowTokenizer(device, max_length=max_length, max_chunks=context_window)
        self.max_length, self.context_window = max_length, context_window
        self.nb, self.up, self.down = cre_neighbour_hood, gene_upstream_neighbour_hood, gene_downstream_neighbour_hood
        self.device = self.tok.device

    @staticmethod
    def _with_record(background: Optional[dict], chrom, pos0, alt: bytes):
        """Sample-variant arrays for one chromosome: the background SNPs plus the query record (applied literally,
        one base replaced), the query record first among equal positions so that it wins the overlap rule."""
        if background is None or chrom not in background:
            pos, rl, gt, alts = np.zeros(0, np.int64), np.zeros(0, np.int32), np.zeros(0, np.uint8), []
        else:
            b = background[chrom]
            pos, rl, gt, alts = b["pos"], b["ref_len"], b["gt"], list(b["alt"])
        k = int(np.searchsorted(pos, pos0, "left"))
        return {chrom: dict(pos=np.insert(pos, k, pos0), ref_len=np.insert(rl, k, 1), gt=np.insert(gt, k, 2),
                            alt=alts[:k] + [alt] + alts[k:])}

    @staticmethod
    def _snps_only(b):
        keep = np.asarray([rl == 1 and len(a) == 1 for rl, a in zip(b["ref_len"], b["alt"])], bool)
        return dict(pos=np.asarray(b["pos"])[keep], ref_len=np.asarray(b["ref_len"])[keep],
                    gt=np.asarray(b["gt"])[keep], alt=[a for a, k in zip(b["alt"], keep) if k])

    def build(self, gene: GeneSpec, variant: Variant, background: Optional[dict] = None):
        """-> the reference's VEP batch dict (3 samples: ref, het, hom) with device tensors, or the empty
        "No overlap" batch.  `background` = per-chromosome variant arrays of a sample (ingest.load_vcf_sample)."""
        minus = gene.strand == "-"
        order, wins = cre_windows(gene, self.nb)
        g0, g1 = gene_window(gene.start, gene.end, gene.strand, self.up, self.down)
        _, cre_hit, unreached, gene_hit = window_hits(wins, minus, variant.pos, g0, g1)
        if cre_hit is None and not gene_hit:
            return {k: [] for k in ("cre_sequences", "cre_attention_masks", "tissue_context", "labels", "ref_labels",
                                    "gene_expression", "strand", "gene_embeddings", "gene_attention_masks")} | \
                   {"variant_type": "No overlap"}
        pos0 = variant.pos - 1
        if background:                                          # the sample contributes SNPs only (variant_type="SNP")
            background = {c: self._snps_only(b) for c, b in background.items()}
        het_alt = get_iupac_code(variant.ref, variant.alt).encode()
        samples = [SampleVariants(background, self.device) if background else None,
                   SampleVariants(self._with_record(background, variant.chrom, pos0, het_alt), self.device),
                   SampleVariants(self._with_record(background, variant.chrom, pos0, variant.alt.encode()), self.device)]
        chroms = [gene.chrom if gene.cre_chrom is None else gene.cre_chrom[i] for i in order]
        labels = torch.from_numpy(np.asarray(gene.cre_labels)[order].copy()).long()
        tissues = torch.as_tensor(variant.tissue if variant.tissue is not None else gene.tissues, dtype=torch.long)
        out = {k: [] for k in ("cre_sequences", "cre_attention_masks", "tissue_context", "labels", "ref_labels",
                               "gene_expression", "gene_embeddings", "gene_attention_masks")}
        gene_pos = []
        for sv in samples:
            seq, lens, err1 = self.tok.sequences(self.genome, chroms, [w[0] for w in wins], [w[1] for w in wins],
                                                 [int(minus)] * len(wins), sv)
            ctok, cmask, _ = self.tok.tokenize_fixed(seq, lens, seq.shape[1], typical_len=self.tok.last_max_window)
            if unreached and sv is not samples[0]:
                useq, ulens, _ = self.tok.sequences(self.genome, [chroms[k] for k in unreached],
                                                    [wins[k][0] for k in unreached], [wins[k][1] for k in unreached],
                                                    [int(minus)] * len(unreached), samples[0])
                utok, umask, _ = self.tok.tokenize_fixed(useq, ulens, useq.shape[1], typical_len=self.tok.last_max_window)
                idx = torch.as_tensor(unreached, device=self.device)
                ctok[idx] = utok; cmask[idx] = umask
            gseq, glens, err2 = self.tok.sequences(self.genome, [gene.chrom], [g0], [g1], [int(minus)], sv)
            cap = self.max_length * self.context_window
            gtok, gcnt, starts = ops.bpe_tokenize(gseq, glens, gseq.shape[1], self.tok.merges, cap, cap, want_starts=True)
            n_tok = int(gcnt[0]); glen = int(glens[0])
            if int(torch.maximum(err1, err2).item()):
                raise RuntimeError("stage-1 kernel error while building a VEP batch")
            G = min(self.context_window, (n_tok + self.max_length - 1) // self.max_length)
            ar = torch.arange(G * self.max_length, device=self.device)
            out["cre_sequences"].append(ctok.long().unsqueeze(1)); out["cre_attention_masks"].append(cmask.unsqueeze(1))
            out["gene_embeddings"].append(gtok[0, :G * self.max_length].view(G, 1, self.max_length).long())
            out["gene_attention_masks"].append((ar >= n_tok).view(G, 1, self.max_length))
            out["tissue_context"].append(tissues); out["labels"].append(torch.zeros(len(wins), dtype=torch.long))
            out["ref_labels"].append(labels); out["gene_expression"].append(torch.tensor([1.0]))
            if gene_hit:
                p = pos0 - g0                                   # offset in the forward window
                if minus:
                    p = glen - p - 1                            # check_if_variant_in_gene_context: len(seq) - pos - 1
                ch = chr(int(gseq[0, p].item())).upper()
                if ch not in "ACGTRYSWKMBDHV":                  # same error as BPEEncoder.encode_with_position (seq.py:93-97)
                    raise ValueError(f"Position {p} points to invalid character '{ch}' which is filtered out during "
                                     "normalization.")
                tok_idx = int((starts[0, :n_tok] <= p).sum().item()) - 1
                gene_pos.append(min(tok_idx // self.max_length, self.context_window - 1))
            else:
                gene_pos.append(float("nan"))
        out["strand"] = torch.tensor([[1 if minus else 0]] * 3, dtype=torch.long)
        out["cre_token_position"] = torch.tensor([[float("nan") if cre_hit is None else float(cre_hit)]] * 3)
        out["gene_token_position"] = torch.tensor([[float(x)] for x in gene_pos])
        out["variant_type"] = ("Gene and CRE overlap" if cre_hit is not None and gene_hit else
                               "CRE overlap only" if cre_hit is not None else "Gene overlap only")
        return out
