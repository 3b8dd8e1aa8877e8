"""HotPath — the batched four-stage pipeline as one call: window tables (host) -> genotype encoding + BPE
(device) -> seq2reg -> seq2gene -> head -> (expression, embeddings).  This is what VCFProcessor / bench.py drive
for slabs of genes; per-item access with the reference's tuple layout lives in datasets/vcfdataset.py."""
from dataclasses import dataclass, field

import os
import numpy as np
import torch

from .engine import Engine
from .stage1 import Genome, SampleVariants, WindowTokenizer, cre_window, gene_window


@dataclass
class GeneSpec:
    """One query row: gene coordinates, its CRE table and the tissues to predict."""
    chrom: str
    start: int
    end: int
    strand: str
    cre_start: np.ndarray
    cre_end: np.ndarray
    cre_labels: np.ndarray              # ids into utils.constants.REF_CREs
    tissues: list
    cre_chrom: list = field(default=None)


class HotPath:
    def __init__(self, engine: Engine, genome: Genome, max_length=200, max_chunks=200, cre_neighbour_hood=50,
                 gene_upstream=1000, gene_downstream=300000):
        self.engine, self.genome = engine, genome
        self.tok = WindowTokenizer(engine.device, max_length=max_length, max_chunks=max_chunks)
        self.nb, self.up, self.down = cre_neighbour_hood, gene_upstream, gene_downstream
        self.max_length, self.max_chunks = max_length, max_chunks

    def tokenize(self, genes, variants: SampleVariants = None):
        """Stage 1 for a slab of genes: two kernel launches for all CRE windows, two for all gene windows.
        -> per-gene lists of device tensors (tokens int32 [n, L], masks bool [n, L]) + host token counts."""
        dev = self.engine.device
        chroms, w0, w1, rc, owner = [], [], [], [], []
        for gi, g in enumerate(genes):
            minus = g.strand == "-"
            order = np.argsort(g.cre_start, kind="stable")
            if minus:
                order = order[::-1]                       # vcfdataset.py:243-246
            for i in order:
                a0, a1 = cre_window(g.cre_start[i], g.cre_end[i], self.nb)
                chroms.append(g.chrom if g.cre_chrom is None else g.cre_chrom[i])
                w0.append(a0); w1.append(a1); rc.append(int(minus)); owner.append(gi)
        seq, lens, err1 = self.tok.sequences(self.genome, chroms, w0, w1, rc, variants)
        ctok, cmask, ccnt = self.tok.tokenize_fixed(seq, lens, seq.shape[1], typical_len=self.tok.last_max_window)
        gw = [gene_window(g.start, g.end, g.strand, self.up, self.down) for g in genes]
        gseq, glens, err2 = self.tok.sequences(self.genome, [g.chrom for g in genes], [x[0] for x in gw],
                                               [x[1] for x in gw], [int(g.strand == "-") for g in genes], variants)
        chunks, gcnt = self.tok.tokenize_chunked(gseq, glens, gseq.shape[1])      # (one small D2H of the counts)
        errs = torch.maximum(err1, err2)
        C = np.bincount(np.asarray(owner), minlength=len(genes))
        off = np.concatenate([[0], np.cumsum(C)])
        ccnt_h = np.minimum(ccnt.cpu().numpy(), self.max_length).astype(np.int64)
        cre_tok = [ctok[off[i]:off[i + 1]] for i in range(len(genes))]
        cre_msk = [cmask[off[i]:off[i + 1]] for i in range(len(genes))]
        gene_tok = [c[0] for c in chunks]; gene_msk = [c[1] for c in chunks]
        glen_h = np.concatenate([np.minimum(self.max_length, np.maximum(
            0, min(int(n), self.max_length * self.max_chunks) - self.max_length * np.arange(t.shape[0])))
            for n, t in zip(gcnt, gene_tok)]).astype(np.int64)
        labels = []
        for g in genes:
            order = np.argsort(g.cre_start, kind="stable")
            labels.append(torch.from_numpy(np.asarray(g.cre_labels)[order[::-1] if g.strand == "-" else order].copy()))
        return dict(cre_tok=cre_tok, cre_msk=cre_msk, gene_tok=gene_tok, gene_msk=gene_msk, labels=labels,
                    lens=(ccnt_h, glen_h), err=errs, cre_seq=(seq, lens), gene_seq=(gseq, glens), gene_count=gcnt)

    def prepare(self, genes, variants: SampleVariants = None):
        """Stage 1 + all host bookkeeping for one slab -> a prepared slab for Engine.run."""
        t = self.tokenize(genes, variants)
        tissues = [torch.as_tensor(g.tissues, dtype=torch.long) for g in genes]
        slab = self.engine.prepare(t["cre_tok"], t["cre_msk"], t["gene_tok"], t["gene_msk"], tissues, t["labels"],
                                   lens=t["lens"])
        slab["err"] = t["err"]
        return slab

    def predict_pipelined(self, slabs, variants: SampleVariants = None, to_host=True):
        """Generator over an iterable of gene lists: while the model (stages 2-4) of slab i runs on the current
        stream, stage 1 and the host bookkeeping of slab i+1 run on a side stream, so their device->host count reads
        and host work no longer leave the GPU idle between slabs.  Yields (pred, emb[, err]) per slab in order."""
        main = torch.cuda.current_stream(self.engine.device)
        if not hasattr(self, "_side"):
            self._side = torch.cuda.Stream(self.engine.device)
        # VF_STAGE1_STREAM=main: no side stream (timing experiments: what the overlap is worth)
        side = main if os.environ.get("VF_STAGE1_STREAM") == "main" else self._side
        side.wait_stream(main)                          # genome / variants / merge tables were uploaded on `main`

        def stage(genes):
            with torch.cuda.stream(side):
                slab = self.prepare(genes, variants)
                ev = torch.cuda.Event(); ev.record(side)
            for v in slab.values():                     # tensors born on the side stream are consumed on `main`
                for x in (v if isinstance(v, (list, tuple)) else [v]):
                    if torch.is_tensor(x) and x.is_cuda:
                        x.record_stream(main)
                    elif hasattr(x, "device_tensors"):
                        for t in x.device_tensors():
                            t.record_stream(main)
            return slab, ev

        it = iter(slabs)
        try:
            nxt = stage(next(it))
        except StopIteration:
            return
        while nxt is not None:
            slab, ev = nxt
            main.wait_event(ev)
            out = self.engine.run(slab)                 # asynchronous launches on `main`
            try:
                nxt = stage(next(it))                   # overlaps with the launches above
            except StopIteration:
                nxt = None
            if to_host:
                pred, emb = out["pred"].cpu().numpy(), out["emb"].cpu().numpy()
                self._raise_on_stage1_error(slab["err"])
                yield pred, emb
            else:
                yield out["pred"], out["emb"], slab["err"]

    def predict_to_parquet(self, slabs, variants: SampleVariants, writer, sample="sample", gene_ids=None, start=0):
        """The production loop (SURVEY 8f rank 3): every slab of `slabs` (an iterable of gene lists) through the
        pipelined path; results leave the device by an asynchronous copy into pinned, double-buffered host memory on a
        copy stream and are written as one Parquet file per slab by `writer` (variantformer_b200.writer.ResultWriter)
        in the background while the next slab computes.  Slabs whose file already exists are skipped, so an interrupted
        run resumes (`start` = index of the first slab of the iterable).  gene_ids: optional callable
        (slab index, position) -> gene id string.  -> number of slabs computed in this call."""
        from .writer import PinnedRing
        dev = self.engine.device
        done = writer.done()
        slabs = list(slabs)
        todo = [(start + i, g) for i, g in enumerate(slabs) if start + i not in done]
        if not todo:
            return 0
        main = torch.cuda.current_stream(dev)
        if not hasattr(self, "_copy"):
            self._copy, self._ring = torch.cuda.Stream(dev), PinnedRing()
        pending = None                                   # (event, slab index, genes, buffer, n, err tensor)

        def flush(p):
            ev, idx, genes, buf, n, err = p
            ev.synchronize()
            self._raise_on_stage1_error(err)
            D = self.engine.w.D
            rows, item = [], 0
            for k, g in enumerate(genes):
                gid = gene_ids(idx, k) if gene_ids is not None else f"{g.chrom}:{g.start}-{g.end}"
                rows += [(item, sample, gid, int(t)) for t in g.tissues]
                item += 1
            writer.submit(idx, rows, buf["pred"][:n].numpy(), buf["emb"][:n * D].view(n, D).numpy(),
                          release=lambda b=buf: self._ring.release(b))
        for (idx, genes), (pred, emb, err) in zip(todo, self.predict_pipelined((g for _, g in todo), variants, to_host=False)):
            n, D = pred.shape[0], emb.shape[1]
            buf = self._ring.acquire(n, D)               # blocks only if both buffers are still being written out
            self._copy.wait_stream(main)
            with torch.cuda.stream(self._copy):
                buf["pred"][:n].copy_(pred, non_blocking=True)
                buf["emb"][:n * D].view(n, D).copy_(emb, non_blocking=True)
                ev = torch.cuda.Event(); ev.record(self._copy)
            pred.record_stream(self._copy); emb.record_stream(self._copy)
            if pending is not None:
                flush(pending)                           # slab i-1 goes to the writer while slab i computes
            pending = (ev, idx, genes, buf, n, err)
        if pending is not None:
            flush(pending)
        writer.flush()                                   # when this returns, every slab of the call is on disk
        return len(todo)

    def predict(self, genes, variants: SampleVariants = None, to_host=True):
        """-> (pred [sum T], emb [sum T, D]) as numpy (to_host) or device tensors."""
        t = self.tokenize(genes, variants)
        tissues = [torch.as_tensor(g.tissues, dtype=torch.long) for g in genes]
        slab = self.engine.prepare(t["cre_tok"], t["cre_msk"], t["gene_tok"], t["gene_msk"], tissues, t["labels"],
                                   lens=t["lens"])
        out = self.engine.run(slab)
        if not to_host:
            return out["pred"], out["emb"], t["err"]
        pred = out["pred"].cpu().numpy(); emb = out["emb"].cpu().numpy()
        self._raise_on_stage1_error(t["err"])
        return pred, emb

    @staticmethod
    def _raise_on_stage1_error(err):
        """The encode kernel flags windows it could not build (their tokens are then all padding): never hand out
        predictions computed from them."""
        code = int(err.item())
        if code:
            raise RuntimeError(f"stage-1 kernel reported error {code} (1: pitch overflow, 2: >2048 variants/window)")
