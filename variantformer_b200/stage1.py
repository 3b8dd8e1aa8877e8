"""Stage 1 host logic: device-resident genome + per-sample variant arrays -> token windows.

Replaces the per-window `samtools faidx | bcftools consensus` subprocess pairs and the
HF-tokenizers encode of datasets/vcfdataset.py:219-303 / utils/data_process.py with two
kernel launches per slab of windows (vf_encode_windows, vf_bpe_tokenize).  Window
arithmetic follows utils/data_process.py:21-24 (CRE) and :387-400 (gene).
"""
import os
from dataclasses import dataclass

import numpy as np
import torch

from . import ops

_MERGES = os.path.join(os.path.dirname(os.path.abspath(__file__)), "vocabs", "bpe500_merges.txt")
ALPHABET = "ABCDGHKMRSTVWY"     # ids 4..17 (vocabs/bpe_vocabulary_500.json)
FLAG_REVCOMP, FLAG_SNP_ONLY = 1, 2


def load_merge_table(path=_MERGES):
    """Rank-ordered merges -> (left, right, new) uint16 numpy arrays + vocab dict.  Asserts the property the
    rank-sweep kernel relies on: every operand of merge r is a base symbol or the product of a merge < r."""
    vocab = {"<pad>": 0, "<s>": 1, "</s>": 2, "<unk>": 3}
    for i, ch in enumerate(ALPHABET):
        vocab[ch] = 4 + i
    left, right, new = [], [], []
    with open(path) as f:
        for line in f:
            line = line.strip()
            if not line or line.startswith("#"):
                continue
            a, b = line.split()
            if a not in vocab or b not in vocab:
                raise ValueError(f"merge '{a} {b}' uses a token that no earlier merge creates")
            if a + b in vocab:
                raise ValueError(f"two merges create the same token '{a + b}'")
            vocab[a + b] = len(vocab)
            left.append(vocab[a]); right.append(vocab[b]); new.append(vocab[a + b])
    return np.asarray(left, np.uint16), np.asarray(right, np.uint16), np.asarray(new, np.uint16), vocab


def merge_batches(left, right, new, max_batch=16):
    """Schedule of the merge table for vf_bpe_tokenize -> (order, batch): `order` permutes the ranks, `batch` is the
    nondecreasing batch id of every permuted rank.

    Two merges whose symbol sets {left, right, new} are disjoint commute (a merge only creates adjacencies that involve
    its own new token), so any order that keeps every pair of INTERACTING ranks in its original relative order gives the
    tokens of the rank-by-rank sweeps.  Rank r gets level 1 + max(level of the earlier ranks it shares a symbol with);
    ranks of one level are pairwise disjoint and become one batch (split at max_batch), applied in one sweep with one
    barrier; a self pair (left == right) needs its detect / apply phases and is a batch of its own.
    bpe500: 482 ranks -> 87 levels -> 113 batches."""
    n = len(left)
    last, level = {}, np.zeros(n, np.int64)
    for r, syms in enumerate(zip(left.tolist(), right.tolist(), new.tolist())):
        level[r] = 1 + max(last.get(s, -1) for s in syms)
        for s in syms:
            last[s] = level[r]
    selfp = np.asarray(left) == np.asarray(right)
    order, batch, k = [], [], 0
    for lv in range(int(level.max()) + 1 if n else 0):
        idx = np.nonzero(level == lv)[0]
        plain = idx[~selfp[idx]]
        for c0 in range(0, len(plain), max_batch):
            chunk = plain[c0:c0 + max_batch]
            order += chunk.tolist(); batch += [k] * len(chunk); k += 1
        for r in idx[selfp[idx]]:
            order.append(int(r)); batch.append(k); k += 1
    return np.asarray(order, np.int64), np.asarray(batch, np.uint16)


def load_merge_table_from_hf_json(path):
    """Same table from a HuggingFace tokenizer JSON (the reference's vocabs/bpe_vocabulary_500.json)."""
    import json
    m = json.load(open(path))["model"]
    vocab = m["vocab"]
    left, right, new = [], [], []
    for a, b in (x if isinstance(x, list) else x.split() for x in m["merges"]):
        left.append(vocab[a]); right.append(vocab[b]); new.append(vocab[a + b])
    for r, (a, b, c) in enumerate(zip(left, right, new)):
        assert a < c and b < c, "merge operands must pre-exist"
    return np.asarray(left, np.uint16), np.asarray(right, np.uint16), np.asarray(new, np.uint16), vocab


@dataclass
class Genome:
    """Reference genome resident in HBM: 1 byte per base exactly as in the FASTA (soft-mask case kept)."""
    seq: torch.Tensor                 # uint8 [total]
    offsets: dict                     # chrom -> (offset, length)

    @staticmethod
    def from_arrays(chroms: dict, device="cuda"):
        off, parts, o = {}, [], 0
        for name, arr in chroms.items():
            arr = np.frombuffer(arr, np.uint8) if isinstance(arr, (bytes, bytearray)) else np.asarray(arr, np.uint8)
            off[name] = (o, len(arr)); parts.append(arr); o += len(arr)
        seq = torch.from_numpy(np.concatenate(parts)).to(device)
        return Genome(seq, off)


class SampleVariants:
    """One sample's variants: per chromosome sorted by position (0-based), one ALT allele per record.
    gt: 0 = hom-ref/missing, 1 = het, 2 = hom-alt.  Symbolic ALTs (<...>) must be dropped by the loader
    (the reference's `-e 'ALT~"<.*>"'`)."""

    def __init__(self, per_chrom: dict, device="cuda"):
        self.ranges, self.host_pos = {}, {}
        # host copies of the rest of each record (variant attribution names a sample's own records by them)
        self.host_ref_len, self.host_alt, self.host_gt = {}, {}, {}
        pos, rl, ao, al, gt, pool = [], [], [], [], [], []
        n = 0; pool_len = 0
        for chrom, v in per_chrom.items():
            p = np.asarray(v["pos"], np.int64)
            assert (np.diff(p) >= 0).all(), "variants must be sorted by position"
            alts = [a.encode() if isinstance(a, str) else bytes(a) for a in v["alt"]]
            lens = np.asarray([len(a) for a in alts], np.int32)
            pos.append(p.astype(np.int32)); rl.append(np.asarray(v["ref_len"], np.int32)); al.append(lens)
            ao.append((np.cumsum(lens) - lens + pool_len).astype(np.int32)); gt.append(np.asarray(v["gt"], np.uint8))
            pool.append(np.frombuffer(b"".join(alts), np.uint8)); pool_len += int(lens.sum())
            self.ranges[chrom] = (n, n + len(p)); self.host_pos[chrom] = p; n += len(p)
            self.host_ref_len[chrom] = rl[-1].astype(np.int64); self.host_alt[chrom] = alts
            self.host_gt[chrom] = gt[-1].copy()

        def cat(xs, dt):
            return torch.from_numpy(np.concatenate(xs).astype(dt) if xs else np.zeros(0, dt)).to(device)
        self.dev = dict(pos=cat(pos, np.int32), ref_len=cat(rl, np.int32), alt_off=cat(ao, np.int32),
                        alt_len=cat(al, np.int32), gt=cat(gt, np.uint8), alt_pool=cat(pool or [np.zeros(0, np.uint8)], np.uint8))
        for k, t in self.dev.items():          # kernels never dereference empty arrays, but need non-NULL
            if t.numel() == 0:
                self.dev[k] = torch.zeros(1, dtype=t.dtype, device=device)

    def window_range(self, chrom, w0, w1):
        if chrom not in self.ranges:
            return 0, 0
        base = self.ranges[chrom][0]
        p = self.host_pos[chrom]
        return base + int(np.searchsorted(p, w0, "left")), base + int(np.searchsorted(p, w1, "left"))


INT32_LIMIT = 2 ** 31 - 1


class CohortVariants:
    """Many samples' variants in one device table: every sample's records concatenated sample-major, then by chromosome,
    then by position, in the six arrays of SampleVariants.dev.  A row (window, sample) of vf_encode_windows points at its
    sample's records through var_lo / var_hi (window_ranges), so one encode batch may mix samples.  The kernels index
    records and ALT bytes with int32: a table past 2^31 of either is refused (split the samples: `blocks`)."""

    def __init__(self, names, per_sample, device="cuda"):
        self.names = list(names)
        assert len(self.names) == len(per_sample)
        self.chroms = list(dict.fromkeys(c for d in per_sample for c in d))
        self.chrom_idx = {c: i for i, c in enumerate(self.chroms)}
        n_rec, n_alt = self.sizes(per_sample)
        if n_rec > INT32_LIMIT or n_alt > INT32_LIMIT:
            raise ValueError(f"{n_rec} records / {n_alt} ALT bytes do not fit int32 indices: split the samples "
                             "(CohortVariants.blocks)")
        keys, pos, rl, al, gt, alts = [], [], [], [], [], []
        nc = len(self.chroms)
        self.n_records = np.zeros(len(self.names), np.int64)
        for s, d in enumerate(per_sample):
            for c in self.chroms:
                if c not in d:
                    continue
                v = d[c]
                p = np.asarray(v["pos"], np.int64)
                assert (np.diff(p) >= 0).all(), "variants must be sorted by position"
                keys.append((s * nc + self.chrom_idx[c]) * (1 << 32) + p)
                pos.append(p.astype(np.int32)); rl.append(np.asarray(v["ref_len"], np.int32))
                gt.append(np.asarray(v["gt"], np.uint8))
                a = [x.encode() if isinstance(x, str) else bytes(x) for x in v["alt"]]
                al.append(np.asarray([len(x) for x in a], np.int32)); alts += a
                self.n_records[s] += len(p)
        cat = lambda xs, dt: np.concatenate(xs).astype(dt) if xs else np.zeros(0, dt)
        self.key = cat(keys, np.int64)               # (segment << 32) + pos: sorted, one segment per (sample, chrom)
        lens = cat(al, np.int32)
        off = (np.cumsum(lens, dtype=np.int64) - lens).astype(np.int32)
        pool = np.frombuffer(b"".join(alts), np.uint8).copy() if alts else np.zeros(0, np.uint8)
        up = lambda a, dt: torch.from_numpy(np.ascontiguousarray(a, dt) if len(a) else np.zeros(1, dt)).to(device)
        self.dev = dict(pos=up(cat(pos, np.int32), np.int32), ref_len=up(cat(rl, np.int32), np.int32),
                        alt_off=up(off, np.int32), alt_len=up(lens, np.int32), gt=up(cat(gt, np.uint8), np.uint8),
                        alt_pool=up(pool, np.uint8))

    @staticmethod
    def sizes(per_sample):
        """(records, ALT bytes) of a list of per-sample dicts."""
        n_rec = sum(len(v["pos"]) for d in per_sample for v in d.values())
        n_alt = sum(len(a) for d in per_sample for v in d.values() for a in v["alt"])
        return n_rec, n_alt

    @staticmethod
    def blocks(per_sample, limit=None):
        """Consecutive sample ranges [a, b) whose tables fit int32 indices (records and ALT bytes <= limit; a single
        sample past it stays alone, and CohortVariants refuses it as SampleVariants' int32 arrays cannot hold it)."""
        limit = INT32_LIMIT if limit is None else limit
        out, a = [], 0
        while a < len(per_sample):
            b, rec, alt = a, 0, 0
            while b < len(per_sample):
                r, x = CohortVariants.sizes([per_sample[b]])
                if b > a and (rec + r > limit or alt + x > limit):
                    break
                rec += r; alt += x; b += 1
            out.append((a, b))
            a = b
        return out

    def window_ranges(self, sample_idx, chroms, w0, w1):
        """Vectorised var_lo / var_hi (int64 numpy) of rows (sample_idx[i], chroms[i], [w0[i], w1[i])) into the
        concatenated arrays: the records of that sample and chromosome with pos in [w0, w1)."""
        s = np.asarray(sample_idx, np.int64)
        names, inv = np.unique(np.asarray(chroms, dtype=object).astype(str), return_inverse=True)
        c = np.asarray([self.chrom_idx.get(x, -1) for x in names], np.int64)[inv.reshape(-1)]
        seg = (s * len(self.chroms) + np.maximum(c, 0)) * (1 << 32)
        lo = np.searchsorted(self.key, seg + np.asarray(w0, np.int64), "left")
        hi = np.searchsorted(self.key, seg + np.asarray(w1, np.int64), "left")
        hi = np.where(c < 0, lo, hi)                 # a chromosome no sample has a record on
        return lo, hi


def cre_window(start, end, nb):
    return max(0, int(start) - nb), int(end) + nb


def gene_window(start, end, strand, up, down):
    start, end = int(start), int(end)
    if strand == "-":
        return max(start, end - down), end + up
    s = max(0, start - up)
    return s, min(end, s + down)


class WindowTokenizer:
    """windows (+ optional sample variants) -> mutated sequence bytes -> BPE tokens, all on the device."""

    def __init__(self, device="cuda", merges_path=None, max_length=200, max_chunks=200):
        a, b, c, self.vocab = (load_merge_table() if merges_path is None else
                               (load_merge_table_from_hf_json(merges_path) if merges_path.endswith(".json")
                                else load_merge_table(merges_path)))
        self.device = torch.device(device)
        order, batch = merge_batches(a, b, c)
        a, b, c = a[order], b[order], c[order]               # the kernel walks the table in this (equivalent) order
        self.merges = tuple(torch.from_numpy(np.ascontiguousarray(x).view(np.int16)).to(self.device) for x in (a, b, c, batch))
        self.max_length, self.max_chunks = max_length, max_chunks
        self._no_var = SampleVariants({}, device=self.device)

    def sequences(self, genome: Genome, chroms, w0, w1, revcomp, variants: SampleVariants = None, snp_only=False,
                  max_insert=4096):
        """-> (uint8 [n, pitch] device, int32 lens device, err flag tensor)."""
        v = variants or self._no_var
        n = len(w0)
        w0 = np.asarray(w0, np.int64); w1 = np.asarray(w1, np.int64)
        base = np.asarray([genome.offsets[c][0] for c in chroms], np.int64)
        for c, b1 in zip(chroms, w1):
            assert b1 <= genome.offsets[c][1], "window runs past the end of the chromosome"
        lo_hi = [v.window_range(c, a, b) for c, a, b in zip(chroms, w0, w1)]
        flags = (np.asarray(revcomp, np.uint8) * FLAG_REVCOMP) | (FLAG_SNP_ONLY if snp_only else 0)
        max_window = int((w1 - w0).max())
        pitch = ((max_window + (max_insert if variants is not None else 0) + 15) // 16) * 16
        t = lambda x, dt: torch.from_numpy(np.ascontiguousarray(x, dt)).to(self.device, non_blocking=True)
        out, out_len, err = ops.encode_windows(
            genome.seq, t(base, np.int64), t(w0, np.int32), t(w1, np.int32), t([x[0] for x in lo_hi], np.int32),
            t([x[1] for x in lo_hi], np.int32), t(flags, np.uint8), v.dev, max_window, pitch)
        self.last_max_window = max_window          # reference span of the longest window (block-size hint)
        return out, out_len, err

    def tokenize_fixed(self, seq, lens, max_len, typical_len=None):
        """CRE windows: pad/truncate to max_length (vcfdataset.py:198-217).  -> tokens int32 [n, L], mask bool."""
        tok, cnt = ops.bpe_tokenize(seq, lens, max_len, self.merges, self.max_length, self.max_length,
                                    typical_len=typical_len)
        ar = torch.arange(self.max_length, device=self.device)[None, :]
        return tok, ar >= cnt.clamp(max=self.max_length)[:, None], cnt

    def tokenize_chunked(self, seq, lens, max_len):
        """Gene windows: consecutive max_length-token chunks, <= max_chunks (vcfdataset.py:338-394).
        -> list of (tokens int32 [G_i, L], mask bool [G_i, L]) per window."""
        cap = self.max_length * self.max_chunks
        tok, cnt = ops.bpe_tokenize(seq, lens, max_len, self.merges, cap, cap)
        cnt_h = cnt.cpu().numpy()
        out = []
        ar = torch.arange(cap, device=self.device)
        for i, c in enumerate(cnt_h):
            g = int(min(self.max_chunks, (int(c) + self.max_length - 1) // self.max_length))
            t = tok[i, : g * self.max_length].view(g, self.max_length)
            m = (ar[: g * self.max_length] >= int(c)).view(g, self.max_length)
            out.append((t, m))
        return out, cnt_h
