"""Host ingest for stage 1: FASTA -> byte arrays, one sample (or many, in one pass) of a VCF -> sorted variant arrays
(SURVEY §8f rank 1).

Replaces what `samtools faidx` / `bcftools consensus` (htslib) read from disk per window
(utils/data_process.py:27,40-59,404,416-435) with ONE pass per genome / per sample through libvf_ingest.so
(csrc/vf_ingest.cpp: C++17, zlib, parallel BGZF inflation and line parsing; C ABI in include/vf_ingest.h).  The parsed
arrays are what stage1.Genome / stage1.SampleVariants upload to HBM.  There is no Python fallback: the pure-Python
restatement of the same semantics lives in oracle/ingest_py.py and is test infrastructure.
"""
import ctypes as C
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.path.join(_HERE, "csrc", "libvf_ingest.so")
_vp, _i32, _i64 = C.c_void_p, C.c_int, C.c_int64

# name -> (argtypes, restype): every symbol include/vf_ingest.h declares
SIGNATURES = {
    "vf_ingest_last_error": ([], C.c_char_p),
    "vf_fasta_open": ([C.c_char_p, _i32], _vp),
    "vf_fasta_num_seqs": ([_vp], _i32),
    "vf_fasta_name": ([_vp, _i32], C.c_char_p),
    "vf_fasta_length": ([_vp, _i32], _i64),
    "vf_fasta_copy": ([_vp, _i32, _vp, _i64], _i64),
    "vf_fasta_close": ([_vp], None),
    "vf_vcf_open": ([C.c_char_p, C.c_char_p, _i32], _vp),
    "vf_vcf_num_chroms": ([_vp], _i32),
    "vf_vcf_chrom": ([_vp, _i32], C.c_char_p),
    "vf_vcf_num_records": ([_vp, _i32], _i64),
    "vf_vcf_alt_bytes": ([_vp, _i32], _i64),
    "vf_vcf_copy": ([_vp, _i32, _vp, _vp, _vp, _vp, _vp, _vp], _i32),
    "vf_vcf_close": ([_vp], None),
    "vf_vcf_open_cohort": ([C.c_char_p, _vp, _i32, C.c_char_p, _i32], _vp),
    "vf_vcf_cohort_num_samples": ([_vp], _i32),
    "vf_vcf_cohort_sample_name": ([_vp, _i32], C.c_char_p),
    "vf_vcf_cohort_num_chroms": ([_vp], _i32),
    "vf_vcf_cohort_chrom": ([_vp, _i32], C.c_char_p),
    "vf_vcf_cohort_num_records": ([_vp, _i32, _i32], _i64),
    "vf_vcf_cohort_alt_bytes": ([_vp, _i32, _i32], _i64),
    "vf_vcf_cohort_copy": ([_vp, _i32, _i32, _vp, _vp, _vp, _vp, _vp, _vp], _i32),
    "vf_vcf_cohort_close": ([_vp], None),
}
_lib = None


class IngestError(RuntimeError):
    pass


def lib():
    global _lib
    if _lib is None:
        if not os.path.exists(LIB_PATH):
            raise IngestError(f"{LIB_PATH} not found: build it with `python -m variantformer_b200.csrc.build`")
        l = C.CDLL(LIB_PATH)
        for name, (args, res) in SIGNATURES.items():
            fn = getattr(l, name)
            fn.argtypes = args
            fn.restype = res
        _lib = l
    return _lib


def _fail(what):
    raise IngestError(f"{what}: {lib().vf_ingest_last_error().decode()}")


def load_fasta(path, chroms=None, threads=0):
    """-> {name: uint8 array} with the FASTA's own case (soft-masking) preserved."""
    l = lib()
    h = l.vf_fasta_open(os.fsencode(path), threads)
    if not h:
        _fail("vf_fasta_open")
    try:
        out = {}
        for i in range(l.vf_fasta_num_seqs(h)):
            name = l.vf_fasta_name(h, i).decode()
            if chroms is not None and name not in chroms:
                continue
            a = np.empty(l.vf_fasta_length(h, i), np.uint8)
            if l.vf_fasta_copy(h, i, a.ctypes.data, a.size) != a.size:
                _fail("vf_fasta_copy")
            out[name] = a
        return out
    finally:
        l.vf_fasta_close(h)


def _copy_records(n, nb, copy, what):
    """Arrays of one chromosome through a vf_vcf_copy-shaped call -> dict(pos, ref_len, gt, alt [bytes])."""
    pos = np.empty(n, np.int64); ref_len = np.empty(n, np.int32); off = np.empty(n, np.int32)
    ln = np.empty(n, np.int32); gt = np.empty(n, np.uint8); pool = np.empty(nb, np.uint8)
    if copy(pos.ctypes.data, ref_len.ctypes.data, off.ctypes.data, ln.ctypes.data, gt.ctypes.data, pool.ctypes.data) != 0:
        _fail(what)
    pb = pool.tobytes()
    return dict(pos=pos, ref_len=ref_len, gt=gt, alt=[pb[o:o + k] for o, k in zip(off.tolist(), ln.tolist())])


def load_vcf_sample(path, sample=None, chroms=None, threads=0):
    """One sample's genotypes -> {chrom: dict(pos int64 0-based, ref_len int32, alt [bytes], gt uint8)}, sorted by
    position (semantics: include/vf_ingest.h)."""
    l = lib()
    h = l.vf_vcf_open(os.fsencode(path), None if sample is None else sample.encode(), threads)
    if not h:
        _fail("vf_vcf_open")
    try:
        per = {}
        for c in range(l.vf_vcf_num_chroms(h)):
            name = l.vf_vcf_chrom(h, c).decode()
            if chroms is not None and name not in chroms:
                continue
            per[name] = _copy_records(l.vf_vcf_num_records(h, c), l.vf_vcf_alt_bytes(h, c),
                                      lambda *a: l.vf_vcf_copy(h, c, *a), "vf_vcf_copy")
        return per
    finally:
        l.vf_vcf_close(h)


def regions_bed(regions):
    """(chrom, start, end) intervals, 0-based half-open -> the BED text vf_vcf_open_cohort filters with."""
    return "".join(f"{c}\t{int(a)}\t{int(b)}\n" for c, a, b in regions)


def load_vcf_cohort(path, samples=None, regions=None, threads=0):
    """Many samples of one VCF in ONE parse -> (names, [per sample: load_vcf_sample's dict]).  samples: names (None =
    every sample column, in file order); regions: optional (chrom, start, end) intervals (0-based, half-open): only
    records whose REF span intersects one are kept.  Sample s's dict equals load_vcf_sample(path, s) (restricted to the
    regions)."""
    l = lib()
    if samples is not None:
        samples = [str(s) for s in samples]
        arr = (C.c_char_p * max(1, len(samples)))(*[s.encode() for s in samples])
        h = l.vf_vcf_open_cohort(os.fsencode(path), C.cast(arr, _vp), len(samples),
                                 None if regions is None else regions_bed(regions).encode(), threads)
    else:
        h = l.vf_vcf_open_cohort(os.fsencode(path), None, 0,
                                 None if regions is None else regions_bed(regions).encode(), threads)
    if not h:
        _fail("vf_vcf_open_cohort")
    try:
        names = [l.vf_vcf_cohort_sample_name(h, s).decode() for s in range(l.vf_vcf_cohort_num_samples(h))]
        chroms = [l.vf_vcf_cohort_chrom(h, c).decode() for c in range(l.vf_vcf_cohort_num_chroms(h))]
        per = []
        for s in range(len(names)):
            d = {}
            for c, name in enumerate(chroms):
                n = l.vf_vcf_cohort_num_records(h, s, c)
                if n > 0:                    # load_vcf_sample lists only chromosomes where the sample keeps a record
                    d[name] = _copy_records(n, l.vf_vcf_cohort_alt_bytes(h, s, c),
                                            lambda *a: l.vf_vcf_cohort_copy(h, s, c, *a), "vf_vcf_cohort_copy")
            per.append(d)
        return names, per
    finally:
        l.vf_vcf_cohort_close(h)
