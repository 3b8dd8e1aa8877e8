"""Multi-sample ingest (vf_vcf_open_cohort / ingest.load_vcf_cohort): one parse of an N-column VCF gives every sample
exactly what the single-sample parse and the pure-Python restatement give, in plain, gzip and BGZF form; the region
filter equals filtering afterwards.  CPU only."""
import numpy as np
import pytest

from oracle import ingest_py
from tests.test_ingest_native import _write
from variantformer_b200 import ingest

N_SAMPLES = 18
GTS = [b"0/0", b"0/1", b"1/1", b"1|0", b"0|1", b"1|2", b"2/1", b"./.", b".", b"1", b"0", b"2|2", b"1/1/1", b"0/1/2",
       b"./1", b"2", b"0|0"]


def _cohort_vcf(rng, n=6000, n_samples=N_SAMPLES):
    """Every genotype form of include/vf_ingest.h: multi-allelic sites, hets of two SNP ALTs (IUPAC), haploid and
    polyploid calls, phased / unphased, missing, symbolic and '*' ALTs, runs of equal positions, short lines."""
    names = [f"S{i}" for i in range(n_samples)]
    lines = [b"##fileformat=VCFv4.2", b"#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\t" +
             "\t".join(names).encode()]
    bases = [b"A", b"C", b"G", b"T"]
    pos = 1000
    for _ in range(n):
        chrom = b"chr%d" % int(rng.integers(1, 4))
        if rng.random() > 0.15:                              # otherwise: the same position again (file order matters)
            pos = int(rng.integers(1, 400_000))
        kind = rng.random()
        if kind < 0.6:
            ref = bases[int(rng.integers(4))]
            alt = b",".join(bases[int(x)] for x in rng.choice(4, int(rng.integers(1, 4)), replace=False))
        elif kind < 0.75:
            ref = b"".join(bases[int(x)] for x in rng.integers(0, 4, int(rng.integers(1, 6))))
            alt = bases[int(rng.integers(4))] + b",<DEL>"
        elif kind < 0.9:
            ref = bases[int(rng.integers(4))]
            alt = ref + b"".join(bases[int(x)] for x in rng.integers(0, 4, int(rng.integers(1, 8)))) + b",*"
        else:
            ref = b"N"; alt = b"<INS>,A"
        # common sites: most samples share the genotype; rare sites: most are hom-ref
        common = rng.random() < 0.3
        cols = []
        for _ in range(n_samples):
            g = GTS[int(rng.integers(len(GTS)))] if (rng.random() < (0.8 if common else 0.2)) else b"0/0"
            cols.append(g + (b":12:0.5" if rng.random() < 0.3 else b""))
        if rng.random() < 0.02:
            cols = cols[:int(rng.integers(0, n_samples))]    # a truncated line: the missing columns drop the record
        lines.append(b"\t".join([chrom, str(pos).encode(), b".", ref, alt, b".", b"PASS", b".", b"GT:DP:AF"] + cols))
    return b"\n".join(lines) + b"\n", names


def _same(got, want):
    assert sorted(got) == sorted(want)
    for c in want:
        for k in ("pos", "ref_len", "gt"):
            assert np.array_equal(got[c][k], want[c][k]), (c, k)
        assert got[c]["alt"] == want[c]["alt"], c


@pytest.mark.parametrize("form", ["plain", "gzip", "bgzf"])
def test_cohort_parse_equals_single_sample_parses(tmp_path, form):
    rng = np.random.default_rng(21)
    data, names = _cohort_vcf(rng)
    path = _write(tmp_path / f"c.{form}", data, form)
    got_names, per = ingest.load_vcf_cohort(path, threads=3)
    assert got_names == names and len(per) == N_SAMPLES
    for s, name in enumerate(names):
        _same(per[s], ingest.load_vcf_sample(path, sample=name, threads=2))
        _same(per[s], ingest_py.load_vcf_sample(path, sample=name))
    # a subset in another order: the same per-sample results
    pick = ["S7", "S0", "S17", "S3"]
    sub_names, sub = ingest.load_vcf_cohort(path, samples=pick, threads=1)
    assert sub_names == pick
    for name, d in zip(pick, sub):
        _same(d, per[names.index(name)])


def test_region_filter_equals_filtering_afterwards(tmp_path):
    rng = np.random.default_rng(22)
    data, names = _cohort_vcf(rng, n=4000)
    path = _write(tmp_path / "c.bgzf", data, "bgzf")
    regions = [("chr1", 10_000, 60_000), ("chr1", 50_000, 90_000), ("chr2", 300_000, 300_001), ("chr3", 0, 5),
               ("chr9", 0, 1_000_000), ("chr2", 120_000, 120_000)]
    _, full = ingest.load_vcf_cohort(path)
    _, filt = ingest.load_vcf_cohort(path, regions=regions)

    def hit(c, p, rl):
        return any(c == rc and p < b and p + max(int(rl), 1) > a for rc, a, b in regions)
    n_kept = 0
    for d, f in zip(full, filt):
        want = {}
        for c, v in d.items():
            keep = [i for i, (p, rl) in enumerate(zip(v["pos"], v["ref_len"])) if hit(c, int(p), rl)]
            if keep:
                want[c] = dict(pos=v["pos"][keep], ref_len=v["ref_len"][keep], gt=v["gt"][keep],
                               alt=[v["alt"][i] for i in keep])
                n_kept += len(keep)
        _same(f, want)
    assert n_kept > 0
    # REF spans that straddle an interval's start are kept: a deletion starting before it reaches into it
    vcf = tmp_path / "span.vcf"
    vcf.write_text("#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tA\tB\n"
                   "chr1\t8\t.\tACGTA\tA\t.\t.\t.\tGT\t0/1\t0/0\n"
                   "chr1\t7\t.\tA\tG\t.\t.\t.\tGT\t1/1\t1/1\n"
                   "chr1\t11\t.\tA\tG\t.\t.\t.\tGT\t1/1\t1/1\n")
    _, per = ingest.load_vcf_cohort(str(vcf), regions=[("chr1", 10, 11)])
    assert per[0]["chr1"]["pos"].tolist() == [7, 10] and "chr1" in per[1] and per[1]["chr1"]["pos"].tolist() == [10]


def test_cohort_errors(tmp_path):
    vcf = tmp_path / "s.vcf"
    vcf.write_text("#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\tINFO\tFORMAT\tS1\tS2\nchr1\t5\t.\tA\tG\t.\t.\t.\tGT\t0/1\t1/1\n")
    with pytest.raises(ingest.IngestError, match="not found"):
        ingest.load_vcf_cohort(str(vcf), samples=["S1", "S9"])
    with pytest.raises(ingest.IngestError, match="twice"):
        ingest.load_vcf_cohort(str(vcf), samples=["S2", "S2"])
    with pytest.raises(ingest.IngestError, match="malformed BED"):
        ingest.load_vcf_cohort(str(vcf), regions=[("chr1", 9, 3)])
    with pytest.raises(ingest.IngestError, match="cannot open"):
        ingest.load_vcf_cohort(str(tmp_path / "missing.vcf"))
    sites = tmp_path / "sites.vcf"                           # sites-only: the '#CHROM' line ends at INFO / FORMAT
    for last in ("INFO", "INFO\tFORMAT"):
        sites.write_text(f"#CHROM\tPOS\tID\tREF\tALT\tQUAL\tFILTER\t{last}\n" +
                         "".join(f"chr1\t{p}\t.\tA\tG\t.\t.\t.\n" for p in (5, 9, 12)))
        with pytest.raises(ingest.IngestError, match="no sample columns"):
            ingest.load_vcf_cohort(str(sites))
    names, per = ingest.load_vcf_cohort(str(vcf))
    assert names == ["S1", "S2"] and [d["chr1"]["gt"].tolist() for d in per] == [[1], [2]]
