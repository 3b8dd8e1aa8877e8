"""CPU checks of variant tables in shared passes: the allele-splice rule (numpy restatement of vf_splice_windows against
plain string surgery), the pair planner (grouping, edit dedup, chromosome filter, "No overlap", unreached windows) and
the gene-token-position arithmetic of insertions on both strands."""
import numpy as np
import pytest

from oracle import stage1 as O
from variantformer_b200 import vep_batch
from variantformer_b200.datasets.vepdataset import Variant, cre_windows, window_hits
from variantformer_b200.pipeline import GeneSpec
from variantformer_b200.stage1 import gene_window

CS = np.array([400_000, 400_120, 400_900, 401_000, 401_700])
CE = np.array([400_100, 400_300, 401_600, 401_100, 401_900])


def splice_np(src: bytes, off: int, allele: bytes, rc: bool) -> bytes:
    """numpy restatement of vf_splice_windows for one row: the ONE base at forward offset `off` replaced by `allele`;
    on a reverse-complemented row the reverse complement of the allele replaces the byte at len - 1 - off."""
    row = np.frombuffer(src, np.uint8)
    q = len(src) - 1 - off if rc else off
    a = np.frombuffer(O.reverse_complement(allele.decode()).encode() if rc else allele, np.uint8)
    return np.concatenate([row[:q], a, row[q + 1:]]).tobytes()


def test_splice_np_is_string_surgery_on_either_strand():
    rng = np.random.default_rng(3)
    for n in (1, 2, 17, 300):
        fwd = "".join(rng.choice(list("ACGTacgtNRYKM"), n))
        for k in (1, 2, 5, 31):
            allele = "".join(rng.choice(list("ACGTN"), k))
            for off in sorted({0, n - 1, int(rng.integers(0, n))}):
                edited = fwd[:off] + allele + fwd[off + 1:]                 # forward strand: one base -> the allele
                assert splice_np(fwd.encode(), off, allele.encode(), False) == edited.encode()
                # stored reverse-complemented: the edit of the forward sequence, reverse-complemented
                rc_src = O.reverse_complement(fwd).encode()
                assert splice_np(rc_src, off, allele.encode(), True) == O.reverse_complement(edited).encode()


def _gene(strand, cre_chrom=None, tissues=(62,)):
    return GeneSpec("chr1", 395_000, 420_000, strand, CS, CE, np.arange(5) % 9, list(tissues), cre_chrom=cre_chrom)


def _pair(gene, pos, ref, alt, tissues=(62,), chrom="chr1", gid="G1"):
    return dict(variant=Variant(chrom, pos, ref, alt, tissue=list(tissues)), gene=gene, gene_id=gid)


@pytest.mark.parametrize("strand", ["+", "-"])
def test_planner_groups_dedups_and_filters(strand):
    g = _gene(strand)
    minus = strand == "-"
    _, wins = cre_windows(g, 50)
    g0, g1 = gene_window(g.start, g.end, g.strand, 1000, 300000)
    pos_cre = 400_050                                               # inside windows 0 and 1 (+ strand order)
    pairs = [_pair(g, pos_cre, "A", "G"), _pair(g, pos_cre, "A", "G"),          # duplicate row
             _pair(g, pos_cre, "A", "TTT"),                                     # insertion: het 'N'
             _pair(g, pos_cre, "AC", "G"),                                      # multi-base REF: het 'N' again
             _pair(g, pos_cre, "A", "G", tissues=(3, 62)),                      # same gene, other tissue list
             _pair(g, 5_000_000, "A", "G"),                                     # touches nothing
             _pair(g, pos_cre, "A", "G", gid="G2"),                             # another gene
             _pair(g, pos_cre, "A", "")]                                        # empty ALT: a deletion
    groups, plans = vep_batch.plan_pairs(pairs)
    assert [p.group for p in plans] == [0, 0, 0, 0, 1, 0, 2, 0] and len(groups) == 3
    assert plans[5].variant_type == "No overlap" and plans[5].edits == ()
    assert plans[0].edits == plans[1].edits                          # duplicates share their items
    het_n = groups[0].edit_of[("chr1", pos_cre, b"N")]
    assert plans[2].edits[0] == het_n == plans[3].edits[0]           # the two 'N' hets collide
    assert [e.data for e in groups[0].edits] == [b"R", b"G", b"N", b"TTT", b""]
    assert plans[7].edits[0] == het_n
    hits, cre_hit, unreached, gene_hit = window_hits(wins, minus, pos_cre, g0, g1)
    for p in plans[:5] + plans[6:]:
        e = groups[p.group].edits[p.edits[1]]
        assert e.hits == hits and p.cre_hit == cre_hit and e.gene_hit == gene_hit == p.gene_hit
        assert e.plain_cre == [] and not e.plain_gene                      # every window on the variant's chromosome
    assert plans[0].variant_type == "Gene and CRE overlap"


def test_planner_unreached_windows_and_other_chromosome():
    # minus strand, rows descending by start: the early break can stop before a nested window that holds the variant
    g = _gene("-")
    _, wins = cre_windows(g, 50)
    g0, g1 = gene_window(g.start, g.end, g.strand, 1000, 300000)
    for pos in range(399_900, 402_000):
        hits, cre_hit, unreached, gene_hit = window_hits(wins, True, pos, g0, g1)
        if unreached:
            break
    else:
        pytest.fail("no position with an unreached window")
    groups, plans = vep_batch.plan_pairs([_pair(g, pos, "A", "C")])
    e = groups[0].edits[plans[0].edits[1]]
    assert e.hits == hits and not set(unreached) & set(e.hits)
    # a CRE row on another chromosome: window_hits' cre_hit is kept, but that window is not edited
    other = _gene("+", cre_chrom=["chr1", "chr2", "chr1", "chr1", "chr1"])
    _, wins = cre_windows(other, 50)
    groups, plans = vep_batch.plan_pairs([_pair(other, 400_200, "A", "C")])
    hits, cre_hit, _, _ = window_hits(wins, False, 400_200, g0, g1)
    assert cre_hit == 1 and plans[0].cre_hit == 1
    e = groups[0].edits[plans[0].edits[1]]
    assert e.hits == [k for k in hits if k != 1]
    assert e.plain_cre == [1] and not e.plain_gene          # the het / hom samples hold no background on chr2
    # a variant on another chromosome than the gene: nothing is edited, every window but the unreached ones is read
    # without the background, the token positions still follow the builder
    hits, _, unreached, _ = window_hits(cre_windows(g, 50)[1], True, 400_050, g0, g1)
    groups, plans = vep_batch.plan_pairs([_pair(g, 400_050, "A", "C", chrom="chr2")])
    e = groups[0].edits[plans[0].edits[1]]
    assert e.hits == [] and not e.gene_hit and plans[0].gene_hit and e.plain_gene
    assert e.plain_cre == [k for k in range(len(CS)) if k not in unreached]


def _builder_gene_pos(fwd: str, off: int, allele: str, minus: bool, L=4):
    """VEPBatchBuilder.build's formula on a window it built itself: p = pos0 - g0, len(seq) - p - 1 on the minus
    strand with the EDITED length, then the token covering base p."""
    edited = fwd[:off] + allele + fwd[off + 1:]
    seq = O.reverse_complement(edited) if minus else edited
    p = len(seq) - off - 1 if minus else off
    bounds = np.cumsum([0] + [L] * (len(seq) // L))                  # fixed 4-base tokens stand in for BPE
    return p, seq[p], int((bounds[bounds < len(seq)] <= p).sum()) - 1


@pytest.mark.parametrize("minus", [False, True])
def test_gene_token_position_of_insertions(minus):
    rng = np.random.default_rng(9)
    fwd = "".join(rng.choice(list("ACGT"), 97))
    for allele in ("G", "GT", "TTTTTTTTTTTTTTTTT"):
        for off in (0, 13, 50, 96):
            p, ch, tok = _builder_gene_pos(fwd, off, allele, minus)
            k = len(allele)
            # the planner's arithmetic (ism.build_edit_items): glen0 + k - 1 - off - 1 on the minus strand
            p_plan = len(fwd) + k - 1 - off - 1 if minus else off
            assert p_plan == p
            seq = splice_np(O.reverse_complement(fwd).encode() if minus else fwd.encode(), off, allele.encode(), minus)
            starts = np.arange(0, len(seq), 4)
            assert chr(seq[p]) == ch
            assert vep_batch.gene_token_position(seq, starts, p, max_length=3, context_window=5) == min(tok // 3, 4)
            # on the minus strand the base at p is the last byte of the reverse-complemented allele block
            assert chr(seq[p]) == (O.reverse_complement(allele)[-1] if minus else allele[0])
    with pytest.raises(ValueError, match="invalid character 'N'"):
        vep_batch.gene_token_position(b"ACNT", np.arange(4), 2)
