"""CPU checks of saturation mutagenesis: the host planner (window hits shared with the VEP builder, skip rules), the
strand rule of a single-base substitution, the slab partition, and the shared-window slab of the engine."""
import numpy as np
import pytest
import torch

from oracle import stage1 as O
from tests.common import pearson, rel_err
from tests.test_engine_host_logic import cpu_engine  # noqa: F401  (fixture)
from variantformer_b200 import ism
from variantformer_b200.datasets.vepdataset import cre_windows, get_iupac_code, window_hits
from variantformer_b200.pipeline import GeneSpec
from variantformer_b200.stage1 import cre_window, gene_window

CS = np.array([400_000, 400_120, 400_900, 401_000, 401_700])
CE = np.array([400_100, 400_300, 401_600, 401_100, 401_900])


def _gene(strand):
    return GeneSpec("chr1", 395_000, 420_000, strand, CS, CE, np.arange(5) % 9, [62])


def _walk(wins, minus, pos):
    """The reference's row loop (vepdataset.py:367-407) restated: every reached overlapping row, early break."""
    hits = []
    for k, (a, b) in enumerate(wins):
        if (b < pos) if minus else (a > pos):
            break
        if a < pos <= b:
            hits.append(k)
    return hits


def mutate_np(src: bytes, off: int, base: str, rc: bool) -> bytes:
    """numpy restatement of vf_mutate_windows for one row: the base at forward offset `off`, placed at len-1-off as its
    complement when the stored row is reverse-complemented."""
    row = bytearray(src)
    if rc:
        row[len(row) - 1 - off] = ord(O.reverse_complement(base))
    else:
        row[off] = ord(base)
    return bytes(row)


@pytest.mark.parametrize("strand", ["+", "-"])
def test_planner_hits_equal_the_vep_walk(strand):
    g = _gene(strand)
    minus = strand == "-"
    _, wins = cre_windows(g, 50)
    order = np.argsort(CS, kind="stable"); order = order[::-1] if minus else order
    assert wins == [cre_window(CS[i], CE[i], 50) for i in order]
    g0, g1 = gene_window(g.start, g.end, g.strand, 1000, 300000)
    start, end = 399_900, 402_000
    bases = b"ACGT" * ((end - start + 1) // 4) + b"ACGT"[:(end - start + 1) % 4]
    plan = ism.plan_mutants(g, start, end, bases, zygosity=(1, 2))
    seen = set()
    for m in plan.mutants:
        assert m.hits == _walk(wins, minus, m.pos) and m.gene_hit == (g0 < m.pos <= g1)
        hits, cre_hit, unreached, gene_hit = window_hits(wins, minus, m.pos, g0, g1)
        assert hits == m.hits and cre_hit == (m.hits[-1] if m.hits else None)
        assert set(unreached) == {k for k, (a, b) in enumerate(wins) if a < m.pos <= b} - set(hits)
        seen.add(m.pos)
    assert seen == set(range(start, end + 1))                         # the whole region lies in the gene window
    # overlapping windows: both reached rows get the base, the later one is the CRE hit
    m = next(m for m in plan.mutants if m.pos == 400_101)
    assert m.hits == ([0, 1] if not minus else [3, 4])
    if minus:
        # nested minus-strand row: 401301 lies in row 2 only, but the walk stops at row 1 -> no CRE hit (unreached)
        m = next(m for m in plan.mutants if m.pos == 401_301)
        assert m.hits == [] and m.gene_hit
        assert window_hits(wins, True, 401_301, g0, g1)[2] == [2]


def test_planner_enumeration_and_skip_rules():
    g = _gene("+")
    # region: 3 positions inside the first CRE window, then one far outside every window (own gene, tiny windows)
    bases = b"aNc"
    plan = ism.plan_mutants(g, 400_001, 400_003, bases, bg_bases=b"ANR", zygosity=(2, 1))
    assert plan.skipped["non_acgt"] == [400_002, 400_003]             # N in the genome, R (het SNP) in the background
    assert [(m.pos, m.ref, m.alt, m.zyg) for m in plan.mutants] == \
        [(400_001, "A", a, z) for a in "CGT" for z in (1, 2)]          # alt == ref is never enumerated
    for m in plan.mutants:
        assert m.base == (m.alt if m.zyg == 2 else get_iupac_code(m.ref, m.alt))
    far = GeneSpec("chr1", 395_000, 396_000, "+", CS, CE, np.arange(5) % 9, [62])
    plan = ism.plan_mutants(far, 398_000, 398_004, b"ACGTA", gene_downstream=500)
    assert plan.mutants == [] and plan.skipped["no_overlap"] == list(range(398_000, 398_005))
    with pytest.raises(ValueError):
        ism.plan_mutants(g, 400_001, 400_003, bases, zygosity=(0,))


@pytest.mark.parametrize("rc", [False, True])
def test_substitution_offset_and_complement_follow_the_strand(rc):
    rng = np.random.default_rng(3)
    fwd = bytes(rng.choice(np.frombuffer(b"ACGTacgt", np.uint8), 97))
    for off in (0, 41, 96):
        for base in "ACGTRYKMSW":
            want = fwd[:off] + base.encode() + fwd[off + 1:]              # the variant applied on the forward strand
            want = O.reverse_complement(want) if rc else want
            src = O.reverse_complement(fwd) if rc else fwd
            assert mutate_np(src, off, base, rc) == want


def test_slab_partition_respects_the_rows_budget():
    assert ism.slab_partition(10, 1024, 16384) == [(0, 10)]
    parts = ism.slab_partition(50, 1024, 16384)
    assert parts[0] == (0, 16) and parts[-1] == (48, 50) and sum(b - a for a, b in parts) == 50
    assert all((b - a) * 1024 <= 16384 for a, b in parts)
    assert ism.slab_partition(3, 40000, 16384) == [(0, 1), (1, 2), (2, 3)]      # one item even over budget
    assert ism.slab_partition(0, 10) == []


def test_shared_window_slab_equals_the_explicit_slab(cpu_engine):  # noqa: F811
    """prepare_shared + run_pooled over deduplicated windows gives what prepare + run gives for the items' own tokens."""
    from tests.common import load_model_golden
    batch, _, _ = load_model_golden()
    sq = lambda xs: [x[:, 0, :] for x in xs]
    ct, cm, gt, gm = (sq(batch[k]) for k in ("cre_sequences", "cre_attention_masks", "gene_embeddings",
                                             "gene_attention_masks"))
    tis, lab = batch["tissue_context"], batch["ref_cre_labels"]
    # item 2 = gene 0 with its CRE row 1 replaced by gene 1's CRE row 0 and its last chunk by gene 1's chunk 0
    ct2 = ct[0].clone(); ct2[1] = ct[1][0]; cm2 = cm[0].clone(); cm2[1] = cm[1][0]
    gt2 = gt[0].clone(); gt2[-1] = gt[1][0]; gm2 = gm[0].clone(); gm2[-1] = gm[1][0]
    want = cpu_engine.forward_tokens([ct[0], ct[1], ct2], [cm[0], cm[1], cm2], [gt[0], gt[1], gt2],
                                     [gm[0], gm[1], gm2], [tis[0], tis[1], tis[0]], [lab[0], lab[1], lab[0]])
    # unique windows: both genes' own windows once
    s0 = cpu_engine.prepare(ct[:2], cm[:2], gt[:2], gm[:2], tis[:2], lab[:2])
    cpool, gpool = cpu_engine.pool_windows(s0)
    C0, G0 = ct[0].shape[0], gt[0].shape[0]
    c_rows = [np.arange(C0), C0 + np.arange(ct[1].shape[0]), np.arange(C0)]
    c_rows[2] = c_rows[2].copy(); c_rows[2][1] = C0
    g_rows = [np.arange(G0), G0 + np.arange(gt[1].shape[0]), np.arange(G0)]
    g_rows[2] = g_rows[2].copy(); g_rows[2][-1] = G0
    s = cpu_engine.prepare_shared(c_rows, g_rows, gpool.shape[0], [tis[0], tis[1], tis[0]], [lab[0], lab[1], lab[0]])
    got = cpu_engine.run_pooled(s, cpool, gpool)
    assert got["T"] == want["T"]
    for k in ("pred", "emb"):
        a, b = got[k].float().numpy(), want[k].float().numpy()
        assert rel_err(a, b) <= 1e-2 and pearson(a, b) >= 0.9999, k
    assert not torch.equal(got["emb"][:len(tis[0])], got["emb"][-len(tis[0]):])   # item 2 really differs from gene 0
