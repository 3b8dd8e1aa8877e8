"""vf_bpe_tokenize vs the CPU oracle, bit for bit, at the launch shapes gene slabs reach.

Windows over 8192 symbols run bpe_tokenize_cluster_kernel: 16-CTA clusters for a call of at most 4 windows, 8-CTA
clusters otherwise (vf_encode.cu: bpe_tokenize), so every slab of 5 or more genes runs the 8-CTA instantiation.  Each
CTA holds one segment of the window; merges, look-aheads and self-pair run scans cross segment boundaries through
distributed shared memory.  Every comparison checks the tokens, out_count (the count before truncation), the token
starts and the zero padding after the kept tokens, with no tolerance."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu

from oracle import stage1 as O  # noqa: E402  (checker only)
from tests.test_gpu_pipeline import CFG, HP, _oracle_batch, _world  # noqa: E402
from variantformer_b200 import ops  # noqa: E402
from variantformer_b200.engine import Engine  # noqa: E402
from variantformer_b200.pipeline import HotPath  # noqa: E402
from variantformer_b200.stage1 import Genome, SampleVariants, WindowTokenizer, gene_window  # noqa: E402
from variantformer_b200.utils import random_init, synth  # noqa: E402

DEV = "cuda"
SMEM_SYMS = 8192              # longest window of the shared-memory kernel (kBpeSmemSyms)
GENE_CAP = 200 * 200          # max_length * max_chunks: tokens kept per gene window
SEP = b"N"


@pytest.fixture(scope="module")
def tk():
    return WindowTokenizer(DEV)


@pytest.fixture(scope="module")
def merges(tk):
    return tk.merges


class _Oracle:
    """OracleBPE.encode_with_starts, memoised per sequence, and the length in bases of every token id."""

    def __init__(self):
        self.bpe = O.OracleBPE()
        self.tlen = np.zeros(max(self.bpe.vocab.values()) + 1, np.int64)
        for s, i in self.bpe.vocab.items():
            self.tlen[i] = len(s) if i >= 4 else 0
        self.memo = {}

    def __call__(self, s: bytes):
        if s not in self.memo:
            self.memo[s] = self.bpe.encode_with_starts(s)
        return self.memo[s]

    def covers(self, s: bytes, b: int) -> bool:
        """Some token holds both base b - 1 and base b."""
        tok, st = self(s)
        i = int(np.searchsorted(st, b - 1, "right")) - 1
        return i >= 0 and st[i] + self.tlen[tok[i]] > b


@pytest.fixture(scope="module")
def oracle():
    return _Oracle()


def _seg(n, cl):
    # segment of one CTA in bpe_tokenize_cluster_kernel<CL> (vf_encode.cu): round_up_8(max(8, ceil(n / CL)))
    return (max(8, -(-n // cl)) + 7) // 8 * 8


def _bases(rng, n, alphabet=b"ACGT"):
    return rng.choice(np.frombuffer(alphabet, np.uint8), n).tobytes()


def _run(seqs, max_len, merges, out_cap, pitch, typical_len=None):
    """One ops.bpe_tokenize call over all of `seqs` (bytes) packed at `pitch` -> numpy (tokens, counts, starts)."""
    lens = np.array([len(s) for s in seqs], np.int32)
    buf = np.zeros((len(seqs), pitch), np.uint8)
    for i, s in enumerate(seqs):
        buf[i, :len(s)] = np.frombuffer(s, np.uint8)
    tok, cnt, st = ops.bpe_tokenize(torch.from_numpy(buf).to(DEV), torch.from_numpy(lens).to(DEV), max_len, merges,
                                    out_cap, out_cap, want_starts=True, typical_len=typical_len)
    return tok.cpu().numpy(), cnt.cpu().numpy(), st.cpu().numpy()


def _assert_oracle(res, seqs, oracle, limit, what):
    """Window i must tokenize as the oracle does its first min(len, limit) bases (limit = min(max_len, pitch))."""
    tok, cnt, st = res
    cap = tok.shape[1]
    for i, s in enumerate(seqs):
        want, want_st = oracle(s[:limit])
        k = min(len(want), cap)
        assert cnt[i] == len(want), f"{what}: window {i} (len {len(s)}): count {cnt[i]} != {len(want)}"
        assert np.array_equal(tok[i, :k], want[:k]), f"{what}: window {i} (len {len(s)}): tokens differ"
        assert not tok[i, k:].any(), f"{what}: window {i}: nonzero padding after {k} tokens"
        assert np.array_equal(st[i, :len(want)], want_st), f"{what}: window {i} (len {len(s)}): token starts differ"


def _assert_same(r0, r1, what):
    (t0, c0, s0), (t1, c1, s1) = r0, r1
    assert np.array_equal(c0, c1), f"{what}: counts differ"
    assert np.array_equal(t0, t1), f"{what}: tokens differ"
    for i, c in enumerate(c0):               # starts past the count are never written
        assert np.array_equal(s0[i, :c], s1[i, :c]), f"{what}: window {i}: token starts differ"


def _concat(parts):
    return tuple(np.concatenate(x) for x in zip(*parts))


# ---------------------------------------------------------------------------------------------------------------------
# 1. gene windows on 8-CTA clusters
# ---------------------------------------------------------------------------------------------------------------------

def test_gene_windows_on_8_cta_clusters_match_oracle_and_16_cta_clusters(merges, oracle):
    rng = np.random.default_rng(101)
    lens = [250_000, 262_417, 280_001, 291_999, 305_000, 301_000]
    pitch = -(-(max(lens) + 4096) // 16) * 16              # a slab tokenized with a sample: 4096 bytes of insert room
    seqs = [_bases(rng, n) for n in lens]
    seqs.append(_bases(rng, pitch - 3))                      # grown by insertions to just under the pitch
    seqs.append(synth.make_chromosome(rng, 280_000, softmask_frac=0.3, n_rate=3e-4).tobytes())   # N runs, lowercase
    assert b"N" in seqs[-1] and b"a" in seqs[-1]
    assert len(seqs) >= 8 and pitch > SMEM_SYMS              # more than 4 windows over 8192 symbols: 8-CTA clusters
    r8 = _run(seqs, pitch, merges, GENE_CAP, pitch)
    _assert_oracle(r8, seqs, oracle, pitch, "8-CTA clusters")
    assert (r8[1] > GENE_CAP).all()                          # every window is truncated, out_count is not
    r16 = _concat([_run(seqs[i:i + 4], pitch, merges, GENE_CAP, pitch) for i in range(0, len(seqs), 4)])
    _assert_same(r8, r16, "8-CTA vs 16-CTA clusters")
    r8u = _run(seqs, pitch, merges[:3], GENE_CAP, pitch)     # every rank its own sweep
    _assert_same(r8, r8u, "batched vs unbatched merge table on 8-CTA clusters")


# ---------------------------------------------------------------------------------------------------------------------
# 2. features on the segment boundaries
# ---------------------------------------------------------------------------------------------------------------------
# kind -> offset of the N from the boundary b
SEPARATORS = {"N at b-1": -1, "N at b": 0, "N at b+1": 1}
FEATURES = ("A run, odd", "A run, even", "N at b-1", "N at b", "N at b+1", "lowercase", "IUPAC", "AC repeat")


def _feature(kind, rng):
    """-> (text, lo, hi): text[lo:hi] is the feature proper (the rest are flanks that end a homopolymer run)."""
    if kind == "A run, odd":
        return b"C" + b"A" * 37 + b"G", 1, 38
    if kind == "A run, even":
        return b"T" + b"A" * 38 + b"C", 1, 39
    if kind == "lowercase":
        return _bases(rng, 40, b"acgt"), 0, 40
    if kind == "IUPAC":
        return _bases(rng, 6, b"RYKMSWBDHV"), 0, 6
    if kind == "AC repeat":
        return b"AC" * 15, 0, 30
    raise ValueError(kind)


def _boundary_window(rng, n, cl, w, oracle):
    """A random ACGT window of n bases with one feature across every boundary k * seg (cycling through FEATURES).
    A merge feature is shifted along its boundary until the oracle puts one token across the boundary, so the kernel
    must merge across two CTAs' segments (IUPAC letters never merge: that stretch stays where it was first put).
    -> (bytes, [(kind, b, start, text)])"""
    bg = bytearray(_bases(rng, n))
    seg = _seg(n, cl)
    plan = []
    for k in range(1, cl):
        b = k * seg
        assert b < n
        kind = FEATURES[(w + k) % len(FEATURES)]
        if kind in SEPARATORS:
            plan.append([kind, b, [b + SEPARATORS[kind]], SEP])
        else:
            text, lo, hi = _feature(kind, rng)
            mid = (lo + hi) // 2                              # b - start from the middle outwards, b-1 and b inside
            ds = sorted(range(lo + 1, hi), key=lambda d: abs(d - mid))
            plan.append([kind, b, [b - d for d in ds], text])
    pick = [0] * len(plan)
    for _ in range(12):
        s = bytearray(bg)
        for (kind, b, starts, text), j in zip(plan, pick):
            s[starts[j]:starts[j] + len(text)] = text
        s = bytes(s)
        moved = False
        for i, (kind, b, starts, text) in enumerate(plan):
            if kind not in SEPARATORS and kind != "IUPAC" and not oracle.covers(s, b):
                pick[i] += 1
                moved = True
        if not moved:
            break
    return s, [(kind, b, starts[j], text) for (kind, b, starts, text), j in zip(plan, pick)]


def _long_run_window(rng, n, cl, oracle):
    """One A run of 30 001 bases from just before boundary 1 to past boundary 2, so it covers a whole segment and its
    self-pair scans walk back through more than one CTA (the scans are quadratic in the run length: keep it short).
    Shifted until a token crosses each boundary it spans.  -> (bytes, run start, run end)"""
    seg = _seg(n, cl)
    bg = _bases(rng, n)
    run = b"A" * 30_001
    for shift in range(16):
        a = seg - 1001 - shift
        s = bg[:a - 1] + b"C" + run + b"T" + bg[a + len(run) + 1:]
        bounds = [k * seg for k in range(1, cl) if a < k * seg < a + len(run)]
        if all(oracle.covers(s, b) for b in bounds):
            break
    assert len(s) == n and len(run) > seg and a < seg and 2 * seg < a + len(run)
    return s, a, a + len(run)


@pytest.mark.parametrize("cl", [8, 16])
def test_features_across_segment_boundaries(merges, oracle, cl):
    rng = np.random.default_rng(200 + cl)
    lens = [100_000, 150_011, 203_457, 250_001, 299_999, 301_000] if cl == 8 else [100_003, 211_111, 301_000]
    windows = [_boundary_window(rng, n, cl, w, oracle) for w, n in enumerate(lens)]
    seqs = [s for s, _ in windows]
    seen = set()
    for s, plan in windows:
        seg = _seg(len(s), cl)
        for kind, b, start, text in plan:
            assert b % seg == 0 and 0 < b < len(s)
            seen.add(kind)
            if kind in SEPARATORS:
                p = b + SEPARATORS[kind]
                assert start == p and s[p:p + 1] == SEP and s[p - 1:p] in (b"A", b"C", b"G", b"T") \
                    and s[p + 1:p + 2] in (b"A", b"C", b"G", b"T"), (kind, b)
                continue
            assert start <= b - 1 and b < start + len(text), (kind, b, start)             # straddles b
            if kind == "IUPAC":
                # bpe500 has no merge with an IUPAC letter: each stays a token of its own, and the look-ahead of the
                # bases before it must see it as an alive symbol, not skip it
                tok, st = oracle(s)
                i = int(np.searchsorted(st, b - 1))
                assert st[i] == b - 1 and st[i + 1] == b and oracle.tlen[tok[i]] == oracle.tlen[tok[i + 1]] == 1
            else:
                assert oracle.covers(s, b), f"{kind} at boundary {b}: no token crosses it"
    assert seen == set(FEATURES)
    s, a0, a1 = _long_run_window(rng, 100_000 if cl == 8 else 200_000, cl, oracle)
    seg = _seg(len(s), cl)
    bounds = [k * seg for k in range(1, cl) if a0 < k * seg < a1]
    assert len(bounds) >= 2 and all(oracle.covers(s, b) for b in bounds)
    seqs.append(s)
    assert (len(seqs) > 4) == (cl == 8) and len(seqs) >= 4  # 5 or more windows: 8-CTA clusters; 4 or fewer: 16
    pitch = -(-max(map(len, seqs)) // 16) * 16
    assert pitch > SMEM_SYMS
    res = _run(seqs, pitch, merges, pitch, pitch)
    _assert_oracle(res, seqs, oracle, pitch, f"{cl}-CTA clusters")


# ---------------------------------------------------------------------------------------------------------------------
# 3. mixed lengths in one cluster call
# ---------------------------------------------------------------------------------------------------------------------

def test_mixed_lengths_in_one_cluster_call(merges, oracle):
    rng = np.random.default_rng(303)
    seqs = [b"", b"A", _bases(rng, 7), b"A" * 8, b"A" * 9, b"C" + b"A" * 15 + b"G", b"AC" * 32]
    seqs += [_bases(rng, 8192), _bases(rng, 8193),
             synth.make_chromosome(rng, 9000, n_rate=1e-3).tobytes(), _bases(rng, 60_000, b"ACGTACGTACGTN"),
             synth.make_chromosome(rng, 301_000, n_rate=1e-4).tobytes()]
    assert [len(s) for s in seqs] == [0, 1, 7, 8, 9, 17, 64, 8192, 8193, 9000, 60_000, 301_000]
    max_len = 250_000                                         # below the last window's length: clamped to it
    pitch = -(-301_000 // 16) * 16
    assert len(seqs) > 4 and max_len > SMEM_SYMS             # one call on 8-CTA clusters
    # short windows get 8-symbol segments (17 A's span three CTAs), empty ones lo == hi == n
    assert _seg(17, 8) == 8 and _seg(0, 8) == 8 and _seg(8193, 8) == 1032
    res = _run(seqs, max_len, merges, GENE_CAP, pitch)
    _assert_oracle(res, seqs, oracle, max_len, "mixed lengths")
    assert res[1][-1] == len(oracle(seqs[-1][:max_len])[0]) != len(oracle(seqs[-1])[0])


# ---------------------------------------------------------------------------------------------------------------------
# 4. the 8192 / 8193 switch between the kernels
# ---------------------------------------------------------------------------------------------------------------------

def test_8192_and_8193_symbol_kernels_agree(merges, oracle):
    rng = np.random.default_rng(404)
    seqs = [_bases(rng, 8192), _bases(rng, 8191), synth.make_chromosome(rng, 8192, n_rate=2e-3).tobytes(),
            _bases(rng, 1020) + b"C" + b"A" * 41 + b"T" + _bases(rng, 7126), _bases(rng, 4096), _bases(rng, 17), b""]
    assert [len(s) for s in seqs[:4]] == [8192, 8191, 8192, 8189]
    pitch = 8208
    assert len(seqs) > 4
    shared = _run(seqs, SMEM_SYMS, merges, SMEM_SYMS + 1, pitch)
    cluster = _run(seqs, SMEM_SYMS + 1, merges, SMEM_SYMS + 1, pitch)
    _assert_oracle(shared, seqs, oracle, pitch, "shared-memory kernel, max_len 8192")
    _assert_oracle(cluster, seqs, oracle, pitch, "8-CTA clusters, max_len 8193")
    _assert_same(shared, cluster, "max_len 8192 vs 8193")


# ---------------------------------------------------------------------------------------------------------------------
# 5. the block-size hint
# ---------------------------------------------------------------------------------------------------------------------

def test_block_size_hint_does_not_change_tokens(tk, merges, oracle):
    rng = np.random.default_rng(505)
    lens = [0, 1, 8, 9, 63, 64, 65, 200, 350, 1024, 1025, 2048, 4095, 4096, 4511, 4512, 4513, 6000, 8191, 8192]
    lens += rng.integers(0, 8193, 20).tolist()
    seqs = [synth.make_chromosome(rng, n, n_rate=2e-3).tobytes() if n else b"" for n in lens]
    pitch, max_len = 8192, 4512                              # a CRE call: ~400-base windows + 4096 bytes of insert room
    hints = [None, 200, 1500, 3000, 8000]                    # 1024, 64, 256, 512 and 1024 threads
    buf = np.zeros((len(seqs), pitch), np.uint8)
    for i, s in enumerate(seqs):
        buf[i, :len(s)] = np.frombuffer(s, np.uint8)
    buf = torch.from_numpy(buf).to(DEV)
    lens_d = torch.tensor(lens, dtype=torch.int32, device=DEV)
    full0 = fixed0 = None
    for t in hints:
        full = _run(seqs, max_len, merges, max_len, pitch, typical_len=t)
        _assert_oracle(full, seqs, oracle, max_len, f"typical_len {t}, out_cap {max_len}")
        fixed = tuple(x.cpu().numpy() for x in tk.tokenize_fixed(buf, lens_d, max_len, typical_len=t))
        for i, s in enumerate(seqs):
            want = oracle(s[:max_len])[0]
            o, m = O.adjust_length(want, 200)
            assert fixed[2][i] == len(want), f"typical_len {t}, out_cap 200: window {i} count"
            assert np.array_equal(fixed[0][i], o) and np.array_equal(fixed[1][i], m), f"typical_len {t}: window {i}"
        if full0 is None:
            full0, fixed0 = full, fixed
        _assert_same(full0, full, f"typical_len {hints[0]} vs {t}")
        assert all(np.array_equal(a, b) for a, b in zip(fixed0, fixed)), f"tokenize_fixed: typical_len {hints[0]} vs {t}"


# ---------------------------------------------------------------------------------------------------------------------
# 6. a production slab of 8 genes
# ---------------------------------------------------------------------------------------------------------------------

@pytest.fixture(scope="module")
def slab8():
    chroms, var, genes = _world(seed=82, n_genes=8)
    sd = random_init.make_state_dict(CFG, HP, seed=5)
    return chroms, var, genes, HotPath(Engine(sd, CFG, HP), Genome.from_arrays(chroms, DEV))


def _gene_window_seq(chroms, var, g, use_var):
    """The gene window as _oracle_batch builds it (oracle genotype application, reverse complement on '-')."""
    a0, a1 = gene_window(g.start, g.end, g.strand, 1000, 300000)
    chrom, v = chroms[g.chrom], var[g.chrom]
    if use_var:
        lens = np.array([len(a) for a in v["alt"]], np.int32)
        lo, hi = np.searchsorted(v["pos"], a0), np.searchsorted(v["pos"], a1)
        s = O.apply_variants(chrom, a0, a1, v["pos"][lo:hi], v["ref_len"][lo:hi], (np.cumsum(lens) - lens)[lo:hi],
                             lens[lo:hi], v["gt"][lo:hi], np.frombuffer(b"".join(v["alt"]), np.uint8))
    else:
        s = chrom[a0:a1].tobytes()
    return O.reverse_complement(s) if g.strand == "-" else s


@pytest.mark.parametrize("use_var", [True, False])
def test_slab_of_8_genes_matches_oracle_and_two_slabs_of_4(slab8, oracle, use_var):
    chroms, var, genes, hot = slab8
    assert len(genes) == 8 and {g.strand for g in genes} == {"+", "-"}
    sv = SampleVariants(var, DEV) if use_var else None
    t = hot.tokenize(genes, sv)
    want = _oracle_batch(chroms, var, genes, use_var=use_var)
    assert t["gene_seq"][0].shape[1] > SMEM_SYMS             # 8 gene windows in one call: 8-CTA clusters
    for g in range(len(genes)):
        assert torch.equal(t["cre_tok"][g].cpu().long(), want["cre_sequences"][g][:, 0]), f"CRE tokens gene {g}"
        assert torch.equal(t["cre_msk"][g].cpu(), want["cre_attention_masks"][g][:, 0]), f"CRE mask gene {g}"
        assert torch.equal(t["gene_tok"][g].cpu().long(), want["gene_embeddings"][g][:, 0]), f"gene tokens gene {g}"
        assert torch.equal(t["gene_msk"][g].cpu(), want["gene_attention_masks"][g][:, 0]), f"gene mask gene {g}"
        s = _gene_window_seq(chroms, var, genes[g], use_var)
        assert len(s) > SMEM_SYMS and t["gene_count"][g] == len(oracle(s)[0]), f"gene token count gene {g}"
    halves = [hot.tokenize(genes[:4], sv), hot.tokenize(genes[4:], sv)]   # 4 gene windows per call: 16-CTA clusters
    for key in ("cre_tok", "cre_msk", "gene_tok", "gene_msk"):
        got = halves[0][key] + halves[1][key]
        assert all(torch.equal(a, b) for a, b in zip(t[key], got)), f"{key}: one slab of 8 vs two slabs of 4"
    assert np.array_equal(t["gene_count"], np.concatenate([h["gene_count"] for h in halves]))
