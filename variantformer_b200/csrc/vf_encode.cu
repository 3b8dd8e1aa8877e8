// vf_encode.cu — stage 1 on the GPU: genotype application (IUPAC diploid encoding)
// and BPE-500 tokenisation of every cis-regulatory / gene window.  Integer, byte
// and index work only: HBM/L2-bound, no tensor cores.  Bit-exact against
// oracle/vf_oracle.c (which is pinned to the reference's utils/seq.py + tokenizers).
//
// Replaces, per window:
//   `samtools faidx | bcftools consensus -H I` subprocess pairs  (utils/data_process.py:17-101, :367-467)
//   reverse_complement                                          (utils/functions.py:129-172)
//   BPEEncoder.normalize / encode (HF tokenizers BPE)            (utils/seq.py:32-62)
//   __adjust_length / chunkify_data                              (datasets/vcfdataset.py:198-217, :338-394)
#include <cooperative_groups.h>

#include <stdlib.h>

#include "vf_common.cuh"
#include "vf_internal.h"

namespace vf {

// ---------------------------------------------------------------------------------
// encode_windows: reference slice + sample genotypes -> (optionally reverse-complemented) sequence
// ---------------------------------------------------------------------------------
constexpr int kMaxApplied = 2048;     // applied variants per window kept in shared memory
constexpr int kEncSlice = 16384;      // reference bytes per CTA

__device__ __forceinline__ uint8_t comp_base(uint8_t c) {
    switch (c) {
        case 'A': return 'T'; case 'a': return 't'; case 'C': return 'G'; case 'c': return 'g';
        case 'G': return 'C'; case 'g': return 'c'; case 'T': return 'A'; case 't': return 'a';
        case 'R': return 'Y'; case 'r': return 'y'; case 'Y': return 'R'; case 'y': return 'r';
        case 'K': return 'M'; case 'k': return 'm'; case 'M': return 'K'; case 'm': return 'k';
        case 'B': return 'V'; case 'b': return 'v'; case 'V': return 'B'; case 'v': return 'b';
        case 'D': return 'H'; case 'd': return 'h'; case 'H': return 'D'; case 'h': return 'd';
        default: return c;
    }
}
__device__ __forceinline__ uint8_t iupac_het(uint8_t ref, uint8_t alt) {   // vepdataset.py:75-104
    const int r = ref == 'A' ? 0 : ref == 'C' ? 1 : ref == 'G' ? 2 : ref == 'T' ? 3 : -1;
    const int a = alt == 'A' ? 0 : alt == 'C' ? 1 : alt == 'G' ? 2 : alt == 'T' ? 3 : -1;
    if (r < 0 || a < 0) return 'N';
    const char tbl[17] = "AMRWMCSYRSGKWYKT";
    return (uint8_t)tbl[r * 4 + a];
}

struct EncodeParams {
    const uint8_t* genome;            // concatenated chromosomes, 1 byte/base as in the FASTA (case kept)
    const int64_t* win_base;          // [n_win] offset of the window's chromosome in `genome`
    const int32_t* w0; const int32_t* w1;         // [n_win] window [w0, w1) inside the chromosome
    const int32_t* var_lo; const int32_t* var_hi; // [n_win] range of candidate variants (pos in [w0, w1))
    const uint8_t* flags;             // [n_win] bit0 = reverse-complement, bit1 = SNP-only filter
    const int32_t* v_pos; const int32_t* v_ref_len; const int32_t* v_alt_off; const int32_t* v_alt_len;
    const uint8_t* v_gt;              // 0 skip, 1 het, 2 hom-alt
    const uint8_t* alt_pool;
    uint8_t* out; int64_t pitch;      // [n_win, pitch]
    int32_t* out_len;                 // [n_win]
    int32_t* err;                     // device error flag (1 = pitch overflow, 2 = too many variants)
};

__global__ void __launch_bounds__(256)
encode_windows_kernel(const EncodeParams p) {
    __shared__ int32_t s_vidx[kMaxApplied];     // applied variant index
    __shared__ int32_t s_shift[kMaxApplied];    // cumulative (alt_len - ref_len) BEFORE this variant
    __shared__ int s_n, s_total;
    const int w = blockIdx.y;
    const int w0 = p.w0[w], w1 = p.w1[w];
    const int slice0 = w0 + blockIdx.x * kEncSlice;
    if (slice0 >= w1 && !(blockIdx.x == 0)) return;
    const uint8_t fl = p.flags[w];
    const bool rc = fl & 1, snp_only = fl & 2;
    if (threadIdx.x == 0) {
        // sequential scan: which records are applied (overlap rule needs order) and where they land
        int n = 0, cur = w0, shift = 0, bad = 0;
        for (int i = p.var_lo[w]; i < p.var_hi[w]; ++i) {
            if (p.v_gt[i] == 0) continue;
            const int pos = p.v_pos[i], rl = p.v_ref_len[i], al = p.v_alt_len[i];
            if (pos < cur || pos + rl > w1) continue;
            if (snp_only && !(rl == 1 && al == 1)) continue;
            if (n == kMaxApplied) { bad = 2; break; }
            s_vidx[n] = i; s_shift[n] = shift; ++n;
            shift += al - rl;
            cur = pos + rl;
        }
        s_n = n; s_total = (w1 - w0) + shift;
        if (bad) atomicMax(p.err, bad);
        if (s_total > p.pitch) atomicMax(p.err, 1);
        // an overflowing window writes nothing: report length 0 (plus err = 1) so the tokenizer never reads past the row
        if (blockIdx.x == 0) p.out_len[w] = s_total > p.pitch ? 0 : s_total;
    }
    __syncthreads();
    const int n = s_n, total = s_total;
    if (total > p.pitch) return;
    const uint8_t* ref = p.genome + p.win_base[w];
    uint8_t* out = p.out + (size_t)w * p.pitch;
    const int slice1 = min(w1, slice0 + kEncSlice);
    // (1) reference bytes of this slice that survive (not inside an applied record's REF span)
    for (int x = slice0 + threadIdx.x; x < slice1; x += blockDim.x) {
        // last applied variant with pos <= x
        int lo = 0, hi = n;
        while (lo < hi) { const int mid = (lo + hi) >> 1; if (p.v_pos[s_vidx[mid]] <= x) lo = mid + 1; else hi = mid; }
        int shift = 0;
        if (lo > 0) {
            const int v = s_vidx[lo - 1];
            if (x < p.v_pos[v] + p.v_ref_len[v]) continue;              // replaced by the record's ALT
            shift = s_shift[lo - 1] + p.v_alt_len[v] - p.v_ref_len[v];
        }
        const int o = x - w0 + shift;
        const uint8_t b = ref[x];
        if (rc) out[total - 1 - o] = comp_base(b); else out[o] = b;
    }
    // (2) ALT bytes of the applied records that start inside this slice
    for (int k = threadIdx.x; k < n; k += blockDim.x) {
        const int v = s_vidx[k];
        const int pos = p.v_pos[v];
        if (pos < slice0 || pos >= slice1) continue;
        const int al = p.v_alt_len[v], rl = p.v_ref_len[v];
        const int o0 = pos - w0 + s_shift[k];
        if (al == 1 && rl == 1) {
            uint8_t a = p.alt_pool[p.v_alt_off[v]];
            if (p.v_gt[v] == 1) {
                uint8_t r = ref[pos];
                if (r >= 'a' && r <= 'z') r -= 32;
                a = iupac_het(r, a);
            }
            if (rc) out[total - 1 - o0] = comp_base(a); else out[o0] = a;
        } else {
            for (int j = 0; j < al; ++j) {
                const uint8_t a = p.alt_pool[p.v_alt_off[v] + j];
                if (rc) out[total - 1 - (o0 + j)] = comp_base(a); else out[o0 + j] = a;
            }
        }
    }
}

int encode_windows(const uint8_t* genome, const int64_t* win_base, const int32_t* w0, const int32_t* w1,
                   const int32_t* var_lo, const int32_t* var_hi, const uint8_t* flags, const int32_t* v_pos,
                   const int32_t* v_ref_len, const int32_t* v_alt_off, const int32_t* v_alt_len, const uint8_t* v_gt,
                   const uint8_t* alt_pool, int n_win, int max_window, uint8_t* out, int64_t pitch, int32_t* out_len,
                   int32_t* err, cudaStream_t s) {
    if (n_win == 0) return 0;
    VF_REQUIRE(max_window > 0 && pitch >= max_window, "encode_windows: pitch %lld < max window %d", (long long)pitch,
               max_window);
    EncodeParams p{genome, win_base, w0, w1, var_lo, var_hi, flags, v_pos, v_ref_len, v_alt_off, v_alt_len, v_gt,
                   alt_pool, out, pitch, out_len, err};
    dim3 grid((max_window + kEncSlice - 1) / kEncSlice, n_win);
    encode_windows_kernel<<<grid, 256, 0, s>>>(p);
    VF_LAUNCH_OK("encode_windows_kernel launch");
    return 0;
}

// ---------------------------------------------------------------------------------
// mutate_windows: an encoded window with ONE base replaced (saturation mutagenesis).  Row r of `out` is the source row
// src[row_src[r]] with the base at forward-strand offset row_off[r] set to row_base[r]; a reverse-complemented source
// (flags bit 0) gets it at len - 1 - off as its complement, with the table encode_windows uses (comp_base).
// One CTA per (row, 16 KB slice), 16-byte loads and stores: pure copy bandwidth.
// ---------------------------------------------------------------------------------
constexpr int kMutSlice = 16384;

struct MutateParams {
    const uint8_t* src; int64_t src_pitch; const int32_t* src_len;
    const int32_t* row_src; const int32_t* row_off; const uint8_t* row_base; const uint8_t* flags;
    uint8_t* out; int64_t out_pitch; int32_t* out_len; int32_t* err;
};

__global__ void __launch_bounds__(256)
mutate_windows_kernel(const MutateParams p) {
    const int r = blockIdx.y;
    const int sr = p.row_src[r];
    const int len = p.src_len[sr];
    const int off = p.row_off[r];
    // a row that cannot be built writes nothing but a zero length (and the error flag): the tokenizer then sees an
    // empty window and never reads the unwritten row
    const bool bad_len = len < 0 || (int64_t)len > p.out_pitch || (int64_t)len > p.src_pitch;
    const bool bad_off = off < 0 || off >= len;
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        if (bad_len) atomicMax(p.err, 1);
        else if (bad_off) atomicMax(p.err, 3);
        p.out_len[r] = (bad_len || bad_off) ? 0 : len;
    }
    if (bad_len || bad_off) return;
    const int b0 = blockIdx.x * kMutSlice;
    if (b0 >= len) return;
    const int b1 = min(len, b0 + kMutSlice);
    const bool rc = p.flags[r] & 1;
    const int q = rc ? len - 1 - off : off;                   // where the base lands in the stored (strand-oriented) row
    const uint8_t base = rc ? comp_base(p.row_base[r]) : p.row_base[r];
    const uint4* s4 = reinterpret_cast<const uint4*>(p.src + (size_t)sr * p.src_pitch);
    uint4* o4 = reinterpret_cast<uint4*>(p.out + (size_t)r * p.out_pitch);
    // whole 16-byte groups up to the one holding the last byte: both pitches are multiples of 16 (host check), so the
    // last group stays inside both rows; bytes past len are copied as they are (they are never read)
    const int g0 = b0 >> 4, g1 = (b1 + 15) >> 4;
    for (int g = g0 + threadIdx.x; g < g1; g += blockDim.x) {
        uint4 v = s4[g];
        if (g == (q >> 4)) {                                  // byte q & 15 of the group (selects: no local memory)
            const int word = (q >> 2) & 3, sh = (q & 3) * 8;
            const uint32_t keep = ~(0xFFu << sh), put = (uint32_t)base << sh;
            v.x = word == 0 ? (v.x & keep) | put : v.x;
            v.y = word == 1 ? (v.y & keep) | put : v.y;
            v.z = word == 2 ? (v.z & keep) | put : v.z;
            v.w = word == 3 ? (v.w & keep) | put : v.w;
        }
        o4[g] = v;
    }
}

int mutate_windows(const uint8_t* src, int64_t src_pitch, const int32_t* src_len, const int32_t* row_src,
                   const int32_t* row_off, const uint8_t* row_base, const uint8_t* flags, int n_rows, uint8_t* out,
                   int64_t out_pitch, int32_t* out_len, int32_t* err, cudaStream_t s) {
    if (n_rows == 0) return 0;
    VF_REQUIRE(src_pitch > 0 && src_pitch % 16 == 0 && out_pitch > 0 && out_pitch % 16 == 0,
               "mutate_windows: pitches must be positive multiples of 16 (src %lld, out %lld)", (long long)src_pitch,
               (long long)out_pitch);
    VF_REQUIRE(((uintptr_t)src & 15) == 0 && ((uintptr_t)out & 15) == 0, "mutate_windows: rows must be 16-byte aligned");
    VF_REQUIRE(n_rows <= 65535, "mutate_windows: %d rows in one call (at most 65535)", n_rows);
    const int64_t span = src_pitch < out_pitch ? src_pitch : out_pitch;   // longest row that can be valid
    MutateParams p{src, src_pitch, src_len, row_src, row_off, row_base, flags, out, out_pitch, out_len, err};
    dim3 grid((unsigned)((span + kMutSlice - 1) / kMutSlice), n_rows);
    mutate_windows_kernel<<<grid, 256, 0, s>>>(p);
    VF_LAUNCH_OK("mutate_windows_kernel launch");
    return 0;
}

// ---------------------------------------------------------------------------------
// BPE-500 tokenisation by ascending-rank sweeps in the base-position domain.
//
// HF tokenizers merges the globally lowest-ranked adjacent pair first (leftmost first among
// equals).  Because the token created by rank r can only be consumed by a merge of rank > r
// (verified on the 482-entry table at load), processing ranks 0..R-1 in order and, within a
// rank, all matches left to right (non-overlapping for self pairs) yields the identical
// segmentation (SURVEY App. D.4).  State: one uint16 per base position — token id at the
// token's first base, DEAD on its remaining bases, SEP on non-IUPAC characters (word
// boundaries, utils/seq.py:36-38).  Tokens are <= 8 bases long, so "next alive symbol" is a
// scan over <= 7 DEAD slots and no compaction is needed between sweeps.
// One CTA per window; symbols in shared memory when the window fits, else in a global
// scratch row (gene windows: ~301 k symbols).  Ranks whose operands are absent from the
// window (per-CTA occupancy counters) are skipped without touching the symbols.
//
// Rank BATCHES.  Consecutive ranks whose symbol sets {left, right, new} are pairwise disjoint
// (and none of which is a self pair) commute: a merge only creates adjacencies that involve its
// own new token, the symbol it kills always sits right behind a symbol of its own left type, so
// no match of another rank of the batch appears, disappears or moves.  Such a run is applied in
// ONE sweep with ONE barrier: every position looks its symbol up in a small table (symbol ->
// rank of the batch whose left operand it is).  The host supplies the batch id of every rank
// (merge_batch, nondecreasing; stage1.merge_batches builds it: 482 ranks -> 162 batches of up
// to 12); null = every rank alone.  Self-pair ranks are always alone (detect / apply phases).
// ---------------------------------------------------------------------------------
constexpr int kMaxBatch = 16;
constexpr uint16_t kDead = 0xFFFF, kSep = 0xFFFE;
constexpr int kBpeSmemSyms = 8192;    // windows up to this many symbols stay in shared memory
constexpr int kMaxVocab = 512;

struct BpeParams {
    const uint8_t* seq; int64_t pitch; const int32_t* len;   // [n_win, pitch] bytes
    const uint16_t* merge_a; const uint16_t* merge_b; const uint16_t* merge_new; int n_merges;
    const uint16_t* merge_batch;                              // [n_merges] nondecreasing batch id per rank, or null (see below)
    uint16_t* scratch; int64_t scratch_pitch;                 // [n_win, scratch_pitch] for long windows (may be null)
    int32_t* out_tokens; int out_pitch; int out_cap;          // [n_win, out_pitch]; first out_cap tokens kept, rest of the row zeroed
    int32_t* out_count;                                       // [n_win] total token count (before truncation)
    int32_t* out_start; int64_t start_pitch;                  // optional [n_win, start_pitch]: first base of every token
    int max_len;                                              // lengths are clamped to this (and to pitch): a corrupt or
                                                              // overflowed length can never index past a row
};

__device__ __forceinline__ uint16_t base_symbol(uint8_t c) {
    // upper-case + 14-letter alphabet A,B,C,D,G,H,K,M,R,S,T,V,W,Y -> ids 4..17; everything else separates words
    if (c >= 'a' && c <= 'z') c -= 32;
    switch (c) {
        case 'A': return 4; case 'B': return 5; case 'C': return 6; case 'D': return 7; case 'G': return 8;
        case 'H': return 9; case 'K': return 10; case 'M': return 11; case 'R': return 12; case 'S': return 13;
        case 'T': return 14; case 'V': return 15; case 'W': return 16; case 'Y': return 17;
        default: return kSep;
    }
}

// Shared by both kernels: the ranks [r0, r0 + nb) of the batch that starts at r0, decided by a whole warp at once
// (lane t looks at rank r0 + t): nb from the nondecreasing batch ids, `ok` = both operands of the lane's rank occur in
// the window (two of them for a self pair).  Every warp of the CTA (of the cluster) computes the same answer from the
// same counters, so the decision is uniform without a barrier.
struct BatchPick { int nb; unsigned okmask; uint16_t a, b, c; bool ok; };
__device__ __forceinline__ BatchPick pick_batch(const BpeParams& p, int r0, const int* cnt, int lane) {
    BatchPick q;
    const int r = r0 + lane;
    const bool in = r < p.n_merges && lane < kMaxBatch;
    uint16_t bid = 0xFFFF;
    if (in) bid = p.merge_batch ? p.merge_batch[r] : (uint16_t)(lane == 0 ? 0 : 0xFFFE);
    const uint16_t bid0 = (uint16_t)__shfl_sync(0xffffffffu, (int)bid, 0);
    const unsigned same = __ballot_sync(0xffffffffu, in && bid == bid0);
    q.nb = __ffs(~same) - 1;                              // ids are nondecreasing: `same` is a prefix mask (lane 0 always set)
    q.a = q.b = q.c = 0;
    q.ok = false;
    if (lane < q.nb) {
        q.a = p.merge_a[r]; q.b = p.merge_b[r]; q.c = p.merge_new[r];
        q.ok = cnt[q.a] != 0 && cnt[q.b] != 0 && !(q.a == q.b && cnt[q.a] < 2);
    }
    q.okmask = __ballot_sync(0xffffffffu, q.ok);
    return q;
}

// One group of four symbols against the batch's table, branch-free up to the (rare) store: v[0..3] = the group,
// v[4..11] = the eight slots behind it (a token is at most 8 bases long, so the next alive symbol of v[e] is among
// v[e+1 .. e+8]).  tab[sy] = right operand | new token << 16 of the batch rank whose LEFT operand is sy (0xFFFFFFFF: none).
// Calls hit(e, off, packed) for every match: slot e of the group merges with the alive symbol `off` slots behind it.
// Reading the twelve slots once is sound: a left operand is never killed during its own batch, the alive symbol right
// behind it can only be killed by this very match, and a symbol that equals the wanted right operand is not a left
// operand of the batch (disjoint symbol sets), so it cannot change under us.
template <class Hit>
__device__ __forceinline__ void sweep_group(const uint16_t (&v)[12], const uint32_t* tab, Hit&& hit) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
        const uint32_t sy = v[e];
        if (sy >= (uint32_t)kMaxVocab) continue;                       // DEAD / SEP (cheap, convergent enough)
        const uint32_t t = tab[sy];
        if (t == 0xFFFFFFFFu) continue;                                 // not a left operand of this batch
        uint32_t nxt = kSep, off = 0;
#pragma unroll
        for (int d = 8; d >= 1; --d) {                                  // nearest alive slot wins (selects, no branches)
            const bool alive = v[e + d] != kDead;
            nxt = alive ? (uint32_t)v[e + d] : nxt;
            off = alive ? (uint32_t)d : off;
        }
        if (nxt == (t & 0xFFFFu)) hit(e, (int)off, t);
    }
}
__device__ __forceinline__ void unpack12(uint2 a, uint2 b, uint2 c, uint16_t (&v)[12]) {
    v[0] = (uint16_t)a.x; v[1] = (uint16_t)(a.x >> 16); v[2] = (uint16_t)a.y; v[3] = (uint16_t)(a.y >> 16);
    v[4] = (uint16_t)b.x; v[5] = (uint16_t)(b.x >> 16); v[6] = (uint16_t)b.y; v[7] = (uint16_t)(b.y >> 16);
    v[8] = (uint16_t)c.x; v[9] = (uint16_t)(c.x >> 16); v[10] = (uint16_t)c.y; v[11] = (uint16_t)(c.y >> 16);
}

__global__ void bpe_tokenize_kernel(const BpeParams p) {
    extern __shared__ __align__(16) uint16_t s_sym[];   // this call's longest window, rounded up to 64 symbols
    __shared__ int s_cnt[kMaxVocab];                    // alive symbols per token id
    __shared__ int s_warp_tot[32];
    __shared__ int s_any;
    __shared__ uint32_t s_tab[kMaxVocab];               // left operand -> right operand | new token << 16 of its batch rank
    __shared__ uint8_t s_rk[kMaxVocab];                 // left operand -> index of that rank within the batch
    __shared__ int s_mcnt[kMaxBatch];
    const int w = blockIdx.x;
    const int n = max(0, min(p.len[w], p.max_len));
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31;
    uint16_t* sym = s_sym;
    const uint8_t* src = p.seq + (size_t)w * p.pitch;

    for (int i = tid; i < kMaxVocab; i += nt) { s_cnt[i] = 0; s_tab[i] = 0xFFFFFFFFu; }
    __syncthreads();
    const int n4 = (n + 3) >> 2;                          // the sweeps read 4 + 8 symbols at a time: pad with SEP
    for (int i = tid; i < 4 * n4 + 8; i += nt) {
        const uint16_t b = i < n ? base_symbol(src[i]) : kSep;
        sym[i] = b;
        if (b != kSep) atomicAdd(&s_cnt[b], 1);
    }
    __syncthreads();

    for (int r0 = 0; r0 < p.n_merges;) {
        const BatchPick q = pick_batch(p, r0, s_cnt, lane);
        const int r1 = r0 + q.nb;
        if (!q.okmask) { r0 = r1; continue; }             // uniform: same counters, stable since the last barrier
        const uint16_t a = (uint16_t)__shfl_sync(0xffffffffu, (int)q.a, 0), b = (uint16_t)__shfl_sync(0xffffffffu, (int)q.b, 0),
                       c = (uint16_t)__shfl_sync(0xffffffffu, (int)q.c, 0);
        if (a != b) {
            // every thread must have taken the skip decision above before any occupancy counter moves
            __syncthreads();
            if (tid < q.nb) {
                if (q.ok) { s_tab[q.a] = (uint32_t)q.b | ((uint32_t)q.c << 16); s_rk[q.a] = (uint8_t)tid; }
                s_mcnt[tid] = 0;
            }
            __syncthreads();
            // matches of the batch's ranks can never share a symbol: apply immediately
            const uint2* sym4 = reinterpret_cast<const uint2*>(sym);
            for (int g = tid; g < n4; g += nt) {
                const uint2 w4 = sym4[g];
                if ((w4.x & w4.y) == 0xFFFFFFFFu) continue;           // four DEAD slots
                uint16_t v[12];
                unpack12(w4, sym4[g + 1], sym4[g + 2], v);
                sweep_group(v, s_tab, [&](int e, int off, uint32_t t) {
                    const int i = 4 * g + e;
                    sym[i] = (uint16_t)(t >> 16); sym[i + off] = kDead;
                    atomicAdd(&s_mcnt[s_rk[v[e]]], 1);
                });
            }
            __syncthreads();
            if (tid < q.nb) {                             // symbol sets are disjoint: no two threads touch one counter
                const int m = s_mcnt[tid];
                if (m) { s_cnt[q.c] += m; s_cnt[q.a] -= m; s_cnt[q.b] -= m; }
                s_tab[q.a] = 0xFFFFFFFFu;
            }
        } else {
            int merged = 0;
            // self pair: within a run of consecutive a's merge (1st,2nd), (3rd,4th), ... -> decide from the
            // parity of the number of a's that precede i in its run; detect first, apply after a barrier
            // (the tentative mark c|0x8000 is treated as `a` by concurrent scans, so marking is race-free)
            const uint16_t mark = (uint16_t)(c | 0x8000);
            if (tid == 0) s_any = 0;
            __syncthreads();
            for (int i = tid; i < n; i += nt) {
                if (sym[i] != a) continue;
                int k = 0, qq = i - 1;
                for (;;) {
                    while (qq >= 0 && sym[qq] == kDead) --qq;
                    if (qq < 0) break;
                    const uint16_t sq = sym[qq];
                    if (sq != a && sq != mark) break;
                    ++k; --qq;
                }
                if (k & 1) continue;                     // i is the right half of the previous pair
                int j = i + 1;
                while (j < n && sym[j] == kDead) ++j;
                if (j < n && (sym[j] == a || sym[j] == mark)) { sym[i] = mark; s_any = 1; }
            }
            __syncthreads();
            if (s_any) {
                for (int i = tid; i < n; i += nt) {
                    if (sym[i] != mark) continue;
                    int j = i + 1;
                    while (j < n && sym[j] == kDead) ++j;
                    sym[j] = kDead; sym[i] = c; ++merged;
                }
            }
            if (merged) { atomicAdd(&s_cnt[c], merged); atomicSub(&s_cnt[a], 2 * merged); }
        }
        __syncthreads();
        r0 = r1;
    }

    // ---- ordered compaction: each thread owns a contiguous segment ----
    const int per = (n + nt - 1) / nt;
    const int b0 = min(n, tid * per), b1 = min(n, b0 + per);
    int mine = 0;
    for (int i = b0; i < b1; ++i) mine += (sym[i] < kSep);
    int incl = mine;
    const int wid = tid >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
    if (lane == 31) s_warp_tot[wid] = incl;
    __syncthreads();
    if (wid == 0) {
        int v = lane < (nt >> 5) ? s_warp_tot[lane] : 0;
        int inc2 = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int u = __shfl_up_sync(0xffffffffu, inc2, o); if (lane >= o) inc2 += u; }
        s_warp_tot[lane] = inc2 - v;                       // exclusive warp offsets
        if (lane == 31) s_any = inc2;                      // grand total
    }
    __syncthreads();
    int o = s_warp_tot[wid] + incl - mine;
    const int total = s_any;
    int32_t* out = p.out_tokens + (size_t)w * p.out_pitch;
    int32_t* ost = p.out_start ? p.out_start + (size_t)w * p.start_pitch : nullptr;
    for (int i = b0; i < b1; ++i) {
        const uint16_t sy = sym[i];
        if (sy < kSep) {
            if (o < p.out_cap) out[o] = sy;
            if (ost) ost[o] = i;
            ++o;
        }
    }
    for (int i = min(total, p.out_cap) + tid; i < p.out_pitch; i += nt) out[i] = 0;    // <pad> = 0
    if (tid == 0) p.out_count[w] = total;
}

// ---------------------------------------------------------------------------------
// Long windows (gene windows, ~301 k symbols): one thread-block CLUSTER per window.  Each CTA keeps a contiguous
// segment of the symbol array in its own shared memory; neighbours are reached through distributed shared memory
// (forward "next alive symbol" scans cross a segment boundary by at most 7 slots, self-pair run scans by the run
// length).  One cluster barrier per applied rank (two for self pairs).  The per-token-id occupancy counters that
// drive the uniform skip decision are replicated in every CTA and kept identical by gathering the per-CTA merge
// counts of every applied sweep through DSMEM right after that sweep's cluster barrier.
// ---------------------------------------------------------------------------------

template <int kBpeCluster>
__global__ void __launch_bounds__(1024, 1)
bpe_tokenize_cluster_kernel(const BpeParams p, const int seg_cap) {
    namespace cg = cooperative_groups;
    cg::cluster_group cluster = cg::this_cluster();
    extern __shared__ __align__(16) uint16_t s_sym[];    // seg_cap symbols of this CTA's segment
    __shared__ int s_cnt[2][kMaxVocab];                  // replicated occupancy counters (double buffered)
    __shared__ uint16_t* s_peer[kBpeCluster];
    __shared__ int* s_peer_cnt[kBpeCluster];
    __shared__ int s_segcnt[kBpeCluster];
    __shared__ int s_warp_tot[32];
    const int rank = (int)cluster.block_rank();
    const int w = blockIdx.x / kBpeCluster;
    const int n = max(0, min(p.len[w], p.max_len));
    const int tid = threadIdx.x, nt = blockDim.x;
    const int seg = (max(8, (n + kBpeCluster - 1) / kBpeCluster) + 7) & ~7;   // multiple of 8, <= seg_cap (host guarantees)
    const int lo = min(n, rank * seg), hi = min(n, lo + seg);
    const uint8_t* src = p.seq + (size_t)w * p.pitch;

    if (tid < kBpeCluster) {
        s_peer[tid] = cluster.map_shared_rank(s_sym, tid);
        s_peer_cnt[tid] = cluster.map_shared_rank(&s_cnt[0][0], tid);
    }
    for (int i = tid; i < 2 * kMaxVocab; i += nt) (&s_cnt[0][0])[i] = 0;
    __syncthreads();
    // local histogram in replica 0 slots of a scratch copy: count into registers-free smem then publish
    __shared__ int s_hist[32];                            // base ids 4..17 only
    if (tid < 32) s_hist[tid] = 0;
    cluster.sync();                                       // every CTA's counters are zeroed before anyone publishes
    for (int i = lo + tid; i < lo + (hi < n ? hi - lo : ((hi - lo + 3) & ~3) + 8); i += nt) {   // (4 + 8 slot reads: SEP padding)
        const uint16_t b = i < hi ? base_symbol(src[i]) : kSep;
        s_sym[i - lo] = b;
        if (b != kSep) atomicAdd(&s_hist[b], 1);
    }
    __syncthreads();
    if (tid < 32 && s_hist[tid] != 0) {
        for (int c = 0; c < kBpeCluster; ++c) {
            atomicAdd(s_peer_cnt[c] + tid, s_hist[tid]);
        }
    }
    cluster.sync();

    auto LD = [&](int pos) -> uint16_t {
        if (pos >= lo && pos < hi) return s_sym[pos - lo];
        const int c = pos / seg;
        return s_peer[c][pos - c * seg];
    };
    auto ST = [&](int pos, uint16_t v) {
        if (pos >= lo && pos < hi) { s_sym[pos - lo] = v; return; }
        const int c = pos / seg;
        s_peer[c][pos - c * seg] = v;
    };
    // Per applied batch every CTA posts the merge counts of the batch's ranks in its own shared memory (slot k&1); after
    // the cluster barrier each CTA gathers the 8 count vectors through DSMEM and updates its private replica of the
    // counters, so all replicas stay identical without remote atomics.
    __shared__ int s_pub[2][kMaxBatch];
    __shared__ int s_mcnt[2][kMaxBatch];
    __shared__ uint32_t s_tab[kMaxVocab];                 // left operand -> right operand | new token << 16 of its batch rank
    __shared__ uint8_t s_rk[kMaxVocab];                   // left operand -> index of that rank within the batch
    for (int i = tid; i < kMaxVocab; i += nt) s_tab[i] = 0xFFFFFFFFu;
    if (tid < 2 * kMaxBatch) (&s_mcnt[0][0])[tid] = 0;
    __syncthreads();
    const int lane = tid & 31;
    const int len4 = (hi - lo + 3) >> 2;                  // (segment starts are multiples of 8; slots past hi hold SEP)
    // slots of the local array the 12-slot reads may touch: an inner segment ends where the next CTA's begins; the last
    // segment (and an empty one) is followed by SEP padding written below
    const int local_slots = hi < n ? hi - lo : ((hi - lo + 3) & ~3) + 8;
    int k = 0;                                            // applied batches so far (cluster-uniform)
    for (int r0 = 0; r0 < p.n_merges;) {
        const BatchPick q = pick_batch(p, r0, s_cnt[0], lane);   // uniform over the whole cluster (identical replicas)
        const int r1 = r0 + q.nb, nb = q.nb;
        if (!q.okmask) { r0 = r1; continue; }
        const uint16_t a = (uint16_t)__shfl_sync(0xffffffffu, (int)q.a, 0), b = (uint16_t)__shfl_sync(0xffffffffu, (int)q.b, 0),
                       c = (uint16_t)__shfl_sync(0xffffffffu, (int)q.c, 0);
        const bool self_pair = a == b;                    // (always a batch of its own)
        int* mc = s_mcnt[k & 1];
        if (!self_pair) {
            if (tid < nb && q.ok) { s_tab[q.a] = (uint32_t)q.b | ((uint32_t)q.c << 16); s_rk[q.a] = (uint8_t)tid; }
            __syncthreads();
            const uint2* sym4 = reinterpret_cast<const uint2*>(s_sym);
            for (int g = tid; g < len4; g += nt) {
                const uint2 w4 = sym4[g];
                if ((w4.x & w4.y) == 0xFFFFFFFFu) continue;           // four DEAD slots
                uint16_t v[12];
                if (4 * g + 12 <= local_slots) {
                    unpack12(w4, sym4[g + 1], sym4[g + 2], v);
                } else {                                              // the look-ahead leaves this CTA's segment (last groups)
                    unpack12(w4, make_uint2(0, 0), make_uint2(0, 0), v);
#pragma unroll
                    for (int x = 4; x < 12; ++x) { const int pos = lo + 4 * g + x; v[x] = pos < n ? LD(pos) : kSep; }
                }
                sweep_group(v, s_tab, [&](int e, int off, uint32_t t) {
                    const int i = lo + 4 * g + e;
                    s_sym[i - lo] = (uint16_t)(t >> 16); ST(i + off, kDead);
                    atomicAdd(&mc[s_rk[v[e]]], 1);
                });
            }
        } else {
            int merged = 0;
            const uint16_t mark = (uint16_t)(c | 0x8000);
            for (int i = lo + tid; i < hi; i += nt) {
                if (s_sym[i - lo] != a) continue;
                int kk = 0, qq = i - 1;
                for (;;) {
                    while (qq >= 0 && LD(qq) == kDead) --qq;
                    if (qq < 0) break;
                    const uint16_t sq = LD(qq);
                    if (sq != a && sq != mark) break;
                    ++kk; --qq;
                }
                if (kk & 1) continue;
                int j = i + 1;
                while (j < n && LD(j) == kDead) ++j;
                if (j < n) { const uint16_t sj = LD(j); if (sj == a || sj == mark) s_sym[i - lo] = mark; }
            }
            cluster.sync();
            for (int i = lo + tid; i < hi; i += nt) {
                if (s_sym[i - lo] != mark) continue;
                int j = i + 1;
                while (j < n && LD(j) == kDead) ++j;
                ST(j, kDead); s_sym[i - lo] = c; ++merged;
            }
            if (merged) atomicAdd(&mc[0], merged);
        }
        __syncthreads();
        if (tid < kMaxBatch) {
            s_pub[k & 1][tid] = tid < nb ? mc[tid] : 0;
            s_mcnt[(k + 1) & 1][tid] = 0;
            if (tid < nb && !self_pair) s_tab[q.a] = 0xFFFFFFFFu;
        }
        cluster.sync();                                   // all merges of this batch + every CTA's counts are visible
        constexpr int kRanksPerWarp = 32 / kBpeCluster;   // lanes = (ranks of the warp) x (CTAs of the cluster)
        if (tid < 32 * kMaxBatch / kRanksPerWarp) {
            const int wq = tid >> 5;
            const int rr = kRanksPerWarp * wq + lane / kBpeCluster, cta = lane % kBpeCluster;
            int v = rr < nb ? cluster.map_shared_rank(&s_pub[0][0], cta)[(k & 1) * kMaxBatch + rr] : 0;
#pragma unroll
            for (int o = kBpeCluster / 2; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
            if (cta == 0 && rr < nb && v != 0) {          // symbol sets of a batch are disjoint: one writer per counter
                const uint16_t ra = p.merge_a[r0 + rr], rb = p.merge_b[r0 + rr], rc = p.merge_new[r0 + rr];
                s_cnt[0][rc] += v;
                if (ra == rb) s_cnt[0][ra] -= 2 * v; else { s_cnt[0][ra] -= v; s_cnt[0][rb] -= v; }
            }
        }
        __syncthreads();
        ++k;
        r0 = r1;
    }
    cluster.sync();                                       // no CTA may exit (or reuse s_pub) while peers still read it

    // ---- ordered compaction of this CTA's segment; token offset = alive symbols of the lower-ranked segments ----
    const int len_seg = hi - lo;
    const int per = (len_seg + nt - 1) / nt;
    const int b0 = min(len_seg, tid * per), b1 = min(len_seg, b0 + per);
    int mine = 0;
    for (int i = b0; i < b1; ++i) mine += (s_sym[i] < kSep);
    int incl = mine;
    const int wid = tid >> 5;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
    if (lane == 31) s_warp_tot[wid] = incl;
    __syncthreads();
    if (wid == 0) {
        const int v = lane < (nt >> 5) ? s_warp_tot[lane] : 0;
        int inc2 = v;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) { const int u = __shfl_up_sync(0xffffffffu, inc2, o); if (lane >= o) inc2 += u; }
        s_warp_tot[lane] = inc2 - v;
        if (lane == 31) {
            for (int c2 = 0; c2 < kBpeCluster; ++c2) cluster.map_shared_rank(&s_segcnt[0], c2)[rank] = inc2;
        }
    }
    cluster.sync();
    int base = 0, total = 0;
    for (int c2 = 0; c2 < kBpeCluster; ++c2) { if (c2 < rank) base += s_segcnt[c2]; total += s_segcnt[c2]; }
    int o = base + s_warp_tot[wid] + incl - mine;
    int32_t* out = p.out_tokens + (size_t)w * p.out_pitch;
    int32_t* ost = p.out_start ? p.out_start + (size_t)w * p.start_pitch : nullptr;
    for (int i = b0; i < b1; ++i) {
        const uint16_t sy = s_sym[i];
        if (sy < kSep) {
            if (o < p.out_cap) out[o] = sy;
            if (ost) ost[o] = lo + i;
            ++o;
        }
    }
    for (int i = min(total, p.out_cap) + rank * nt + tid; i < p.out_pitch; i += nt * kBpeCluster) out[i] = 0;
    if (rank == 0 && tid == 0) p.out_count[w] = total;
    cluster.sync();                                       // keep every CTA's shared memory alive until all peers are done
}

int bpe_tokenize(const uint8_t* seq, int64_t pitch, const int32_t* len, int n_win, int max_len,
                 const uint16_t* merge_a, const uint16_t* merge_b, const uint16_t* merge_new,
                 const uint16_t* merge_batch, int n_merges, uint16_t* scratch, int64_t scratch_pitch, int32_t* out_tokens, int out_pitch, int out_cap,
                 int32_t* out_count, int32_t* out_start, int64_t start_pitch, int block_threads, cudaStream_t s) {
    if (n_win == 0) return 0;
    VF_REQUIRE(out_cap <= out_pitch, "bpe_tokenize: out_cap %d > out_pitch %d", out_cap, out_pitch);
    VF_REQUIRE(out_start == nullptr || start_pitch >= max_len, "bpe_tokenize: start_pitch too small");
    BpeParams p{seq, pitch, len, merge_a, merge_b, merge_new, n_merges, merge_batch, scratch, scratch_pitch,
                out_tokens, out_pitch, out_cap, out_count, out_start, start_pitch,
                (int)(pitch < (int64_t)max_len ? pitch : (int64_t)max_len)};
    if (max_len > kBpeSmemSyms) {
        // cluster path: CL CTAs per window, segment of the symbol array per CTA in shared memory.  16-CTA clusters (non
        // portable size, VF_BPE_CLUSTER=16) put a slab's 8 gene windows on 128 SMs instead of 64 but the cluster barrier
        // grows faster than the sweep shrinks: 3.1 ms against 2.6-2.8 ms per slab with the portable size (the default).
        // A call with few windows (single-gene latency) cannot fill the machine either way: there the larger cluster wins
        // (one 301 k-symbol window: 1.1 ms against 1.8 ms).
        static int cl_env = -1;
        if (cl_env < 0) {
            const char* e = getenv("VF_BPE_CLUSTER");
            cl_env = e ? atoi(e) : 0;
        }
        const int cl = (cl_env == 8 || cl_env == 16) ? cl_env : (n_win <= 4 ? 16 : 8);
        auto launch = [&](auto kern, int CL) -> int {
            const int seg_cap = (max_len + CL - 1) / CL + 32;
            const size_t smem = (size_t)seg_cap * sizeof(uint16_t);
            VF_REQUIRE(smem <= 200 * 1024, "bpe_tokenize: window of %d symbols exceeds the cluster kernel's capacity", max_len);
            VF_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            if (CL > 8) VF_CUDA_OK(cudaFuncSetAttribute(kern, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
            cudaLaunchConfig_t cfg = {};
            cfg.gridDim = dim3(n_win * CL); cfg.blockDim = dim3(1024); cfg.dynamicSmemBytes = smem; cfg.stream = s;
            cudaLaunchAttribute at[1];
            at[0].id = cudaLaunchAttributeClusterDimension;
            at[0].val.clusterDim.x = CL; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
            cfg.attrs = at; cfg.numAttrs = 1;
            VF_CUDA_OK(cudaLaunchKernelEx(&cfg, kern, p, seg_cap));
            VF_LAUNCH_OK("bpe_tokenize_cluster_kernel launch");
            return 0;
        };
        return cl == 16 ? launch(bpe_tokenize_cluster_kernel<16>, 16) : launch(bpe_tokenize_cluster_kernel<8>, 8);
    }
    // Block size is a pure performance hint (typical window length); any value works for any window.  Short windows are
    // latency bound (one barrier per rank batch, a handful of symbols per thread): what pays is WINDOWS IN FLIGHT, so
    // the shared-memory footprint is sized to this call's longest window (not the 8192-symbol maximum) and cCRE-sized
    // windows run on 64 threads — 32 resident CTAs per SM instead of 11.
    const int threads = (block_threads == 64 || block_threads == 128 || block_threads == 256 || block_threads == 512 ||
                         block_threads == 1024) ? block_threads : (max_len <= 1024 ? 64 : 1024);
    const size_t smem = (size_t)((max_len + 16 + 63) / 64 * 64) * sizeof(uint16_t);   // + the sweeps' 8-slot look-ahead
    static size_t attr_smem1 = 0;
    if (smem > 40 * 1024 && smem > attr_smem1) {
        VF_CUDA_OK(cudaFuncSetAttribute(bpe_tokenize_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        attr_smem1 = smem;
    }
    bpe_tokenize_kernel<<<n_win, threads, smem, s>>>(p);
    VF_LAUNCH_OK("bpe_tokenize_kernel launch");
    return 0;
}

}  // namespace vf
