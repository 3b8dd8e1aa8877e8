// vf_attention_mc.cu — variable-length non-causal attention on the 5th-gen tensor cores, TWO CTAs PER SM.
//
// Same contract as vf_attention_tc.cu (flash_attn varlen call sites: seq2reg/modules.py:159-171,
// seq2gene/modules/layers.py:372-467): softmax((q·k)/sqrt(hd) - slope_h*|i + Sk - Sq - j|) v, fp32 statistics.
//
// Why a second kernel: at head_dim 48/64 attention is bound by the softmax (one ex2 per score, 16/clk/SM), not by
// the tensor pipe, and with one CTA per SM the 8 softmax warps (2 per scheduler) leave most issue slots and ~60 % of
// the MUFU pipe idle behind TMEM-load, barrier and MUFU latencies (ncu: profiles/r01_attention_tc_*).  This kernel
// halves every per-CTA resource (256 TMEM columns, ~106 KB shared memory, 2 query tiles per work item) so that two
// CTAs are co-resident: 16 softmax warps per SM in four independent pipelines whose bubbles overlap.
//
// One CTA = 384 threads = 3 warpgroups:
//   warp 0      TMA producer: Q tiles of the item's (up to) two SLOTS, K / V blocks of 64 keys through 3- / 2-stage
//               rings; all tiles are [rows, 64 cols] bf16, SWIZZLE_128B (hd=48 over-fetches 16 columns never read)
//   warps 1, 2  tcgen05.mma issuers, ONE PER SLOT (neither slot waits behind the other's barriers):
//               S_s = Q_s K^T (M128 x N64 x K=hd) into slot s's TMEM score buffer, issued as soon as the previous
//               scores are in registers; O_s += P_s V (M128 x N=hd x K64), P from shared memory (K-major), V as an
//               MN-major operand
//   warp 3      idle (warpgroup 0 hands its registers to the softmax warps with setmaxnreg)
//   warps 4-11  two softmax warpgroups, warpgroup s owns slot s: ONE THREAD PER QUERY ROW, the 64 scores of a row
//               come straight from TMEM (tcgen05.ld 32x32b) into registers; the 8 warps never synchronise with each
//               other, only with their slot's issuer through mbarriers
// A work item is (head, two slots); a slot is a 128-row query tile of some sequence, described by a host-built record
// {first query row, valid rows, first key row, keys, ALiBi position of row 0} (absolute row numbers: no cu_seqlens
// lookups on the device).  Two slots with the same key range share one K/V stream (long sequences: every K/V block
// feeds two query tiles); slots of different sequences (short sequences, <= 128 rows: seq2reg windows) stream their
// own K/V, so both warpgroups stay busy either way.
//
// Softmax: single pass with a LAZY reference maximum (exact arithmetic): P = exp2(x - m_ref) may reach 2^8 before
// m_ref is raised; raising rescales l and (through tcgen05.ld/st) O_s by exp2(m_old - m_new).  The whole 64-key
// score row is in registers before anything is written, so a raise never needs a restart.  The affine part of the
// exponent (scale, -m_ref, and away from the diagonal the ALiBi term, which is linear in the key index there) is
// folded into one or two FFMA per score.
// TMEM (256 columns per CTA): [64 s, +64) scores of slot s, [128 + 64 s, +64) O_s.
#include <cuda.h>

#include "vf_common.cuh"
#include "vf_internal.h"

namespace vf {
namespace mc {

constexpr int kQT = 128;            // query rows per slot
constexpr int kKB = 64;             // keys per block
constexpr int kKStages = 3, kVStages = 2;
constexpr uint32_t kQBytes = 128 * 64 * 2;                    // one [128 x 64] bf16 tile (Q tile, P buffer)
constexpr uint32_t kKvBytes = kKB * 64 * 2;                   // one [64 keys x 64] bf16 tile
constexpr int kThreads = 384;
constexpr int kFirstSoftmaxWarp = 4;
constexpr uint32_t kTmemCols = 256;
constexpr size_t kSmem = 1024 + 2 * kQBytes + (size_t)(kKStages + kVStages) * kKvBytes + 2 * kQBytes + 384;
constexpr float kLazyThreshold = 8.0f;      // log2 units: P stays below 2^8 between reference-max updates

// one slot of a work item (32 bytes): nrows == 0 marks an empty slot
struct SlotRec { int qrow, nrows, krow, Sk, qpos0, pad0, pad1, pad2; };

struct Params {
    const SlotRec* slots;                         // [n_items][2]
    int n_items, heads;
    __nv_bfloat16* o; int ldo;
    const float* slopes;
    float scale_log2;
};

constexpr uint32_t kRegsLo = 32;    // producer / MMA issuer warpgroup; 128 * kRegsLo + 256 * kRegsHi <= 384 * 80
constexpr uint32_t kRegsHi = 104;   // softmax warpgroups

__device__ __forceinline__ float ex2_approx(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

// O_s row *= corr, in tensor memory, 8 columns at a time (few live registers: the caller holds a whole score row).
// Warp-collective; lanes that need no change pass corr = 1.
template <int HD>
__device__ __forceinline__ void rescale_o(uint32_t o_addr, float corr) {
#pragma unroll 1
    for (int c = 0; c < HD; c += 8) {
        uint32_t u[8];
        tmem_ld_32x8(o_addr + c, u);
        tmem_ld_wait();
#pragma unroll
        for (int e = 0; e < 8; ++e) u[e] = __float_as_uint(__uint_as_float(u[e]) * corr);
        tmem_st_32x8(o_addr + c, u);
    }
    tmem_st_wait();
}

// Packed fp32 pairs (sm_100 FFMA2 / FADD2: one issue slot for two lanes of arithmetic) and the 3-input maximum.  The
// softmax warps are bound by the instructions they issue, not by any single pipe, so the per-score count is what
// matters: 3.0 (no positional term), 3.5 (ALiBi off the diagonal), 4.5 (diagonal block) instead of 4.5 / 5.5 / 7.5.
__device__ __forceinline__ float max3(float a, float b, float c) {
    float d;
    asm("max.f32 %0, %1, %2, %3;" : "=f"(d) : "f"(a), "f"(b), "f"(c));
    return d;
}

// {2i, 2i+1} and its negative as packed fp32 pairs (little-endian: low word = first key)
#define VF_KP(i) (((uint64_t)__builtin_bit_cast(uint32_t, (float)(2 * (i) + 1)) << 32) | __builtin_bit_cast(uint32_t, (float)(2 * (i))))
#define VF_NKP(i) (((uint64_t)__builtin_bit_cast(uint32_t, -(float)(2 * (i) + 1)) << 32) | __builtin_bit_cast(uint32_t, -(float)(2 * (i))))
#define VF_ROW8(M, b) M(b), M(b + 1), M(b + 2), M(b + 3), M(b + 4), M(b + 5), M(b + 6), M(b + 7)
__constant__ uint64_t kKeyPair[32] = {VF_ROW8(VF_KP, 0), VF_ROW8(VF_KP, 8), VF_ROW8(VF_KP, 16), VF_ROW8(VF_KP, 24)};
__constant__ uint64_t kNegKeyPair[32] = {VF_ROW8(VF_NKP, 0), VF_ROW8(VF_NKP, 8), VF_ROW8(VF_NKP, 16), VF_ROW8(VF_NKP, 24)};

// First pass over one row of a 128 x 64 score tile.  Exponent of a score (base 2, against the current reference
// `base`): x = raw * scale + bias - base.  Returns the row maximum of x.
// MODE 0: no positional term: the maximum is taken on the raw scores, r is left as it is and the affine map is applied
//         in the exponential pass (where it overlaps the MUFU pipe).
// MODE 1: ALiBi with the whole 64-key block on one side of the diagonal for every row of the warp: the bias is linear
//         in the key index.
// MODE 2: ALiBi across the diagonal.   MODE 3: MODE 2 + tail mask (keys >= nvalid -> -inf); slope may be 0; works on
//         whole 16-key groups up to nvalid only.
// Modes 1-3 write x back into r.  Key index pairs come from constant memory (operands of the packed instructions):
// no running sums, the 32 pairs stay independent.
template <int MODE>
__device__ __forceinline__ float exponents(uint32_t (&r)[64], float scale, float slope, float d0, float base, int nvalid) {
    float m0 = -INFINITY, m1 = -INFINITY;
    if constexpr (MODE == 0) {
#pragma unroll
        for (int i = 0; i < 32; i += 2) {
            m0 = max3(m0, __uint_as_float(r[2 * i]), __uint_as_float(r[2 * i + 1]));
            m1 = max3(m1, __uint_as_float(r[2 * i + 2]), __uint_as_float(r[2 * i + 3]));
        }
        return fmaf(fmaxf(m0, m1), scale, -base);               // scale > 0
    } else {
        const uint64_t scale2 = f2_pack(scale, scale);
        uint64_t sl2 = 0, c2 = 0, d2 = 0;
        if constexpr (MODE == 1) {
            // |d0 - e| = +-(d0 - e) for the whole block: bias(e) = -slope |d0| - base + sl e
            const float sl = d0 > 0.f ? slope : -slope;
            const float c = fmaf(-slope, fabsf(d0), -base);
            sl2 = f2_pack(sl, sl);
            c2 = f2_pack(c, c);
        } else {
            d2 = f2_pack(d0, d0);
        }
#pragma unroll
        for (int i = 0; i < 32; ++i) {
            if (MODE == 3 && (i & 7) == 0 && 2 * i >= nvalid) break;   // whole groups past the end
            uint64_t bias2;
            if constexpr (MODE == 1) {
                bias2 = f2_fma(kKeyPair[i], sl2, c2);
            } else {
                float t0, t1;
                f2_unpack(f2_add(d2, kNegKeyPair[i]), t0, t1);                          // d0 - e
                bias2 = f2_pack(fmaf(-slope, fabsf(t0), -base), fmaf(-slope, fabsf(t1), -base));
            }
            float x0, x1;
            f2_unpack(f2_fma(f2_pack(r[2 * i], r[2 * i + 1]), scale2, bias2), x0, x1);
            if constexpr (MODE == 3) {
                if (2 * i >= nvalid) x0 = -INFINITY;
                if (2 * i + 1 >= nvalid) x1 = -INFINITY;
            }
            r[2 * i] = __float_as_uint(x0);
            r[2 * i + 1] = __float_as_uint(x1);
            if (i & 1) m1 = max3(m1, x0, x1);
            else m0 = max3(m0, x0, x1);
        }
        return fmaxf(m0, m1);
    }
}

// Everything after the first pass: lazy raise of the reference maximum (O_s rescaled in TMEM), exponentials, P -> shared
// memory (bf16, K-major SWIZZLE_128B: 16-byte chunk index XOR (row & 7)), running row sum.
// KIND 0: r holds raw scores (exponents<0>).  KIND 1: r holds x.  KIND 3: x, tail block (groups past nvalid: P = 0; the
// issuer still runs all four P V steps).
// The four warps of a slot meet different ALiBi block kinds in the same tile, so modes 1 and 2 share ONE copy of this
// code (a copy per mode was measured 20 % slower on 201-token sequences: instruction fetch); tails and the no-bias
// kind are uniform over the slot and get their own.
template <int HD, int KIND, bool PRESWZ>
__device__ __forceinline__ void softmax_rest(uint32_t (&r)[64], float mx, float base, float scale, int nvalid,
                                             uint32_t o_addr, bool first, SmemBar p_empty_bar, uint32_t p_empty_parity,
                                             float& m_ref, float& l, uint32_t p_row, int row, float gate) {
    // The PV of this slot's previous step is the last reader of the P buffer and the last writer of O_s.  It was issued
    // at the end of the previous tile, so waiting for it HERE (before the exponentials) can stall every softmax warp
    // of the slot; only a raise of the reference maximum needs it this early (it rescales O_s).  The common path
    // takes the exponentials first, packed into the registers the scores occupied, and waits right before the stores.
    bool waited = false;
    float delta = 0.f;
    // Only LIVE rows vote: the rows of a tile past the sequence's last query row hold whatever follows in the q tensor
    // (rows of other sequences), and a raise they triggered would change the rounding of the live rows' probabilities —
    // results would depend on what a sequence is batched with.  (A dead row may overflow; nobody reads it.)
    // (`gate` = kLazyThreshold for a live row, +inf for a dead one: one register the caller sets once per item; a bool
    // was recomputed from SR_TID at every tile.)
    if (first || __any_sync(0xffffffffu, mx > gate)) {
        // first tile: the exact row maximum becomes the reference (may be negative).  later: raise by max(mx, 0).
        delta = first ? mx : fmaxf(mx, 0.f);
        const float corr = first ? 0.f : ex2_approx(-delta);
        l *= corr;
        if (!first) {
            mbar_wait(p_empty_bar, p_empty_parity);
            tc_fence_after();
            waited = true;
            rescale_o<HD>(o_addr, corr);
        }
        m_ref = base + delta;
        if constexpr (KIND != 0) {
            const uint64_t nd2 = f2_pack(-delta, -delta);
#pragma unroll
            for (int i = 0; i < 32; ++i) {
                if (KIND == 3 && (i & 7) == 0 && 2 * i >= nvalid) break;
                f2_unpack(f2_add(f2_pack(r[2 * i], r[2 * i + 1]), nd2), r[2 * i], r[2 * i + 1]);
            }
        }
    }
    // (Serialising this section per scheduler with a lock — to break up convoys on the MUFU pipe — was measured 1.6x
    // SLOWER: one warp alone does not keep the pipe busy.)
    const uint64_t scale2 = f2_pack(scale, scale);
    const float c0 = -(base + delta);
    const uint64_t c2 = f2_pack(c0, c0);
    uint64_t acc0 = f2_pack(0.f, 0.f), acc1 = acc0;
    int ndone = 32;
#pragma unroll
    for (int i = 0; i < 32; ++i) {                            // r[i] <- bf16x2(p[2i], p[2i+1]); i <= 2i: in place
        if (KIND == 3 && (i & 7) == 0 && 2 * i >= nvalid) { ndone = i; break; }
        float x0, x1;
        if constexpr (KIND == 0) f2_unpack(f2_fma(f2_pack(r[2 * i], r[2 * i + 1]), scale2, c2), x0, x1);
        else { x0 = __uint_as_float(r[2 * i]); x1 = __uint_as_float(r[2 * i + 1]); }
        const float p0 = ex2_approx(x0), p1 = ex2_approx(x1);
        if (i & 1) acc1 = f2_add(acc1, f2_pack(p0, p1));
        else acc0 = f2_add(acc0, f2_pack(p0, p1));
        r[i] = pack_bf16x2(p0, p1);
    }
    if (!waited) {
        mbar_wait(p_empty_bar, p_empty_parity);
        tc_fence_after();
    }
#pragma unroll
    for (int q8 = 0; q8 < 8; ++q8) {                          // 8 probabilities -> one 16-byte chunk of the P row
        // PRESWZ: p_row already carries the row's swizzle term (see the caller)
        const uint32_t dst = PRESWZ ? p_row ^ (q8 * 16) : p_row + ((q8 ^ (row & 7)) * 16);
        if (KIND == 3 && 4 * q8 >= ndone)
            asm volatile("st.shared.v4.b32 [%0], {%1, %1, %1, %1};" ::"r"(dst), "r"(0u) : "memory");
        else
            asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(dst), "r"(r[q8 * 4]), "r"(r[q8 * 4 + 1]),
                         "r"(r[q8 * 4 + 2]), "r"(r[q8 * 4 + 3]) : "memory");
    }
    float s0, s1;
    f2_unpack(f2_add(acc0, acc1), s0, s1);
    l += s0 + s1;
}

template <int HD, bool ALIBI>
__device__ __forceinline__ void softmax_tile(uint32_t (&r)[64], uint32_t o_addr, bool first, SmemBar p_empty_bar,
                                             uint32_t p_empty_parity, float scale, float slope, float qpos, int key0,
                                             int Sk, float& m_ref, float& l, uint32_t p_row, int row, int lane, float gate) {
    const float base = first ? 0.f : m_ref;                  // exponents are first taken against `base`
    const float d0 = qpos - (float)key0;                     // query position minus the block's first key
    const int nvalid = Sk - key0;
    if (nvalid < kKB) {
        const float mx = exponents<3>(r, scale, ALIBI ? slope : 0.f, d0, base, nvalid);
        softmax_rest<HD, 3, !ALIBI>(r, mx, base, scale, nvalid, o_addr, first, p_empty_bar, p_empty_parity, m_ref, l, p_row, row, gate);
    } else if constexpr (ALIBI) {
        float mx;
        if (__all_sync(0xffffffffu, d0 >= 63.f) || __all_sync(0xffffffffu, d0 <= 0.f))
            mx = exponents<1>(r, scale, slope, d0, base, nvalid);
        else
            mx = exponents<2>(r, scale, slope, d0, base, nvalid);
        softmax_rest<HD, 1, !ALIBI>(r, mx, base, scale, nvalid, o_addr, first, p_empty_bar, p_empty_parity, m_ref, l, p_row, row, gate);
    } else {
        const float mx = exponents<0>(r, scale, 0.f, d0, base, nvalid);
        softmax_rest<HD, 0, !ALIBI>(r, mx, base, scale, nvalid, o_addr, first, p_empty_bar, p_empty_parity, m_ref, l, p_row, row, gate);
    }
}

// Shared-memory counters "K / V blocks issued so far", written by the TMA producer, read by the MMA issuers.
// mbarrier waits are parity waits: they are only sound while the waiter is at most ONE phase behind the barrier.  An
// issuer does not consume every block that passes through a ring stage (the other slot's blocks of a split-key item,
// items in which its slot is empty), so the stage's `full` barrier can be more than one phase behind the use the
// issuer is about to wait for, and a parity test then answers for the wrong phase (round 1: one wrong launch in 12 000
// on split-key items).  The producer issues load number idx only after BOTH release barriers of the stage's previous
// use have completed, i.e. after that use's `full` phase has completed; so once an issuer has seen issued > idx the
// barrier is either in the phase it waits for or one past it, and the parity test is exact.
__device__ __forceinline__ uint32_t lds_acquire(uint32_t addr) {
    uint32_t v;
    asm volatile("ld.acquire.cta.shared::cta.u32 %0, [%1];" : "=r"(v) : "r"(addr) : "memory");
    return v;
}
__device__ __forceinline__ void sts_release(uint32_t addr, uint32_t v) {
    asm volatile("st.release.cta.shared::cta.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}

// global position of K/V block (j, slot) of an item inside the CTA's K / V rings, relative to the item's first load.
// One stream when the slots share their keys; otherwise the blocks of the two slots alternate while both have keys.
__device__ __forceinline__ int ring_offset(int j, int s, bool same, int nk0, int nk1) {
    if (same) return j;
    return min(j, nk0) + min(j, nk1) + ((s == 1 && j < nk0) ? 1 : 0);
}

template <int HD, bool ALIBI>
__global__ void __launch_bounds__(kThreads, 2)
attention_mc_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                    const __grid_constant__ CUtensorMap tmV, const Params p) {
    extern __shared__ uint8_t smem_raw[];
    // Everything in shared memory is named by its 32-bit shared-space address (see SmemBar): one base register, constant
    // offsets.
    uint32_t smem_a = (smem_u32(smem_raw) + 1023u) & ~1023u;
    // HD = 48: opaque, so the base stays in a register instead of being rebuilt (S2UR + ULEA) at every hand-shake
    // (201-token self-attention 0.69 -> 0.63 ms).  HD = 64 has no register to spare in the softmax warps.
    if constexpr (HD == 48) asm volatile("mov.b32 %0, %0;" : "+r"(smem_a));
    const uint32_t sm_q = smem_a;                                 // 2 slots x 16 KB
    const uint32_t sm_k = sm_q + 2 * kQBytes;                     // kKStages x 8 KB
    const uint32_t sm_v = sm_k + kKStages * kKvBytes;             // kVStages x 8 KB
    const uint32_t sm_p = sm_v + kVStages * kKvBytes;             // 2 slots x 16 KB
    const SmemBar bars{sm_p + 2 * kQBytes};
    const SmemBar q_full = bars[0], q_empty = bars[2];            // [slot]
    const SmemBar s_full = bars[4], s_empty = bars[6];            // [slot]
    const SmemBar p_full = bars[8], p_empty = bars[10];           // [slot]
    const SmemBar o_full = bars[12], o_empty = bars[14];          // [slot]
    // a K / V stage has TWO release barriers, one per slot: both slots arrive (tcgen05.commit) when they share the
    // block, its only user arrives on both otherwise.  (Two commits on ONE barrier with count 2 are not reliable: when
    // both are pending on the same MMAs they can be merged into a single arrival.)
    const SmemBar k_full = bars[16], k_empty = k_full[kKStages];  // k_empty[2 * stage + slot]
    const SmemBar v_full = k_empty[2 * kKStages], v_empty = v_full[kVStages];
    const uint32_t tmem_slot = v_empty[2 * kVStages].addr;
    const uint32_t k_issued = tmem_slot + 8, v_issued = tmem_slot + 12;   // blocks issued so far (see lds_acquire)

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int n_work = p.n_items * p.heads;

    if (warp == 0 && elect_one()) {
        tma_prefetch_desc(&tmQ); tma_prefetch_desc(&tmK); tma_prefetch_desc(&tmV);
        for (int i = 0; i < 2; ++i) {
            mbar_init(q_full[i], 1); mbar_init(q_empty[i], 1);
            mbar_init(s_full[i], 1); mbar_init(s_empty[i], 4);      // 4 softmax warps per slot
            mbar_init(p_full[i], 4); mbar_init(p_empty[i], 1);
            mbar_init(o_full[i], 1); mbar_init(o_empty[i], 4);
        }
        for (int i = 0; i < kKStages; ++i) { mbar_init(k_full[i], 1); mbar_init(k_empty[2 * i], 1); mbar_init(k_empty[2 * i + 1], 1); }
        for (int i = 0; i < kVStages; ++i) { mbar_init(v_full[i], 1); mbar_init(v_empty[2 * i], 1); mbar_init(v_empty[2 * i + 1], 1); }
        sts_release(k_issued, 0u); sts_release(v_issued, 0u);
        fence_barrier_init();
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(tmem_slot), "r"((uint32_t)kTmemCols) : "memory");
        tmem_relinquish();
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    uint32_t tmem_base;
    asm volatile("ld.shared.b32 %0, [%1];" : "=r"(tmem_base) : "r"(tmem_slot) : "memory");

    // work index w -> (head, item): head-major so concurrently running CTAs share one head's K/V in L2.  Every role
    // reads only the fields it needs from the item's two slot records.
    const int4* recs = reinterpret_cast<const int4*>(p.slots);         // 4 int4 per item: {s0.lo, s0.hi, s1.lo, s1.hi}

    if (warp < kFirstSoftmaxWarp) {
        reg_dealloc<kRegsLo>();
        if (warp == 0 && elect_one()) {
            // ============================ TMA producer ============================
            uint32_t ring = 0;                               // K / V blocks loaded so far (same count for both rings)
            uint32_t nq[2] = {0, 0};                         // Q tiles loaded so far per slot
            for (int w = blockIdx.x; w < n_work; w += gridDim.x) {
                const int head = w / p.n_items, item = w - head * p.n_items;
                const int4 r0 = __ldg(recs + 4 * item), r1 = __ldg(recs + 4 * item + 2);   // {qrow, nrows, krow, Sk}
                const int qrow[2] = {r0.x, r1.x}, krow[2] = {r0.z, r1.z};
                const int nk[2] = {r0.y > 0 ? (r0.w + kKB - 1) / kKB : 0, r1.y > 0 ? (r1.w + kKB - 1) / kKB : 0};
                const bool same = nk[0] > 0 && nk[1] > 0 && r0.z == r1.z && r0.w == r1.w;
                const int col = head * HD;
#pragma unroll
                for (int s = 0; s < 2; ++s) {
                    if (nk[s] == 0) continue;
                    const uint32_t m = nq[s]++;
                    mbar_wait(q_empty[s], (m & 1) ^ 1);
                    mbar_arrive_expect_tx(q_full[s], kQBytes);
                    tma_load_2d(sm_q + s * kQBytes, &tmQ, q_full[s], col, qrow[s]);
                }
                // K / V blocks in exactly the order the MMA warps consume them: K of block j+1 before V of block j
                const int nkmax = max(nk[0], nk[1]);
                const uint32_t base = ring;
                auto load_k = [&](int j, int s) {
                    const uint32_t idx = base + ring_offset(j, s, same, nk[0], nk[1]);
                    const uint32_t st = idx % kKStages;
                    mbar_wait(k_empty[2 * st], ((idx / kKStages) & 1) ^ 1);
                    mbar_wait(k_empty[2 * st + 1], ((idx / kKStages) & 1) ^ 1);
                    mbar_arrive_expect_tx(k_full[st], kKvBytes);
                    tma_load_2d(sm_k + st * kKvBytes, &tmK, k_full[st], col, krow[s] + j * kKB);
                    sts_release(k_issued, idx + 1);
                };
                auto load_v = [&](int j, int s) {
                    const uint32_t idx = base + ring_offset(j, s, same, nk[0], nk[1]);
                    const uint32_t st = idx % kVStages;
                    mbar_wait(v_empty[2 * st], ((idx / kVStages) & 1) ^ 1);
                    mbar_wait(v_empty[2 * st + 1], ((idx / kVStages) & 1) ^ 1);
                    mbar_arrive_expect_tx(v_full[st], kKvBytes);
                    tma_load_2d(sm_v + st * kKvBytes, &tmV, v_full[st], col, krow[s] + j * kKB);
                    sts_release(v_issued, idx + 1);
                };
#pragma unroll
                for (int s = 0; s < 2; ++s) if (nk[s] > 0 && !(s == 1 && same)) load_k(0, s);
                for (int j = 0; j < nkmax; ++j) {
#pragma unroll
                    for (int s = 0; s < 2; ++s) if (j + 1 < nk[s] && !(s == 1 && same)) load_k(j + 1, s);
#pragma unroll
                    for (int s = 0; s < 2; ++s) if (j < nk[s] && !(s == 1 && same)) load_v(j, s);
                }
                ring += same ? nk[0] : nk[0] + nk[1];
            }
        } else if (warp == 1 || warp == 2) {
            // ============================ MMA issuer of slot s = warp - 1 ============================
            // One issuer per slot: neither slot ever waits behind the other's barriers.  S(j+1) = Q K^T is issued as
            // soon as the four softmax warps have S(j) in registers, i.e. BEFORE waiting for P(j); the first Q K^T of
            // the next item follows the last P V of the current one.
            const int s = warp - 1;
            constexpr uint32_t idesc_qk = umma_idesc_bf16(128, kKB);                         // A, B K-major
            constexpr uint32_t idesc_pv = umma_idesc_bf16(128, HD) | (1u << 16);            // B (= V) MN-major
            const uint32_t s_tmem = tmem_base + s * kKB, o_tmem = tmem_base + 128 + s * 64;
            const uint64_t q_desc = umma_desc_kmajor_sw128(sm_q + s * kQBytes);
            const uint64_t p_desc = umma_desc_kmajor_sw128(sm_p + s * kQBytes);
            // One work item as this issuer sees it, packed into four registers (the warpgroup runs on 32 registers per
            // thread and every spill here is on the critical path of short sequences): key-block counts of both slots,
            // own block count, keys in the own last block, flags, first ring position, first score tile.
            struct It {
                uint32_t nks, meta, base, tile0;
                __device__ __forceinline__ int nk0() const { return (int)(nks & 0xFFFFu); }
                __device__ __forceinline__ int nk1() const { return (int)(nks >> 16); }
                __device__ __forceinline__ int my_nk() const { return (int)(meta & 0xFFFFu); }
                __device__ __forceinline__ int tail() const { return (int)((meta >> 16) & 0xFFu); }
                __device__ __forceinline__ bool same() const { return (meta >> 24) & 1u; }
                __device__ __forceinline__ bool all_mine() const { return (meta >> 25) & 1u; }
            };
            bool skipped = false, prev_all_mine = false;
            uint32_t ring = 0, n_tiles = 0, n_q = 0, n_done = 0;      // ring position, score tiles / items started / finished
            uint32_t run0 = 0xF0000000u;                              // see `issued` (no run yet)
            int w = blockIdx.x;
            // next work item in which this slot is occupied (the ring position advances over every item)
            auto next_valid = [&](It& it) -> bool {
                for (; w < n_work; w += gridDim.x) {
                    const int item = w % p.n_items;
                    const int4 r0 = __ldg(recs + 4 * item), r1 = __ldg(recs + 4 * item + 2);
                    const int nk0 = r0.y > 0 ? (r0.w + kKB - 1) / kKB : 0;
                    const int nk1 = r1.y > 0 ? (r1.w + kKB - 1) / kKB : 0;
                    const bool same = nk0 > 0 && nk1 > 0 && r0.z == r1.z && r0.w == r1.w;
                    it.base = ring;
                    ring += same ? nk0 : nk0 + nk1;
                    const int my_nk = s == 0 ? nk0 : nk1;
                    const int tail = (s == 0 ? r0.w : r1.w) - (my_nk - 1) * kKB;      // keys in the own last block (1..64)
                    // does this issuer consume every ring position of the item?  (shared stream, or the only occupied slot)
                    const bool all_mine = my_nk > 0 && (same || (s == 0 ? nk1 : nk0) == 0);
                    it.nks = (uint32_t)nk0 | ((uint32_t)nk1 << 16);
                    it.meta = (uint32_t)my_nk | ((uint32_t)(tail & 0xFF) << 16) | ((uint32_t)same << 24) | ((uint32_t)all_mine << 25);
                    if (my_nk > 0) {
                        // a run continues only from an item consumed in full, with no item skipped in between
                        if (!all_mine) run0 = 0xF0000000u;
                        else if (!prev_all_mine || skipped) run0 = it.base;
                        prev_all_mine = all_mine; skipped = false;
                        w += gridDim.x;
                        return true;
                    }
                    skipped = true;                                   // ring positions pass by that this issuer never sees
                }
                return false;
            };
            auto ready = [&](SmemBar bar, uint32_t parity, bool blocking) -> bool {
                if (blocking) { mbar_wait(bar, parity); return true; }
                // one lane's answer for the whole warp: the lanes keep the (uniform) books of the pipeline, so they
                // must never disagree on whether the early Q K^T went out
                return __shfl_sync(0xffffffffu, (int)mbar_test_wait(bar, parity), 0) != 0;
            };
            // Has the producer issued block idx of a ring?  Needed only when this issuer did not consume the stage's
            // previous use itself (idx - stages): `run0` is the ring position from which it has consumed EVERY block
            // (shared streams of items in which its slot is occupied), so inside such a run no check is made at all.
            // Blocking mode: every lane polls for itself (each one's own later parity test is then sound); non-blocking
            // mode: one lane's answer for the warp, the lanes must agree on whether the early Q K^T went out.
            auto issued = [&](uint32_t ctr, uint32_t idx, uint32_t stages, bool blocking) -> bool {
                if (idx >= run0 + stages) return true;
                if (!blocking) return __shfl_sync(0xffffffffu, lds_acquire(ctr), 0) > idx;
                uint32_t spins = 0;
                while (lds_acquire(ctr) <= idx)
                    if ((++spins & 0xFFFFFFu) == 0) __trap();                     // ~seconds: a pipeline bug, never a wait
                return true;
            };
            // S(j) = Q K(j)^T of item `it`; non-blocking mode gives up (nothing issued) if an input has not landed yet
            auto issue_qk = [&](It& it, int j, bool blocking) -> bool {
                const uint32_t idx = it.base + ring_offset(j, s, it.same(), it.nk0(), it.nk1());
                const uint32_t st = idx % kKStages;
                if (j == 0 && !ready(q_full[s], n_q & 1, blocking)) return false;
                if (!issued(k_issued, idx, kKStages, blocking)) return false;
                if (!ready(k_full[st], (idx / kKStages) & 1, blocking)) return false;
                if (!ready(s_empty[s], (n_tiles & 1) ^ 1, blocking)) return false;      // previous scores are in registers
                if (j == 0) { ++n_q; it.tile0 = n_tiles; }
                ++n_tiles;
                tc_fence_after();
                if (elect_one()) {                            // the whole warp keeps the (uniform) books, one lane issues
                    const uint64_t db = umma_desc_kmajor_sw128(sm_k + st * kKvBytes);
#pragma unroll
                    for (int k = 0; k < HD / 16; ++k) umma_bf16(s_tmem, q_desc + 2 * k, db + 2 * k, idesc_qk, k != 0);
                    umma_commit(s_full[s]);
                    umma_commit(k_empty[2 * st + s]);
                    if (!it.same()) umma_commit(k_empty[2 * st + (s ^ 1)]);    // sole user: the other slot's release too
                    if (j + 1 == it.my_nk()) umma_commit(q_empty[s]);          // last Q K^T of the item: Q slot may be refilled
                }
                __syncwarp();
                return true;
            };
            It cur, nxt;
            bool have = next_valid(cur);
            if (have) issue_qk(cur, 0, true);
            while (have) {
                const bool have_next = next_valid(nxt);
                bool next_started = false;
                for (int j = 0; j < cur.my_nk(); ++j) {
                    // S(j+1) is issued as soon as the four softmax warps have S(j) in registers, i.e. BEFORE waiting for
                    // P(j).  At the last block the first score tile of the NEXT item goes out instead — but only if its
                    // inputs have already landed: blocking on them here could deadlock (the producer may need the V
                    // block this slot is about to release before it can reach the next item's loads).
                    if (j + 1 < cur.my_nk()) issue_qk(cur, j + 1, true);
                    else if (have_next) next_started = issue_qk(nxt, 0, false);
                    // ---- O += P(j) V(j) ----
                    const uint32_t idx = cur.base + ring_offset(j, s, cur.same(), cur.nk0(), cur.nk1());
                    const uint32_t st = idx % kVStages;
                    if (j == 0) mbar_wait(o_empty[s], (n_done & 1) ^ 1);   // previous item's O has been read out
                    issued(v_issued, idx, kVStages, true);
                    mbar_wait(v_full[st], (idx / kVStages) & 1);
                    const uint32_t vb = sm_v + st * kKvBytes;
                    int nkk = kKB / 16;                          // 16-key steps of this block's P V
                    if (j + 1 == cur.my_nk() && cur.tail() < kKB) {
                        // The last block of a sequence over-fetches rows of whatever follows it in the K/V tensors.  Their
                        // probabilities are exactly 0, but 0 x NaN/Inf would still poison O.  Whole 16-key groups past the
                        // last key are not multiplied at all; in the partial group the V rows past the end are cleared
                        // (a row of the [64 keys x 64] SWIZZLE_128B tile is 128 contiguous bytes; at most 15 rows).  Both
                        // issuers of a shared stream write the same zeros.
                        nkk = (cur.tail() + 15) >> 4;
                        if (cur.tail() & 15) {
                            for (int r = cur.tail() + (lane >> 3); r < nkk * 16; r += 4)
                                asm volatile("st.shared.v4.b32 [%0], {%1, %1, %1, %1};" ::"r"(vb + r * 128 + (lane & 7) * 16), "r"(0u) : "memory");
                            fence_proxy_async_smem();
                            __syncwarp();
                        }
                    }
                    mbar_wait(p_full[s], (cur.tile0 + j) & 1);
                    tc_fence_after();
                    if (elect_one()) {
                        for (int kk = 0; kk < nkk; ++kk)
                            umma_bf16(o_tmem, p_desc + 2 * kk, umma_desc_kmajor_sw128(vb + kk * 2048), idesc_pv, (j | kk) != 0);
                        umma_commit(p_empty[s]);
                        umma_commit(v_empty[2 * st + s]);
                        if (!cur.same()) umma_commit(v_empty[2 * st + (s ^ 1)]);
                        if (j + 1 == cur.my_nk()) umma_commit(o_full[s]);
                    }
                    __syncwarp();
                }
                ++n_done;
                if (have_next && !next_started) issue_qk(nxt, 0, true);   // everything of `cur` is consumed: blocking is safe
                cur = nxt;
                have = have_next;
            }
        }
    } else {
        // ============================ softmax warps (fully independent of each other) ============================
        reg_alloc<kRegsHi>();
        const int s = (warp - kFirstSoftmaxWarp) >> 2;        // slot owned by this warpgroup
        const int quad = warp & 3;                            // TMEM lane quadrant of this warp
        const int row = quad * 32 + lane;                     // row inside the 128-row query tile
        const uint32_t t_lane = tmem_base + ((uint32_t)(quad * 32) << 16);
        uint32_t s_addr = t_lane + s * kKB;
        const uint32_t o_addr = t_lane + 128 + s * 64;
        // opaque: otherwise the address is REBUILT from SR_TID and the (spilled) TMEM base at every tile — S2R + LDL + 8
        // integer instructions whose scoreboard waits were 6 % of the softmax warps' samples
        asm volatile("mov.b32 %0, %0;" : "+r"(s_addr));
        // this row of the P tile (shared-space address, 128-byte aligned) with the row's SWIZZLE_128B term folded in:
        // chunk q8 of the row lives at my_p ^ (q8 * 16)
        // (not in the ALiBi kernels: measured 3 % slower there, 0.6 % faster without the bias)
        const uint32_t my_p = (sm_p + s * kQBytes + row * 128) ^ (ALIBI ? 0u : (uint32_t)((row & 7) * 16));
        // this slot's barriers, relative to ONE register (index = the [slot] arrays' offsets from `bars`)
        uint32_t sb_a = bars[s].addr;
        if constexpr (HD == 48 && !ALIBI) asm volatile("mov.b32 %0, %0;" : "+r"(sb_a));   // (a register too many with ALiBi)
        const SmemBar sb{sb_a};
        const SmemBar my_s_full = sb[4], my_s_empty = sb[6], my_p_full = sb[8], my_p_empty = sb[10], my_o_full = sb[12],
                      my_o_empty = sb[14];
        uint32_t n_tiles = 0, n_mine = 0;                     // score tiles / items this slot has processed so far
        for (int w = blockIdx.x; w < n_work; w += gridDim.x) {
            const int head = w / p.n_items, item = w - head * p.n_items;
            const int4 me = __ldg(recs + 4 * item + 2 * s);                       // {qrow, nrows, krow, Sk}
            const int my_nk = me.y > 0 ? (me.w + kKB - 1) / kKB : 0;
            if (my_nk == 0) continue;
            const int qpos0 = __ldg(reinterpret_cast<const int*>(recs + 4 * item + 2 * s + 1));
            const float slope = ALIBI ? p.slopes[head] * 1.4426950408889634f : 0.f;
            const float qpos = (float)(qpos0 + row);
            float m_ref = 0.f, l_run = 0.f;
            float gate = row < me.y ? kLazyThreshold : INFINITY;      // only live rows vote on a raise (softmax_rest)
            asm volatile("mov.b32 %0, %0;" : "+f"(gate));
            for (int j = 0; j < my_nk; ++j) {
                const uint32_t m = n_tiles++;
                mbar_wait(my_s_full, m & 1);
                tc_fence_after();
                // ---- scores of this row -> registers; then the score buffer is free for the next Q K^T ----
                uint32_t r[64];
                tmem_ld_32x32(s_addr, *reinterpret_cast<uint32_t(*)[32]>(&r[0]));
                if (me.w - j * kKB > 32)                      // (a tail block's softmax reads only its groups of keys)
                    tmem_ld_32x32(s_addr + 32, *reinterpret_cast<uint32_t(*)[32]>(&r[32]));
                tmem_ld_wait();
                tc_fence_before();
                __syncwarp();
                // one lane arrives on the warp's behalf: `elect.sync` needs no register and no S2R (the compiler does not
                // keep `lane` alive across the tile loop at 104 registers: it re-read SR_TID at every arrive)
                if (elect_one()) mbar_arrive(my_s_empty);
                softmax_tile<HD, ALIBI>(r, o_addr, j == 0, my_p_empty, (m & 1) ^ 1, p.scale_log2, slope, qpos, j * kKB,
                                        me.w, m_ref, l_run, my_p, row, lane, gate);
                fence_proxy_async_smem();                     // generic-proxy P writes -> visible to the UMMA (async proxy)
                tc_fence_before();                            // orders a possible tcgen05.st rescale before the PV
                __syncwarp();
                if (elect_one()) mbar_arrive(my_p_full);
            }
            // ---- epilogue: O_s / l -> bf16 -> global ----
            mbar_wait(my_o_full, n_mine & 1);
            ++n_mine;
            tc_fence_after();
            uint32_t o0[32], o1[32];
            tmem_ld_32x32(o_addr, o0);
            if constexpr (HD > 48) tmem_ld_32x32(o_addr + 32, o1);
            else tmem_ld_32x16(o_addr + 32, *reinterpret_cast<uint32_t(*)[16]>(&o1[0]));
            tmem_ld_wait();
            tc_fence_before();
            __syncwarp();
            if (elect_one()) mbar_arrive(my_o_empty);          // O_s may be overwritten by the next item's first P V
            if (row < me.y) {
                const float inv = 1.0f / l_run;
                __nv_bfloat16* dst = p.o + (size_t)(me.x + row) * p.ldo + head * HD;
#pragma unroll
                for (int e = 0; e < 32; e += 8)
                    *reinterpret_cast<uint4*>(dst + e) = make_uint4(
                        pack_bf16x2(__uint_as_float(o0[e]) * inv, __uint_as_float(o0[e + 1]) * inv),
                        pack_bf16x2(__uint_as_float(o0[e + 2]) * inv, __uint_as_float(o0[e + 3]) * inv),
                        pack_bf16x2(__uint_as_float(o0[e + 4]) * inv, __uint_as_float(o0[e + 5]) * inv),
                        pack_bf16x2(__uint_as_float(o0[e + 6]) * inv, __uint_as_float(o0[e + 7]) * inv));
#pragma unroll
                for (int e = 0; e < HD - 32; e += 8)
                    *reinterpret_cast<uint4*>(dst + 32 + e) = make_uint4(
                        pack_bf16x2(__uint_as_float(o1[e]) * inv, __uint_as_float(o1[e + 1]) * inv),
                        pack_bf16x2(__uint_as_float(o1[e + 2]) * inv, __uint_as_float(o1[e + 3]) * inv),
                        pack_bf16x2(__uint_as_float(o1[e + 4]) * inv, __uint_as_float(o1[e + 5]) * inv),
                        pack_bf16x2(__uint_as_float(o1[e + 6]) * inv, __uint_as_float(o1[e + 7]) * inv));
            }
        }
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) { tc_fence_after(); tmem_dealloc(tmem_base, kTmemCols); }
}

// ---------------------------------------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static int make_tmap_rows64(CUtensorMap* tm, const void* base, long rows, int cols, int ld, int box_rows) {
    static PFN_encodeTiled enc = nullptr;
    if (!enc) {
        void* fp = nullptr; cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fp, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            enc = reinterpret_cast<PFN_encodeTiled>(fp);
    }
    VF_REQUIRE(enc, "cuTensorMapEncodeTiled entry point not available");
    VF_REQUIRE((reinterpret_cast<uintptr_t>(base) & 15) == 0 && ld % 8 == 0, "attention operands must be 16-byte aligned");
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
    cuuint32_t box[2] = {64, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    VF_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed (%d) for an attention operand", (int)r);
    return 0;
}

template <int HD, bool ALIBI>
static int launch(const CUtensorMap& tq, const CUtensorMap& tk, const CUtensorMap& tv, const Params& p, cudaStream_t s) {
    static bool attr_set = false;
    if (!attr_set) {
        VF_CUDA_OK(cudaFuncSetAttribute(attention_mc_kernel<HD, ALIBI>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)kSmem));
        VF_CUDA_OK(cudaFuncSetAttribute(attention_mc_kernel<HD, ALIBI>, cudaFuncAttributePreferredSharedMemoryCarveout,
                                        cudaSharedmemCarveoutMaxShared));
        // (cudaOccupancyMaxActiveBlocksPerMultiprocessor reports 1 for every kernel that allocates tensor memory;
        //  tools/ubench/occ.cu shows two such CTAs with 256 columns and 108 KB each are in fact co-resident.)
        attr_set = true;
    }
    int dev = 0, sms = 0;
    VF_CUDA_OK(cudaGetDevice(&dev));
    VF_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    const long work = (long)p.n_items * p.heads;
    const int grid = (int)(work < 2L * sms ? work : 2L * sms);
    attention_mc_kernel<HD, ALIBI><<<grid, kThreads, kSmem, s>>>(tq, tk, tv, p);
    VF_LAUNCH_OK("attention_mc_kernel launch");
    return 0;
}

}  // namespace mc

int attention_mc_varlen(const void* q, int ldq, const void* k, int ldk, const void* v, int ldv, void* o, int ldo,
                        long rows_q, long rows_k, const int* slots, int n_items, int heads, int head_dim,
                        const float* slopes, cudaStream_t stream) {
    using namespace mc;
    VF_REQUIRE(head_dim == 48 || head_dim == 64, "attention_mc: head_dim %d not supported (48/64)", head_dim);
    VF_REQUIRE(ldo % 8 == 0, "attention_mc: output stride must keep 16-byte alignment");
    if (n_items == 0) return 0;
    const int d = heads * head_dim;
    CUtensorMap tq, tk, tv;
    if (make_tmap_rows64(&tq, q, rows_q, d, ldq, kQT)) return -1;
    if (make_tmap_rows64(&tk, k, rows_k, d, ldk, kKB)) return -1;
    if (make_tmap_rows64(&tv, v, rows_k, d, ldv, kKB)) return -1;
    Params p;
    VF_REQUIRE((reinterpret_cast<uintptr_t>(slots) & 15) == 0, "attention_mc: slot table must be 16-byte aligned");
    p.slots = reinterpret_cast<const SlotRec*>(slots); p.n_items = n_items; p.heads = heads;
    p.o = (__nv_bfloat16*)o; p.ldo = ldo; p.slopes = slopes;
    p.scale_log2 = (1.0f / sqrtf((float)head_dim)) * 1.4426950408889634f;
    if (head_dim == 48) return slopes ? launch<48, true>(tq, tk, tv, p, stream) : launch<48, false>(tq, tk, tv, p, stream);
    return slopes ? launch<64, true>(tq, tk, tv, p, stream) : launch<64, false>(tq, tk, tv, p, stream);
}

}  // namespace vf
