// vf_attn_probs.cu — the probabilities of a cross-attention for selected query rows (vf_cross_attention_probs).
//
// The fused attention kernel (vf_attention_mc.cu) keeps P in TMEM and shared memory only.  This kernel recomputes P for a
// few query rows per key range — the registry (tissue) rows of every gene against the gene's CREs — and writes it in
// fp32.  The work is n_rows x keys x head_dim per head, small next to the layer's GEMMs, so it runs on CUDA cores:
//   one CTA per (group, head); up to 64 query rows of the group in shared memory (fp32), K streamed through a 64-key
//   shared-memory tile with 16-byte loads;
//   pass 1: every lane keeps a running (max, sum) per row over its keys; a butterfly merges the lanes (IEEE max and
//   the two-term sum are commutative, so every lane ends with the same bits);
//   pass 2: the same score code again, exp(s - max) / sum stored along the keys (coalesced).
// A row's result depends on its own q, its group's keys and nothing else: not on its position in the group, the group's
// size, or the other groups of the launch.
#include <math.h>

#include "vf_common.cuh"
#include "vf_internal.h"

namespace vf {
namespace {

constexpr int kWarps = 8;
constexpr int kRowsPerWarp = 8;
constexpr int kRows = kWarps * kRowsPerWarp;   // query rows per K stream
constexpr int kKeys = 64;                      // keys per shared-memory tile: two per lane
constexpr int kThreads = kWarps * 32;

__device__ __forceinline__ void unpack8(const uint4 v, float* dst) {
    const __nv_bfloat162* p = reinterpret_cast<const __nv_bfloat162*>(&v);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        const float2 f = __bfloat1622float2(p[i]);
        dst[2 * i] = f.x; dst[2 * i + 1] = f.y;
    }
}

// keys [c0, c0 + kKeys) of head h into ks (rows past nk zero-filled: never read from global memory)
template <int HD, int KS>
__device__ __forceinline__ void load_key_tile(float (*ks)[KS], const __nv_bfloat16* __restrict__ k, int ldk, long k0,
                                              int c0, int nk, int h) {
    constexpr int V = HD / 8;
    for (int i = threadIdx.x; i < kKeys * V; i += kThreads) {
        const int j = i / V, u = i % V;
        uint4 v = make_uint4(0, 0, 0, 0);
        if (c0 + j < nk) v = *reinterpret_cast<const uint4*>(k + (k0 + c0 + j) * (long)ldk + h * HD + u * 8);
        unpack8(v, &ks[j][u * 8]);
    }
}

// scaled scores of this warp's rows against this lane's two keys of the tile
template <int HD, int KS>
__device__ __forceinline__ void tile_scores(const float (*qs)[HD], const float (*ks)[KS], int warp, int lane, float scale,
                                            float (&s)[kRowsPerWarp][2]) {
    float acc[kRowsPerWarp][2];
#pragma unroll
    for (int j = 0; j < kRowsPerWarp; ++j) acc[j][0] = acc[j][1] = 0.f;
#pragma unroll 4
    for (int d = 0; d < HD; ++d) {
        const float k0 = ks[lane][d], k1 = ks[lane + 32][d];
#pragma unroll
        for (int j = 0; j < kRowsPerWarp; ++j) {
            const float qv = qs[warp + kWarps * j][d];
            acc[j][0] = fmaf(qv, k0, acc[j][0]);
            acc[j][1] = fmaf(qv, k1, acc[j][1]);
        }
    }
#pragma unroll
    for (int j = 0; j < kRowsPerWarp; ++j) {                // __fmul_rn: never contracted into the exp argument
        s[j][0] = __fmul_rn(acc[j][0], scale);
        s[j][1] = __fmul_rn(acc[j][1], scale);
    }
}

template <int HD>
__global__ void __launch_bounds__(kThreads) cross_attention_probs_kernel(
    const __nv_bfloat16* __restrict__ q, int ldq, const int32_t* __restrict__ q_rows, const int32_t* __restrict__ group_q,
    const __nv_bfloat16* __restrict__ k, int ldk, const int32_t* __restrict__ group_k, int heads, float* __restrict__ out,
    const int64_t* __restrict__ out_off, int layer, float scale) {
    constexpr int KS = HD + 1;                         // padded: the lanes of a warp read 32 different key rows
    constexpr int V = HD / 8;
    __shared__ float qs[kRows][HD];
    __shared__ float ks[kKeys][KS];
    const int g = blockIdx.x, h = blockIdx.y;
    const int q0 = group_q[2 * g], nq = group_q[2 * g + 1];
    const long k0 = group_k[2 * g];
    const int nk = group_k[2 * g + 1];
    if (nq <= 0 || nk <= 0) return;
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const long head_off = ((long)layer * heads + h) * nk;
    for (int r0 = 0; r0 < nq; r0 += kRows) {
        const int nr = min(kRows, nq - r0);
        __syncthreads();                               // the previous chunk's readers of qs / ks are done
        for (int i = threadIdx.x; i < kRows * V; i += kThreads) {
            const int r = i / V, u = i % V;
            uint4 v = make_uint4(0, 0, 0, 0);
            if (r < nr) {
                const int qi = q0 + r0 + r;
                const long row = q_rows ? q_rows[qi] : qi;
                v = *reinterpret_cast<const uint4*>(q + row * ldq + h * HD + u * 8);
            }
            unpack8(v, &qs[r][u * 8]);
        }
        const bool active = warp < nr;                 // warp-uniform: this warp has at least one live row
        float m[kRowsPerWarp], l[kRowsPerWarp], s[kRowsPerWarp][2];
#pragma unroll
        for (int j = 0; j < kRowsPerWarp; ++j) { m[j] = -INFINITY; l[j] = 0.f; }
        // ---- pass 1: running (max, sum) per (lane, row) ----
        for (int c0 = 0; c0 < nk; c0 += kKeys) {
            __syncthreads();
            load_key_tile<HD, KS>(ks, k, ldk, k0, c0, nk, h);
            __syncthreads();
            if (!active) continue;
            tile_scores<HD, KS>(qs, ks, warp, lane, scale, s);
            const bool v0 = c0 + lane < nk, v1 = c0 + lane + 32 < nk;
#pragma unroll
            for (int j = 0; j < kRowsPerWarp; ++j) {
                const float a = v0 ? s[j][0] : -INFINITY, b = v1 ? s[j][1] : -INFINITY;
                const float mn = fmaxf(m[j], fmaxf(a, b));
                if (mn == -INFINITY) continue;
                l[j] = l[j] * expf(m[j] - mn) + expf(a - mn) + expf(b - mn);
                m[j] = mn;
            }
        }
        if (active) {
#pragma unroll
            for (int j = 0; j < kRowsPerWarp; ++j) {
#pragma unroll
                for (int o = 16; o; o >>= 1) {
                    const float mo = __shfl_xor_sync(0xffffffffu, m[j], o), lo = __shfl_xor_sync(0xffffffffu, l[j], o);
                    const float mn = fmaxf(m[j], mo);
                    l[j] = mn == -INFINITY ? 0.f : l[j] * expf(m[j] - mn) + lo * expf(mo - mn);
                    m[j] = mn;
                }
            }
        }
        // ---- pass 2: the same scores, normalised ----
        int64_t base[kRowsPerWarp];
#pragma unroll
        for (int j = 0; j < kRowsPerWarp; ++j) {
            const int r = warp + kWarps * j;
            base[j] = r < nr ? out_off[q0 + r0 + r] + head_off : -1;
        }
        for (int c0 = 0; c0 < nk; c0 += kKeys) {
            __syncthreads();
            load_key_tile<HD, KS>(ks, k, ldk, k0, c0, nk, h);
            __syncthreads();
            if (!active) continue;
            tile_scores<HD, KS>(qs, ks, warp, lane, scale, s);
            const int c = c0 + lane;
#pragma unroll
            for (int j = 0; j < kRowsPerWarp; ++j) {
                if (base[j] < 0) continue;
                if (c < nk) out[base[j] + c] = expf(s[j][0] - m[j]) / l[j];
                if (c + 32 < nk) out[base[j] + c + 32] = expf(s[j][1] - m[j]) / l[j];
            }
        }
    }
}

}  // namespace

int cross_attention_probs(const void* q, int ldq, const int32_t* q_rows, const int32_t* group_q, int n_groups, const void* k,
                          int ldk, const int32_t* group_k, int heads, int head_dim, float* out, const int64_t* out_off,
                          int layer, cudaStream_t s) {
    VF_REQUIRE(n_groups >= 0 && heads > 0 && heads <= 65535 && layer >= 0,
               "cross_attention_probs: n_groups %d, heads %d, layer %d out of range", n_groups, heads, layer);
    VF_REQUIRE(head_dim == 48 || head_dim == 64, "cross_attention_probs: head_dim %d not in {48, 64}", head_dim);
    VF_REQUIRE(ldq >= heads * head_dim && ldk >= heads * head_dim && ldq % 8 == 0 && ldk % 8 == 0,
               "cross_attention_probs: ldq %d / ldk %d must be multiples of 8 and >= heads * head_dim", ldq, ldk);
    VF_REQUIRE((reinterpret_cast<uintptr_t>(q) & 15) == 0 && (reinterpret_cast<uintptr_t>(k) & 15) == 0,
               "cross_attention_probs: q and k must be 16-byte aligned");
    VF_REQUIRE((reinterpret_cast<uintptr_t>(out) & 3) == 0 && (reinterpret_cast<uintptr_t>(out_off) & 7) == 0 &&
               (reinterpret_cast<uintptr_t>(q_rows) & 3) == 0 && (reinterpret_cast<uintptr_t>(group_q) & 3) == 0 &&
               (reinterpret_cast<uintptr_t>(group_k) & 3) == 0,
               "cross_attention_probs: misaligned out / out_off / index tables");
    if (n_groups == 0) return 0;
    VF_REQUIRE(q && k && group_q && group_k && out && out_off, "cross_attention_probs: NULL operand");
    const dim3 grid(n_groups, heads);
    const float scale = 1.0f / sqrtf((float)head_dim);
    if (head_dim == 48)
        cross_attention_probs_kernel<48><<<grid, kThreads, 0, s>>>((const __nv_bfloat16*)q, ldq, q_rows, group_q,
                                                                   (const __nv_bfloat16*)k, ldk, group_k, heads, out,
                                                                   out_off, layer, scale);
    else
        cross_attention_probs_kernel<64><<<grid, kThreads, 0, s>>>((const __nv_bfloat16*)q, ldq, q_rows, group_q,
                                                                   (const __nv_bfloat16*)k, ldk, group_k, heads, out,
                                                                   out_off, layer, scale);
    VF_LAUNCH_OK("cross_attention_probs_kernel launch");
    return 0;
}

}  // namespace vf

extern "C" int vf_cross_attention_probs(const void* q, int ldq, const int32_t* q_rows, const int32_t* group_q, int n_groups,
                                        const void* k, int ldk, const int32_t* group_k, int heads, int head_dim, float* out,
                                        const int64_t* out_off, int layer, void* stream) {
    return vf::cross_attention_probs(q, ldq, q_rows, group_q, n_groups, k, ldk, group_k, heads, head_dim, out, out_off,
                                     layer, reinterpret_cast<cudaStream_t>(stream));
}
