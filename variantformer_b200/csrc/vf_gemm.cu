// vf_gemm.cu — bf16 GEMM  D[M,N] = A[M,K] · W[N,K]^T  (+ fused epilogues) on the
// 5th-gen tensor cores: TMA (128B-swizzled K-major tiles) -> shared memory ->
// tcgen05.mma with fp32 accumulators in TMEM -> tcgen05.ld epilogue.
//
// Replaces every nn.Linear on the reference's hot path (cuBLASLt under autocast):
//   seq2reg/modules.py:140-147 (Wqkv, out_proj, linear_geglu_1/2),
//   seq2gene/modules/layers.py:63-80 (mixer/crossMHA projections, GeGLU FFN),
//   seq2gene/model_combined_modulator.py:502-507 (gene_map, cre_map),
//   seq2gene/modules/layers.py:1078-1087 (head Linear layers).
//
// Kernel shape: persistent, one CTA per SM, 384 threads = 3 warpgroups:
//   warp 0    : TMA producer (one elected lane)       smem ring of kStages x (A 128x64 + W 256x64) bf16
//   warp 1    : TMEM allocator + tcgen05.mma issuer   UMMA 128x256x16, 4 per k-block
//   warps 2-3 : idle (they only exist so that warpgroup 0 can give its registers away with setmaxnreg)
//   warps 4-11: epilogue (TMEM lane quadrant = warp%4, two warps per quadrant), 232 registers each: pipelined
//               tcgen05.ld, LayerNorm fold / bias / GeGLU / GELU / +residual, transposed through a swizzled smem
//               tile for fully coalesced stores, optional bf16 mirror and per-row (sum, sum of squares)
// Two 256-column fp32 accumulators (all 512 TMEM columns) double-buffer the
// epilogue of tile i against the mainloop of tile i+1.
//
// LayerNorm fold (seq2reg/modules.py:143-144, layers.py:74-76 feed every LN straight into a Linear):
//   LN(x) W^T + b = rstd_r * (x (W*gamma)^T - mean_r * colsum(W*gamma)) + (b + W beta)
// so a GEMM whose A operand is the bf16 mirror of the un-normalised fp32 stream, with gamma folded into W at load
// time, only needs the per-row (sum, sum of squares) of x in its epilogue.  Those are written by the epilogue
// of the GEMM that PRODUCED x (stats_out) as one partial per (column tile, epilogue half) — plain stores, summed in a
// fixed order by the consumer, so results are bit-reproducible — and no separate LayerNorm pass ever reads the stream.
#include <cuda.h>
#include <stdio.h>

#include "vf_common.cuh"
#include "vf_internal.h"

namespace vf {

constexpr int BM = 128, BN = 256, BK = 64, kStages = 4;
constexpr int kStagesPair = 6;                        // CTA-pair kernel: 6 x 32 KB stages in the same shared memory
constexpr int kEpiWarps = 8;                          // two warps per TMEM lane quadrant
constexpr int kFirstEpiWarp = 4;                      // warpgroup 0 = TMA + MMA (+2 idle warps), warpgroups 1-2 = epilogue
constexpr int kGemmThreads = (kFirstEpiWarp + kEpiWarps) * 32;
constexpr uint32_t kTmemCols = 512;
constexpr uint32_t kABytes = BM * BK * 2, kBBytes = BN * BK * 2, kStageBytes = kABytes + kBBytes;
constexpr uint32_t kStageOutBytes = 32 * 32 * 4;      // per-epilogue-warp staging tile: 32 rows x 32 fp32 columns
constexpr uint32_t kColVecBytes = 2 * BN * 4;         // bias and LayerNorm column sums of the tile's 256 columns
// (no alignment slack: the dynamic shared memory of a kernel without static shared memory starts 1 KB aligned; the
// kernel traps otherwise)
constexpr size_t kGemmSmem = (size_t)kStages * kStageBytes + kEpiWarps * kStageOutBytes + 256 /*barriers*/ + kColVecBytes;
// "RT" residual epilogue (CTA-pair kernel, bf16 residual in, bf16 mirror + row statistics out: the out_proj shapes): the
// residual slabs come in by TMA into a per-warp ring (3 x 2 KB, SWIZZLE_64B) and the mirror slabs leave by TMA from a
// 2 KB tile, so a warp owns 8 KB instead of 4; one operand stage (32 KB) pays for it.
constexpr int kStagesPairRT = 5, kStagesPairRT2 = 4;      // (RT 2, the FFN2 form: 12 KB per warp, see the epilogue)
constexpr uint32_t kStageOutBytesRT = 8192, kStageOutBytesRT2 = 12288, kBarBytesRT = 512;
constexpr size_t kGemmSmemRT = (size_t)kStagesPairRT * (kABytes + kBBytes / 2) + kEpiWarps * kStageOutBytesRT + kBarBytesRT + kColVecBytes;
static_assert(kGemmSmemRT <= 227 * 1024, "shared memory budget (RT)");
static_assert((size_t)kStagesPairRT2 * (kABytes + kBBytes / 2) + kEpiWarps * kStageOutBytesRT2 + kBarBytesRT + kColVecBytes <= kGemmSmemRT, "RT 2 fits the RT budget");

struct GemmParams {
    int M, N, K;
    const float* bias;       // [N] (GeGLU: tile-interleaved like W) or nullptr
    const float* resid;      // fp32 [M, ldr] or nullptr
    const __nv_bfloat16* resid16;   // ... or a bf16 residual [M, ldr] (intra-layer temporaries, see engine.py)
    int ldr;
    void* out;               // bf16 or fp32, row stride ldo (elements)
    int ldo;
    __nv_bfloat16* out2;     // optional bf16 mirror of an fp32 output (row stride ldo2)
    int ldo2;
    const float* ln_stats;   // LayerNorm fold: fp32 [M, ln_parts, 2] partial (sum, sum of squares) of the rows A mirrors
    int ln_parts;            //                 (nullptr = no fold)
    const float* ln_colsum;  //                 fp32 [N] column sums of the gamma-folded weight (layout of `bias`)
    float ln_inv_d, ln_eps;  //                 1 / normalised width, eps
    float* stats_out;        // fp32 outputs: partial (sum, sum of squares) of every output row -> [M, 2*n_tiles, 2], or nullptr
    int tile_chunked;        // tile schedule: 1 = each unit walks a contiguous run of tiles (n fastest), 0 = round-robin
};

template <int EPI>
constexpr bool epi_is_bf16() {
    return EPI == VF_EPI_BIAS_BF16 || EPI == VF_EPI_BIAS_GEGLU_BF16 || EPI == VF_EPI_BIAS_GELU_BF16;
}

// One 32-row x 32-column slab (thread = row, v = its 32 finished values) -> global memory, transposed through the
// warp's private shared-memory tile so that every global access is a run of full 32-byte sectors:
//   bf16 out : rows are 64 B; a warp instruction stores 8 rows x 64 B
//   fp32 out : rows are 128 B; a warp instruction loads the residual / stores 4 rows x 128 B
// 16-byte chunks are XOR-swizzled inside the tile so both the row-wise writes and the column-wise reads are
// bank-conflict free.
// Residual slab prefetch: the 8 float4 this lane will add in the coalesced phase (4 rows x 128 B per warp request).
// Issued as one batch well before they are needed so the memory latency overlaps the TMEM load and the staging writes
// (loads cannot be hoisted by the compiler itself: `out` may alias `resid`).
__device__ __forceinline__ void load_resid_slab(const GemmParams& p, int row0, int col0, int lane, float4 (&rr4)[8]) {
    // interior slab (warp-uniform test): one base pointer, constant row stride, no per-row predicates — the bounds
    // checks, 64-bit address products and the branches around them were ~45 % of the residual epilogue's instructions
    if (row0 + 32 <= p.M && col0 + 32 <= p.N) {
        const int r = row0 + (lane >> 3), c = col0 + (lane & 7) * 4;
        if (p.resid16) {
            const __nv_bfloat16* src = p.resid16 + (size_t)r * p.ldr + c;
            const size_t st = 4 * (size_t)p.ldr;
#pragma unroll
            for (int it = 0; it < 8; ++it) {
                const uint2 h = *reinterpret_cast<const uint2*>(src + it * st);
                rr4[it] = make_float4(__uint_as_float(h.x), __uint_as_float(h.y), 0.f, 0.f);
            }
            return;
        }
        if (p.resid) {
            const float* src = p.resid + (size_t)r * p.ldr + c;
            const size_t st = 4 * (size_t)p.ldr;
#pragma unroll
            for (int it = 0; it < 8; ++it) rr4[it] = *reinterpret_cast<const float4*>(src + it * st);
            return;
        }
    }
#pragma unroll
    for (int it = 0; it < 8; ++it) {
        const int grow = row0 + it * 4 + (lane >> 3), gcol = col0 + (lane & 7) * 4;
        const bool ok = grow < p.M && gcol + 4 <= p.N;
        if (p.resid16) {
            uint2 h = make_uint2(0u, 0u);
            if (ok) h = *reinterpret_cast<const uint2*>(p.resid16 + (size_t)grow * p.ldr + gcol);
            // raw bits only: widening them HERE would put a consumer right behind the load and stall the warp for
            // the whole DRAM round trip (measured: the bf16-residual epilogue ran 2x slower than the fp32 one)
            rr4[it] = make_float4(__uint_as_float(h.x), __uint_as_float(h.y), 0.f, 0.f);
        } else {
            rr4[it] = (p.resid && ok) ? *reinterpret_cast<const float4*>(p.resid + (size_t)grow * p.ldr + gcol)
                                      : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    }
}

// Per-warp running (sum, sum of squares) of the fp32 rows it stores: lane holds the partial of rows it*4 + (lane>>3)
// over its own 4 columns of every slab; reduced over the 8 lanes of a row group once per tile.
struct RowStats {
    float s1[8], s2[8];
    __device__ __forceinline__ void clear() {
#pragma unroll
        for (int i = 0; i < 8; ++i) { s1[i] = 0.f; s2[i] = 0.f; }
    }
    // 8 values x 8 lanes -> lane k of each 8-lane group ends with the group total of value k (7 shuffles per array)
    static __device__ __forceinline__ float reduce8(const float (&s)[8], int lane) {
        float t[4], u[2];
        const bool b4 = lane & 4, b2 = lane & 2, b1 = lane & 1;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            const float mine = b4 ? s[i + 4] : s[i], other = b4 ? s[i] : s[i + 4];
            t[i] = mine + __shfl_xor_sync(0xffffffffu, other, 4);
        }
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const float mine = b2 ? t[i + 2] : t[i], other = b2 ? t[i] : t[i + 2];
            u[i] = mine + __shfl_xor_sync(0xffffffffu, other, 2);
        }
        const float mine = b1 ? u[1] : u[0], other = b1 ? u[0] : u[1];
        return mine + __shfl_xor_sync(0xffffffffu, other, 1);
    }
    __device__ __forceinline__ void flush(float* stats_out, int row0, int M, int part, int parts, int lane) {
        const float a = reduce8(s1, lane), b = reduce8(s2, lane);
        const int grow = row0 + (lane & 7) * 4 + (lane >> 3);          // lane publishes row (lane&7)*4 + (lane>>3)
        if (grow < M) *reinterpret_cast<float2*>(stats_out + 2 * ((size_t)grow * parts + part)) = make_float2(a, b);
    }
};

template <int EPI>
__device__ __forceinline__ void epilogue_store_slab(const GemmParams& p, uint32_t stage, int row0, int col0, int n_out,
                                                    const float (&v)[32], int lane, const float4 (&rr4)[8],
                                                    RowStats& rs, const CUtensorMap* tmO = nullptr, int half_buf = 0) {
    // `stage` = shared-space address of the warp's 4 KB tile.
    if constexpr (epi_is_bf16<EPI>()) {
        // The slab leaves through ONE bulk tensor store: the staging layout ([32 rows][4 chunks of 16 B], chunk index
        // XOR (row >> 1) & 3) is exactly SWIZZLE_64B, so the TMA unit reads it as it lies; rows / columns past M / N
        // are clipped by the hardware.  The warp's 4 KB tile holds two bf16 slabs: while one is being read out by the
        // TMA unit the next is written (at most one store group outstanding when a half is rewritten).
        stage += half_buf * 2048;
        if (lane == 0) tma_store_wait_read<1>();
        __syncwarp();
#pragma unroll
        for (int j = 0; j < 4; ++j)
            sts128(stage + (lane * 4 + (j ^ ((lane >> 1) & 3))) * 16, pack_bf16x2(v[j * 8 + 0], v[j * 8 + 1]),
                   pack_bf16x2(v[j * 8 + 2], v[j * 8 + 3]), pack_bf16x2(v[j * 8 + 4], v[j * 8 + 5]),
                   pack_bf16x2(v[j * 8 + 6], v[j * 8 + 7]));
        fence_proxy_async_smem();
        __syncwarp();
        if (lane == 0) { tma_store_2d(tmO, stage, col0, row0); tma_store_commit(); }
    } else {
        // All reads of the transposed tile are issued as one batch (no branch in between), then the global stores follow.
#pragma unroll
        for (int j = 0; j < 8; ++j)                                     // [32 rows][8 chunks of 16 B]
            sts128(stage + (lane * 8 + (j ^ (lane & 7))) * 16, __float_as_uint(v[j * 4]), __float_as_uint(v[j * 4 + 1]),
                   __float_as_uint(v[j * 4 + 2]), __float_as_uint(v[j * 4 + 3]));
        __syncwarp();
        uint4 q[8];
#pragma unroll
        for (int it = 0; it < 8; ++it) {
            const int rr = it * 4 + (lane >> 3), jj = lane & 7;
            q[it] = lds128(stage + (rr * 8 + (jj ^ (rr & 7))) * 16);
        }
        __syncwarp();
        float* o = reinterpret_cast<float*>(p.out);
        const int gcol = col0 + (lane & 7) * 4;
        if (row0 + 32 <= p.M && col0 + 32 <= n_out) {                   // interior slab (warp-uniform): see load_resid_slab
            const int r = row0 + (lane >> 3);
            float* op = o ? o + (size_t)r * p.ldo + gcol : nullptr;
            __nv_bfloat16* mp = p.out2 ? p.out2 + (size_t)r * p.ldo2 + gcol : nullptr;
            const size_t so = 4 * (size_t)p.ldo, sm = 4 * (size_t)p.ldo2;
#pragma unroll
            for (int it = 0; it < 8; ++it) {
                float4 f = make_float4(__uint_as_float(q[it].x), __uint_as_float(q[it].y), __uint_as_float(q[it].z),
                                       __uint_as_float(q[it].w));
                if constexpr (EPI == VF_EPI_BIAS_RESID_F32) {
                    float4 rv = rr4[it];
                    if (p.resid16) {
                        const uint32_t hx = __float_as_uint(rv.x), hy = __float_as_uint(rv.y);
                        rv = make_float4(__uint_as_float(hx << 16), __uint_as_float(hx & 0xffff0000u),
                                         __uint_as_float(hy << 16), __uint_as_float(hy & 0xffff0000u));
                    }
                    f.x += rv.x; f.y += rv.y; f.z += rv.z; f.w += rv.w;
                }
                if (op) *reinterpret_cast<float4*>(op + it * so) = f;
                if (mp) {
                    uint2 h; h.x = pack_bf16x2(f.x, f.y); h.y = pack_bf16x2(f.z, f.w);
                    *reinterpret_cast<uint2*>(mp + it * sm) = h;
                }
                rs.s1[it] += (f.x + f.y) + (f.z + f.w);
                rs.s2[it] += fmaf(f.x, f.x, f.y * f.y) + fmaf(f.z, f.z, f.w * f.w);
            }
            return;
        }
        if (gcol + 4 <= n_out) {
#pragma unroll
            for (int it = 0; it < 8; ++it) {
                const int grow = row0 + it * 4 + (lane >> 3);
                float4 f = make_float4(__uint_as_float(q[it].x), __uint_as_float(q[it].y), __uint_as_float(q[it].z),
                                       __uint_as_float(q[it].w));
                if constexpr (EPI == VF_EPI_BIAS_RESID_F32) {
                    float4 rv = rr4[it];
                    if (p.resid16) {                          // bf16 pairs travel as raw bits (load_resid_slab)
                        const uint32_t hx = __float_as_uint(rv.x), hy = __float_as_uint(rv.y);
                        rv = make_float4(__uint_as_float(hx << 16), __uint_as_float(hx & 0xffff0000u),
                                         __uint_as_float(hy << 16), __uint_as_float(hy & 0xffff0000u));
                    }
                    f.x += rv.x; f.y += rv.y; f.z += rv.z; f.w += rv.w;
                }
                if (grow < p.M) {
                    if (o) *reinterpret_cast<float4*>(o + (size_t)grow * p.ldo + gcol) = f;
                    if (p.out2) {
                        uint2 h; h.x = pack_bf16x2(f.x, f.y); h.y = pack_bf16x2(f.z, f.w);
                        *reinterpret_cast<uint2*>(p.out2 + (size_t)grow * p.ldo2 + gcol) = h;
                    }
                    rs.s1[it] += (f.x + f.y) + (f.z + f.w);
                    rs.s2[it] += fmaf(f.x, f.x, f.y * f.y) + fmaf(f.z, f.z, f.w * f.w);
                }
            }
        }
    }
}

// CTAS = 1: one CTA per 128 x 256 tile.  CTAS = 2: a CTA PAIR (cluster of 2, tcgen05 cta_group::2) per 256 x 256
// tile: each CTA stages its own 128 A rows and HALF of the W rows (32 KB per stage instead of 48: a third less
// L2 -> SM operand traffic and room for more stages), the pair leader issues M=256 MMAs that read both CTAs' shared
// memory and write each CTA's 128 accumulator rows into its own TMEM; every CTA runs its own epilogue.
template <int EPI, int CTAS, int RT = 0>
__global__ void __cluster_dims__(CTAS, 1, 1) __launch_bounds__(kGemmThreads, 1)
gemm_tcgen05_kernel(const __grid_constant__ CUtensorMap tmA, const __grid_constant__ CUtensorMap tmB,
                    const __grid_constant__ CUtensorMap tmR, const __grid_constant__ CUtensorMap tmO,
                    const GemmParams p_in) {
    // Local copy: the fields live in registers.  Read through the parameter itself they are re-fetched from the
    // constant bank (LDCU, a scoreboard wait each) after every asm statement with a memory clobber — in the epilogue
    // that is several times per slab.
    const GemmParams p = p_in;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = smem_raw;
    if (smem_u32(smem_raw) & 1023u) __trap();                // SWIZZLE_128B tiles need 1 KB alignment
    static_assert(RT == 0 || (CTAS == 2 && EPI == VF_EPI_BIAS_RESID_F32), "RT is a variant of the pair kernel's residual epilogue");
    constexpr int kStg = CTAS == 2 ? (RT == 2 ? kStagesPairRT2 : RT == 1 ? kStagesPairRT : kStagesPair) : kStages;
    constexpr uint32_t kBBytesC = kBBytes / CTAS, kStageBytesC = kABytes + kBBytesC;
    constexpr uint32_t kOutW = RT == 2 ? kStageOutBytesRT2 : RT == 1 ? kStageOutBytesRT : kStageOutBytes;
    uint8_t* smem_a = smem;                                  // kStg x 16 KB
    uint8_t* smem_b = smem + kStg * kABytes;                 // kStg x 32 KB (16 KB per CTA of a pair)
    uint8_t* smem_out = smem + kStg * kStageBytesC;          // kEpiWarps x 4 KB staging tiles (RT: 8 KB)
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_out + kEpiWarps * kOutW);
    uint64_t* full = bars;                 // [kStg]
    uint64_t* empty = bars + kStg;         // [kStg]
    uint64_t* tmem_full = bars + 2 * kStg;          // [2]
    uint64_t* tmem_empty = bars + 2 * kStg + 2;     // [2]
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * kStg + 4);
    uint64_t* rbars = bars + 2 * kStg + 6;                   // RT: [kEpiWarps][3] "residual slab landed"
    const uint32_t colvec = smem_u32(bars) + (RT ? kBarBytesRT : 256u);   // [256] bias | [256] LayerNorm column sums (shared-space address)

    const int warp = threadIdx.x >> 5;
    // work unit = CTA (CTAS 1) or CTA pair (CTAS 2); `rank` = this CTA's half of the pair's 256 rows / 256 W rows
    const int unit = CTAS == 2 ? (int)(blockIdx.x >> 1) : (int)blockIdx.x;
    const int n_units = CTAS == 2 ? (int)(gridDim.x >> 1) : (int)gridDim.x;
    const int rank = CTAS == 2 ? (int)cluster_ctarank() : 0;
    const int m_tiles = (p.M + BM * CTAS - 1) / (BM * CTAS), n_tiles = (p.N + BN - 1) / BN;
    const int num_tiles = m_tiles * n_tiles;
    // Tile schedule of this unit: t = t_first + i * t_step, i < t_count.  Tiles are numbered n-fastest.  "chunked": a unit
    // owns a contiguous run, i.e. it walks the n-tiles of one row block one after the other, so the LayerNorm row
    // statistics are reduced once per row block instead of once per tile (their load was the top stall of the K = 512
    // epilogues) and the A tile is re-read while it is hot.  "strided": round-robin over the units.
    int t_first, t_step, t_count;
    if (p.tile_chunked) {
        const int per = (num_tiles + n_units - 1) / n_units;
        t_first = unit * per; t_step = 1; t_count = max(0, min(per, num_tiles - t_first));
    } else {
        t_first = unit; t_step = n_units; t_count = unit < num_tiles ? (num_tiles - unit + n_units - 1) / n_units : 0;
    }
    const int k_blocks = (p.K + BK - 1) / BK;

    if (warp == 0 && elect_one()) {
        tma_prefetch_desc(&tmA);
        tma_prefetch_desc(&tmB);
        if constexpr (RT != 0) { tma_prefetch_desc(&tmR); tma_prefetch_desc(&tmO); }
        if constexpr (epi_is_bf16<EPI>()) tma_prefetch_desc(&tmO);
        for (int s = 0; s < kStg; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
        // the leader's tmem_empty collects the epilogue warps of BOTH CTAs of a pair
        for (int a = 0; a < 2; ++a) { mbar_init(&tmem_full[a], 1); mbar_init(&tmem_empty[a], kEpiWarps * CTAS); }
        if constexpr (RT != 0) for (int i = 0; i < kEpiWarps * 3; ++i) mbar_init(&rbars[i], 1);
        fence_barrier_init();
    }
    if constexpr (CTAS == 2) cluster_sync_all();             // both CTAs' barriers exist before anyone signals the peer's
    if (warp == 1) {
        if constexpr (CTAS == 2) { tmem_alloc_pair(tmem_slot, kTmemCols); tmem_relinquish_pair(); }
        else { tmem_alloc(tmem_slot, kTmemCols); tmem_relinquish(); }
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;

    if (warp < kFirstEpiWarp) {
        reg_dealloc<40>();                                   // warpgroup 0 hands its registers to the epilogue warps
        if (warp == 0) {
            // ================= TMA producer =================
            if (elect_one()) {
                int stage = 0; uint32_t phase = 0;
                for (int ti = 0; ti < t_count; ++ti) {
                    const int t = t_first + ti * t_step;
                    const int m0 = (t / n_tiles) * BM * CTAS + rank * BM, n0 = (t % n_tiles) * BN;
                    for (int kb = 0; kb < k_blocks; ++kb) {
                        mbar_wait(&empty[stage], phase ^ 1);
                        if constexpr (CTAS == 2) {
                            // all four loads of the pair complete on the LEADER's barrier, which expects their total
                            if (rank == 0) mbar_arrive_expect_tx(&full[stage], 2 * kStageBytesC);
                            tma_load_2d_pair(smem_a + stage * kABytes, &tmA, &full[stage], kb * BK, m0);
                            tma_load_2d_pair(smem_b + stage * kBBytesC, &tmB, &full[stage], kb * BK, n0 + rank * (BN / 2));
                        } else {
                            mbar_arrive_expect_tx(&full[stage], kStageBytes);
                            tma_load_2d(smem_a + stage * kABytes, &tmA, &full[stage], kb * BK, m0);
                            tma_load_2d(smem_b + stage * kBBytes, &tmB, &full[stage], kb * BK, n0);
                        }
                        if (++stage == kStg) { stage = 0; phase ^= 1; }
                    }
                }
            }
            __syncwarp();
        } else if (warp == 1) {
            // ================= MMA issuer =================
            if (rank == 0 && elect_one()) {                  // the pair's leader issues for both CTAs
                constexpr uint32_t idesc = umma_idesc_bf16(BM * CTAS, BN);
                int stage = 0; uint32_t phase = 0; int it = 0;
                for (; it < t_count; ++it) {
                    const int acc = it & 1; const uint32_t acc_phase = (it >> 1) & 1;
                    mbar_wait(&tmem_empty[acc], acc_phase ^ 1);
                    tc_fence_after();
                    const uint32_t d_tmem = tmem_base + acc * BN;
                    for (int kb = 0; kb < k_blocks; ++kb) {
                        mbar_wait(&full[stage], phase);
                        tc_fence_after();
                        const uint64_t da = umma_desc_kmajor_sw128(smem_u32(smem_a + stage * kABytes));
                        const uint64_t db = umma_desc_kmajor_sw128(smem_u32(smem_b + stage * kBBytesC));
#pragma unroll
                        for (int k = 0; k < BK / 16; ++k) {
                            // +32 bytes per UMMA_K step inside the 128-byte swizzle row (start address is in 16 B units)
                            if constexpr (CTAS == 2) umma_bf16_pair(d_tmem, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0);
                            else umma_bf16(d_tmem, da + 2 * k, db + 2 * k, idesc, (kb | k) != 0);
                        }
                        if constexpr (CTAS == 2) {                       // (multicast: the barrier of BOTH CTAs)
                            umma_commit_pair(&empty[stage]);
                            if (kb == k_blocks - 1) umma_commit_pair(&tmem_full[acc]);
                        } else {
                            umma_commit(&empty[stage]);                  // frees the smem slot when these MMAs retire
                            if (kb == k_blocks - 1) umma_commit(&tmem_full[acc]);
                        }
                        if (++stage == kStg) { stage = 0; phase ^= 1; }
                    }
                }
            }
            __syncwarp();
        }
    } else {
        // ================= epilogue warps =================
        // warp%4 selects the TMEM lane quadrant (hardware rule); the two warps of a quadrant interleave the
        // 32-column slabs (even / odd).  TMEM loads are software-pipelined: slab i+1 is in flight while slab i is
        // converted and stored.
        reg_alloc<232>();
        const int quad = warp & 3;
        const int half = (warp - kFirstEpiWarp) >> 2;
        const int lane = threadIdx.x & 31;
        const uint32_t stage_out = smem_u32(smem_out + (warp - kFirstEpiWarp) * kOutW);
        constexpr int kSlabs = (EPI == VF_EPI_BIAS_GEGLU_BF16) ? 2 : 4;      // per warp per tile
        const int n_out = (EPI == VF_EPI_BIAS_GEGLU_BF16) ? p.N / 2 : p.N;
        const bool ln = epi_is_bf16<EPI>() && p.ln_stats != nullptr;
        const bool want_stats = !epi_is_bf16<EPI>() && p.stats_out != nullptr;
        RowStats rs;
        float4 rr4[4][8];                                     // residual of slab i of a tile (RESID epilogue only)
        // RT: slab stream of this warp: slab G = (tile G / 4 of the unit's schedule, column slab half + 2 * (G % 4)); ring
        // slot G % 3; lane 0 keeps the loads of the next two slabs in flight.
        const SmemBar rbar = smem_bar(rbars + (warp - kFirstEpiWarp) * 3);
        uint32_t rt_g = 0;                                    // slabs consumed so far
        auto rt_issue = [&](uint32_t G) {                     // (lane 0 only)
            const int ti = (int)(G >> 2);
            if (ti >= t_count) return;
            const int tt = t_first + ti * t_step;
            const int r0 = (tt / n_tiles) * BM * CTAS + rank * BM + quad * 32, c0 = (tt % n_tiles) * BN + (half + 2 * (int)(G & 3)) * 32;
            if constexpr (RT == 2) {                          // fp32 slabs: two 4 KB slots
                const uint32_t k = G & 1;
                mbar_arrive_expect_tx(rbar[k], 4096);
                tma_load_2d(stage_out + k * 4096, &tmR, rbar[k], c0, r0);
            } else {                                          // bf16 slabs: three 2 KB slots
                const uint32_t k = G % 3;
                mbar_arrive_expect_tx(rbar[k], 2048);
                tma_load_2d(stage_out + k * 2048, &tmR, rbar[k], c0, r0);
            }
        };
        if constexpr (RT == 1) {
            if (lane == 0) { rt_issue(0); rt_issue(1); }
        }
        if constexpr (RT == 2) {
            if (lane == 0) rt_issue(0);
        }
        if constexpr (EPI == VF_EPI_BIAS_RESID_F32 && RT == 0) {
            if (t_count > 0) {                                // prime the slab stream: slabs 0 and 1 of the first tile
                const int m0f = (t_first / n_tiles) * BM * CTAS + rank * BM, n0f = (t_first % n_tiles) * BN;
                load_resid_slab(p, m0f + quad * 32, n0f + half * 32, lane, rr4[0]);
                load_resid_slab(p, m0f + quad * 32, n0f + (half + 2) * 32, lane, rr4[1]);
                load_resid_slab(p, m0f + quad * 32, n0f + (half + 4) * 32, lane, rr4[2]);
            }
        }
        int last_m0 = -1;
        float ln_a = 1.f, ln_c = 0.f;
        // Per-column epilogue vectors of a tile (bias, LayerNorm column sums) go through shared memory: one value per
        // epilogue thread, requested a whole tile ahead, instead of 16-32 global loads per slab and warp whose L2 latency
        // sat on the critical path of the K = 512 epilogues (39 % of their samples on the long scoreboard; only ~28 KB of
        // L1 is left next to the operand ring).
        const int etid = threadIdx.x - kFirstEpiWarp * 32;    // 0..255 = column of the tile
        auto col_values = [&](int tile, float& b, float& cs) {
            const int col = (tile % n_tiles) * BN + etid;
            b = (p.bias && col < p.N) ? __ldg(p.bias + col) : 0.f;
            cs = (ln && col < p.N) ? __ldg(p.ln_colsum + col) : 0.f;
        };
        float nb = 0.f, ncs = 0.f;
        if (t_count > 0) col_values(t_first, nb, ncs);
        for (int it = 0; it < t_count; ++it) {
            const int t = t_first + it * t_step;
            const int acc = it & 1; const uint32_t acc_phase = (it >> 1) & 1;
            const int m0 = (t / n_tiles) * BM * CTAS + rank * BM, n0 = (t % n_tiles) * BN;
            const int row0 = m0 + quad * 32;
            asm volatile("bar.sync 1, %0;" ::"n"(kEpiWarps * 32) : "memory");      // previous tile's vectors are no longer read
            asm volatile("st.shared.f32 [%0], %1;" ::"r"(colvec + etid * 4), "f"(nb) : "memory");
            asm volatile("st.shared.f32 [%0], %1;" ::"r"(colvec + BN * 4 + etid * 4), "f"(ncs) : "memory");
            asm volatile("bar.sync 1, %0;" ::"n"(kEpiWarps * 32) : "memory");
            if (it + 1 < t_count) col_values(t + t_step, nb, ncs);
            // LayerNorm fold: this thread's row is normalised as  ln_a * acc + ln_c * colsum[n] + bias'[n]; the pair is
            // kept while the unit stays on the same row block
            if (ln && m0 != last_m0) { ln_a = 1.f; ln_c = 0.f; }
            if (ln && m0 != last_m0 && row0 + lane < p.M) {
                const float2* sp = reinterpret_cast<const float2*>(p.ln_stats) + (size_t)(row0 + lane) * p.ln_parts;
                float2 st = make_float2(0.f, 0.f);
                if (p.ln_parts > 1 && p.ln_parts <= 16 && (p.ln_parts & 1) == 0) {
                    // the row's partials as ONE batch of 16-byte loads (a dependent loop pays a memory round trip per
                    // partial: 12 per tile for a 1536-wide stream), summed in index order.  (Requesting them a whole
                    // tile ahead was measured: no gain, 32 more live registers.)
                    float4 q[8];
#pragma unroll
                    for (int i = 0; i < 8; ++i)
                        q[i] = 2 * i < p.ln_parts ? __ldg(reinterpret_cast<const float4*>(sp) + i) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
                    for (int i = 0; i < 8; ++i) { st.x += q[i].x; st.y += q[i].y; st.x += q[i].z; st.y += q[i].w; }
                } else {
                    st = __ldg(sp);
                    for (int i = 1; i < p.ln_parts; ++i) { const float2 t2 = __ldg(sp + i); st.x += t2.x; st.y += t2.y; }
                }
                const float mean = st.x * p.ln_inv_d;
                const float var = fmaxf(fmaf(st.y, p.ln_inv_d, -mean * mean), 0.f);
                ln_a = rsqrtf(var + p.ln_eps);
                ln_c = -ln_a * mean;
            }
            last_m0 = m0;
            rs.clear();
            mbar_wait(&tmem_full[acc], acc_phase);
            tc_fence_after();
            const uint32_t t_row = tmem_base + ((uint32_t)(quad * 32) << 16) + acc * BN;
            if constexpr (EPI == VF_EPI_BIAS_GEGLU_BF16) {
                // W rows are tile-interleaved: accumulator columns [0,128) = u, [128,256) = gate of the same 128
                // output columns (layers.py:159-160: u, gate = chunk(2); out = u * gelu(gate)).
                const int out0 = (n0 / BN) * (BN / 2);
                uint32_t ru[2][32], rg[2][32];
                tmem_ld_32x32(t_row + half * 32, ru[0]);
                tmem_ld_32x32(t_row + 128 + half * 32, rg[0]);
#pragma unroll
                for (int i = 0; i < kSlabs; ++i) {
                    const int c = half + 2 * i;                           // 32-column slab of the 128 outputs
                    tmem_ld_wait();
                    if (i + 1 < kSlabs) {
                        tmem_ld_32x32(t_row + (c + 2) * 32, ru[(i + 1) & 1]);
                        tmem_ld_32x32(t_row + 128 + (c + 2) * 32, rg[(i + 1) & 1]);
                    }
                    float v[32];
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        // bias (+ LayerNorm column-sum term) of these four columns, from the tile's shared-memory vectors
                        // (read where they are used: as arrays they cost 64 registers the packed arithmetic needs)
                        float4 b0 = lds_f4(colvec + (c * 32 + j) * 4), b1 = lds_f4(colvec + (128 + c * 32 + j) * 4);
                        if (ln) {
                            const float4 su = lds_f4(colvec + (BN + c * 32 + j) * 4), sg = lds_f4(colvec + (BN + 128 + c * 32 + j) * 4);
                            b0.x = fmaf(ln_c, su.x, b0.x); b0.y = fmaf(ln_c, su.y, b0.y); b0.z = fmaf(ln_c, su.z, b0.z); b0.w = fmaf(ln_c, su.w, b0.w);
                            b1.x = fmaf(ln_c, sg.x, b1.x); b1.y = fmaf(ln_c, sg.y, b1.y); b1.z = fmaf(ln_c, sg.z, b1.z); b1.w = fmaf(ln_c, sg.w, b1.w);
                        }
                        // u * gelu(gate) on packed pairs (FFMA2 / FMUL2)
                        const uint64_t la2 = f2_bcast(ln_a);
                        float g0, g1, g2, g3, y0, y1, y2, y3;
                        f2_unpack(f2_fma(f2_pack(rg[i & 1][j + 0], rg[i & 1][j + 1]), la2, f2_pack(b1.x, b1.y)), g0, g1);
                        f2_unpack(f2_fma(f2_pack(rg[i & 1][j + 2], rg[i & 1][j + 3]), la2, f2_pack(b1.z, b1.w)), g2, g3);
                        gelu_erf_fast2(g0, g1, y0, y1);
                        gelu_erf_fast2(g2, g3, y2, y3);
                        const uint64_t u01 = f2_fma(f2_pack(ru[i & 1][j + 0], ru[i & 1][j + 1]), la2, f2_pack(b0.x, b0.y));
                        const uint64_t u23 = f2_fma(f2_pack(ru[i & 1][j + 2], ru[i & 1][j + 3]), la2, f2_pack(b0.z, b0.w));
                        f2_unpack(f2_mul(u01, f2_pack(y0, y1)), v[j + 0], v[j + 1]);
                        f2_unpack(f2_mul(u23, f2_pack(y2, y3)), v[j + 2], v[j + 3]);
                    }
                    float4 none[8];
                    epilogue_store_slab<EPI>(p, stage_out, row0, out0 + c * 32, n_out, v, lane, none, rs, &tmO, i & 1);
                }
            } else if constexpr (RT == 2) {
                // FFN2 form, IN PLACE (out == resid: the fp32 stream): a slab's residual arrives by TMA in a SWIZZLE_128B
                // tile, the sum is formed in the accumulator's layout (lane = row) and written back into the same tile,
                // which then leaves by a bulk tensor store through the same tensor map; the mirror leaves from a 2 KB
                // SWIZZLE_64B tile.  Two fp32 slots and two mirror tiles per warp: while slab G is computed, slot G ^ 1
                // (stored at the end of slab G - 1) is refilled with slab G + 1 — a lead of one slab (2-4 us, several DRAM
                // round trips).
                // Row statistics in EXACTLY the association of the register-prefetch epilogue (RowStats: one partial per
                // group of four columns, slabs added in order, then ((S0+S4)+(S2+S6)) + ((S1+S5)+(S3+S7))): which kernel a
                // GEMM runs through depends on M, and results must not depend on how rows are batched.
                float st1[8], st2[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) { st1[j] = 0.f; st2[j] = 0.f; }
                uint32_t r[32];
#pragma unroll
                for (int i = 0; i < kSlabs; ++i) {
                    const int c = half + 2 * i;
                    const int col0 = n0 + c * 32;
                    const uint32_t k = rt_g & 1;
                    const uint32_t slot = stage_out + k * 4096, mt = stage_out + 8192 + k * 2048;
                    if (lane == 0) { tma_store_wait_read<0>(); rt_issue(rt_g + 1); }   // slot k ^ 1 has been read out
                    tmem_ld_32x32(t_row + c * 32, r);
                    float4 bb[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) bb[j] = lds_f4(colvec + (c * 32 + 4 * j) * 4);
                    mbar_wait(rbar[k], (rt_g >> 1) & 1);
                    float4 rq[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) rq[j] = lds_f4(slot + (lane * 8 + (j ^ (lane & 7))) * 16);
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 8; ++j) {
                        float4 f;
                        f.x = (__uint_as_float(r[4 * j + 0]) + bb[j].x) + rq[j].x;
                        f.y = (__uint_as_float(r[4 * j + 1]) + bb[j].y) + rq[j].y;
                        f.z = (__uint_as_float(r[4 * j + 2]) + bb[j].z) + rq[j].z;
                        f.w = (__uint_as_float(r[4 * j + 3]) + bb[j].w) + rq[j].w;
                        st1[j] += (f.x + f.y) + (f.z + f.w);
                        st2[j] += fmaf(f.x, f.x, f.y * f.y) + fmaf(f.z, f.z, f.w * f.w);
                        rq[j] = f;
                    }
#pragma unroll
                    for (int j = 0; j < 8; ++j)
                        sts128(slot + (lane * 8 + (j ^ (lane & 7))) * 16, __float_as_uint(rq[j].x), __float_as_uint(rq[j].y),
                               __float_as_uint(rq[j].z), __float_as_uint(rq[j].w));
                    if (p.out2) {
#pragma unroll
                        for (int j = 0; j < 4; ++j)
                            sts128(mt + (lane * 4 + (j ^ ((lane >> 1) & 3))) * 16, pack_bf16x2(rq[2 * j].x, rq[2 * j].y),
                                   pack_bf16x2(rq[2 * j].z, rq[2 * j].w), pack_bf16x2(rq[2 * j + 1].x, rq[2 * j + 1].y),
                                   pack_bf16x2(rq[2 * j + 1].z, rq[2 * j + 1].w));
                    }
                    fence_proxy_async_smem();
                    __syncwarp();
                    if (lane == 0) {
                        tma_store_2d(&tmR, slot, col0, row0);
                        if (p.out2) tma_store_2d(&tmO, mt, col0, row0);
                        tma_store_commit();
                    }
                    ++rt_g;
                }
                if (want_stats && row0 + lane < p.M)
                    *reinterpret_cast<float2*>(p.stats_out + 2 * ((size_t)(row0 + lane) * (2 * n_tiles) + (t % n_tiles) * 2 + half)) =
                        make_float2(((st1[0] + st1[4]) + (st1[2] + st1[6])) + ((st1[1] + st1[5]) + (st1[3] + st1[7])),
                                    ((st2[0] + st2[4]) + (st2[2] + st2[6])) + ((st2[1] + st2[5]) + (st2[3] + st2[7])));
            } else if constexpr (RT == 1) {
                // acc + bias + residual in the accumulator's own layout (lane = row): the residual row comes out of the
                // TMA-filled SWIZZLE_64B tile with four conflict-free 16-byte reads, the row statistics need no shuffles,
                // the bf16 mirror leaves through one bulk tensor store per slab.  No transposed read-back, no per-row
                // address arithmetic, no prefetch registers.
                float st1[8], st2[8];                         // (same association as RowStats, see the FFN2 form above)
#pragma unroll
                for (int j = 0; j < 8; ++j) { st1[j] = 0.f; st2[j] = 0.f; }
                uint32_t r[32];
#pragma unroll
                for (int i = 0; i < kSlabs; ++i) {
                    const int c = half + 2 * i;
                    const int col0 = n0 + c * 32;
                    const uint32_t k = rt_g % 3;
                    if (lane == 0) rt_issue(rt_g + 2);        // slot (rt_g + 2) % 3 was read out one slab ago
                    tmem_ld_32x32(t_row + c * 32, r);
                    float4 bb[8];
#pragma unroll
                    for (int j = 0; j < 8; ++j) bb[j] = lds_f4(colvec + (c * 32 + 4 * j) * 4);
                    mbar_wait(rbar[k], (rt_g / 3) & 1);
                    uint4 rq[4];
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        rq[j] = lds128(stage_out + k * 2048 + (lane * 4 + (j ^ ((lane >> 1) & 3))) * 16);
                    tmem_ld_wait();
                    float v[32];
#pragma unroll
                    for (int j = 0; j < 4; ++j) {
                        const uint32_t w[4] = {rq[j].x, rq[j].y, rq[j].z, rq[j].w};
#pragma unroll
                        for (int e = 0; e < 4; ++e) {
                            const int q = j * 8 + e * 2;
                            const float4 b = bb[q >> 2];
                            const float b0 = (q & 2) ? b.z : b.x, b1 = (q & 2) ? b.w : b.y;
                            v[q] = (__uint_as_float(r[q]) + b0) + __uint_as_float(w[e] << 16);
                            v[q + 1] = (__uint_as_float(r[q + 1]) + b1) + __uint_as_float(w[e] & 0xffff0000u);
                        }
                    }
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        st1[j >> 2] += (v[j] + v[j + 1]) + (v[j + 2] + v[j + 3]);
                        st2[j >> 2] += fmaf(v[j], v[j], v[j + 1] * v[j + 1]) + fmaf(v[j + 2], v[j + 2], v[j + 3] * v[j + 3]);
                    }
                    // mirror slab -> the warp's out tile (SWIZZLE_64B as it lies) -> one bulk store
                    const uint32_t ot = stage_out + 6144;
                    if (lane == 0) tma_store_wait_read<0>();  // the previous slab's store has read the tile
                    __syncwarp();
#pragma unroll
                    for (int j = 0; j < 4; ++j)
                        sts128(ot + (lane * 4 + (j ^ ((lane >> 1) & 3))) * 16, pack_bf16x2(v[j * 8 + 0], v[j * 8 + 1]),
                               pack_bf16x2(v[j * 8 + 2], v[j * 8 + 3]), pack_bf16x2(v[j * 8 + 4], v[j * 8 + 5]),
                               pack_bf16x2(v[j * 8 + 6], v[j * 8 + 7]));
                    fence_proxy_async_smem();
                    __syncwarp();
                    if (lane == 0) { tma_store_2d(&tmO, ot, col0, row0); tma_store_commit(); }
                    ++rt_g;
                }
                if (want_stats && row0 + lane < p.M)
                    *reinterpret_cast<float2*>(p.stats_out + 2 * ((size_t)(row0 + lane) * (2 * n_tiles) + (t % n_tiles) * 2 + half)) =
                        make_float2(((st1[0] + st1[4]) + (st1[2] + st1[6])) + ((st1[1] + st1[5]) + (st1[3] + st1[7])),
                                    ((st2[0] + st2[4]) + (st2[2] + st2[6])) + ((st2[1] + st2[5]) + (st2[3] + st2[7])));
            } else if constexpr (EPI == VF_EPI_BIAS_RESID_F32) {
                // The fp32 residual is the long-latency input of this epilogue (one DRAM round trip per slab) and it
                // does not depend on the MMA: the slab stream of this warp (4 per tile, tile after tile) keeps the
                // residual of the NEXT THREE slabs in flight in registers — across the tile boundary too — while the
                // current slab is converted and stored.  rr4[i] belongs to slab i of a tile; slabs 0-2 of the first
                // tile were primed before the loop.
                uint32_t r[32];
#pragma unroll
                for (int i = 0; i < kSlabs; ++i) {
                    const int c = half + 2 * i;
                    const int col0 = n0 + c * 32;
                    {   // prefetch distance 3 (the buffer slab i-1 just left): slab i+3 of this tile, or slab i-1 of
                        // this warp's next tile.  (Distance 2 left the residual add on the long scoreboard for ~12 % of
                        // the kernel's samples.)
                        const int tn = i + 3 < kSlabs ? t : (it + 1 < t_count ? t + t_step : num_tiles);
                        const int cn = half + 2 * ((i + 3) & 3);
                        const int m0n = (tn / n_tiles) * BM * CTAS + rank * BM, n0n = (tn % n_tiles) * BN;
                        if (tn < num_tiles) load_resid_slab(p, m0n + quad * 32, n0n + cn * 32, lane, rr4[(i + 3) & 3]);
                    }
                    if (col0 < p.N) {                                     // warp-uniform
                        tmem_ld_32x32(t_row + c * 32, r);
                        float4 bb[8];
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            bb[j] = lds_f4(colvec + (c * 32 + 4 * j) * 4);
                        }
                        tmem_ld_wait();
                        float v[32];
#pragma unroll
                        for (int j = 0; j < 32; j += 4) {
                            const float4 b = bb[j >> 2];
                            v[j + 0] = __uint_as_float(r[j + 0]) + b.x; v[j + 1] = __uint_as_float(r[j + 1]) + b.y;
                            v[j + 2] = __uint_as_float(r[j + 2]) + b.z; v[j + 3] = __uint_as_float(r[j + 3]) + b.w;
                        }
                        epilogue_store_slab<EPI>(p, stage_out, row0, col0, n_out, v, lane, rr4[i], rs);
                    }
                }
            } else {
                uint32_t r[2][32];
                float4 none[8];
                const bool any = n0 + half * 32 < p.N;
                if (any) tmem_ld_32x32(t_row + half * 32, r[0]);
#pragma unroll
                for (int i = 0; i < kSlabs; ++i) {
                    const int c = half + 2 * i;
                    const int col0 = n0 + c * 32;
                    if (col0 >= p.N) break;                               // warp-uniform
                    float4 bb[8];                                         // bias (+ LayerNorm term) of the slab: one batch of
#pragma unroll                                                            // broadcast loads issued before the TMEM wait
                    for (int j = 0; j < 8; ++j) {
                        bb[j] = lds_f4(colvec + (c * 32 + 4 * j) * 4);
                    }
                    if constexpr (epi_is_bf16<EPI>()) {
                        if (ln) {
#pragma unroll
                            for (int j = 0; j < 8; ++j) {
                                {
                                    const float4 sc = lds_f4(colvec + (BN + c * 32 + 4 * j) * 4);
                                    bb[j].x = fmaf(ln_c, sc.x, bb[j].x); bb[j].y = fmaf(ln_c, sc.y, bb[j].y);
                                    bb[j].z = fmaf(ln_c, sc.z, bb[j].z); bb[j].w = fmaf(ln_c, sc.w, bb[j].w);
                                }
                            }
                        }
                    }
                    tmem_ld_wait();
                    if (i + 1 < kSlabs && col0 + 64 < p.N) tmem_ld_32x32(t_row + (c + 2) * 32, r[(i + 1) & 1]);
                    float v[32];
#pragma unroll
                    for (int j = 0; j < 32; j += 4) {
                        const float4 b = bb[j >> 2];
                        v[j + 0] = fmaf(__uint_as_float(r[i & 1][j + 0]), ln_a, b.x);
                        v[j + 1] = fmaf(__uint_as_float(r[i & 1][j + 1]), ln_a, b.y);
                        v[j + 2] = fmaf(__uint_as_float(r[i & 1][j + 2]), ln_a, b.z);
                        v[j + 3] = fmaf(__uint_as_float(r[i & 1][j + 3]), ln_a, b.w);
                    }
                    if constexpr (EPI == VF_EPI_BIAS_GELU_BF16) {
#pragma unroll
                        for (int j = 0; j < 32; ++j) v[j] = gelu_erf(v[j]);
                    }
                    epilogue_store_slab<EPI>(p, stage_out, row0, col0, n_out, v, lane, none, rs, &tmO, i & 1);
                }
            }
            // all TMEM reads of this accumulator are complete (wait::ld above) -> hand it back to the MMA warp
            tmem_ld_wait();
            tc_fence_before();
            __syncwarp();
            if (lane == 0) {
                if constexpr (CTAS == 2) mbar_arrive_leader(&tmem_empty[acc]);
                else mbar_arrive(&tmem_empty[acc]);
            }
            if constexpr (!epi_is_bf16<EPI>()) {
                if (RT == 0 && want_stats) rs.flush(p.stats_out, row0, p.M, (t % n_tiles) * 2 + half, 2 * n_tiles, lane);
            }
        }
    }

    if constexpr (epi_is_bf16<EPI>() || RT != 0) tma_store_wait_read<0>();   // (no-op for threads that issued no bulk store)
    tc_fence_before();
    __syncthreads();
    if constexpr (CTAS == 2) cluster_sync_all();             // the leader's MMAs read the peer's shared memory until the end
    if (warp == 1) {
        tc_fence_after();
        if constexpr (CTAS == 2) tmem_dealloc_pair(tmem_base, kTmemCols);
        else tmem_dealloc(tmem_base, kTmemCols);
    }
}

// ---------------------------------------------------------------------------------
// Debug cross-check path (VF_GEMM_DEBUG_SIMT=1): plain CUDA-core tiled GEMM into an
// fp32 scratch + elementwise epilogue.  Exists only to bisect tcgen05/TMA descriptor
// bugs on the GPU box; never selected by default and never a fallback.
// ---------------------------------------------------------------------------------
__global__ void gemm_simt_raw_kernel(const __nv_bfloat16* __restrict__ A, int lda, const __nv_bfloat16* __restrict__ W,
                                     int ldw, float* __restrict__ C, int M, int N, int K) {
    __shared__ float sa[32][33], sw[32][33];
    const int tx = threadIdx.x, ty = threadIdx.y;
    const int row = blockIdx.y * 32 + ty, col = blockIdx.x * 32 + tx;
    float acc = 0.f;
    for (int k0 = 0; k0 < K; k0 += 32) {
        const int ka = k0 + tx;
        sa[ty][tx] = (row < M && ka < K) ? __bfloat162float(A[(size_t)row * lda + ka]) : 0.f;
        const int wr = blockIdx.x * 32 + ty;
        sw[ty][tx] = (wr < N && ka < K) ? __bfloat162float(W[(size_t)wr * ldw + ka]) : 0.f;
        __syncthreads();
#pragma unroll
        for (int k = 0; k < 32; ++k) acc += sa[ty][k] * sw[tx][k];
        __syncthreads();
    }
    if (row < M && col < N) C[(size_t)row * N + col] = acc;
}

template <int EPI>
__global__ void gemm_simt_epilogue_kernel(const float* __restrict__ C, const GemmParams p) {
    const int n_out = (EPI == VF_EPI_BIAS_GEGLU_BF16) ? p.N / 2 : p.N;
    const size_t total = (size_t)p.M * n_out;
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int row = (int)(i / n_out), col = (int)(i % n_out);
        float v, ln_a = 1.f, ln_c = 0.f;
        if (p.ln_stats) {
            float s1 = 0.f, s2 = 0.f;
            for (int i = 0; i < p.ln_parts; ++i) {
                s1 += p.ln_stats[2 * ((size_t)row * p.ln_parts + i)]; s2 += p.ln_stats[2 * ((size_t)row * p.ln_parts + i) + 1];
            }
            const float mean = s1 * p.ln_inv_d;
            const float var = fmaxf(s2 * p.ln_inv_d - mean * mean, 0.f);
            ln_a = rsqrtf(var + p.ln_eps); ln_c = -ln_a * mean;
        }
        if constexpr (EPI == VF_EPI_BIAS_GEGLU_BF16) {
            const int cu = (col / 128) * 256 + (col % 128), cg = cu + 128;   // tile-interleaved columns
            float u = C[(size_t)row * p.N + cu], g = C[(size_t)row * p.N + cg];
            if (p.ln_stats) { u = ln_a * u + ln_c * p.ln_colsum[cu]; g = ln_a * g + ln_c * p.ln_colsum[cg]; }
            if (p.bias) { u += p.bias[cu]; g += p.bias[cg]; }
            v = u * gelu_erf(g);
        } else {
            v = C[(size_t)row * p.N + col];
            if (p.ln_stats && EPI != VF_EPI_BIAS_RESID_F32 && EPI != VF_EPI_BIAS_F32) v = ln_a * v + ln_c * p.ln_colsum[col];
            if (p.bias) v += p.bias[col];
            if (EPI == VF_EPI_BIAS_RESID_F32 && p.resid) v += p.resid[(size_t)row * p.ldr + col];
            if (EPI == VF_EPI_BIAS_RESID_F32 && p.resid16) v += __bfloat162float(p.resid16[(size_t)row * p.ldr + col]);
            if (EPI == VF_EPI_BIAS_GELU_BF16) v = gelu_erf(v);
        }
        if constexpr (EPI == VF_EPI_BIAS_BF16 || EPI == VF_EPI_BIAS_GEGLU_BF16 || EPI == VF_EPI_BIAS_GELU_BF16) {
            reinterpret_cast<__nv_bfloat16*>(p.out)[(size_t)row * p.ldo + col] = __float2bfloat16_rn(v);
        } else {
            if (p.out) reinterpret_cast<float*>(p.out)[(size_t)row * p.ldo + col] = v;
            if (p.out2) p.out2[(size_t)row * p.ldo2 + col] = __float2bfloat16_rn(v);
            if (p.stats_out) {      // debug path: everything lands in part 0 (the buffer was zeroed by the launcher)
                const int parts = 2 * ((p.N + BN - 1) / BN);
                atomicAdd(p.stats_out + 2 * (size_t)row * parts, v); atomicAdd(p.stats_out + 2 * (size_t)row * parts + 1, v * v);
            }
        }
    }
}

// ---------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static PFN_encodeTiled get_encode_fn() {
    static PFN_encodeTiled fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<PFN_encodeTiled>(p);
    }
    return fn;
}

// K-major bf16 matrix [rows, cols] with row stride ld (elements) -> TMA map with box {64, box_rows}, 128B swizzle.
static int make_tmap_kmajor(CUtensorMap* tm, const void* base, int rows, int cols, int ld, int box_rows) {
    PFN_encodeTiled enc = get_encode_fn();
    VF_REQUIRE(enc, "cuTensorMapEncodeTiled entry point not available (driver too old?)");
    VF_REQUIRE((reinterpret_cast<uintptr_t>(base) & 15) == 0 && (ld % 8) == 0,
               "GEMM operand must be 16-byte aligned with a row stride that is a multiple of 8 elements");
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
    cuuint32_t box[2] = {(cuuint32_t)BK, (cuuint32_t)box_rows};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, const_cast<void*>(base), dims, strides, box, estr,
                     CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                     CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    VF_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled failed with CUresult %d (rows=%d cols=%d ld=%d)", (int)r,
               rows, cols, ld);
    return 0;
}

// bf16 output [rows, cols] with row stride ld -> map with box {32 columns, 32 rows}, 64-byte swizzle: the layout of an
// epilogue warp's staging slab.
// fp32 [rows, cols] tile map, box 32 x 32 (128-byte rows), SWIZZLE_128B: the in-place slabs of the RT == 2 epilogue
static int make_tmap_slab_f32(CUtensorMap* tm, void* base, int rows, int cols, int ld) {
    PFN_encodeTiled enc = get_encode_fn();
    VF_REQUIRE(enc, "cuTensorMapEncodeTiled entry point not available (driver too old?)");
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * 4};
    cuuint32_t box[2] = {32, 32};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 2, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    VF_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled (fp32 slab) failed with CUresult %d (rows=%d cols=%d ld=%d)", (int)r,
               rows, cols, ld);
    return 0;
}

static int make_tmap_out_bf16(CUtensorMap* tm, void* base, int rows, int cols, int ld) {
    PFN_encodeTiled enc = get_encode_fn();
    VF_REQUIRE(enc, "cuTensorMapEncodeTiled entry point not available (driver too old?)");
    cuuint64_t dims[2] = {(cuuint64_t)cols, (cuuint64_t)rows};
    cuuint64_t strides[1] = {(cuuint64_t)ld * 2};
    cuuint32_t box[2] = {32, 32};
    cuuint32_t estr[2] = {1, 1};
    CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, base, dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    VF_REQUIRE(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled (output) failed with CUresult %d (rows=%d cols=%d ld=%d)", (int)r,
               rows, cols, ld);
    return 0;
}

static int g_num_sms = 0;
static bool g_debug_simt = false;
// CTA-pair kernel for M >= kPairMinRows and K >= kPairMinK: measured 6-12 % faster than the single-CTA kernel at
// K = 1024 / 1536 (Wqkv 101k x 4608 x 1536: 1.03 -> 0.90 ms = 1590 TFLOP/s, cuBLAS 0.91).  Round 1 kept K = 512 on the
// single-CTA kernel (its epilogue was the limit then); with the leaner epilogues of round 2 (shared-memory column
// vectors, packed GeGLU, TMA stores) the operand traffic is the limit there too: 48 KB of operands per 512-cycle k-step
// and SM against 32 KB for a pair — LN-folded Wqkv 1.11 M x 1536 x 512 1.61 -> 1.49 ms, GeGLU1 x 2048 2.11-2.24 ->
// 1.95 ms (cuBLAS 1.44-1.64 / 2.02-2.31).
constexpr int kPairMinRows = 1024, kPairMinK = 512;
static bool g_inited = false;

template <int EPI>
static int launch_tc(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tr, const CUtensorMap& to,
                     const GemmParams& p, cudaStream_t s) {
    static bool attr_set = false;
    if (!attr_set) {
        VF_CUDA_OK(cudaFuncSetAttribute(gemm_tcgen05_kernel<EPI, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)kGemmSmem));
        attr_set = true;
    }
    const int tiles = ((p.M + BM - 1) / BM) * ((p.N + BN - 1) / BN);
    const int grid = tiles < g_num_sms ? tiles : g_num_sms;
    gemm_tcgen05_kernel<EPI, 1><<<grid, kGemmThreads, kGemmSmem, s>>>(ta, tb, tr, to, p);
    VF_LAUNCH_OK("gemm_tcgen05_kernel launch");
    return 0;
}

// CTA-pair variant: grid = 2 x (number of pairs that can be co-scheduled, asked from the driver once)
static int g_max_pairs = 0;
template <int EPI, int RT = 0>
static int launch_tc_pair(const CUtensorMap& ta, const CUtensorMap& tb, const CUtensorMap& tr, const CUtensorMap& to,
                          const GemmParams& p, cudaStream_t s) {
    constexpr size_t kSmem = RT ? kGemmSmemRT : kGemmSmem;
    static bool attr_set = false;
    if (!attr_set) {
        VF_CUDA_OK(cudaFuncSetAttribute(gemm_tcgen05_kernel<EPI, 2, RT>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                        (int)kSmem));
        attr_set = true;
    }
    if (g_max_pairs == 0) {
        cudaLaunchConfig_t cfg = {};
        cfg.gridDim = dim3(g_num_sms & ~1); cfg.blockDim = dim3(kGemmThreads); cfg.dynamicSmemBytes = kSmem;
        cudaLaunchAttribute at; at.id = cudaLaunchAttributeClusterDimension; at.val.clusterDim.x = 2;
        at.val.clusterDim.y = 1; at.val.clusterDim.z = 1;
        cfg.attrs = &at; cfg.numAttrs = 1;
        int n = 0;
        cudaError_t e = cudaOccupancyMaxActiveClusters(&n, gemm_tcgen05_kernel<EPI, 2, RT>, &cfg);
        g_max_pairs = (e == cudaSuccess && n > 0) ? n : g_num_sms / 2;
        if (g_max_pairs > g_num_sms / 2) g_max_pairs = g_num_sms / 2;
        (void)cudaGetLastError();
    }
    const int tiles = ((p.M + 2 * BM - 1) / (2 * BM)) * ((p.N + BN - 1) / BN);
    const int pairs = tiles < g_max_pairs ? tiles : g_max_pairs;
    gemm_tcgen05_kernel<EPI, 2, RT><<<2 * pairs, kGemmThreads, kSmem, s>>>(ta, tb, tr, to, p);
    VF_LAUNCH_OK("gemm_tcgen05_kernel (CTA pair) launch");
    return 0;
}

template <int EPI>
static int launch_simt(const __nv_bfloat16* A, int lda, const __nv_bfloat16* W, int ldw, const GemmParams& p,
                       cudaStream_t s) {
    float* scratch = nullptr;
    VF_CUDA_OK(cudaMallocAsync(&scratch, (size_t)p.M * p.N * sizeof(float), s));
    dim3 grid((p.N + 31) / 32, (p.M + 31) / 32), block(32, 32);
    gemm_simt_raw_kernel<<<grid, block, 0, s>>>(A, lda, W, ldw, scratch, p.M, p.N, p.K);
    VF_LAUNCH_OK("gemm_simt_raw_kernel launch");
    gemm_simt_epilogue_kernel<EPI><<<1184, 256, 0, s>>>(scratch, p);
    VF_LAUNCH_OK("gemm_simt_epilogue_kernel launch");
    VF_CUDA_OK(cudaFreeAsync(scratch, s));
    return 0;
}

int gemm_bf16(const void* A, int lda, const void* W, int ldw, int M, int N, int K, int epi, const float* bias,
              const void* resid, int resid_bf16, int ldr, void* out, int ldo, void* out2, int ldo2, const float* ln_stats,
              int ln_parts, const float* ln_colsum, int ln_dim, float ln_eps, float* stats_out, cudaStream_t stream) {
    if (!g_inited) {
        int dev = 0;
        VF_CUDA_OK(cudaGetDevice(&dev));
        VF_CUDA_OK(cudaDeviceGetAttribute(&g_num_sms, cudaDevAttrMultiProcessorCount, dev));
        const char* e = getenv("VF_GEMM_DEBUG_SIMT");
        g_debug_simt = e && e[0] == '1';
        g_inited = true;
    }
    VF_REQUIRE(M >= 0 && N > 0 && K > 0, "gemm: bad shape M=%d N=%d K=%d", M, N, K);
    // Every operand the epilogue writes or reads with vector accesses (uint4 / float4 rows of out, uint2 of the mirror
    // and of a bf16 residual, float2 statistics, float4 batches of the LayerNorm partials) must be aligned for them: a
    // misaligned view is an error here, not a misaligned-address fault in the kernel.  Checked before the M == 0 return
    // so that a caller's bad view is reported whatever its row count.
    const auto misaligned = [](const void* q, uintptr_t bytes) { return (reinterpret_cast<uintptr_t>(q) & (bytes - 1)) != 0; };
    VF_REQUIRE(!misaligned(out, 16), "gemm: output must be 16-byte aligned");
    VF_REQUIRE(!misaligned(out2, 16) && (!out2 || ldo2 % 8 == 0),
               "gemm: bf16 mirror must be 16-byte aligned with a row stride that is a multiple of 8 elements (ldo2=%d)", ldo2);
    VF_REQUIRE(!misaligned(resid, 16) && (!resid || ldr % (resid_bf16 ? 8 : 4) == 0),
               "gemm: residual must be 16-byte aligned with a row stride that is a multiple of 16 bytes (ldr=%d)", ldr);
    VF_REQUIRE(!misaligned(stats_out, 8), "gemm: stats_out must be 8-byte aligned");
    // (the epilogue reads a row's partials as float4 batches when 2 <= ln_parts <= 16 and ln_parts is even)
    VF_REQUIRE(!misaligned(ln_stats, ln_parts > 1 && ln_parts <= 16 && ln_parts % 2 == 0 ? 16 : 8),
               "gemm: ln_stats must be 8-byte aligned (16-byte for an even partial count of 2 to 16: such rows are read as "
               "float4)");
    if (M == 0) return 0;
    VF_REQUIRE(N % 8 == 0 && K % 8 == 0, "gemm: N and K must be multiples of 8 (N=%d K=%d)", N, K);
    VF_REQUIRE(epi >= 0 && epi < VF_EPI_COUNT, "gemm: unknown epilogue %d", epi);
    if (epi == VF_EPI_BIAS_GEGLU_BF16) VF_REQUIRE(N % 256 == 0, "gemm: GeGLU epilogue needs N %% 256 == 0 (N=%d)", N);
    const int n_out = epi == VF_EPI_BIAS_GEGLU_BF16 ? N / 2 : N;
    const bool out_f32 = epi == VF_EPI_BIAS_RESID_F32 || epi == VF_EPI_BIAS_F32;
    VF_REQUIRE(out || (out_f32 && out2), "gemm: no output buffer (only the fp32 epilogues may write their bf16 mirror alone)");
    VF_REQUIRE(!out || (ldo >= n_out && (ldo % 8) == 0), "gemm: bad output stride %d", ldo);
    VF_REQUIRE(!resid_bf16 || epi == VF_EPI_BIAS_RESID_F32, "gemm: a bf16 residual needs the residual epilogue");
    GemmParams p{};
    p.M = M; p.N = N; p.K = K; p.bias = bias; p.ldr = ldr; p.out = out; p.ldo = ldo;
    p.resid = resid_bf16 ? nullptr : reinterpret_cast<const float*>(resid);
    p.resid16 = resid_bf16 ? reinterpret_cast<const __nv_bfloat16*>(resid) : nullptr;
    p.out2 = reinterpret_cast<__nv_bfloat16*>(out2); p.ldo2 = ldo2;
    const bool out_bf16 = epi == VF_EPI_BIAS_BF16 || epi == VF_EPI_BIAS_GEGLU_BF16 || epi == VF_EPI_BIAS_GELU_BF16;
    VF_REQUIRE(!ln_stats || (out_bf16 && ln_colsum && ln_dim > 0 && ln_parts > 0),
               "gemm: the LayerNorm fold needs a bf16 epilogue, column sums, the normalised width and the partial count");
    VF_REQUIRE(!stats_out || !out_bf16, "gemm: row statistics are produced by the fp32 epilogues only");
    p.ln_stats = ln_stats; p.ln_parts = ln_parts; p.ln_colsum = ln_colsum;
    p.ln_inv_d = ln_dim > 0 ? 1.0f / (float)ln_dim : 0.f; p.ln_eps = ln_eps; p.stats_out = stats_out;
    // Tile schedule: chunked for LayerNorm-folded epilogues with K <= 512, whose epilogue is the critical path (+5-10 %
    // there); round-robin otherwise: concurrently running CTAs then share A tiles in L2, worth 15 % at K = 1536.
    p.tile_chunked = ln_stats != nullptr && K <= 512;
    if (g_debug_simt) {
        if (stats_out)
            VF_CUDA_OK(cudaMemsetAsync(stats_out, 0, (size_t)M * 2 * ((N + BN - 1) / BN) * 2 * sizeof(float), stream));
        const __nv_bfloat16* a = reinterpret_cast<const __nv_bfloat16*>(A);
        const __nv_bfloat16* w = reinterpret_cast<const __nv_bfloat16*>(W);
        switch (epi) {
            case VF_EPI_BIAS_BF16: return launch_simt<VF_EPI_BIAS_BF16>(a, lda, w, ldw, p, stream);
            case VF_EPI_BIAS_GEGLU_BF16: return launch_simt<VF_EPI_BIAS_GEGLU_BF16>(a, lda, w, ldw, p, stream);
            case VF_EPI_BIAS_RESID_F32: return launch_simt<VF_EPI_BIAS_RESID_F32>(a, lda, w, ldw, p, stream);
            case VF_EPI_BIAS_GELU_BF16: return launch_simt<VF_EPI_BIAS_GELU_BF16>(a, lda, w, ldw, p, stream);
            default: return launch_simt<VF_EPI_BIAS_F32>(a, lda, w, ldw, p, stream);
        }
    }
    const bool pair = M >= kPairMinRows && K >= kPairMinK;
    CUtensorMap ta, tb;
    if (make_tmap_kmajor(&ta, A, M, K, lda, BM)) return -1;
    if (make_tmap_kmajor(&tb, W, N, K, ldw, pair ? BN / 2 : BN)) return -1;
    CUtensorMap tr = ta, to = ta;                                      // (placeholders where a kernel reads neither)
    // bf16 epilogues store through TMA: out (always given for them) and ldo were checked above for the alignment the
    // tensor map needs
    if (out_bf16 && make_tmap_out_bf16(&to, out, M, n_out, ldo)) return -1;
    if (pair && epi == VF_EPI_BIAS_RESID_F32 && resid_bf16 && !out && out2 && N % BN == 0) {
        // out_proj shape: bf16 residual in, bf16 mirror + row statistics out -> TMA-staged epilogue (see kGemmSmemRT)
        if (make_tmap_out_bf16(&tr, const_cast<void*>(resid), M, N, ldr)) return -1;
        if (make_tmap_out_bf16(&to, out2, M, N, ldo2)) return -1;
        return launch_tc_pair<VF_EPI_BIAS_RESID_F32, 1>(ta, tb, tr, to, p, stream);
    }
    if (pair && epi == VF_EPI_BIAS_RESID_F32 && resid && !resid_bf16 && out == resid && ldo == ldr && N % BN == 0) {
        // FFN2 form, in place on the fp32 stream (+ mirror, statistics)
        if (make_tmap_slab_f32(&tr, out, M, N, ldo)) return -1;
        if (out2 && make_tmap_out_bf16(&to, out2, M, N, ldo2)) return -1;
        return launch_tc_pair<VF_EPI_BIAS_RESID_F32, 2>(ta, tb, tr, to, p, stream);
    }
    if (pair) {
        switch (epi) {
            case VF_EPI_BIAS_BF16: return launch_tc_pair<VF_EPI_BIAS_BF16>(ta, tb, tr, to, p, stream);
            case VF_EPI_BIAS_GEGLU_BF16: return launch_tc_pair<VF_EPI_BIAS_GEGLU_BF16>(ta, tb, tr, to, p, stream);
            case VF_EPI_BIAS_RESID_F32: return launch_tc_pair<VF_EPI_BIAS_RESID_F32>(ta, tb, tr, to, p, stream);
            case VF_EPI_BIAS_GELU_BF16: return launch_tc_pair<VF_EPI_BIAS_GELU_BF16>(ta, tb, tr, to, p, stream);
            default: return launch_tc_pair<VF_EPI_BIAS_F32>(ta, tb, tr, to, p, stream);
        }
    }
    switch (epi) {
        case VF_EPI_BIAS_BF16: return launch_tc<VF_EPI_BIAS_BF16>(ta, tb, tr, to, p, stream);
        case VF_EPI_BIAS_GEGLU_BF16: return launch_tc<VF_EPI_BIAS_GEGLU_BF16>(ta, tb, tr, to, p, stream);
        case VF_EPI_BIAS_RESID_F32: return launch_tc<VF_EPI_BIAS_RESID_F32>(ta, tb, tr, to, p, stream);
        case VF_EPI_BIAS_GELU_BF16: return launch_tc<VF_EPI_BIAS_GELU_BF16>(ta, tb, tr, to, p, stream);
        default: return launch_tc<VF_EPI_BIAS_F32>(ta, tb, tr, to, p, stream);
    }
}

}  // namespace vf
