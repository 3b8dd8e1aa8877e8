// vf_common.cuh — shared device helpers for the sm_100a kernels (PTX wrappers,
// error plumbing).  No torch types anywhere in csrc/: the library is a plain
// C-ABI .so (include/vf_b200.h).
#pragma once
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#ifndef VF_WATCHDOG_NS
// mbarrier waits trap instead of hanging the GPU box when a pipeline bug deadlocks a kernel (a hang is a strike on
// the shared pool): a wait that lasts longer than this many nanoseconds of %globaltimer is reported and killed.
#define VF_WATCHDOG_NS 4000000000ull
#endif

namespace vf {

// ---- error plumbing (thread-local last error string) -----------------------
void set_error(const char* fmt, ...);
int  cuda_fail(cudaError_t e, const char* what);
#define VF_CUDA_OK(call)                                                 \
    do {                                                                 \
        cudaError_t e__ = (call);                                        \
        if (e__ != cudaSuccess) return ::vf::cuda_fail(e__, #call);      \
    } while (0)
// every kernel launch of the library passes through here: g_launches is what vf_launch_count() reports
extern unsigned long long g_launches;
#define VF_LAUNCH_OK(what)                                               \
    do {                                                                 \
        cudaError_t e__ = cudaGetLastError();                            \
        if (e__ != cudaSuccess) return ::vf::cuda_fail(e__, what);       \
        __atomic_add_fetch(&::vf::g_launches, 1ull, __ATOMIC_RELAXED);   \
    } while (0)
#define VF_REQUIRE(cond, ...)                                            \
    do {                                                                 \
        if (!(cond)) { ::vf::set_error(__VA_ARGS__); return -1; }        \
    } while (0)

// ---- small device utilities ------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) {
    return static_cast<uint32_t>(__cvta_generic_to_shared(p));
}
__device__ __forceinline__ uint32_t lane_id() { return threadIdx.x & 31; }

__device__ __forceinline__ bool elect_one() {
    uint32_t pred = 0;
    asm volatile(
        "{\n\t.reg .pred P1;\n\t"
        "elect.sync _|P1, 0xffffffff;\n\t"
        "selp.b32 %0, 1, 0, P1;\n\t}\n"
        : "=r"(pred));
    return pred != 0;
}

__device__ __forceinline__ uint32_t pack_bf16x2(float lo, float hi) {
    __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
    return *reinterpret_cast<uint32_t*>(&v);
}

__device__ __forceinline__ float gelu_erf(float x) {   // nn.GELU() default (exact erf form)
    return 0.5f * x * (1.0f + erff(x * 0.70710678118654752440f));
}
// Same function for the GEMM epilogues that are instruction bound (GeGLU at K = 512: erff costs ~35 instructions per
// output).  erf(x / sqrt 2) = sign(x) * min(1, a * P(2 a^2 / X^2 - 1)), a = min(|x|, X), X = 4.8, P = degree-10
// minimax fit (tools: see DESIGN.md): |error| of erf <= 3.9e-6, of gelu <= 9.3e-6 absolute over all of R — two
// orders of magnitude below the bf16 rounding of the result.  ~17 instructions.
__device__ __forceinline__ float gelu_erf_fast(float x) {
    const float a = fminf(fabsf(x), 4.8f);
    const float t = fmaf(a * a, 2.0f / (4.8f * 4.8f), -1.0f);
    float p = 3.602446076e-03f;
    p = fmaf(p, t, -8.992323659e-03f); p = fmaf(p, t, 9.407739340e-03f); p = fmaf(p, t, -1.378258884e-02f);
    p = fmaf(p, t, 2.861803474e-02f);  p = fmaf(p, t, -4.503236200e-02f); p = fmaf(p, t, 6.122043364e-02f);
    p = fmaf(p, t, -8.099147498e-02f); p = fmaf(p, t, 1.058257807e-01f);  p = fmaf(p, t, -1.459672796e-01f);
    p = fmaf(p, t, 2.944253756e-01f);
    const float e = copysignf(fminf(p * a, 1.0f), x);
    const float h = 0.5f * x;
    return fmaf(h, e, h);
}

// ---- packed fp32 pairs (sm_100: FFMA2 / FADD2 / FMUL2, one issue slot for two lanes of arithmetic) ----
__device__ __forceinline__ uint64_t f2_pack(float lo, float hi) {
    uint64_t v;
    asm("mov.b64 %0, {%1, %2};" : "=l"(v) : "f"(lo), "f"(hi));
    return v;
}
__device__ __forceinline__ uint64_t f2_pack(uint32_t lo, uint32_t hi) {
    uint64_t v;
    asm("mov.b64 %0, {%1, %2};" : "=l"(v) : "r"(lo), "r"(hi));
    return v;
}
__device__ __forceinline__ void f2_unpack(uint64_t v, uint32_t& lo, uint32_t& hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=r"(lo), "=r"(hi) : "l"(v));
}
__device__ __forceinline__ void f2_unpack(uint64_t v, float& lo, float& hi) {
    asm("mov.b64 {%0, %1}, %2;" : "=f"(lo), "=f"(hi) : "l"(v));
}
__device__ __forceinline__ uint64_t f2_fma(uint64_t a, uint64_t b, uint64_t c) {
    uint64_t d;
    asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(d) : "l"(a), "l"(b), "l"(c));
    return d;
}
__device__ __forceinline__ uint64_t f2_add(uint64_t a, uint64_t b) {
    uint64_t d;
    asm("add.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ uint64_t f2_mul(uint64_t a, uint64_t b) {
    uint64_t d;
    asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(d) : "l"(a), "l"(b));
    return d;
}
__device__ __forceinline__ uint64_t f2_bcast(float x) { return f2_pack(x, x); }

// gelu_erf_fast on a pair: the polynomial, the squares and the final products run as packed instructions (21
// instructions for two values instead of 2 x 19): the GeGLU epilogue at K = 512 is bound by the instructions it issues.
__device__ __forceinline__ void gelu_erf_fast2(float x0, float x1, float& y0, float& y1) {
    const float a0 = fminf(fabsf(x0), 4.8f), a1 = fminf(fabsf(x1), 4.8f);
    const uint64_t a = f2_pack(a0, a1), x = f2_pack(x0, x1);
    const uint64_t t = f2_fma(f2_mul(a, a), f2_bcast(2.0f / (4.8f * 4.8f)), f2_bcast(-1.0f));
    uint64_t p = f2_bcast(3.602446076e-03f);
    p = f2_fma(p, t, f2_bcast(-8.992323659e-03f)); p = f2_fma(p, t, f2_bcast(9.407739340e-03f));
    p = f2_fma(p, t, f2_bcast(-1.378258884e-02f)); p = f2_fma(p, t, f2_bcast(2.861803474e-02f));
    p = f2_fma(p, t, f2_bcast(-4.503236200e-02f)); p = f2_fma(p, t, f2_bcast(6.122043364e-02f));
    p = f2_fma(p, t, f2_bcast(-8.099147498e-02f)); p = f2_fma(p, t, f2_bcast(1.058257807e-01f));
    p = f2_fma(p, t, f2_bcast(-1.459672796e-01f)); p = f2_fma(p, t, f2_bcast(2.944253756e-01f));
    float e0, e1;
    f2_unpack(f2_mul(p, a), e0, e1);
    e0 = copysignf(fminf(e0, 1.0f), x0);
    e1 = copysignf(fminf(e1, 1.0f), x1);
    const uint64_t h = f2_mul(x, f2_bcast(0.5f));
    f2_unpack(f2_fma(h, f2_pack(e0, e1), h), y0, y1);
}

// ---- explicit shared-memory accesses (32-bit shared-space addresses).  Going through a generic pointer the
// compiler emits LD.E / ST.E with 64-bit address arithmetic, tracked on the long scoreboard like global memory. ----
__device__ __forceinline__ void sts128(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}
__device__ __forceinline__ uint4 lds128(uint32_t addr) {
    uint4 v;
    asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(addr) : "memory");
    return v;
}

__device__ __forceinline__ float4 lds_f4(uint32_t addr) {
    float4 v;
    asm volatile("ld.shared.v4.f32 {%0, %1, %2, %3}, [%4];" : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w) : "r"(addr) : "memory");
    return v;
}

// ---- mbarrier ----------------------------------------------------------------
// A barrier named by its 32-bit shared-space address.  Kernels whose warps hand-shake every few hundred cycles keep
// ONE such base in a register and index it: going through a generic pointer makes the compiler rebuild the shared
// window base (S2UR + ULEA, a short-scoreboard stall) at every use.
struct SmemBar {
    uint32_t addr;
    __device__ __forceinline__ SmemBar operator[](int i) const { return SmemBar{addr + 8u * (uint32_t)i}; }
};
__device__ __forceinline__ SmemBar smem_bar(uint64_t* bar) { return SmemBar{smem_u32(bar)}; }
__device__ __forceinline__ void mbar_init(SmemBar bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar.addr), "r"(count));
}
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) { mbar_init(smem_bar(bar), count); }
__device__ __forceinline__ void fence_barrier_init() {
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
}
__device__ __forceinline__ void fence_proxy_async_smem() {
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void mbar_arrive(SmemBar bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar.addr) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) { mbar_arrive(smem_bar(bar)); }
__device__ __forceinline__ void mbar_arrive_expect_tx(SmemBar bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar.addr), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive_expect_tx(uint64_t* bar, uint32_t bytes) {
    mbar_arrive_expect_tx(smem_bar(bar), bytes);
}
// Non-blocking test of a phase.
__device__ __forceinline__ bool mbar_test_wait(SmemBar bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n\t.reg .pred P1;\n\t"
        "mbarrier.test_wait.parity.shared::cta.b64 P1, [%1], %2;\n\t"
        "selp.b32 %0, 1, 0, P1;\n\t}\n"
        : "=r"(ok)
        : "r"(bar.addr), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ bool mbar_test_wait(uint64_t* bar, uint32_t parity) { return mbar_test_wait(smem_bar(bar), parity); }
__device__ __forceinline__ uint64_t global_timer_ns() {
    uint64_t t;
    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t));
    return t;
}
// Wait for a phase.  Pure spin on the NON-blocking test: `mbarrier.try_wait` lets the hardware suspend the thread, and
// the wake-up after the phase completes costs on the order of a microsecond — measured on the attention kernels, whose
// softmax <-> MMA hand-shakes happen every ~2 us: 31 % (201-token items) to 5 % (1024-key items) slower than spinning.
// Every 2^20 spins the loop looks at %globaltimer: a wait longer than VF_WATCHDOG_NS kills the kernel (`trap`), so a
// pipeline bug cannot hang the GPU.  The loop must not contain a call: a printf here (even on the cold path) gives
// every kernel that waits on a barrier an ABI stack frame and cost the attention kernels the whole 31 % again; build
// with -DVF_WATCHDOG_VERBOSE to get the message (block, thread, barrier, parity) when chasing a deadlock.
__device__ __forceinline__ void mbar_wait(SmemBar bar, uint32_t parity) {
    uint32_t spins = 0;
    uint64_t t0 = 0;
    while (!mbar_test_wait(bar, parity)) {
        if ((++spins & 0xFFFFFu) == 0) {
            const uint64_t now = global_timer_ns();
            if (t0 == 0) t0 = now;
            if (now - t0 > VF_WATCHDOG_NS) {
#ifdef VF_WATCHDOG_VERBOSE
                unsigned long long raw;
                asm volatile("ld.shared.b64 %0, [%1];" : "=l"(raw) : "r"(bar.addr) : "memory");
                printf("vf: mbarrier watchdog: block %d thread %d barrier smem+0x%x parity %u state 0x%016llx\n", blockIdx.x,
                       threadIdx.x, bar.addr, parity, raw);
#pragma unroll 1
                for (int i = 0; i < 1000; ++i) __nanosleep(1000000);
#endif
                __trap();
            }
        }
    }
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) { mbar_wait(smem_bar(bar), parity); }

// ---- TMA (cp.async.bulk.tensor) -----------------------------------------------
__device__ __forceinline__ void tma_prefetch_desc(const void* tmap) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(reinterpret_cast<uint64_t>(tmap)) : "memory");
}
// 2-D tile load: coordinates are (c0 = innermost element index, c1 = row index)
__device__ __forceinline__ void tma_load_2d(uint32_t smem_dst, const void* tmap, SmemBar bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_dst), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(bar.addr), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const void* tmap, uint64_t* bar, int c0, int c1) {
    tma_load_2d(smem_u32(smem_dst), tmap, smem_bar(bar), c0, c1);
}

// TMA store of one box from shared memory (bulk async group): smem -> global, rows / columns past the tensor's extent
// are clipped by the hardware.  The writer must make its generic-proxy shared-memory writes visible to the async proxy
// first (fence_proxy_async_smem) and may overwrite the buffer only after tma_store_wait_read<N>().
__device__ __forceinline__ void tma_store_2d(const void* tmap, uint32_t smem_src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                 ::"l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_src), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }

// ---- warpgroup register reallocation (all 4 warps of a warpgroup must execute the same one) ----
template <uint32_t R>
__device__ __forceinline__ void reg_alloc() { asm volatile("setmaxnreg.inc.sync.aligned.u32 %0;" ::"n"(R)); }
template <uint32_t R>
__device__ __forceinline__ void reg_dealloc() { asm volatile("setmaxnreg.dec.sync.aligned.u32 %0;" ::"n"(R)); }

// ---- tcgen05 / TMEM -------------------------------------------------------------
__device__ __forceinline__ void tmem_alloc(uint32_t* smem_dst, uint32_t ncols) {   // whole warp, .sync.aligned
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)),
                 "r"(ncols)
                 : "memory");
}
__device__ __forceinline__ void tmem_relinquish() {
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {      // whole warp
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

// D[tmem] (+)= A[smem desc] * B[smem desc]; bf16 inputs, fp32 accumulate; issued by ONE thread.
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                          uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// Arrive on an mbarrier once all previously issued tcgen05.mma of this thread retire
// (implies tcgen05.fence::before_thread_sync).
__device__ __forceinline__ void umma_commit(SmemBar bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(bar.addr)
                 : "memory");
}
__device__ __forceinline__ void umma_commit(uint64_t* bar) { umma_commit(smem_bar(bar)); }
// ---- CTA pair (cta_group::2): two CTAs of a cluster cooperate on one 256-row UMMA tile.  The leader (even rank)
// issues the MMA; each CTA loads its own A rows and its half of the B rows; barriers of the leader are addressed from
// the peer by clearing the rank bit of the shared::cluster address (same offset in the even CTA of the pair). ----
constexpr uint32_t kPeerBitMask = 0xFEFFFFFFu;
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ void tma_load_2d_pair(void* smem_dst, const void* tmap, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        ::"r"(smem_u32(smem_dst)), "l"(reinterpret_cast<uint64_t>(tmap)), "r"(smem_u32(bar) & kPeerBitMask), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void mbar_arrive_leader(uint64_t* bar) {      // arrive on the pair leader's copy of `bar`
    // (no .release.cluster: that form puts a MEMBAR + ERRBAR in front of the arrive, i.e. the epilogue warp waits for
    // all of its global stores to be acknowledged before it hands the accumulator back — 5 % of the kernel's samples.
    // What the arrive orders are TMEM reads, and tcgen05.wait::ld + tcgen05.fence::before_thread_sync do that.)
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" ::"r"(smem_u32(bar) & kPeerBitMask) : "memory");
}
__device__ __forceinline__ void tmem_alloc_pair(uint32_t* smem_dst, uint32_t ncols) {
    asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(smem_dst)), "r"(ncols) : "memory");
}
__device__ __forceinline__ void tmem_relinquish_pair() {
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc_pair(uint32_t taddr, uint32_t ncols) {
    asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols) : "memory");
}
__device__ __forceinline__ void umma_bf16_pair(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc,
                                               uint32_t accumulate) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
        ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
        : "memory");
}
// arrive (once all previously issued MMAs retire) on the barrier at this offset in BOTH CTAs of the pair
__device__ __forceinline__ void umma_commit_pair(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 ::"r"(smem_u32(bar)), "h"((uint16_t)3)
                 : "memory");
}

// TMEM -> registers: 32 lanes x 32 consecutive fp32 columns (one row per thread of the warp).
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// registers -> TMEM: the inverse of tmem_ld_32x32 (one row per thread, 32 consecutive fp32 columns)
__device__ __forceinline__ void tmem_st_32x32(uint32_t taddr, const uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x32.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16, "
        "%17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31, %32};"
        ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
          "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15]),
          "r"(r[16]), "r"(r[17]), "r"(r[18]), "r"(r[19]), "r"(r[20]), "r"(r[21]), "r"(r[22]), "r"(r[23]),
          "r"(r[24]), "r"(r[25]), "r"(r[26]), "r"(r[27]), "r"(r[28]), "r"(r[29]), "r"(r[30]), "r"(r[31])
        : "memory");
}
// 16-column variants (head_dim 48: the O accumulator is 32 + 16 columns wide)
__device__ __forceinline__ void tmem_ld_32x16(uint32_t taddr, uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr)
        : "memory");
}
__device__ __forceinline__ void tmem_st_32x16(uint32_t taddr, const uint32_t (&r)[16]) {
    asm volatile(
        "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], "
        "{%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
        ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7]),
          "r"(r[8]), "r"(r[9]), "r"(r[10]), "r"(r[11]), "r"(r[12]), "r"(r[13]), "r"(r[14]), "r"(r[15])
        : "memory");
}
__device__ __forceinline__ void tmem_ld_32x8(uint32_t taddr, uint32_t (&r)[8]) {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr)
                 : "memory");
}
__device__ __forceinline__ void tmem_st_32x8(uint32_t taddr, const uint32_t (&r)[8]) {
    asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
                 ::"r"(taddr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
                 : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// K-major operand tile in shared memory, rows of 64 bf16 (= 128 B), 128-byte swizzle
// (what a TMA box {64, rows} with CU_TENSOR_MAP_SWIZZLE_128B produces): 8-row core groups
// are 1024 B apart (SBO), LBO unused for swizzled K-major, descriptor version 1 (Blackwell).
__device__ __forceinline__ uint64_t umma_desc_kmajor_sw128(uint32_t smem_addr) {
    uint64_t d = 0;
    d |= (uint64_t)((smem_addr & 0x3FFFF) >> 4);          // [0,14)  start address >> 4
    d |= (uint64_t)1 << 16;                                // [16,30) leading byte offset (ignored, canonical 1)
    d |= (uint64_t)(1024 >> 4) << 32;                      // [32,46) stride byte offset = 1024 B
    d |= (uint64_t)1 << 46;                                // [46,48) descriptor version = 1
    d |= (uint64_t)2 << 61;                                // [61,64) SWIZZLE_128B
    return d;
}
// kind::f16 instruction descriptor: D=f32, A=B=bf16, both K-major, shape M x N.
__host__ __device__ constexpr uint32_t umma_idesc_bf16(int m, int n) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(n >> 3) << 17) | ((uint32_t)(m >> 4) << 24);
}

// ---- legacy warp-level MMA (attention, round 1) -----------------------------------
__device__ __forceinline__ void mma_bf16_16816(float (&c)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void ldmatrix_x4(uint32_t (&r)[4], uint32_t addr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
                 : "r"(addr));
}
__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t (&r)[4], uint32_t addr) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
                 : "r"(addr));
}
__device__ __forceinline__ void cp_async_16(uint32_t smem_addr, const void* gptr, bool valid) {
    int sz = valid ? 16 : 0;   // src-size 0 => zero fill
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(smem_addr), "l"(gptr), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" ::"n"(N) : "memory"); }

}  // namespace vf
