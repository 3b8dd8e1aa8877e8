// vf_forward.cu — the coarse entry points of the C ABI: whole-module forwards with the layer loop in C++, a weight-pointer
// table in, caller-owned workspace, no Python between launches (SURVEY 8b: vf_seq2reg_forward / vf_seq2gene_forward /
// *_workspace_bytes), plus the host-side builder of the attention work tables.
//
// Reference call sites replaced:
//   vf_seq2reg_forward   Seq2RegPredictor.forward(only_embed=True)        seq2reg/model.py:193-279, seq2reg/modules.py:149-191
//   vf_seq2gene_forward  cre_map / gene_map, MultiRegistry, CombinedModulator.forward, pool_outputs, TissueExpressionHeads
//                        seq2gene/model_combined_modulator.py:137-328, 540-720; seq2gene/modules/layers.py:88-165, 508-521,
//                        1078-1144
// Schedule and numerics are exactly those of variantformer_b200/engine.py (the fine-grained path through the same
// kernels): tissue-deduplicated CRE stream on a second CUDA stream, tissue copies stacked on the M axis, 9-class label
// attention, LayerNorm folded into the consuming GEMM, row-centred fp32 residual streams, last gene layer on the rows
// that are read.  Results are bit-identical to the fine-grained path (tests/test_gpu_forward_abi.py).
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <vector>

#include "vf_common.cuh"
#include "vf_internal.h"

namespace vf {

// ---- workspace carving --------------------------------------------------------------------------------------------
struct Carver {
    uint8_t* base; size_t off = 0;
    explicit Carver(void* p) : base(reinterpret_cast<uint8_t*>(p)) {}
    template <class T> T* take(size_t n) {
        off = (off + 255) & ~size_t(255);
        T* p = base ? reinterpret_cast<T*>(base + off) : nullptr;
        off += n * sizeof(T);
        return p;
    }
};
static inline int stats_parts(int n) { return 2 * ((n + 255) / 256); }
using bf16 = uint16_t;

// ---- one LayerNorm-folded or plain linear ---------------------------------------------------------------------------
static int linear(const vf_linear_t& L, const void* a, int lda, int M, int N, int K, int epi, const void* resid, int resid16,
                  int ldr, void* out, int ldo, void* out2, int ldo2, const float* ln_stats, int ln_parts, float eps,
                  float* stats_out, cudaStream_t s) {
    return gemm_bf16(a, lda, L.w, K, M, N, K, epi, L.b, resid, resid16, ldr, out, ldo, out2, ldo2, ln_stats,
                     ln_stats ? ln_parts : 0, ln_stats ? L.cs : nullptr, ln_stats ? K : 0, eps, stats_out, s);
}

// ====================================================================================================================
// seq2reg
// ====================================================================================================================
struct Seq2RegWs {
    int32_t *ids, *pos; float *x, *piv, *xs0, *xs, *s1; bf16 *xb, *qkv, *a, *f; size_t bytes;
};
static Seq2RegWs carve_seq2reg(const vf_seq2reg_weights_t& w, int64_t n, void* ws) {
    Carver c(ws); Seq2RegWs r;
    const int d = w.d, P = stats_parts(d);
    r.ids = c.take<int32_t>(n); r.pos = c.take<int32_t>(n);
    r.x = c.take<float>(n * d); r.piv = c.take<float>(n); r.xs0 = c.take<float>(n * 2);
    r.xs = c.take<float>(n * P * 2); r.s1 = c.take<float>(n * P * 2);
    r.xb = c.take<bf16>(n * d); r.qkv = c.take<bf16>(n * 3 * d); r.a = c.take<bf16>(n * d);
    r.f = c.take<bf16>(n * (w.ffn_hidden / 2));
    r.bytes = c.off + 256;
    return r;
}

static int seq2reg_forward(const vf_seq2reg_weights_t& w, const int32_t* tokens, const uint8_t* pad_mask, const int32_t* cu,
                           int n_win, int L, int64_t n_tok, const int32_t* slots, int n_items, void* ws, size_t ws_bytes,
                           void* out_bf16, cudaStream_t s) {
    VF_REQUIRE(w.layers && w.emb && w.n_layers >= 1 && w.d % w.heads == 0, "seq2reg_forward: incomplete weight table");
    if (n_win == 0 || n_tok == 0) return 0;
    Seq2RegWs b = carve_seq2reg(w, n_tok, ws);
    VF_REQUIRE(ws && ws_bytes >= b.bytes, "seq2reg_forward: workspace of %zu bytes < %zu needed", ws_bytes, b.bytes);
    VF_REQUIRE((reinterpret_cast<uintptr_t>(ws) & 255) == 0, "seq2reg_forward: workspace must be 256-byte aligned");
    const int d = w.d, H = w.heads, hd = d / H, P = stats_parts(d), n = (int)n_tok, F = w.ffn_hidden;
    int rc;
    if ((rc = compact_tokens(tokens, pad_mask, cu, n_win, L, b.ids, b.pos, s))) return rc;
    if ((rc = embed_center(b.ids, b.pos, w.emb, w.pe, n, d, b.x, b.piv, b.xs0, b.xb, s))) return rc;
    for (int l = 0; l < w.n_layers; ++l) {
        const vf_seq2reg_layer_t& Lr = w.layers[l];
        if ((rc = linear(Lr.qkv, b.xb, d, n, 3 * d, d, VF_EPI_BIAS_BF16, nullptr, 0, 0, b.qkv, 3 * d, nullptr, 0,
                         l == 0 ? b.xs0 : b.xs, l == 0 ? 1 : P, w.ln_eps, nullptr, s))) return rc;
        if ((rc = attention_mc_varlen(b.qkv, 3 * d, b.qkv + d, 3 * d, b.qkv + 2 * d, 3 * d, b.a, d, n, n, slots, n_items, H, hd,
                                      w.slopes, s))) return rc;
        // x1 = x + MHA(..): bf16 mirror + row statistics only (the layer's residual is its INPUT, modules.py:189); its
        // residual is read from the bf16 mirror of x (see engine.py: Engine.seq2reg)
        if ((rc = linear(Lr.out, b.a, d, n, d, d, VF_EPI_BIAS_RESID_F32, b.xb, 1, d, nullptr, 0, b.xb, d, nullptr, 0, 0.f, b.s1,
                         s))) return rc;
        if ((rc = linear(Lr.g1, b.xb, d, n, F, d, VF_EPI_BIAS_GEGLU_BF16, nullptr, 0, 0, b.f, F / 2, nullptr, 0, b.s1, P,
                         w.ln_eps, nullptr, s))) return rc;
        if ((rc = linear(Lr.g2, b.f, F / 2, n, d, F / 2, VF_EPI_BIAS_RESID_F32, b.x, 0, d, b.x, d, b.xb, d, nullptr, 0, 0.f,
                         b.xs, s))) return rc;
    }
    return masked_meanpool(b.x, d, cu, n_win, d, b.piv, out_bf16, nullptr, d, s);
}

// ====================================================================================================================
// seq2gene
// ====================================================================================================================
struct StreamBufs { bf16 *hb, *qkv, *a, *f; float *s1, *xs; };
static StreamBufs carve_stream(Carver& c, size_t M, int D, int F) {
    StreamBufs r; const int P = stats_parts(D);
    r.hb = c.take<bf16>(M * D); r.qkv = c.take<bf16>(M * 3 * D); r.a = c.take<bf16>(M * D); r.f = c.take<bf16>(M * (F / 2));
    r.s1 = c.take<float>(M * P * 2); r.xs = c.take<float>(M * P * 2);
    return r;
}
struct Seq2GeneWs {
    float *cx, *cpiv, *cxs0, *gene_emb, *gx, *gpiv, *gxs0, *h1, *lastf, *tokf; bf16 *ctx, *cxb, *gxb, *kv, *h1n, *h2, *lastb;
    StreamBufs cs, gs;
    // last layer, needed rows only
    float *xR, *stR, *s1R; bf16 *xbR, *qR, *aR, *hbR, *fR;
    size_t bytes;
};
static Seq2GeneWs carve_seq2gene(const vf_seq2gene_weights_t& w, const vf_seq2gene_slab_t& t, void* ws) {
    Carver c(ws); Seq2GeneWs r;
    const size_t nC = t.n_cre, Mg = t.n_gene_rows, R = t.n_need;
    const int D = w.D, F = w.ffn_hidden, P = stats_parts(D), NL = w.n_layers;
    r.cx = c.take<float>(nC * D); r.cpiv = c.take<float>(nC); r.cxs0 = c.take<float>(nC * 2);
    r.ctx = c.take<bf16>(nC * D); r.cxb = c.take<bf16>(nC * D);
    r.gene_emb = c.take<float>((size_t)t.n_gene_chunks * D);
    r.gx = c.take<float>(Mg * D); r.gpiv = c.take<float>(Mg); r.gxs0 = c.take<float>(Mg * 2); r.gxb = c.take<bf16>(Mg * D);
    r.kv = c.take<bf16>((size_t)NL * nC * 2 * D);               // K/V of every gene layer's cross-attention
    r.cs = carve_stream(c, nC, D, F); r.gs = carve_stream(c, Mg, D, F);
    r.xR = c.take<float>(R * D); r.xbR = c.take<bf16>(R * D); r.stR = c.take<float>(R * P * 2); r.s1R = c.take<float>(R * P * 2);
    r.qR = c.take<bf16>(R * D); r.aR = c.take<bf16>(R * D); r.hbR = c.take<bf16>(R * D); r.fR = c.take<bf16>(R * (F / 2));
    r.lastf = c.take<float>(R * D); r.lastb = c.take<bf16>(R * D); r.tokf = c.take<float>((size_t)std::max(t.n_reg, 1) * D);
    r.h1 = c.take<float>((size_t)t.n_reg * D); r.h1n = c.take<bf16>((size_t)t.n_reg * D); r.h2 = c.take<bf16>((size_t)t.n_reg * D);
    r.bytes = c.off + 256;
    return r;
}

// ContextFlashAttentionEncoderLayer on an unpadded row-centred stream (engine.py: Engine._layer)
template <class SelfAttn, class CrossAttn>
static int context_layer(const vf_context_layer_t& L, const vf_seq2gene_weights_t& w, float* x, bf16* xb, const float* xs,
                         int xs_parts, int M, StreamBufs& b, SelfAttn&& self_attn, CrossAttn&& cross_attn, float** xs_out,
                         cudaStream_t s) {
    const int D = w.D, F = w.ffn_hidden, P = stats_parts(D);
    int rc;
    if ((rc = linear(L.qkv, xb, D, M, 3 * D, D, VF_EPI_BIAS_BF16, nullptr, 0, 0, b.qkv, 3 * D, nullptr, 0, xs, xs_parts,
                     w.ln_eps, nullptr, s))) return rc;
    if ((rc = self_attn(b.qkv, b.a))) return rc;
    if ((rc = linear(L.out, b.a, D, M, D, D, VF_EPI_BIAS_RESID_F32, xb, 1, D, nullptr, 0, b.hb, D, nullptr, 0, 0.f, b.s1, s)))
        return rc;
    if ((rc = linear(L.q, b.hb, D, M, D, D, VF_EPI_BIAS_BF16, nullptr, 0, 0, b.qkv, 3 * D, nullptr, 0, b.s1, P, w.ln_eps,
                     nullptr, s))) return rc;
    if ((rc = cross_attn(b.qkv, b.a))) return rc;
    if ((rc = linear(L.out2, b.a, D, M, D, D, VF_EPI_BIAS_RESID_F32, b.hb, 1, D, nullptr, 0, b.hb, D, nullptr, 0, 0.f, b.s1, s)))
        return rc;
    if ((rc = linear(L.g1, b.hb, D, M, F, D, VF_EPI_BIAS_GEGLU_BF16, nullptr, 0, 0, b.f, F / 2, nullptr, 0, b.s1, P, w.ln_eps,
                     nullptr, s))) return rc;
    if ((rc = linear(L.g2, b.f, F / 2, M, D, F / 2, VF_EPI_BIAS_RESID_F32, x, 0, D, x, D, xb, D, nullptr, 0, 0.f, b.xs, s)))
        return rc;
    *xs_out = b.xs;
    return 0;
}

// the library's own side stream + events for the CRE stack (one set per device, created on first use)
struct SideStream { cudaStream_t s = nullptr; std::vector<cudaEvent_t> ev; cudaEvent_t start = nullptr; };
static SideStream& side_stream(int n_events) {
    static SideStream g[16];
    int dev = 0;
    cudaGetDevice(&dev);
    SideStream& t = g[dev & 15];
    if (!t.s) { cudaStreamCreateWithFlags(&t.s, cudaStreamNonBlocking); cudaEventCreateWithFlags(&t.start, cudaEventDisableTiming); }
    while ((int)t.ev.size() < n_events) {
        cudaEvent_t e; cudaEventCreateWithFlags(&e, cudaEventDisableTiming); t.ev.push_back(e);
    }
    return t;
}

static int seq2gene_forward(const vf_seq2gene_weights_t& w, const vf_seq2gene_slab_t& t, const void* cre_pooled,
                            const void* gene_pooled, void* ws, size_t ws_bytes, float* pred, float* emb,
                            float* gene_token_emb, float* cre_token_emb, const vf_cre_attention_t* attn, cudaStream_t main) {
    VF_REQUIRE(w.cre_layers && w.gene_layers && w.n_layers >= 1 && w.D % w.heads == 0, "seq2gene_forward: incomplete weight table");
    VF_REQUIRE(t.n_need >= t.n_reg && t.n_reg > 0 && t.n_cre > 0 && t.n_gene_rows > 0, "seq2gene_forward: empty slab");
    if (attn) {
        VF_REQUIRE(attn->n_groups >= 0 && attn->group_q && attn->group_k && attn->reg_rows && attn->out && attn->out_off,
                   "seq2gene_forward: incomplete CRE attention table");
        VF_REQUIRE((reinterpret_cast<uintptr_t>(attn->out) & 3) == 0 && (reinterpret_cast<uintptr_t>(attn->out_off) & 7) == 0,
                   "seq2gene_forward: CRE attention out / out_off misaligned");
    }
    Seq2GeneWs b = carve_seq2gene(w, t, ws);
    VF_REQUIRE(ws && ws_bytes >= b.bytes, "seq2gene_forward: workspace of %zu bytes < %zu needed", ws_bytes, b.bytes);
    VF_REQUIRE((reinterpret_cast<uintptr_t>(ws) & 255) == 0, "seq2gene_forward: workspace must be 256-byte aligned");
    const int D = w.D, H = w.heads, hd = D / H, P = stats_parts(D), NL = w.n_layers, F = w.ffn_hidden;
    const int nC = t.n_cre, Mg = t.n_gene_rows, R = t.n_need, n_reg = t.n_reg;
    int rc;
    // the cross-attention maps of gene layer `layer` from the queries the attention kernel just read (q_rows NULL: the
    // pruned last layer's query rows, registry rows first)
    auto maps = [&](const bf16* q, int ldq, const int32_t* q_rows, const bf16* k, int layer) {
        if (!attn) return 0;
        return cross_attention_probs(q, ldq, q_rows, attn->group_q, attn->n_groups, k, 2 * D, attn->group_k, H, hd, attn->out,
                                     attn->out_off, layer, main);
    };
    // ---- stream set-up: cre_map (raw bf16 copy = context of gene layer 0), gene_map + registry gather, row centring ----
    if ((rc = linear(w.cre_map, cre_pooled, w.token_dim, nC, D, w.token_dim, VF_EPI_BIAS_F32, nullptr, 0, 0, b.cx, D, b.ctx, D,
                     nullptr, 0, 0.f, nullptr, main))) return rc;
    if ((rc = center_rows(b.cx, D, nC, D, b.cpiv, b.cxs0, b.cxb, D, main))) return rc;
    if ((rc = linear(w.gene_map, gene_pooled, w.token_dim, t.n_gene_chunks, D, w.token_dim, VF_EPI_BIAS_F32, nullptr, 0, 0,
                     b.gene_emb, D, nullptr, 0, nullptr, 0, 0.f, nullptr, main))) return rc;
    if ((rc = gather_rows(b.gene_emb, D, w.registry, D, t.gene_idx, Mg, D, b.gx, nullptr, D, main))) return rc;
    if ((rc = center_rows(b.gx, D, Mg, D, b.gpiv, b.gxs0, b.gxb, D, main))) return rc;

    auto kv_of = [&](int i) { return b.kv + (size_t)i * nC * 2 * D; };
    auto project_kv = [&](int i, cudaStream_t s) {           // K/V of gene layer i's cross-attention: shared by every tissue copy
        return linear(w.gene_layers[i].kv, b.ctx, D, nC, 2 * D, D, VF_EPI_BIAS_BF16, nullptr, 0, 0, kv_of(i), 2 * D, nullptr, 0,
                      nullptr, 0, 0.f, nullptr, s);
    };
    const float* cxs = b.cxs0; int cxs_parts = 1;
    auto cre_layer = [&](int i, cudaStream_t s) -> int {
        float* out_stats = nullptr;
        int r2 = context_layer(w.cre_layers[i], w, b.cx, b.cxb, cxs, cxs_parts, nC, b.cs,
            [&](bf16* qkv, bf16* o) { return attention_mc_varlen(qkv, 3 * D, qkv + D, 3 * D, qkv + 2 * D, 3 * D, o, D, nC, nC,
                                                                 t.slots_cself, t.n_cself, H, hd, w.slopes, s); },
            [&](bf16* q, bf16* o) { return label_attention(q, 3 * D, w.cre_layers[i].kv9, t.logc, t.row_seq, nC, H, hd, o, D, s); },
            &out_stats, s);
        if (r2) return r2;
        cxs = out_stats; cxs_parts = P;
        return uncenter_rows(b.cx, D, b.cpiv, nullptr, nC, D, nullptr, b.ctx, D, s);      // context of gene layer i + 1
    };
    // ---- the CRE stack runs ahead on the library's side stream; gene layer i waits for event i ----
    const bool two = t.single_stream == 0 && NL > 1;
    SideStream& ss = side_stream(NL);
    cudaStream_t side = two ? ss.s : main;
    if (two) {
        VF_CUDA_OK(cudaEventRecord(ss.start, main));
        VF_CUDA_OK(cudaStreamWaitEvent(side, ss.start, 0));
        if ((rc = project_kv(0, side))) return rc;
        VF_CUDA_OK(cudaEventRecord(ss.ev[0], side));
        for (int i = 0; i + 1 < NL; ++i) {
            if ((rc = cre_layer(i, side))) return rc;
            if ((rc = project_kv(i + 1, side))) return rc;
            VF_CUDA_OK(cudaEventRecord(ss.ev[i + 1], side));
        }
    }
    const float* gxs = b.gxs0; int gxs_parts = 1;
    const bool prune = NL > 1;
    for (int i = 0; i < NL; ++i) {
        if (two) VF_CUDA_OK(cudaStreamWaitEvent(main, ss.ev[i], 0));
        else {
            if (i > 0 && (rc = cre_layer(i - 1, main))) return rc;
            if ((rc = project_kv(i, main))) return rc;
        }
        if (i < NL - 1 || !prune) {
            float* out_stats = nullptr;
            bf16* kv = kv_of(i);
            if ((rc = context_layer(w.gene_layers[i], w, b.gx, b.gxb, gxs, gxs_parts, Mg, b.gs,
                [&](bf16* qkv, bf16* o) { return attention_mc_varlen(qkv, 3 * D, qkv + D, 3 * D, qkv + 2 * D, 3 * D, o, D, Mg, Mg,
                                                                     t.slots_gself, t.n_gself, H, hd, w.slopes, main); },
                [&](bf16* q, bf16* o) {
                    int r2 = attention_mc_varlen(q, 3 * D, kv, 2 * D, kv + D, 2 * D, o, D, Mg, nC, t.slots_gcross, t.n_gcross, H,
                                                 hd, nullptr, main);
                    return r2 ? r2 : maps(q, 3 * D, attn ? attn->reg_rows : nullptr, kv, i);
                },
                &out_stats, main))) return rc;
            gxs = out_stats; gxs_parts = P;
        }
    }
    const float* last = nullptr;                              // [R, D] fp32, raw (un-centred)
    if (prune) {
        // last gene layer on the rows whose output is read (engine.py: _gene_layer_last)
        const vf_context_layer_t& L = w.gene_layers[NL - 1];
        bf16* kvs = b.gs.qkv + D;                             // K | V of every row (Q columns unused)
        vf_linear_t kvw{reinterpret_cast<const bf16*>(L.qkv.w) + (size_t)D * D, L.qkv.b + D, L.qkv.cs + D};
        vf_linear_t qw{L.qkv.w, L.qkv.b, L.qkv.cs};
        if ((rc = gemm_bf16(b.gxb, D, kvw.w, D, Mg, 2 * D, D, VF_EPI_BIAS_BF16, kvw.b, nullptr, 0, 0, kvs, 3 * D, nullptr, 0, gxs,
                            gxs_parts, kvw.cs, D, w.ln_eps, nullptr, main))) return rc;
        if ((rc = gather_rows(b.gx, D, nullptr, 0, t.last_rows, R, D, b.xR, b.xbR, D, main))) return rc;
        if ((rc = gather_rows(gxs, 2 * gxs_parts, nullptr, 0, t.last_rows, R, 2 * gxs_parts, b.stR, nullptr, 2 * gxs_parts, main)))
            return rc;
        if ((rc = gemm_bf16(b.xbR, D, qw.w, D, R, D, D, VF_EPI_BIAS_BF16, qw.b, nullptr, 0, 0, b.qR, D, nullptr, 0, b.stR, gxs_parts,
                            qw.cs, D, w.ln_eps, nullptr, main))) return rc;
        if ((rc = attention_mc_varlen(b.qR, D, kvs, 3 * D, kvs + D, 3 * D, b.aR, D, R, Mg, t.slots_last_self, t.n_last_self, H, hd,
                                      w.slopes, main))) return rc;
        if ((rc = linear(L.out, b.aR, D, R, D, D, VF_EPI_BIAS_RESID_F32, b.xbR, 1, D, nullptr, 0, b.hbR, D, nullptr, 0, 0.f, b.s1R,
                         main))) return rc;
        if ((rc = linear(L.q, b.hbR, D, R, D, D, VF_EPI_BIAS_BF16, nullptr, 0, 0, b.qR, D, nullptr, 0, b.s1R, P, w.ln_eps, nullptr,
                         main))) return rc;
        bf16* kv = kv_of(NL - 1);
        if ((rc = attention_mc_varlen(b.qR, D, kv, 2 * D, kv + D, 2 * D, b.aR, D, R, nC, t.slots_last_cross, t.n_last_cross, H, hd,
                                      nullptr, main))) return rc;
        if ((rc = maps(b.qR, D, nullptr, kv, NL - 1))) return rc;
        if ((rc = linear(L.out2, b.aR, D, R, D, D, VF_EPI_BIAS_RESID_F32, b.hbR, 1, D, nullptr, 0, b.hbR, D, nullptr, 0, 0.f, b.s1R,
                         main))) return rc;
        if ((rc = linear(L.g1, b.hbR, D, R, F, D, VF_EPI_BIAS_GEGLU_BF16, nullptr, 0, 0, b.fR, F / 2, nullptr, 0, b.s1R, P, w.ln_eps,
                         nullptr, main))) return rc;
        if ((rc = linear(L.g2, b.fR, F / 2, R, D, F / 2, VF_EPI_BIAS_RESID_F32, b.xR, 0, D, b.xR, D, nullptr, 0, nullptr, 0, 0.f,
                         nullptr, main))) return rc;
        if ((rc = uncenter_rows(b.xR, D, b.gpiv, t.last_rows, R, D, b.lastf, b.lastb, D, main))) return rc;
        last = b.lastf;
    } else {
        if ((rc = gather_rows(b.gx, D, nullptr, 0, t.last_rows, R, D, b.xR, nullptr, D, main))) return rc;
        if ((rc = uncenter_rows(b.xR, D, b.gpiv, t.last_rows, R, D, b.lastf, b.lastb, D, main))) return rc;
        last = b.lastf;
    }
    // ---- registry rows -> embeddings -> head (layers.py:1078-1087) ----
    VF_CUDA_OK(cudaMemcpyAsync(emb, last, (size_t)n_reg * D * sizeof(float), cudaMemcpyDeviceToDevice, main));
    if (gene_token_emb && R > n_reg)
        VF_CUDA_OK(cudaMemcpyAsync(gene_token_emb, last + (size_t)n_reg * D, (size_t)(R - n_reg) * D * sizeof(float),
                                   cudaMemcpyDeviceToDevice, main));
    if ((rc = linear(w.h0, b.lastb, D, n_reg, D, D, VF_EPI_BIAS_F32, nullptr, 0, 0, b.h1, D, nullptr, 0, nullptr, 0, 0.f, nullptr,
                     main))) return rc;
    if ((rc = layernorm(b.h1, D, w.hn_g, w.hn_b, n_reg, D, w.ln_eps, b.h1n, D, 1, main))) return rc;
    if ((rc = linear(w.h4, b.h1n, D, n_reg, D, D, VF_EPI_BIAS_GELU_BF16, nullptr, 0, 0, b.h2, D, nullptr, 0, nullptr, 0, 0.f, nullptr,
                     main))) return rc;
    if ((rc = head_out(b.h2, D, w.h6_w, w.h6_b, n_reg, D, 1, pred, main))) return rc;
    if (cre_token_emb && t.cre_pos_idx) {
        if ((rc = gather_rows(b.cx, D, nullptr, 0, t.cre_pos_idx, n_reg, D, b.tokf, nullptr, D, main))) return rc;
        if ((rc = uncenter_rows(b.tokf, D, b.cpiv, t.cre_pos_idx, n_reg, D, cre_token_emb, nullptr, D, main))) return rc;
    }
    return 0;
}

// CRE-token rows of the forward that just ran: the final CRE stream and its pivots are still in the workspace
static int seq2gene_cre_rows(const vf_seq2gene_weights_t& w, const vf_seq2gene_slab_t& t, void* ws, size_t ws_bytes,
                             const int32_t* rows, int n, float* out, cudaStream_t s) {
    if (n == 0) return 0;
    Seq2GeneWs b = carve_seq2gene(w, t, ws);
    VF_REQUIRE(ws && ws_bytes >= b.bytes, "seq2gene_cre_rows: workspace of %zu bytes < %zu needed", ws_bytes, b.bytes);
    VF_REQUIRE(rows && out, "seq2gene_cre_rows: NULL rows / out");
    int rc;
    if ((rc = gather_rows(b.cx, w.D, nullptr, 0, rows, n, w.D, out, nullptr, w.D, s))) return rc;
    return uncenter_rows(out, w.D, b.cpiv, rows, n, w.D, out, nullptr, w.D, s);
}

// ====================================================================================================================
// attention work tables (host): the C counterpart of variantformer_b200.ops.SlotMap
// ====================================================================================================================
static int build_slots(const int32_t* q_lens, const int32_t* k_lens, int n_seq, int pair_unrelated, int32_t* out, int max_items) {
    struct Rec { int32_t v[8]; };
    std::vector<Rec> pairs, singles;
    long cq = 0, ck = 0;
    for (int i = 0; i < n_seq; ++i) {
        const int ql = q_lens[i], kl = k_lens ? k_lens[i] : q_lens[i];
        const int nt = (ql + 127) / 128;
        for (int t = 0; t < nt && kl > 0; ++t) {
            Rec r{};
            r.v[0] = (int32_t)(cq + 128 * t); r.v[1] = std::min(128, ql - 128 * t); r.v[2] = (int32_t)ck; r.v[3] = kl;
            r.v[4] = 128 * t + kl - ql;
            ((t == nt - 1 && (nt & 1)) ? singles : pairs).push_back(r);
        }
        cq += ql; ck += kl;
    }
    const size_t n_pair_items = pairs.size() / 2;
    const size_t n_single_items = pair_unrelated ? (singles.size() + 1) / 2 : singles.size();
    const size_t n_items = n_pair_items + n_single_items;
    if (!out) return (int)n_items;
    VF_REQUIRE((size_t)max_items >= n_items, "attention_build_slots: table of %d items < %zu needed", max_items, n_items);
    memset(out, 0, n_items * 16 * sizeof(int32_t));
    for (size_t i = 0; i < pairs.size(); ++i) memcpy(out + i * 8, pairs[i].v, 32);
    int32_t* o = out + n_pair_items * 16;
    for (size_t i = 0; i < singles.size(); ++i) {
        const size_t item = pair_unrelated ? i / 2 : i, slot = pair_unrelated ? i % 2 : 0;
        memcpy(o + item * 16 + slot * 8, singles[i].v, 32);
    }
    return (int)n_items;
}

}  // namespace vf

using namespace vf;
#define ST(s) reinterpret_cast<cudaStream_t>(s)

extern "C" {

int vf_attention_build_slots(const int32_t* q_lens, const int32_t* k_lens, int n_seq, int pair_unrelated, int32_t* out_table,
                             int max_items) {
    return build_slots(q_lens, k_lens, n_seq, pair_unrelated, out_table, max_items);
}

size_t vf_seq2reg_workspace_bytes(const vf_seq2reg_weights_t* w, int64_t n_tok) {
    return w ? carve_seq2reg(*w, n_tok, nullptr).bytes : 0;
}

int vf_seq2reg_forward(const vf_seq2reg_weights_t* w, const int32_t* tokens, const uint8_t* pad_mask, const int32_t* cu,
                       int n_win, int L, int64_t n_tok, const int32_t* slots, int n_items, void* workspace,
                       size_t workspace_bytes, void* out_bf16, void* stream) {
    VF_REQUIRE(w, "seq2reg_forward: NULL weight table");
    return seq2reg_forward(*w, tokens, pad_mask, cu, n_win, L, n_tok, slots, n_items, workspace, workspace_bytes, out_bf16,
                           ST(stream));
}

size_t vf_seq2gene_workspace_bytes(const vf_seq2gene_weights_t* w, const vf_seq2gene_slab_t* slab) {
    return (w && slab) ? carve_seq2gene(*w, *slab, nullptr).bytes : 0;
}

int vf_seq2gene_forward(const vf_seq2gene_weights_t* w, const vf_seq2gene_slab_t* slab, const void* cre_pooled_bf16,
                        const void* gene_pooled_bf16, void* workspace, size_t workspace_bytes, float* pred, float* emb,
                        float* gene_token_emb, float* cre_token_emb, void* stream) {
    VF_REQUIRE(w && slab, "seq2gene_forward: NULL weight table / slab");
    return seq2gene_forward(*w, *slab, cre_pooled_bf16, gene_pooled_bf16, workspace, workspace_bytes, pred, emb, gene_token_emb,
                            cre_token_emb, nullptr, ST(stream));
}

int vf_seq2gene_forward_attn(const vf_seq2gene_weights_t* w, const vf_seq2gene_slab_t* slab, const void* cre_pooled_bf16,
                             const void* gene_pooled_bf16, void* workspace, size_t workspace_bytes, float* pred, float* emb,
                             float* gene_token_emb, float* cre_token_emb, const vf_cre_attention_t* attn, void* stream) {
    VF_REQUIRE(w && slab, "seq2gene_forward: NULL weight table / slab");
    return seq2gene_forward(*w, *slab, cre_pooled_bf16, gene_pooled_bf16, workspace, workspace_bytes, pred, emb, gene_token_emb,
                            cre_token_emb, attn, ST(stream));
}

int vf_seq2gene_cre_rows(const vf_seq2gene_weights_t* w, const vf_seq2gene_slab_t* slab, void* workspace,
                         size_t workspace_bytes, const int32_t* rows, int n, float* out_f32, void* stream) {
    VF_REQUIRE(w && slab, "seq2gene_cre_rows: NULL weight table / slab");
    return seq2gene_cre_rows(*w, *slab, workspace, workspace_bytes, rows, n, out_f32, ST(stream));
}

}  // extern "C"
