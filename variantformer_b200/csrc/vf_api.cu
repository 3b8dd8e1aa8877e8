// vf_api.cu — the extern "C" surface declared in include/vf_b200.h (plain pointers and sizes only).
#include <stdarg.h>
#include <stdio.h>

#include "vf_common.cuh"
#include "vf_internal.h"

namespace vf {
unsigned long long g_launches = 0;
static thread_local char g_err[512] = "";
void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
int cuda_fail(cudaError_t e, const char* what) {
    set_error("%s: %s (%s)", what, cudaGetErrorName(e), cudaGetErrorString(e));
    return -2;
}
}  // namespace vf

using namespace vf;
#define ST(s) reinterpret_cast<cudaStream_t>(s)

extern "C" {

const char* vf_last_error(void) { return g_err; }
int vf_abi_version(void) { return VF_B200_ABI_VERSION; }
unsigned long long vf_launch_count(void) { return __atomic_load_n(&g_launches, __ATOMIC_RELAXED); }

int vf_device_check(int* sm_count) {
    int dev = 0, major = 0, sms = 0;
    VF_CUDA_OK(cudaGetDevice(&dev));
    VF_CUDA_OK(cudaDeviceGetAttribute(&major, cudaDevAttrComputeCapabilityMajor, dev));
    VF_CUDA_OK(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
    if (sm_count) *sm_count = sms;
    VF_REQUIRE(major == 10, "libvf_b200 is built for sm_100a only; current device has compute capability %d.x", major);
    return 0;
}

int vf_gemm_bf16(const void* A, int lda, const void* W, int ldw, int M, int N, int K, int epilogue, const float* bias,
                 const float* resid, int ldr, void* out, int ldo, void* out2_bf16, int ldo2, void* stream) {
    return gemm_bf16(A, lda, W, ldw, M, N, K, epilogue, bias, resid, 0, ldr, out, ldo, out2_bf16, ldo2, nullptr, 0, nullptr,
                     0, 0.f, nullptr, ST(stream));
}
int vf_gemm_bf16_ln(const void* A, int lda, const void* W, int ldw, int M, int N, int K, int epilogue,
                    const float* bias, const void* resid, int resid_bf16, int ldr, void* out, int ldo, void* out2_bf16, int ldo2,
                    const float* ln_stats, int ln_parts, const float* ln_colsum, int ln_dim, float ln_eps,
                    float* stats_out, void* stream) {
    return gemm_bf16(A, lda, W, ldw, M, N, K, epilogue, bias, resid, resid_bf16, ldr, out, ldo, out2_bf16, ldo2, ln_stats,
                     ln_parts, ln_colsum, ln_dim, ln_eps, stats_out, ST(stream));
}
int vf_rowstats(const float* x, int ldx, int M, int d, float* stats, void* out_bf16, int ldo, void* stream) {
    return rowstats(x, ldx, M, d, stats, out_bf16, ldo, ST(stream));
}
int vf_attention_mc_varlen(const void* q, int ldq, const void* k, int ldk, const void* v, int ldv, void* o, int ldo,
                           int64_t rows_q, int64_t rows_k, const int32_t* slots, int n_items, int heads,
                           int head_dim, const float* slopes, void* stream) {
    return attention_mc_varlen(q, ldq, k, ldk, v, ldv, o, ldo, (long)rows_q, (long)rows_k, slots, n_items, heads,
                               head_dim, slopes, ST(stream));
}
int vf_label_attention(const void* q, int ldq, const float* kv9, const float* logc, const int32_t* row_seq, int n_rows,
                       int heads, int head_dim, void* out, int ldo, void* stream) {
    return label_attention(q, ldq, kv9, logc, row_seq, n_rows, heads, head_dim, out, ldo, ST(stream));
}
int vf_layernorm(const float* x, int ldx, const float* gamma, const float* beta, int M, int d, float eps,
                 void* out_bf16, int ldo, int act_gelu, void* stream) {
    return layernorm(x, ldx, gamma, beta, M, d, eps, out_bf16, ldo, act_gelu, ST(stream));
}
int vf_window_lengths(const uint8_t* pad_mask, int n_win, int L, int32_t* lens, void* stream) {
    return window_lengths(pad_mask, n_win, L, lens, ST(stream));
}
int vf_compact_tokens(const int32_t* tokens, const uint8_t* pad_mask, const int32_t* cu, int n_win, int L,
                      int32_t* out_ids, int32_t* out_pos, void* stream) {
    return compact_tokens(tokens, pad_mask, cu, n_win, L, out_ids, out_pos, ST(stream));
}
int vf_embed_tokens(const int32_t* ids, const int32_t* pos, const float* emb, const float* pe, int n_tok, int d,
                    float* out, void* stream) {
    return embed_tokens(ids, pos, emb, pe, n_tok, d, out, ST(stream));
}
int vf_masked_meanpool(const float* x, int ldx, const int32_t* cu, int n_win, int d, const float* pivot, void* out_bf16,
                       float* out_f32, int ldo, void* stream) {
    return masked_meanpool(x, ldx, cu, n_win, d, pivot, out_bf16, out_f32, ldo, ST(stream));
}
int vf_center_rows(float* x, int ldx, int M, int d, float* pivot, float* stats, void* out_bf16, int ldo, void* stream) {
    return center_rows(x, ldx, M, d, pivot, stats, out_bf16, ldo, ST(stream));
}
int vf_uncenter_rows(const float* x, int ldx, const float* pivot, const int32_t* idx, int M, int d, float* out_f32,
                     void* out_bf16, int ldo, void* stream) {
    return uncenter_rows(x, ldx, pivot, idx, M, d, out_f32, out_bf16, ldo, ST(stream));
}
int vf_gather_rows(const float* table_a, int lda, const float* table_b, int ldb, const int32_t* idx, int n_rows, int d,
                   float* out_f32, void* out_bf16, int ldo, void* stream) {
    return gather_rows(table_a, lda, table_b, ldb, idx, n_rows, d, out_f32, out_bf16, ldo, ST(stream));
}
int vf_head_out(const void* h_bf16, int ldh, const float* w, const float* b, int n_rows, int d, int softplus,
                float* out, void* stream) {
    return head_out(h_bf16, ldh, w, b, n_rows, d, softplus, out, ST(stream));
}
int vf_cast_f32_to_bf16(const float* x, void* y_bf16, size_t n, void* stream) {
    return cast_f32_to_bf16(x, y_bf16, n, ST(stream));
}
int vf_forest_predict(const float* x, int ldx, int n_rows, int d, const int32_t* row_forest, const int32_t* forest_tree_off,
                      const float* forest_base, const int32_t* tree_root, const int32_t* node_feat, const float* node_thr,
                      const int32_t* node_left, const int32_t* node_right, const float* node_value, int op_lt, float* out,
                      void* stream) {
    return forest_predict(x, ldx, n_rows, d, row_forest, forest_tree_off, forest_base, tree_root, node_feat, node_thr,
                          node_left, node_right, node_value, op_lt, out, ST(stream));
}
int vf_encode_windows(const uint8_t* genome, const int64_t* win_base, const int32_t* w0, const int32_t* w1,
                      const int32_t* var_lo, const int32_t* var_hi, const uint8_t* flags, const int32_t* v_pos,
                      const int32_t* v_ref_len, const int32_t* v_alt_off, const int32_t* v_alt_len, const uint8_t* v_gt,
                      const uint8_t* alt_pool, int n_win, int max_window, uint8_t* out, int64_t pitch, int32_t* out_len,
                      int32_t* err, void* stream) {
    return encode_windows(genome, win_base, w0, w1, var_lo, var_hi, flags, v_pos, v_ref_len, v_alt_off, v_alt_len,
                          v_gt, alt_pool, n_win, max_window, out, pitch, out_len, err, ST(stream));
}
int vf_mutate_windows(const uint8_t* src, int64_t src_pitch, const int32_t* src_len, const int32_t* row_src,
                      const int32_t* row_off, const uint8_t* row_base, const uint8_t* flags, int n_rows, uint8_t* out,
                      int64_t out_pitch, int32_t* out_len, int32_t* err, void* stream) {
    return mutate_windows(src, src_pitch, src_len, row_src, row_off, row_base, flags, n_rows, out, out_pitch, out_len, err,
                          ST(stream));
}
int vf_bpe_tokenize(const uint8_t* seq, int64_t pitch, const int32_t* len, int n_win, int max_len,
                    const uint16_t* merge_a, const uint16_t* merge_b, const uint16_t* merge_new,
                    const uint16_t* merge_batch, int n_merges, uint16_t* scratch, int64_t scratch_pitch, int32_t* out_tokens, int out_pitch, int out_cap,
                    int32_t* out_count, int32_t* out_start, int64_t start_pitch, int block_threads, void* stream) {
    return bpe_tokenize(seq, pitch, len, n_win, max_len, merge_a, merge_b, merge_new, merge_batch, n_merges, scratch,
                        scratch_pitch, out_tokens, out_pitch, out_cap, out_count, out_start, start_pitch, block_threads,
                        ST(stream));
}

}  // extern "C"
