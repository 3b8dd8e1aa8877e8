// vf_internal.h — declarations shared between the .cu translation units (not installed).
#pragma once
#include <cuda_runtime.h>
#include <stddef.h>
#include <stdint.h>

#include "../../include/vf_b200.h"

namespace vf {

int gemm_bf16(const void* A, int lda, const void* W, int ldw, int M, int N, int K, int epi, const float* bias,
              const void* resid, int resid_bf16, int ldr, void* out, int ldo, void* out2, int ldo2, const float* ln_stats,
              int ln_parts, const float* ln_colsum, int ln_dim, float ln_eps, float* stats_out, cudaStream_t stream);

int attention_mc_varlen(const void* q, int ldq, const void* k, int ldk, const void* v, int ldv, void* o, int ldo,
                        long rows_q, long rows_k, const int* slots, int n_items, int heads, int head_dim,
                        const float* slopes, cudaStream_t stream);

int layernorm(const float* x, int ldx, const float* gamma, const float* beta, int M, int d, float eps, void* out,
              int ldo, int act_gelu, cudaStream_t s);
int rowstats(const float* x, int ldx, int M, int d, float* stats, void* out_bf16, int ldo, cudaStream_t s);
int window_lengths(const uint8_t* pad_mask, int n_win, int L, int* lens, cudaStream_t s);
int compact_tokens(const int* tokens, const uint8_t* pad_mask, const int* cu, int n_win, int L, int* out_ids,
                   int* out_pos, cudaStream_t s);
int embed_tokens(const int* ids, const int* pos, const float* emb, const float* pe, int n_tok, int d, float* out,
                 cudaStream_t s);
int center_rows(float* x, int ldx, int M, int d, float* pivot, float* stats, void* out_bf16, int ldo, cudaStream_t s);
int embed_center(const int* ids, const int* pos, const float* emb, const float* pe, int n_tok, int d, float* x,
                 float* pivot, float* stats, void* out_bf16, cudaStream_t s);
int uncenter_rows(const float* x, int ldx, const float* pivot, const int* idx, int M, int d, float* out_f32,
                  void* out_bf16, int ldo, cudaStream_t s);
int masked_meanpool(const float* x, int ldx, const int* cu, int n_win, int d, const float* pivot, void* out_bf16,
                    float* out_f32, int ldo, cudaStream_t s);
int gather_rows(const float* ta, int lda, const float* tb, int ldb, const int* idx, int n_rows, int d, float* out_f32,
                void* out_bf16, int ldo, cudaStream_t s);
int label_attention(const void* q, int ldq, const float* kv9, const float* logc, const int* row_seq, int n_rows, int H,
                    int HD, void* out, int ldo, cudaStream_t s);
int head_out(const void* h, int ldh, const float* w, const float* b, int n_rows, int d, int softplus, float* out,
             cudaStream_t s);
int cast_f32_to_bf16(const float* x, void* y, size_t n, cudaStream_t s);
int forest_predict(const float* x, int ldx, int n_rows, int d, const int* row_forest, const int* forest_tree_off,
                   const float* forest_base, const int* tree_root, const int* node_feat, const float* node_thr,
                   const int* node_left, const int* node_right, const float* node_value, int op_lt, float* out,
                   cudaStream_t s);

int encode_windows(const uint8_t* genome, const int64_t* win_base, const int32_t* w0, const int32_t* w1,
                   const int32_t* var_lo, const int32_t* var_hi, const uint8_t* flags, const int32_t* v_pos,
                   const int32_t* v_ref_len, const int32_t* v_alt_off, const int32_t* v_alt_len, const uint8_t* v_gt,
                   const uint8_t* alt_pool, int n_win, int max_window, uint8_t* out, int64_t pitch, int32_t* out_len,
                   int32_t* err, cudaStream_t s);
int mutate_windows(const uint8_t* src, int64_t src_pitch, const int32_t* src_len, const int32_t* row_src,
                   const int32_t* row_off, const uint8_t* row_base, const uint8_t* flags, int n_rows, uint8_t* out,
                   int64_t out_pitch, int32_t* out_len, int32_t* err, cudaStream_t s);
int bpe_tokenize(const uint8_t* seq, int64_t pitch, const int32_t* len, int n_win, int max_len,
                 const uint16_t* merge_a, const uint16_t* merge_b, const uint16_t* merge_new,
                 const uint16_t* merge_batch, int n_merges, uint16_t* scratch, int64_t scratch_pitch, int32_t* out_tokens, int out_pitch, int out_cap,
                 int32_t* out_count, int32_t* out_start, int64_t start_pitch, int block_threads, cudaStream_t s);

}  // namespace vf
