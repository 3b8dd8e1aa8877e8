/*
 * vf_b200.h — C ABI of libvf_b200.so: the sm_100a CUDA kernels behind VariantFormer's
 * batched-inference hot path.
 *
 * The reference has no FFI of its own: its boundary is a set of Python call sites that
 * reach third-party native code (flash_attn, cuBLASLt via nn.Linear, ATen, HuggingFace
 * tokenizers, samtools/bcftools subprocesses).  Each entry point below names the reference
 * call site (file:line under the reference checkout) it replaces; INTEGRATION.md shows the
 * ctypes stub a maintainer of the reference would add.
 *
 * Conventions
 *   - every function returns 0 on success and a negative value on error;
 *     vf_last_error() then returns a thread-local message.  Nothing throws, nothing
 *     allocates device memory (callers own every buffer), nothing synchronises the device.
 *   - all pointers are DEVICE pointers unless noted; `stream` is a cudaStream_t passed as void*.
 *   - bf16 buffers are plain uint16 storage (__nv_bfloat16); "ld*" are row strides in ELEMENTS.
 *   - re-entrant per stream; the only global state is read-only after first use.
 */
#ifndef VF_B200_H
#define VF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VF_B200_ABI_VERSION 2

const char* vf_last_error(void);
int vf_abi_version(void);
/* Kernels launched by this library since it was loaded (process-wide; bench.py reports the difference over its timed
 * region as gpu_launches). */
unsigned long long vf_launch_count(void);
/* Device sanity: returns 0 iff the current device is compute capability 10.x; fills sm_count. */
int vf_device_check(int* sm_count);

/* ---- GEMM epilogues ------------------------------------------------------------------- */
enum {
    VF_EPI_BIAS_BF16 = 0,       /* out bf16 [M,N]   = A·W^T + bias                                     */
    VF_EPI_BIAS_GEGLU_BF16 = 1, /* out bf16 [M,N/2] = (u+bu) * gelu_erf(g+bg); W/bias rows tile-interleaved:
                                   rows [256j,256j+128) = u columns [128j,128j+128), next 128 rows = their gates */
    VF_EPI_BIAS_RESID_F32 = 2,  /* out fp32 [M,N]   = A·W^T + bias + resid (out may alias resid); optional bf16 mirror */
    VF_EPI_BIAS_F32 = 3,        /* out fp32 [M,N]   = A·W^T + bias; optional bf16 mirror                 */
    VF_EPI_BIAS_GELU_BF16 = 4,  /* out bf16 [M,N]   = gelu_erf(A·W^T + bias)                             */
    VF_EPI_COUNT = 5
};

/*
 * D = A[M,K] (bf16, row stride lda) x W[N,K]^T (bf16 nn.Linear weight layout, row stride ldw), fp32
 * accumulation on tcgen05 tensor cores (TMA-fed, TMEM accumulators).
 * Replaces nn.Linear under bf16 autocast (cuBLASLt): seq2reg/modules.py:140-147;
 * seq2gene/modules/layers.py:63-80 + flash_attn MHA Wqkv/Wq/Wkv/out_proj;
 * seq2gene/model_combined_modulator.py:502-507,610-612; seq2gene/modules/layers.py:1078-1087.
 * N % 8 == 0, K % 8 == 0, 16-byte aligned operands.  bias/resid/out2 may be NULL.
 * Alignment: A, W, out, out2_bf16 and resid 16-byte aligned; lda, ldw, ldo, ldo2 multiples of 8 elements; ldr a
 * multiple of 4 elements (fp32 residual) or of 8 (bf16 residual); stats_out and ln_stats (vf_gemm_bf16_ln) 8-byte
 * aligned, ln_stats 16-byte aligned when ln_parts is even and at most 16.  A violation returns an error and launches
 * nothing; the operands the epilogue writes or reads (out, out2, resid, stats_out, ln_stats) are checked even when
 * M == 0.
 */
int vf_gemm_bf16(const void* A, int lda, const void* W, int ldw, int M, int N, int K, int epilogue,
                 const float* bias, const float* resid, int ldr, void* out, int ldo, void* out2_bf16, int ldo2,
                 void* stream);

/*
 * Same GEMM with the LayerNorm that precedes the Linear folded in, and/or row statistics of the output:
 *   ln_stats (fp32 [M, ln_parts, 2] = partial per-row sums and sums of squares of the fp32 rows that A mirrors in bf16;
 *   the partials of a row are added in index order), ln_colsum (fp32 [N], column sums of the gamma-folded weight, same
 *   layout as bias), ln_dim (normalised width), ln_eps:
 *     out = epilogue( rstd_r * (A·W'^T - mean_r * colsum) + bias' ),  W' = W*gamma, bias' = bias + W·beta
 *   which equals Linear(LayerNorm(x)) (seq2reg/modules.py:143-147,176-189; seq2gene/modules/layers.py:74-76,116-163).
 *   Allowed with the bf16 epilogues only.  NULL ln_stats = plain GEMM.
 *   stats_out (fp32 [M, 2*ceil(N/256), 2]): the fp32 epilogues store one partial (sum, sum of squares) of every output
 *   row per 128-column half tile (plain stores: deterministic), i.e. the ln_stats of the next folded GEMM with
 *   ln_parts = 2*ceil(N/256).  NULL = off.
 *   resid_bf16 != 0: the residual of VF_EPI_BIAS_RESID_F32 is a bf16 matrix (row stride ldr elements).  The fp32
 *   epilogues accept out == NULL when out2_bf16 is given: only the bf16 mirror (and the statistics) are written.  Both
 *   serve the intra-layer temporaries x1 = MHA(LN(x)) + x of the encoder layers, which are consumed only through a
 *   LayerNorm feeding a bf16 GEMM (the layer's residual path is the layer INPUT: layers.py:163, modules.py:189).
 */
int vf_gemm_bf16_ln(const void* A, int lda, const void* W, int ldw, int M, int N, int K, int epilogue,
                    const float* bias, const void* resid, int resid_bf16, int ldr, void* out, int ldo, void* out2_bf16, int ldo2,
                    const float* ln_stats, int ln_parts, const float* ln_colsum, int ln_dim, float ln_eps,
                    float* stats_out, void* stream);
/* Per-row (sum, sum of squares) of an fp32 matrix [M,d] into stats [M,1,2] + optional bf16 mirror: the statistics of a
 * stream at the point it is assembled (seq2reg/model.py:214-220 embeddings; layers.py:508-521 registry prepend). */
int vf_rowstats(const float* x, int ldx, int M, int d, float* stats, void* out_bf16, int ldo, void* stream);

/*
 * Variable-length non-causal attention, one launch for all sequences and heads:
 *   o = softmax(q k^T / sqrt(head_dim) - slope_h * |i + Sk - Sq - j|) v      (fp32 statistics, bf16 operands)
 * tcgen05 tensor cores (TMA-staged Q/K/V tiles, S and O accumulators in TMEM, one softmax thread per query row,
 * single-pass softmax with a lazily raised reference maximum), two co-resident CTAs per SM.
 * q/k/v/o: bf16, head h at columns [h*head_dim, (h+1)*head_dim) of each row; packed QKV/KV buffers are addressed by
 * passing offset base pointers.  rows_q / rows_k = total rows of the q and k/v tensors (TMA bounds).
 * A work item has two SLOTS, each a query tile of up to 128 rows of one sequence.
 * slots: int32 [n_items][2][8], 16-byte aligned, per slot {first query row (absolute row of q/o), valid rows (0 = empty
 * slot; slot 0 of an item is never the empty one), first key row (absolute row of k/v), number of keys (> 0),
 * i + Sk - Sq of the tile's first row (ALiBi position), 0, 0, 0}.  Two slots with the same (first key row, keys) share
 * one K/V stream; two slots with different key ranges stream their own keys (any mixture of the two kinds of item in
 * one launch is fine: the MMA issuers order their ring waits behind the producer's issue counters, DESIGN.md section 5).
 * Rows past a sequence's last key that a 64-key block over-fetches are masked in S and cleared in V, so non-finite
 * values in a neighbouring sequence never reach this one.  slopes: fp32 [heads] ALiBi slopes or NULL.
 * head_dim in {48, 64}.
 * Replaces flash_attn_varlen_qkvpacked_func / flash_attn_varlen_kvpacked_func as called through
 * flash_attn.modules.mha.MHA at seq2reg/modules.py:159-171 and seq2gene/modules/layers.py:344-351, 372-467.
 */
int vf_attention_mc_varlen(const void* q, int ldq, const void* k, int ldk, const void* v, int ldv, void* o, int ldo,
                           int64_t rows_q, int64_t rows_k, const int32_t* slots, int n_items, int heads,
                           int head_dim, const float* slopes, void* stream);

/*
 * Attention probabilities of a cross-attention for selected query rows (no positional bias), fp32:
 *   out[out_off[i] + (layer * heads + h) * n_keys + c] = softmax_c( q[row_i, h] . k[first_key + c, h] / sqrt(head_dim) )
 * for every query index i of group g (i in [group_q[2g], group_q[2g] + group_q[2g+1])), head h and key c in
 * [0, n_keys), where (first_key, n_keys) = (group_k[2g], group_k[2g+1]) and row_i = q_rows[i] (q_rows NULL: row_i = i).
 * Scores and softmax in fp32 over the whole key range (exact maximum, no lazy rescaling); bf16 operands as the fused
 * kernel reads them.  Per prediction the blocks of all layers form one [n_layers, heads, n_keys] array at out_off[i].
 * q / k: bf16, head h at columns [h*head_dim, (h+1)*head_dim) of each row (k: the K half of a packed KV buffer).
 * Groups of any size (64 query rows share one K stream); a group with <= 0 rows or keys writes nothing.  One CTA per
 * (group, head), CUDA cores.  Errors before any launch: head_dim not in {48, 64}, n_groups / layer < 0, heads not in
 * [1, 65535], q or k not 16-byte aligned, ldq / ldk not multiples of 8 or < heads * head_dim, out / q_rows / group
 * tables not 4-byte aligned, out_off not 8-byte aligned.
 * Serves the gene -> CRE cross-attention maps (seq2gene/modules/layers.py:142-150 with the gene stream as query).
 */
int vf_cross_attention_probs(const void* q, int ldq, const int32_t* q_rows, const int32_t* group_q, int n_groups,
                             const void* k, int ldk, const int32_t* group_k, int heads, int head_dim, float* out,
                             const int64_t* out_off, int layer, void* stream);

/*
 * CRE x reference-label cross-attention collapsed to the 9 cCRE classes (exact identity):
 * q bf16 [n_rows, H*HD]; kv9 fp32 [9, 2*H*HD] = Wkv·Emb9 + b ((two,h,d) order); logc fp32 [n_seq,9] =
 * log(#CREs of the class in the row's gene) (-inf when absent); row_seq int32 [n_rows].
 * Replaces the crossMHA call of the CRE stream: seq2gene/modules/layers.py:142-150 with
 * context = second_level_context_embedding(ref_labels) (model_combined_modulator.py:168,261-267).
 */
int vf_label_attention(const void* q, int ldq, const float* kv9, const float* logc, const int32_t* row_seq,
                       int n_rows, int heads, int head_dim, void* out, int ldo, void* stream);

/* nn.LayerNorm(eps) + optional exact GELU, fp32 [M,d] -> bf16 (seq2reg/modules.py:143-144;
 * seq2gene/modules/layers.py:74-76; head LayerNorm+GELU :1080-1081). */
int vf_layernorm(const float* x, int ldx, const float* gamma, const float* beta, int M, int d, float eps,
                 void* out_bf16, int ldo, int act_gelu, void* stream);

/* Valid-token counts per window from a pad mask (uint8, 1 = padding) [n_win, L]
 * (flash_attn.bert_padding.unpad_input at seq2reg/modules.py:156-161). */
int vf_window_lengths(const uint8_t* pad_mask, int n_win, int L, int32_t* lens, void* stream);
/* Ordered compaction of valid tokens: cu int32 [n_win+1] -> ids/pos int32 [n_tok]. */
int vf_compact_tokens(const int32_t* tokens, const uint8_t* pad_mask, const int32_t* cu, int n_win, int L,
                      int32_t* out_ids, int32_t* out_pos, void* stream);
/* x[t] = E[ids[t]] + PE[pos[t]] (pe may be NULL): seq2reg/model.py:214-220. */
int vf_embed_tokens(const int32_t* ids, const int32_t* pos, const float* emb, const float* pe, int n_tok, int d,
                    float* out, void* stream);
/* Mean over each window's tokens (seq2reg/model.py:263-267); empty window -> NaN as upstream.
 * pivot (fp32 [n_tok] or NULL): the rows are a centred stream (vf_center_rows); their pivots are added back. */
int vf_masked_meanpool(const float* x, int ldx, const int32_t* cu, int n_win, int d, const float* pivot, void* out_bf16,
                       float* out_f32, int ldo, void* stream);
/*
 * Row-centred residual streams.  Every consumer of a residual stream of the path is a LayerNorm (invariant under a
 * per-row shift: seq2reg/modules.py:176,185; layers.py:116,140,158) or a residual add (which carries a shift along), so
 * a stream may be kept as x' = x - pivot_r.  With pivot_r = the row mean where the stream is assembled, the bf16 mirror
 * that the LayerNorm-folded GEMMs read keeps the bits of the NORMALISED signal even when |mean| >> std (the reference
 * normalises in fp32 before rounding to bf16).
 * vf_center_rows: x <- x - mean_r in place (fp32 [M,d]); pivot[r] = mean_r; stats [M,1,2] = (sum, sum of squares) of
 * the shifted row; optional bf16 mirror.  Replaces vf_rowstats where a stream is born.
 * vf_uncenter_rows: out[r] = x[r] + pivot[idx ? idx[r] : r] (fp32 and/or bf16): raw values for the cross-attention
 * context (layers.py:142-150: context is not normalised) and for the returned embeddings.
 */
int vf_center_rows(float* x, int ldx, int M, int d, float* pivot, float* stats, void* out_bf16, int ldo, void* stream);
int vf_uncenter_rows(const float* x, int ldx, const float* pivot, const int32_t* idx, int M, int d, float* out_f32,
                     void* out_bf16, int ldo, void* stream);
/* out[r] = idx[r] >= 0 ? table_a[idx[r]] : table_b[-idx[r]-1]  (registry-token prepend / tissue replication:
 * seq2gene/modules/layers.py:508-521, model_combined_modulator.py:622-649; pool_outputs :391-392). */
int vf_gather_rows(const float* table_a, int lda, const float* table_b, int ldb, const int32_t* idx, int n_rows, int d,
                   float* out_f32, void* out_bf16, int ldo, void* stream);
/* y = softplus(h·w + b) per row (h bf16): last Linear(emb,1)+Softplus of the head, layers.py:1084-1087. */
int vf_head_out(const void* h_bf16, int ldh, const float* w, const float* b, int n_rows, int d, int softplus,
                float* out, void* stream);
int vf_cast_f32_to_bf16(const float* x, void* y_bf16, size_t n, void* stream);

/*
 * Gradient-boosted forest inference on embeddings — the AD-risk head.  Replaces treelite.gtil.predict per (gene, tissue)
 * row (processors/ad_risk.py:41-52, 157-176).  x fp32 [n_rows, d]; row_forest int32 [n_rows] = forest of every row;
 * forest_tree_off int32 [n_forests + 1] = range of the forest's trees in tree_root; forest_base fp32 [n_forests] = raw
 * score offset; tree_root int32 [n_trees] = root node of every tree; nodes (SoA over all forests): node_feat int32 (-1 =
 * leaf; bit 31 set on a split = missing values go left), node_thr fp32, node_left / node_right int32 (absolute node
 * indices), node_value fp32 (leaf contribution, learning rate folded in).  op_lt: 0 = "x <= thr goes left" (sklearn,
 * treelite "<="), 1 = "x < thr" (xgboost).  out fp32 [n_rows] = sigmoid(base + sum of leaf values) = P(class 1).
 */
int vf_forest_predict(const float* x, int ldx, int n_rows, int d, const int32_t* row_forest, const int32_t* forest_tree_off,
                      const float* forest_base, const int32_t* tree_root, const int32_t* node_feat, const float* node_thr,
                      const int32_t* node_left, const int32_t* node_right, const float* node_value, int op_lt, float* out,
                      void* stream);

/* ---- stage 1: genotype -> IUPAC sequence -> BPE-500 tokens (integer work, bit-exact) -------------- */
/*
 * Per window w: slice [w0,w1) of the chromosome starting at genome + win_base[w], apply the sample's
 * variants var_lo[w]..var_hi[w] (sorted by position; gt 0 skip / 1 het / 2 hom-alt): het SNP -> IUPAC code,
 * hom SNP -> ALT, indel/MNP -> REF span replaced by ALT, overlapping or window-straddling records skipped;
 * flags bit0 = reverse-complement the result, bit1 = SNP-only filter.
 * out: uint8 [n_win, pitch]; out_len int32 [n_win]; err: device int32 flag (1 pitch overflow, 2 >2048 records;
 * vf_encode_windows_edits also 4: a row's extra records are not sorted by pos; vf_encode_windows_overrides also 8: a
 * row's override list is malformed).
 * Any n_win: batches of more than 65535 windows are launched in chunks of 65535.
 * Replaces the `samtools faidx | bcftools consensus -H I -e 'ALT~"<.*>"'` subprocess pair per window
 * (utils/data_process.py:17-101, :367-467) and utils/functions.py:129-172 (reverse_complement).
 */
int vf_encode_windows(const uint8_t* genome, const int64_t* win_base, const int32_t* w0, const int32_t* w1,
                      const int32_t* var_lo, const int32_t* var_hi, const uint8_t* flags, const int32_t* v_pos,
                      const int32_t* v_ref_len, const int32_t* v_alt_off, const int32_t* v_alt_len, const uint8_t* v_gt,
                      const uint8_t* alt_pool, int n_win, int max_window, uint8_t* out, int64_t pitch, int32_t* out_len,
                      int32_t* err, void* stream);
/*
 * vf_encode_windows with ONE extra record per row (in-silico deletions, variant edits against a sample background): row w
 * is encoded as vf_encode_windows encodes it on the table with the record {pos e_pos[w], ref_len e_ref_len[w], ALT
 * e_alt_pool[e_alt_off[w], + e_alt_len[w]), gt 2 (hom-alt)} inserted into [var_lo[w], var_hi[w]) right after every record
 * with pos <= e_pos[w], bit for bit: the same rule decides, in the same kernel body, whether it applies.  The extra
 * record counts toward the 2048-record cap.  applied uint8 [n_win] = 1 iff row w's extra record was applied (it then
 * lies in [w0, w1), no earlier applied record overlaps its position and it is not dropped by the SNP-only filter).
 * Other arguments, outputs and errors as vf_encode_windows; n_win < 0 or a NULL array fails before any launch.
 */
int vf_encode_windows_edit(const uint8_t* genome, const int64_t* win_base, const int32_t* w0, const int32_t* w1,
                           const int32_t* var_lo, const int32_t* var_hi, const uint8_t* flags, const int32_t* v_pos,
                           const int32_t* v_ref_len, const int32_t* v_alt_off, const int32_t* v_alt_len,
                           const uint8_t* v_gt, const uint8_t* alt_pool, const int32_t* e_pos, const int32_t* e_ref_len,
                           const int32_t* e_alt_off, const int32_t* e_alt_len, const uint8_t* e_alt_pool, int n_win,
                           int max_window, uint8_t* out, int64_t pitch, int32_t* out_len, uint8_t* applied,
                           int32_t* err, void* stream);
/*
 * vf_encode_windows with a LIST of extra records per row (variant sets: haplotypes, pairs, edits against a sample
 * background), in CSR form: row w owns the records [e_off[w], e_off[w + 1]) (e_off int32 [n_win + 1], nondecreasing,
 * ranges disjoint), each {pos e_pos, ref_len e_ref_len, ALT e_alt_pool[e_alt_off, + e_alt_len), gt e_gt (0 skip, 1 het,
 * 2 hom-alt)}, sorted by pos within the row.  Row w is encoded as vf_encode_windows encodes it on the table with each of
 * its records inserted right after every background record with pos <= its own (records of one pos in list order), bit
 * for bit, in the same kernel body.  Extras count toward the 2048-record cap.  applied uint8 [e_off[n_win]] = 1 iff that
 * extra record was applied.  A row whose records are not sorted by pos sets *err to 4 and writes length 0.
 * vf_encode_windows_edit is the one-record case: row w's list is record w, gt 2.  Other arguments, outputs and errors
 * as vf_encode_windows; n_win < 0 or a NULL array fails before any launch.
 */
int vf_encode_windows_edits(const uint8_t* genome, const int64_t* win_base, const int32_t* w0, const int32_t* w1,
                            const int32_t* var_lo, const int32_t* var_hi, const uint8_t* flags, const int32_t* v_pos,
                            const int32_t* v_ref_len, const int32_t* v_alt_off, const int32_t* v_alt_len,
                            const uint8_t* v_gt, const uint8_t* alt_pool, const int32_t* e_off, const int32_t* e_pos,
                            const int32_t* e_ref_len, const int32_t* e_alt_off, const int32_t* e_alt_len,
                            const uint8_t* e_gt, const uint8_t* e_alt_pool, int n_win, int max_window, uint8_t* out,
                            int64_t pitch, int32_t* out_len, uint8_t* applied, int32_t* err, void* stream);
/*
 * vf_encode_windows with a list of GENOTYPE OVERRIDES per row (variant attribution: the sample's own records removed or
 * re-genotyped), in CSR form: row w owns the overrides [o_off[w], o_off[w + 1]) (o_off int32 [n_win + 1],
 * nondecreasing), each {record o_idx (an index into the variant table), new gt o_gt (0 removed, 1 het, 2 hom-alt)},
 * indices strictly increasing within the row and inside [var_lo[w], var_hi[w]).  Row w is encoded as vf_encode_windows
 * encodes it on the table with those records' gts replaced, bit for bit, in the same kernel body (gt 0 is the line
 * removed: the encoder skips gt 0 records).  A row whose indices are unsorted, repeated or outside its range sets *err to
 * 8 and writes length 0; other rows are not affected.  Other arguments, outputs and errors as vf_encode_windows;
 * n_win < 0 or a NULL array fails before any launch.
 */
int vf_encode_windows_overrides(const uint8_t* genome, const int64_t* win_base, const int32_t* w0, const int32_t* w1,
                                const int32_t* var_lo, const int32_t* var_hi, const uint8_t* flags, const int32_t* v_pos,
                                const int32_t* v_ref_len, const int32_t* v_alt_off, const int32_t* v_alt_len,
                                const uint8_t* v_gt, const uint8_t* alt_pool, const int32_t* o_off, const int32_t* o_idx,
                                const uint8_t* o_gt, int n_win, int max_window, uint8_t* out, int64_t pitch,
                                int32_t* out_len, int32_t* err, void* stream);
/*
 * Which rows of a cohort encode to the same bytes.  Row r = one (window, sample): w0/w1/flags/var_lo/var_hi as in
 * vf_encode_windows (flags bit1 = SNP-only), the variant arrays those of vf_encode_windows (one concatenated table may
 * hold every sample's records; each row's [var_lo, var_hi) points at its sample's).  The applied records of a row are
 * selected with exactly vf_encode_windows' rule (one device function serves both).
 * vf_window_genotype_keys: keys uint64 [n_rows, 2] = a 128-bit hash of the applied records' (pos, ref_len, gt, alt_len,
 *   ALT bytes), 0 for a row with none (the reference window); count int32 [n_rows] = the number applied, or -1 where a
 *   2049th record would apply: such a row sets *err to 2, exactly where vf_encode_windows does; out_len int32
 *   [n_rows] or NULL = the length vf_encode_windows gives the row, (w1 - w0) + sum(alt_len - ref_len) over the applied
 *   records (over the first 2048 on a capped row): the row overflows a pitch iff out_len > pitch.
 * vf_window_genotype_equal: equal int32 [n_rows] = 1 iff row r and row rep[r] (same w0, w1, flags bits 0-1) apply equal
 *   record lists, element by element; rows of equal lists encode to identical bytes.
 * One thread per row; any n_rows >= 0; NULL arrays for n_rows > 0 fail before any launch.
 */
int vf_window_genotype_keys(const int32_t* w0, const int32_t* w1, const int32_t* var_lo, const int32_t* var_hi,
                            const uint8_t* flags, const int32_t* v_pos, const int32_t* v_ref_len, const int32_t* v_alt_off,
                            const int32_t* v_alt_len, const uint8_t* v_gt, const uint8_t* alt_pool, int n_rows,
                            unsigned long long* keys, int32_t* count, int32_t* out_len, int32_t* err, void* stream);
int vf_window_genotype_equal(const int32_t* w0, const int32_t* w1, const int32_t* var_lo, const int32_t* var_hi,
                             const uint8_t* flags, const int32_t* v_pos, const int32_t* v_ref_len, const int32_t* v_alt_off,
                             const int32_t* v_alt_len, const uint8_t* v_gt, const uint8_t* alt_pool, int n_rows,
                             const int32_t* rep, int32_t* equal, void* stream);
/*
 * The same keys and comparison for rows with a list of extra records (variant sets across a cohort), the records in the
 * CSR form of vf_encode_windows_edits (e_off int32 [n_rows + 1], e_pos, e_ref_len, e_alt_off, e_alt_len, e_gt, e_alt_pool):
 * a row's applied list is what vf_encode_windows_edits applies for it, background and extra records merged by the same
 * device walk.  The hash and the comparison read record content only, so a row whose extras are all blocked keys and
 * compares equal to its window without them, and a row with no extras gets vf_window_genotype_keys' key, count and
 * out_len bit for bit.  vf_window_genotype_keys_edits also writes applied uint8 [e_off[n_rows]], equal to what
 * vf_encode_windows_edits writes for the row.  A row whose extras are not sorted by pos sets *err to 4, count -1 and
 * out_len 0, and compares equal to no other row.  Other arguments, outputs and errors as vf_window_genotype_keys /
 * vf_window_genotype_equal; n_rows < 0 or a NULL array fails before any launch.
 */
int vf_window_genotype_keys_edits(const int32_t* w0, const int32_t* w1, const int32_t* var_lo, const int32_t* var_hi,
                                  const uint8_t* flags, const int32_t* v_pos, const int32_t* v_ref_len,
                                  const int32_t* v_alt_off, const int32_t* v_alt_len, const uint8_t* v_gt,
                                  const uint8_t* alt_pool, const int32_t* e_off, const int32_t* e_pos,
                                  const int32_t* e_ref_len, const int32_t* e_alt_off, const int32_t* e_alt_len,
                                  const uint8_t* e_gt, const uint8_t* e_alt_pool, int n_rows, unsigned long long* keys,
                                  int32_t* count, int32_t* out_len, uint8_t* applied, int32_t* err, void* stream);
int vf_window_genotype_equal_edits(const int32_t* w0, const int32_t* w1, const int32_t* var_lo, const int32_t* var_hi,
                                   const uint8_t* flags, const int32_t* v_pos, const int32_t* v_ref_len,
                                   const int32_t* v_alt_off, const int32_t* v_alt_len, const uint8_t* v_gt,
                                   const uint8_t* alt_pool, const int32_t* e_off, const int32_t* e_pos,
                                   const int32_t* e_ref_len, const int32_t* e_alt_off, const int32_t* e_alt_len,
                                   const uint8_t* e_gt, const uint8_t* e_alt_pool, int n_rows, const int32_t* rep,
                                   int32_t* equal, void* stream);
/*
 * Single-base substitution of encoded windows (in-silico saturation mutagenesis): row r of out = the source row
 * src[row_src[r]] (src_len[row_src[r]] bytes, as vf_encode_windows wrote it) with ONE base replaced by row_base[r].
 * row_off[r] = forward-strand offset pos0 - w0 of the base; flags[r] bit0 = the source was reverse-complemented: the base
 * goes to len - 1 - row_off[r] as its IUPAC complement (the table vf_encode_windows applies).  The caller passes the
 * base of the datasets/vepdataset.py:94-131 rule: the ALT base (hom) or get_iupac_code(ref, alt) (het).
 * out: uint8 [n_rows, out_pitch]; out_len int32 [n_rows]; err: device int32 flag (1 row longer than a pitch, 3 offset
 * outside the row; such a row gets length 0).  Pitches: multiples of 16, rows 16-byte aligned; any n_rows.
 * The rows then go through vf_bpe_tokenize like any encoded window.  Same kernel as vf_splice_windows with k = 1.
 */
int vf_mutate_windows(const uint8_t* src, int64_t src_pitch, const int32_t* src_len, const int32_t* row_src,
                      const int32_t* row_off, const uint8_t* row_base, const uint8_t* flags, int n_rows, uint8_t* out,
                      int64_t out_pitch, int32_t* out_len, int32_t* err, void* stream);
/*
 * Allele splice of encoded windows (variant tables): row r of out = the source row src[row_src[r]] with the ONE base at
 * forward-strand offset row_off[r] replaced by the k = allele_len[r] >= 0 bytes allele_pool[allele_off[r], + k) (a
 * multi-base allele is an insertion, an empty one deletes the base; nothing else is deleted: the
 * datasets/vepdataset.py:94-131 rule).  flags[r] bit0 = the
 * source was reverse-complemented: the reverse complement of the allele (vf_encode_windows' table) replaces the byte at
 * len - 1 - row_off[r].  out_len[r] = len + k - 1.  allele_off == allele_len == NULL: row r's allele is allele_pool[r],
 * k = 1 (vf_mutate_windows).  err: device int32 flag (1 output row longer than out_pitch, 3 offset outside the row or
 * k < 0; such a row gets length 0).  Pitches: multiples of 16, rows 16-byte aligned; any n_rows (launched in chunks of
 * 65535).
 */
int vf_splice_windows(const uint8_t* src, int64_t src_pitch, const int32_t* src_len, const int32_t* row_src,
                      const int32_t* row_off, const uint8_t* allele_pool, const int32_t* allele_off,
                      const int32_t* allele_len, const uint8_t* flags, int n_rows, uint8_t* out, int64_t out_pitch,
                      int32_t* out_len, int32_t* err, void* stream);
/*
 * BPE tokenisation of n_win byte sequences (upper-cased; non-IUPAC characters split words).
 * merge_a/merge_b/merge_new: uint16 [n_merges] rank-ordered merge table.  merge_batch: uint16 [n_merges] nondecreasing
 * batch ids, or NULL: consecutive ranks with one id are applied in a single sweep with a single barrier — legal when
 * their {left, right, new} symbol sets are pairwise disjoint and none is a self pair (such merges commute);
 * at most 16 ranks per batch; NULL = every rank alone (same tokens, three times the barriers).  out_tokens int32 [n_win, out_pitch]:
 * the first min(count, out_cap) ids, remainder of the row zero (<pad>); out_count int32 [n_win] = untruncated
 * token count; out_start (optional) int32 [n_win, start_pitch] = first base index of every token.
 * Windows longer than 8192 symbols run on the cluster/DSMEM kernel (8 CTAs per window); scratch is unused there.
 * block_threads: 0 = auto, or 128/256/512/1024 (performance hint for the single-CTA kernel).
 * Replaces utils/seq.py:32-62 (BPEEncoder.normalize/encode -> HF tokenizers), :68-174 (token offsets) and the
 * pad/truncate/chunk steps datasets/vcfdataset.py:198-217, :338-394.
 */
int vf_bpe_tokenize(const uint8_t* seq, int64_t pitch, const int32_t* len, int n_win, int max_len,
                    const uint16_t* merge_a, const uint16_t* merge_b, const uint16_t* merge_new,
                    const uint16_t* merge_batch, int n_merges, uint16_t* scratch, int64_t scratch_pitch, int32_t* out_tokens, int out_pitch, int out_cap,
                    int32_t* out_count, int32_t* out_start, int64_t start_pitch, int block_threads, void* stream);

/* ---- coarse entry points: whole-module forwards, layer loop inside the library ---------------------------------- */
/*
 * Weight-pointer tables.  Every pointer is a DEVICE pointer; the tables themselves (and the per-layer arrays they point
 * to) live in HOST memory and are only read during the call.  A linear is {w bf16 [N, K] (nn.Linear layout), b fp32 [N],
 * cs fp32 [N] or NULL}: with cs != NULL the LayerNorm in front of the Linear is folded in — w = bf16(W * gamma),
 * b = bias + W beta, cs = row sums of that bf16 w (vf_gemm_bf16_ln).  linear_geglu_1 (w, b, cs) is tile-interleaved as
 * VF_EPI_BIAS_GEGLU_BF16 wants it.  variantformer_b200/engine.py builds exactly these tables from a reference state_dict.
 */
typedef struct { const void* w; const float* b; const float* cs; } vf_linear_t;

/* seq2reg/modules.py:129-147: qkv = Wqkv(norm1 folded), out = out_proj, g1 = linear_geglu_1(norm2 folded), g2 = linear_geglu_2 */
typedef struct { vf_linear_t qkv, out, g1, g2; } vf_seq2reg_layer_t;
typedef struct {
    int d, heads, n_layers, ffn_hidden, token_length;   /* 512, 8, 6, 2048, 200 for the configured tokenizers */
    float ln_eps;
    const float* emb;                                   /* fp32 [vocab, d]           seq2reg/model.py:214 */
    const float* pe;                                    /* fp32 [token_length, d] or NULL (ALiBi)   :15-37, :219-220 */
    const float* slopes;                                /* fp32 [heads] ALiBi slopes or NULL */
    const vf_seq2reg_layer_t* layers;                   /* host array [n_layers] */
} vf_seq2reg_weights_t;

/*
 * Seq2RegPredictor.forward(only_embed=True) for n_win windows (seq2reg/model.py:193-279, seq2reg/modules.py:149-191):
 * tokens int32 [n_win, L], pad_mask uint8 [n_win, L] (1 = padding), cu int32 [n_win + 1] prefix sums of the valid
 * counts, n_tok = cu[n_win]; slots / n_items = attention work table of the windows' valid lengths
 * (vf_attention_build_slots); workspace: caller-owned device memory of vf_seq2reg_workspace_bytes(w, n_tok) bytes,
 * 256-byte aligned.  out_bf16 [n_win, d] = mean over each window's valid tokens of the last layer (NaN for an empty
 * window, as upstream).
 */
size_t vf_seq2reg_workspace_bytes(const vf_seq2reg_weights_t* w, int64_t n_tok);
int vf_seq2reg_forward(const vf_seq2reg_weights_t* w, const int32_t* tokens, const uint8_t* pad_mask, const int32_t* cu,
                       int n_win, int L, int64_t n_tok, const int32_t* slots, int n_items, void* workspace,
                       size_t workspace_bytes, void* out_bf16, void* stream);

/* layers.py:47-86: qkv = mixer Wqkv(norm1), out = mixer out_proj, q = crossMHA Wq(norm2), kv = crossMHA Wkv (plain; w NULL
 * for a CRE layer), out2 = crossMHA out_proj, g1 = linear_geglu_1(norm3), g2 = linear_geglu_2; kv9 fp32 [9, 2D] =
 * Wkv Emb9 + b of a CRE layer (vf_label_attention), NULL for a gene layer. */
typedef struct { vf_linear_t qkv, out, q, kv, out2, g1, g2; const float* kv9; } vf_context_layer_t;
typedef struct {
    int D, heads, n_layers, ffn_hidden, token_dim;      /* 1536, 32, 25, 2048, 512 */
    float ln_eps;
    const float* slopes;                                /* fp32 [heads] ALiBi slopes (self-attention) or NULL */
    const float* registry;                              /* fp32 [num_tissues, D]  start_tkn.registry_tokens (layers.py:508-521) */
    vf_linear_t cre_map, gene_map;                      /* model_combined_modulator.py:502-507 (plain linears) */
    const vf_context_layer_t* cre_layers;               /* host array [n_layers - 1] */
    const vf_context_layer_t* gene_layers;              /* host array [n_layers] */
    vf_linear_t h0, h4;                                 /* tissue_heads.tissue_expressions.0 / .4 (layers.py:1078-1087) */
    const float* hn_g; const float* hn_b;               /* ... .1 LayerNorm */
    const float* h6_w; const float* h6_b;               /* ... .6 Linear(D, 1) */
} vf_seq2gene_weights_t;
/*
 * Index tables of one slab of genes (device pointers, built by the caller: engine.py:Engine.prepare is the reference
 * builder).  Gene-stream rows: per gene, per tissue: [registry(tissue); chunk_0 .. chunk_{G-1}], tissues of a gene
 * contiguous.  n_reg = sum of tissues over the slab's genes = number of predictions.
 */
typedef struct {
    int n_cre, n_gene_chunks, n_gene_rows, n_reg, n_need;
    int single_stream;              /* != 0: CRE stack on the caller's stream (profiling); 0: on the library's side stream */
    const int32_t* gene_idx;        /* [n_gene_rows]: >= 0 row of gene_map's output, < 0 registry token -(tissue + 1) */
    const int32_t* row_seq;         /* [n_cre] gene of every CRE row */
    const float* logc;              /* [genes, 9] log(#CREs of the class in the gene), -inf when absent */
    const int32_t* last_rows;       /* [n_need] rows whose last-layer output is read: the n_reg registry rows first */
    const int32_t* cre_pos_idx;     /* [n_reg] CRE row per prediction (VEP token gather) or NULL */
    const int32_t* slots_gself; int n_gself;            /* work tables (vf_attention_build_slots layout): gene self, */
    const int32_t* slots_gcross; int n_gcross;          /* stacked gene -> CRE cross (queries: all tissue copies of a gene), */
    const int32_t* slots_cself; int n_cself;            /* CRE self, */
    const int32_t* slots_last_self; int n_last_self;    /* last layer: one-row query tiles against their own sequence, */
    const int32_t* slots_last_cross; int n_last_cross;  /* last layer: runs of one gene's needed rows against its CREs */
} vf_seq2gene_slab_t;
/*
 * cre_map / gene_map, registry-token assembly, CombinedModulator, pool_outputs and the expression head for one slab
 * (model_combined_modulator.py:137-328, 540-720; layers.py:88-165, 508-521, 1078-1144).  cre_pooled_bf16 [n_cre,
 * token_dim] / gene_pooled_bf16 [n_gene_chunks, token_dim]: outputs of vf_seq2reg_forward.  pred fp32 [n_reg]
 * (Softplus applied), emb fp32 [n_reg, D]; gene_token_emb fp32 [n_need - n_reg, D] and cre_token_emb fp32 [n_reg, D]
 * may be NULL.  The CRE stack runs on a side stream owned by the library (one forward in flight per device).
 */
/*
 * Rows of the final CRE stream of the forward that just ran (CRE-token embeddings of arbitrary rows, e.g. several per
 * prediction in a slab whose items share windows): out_f32 [n, D] = raw (un-centred) value of CRE row rows[r] of the
 * slab, the same gather + un-centring as cre_token_emb.  PRECONDITION: called on the same stream right after
 * vf_seq2gene_forward with the same weight table, slab and workspace (untouched in between): it reads the stream that
 * call left in the workspace.  rows int32 [n], each in [0, n_cre).
 */
int vf_seq2gene_cre_rows(const vf_seq2gene_weights_t* w, const vf_seq2gene_slab_t* slab, void* workspace,
                         size_t workspace_bytes, const int32_t* rows, int n, float* out_f32, void* stream);
size_t vf_seq2gene_workspace_bytes(const vf_seq2gene_weights_t* w, const vf_seq2gene_slab_t* slab);
int vf_seq2gene_forward(const vf_seq2gene_weights_t* w, const vf_seq2gene_slab_t* slab, const void* cre_pooled_bf16,
                        const void* gene_pooled_bf16, void* workspace, size_t workspace_bytes, float* pred, float* emb,
                        float* gene_token_emb, float* cre_token_emb, void* stream);
/*
 * Gene -> CRE cross-attention maps of one slab (vf_cross_attention_probs layout): one group per gene, its predictions'
 * registry rows as queries, its CREs as keys.  group_q int32 [n_groups][2] = {first prediction, predictions} (index
 * into the n_reg predictions / the registry rows of the slab, in gene-stream order); group_k int32 [n_groups][2] =
 * {first CRE row, CREs}; reg_rows int32 [n_reg] = gene-stream row of every prediction's registry token; out fp32,
 * out_off int64 [n_reg] = start of each prediction's [n_layers, heads, CREs] block.
 */
typedef struct {
    int n_groups;
    const int32_t* group_q;
    const int32_t* group_k;
    const int32_t* reg_rows;
    float* out;
    const int64_t* out_off;
} vf_cre_attention_t;
/*
 * vf_seq2gene_forward that also writes the maps: after the cross-attention of every gene layer, on the caller's stream,
 * one vf_cross_attention_probs launch on the layer's queries (the registry rows of the query buffer; the pruned last
 * layer's query rows, whose first n_reg are the registry rows).  Same workspace, same launches otherwise: pred, emb and
 * the token embeddings are bit-identical to vf_seq2gene_forward.  attn NULL = vf_seq2gene_forward.
 */
int vf_seq2gene_forward_attn(const vf_seq2gene_weights_t* w, const vf_seq2gene_slab_t* slab, const void* cre_pooled_bf16,
                             const void* gene_pooled_bf16, void* workspace, size_t workspace_bytes, float* pred, float* emb,
                             float* gene_token_emb, float* cre_token_emb, const vf_cre_attention_t* attn, void* stream);
/*
 * HOST helper: work table of vf_attention_mc_varlen for n_seq sequences of q_lens query rows and k_lens keys (NULL =
 * self-attention), rows packed back to back.  out_table: HOST int32 [max_items][2][8] (NULL: only count).  Consecutive
 * 128-row tiles of a sequence share an item; left-over tiles are paired with each other when pair_unrelated != 0.
 * Returns the number of items (>= 0) or a negative error.  Same tables as variantformer_b200.ops.SlotMap.
 */
int vf_attention_build_slots(const int32_t* q_lens, const int32_t* k_lens, int n_seq, int pair_unrelated,
                             int32_t* out_table, int max_items);

#ifdef __cplusplus
}
#endif
#endif /* VF_B200_H */
