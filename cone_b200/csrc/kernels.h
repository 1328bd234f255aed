// Internal launcher declarations shared by the .cu files of libcone_b200.
#pragma once
#include "common.cuh"

namespace cone {

// bytes per element of a raw feature tensor of dtype CONE_DTYPE_*; 0 = unknown code
inline size_t feature_elem_bytes(int dtype) {
    return dtype == CONE_DTYPE_F32 ? 4 : (dtype == CONE_DTYPE_F16 || dtype == CONE_DTYPE_BF16) ? 2 : 0;
}

// ---------------------------------------------------------------- gemm_simt.cu
// C[M,N] = epi(A[M,K] * W[N,K]^T): both operands K-major (row-major activations x nn.Linear weight).
struct GemmParams {
    const float* A = nullptr;
    int64_t lda = 0;
    const float* W = nullptr;
    int64_t ldw = 0;
    float* C = nullptr;
    int64_t ldc = 0;
    const float* bias = nullptr;  // [N] or null
    const float* R = nullptr;     // residual [M,N] or null, added after bias, before relu
    int64_t ldr = 0;
    int64_t M = 0;
    int N = 0, K = 0;
    int relu = 0;
};
int sgemm_nt(const GemmParams& p, cudaStream_t s);

// Grouped frame-score GEMM: for video v, C_v[q, f] = cls[q] . ctx[f]   (q in the video's queries)
int sgemm_frame_scores(const float* ctx, const float* cls, int K, const int64_t* video_offsets, const int32_t* q_first,
                       int n_videos, int max_video_frames, int max_video_queries, float* score,
                       const int64_t* score_offsets, cudaStream_t s);

// out[row, n] = epi(x[row,:K] . W[n,:K] + bias[n]) for tiny N (<= 8). mode: 0 none, 1 sigmoid,
// 2 "softmax over the N outputs, write element 0 only" (out has 1 column), 3 softmax all
// group_out/group_in > 0 remap rows: output row r reads input row (r / group_out) * group_in + r % group_out
int rowdot_small(const float* x, int64_t ldx, const float* W, const float* bias, float* out, int64_t rows, int N, int K,
                 int mode, cudaStream_t s, int group_out = 0, int group_in = 0);

// ---------------------------------------------------------------- rowops.cu
// x_dtype (CONE_DTYPE_*) is the element type of the raw rows x; residual, gamma, beta and out are fp32
int layernorm_rows(const void* x, int x_dtype, const float* residual, const float* gamma, const float* beta, float* out,
                   int64_t rows, int D, float eps, cudaStream_t s);
inline int layernorm_rows(const float* x, const float* residual, const float* gamma, const float* beta, float* out,
                          int64_t rows, int D, float eps, cudaStream_t s) {
    return layernorm_rows(x, CONE_DTYPE_F32, residual, gamma, beta, out, rows, D, eps, s);
}
int l2norm_rows(const void* x, int x_dtype, float* out, int64_t rows, int D, float eps, cudaStream_t s);
inline int l2norm_rows(const float* x, float* out, int64_t rows, int D, float eps, cudaStream_t s) {
    return l2norm_rows(x, CONE_DTYPE_F32, out, rows, D, eps, s);
}
int build_pos_table(float* table, int max_v_l, int d, cudaStream_t s);  // [max_v_l+1, max_v_l, d]
// window rows: src[b*S + r] = r < Lv ? vidproj[min(vid_base[b]+r, n_vid_rows-1)] : txtproj[txt_base[b] + r - Lv]
int gather_window_rows(const float* vidproj, int64_t n_vid_rows, const int64_t* vid_base, const float* txtproj,
                       const int64_t* txt_base, float* src, int64_t B, int Lv, int Lt, int d, cudaStream_t s);
// out[b*S + r] = src[b*S + r] + (r < Lv ? pos[vlen[b]][r] : 0)
int add_pos_rows(const float* src, const float* pos_table, const int32_t* vlen, float* out, int64_t B, int Lv, int Lt,
                 int d, int table_lv, cudaStream_t s);
int gather_window_rows_f16(const float* vidproj, int64_t n_vid_rows, const int64_t* vid_base, const float* txtproj,
                           const int64_t* txt_base, uint16_t* src16, int64_t B, int Lv, int Lt, int d, cudaStream_t s,
                           uint16_t* src16lo = nullptr);  // src16lo (nullable): fp16(value - fp16(value))
// hi = fp16(x), lo = fp16(x - hi) (lo nullable) over n contiguous elements; and out = hi + lo
int split_hilo_rows(const float* x, uint16_t* hi, uint16_t* lo, int64_t n, cudaStream_t s);
int combine_hilo_rows(const uint16_t* hi, const uint16_t* lo, float* out, int64_t n, cudaStream_t s);
// same gather from fp16 source rows (bit-identical to rounding the fp32 rows)
int gather_window_rows_h2h(const uint16_t* vid16, int64_t n_vid_rows, const int64_t* vid_base, const uint16_t* txt16,
                           const int64_t* txt_base, uint16_t* src16, int64_t B, int Lv, int Lt, int d, cudaStream_t s);
// fp16 operands for the tensor-core path: plain16 = fp16(src), pos16 = fp16(src + pos); either may be null
int add_pos_rows_f16(const float* src, const float* pos_table, const int32_t* vlen, uint16_t* plain16, uint16_t* pos16,
                     int64_t B, int Lv, int Lt, int d, int table_lv, cudaStream_t s);
// out[row] = x[row] + table[row % period]   (x may be null = zeros)
int add_row_table(const float* x, const float* table, float* out, int64_t rows, int period, int d, cudaStream_t s);
// same, rounded to fp16 (GEMM operand of the tensor-core decoder chain)
int add_row_table_f16(const float* x, const float* table, uint16_t* out16, int64_t rows, int period, int d, cudaStream_t s);
int fill_window_desc_dense(int64_t* vid_base, int64_t* txt_base, int32_t* qidx, int64_t B, int Lv, int Lt,
                           cudaStream_t s);
int fill_i32(int32_t* p, int64_t n, int32_t value, cudaStream_t s);

// ---------------------------------------------------------------- attention.cu
// encoder self-attention over S = Lv+Lt rows per window, head_dim 32
int enc_self_attention(const float* qk, int64_t ldqk, const float* v, int64_t ldv, float* o, int64_t ldo,
                       const int32_t* vlen, const int32_t* tlen, int64_t B, int Lv, int Lt, int nheads,
                       cudaStream_t s);
// tensor-core variant: fp16 q|k [R, ldqk], v, o (passed as void* to keep cuda_fp16.h out of this header)
// posqk (nullable): per-layer table [(table_lv+1)*table_lv, 2*d] = pos . [Wq; Wk]^T added to q | k of video rows
int enc_self_attention_f16(const void* qk, int64_t ldqk, const void* v, int64_t ldv, void* o, int64_t ldo,
                           const int32_t* vlen, const int32_t* tlen, int64_t B, int Lv, int Lt, int nheads,
                           const void* posqk16, int table_lv, cudaStream_t s, const void* frame_qkv = nullptr,
                           const void* token_qkv = nullptr, const int64_t* vid_base = nullptr,
                           const int64_t* txt_base = nullptr, int64_t n_frames = 0);
// tcgen05 version (enc_attn_tc.cu): qkv = dense window rows [B S, 768] (token_qkv null) or the per-frame rows [rows, 768] with
// token_qkv [n_tok, 768] and the window descriptors; posqk16 = fp16 copy of the position-projection table
bool enc_attn_tc_supported(int Lv, int Lt, int d_model, int nheads);
int enc_attn_tc_run(const void* qkv, int64_t rows, void* o, int64_t ldo, const int32_t* vlen, const int32_t* tlen, int64_t B, int Lv,
                    int Lt, const void* posqk16, int table_lv, const void* token_qkv, int64_t n_tok, const int64_t* vid_base,
                    const int64_t* txt_base, int num_sms, cudaStream_t s);
// frame_qkv / token_qkv (nullable): fp16 q|k|v rows [n, 3 d] of every frame / token; window row r then reads
// frame vid_base[b] + r (r < Lv) or token txt_base[b] + r - Lv instead of qk / v
// decoder self-attention over nq slots (no mask)
// qk / v / o are fp32 (f16 = 0) or fp16 (f16 = 1)
int dec_self_attention(const void* qk, int64_t ldqk, const void* v, int64_t ldv, void* o, int64_t ldo, int64_t B,
                       int nq, int nheads, int f16, cudaStream_t s);
// decoder cross-attention of the fp32 mode: nq queries x S memory keys with key-padding mask, fp32 q / k / v / o
// (kv_f16 must be 0: the tensor-core decoder uses dec_cross_attention_mem below)
int dec_cross_attention(const void* q, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv,
                        void* o, int64_t ldo, const int32_t* vlen, const int32_t* tlen, int64_t B, int nq, int Lv,
                        int Lt, int nheads, int kv_f16, const void* posk, int64_t ldposk, int table_lv,
                        cudaStream_t s);  // posk: fp32 table (kv_f16 = 0) or fp16 table (kv_f16 = 1), or null

// memory-direct cross-attention of the tensor-core decoder: mem [B S, 256] fp16 raw encoder output, qqt [B nq, 9 * 256] fp16
// = q (softmax scale folded in) | q pushed through Wk_h^T per head; pm [B nq, 8 * 256] fp16 = per-head attention-pooled
// memory (Wv and the output projection are applied by the next GEMM); posk = fp16 pos.Wk^T table
int dec_cross_attention_mem(const void* mem, int64_t ldm, const void* qqt, int64_t ldq, void* pm, int64_t ldp,
                            const int32_t* vlen, const int32_t* tlen, int64_t B, int nq, int Lv, int Lt, const void* posk,
                            int64_t ldposk, int table_lv, cudaStream_t s, int q_bcast = 0);
// q_bcast = 1: the queries are the same for every window (decoder layer 0: tgt starts at zero) — qqt holds nq rows

// ---------------------------------------------------------------- prefilter.cu
int window_ranklist(const float* frame_score, const int64_t* score_offsets, const int32_t* frame_count, int n_queries,
                    int max_v_l, int32_t* ranklist, float* winscore, int ranklist_stride, cudaStream_t s);
// window descriptors of the first `topk` ranked windows of each query
int prefilter_desc(int64_t* video_offsets, int32_t* q_first, int64_t* score_offsets, int32_t* frame_count, int64_t L,
                   int n_queries, cudaStream_t s);
int take_topk(const int32_t* ranklist, const float* winscore, int ranklist_stride, int n_queries, int topk, int32_t* win_idx,
              float* win_score, cudaStream_t s);
int build_windows(const int32_t* ranklist, int ranklist_stride, const int32_t* q_video_len, int n_queries, int topk,
                  int max_v_l, int32_t* win_start, int32_t* win_len, cudaStream_t s);
int batch_max_len(const int32_t* win_len, const int32_t* q_batch, int n_queries, int topk, int32_t* batch_max,
                  int n_batches, cudaStream_t s);
// per-chunk descriptors for queries [q0, q0+nq)
int fill_window_desc_chunk(const int64_t* q_video_start, const int32_t* win_start, const int32_t* win_len,
                           const int32_t* tok_len, const int32_t* q_batch, const int32_t* batch_max, int q0, int nqc,
                           int topk, int Lt, int fixed_pad, int64_t* vid_base, int32_t* vlen, int64_t* txt_base,
                           int32_t* tlen, int32_t* pad_len, int32_t* qidx, cudaStream_t s);  // q_batch null: pad_len = fixed_pad

// ---------------------------------------------------------------- pool_match.cu
// pooled[(b*nq+j), :] = mean of zero-padded window rows [start, min(end, pad_len)) (model.py:186-200)
// frames_dtype (CONE_DTYPE_*): element type of the raw rows; pooled is fp32
int span_mean_pool(const void* frames, int frames_dtype, int64_t n_frames, const int64_t* vid_base, const int32_t* vlen,
                   const int32_t* pad_len, const float* spans, float* pooled, int64_t B, int nq, int Dv,
                   cudaStream_t s);
// out[b*nq+j] = (p / ||p||) . t[qidx[b]]
int norm_dot(const float* p, const float* t, const int32_t* qidx, float* out, int64_t B, int nq, int Dv,
             cudaStream_t s);

// ---------------------------------------------------------------- fuse_nms.cu
int fuse_nms(const float* pred_spans, const float* prob_fg, const float* match, const int32_t* win_start,
             const int32_t* win_len, int n_queries, int topk, int nq, float clip_length, double nms_thd,
             int max_before_nms, int max_after_nms, double* out, int32_t* out_count, double* rows_out,
             int32_t* rows_count, cudaStream_t s, int fixed_duration = 0, int sort_windows = 1);
int temporal_nms_single(const double* st, const double* ed, const double* score, int n, double nms_thd,
                        int max_after_nms, int32_t* keep_out, int32_t* n_keep_out, cudaStream_t s);


// ---------------------------------------------------------------- eval.cu
// R@K / IoU hit counters from the stage-3 output (flavour 0: evaluate_mad.py, 1: evaluate_ego4d_nlq.py); topk / thr are
// HOST arrays; hits [3, n_topk, n_thr] int64 is ACCUMULATED into; top1_iou (nullable) [n_queries, 3] fp64
int eval_recall(const double* nms, const int32_t* nms_count, const double* gt, int n_queries, int max_after,
                const int32_t* topk_host, int n_topk, const double* thr_host, int n_thr, int flavour, int64_t* hits,
                double* top1_iou, cudaStream_t s);
// window pre-filtering recall (evaluate_pre_filtered_window.py); hits [n_topk] int64 is accumulated into
int eval_window_recall(const int32_t* ranklist, int ranklist_stride, const double* gt, int n_queries, double clip_length,
                       int max_v_l, const int32_t* topk_host, int n_topk, int64_t* hits, cudaStream_t s);

}  // namespace cone
