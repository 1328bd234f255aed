/*
 * cone_b200.h — C ABI of the B200-native CONE coarse-to-fine inference path.
 *
 * The reference (houzhijian/CONE) is pure Python/PyTorch and has no FFI layer; its "operator
 * surface" is the set of Python call sites in cone/inference.py (SURVEY.md §8b).  Each entry point
 * below names the reference code it replaces (paths relative to the reference root).  The Python
 * shim in cone_b200/ binds these with ctypes (see INTEGRATION.md).
 *
 * Conventions
 *   - every pointer is a DEVICE pointer unless the name ends in _host; tensors are row-major,
 *     contiguous, fp32 unless stated; the caller owns all buffers, outputs and the workspace;
 *   - every call is asynchronous on `stream` (a cudaStream_t passed as void*) and allocates nothing
 *     per call: the weights handle is the only owner of hidden device memory (the packed state
 *     dict, derived tables and, on first use of CONE_PREC_TC, fp16 weight copies).  Calls may be
 *     queued on different streams with different workspaces; calls that share one weights handle
 *     must come from one host thread at a time (the handle caches per-call scratch pointers);
 *   - return value 0 = OK, negative = error (CONE_ERR_*); cone_last_error() gives the message
 *     of the calling thread's last failure;
 *   - masks of the reference API are prefix masks (1 = valid, then 0 = pad), which is the only
 *     kind `start_end_collate` produces (cone/ego4d_mad_dataloader.py:305-344); they are passed
 *     here as per-row valid lengths.
 */
#ifndef CONE_B200_H
#define CONE_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CONE_OK 0
#define CONE_ERR_INVALID (-1)   /* bad argument / unsupported shape */
#define CONE_ERR_WORKSPACE (-2) /* workspace too small */
#define CONE_ERR_CUDA (-3)      /* CUDA runtime error */

/* compute precision of the dense projections */
#define CONE_PREC_FP32 0 /* fp32 CUDA-core GEMMs: parity mode, 1e-5 vs the reference */
#define CONE_PREC_TC 1   /* tcgen05 tensor-core GEMMs (fp16 operands, fp32 accumulate): 1e-3 */
#define CONE_PREC_TC_SPLIT 2 /* cone_linear only: 3-product split-fp16 GEMM on tcgen05, fp32-class accuracy (what
                                CONE_PREC_TC uses for the input projections and the span head) */

/* storage type of a raw feature tensor (frames, motion rows, tokens, CLS) passed to an _ex entry point.  fp16 and bf16
 * values convert to fp32 exactly and the kernels that read raw rows keep their fp32 reduction order, so a call on 16-bit
 * features gives the same bits as the same call on the fp32 upcast.  A 16-bit feature pointer must be 8-byte aligned. */
#define CONE_DTYPE_F32 0
#define CONE_DTYPE_F16 1
#define CONE_DTYPE_BF16 2

/* Longest window the library runs: max_v_l + max_q_l (and Lv + Lt of cone_forward) <= 512 rows.  Windows of up to 256
 * rows run the short-window attention kernels; 257..512 rows run their long-window variants, chosen per call from the
 * row count with the same accuracy contract.  Longer windows are refused (CONE_ERR_INVALID, the message names the
 * limit).  The handle's position tables grow as (max_v_l + 1) * max_v_l rows: about 2.4 GB at max_v_l = 480 in
 * CONE_PREC_TC mode (DESIGN.md §4). */
#define CONE_MAX_WINDOW_ROWS 512

/* Model / window hyper-parameters (cone/config.py:73-125; values per dataset in
 * cone/scripts/train_{ego4d,mad}.sh). */
typedef struct cone_dims {
    int32_t v_dim;       /* Dv: video feature dim (= CLS dim)            --v_appear_feat_dim */
    int32_t t_dim;       /* Dt: text token feature dim                   --t_feat_dim        */
    int32_t hidden;      /* d = 256                                      --hidden_dim        */
    int32_t nheads;      /* 8                                            --nheads            */
    int32_t ffn;         /* 1024                                         --dim_feedforward   */
    int32_t enc_layers;  /* 2                                            --enc_layers        */
    int32_t dec_layers;  /* 2                                            --dec_layers        */
    int32_t num_queries; /* 5 moment slots per window                    --num_queries       */
    int32_t max_v_l;     /* window length in frames                      --max_v_l           */
    int32_t max_q_l;     /* max text tokens (max_v_l + max_q_l <= 512)   --max_q_l           */
    int32_t m_dim;       /* Dm: motion feature dim, the input width of   --v_motion_feat_dim
                            input_vid_proj; 0 = Dv (one feature source for both roles) */
} cone_dims;

typedef struct cone_weights cone_weights; /* opaque: packed state dict + derived tables, on device */

const char* cone_last_error(void);
int cone_version(void);

/* ---- weights ------------------------------------------------------------------------------
 * Replaces `build_model` + `model.load_state_dict(checkpoint["model"])` (cone/model.py:468-521,
 * cone/inference.py:505-528).  `blob_host` is the state dict flattened to fp32 in the canonical
 * key order of cone_b200/weights.py::state_dict_shapes (n_floats must match exactly). */
int cone_weights_create(const float* blob_host, size_t n_floats, const cone_dims* dims, void* stream,
                        cone_weights** out);
void cone_weights_destroy(cone_weights* w);
/* Live weights: `model.load_state_dict` on an existing model, as the training loop's periodic
 * `eval_epoch` sees it (cone/train.py:164-168).  Writes the new state dict into the handle's existing
 * device buffers and recomputes every derived tensor in place: device pointers, TMA descriptors and
 * CUDA graphs captured over this handle stay valid.  Ordered after prior work on `stream`. */
int cone_weights_update(cone_weights* w, const float* blob_host, size_t n_floats, void* stream);
size_t cone_weights_expected_floats(const cone_dims* dims);

/* ---- workspace sizing ---------------------------------------------------------------------- */
/* bytes needed by cone_ground_windows / cone_forward for `n_windows` windows in flight */
size_t cone_workspace_bytes(const cone_dims* dims, int64_t n_windows, int32_t lv, int32_t lt);
/* bytes needed by cone_video_prepare / cone_video_prepare_motion for `n_frames` rows in flight */
size_t cone_prepare_workspace_bytes(const cone_dims* dims, int64_t n_frames);

/* ---- A1  host L2 normalisation: x / (||x|| + eps)  (utils/basic_utils.py:97-99, applied at
 * cone/ego4d_mad_dataloader.py:274-280, 459, 472).  eps = 0 gives x / ||x||.  eps < 0 selects
 * torch's F.normalize form x / max(||x||, -eps) (run_on_video/cone_localizator.py:127, 131).
 * In place if out == x. */
int cone_l2_normalize(const float* x, float* out, int64_t rows, int32_t dim, float eps, void* stream);
/* Same on x of storage type x_dtype (CONE_DTYPE_*); out stays fp32 (so out == x only for fp32).
 * cone_l2_normalize == cone_l2_normalize_ex(x_dtype CONE_DTYPE_F32). */
int cone_l2_normalize_ex(const void* x, int32_t x_dtype, float* out, int64_t rows, int32_t dim, float eps, void* stream);

/* ---- A2  stage 0 (cone/inference.py:250-260) + per-frame `input_vid_proj` (cone/model.py:100).
 * frames_raw [n_frames, Dv] raw features.  ctx_out [n_frames, Dv] = normalised adapted context
 * features; vidproj_out [n_frames, d] = input_vid_proj(raw) — the reference recomputes this per
 * window (A6); it is row-wise so it is computed once per frame here.  Either output may be NULL.
 * Raw appearance rows are the motion input only when one feature source serves both roles: on a handle with
 * m_dim != v_dim a non-NULL vidproj_out is CONE_ERR_INVALID (use cone_video_prepare_motion). */
int cone_video_prepare(const cone_weights* w, const float* frames_raw, int64_t n_frames, float* ctx_out,
                       float* vidproj_out, void* workspace, size_t workspace_bytes, int precision, void* stream);
/* Same on frames_raw of storage type frames_dtype (CONE_DTYPE_*); outputs stay fp32.
 * cone_video_prepare == cone_video_prepare_ex(frames_dtype CONE_DTYPE_F32). */
int cone_video_prepare_ex(const cone_weights* w, const void* frames_raw, int32_t frames_dtype, int64_t n_frames,
                          float* ctx_out, float* vidproj_out, void* workspace, size_t workspace_bytes, int precision,
                          void* stream);

/* Per-frame `input_vid_proj` of a separate motion stream (--motion_feat_dir): motion_raw [n_frames, Dm] raw features
 * are L2-normalised per frame, x / (||x|| + 1e-5) (cone/ego4d_mad_dataloader.py:284-292), then projected:
 * vidproj_out [n_frames, d], the `vidproj` of cone_ground_windows.  Frames run in slabs sized to the workspace
 * (cone_prepare_workspace_bytes); the result does not depend on the slab size. */
int cone_video_prepare_motion(const cone_weights* w, const float* motion_raw, int64_t n_frames, float* vidproj_out,
                              void* workspace, size_t workspace_bytes, int precision, void* stream);
/* Same on motion_raw of storage type motion_dtype (CONE_DTYPE_*); vidproj_out stays fp32.
 * cone_video_prepare_motion == cone_video_prepare_motion_ex(motion_dtype CONE_DTYPE_F32). */
int cone_video_prepare_motion_ex(const cone_weights* w, const void* motion_raw, int32_t motion_dtype, int64_t n_frames,
                                 float* vidproj_out, void* workspace, size_t workspace_bytes, int precision, void* stream);

/* `adapter_layer(x) + x` on arbitrary rows (cone/model.py:80; inference.py:255): the
 * `model.adapter_layer` attribute of the drop-in surface. `residual` = 1 adds x. */
int cone_adapter(const cone_weights* w, const float* x, float* out, int64_t rows, int residual, void* workspace,
                 size_t workspace_bytes, int precision, void* stream);

/* `torch.nn.functional.linear` on rows, the primitive every projection of the reference reduces to
 * (cone/model.py:437-440, 458-465; nn.MultiheadAttention in/out projections):
 * y[M,N] = act(x[M,K] * W[N,K]^T + bias (+ residual[M,N])).  W is any fp32 device matrix; with
 * CONE_PREC_TC its fp16 copy is cached inside the weights handle. */
int cone_linear(const cone_weights* w, const float* x, const float* W, const float* bias, int64_t M, int32_t N,
                int32_t K, int relu, const float* residual, float* y, void* workspace, size_t workspace_bytes,
                int precision, void* stream);

/* Tail of one encoder layer as the tensor-core mode runs it (cone/transformer.py:239-245):
 *     x   = norm1(res + out_proj(att))            out = norm2(x + linear2(relu(linear1(x))))
 * for encoder layer `layer` of the handle, on M rows of width 256: ONE fused tcgen05 kernel (csrc/enc_tail.cu).
 * Operator-level parity surface: att / res / out are fp32 [M, 256] device arrays here (att is rounded to fp16 as
 * the attention kernel's output is, res travels as fp16 hi + lo); inside cone_ground_windows / cone_forward the
 * same kernel runs directly on the fp16 streams.  cta_group: 1, 2 (tcgen05 CTA pair) or 0 = default.
 * workspace >= 10 * M * 256 bytes. */
int cone_encoder_tail(const cone_weights* w, int32_t layer, const float* att, const float* res, int64_t M, float* out,
                      int32_t cta_group, void* workspace, size_t workspace_bytes, void* stream);

/* ---- A3  stage 1 (cone/inference.py:276-299).
 * Frame scores `einsum('db,b->d')` (inference.py:284) for all queries of a set of videos in one
 * grouped GEMM: queries must be grouped by video.  ctx [n_frames_total, Dv]; video_offsets
 * [n_videos+1] int64 frame offsets; q_first [n_videos+1] int32 = first query of each video;
 * cls_norm [n_queries, Dv] normalised CLS (all device arrays).  max_video_frames /
 * max_video_queries size the launch grid.  score_out is ragged: query q's scores are
 * score_out[score_offsets[q] ... + L_video(q)), score_offsets [n_queries] int64.
 * Always fp32: the window ranking must be bit-stable (precision is accepted for symmetry). */
int cone_frame_scores(const float* ctx, int32_t v_dim, const int64_t* video_offsets, const int32_t* q_first,
                      int32_t n_videos, int32_t max_video_frames, int32_t max_video_queries, const float* cls_norm,
                      float* score_out, const int64_t* score_offsets, int precision, void* stream);

/* Window scores + full rank-list (score descending, window index ascending on ties; NaN first, as
 * torch.sort orders it).  frame_score ragged as above (device), score_offsets / frame_count
 * [n_queries] device arrays.  ranklist_out [n_queries, ranklist_stride] int32, filled up to
 * num_window(q) = ceil(L/stride)+1, rest -1; winscore_out (nullable) same shape fp32.
 * Also the parity surface of the function form `compute_window_ranklist`
 * (run_on_video/cone_localizator.py:83-100). */
int cone_window_ranklist(const float* frame_score, const int64_t* score_offsets, const int32_t* frame_count,
                         int32_t n_queries, int32_t max_v_l, int32_t* ranklist_out, float* winscore_out,
                         int32_t ranklist_stride, void* stream);

/* ---- A1-A3 for ONE video in one call: the `cone_prefilter` of SURVEY.md §8(b) — host L2 normalisation of the raw frames and
 * CLS vectors (cone/ego4d_mad_dataloader.py:459, 472), stage 0 (cone/inference.py:250-260) and stage 1
 * (cone/inference.py:276-299; the same pre-filter runs in cone_2dtan/moment_localization/test.py:173-239).
 *   frames_raw [L, Dv] raw features of the video, cls_raw [n_queries, Dv] raw CLS features (device)
 *   win_idx   [n_queries, topk] int32: the first topk window ids of each query's rank-list, -1 where the video has fewer
 *   win_score [n_queries, topk] fp32 (nullable): the window scores (max frame score) of those windows
 * Always fp32 (the ranking must be bit-stable).  The window length is the handle's max_v_l.
 * Composition of cone_l2_normalize, cone_video_prepare, cone_frame_scores, cone_window_ranklist: bit-identical to them. */
size_t cone_prefilter_workspace_bytes(const cone_dims* dims, int64_t n_frames, int32_t n_queries);
int cone_prefilter(const cone_weights* w, const float* frames_raw, int64_t n_frames, const float* cls_raw, int32_t n_queries,
                   int32_t topk, int32_t* win_idx, float* win_score, void* workspace, size_t workspace_bytes, void* stream);
/* Same with frames_raw of storage type frames_dtype and cls_raw of storage type cls_dtype (CONE_DTYPE_*, independent).
 * cone_prefilter == cone_prefilter_ex(both CONE_DTYPE_F32). */
int cone_prefilter_ex(const cone_weights* w, const void* frames_raw, int32_t frames_dtype, int64_t n_frames,
                      const void* cls_raw, int32_t cls_dtype, int32_t n_queries, int32_t topk, int32_t* win_idx,
                      float* win_score, void* workspace, size_t workspace_bytes, void* stream);

/* ---- A4-A9  stage 2: slice the top-k windows of every query straight out of the frame tensors,
 * run Moment-DETR on them and score the proposals (cone/ego4d_mad_dataloader.py:144-159, 305-358;
 * cone/model.py:82-152; cone/inference.py:46-52).
 *   frames_raw [n_frames, Dv] raw appearance rows (pooled for matching), vidproj [n_frames, d] projected motion rows
 *       (from cone_video_prepare, or cone_video_prepare_motion for a separate motion stream)
 *   q_video_start / q_video_len [n_queries]  frame offset and length of each query's video
 *   ranklist [n_queries, ranklist_stride]    from cone_window_ranklist
 *   tok [n_queries, max_q_l, Dt] L2-normalised tokens, zero padded; tok_len [n_queries]
 *   cls_norm [n_queries, Dv]
 *   q_batch [n_queries] id of the reference eval batch the query falls in (dataset index /
 *       eval_bsz): proposals are mean-pooled over the window zero-padded to that batch's longest
 *       window, exactly as the reference does (SURVEY.md §8 A9); n_batches = max id + 1.
 *       NULL = every window is pooled over max_v_l zero-padded rows, the fixed padding of the
 *       single-video front end (run_on_video/cone_localizator.py:141-165)
 * Outputs, [n_queries, topk, nq, ...]: pred_spans (cx,w), prob_fg = softmax(logits)[0], match;
 * win_start / win_len [n_queries, topk] int32 (len 0 = window absent: video has < topk windows). */
int cone_ground_windows(const cone_weights* w, const float* frames_raw, int64_t n_frames, const float* vidproj,
                        const int64_t* q_video_start, const int32_t* q_video_len, const int32_t* ranklist,
                        int32_t ranklist_stride, const float* tok, const int32_t* tok_len, const float* cls_norm,
                        const int32_t* q_batch, int32_t n_batches, int32_t n_queries, int32_t topk,
                        float* pred_spans, float* prob_fg, float* match, int32_t* win_start, int32_t* win_len,
                        void* workspace, size_t workspace_bytes, int precision, void* stream);
/* Same with frames_raw (the rows pooled for matching) of storage type frames_dtype (CONE_DTYPE_*); every other
 * input is fp32 as above.  cone_ground_windows == cone_ground_windows_ex(frames_dtype CONE_DTYPE_F32). */
int cone_ground_windows_ex(const cone_weights* w, const void* frames_raw, int32_t frames_dtype, int64_t n_frames,
                           const float* vidproj, const int64_t* q_video_start, const int32_t* q_video_len,
                           const int32_t* ranklist, int32_t ranklist_stride, const float* tok, const int32_t* tok_len,
                           const float* cls_norm, const int32_t* q_batch, int32_t n_batches, int32_t n_queries,
                           int32_t topk, float* pred_spans, float* prob_fg, float* match, int32_t* win_start,
                           int32_t* win_len, void* workspace, size_t workspace_bytes, int precision, void* stream);

/* ---- A6-A8  reference-shaped forward: `model(src_txt, src_txt_mask, src_vid_motion,
 * src_vid_motion_mask)` (cone/model.py:82-128).  src_vid [B, Lv, Dm] (= src_vid_motion), src_txt [B, Lt, Dt], valid
 * lengths vid_len / txt_len [B] int32, Lv <= max_v_l of the handle, Lv + Lt <= CONE_MAX_WINDOW_ROWS.
 * Outputs: pred_logits [B,nq,2], pred_spans [B,nq,2];
 * nullable: saliency [B,Lv], aux_logits / aux_spans [dec_layers-1, B, nq, 2]. */
int cone_forward(const cone_weights* w, const float* src_txt, const int32_t* txt_len, const float* src_vid,
                 const int32_t* vid_len, int32_t B, int32_t Lt, int32_t Lv, float* pred_logits, float* pred_spans,
                 float* saliency, float* aux_logits, float* aux_spans, void* workspace, size_t workspace_bytes,
                 int precision, void* stream);

/* ---- A9  `model.forward_clip_matching(src_cls_txt, src_vid_appear, src_vid_appear_mask,
 * proposal=pred_spans)` (cone/model.py:130-152, 178-210).  src_vid_appear [B, Lv, Dv] zero padded,
 * vid_len [B]; spans [B, nq, 2]; out [B, nq]. */
int cone_clip_matching(const cone_weights* w, const float* src_cls_txt, const float* src_vid_appear,
                       const int32_t* vid_len, const float* spans, int32_t B, int32_t Lv, int32_t nq, float* out,
                       void* workspace, size_t workspace_bytes, int precision, void* stream);

/* ---- A10-A13  stage 3 (cone/inference.py:70-91, 103-217; utils/temporal_nms.py).
 * Per query: spans -> seconds, 4-decimal rounding, per-window sort, min-max score fusion,
 * (st,ed) de-duplication, and for each of the three rankings (0 fusion, 1 proposal, 2 matching)
 * stable sort + greedy temporal NMS.  nms_thd = -1 disables NMS (inference.py:125-127).
 * out [n_queries, 3, max_after_nms, 5] fp64 rows [st, ed, score, match, fusion]; out_count
 * [n_queries, 3]; rows_out (nullable) [n_queries, topk*nq, 4] fp64 = the reference's
 * `pred_relevant_windows` rows, rows_count (nullable) [n_queries]. */
int cone_fuse_nms(const float* pred_spans, const float* prob_fg, const float* match, const int32_t* win_start,
                  const int32_t* win_len, int32_t n_queries, int32_t topk, int32_t nq, float clip_length,
                  double nms_thd, int32_t max_before_nms, int32_t max_after_nms, double* out, int32_t* out_count,
                  double* rows_out, int32_t* rows_count, void* stream);

/* Same with the two knobs of the single-video front end (run_on_video/cone_localizator.py:183-219):
 * fixed_duration > 0 scales every span by that many frames instead of the window's own length
 * (`span_cxw_to_xx(spans) * args.max_v_l`), sort_within_window = 0 keeps the moment slots of a window
 * in slot order.  cone_fuse_nms == cone_fuse_nms_ex(fixed_duration 0, sort_within_window 1). */
int cone_fuse_nms_ex(const float* pred_spans, const float* prob_fg, const float* match, const int32_t* win_start,
                     const int32_t* win_len, int32_t n_queries, int32_t topk, int32_t nq, float clip_length,
                     double nms_thd, int32_t max_before_nms, int32_t max_after_nms, int32_t fixed_duration,
                     int32_t sort_within_window, double* out, int32_t* out_count, double* rows_out,
                     int32_t* rows_count, void* stream);

/* ---- A13  `temporal_nms(predictions, nms_thd, max_after_nms)` (utils/temporal_nms.py:25-74) on
 * one list: st/ed/score [n] fp64 in input order; keep_out [max_after_nms] indices into the input in
 * output order; n_keep_out [1]. */
int cone_temporal_nms(const double* st, const double* ed, const double* score, int32_t n, double nms_thd,
                      int32_t max_after_nms, int32_t* keep_out, int32_t* n_keep_out, void* stream);

/* ---- A14 / SURVEY.md §8(f)1  metric counters on the device, straight from cone_fuse_nms' output.
 * cone_eval_recall: for each query and each of the 3 rankings, IoU of its first max(topk) predictions
 * with the ground truth gt [n_queries, 2] fp64 (seconds) and, per (rank K, threshold), whether any of
 * the first K exceeds it (strict >).  flavour 0 = standalone_eval/evaluate_mad.py:32-37, 60-104
 * (float32 hull IoU against float32 thresholds), flavour 1 =
 * standalone_eval/evaluate_ego4d_nlq.py:41-62, 65-117 (float64).  topk_host / thresholds_host are
 * HOST arrays (at most CONE_EVAL_MAX_TOPK / CONE_EVAL_MAX_THRESHOLDS entries).  hits
 * [3, n_topk, n_thr] int64 is ADDED to (zero it first; counters of several steps or ranks simply
 * add up; recall = hits / #queries); top1_iou (nullable) [n_queries, 3] fp64 = IoU of the first
 * prediction (Ego4D's mIoU is its mean).
 * cone_eval_window_recall: standalone_eval/evaluate_pre_filtered_window.py:30-72: whether any of the
 * first K ranked windows lies in range(floor(st/clip_length/stride), ceil(ed/clip_length/stride)+1),
 * stride = int(max_v_l / 2).  hits [n_topk] int64 is added to. */
#define CONE_EVAL_MAX_TOPK 8
#define CONE_EVAL_MAX_THRESHOLDS 8
int cone_eval_recall(const double* nms, const int32_t* nms_count, const double* gt, int32_t n_queries,
                     int32_t max_after_nms, const int32_t* topk_host, int32_t n_topk, const double* thresholds_host,
                     int32_t n_thresholds, int32_t flavour, int64_t* hits, double* top1_iou, void* stream);
int cone_eval_window_recall(const int32_t* ranklist, int32_t ranklist_stride, const double* gt, int32_t n_queries,
                            double clip_length, int32_t max_v_l, const int32_t* topk_host, int32_t n_topk,
                            int64_t* hits, void* stream);

/* ---- measurement hooks (no reference counterpart) --------------------------------------------
 * Per-kernel timing: when enabled, every launch of the calling thread is bracketed by CUDA events on
 * its stream; cone_profile_read waits for them and returns, per category, the summed device time
 * (ms), launch count and the algorithmic FLOPs / bytes the launches were given. */
void cone_profile_enable(int on);
int cone_profile_categories(void);
const char* cone_profile_name(int category);
int cone_profile_read(double* ms, int64_t* launches, double* flops, double* bytes, int n_categories);

/* number of kernels launched by this library on the calling thread since the last reset */
int64_t cone_launch_count(void);
void cone_launch_count_reset(void);

#ifdef __cplusplus
}
#endif
#endif /* CONE_B200_H */
