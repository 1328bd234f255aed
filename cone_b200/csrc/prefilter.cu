// Stage 1 of the reference (cone/inference.py:286-299): window score = max frame score inside each
// 50%-overlapping window, then the full rank-list by (score descending, window index ascending).
// Every (frame, query) score is computed once (gemm) and windows take the max of STORED values, so the
// exact ties between overlapping windows that share their best frame survive (SURVEY.md §7 H1).
#include <math_constants.h>

#include "kernels.h"

namespace cone {

namespace {

// torch.max propagates NaN; torch.sort(descending=True) puts NaN first.
__device__ __forceinline__ float nanmax(float a, float b) { return (a != a) ? a : ((b != b) ? b : fmaxf(a, b)); }

// monotone map float -> uint32 (ascending); -0.0 == +0.0; NaN largest
__device__ __forceinline__ uint32_t orderable(float f) {
    if (f != f) return 0xFFFFFFFFu;
    f = f + 0.0f;  // -0.0 -> +0.0
    const uint32_t u = __float_as_uint(f);
    return (u & 0x80000000u) ? ~u : (u | 0x80000000u);
}

// one CTA per query: window maxima into shared memory, then a bitonic sort of 64-bit keys
// key = (~orderable(score) << 32) | window_index, ascending  ==  score descending, index ascending.
__global__ void __launch_bounds__(256)
window_ranklist_kernel(const float* __restrict__ frame_score, const int64_t* __restrict__ score_offsets,
                       const int32_t* __restrict__ frame_count, int max_v_l, int32_t* __restrict__ ranklist,
                       float* __restrict__ winscore, int ranklist_stride, int npad) {
    extern __shared__ unsigned long long keys[];
    const int q = blockIdx.x;
    const int L = frame_count[q];
    const int stride = max_v_l / 2;
    const int nw = (L + stride - 1) / stride + 1;
    const float* fs = frame_score + score_offsets[q];
    if (nw > npad) {  // windows past npad cannot enter the sort: no rank-list rather than the best of a prefix
        for (int i = threadIdx.x; i < ranklist_stride; i += blockDim.x) {
            ranklist[(int64_t)q * ranklist_stride + i] = -1;
            if (winscore) winscore[(int64_t)q * ranklist_stride + i] = CUDART_NAN_F;
        }
        return;
    }
    for (int i = threadIdx.x; i < npad; i += blockDim.x) {
        unsigned long long key = ~0ull;
        if (i < nw) {
            const int s = max((i - 1) * stride, 0);
            const int e = min((i - 1) * stride + max_v_l, L);
            float m = -CUDART_INF_F;
            if (e > s) {
                m = fs[s];
                for (int f = s + 1; f < e; ++f) m = nanmax(m, fs[f]);
            }
            if (winscore && i < ranklist_stride) winscore[(int64_t)q * ranklist_stride + i] = m;
            key = ((unsigned long long)(~orderable(m)) << 32) | (unsigned)i;
        }
        keys[i] = key;
    }
    __syncthreads();
    for (int k = 2; k <= npad; k <<= 1) {
        for (int j = k >> 1; j > 0; j >>= 1) {
            for (int i = threadIdx.x; i < npad; i += blockDim.x) {
                const int ixj = i ^ j;
                if (ixj > i) {
                    const unsigned long long a = keys[i], b = keys[ixj];
                    const bool up = ((i & k) == 0);
                    if ((a > b) == up) {
                        keys[i] = b;
                        keys[ixj] = a;
                    }
                }
            }
            __syncthreads();
        }
    }
    for (int i = threadIdx.x; i < ranklist_stride; i += blockDim.x)
        ranklist[(int64_t)q * ranklist_stride + i] = (i < nw) ? (int32_t)(keys[i] & 0xFFFFFFFFull) : -1;
}

__global__ void build_windows_kernel(const int32_t* __restrict__ ranklist, int ranklist_stride,
                                     const int32_t* __restrict__ q_video_len, int n_queries, int topk, int max_v_l,
                                     int32_t* __restrict__ win_start, int32_t* __restrict__ win_len) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_queries * topk) return;
    const int q = i / topk, j = i % topk;
    const int L = q_video_len[q];
    const int stride = max_v_l / 2;
    const int nw = (L + stride - 1) / stride + 1;
    int s = 0, n = 0;
    if (j < nw && j < ranklist_stride) {  // `ranklist[:topk_window]` yields min(k, num_window) windows
        const int w = ranklist[(int64_t)q * ranklist_stride + j];
        s = max((w - 1) * stride, 0);
        const int e = min((w - 1) * stride + max_v_l, L);
        n = max(e - s, 0);
    }
    win_start[i] = s;
    win_len[i] = n;
}

__global__ void batch_max_len_kernel(const int32_t* __restrict__ win_len, const int32_t* __restrict__ q_batch,
                                     int n_queries, int topk, int32_t* __restrict__ batch_max) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_queries * topk) return;
    atomicMax(&batch_max[q_batch[i / topk]], win_len[i]);
}

// descriptors of the flat windows g0 .. g0+nw of [n_queries, topk]; query indices relative to q_lo (the chunk's first query)
__global__ void fill_window_desc_chunk_kernel(const int64_t* __restrict__ q_video_start,
                                              const int32_t* __restrict__ win_start, const int32_t* __restrict__ win_len,
                                              const int32_t* __restrict__ tok_len, const int32_t* __restrict__ q_batch,
                                              const int32_t* __restrict__ batch_max, int64_t g0, int nw, int q_lo, int topk,
                                              int Lt, int fixed_pad, int64_t* vid_base, int32_t* vlen, int64_t* txt_base,
                                              int32_t* tlen, int32_t* pad_len, int32_t* qidx) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= nw) return;
    const int64_t g = g0 + i;
    const int q = (int)(g / topk);
    const int ql = q - q_lo;
    vid_base[i] = q_video_start[q] + win_start[g];
    vlen[i] = win_len[g];
    txt_base[i] = (int64_t)ql * Lt;
    tlen[i] = tok_len[q];
    // q_batch == null: every window is padded to `fixed_pad` rows (run_on_video/cone_localizator.py:141-165)
    pad_len[i] = q_batch ? batch_max[q_batch[q]] : fixed_pad;
    qidx[i] = ql;
}

}  // namespace

int window_ranklist(const float* frame_score, const int64_t* score_offsets, const int32_t* frame_count, int n_queries,
                    int max_v_l, int32_t* ranklist, float* winscore, int ranklist_stride, cudaStream_t s) {
    if (n_queries == 0) return CONE_OK;
    CONE_REQUIRE(max_v_l >= 2, "window_ranklist: max_v_l must be >= 2");
    int npad = 32;
    while (npad < ranklist_stride) npad <<= 1;
    CONE_REQUIRE(npad <= 16384, "window_ranklist: more than 16384 windows per video is not supported");
    const size_t smem = (size_t)npad * sizeof(unsigned long long);
    if (smem > 48 * 1024) {
        CONE_CUDA(cudaFuncSetAttribute(window_ranklist_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    }
    ProfScope ps(s, P_RANKLIST);
    window_ranklist_kernel<<<n_queries, 256, smem, s>>>(frame_score, score_offsets, frame_count, max_v_l, ranklist,
                                                        winscore, ranklist_stride, npad);
    CONE_LAUNCH_CHECK("window_ranklist");
    return CONE_OK;
}

namespace {
// descriptors of the single-video form: every query sees the same L frames
__global__ void prefilter_desc_kernel(int64_t* video_offsets, int32_t* q_first, int64_t* score_offsets, int32_t* frame_count,
                                      int64_t L, int n_queries) {
    const int q = blockIdx.x * blockDim.x + threadIdx.x;
    if (q == 0) {
        video_offsets[0] = 0; video_offsets[1] = L;
        q_first[0] = 0; q_first[1] = n_queries;
    }
    if (q < n_queries) {
        score_offsets[q] = (int64_t)q * L;
        frame_count[q] = (int32_t)L;
    }
}
// first `topk` entries of each rank-list and the scores of those windows; -1 / NaN past the video's window count
__global__ void take_topk_kernel(const int32_t* __restrict__ ranklist, const float* __restrict__ winscore, int ranklist_stride,
                                 int n_queries, int topk, int32_t* __restrict__ win_idx, float* __restrict__ win_score) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n_queries * topk) return;
    const int q = i / topk, j = i - q * topk;
    const int32_t w = j < ranklist_stride ? ranklist[(int64_t)q * ranklist_stride + j] : -1;
    win_idx[i] = w;
    if (win_score) win_score[i] = w >= 0 ? winscore[(int64_t)q * ranklist_stride + w] : __int_as_float(0x7fc00000);
}
}  // namespace

int prefilter_desc(int64_t* video_offsets, int32_t* q_first, int64_t* score_offsets, int32_t* frame_count, int64_t L,
                   int n_queries, cudaStream_t s) {
    prefilter_desc_kernel<<<cdiv(n_queries > 0 ? n_queries : 1, 256), 256, 0, s>>>(video_offsets, q_first, score_offsets, frame_count, L,
                                                                                  n_queries);
    CONE_LAUNCH_CHECK("prefilter_desc");
    return CONE_OK;
}

int take_topk(const int32_t* ranklist, const float* winscore, int ranklist_stride, int n_queries, int topk, int32_t* win_idx,
              float* win_score, cudaStream_t s) {
    if (n_queries == 0 || topk == 0) return CONE_OK;
    take_topk_kernel<<<cdiv(n_queries * topk, 256), 256, 0, s>>>(ranklist, winscore, ranklist_stride, n_queries, topk, win_idx,
                                                                win_score);
    CONE_LAUNCH_CHECK("take_topk");
    return CONE_OK;
}

int build_windows(const int32_t* ranklist, int ranklist_stride, const int32_t* q_video_len, int n_queries, int topk,
                  int max_v_l, int32_t* win_start, int32_t* win_len, cudaStream_t s) {
    if (n_queries == 0) return CONE_OK;
    build_windows_kernel<<<cdiv(n_queries * topk, 256), 256, 0, s>>>(ranklist, ranklist_stride, q_video_len, n_queries,
                                                                    topk, max_v_l, win_start, win_len);
    CONE_LAUNCH_CHECK("build_windows");
    return CONE_OK;
}

int batch_max_len(const int32_t* win_len, const int32_t* q_batch, int n_queries, int topk, int32_t* batch_max,
                  int n_batches, cudaStream_t s) {
    if (n_queries == 0) return CONE_OK;
    CONE_CUDA(cudaMemsetAsync(batch_max, 0, sizeof(int32_t) * n_batches, s));
    batch_max_len_kernel<<<cdiv(n_queries * topk, 256), 256, 0, s>>>(win_len, q_batch, n_queries, topk, batch_max);
    CONE_LAUNCH_CHECK("batch_max_len");
    return CONE_OK;
}

int fill_window_desc_chunk(const int64_t* q_video_start, const int32_t* win_start, const int32_t* win_len,
                           const int32_t* tok_len, const int32_t* q_batch, const int32_t* batch_max, int64_t g0, int nw,
                           int q_lo, int topk, int Lt, int fixed_pad, int64_t* vid_base, int32_t* vlen, int64_t* txt_base,
                           int32_t* tlen, int32_t* pad_len, int32_t* qidx, cudaStream_t s) {
    if (nw == 0) return CONE_OK;
    fill_window_desc_chunk_kernel<<<cdiv(nw, 256), 256, 0, s>>>(q_video_start, win_start, win_len, tok_len, q_batch,
                                                                batch_max, g0, nw, q_lo, topk, Lt, fixed_pad, vid_base,
                                                                vlen, txt_base, tlen, pad_len, qidx);
    CONE_LAUNCH_CHECK("fill_window_desc_chunk");
    return CONE_OK;
}

}  // namespace cone
