// Fine-grained proposal ranking (cone/model.py:130-152, 178-210): span -> [floor, ceil) frame bounds,
// mean-pool the RAW appearance rows of the zero-padded window, (adapter + residual via the GEMM path),
// L2-normalise, dot with the normalised CLS vector.  HBM/L2-bound: coalesced float4 row reads.
// The pooling kernels also read raw rows stored as fp16 / bf16 (features.cuh): 4 columns per thread as in fp32, each
// column's rows added in row order into its own fp32 accumulator, so the pooled rows are those of the upcast input.
#include <math_constants.h>

#include <type_traits>

#include "features.cuh"
#include "kernels.h"

namespace cone {

namespace {

// One CTA per (window, slot).  Bounds follow the reference's fp32 operation order exactly:
//   x1 = cx - 0.5*w ; x2 = cx + 0.5*w                     (span_cxw_to_xx, cone/span_utils.py:39-40)
//   start = relu(int(floor(x1 * dur))) ; end = int(ceil(x2 * dur))          (model.py:187-192)
// `feat[start:end]` is a Python slice of the window zero-padded to pad_len rows: `end` clips to pad_len,
// pad rows inside the slice are averaged in (they are zeros), an empty slice gives NaN.
template <class T>
__global__ void __launch_bounds__(256)
span_mean_pool_kernel(const T* __restrict__ frames, int64_t n_frames, const int64_t* __restrict__ vid_base,
                      const int32_t* __restrict__ vlen, const int32_t* __restrict__ pad_len,
                      const float* __restrict__ spans, float* __restrict__ pooled, int nq, int Dv) {
    const int64_t p = blockIdx.x;  // window * nq + slot
    const int64_t b = p / nq;
    const float cx = spans[p * 2 + 0], w = spans[p * 2 + 1];
    const int len = vlen[b];
    const float dur = (float)len;
    const float hw = __fmul_rn(0.5f, w);
    const float x1 = __fmul_rn(__fsub_rn(cx, hw), dur);
    const float x2 = __fmul_rn(__fadd_rn(cx, hw), dur);
    int start = (int)floorf(x1);
    start = start < 0 ? 0 : start;
    int end = (int)ceilf(x2);
    const int pl = pad_len[b];
    if (end > pl) end = pl;
    const int n = end - start;            // rows in the slice, pad rows included
    const int vend = end < len ? end : len;  // rows that hold data
    const int64_t base = vid_base[b];
    const int nv = Dv >> 2;
    for (int c = threadIdx.x; c < nv; c += blockDim.x) {
        float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
        // rows are summed in order (start, start+1, ...) as the reference's mean does; 8 loads are in flight at a
        // time so the column is not one memory round trip per row
        const int64_t last = (base + vend < n_frames ? base + vend : n_frames) - base;  // rows past the tensor end: none
        for (int r = start; r < last; r += 8) {
            float4 v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u)
                v[u] = (r + u < last) ? ldg_feat4(frames + (base + r + u) * Dv + 4 * c) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int u = 0; u < 8; ++u) {
                if (r + u < last) {
                    acc.x += v[u].x; acc.y += v[u].y; acc.z += v[u].z; acc.w += v[u].w;
                }
            }
        }
        float4 o;
        if (n > 0) {
            const float fn = (float)n;
            o = make_float4(acc.x / fn, acc.y / fn, acc.z / fn, acc.w / fn);
        } else {
            o = make_float4(CUDART_NAN_F, CUDART_NAN_F, CUDART_NAN_F, CUDART_NAN_F);
        }
        reinterpret_cast<float4*>(pooled + p * Dv)[c] = o;
    }
}

// One CTA per WINDOW: the rows between the earliest start and the latest end of the window's NQ proposals are read once
// and every row is added to the accumulators of the proposals whose slice contains it.  Each proposal's rows are
// still added in increasing order into its own accumulator, so the result is bit-identical to the per-proposal kernel
// above; what changes is the traffic: the proposals of a window overlap (ncu: 39 rows per proposal on average, 195 per
// window, against at most Lv = 125 distinct rows).
template <int NQ, class T>
__global__ void __launch_bounds__(256)
span_mean_pool_window_kernel(const T* __restrict__ frames, int64_t n_frames, const int64_t* __restrict__ vid_base,
                             const int32_t* __restrict__ vlen, const int32_t* __restrict__ pad_len,
                             const float* __restrict__ spans, float* __restrict__ pooled, int nq, int Dv) {
    const int64_t b = blockIdx.x;
    const int len = vlen[b];
    const float dur = (float)len;
    const int pl = pad_len[b];
    const int64_t base = vid_base[b];
    int st[NQ], en[NQ], cnt[NQ];  // data rows [st, en) and slice length (pad rows included) of every proposal
    int lo = 0x7fffffff, hi = 0;
#pragma unroll
    for (int j = 0; j < NQ; ++j) {
        st[j] = en[j] = cnt[j] = 0;
        if (j < nq) {
            const float cx = spans[(b * nq + j) * 2 + 0], w = spans[(b * nq + j) * 2 + 1];
            const float hw = __fmul_rn(0.5f, w);
            const float x1 = __fmul_rn(__fsub_rn(cx, hw), dur);
            const float x2 = __fmul_rn(__fadd_rn(cx, hw), dur);
            int start = (int)floorf(x1);
            start = start < 0 ? 0 : start;
            int end = (int)ceilf(x2);
            if (end > pl) end = pl;
            cnt[j] = end - start;
            int vend = end < len ? end : len;                                  // rows that hold data
            const int64_t room = n_frames - base;                              // rows past the tensor end: none
            if ((int64_t)vend > room) vend = (int)(room < 0 ? 0 : room);
            st[j] = start;
            en[j] = vend > start ? vend : start;
            if (en[j] > st[j]) {
                lo = st[j] < lo ? st[j] : lo;
                hi = en[j] > hi ? en[j] : hi;
            }
        }
    }
    const int nv = Dv >> 2;
    for (int c = threadIdx.x; c < nv; c += blockDim.x) {
        float4 acc[NQ];
#pragma unroll
        for (int j = 0; j < NQ; ++j) acc[j] = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int r = lo; r < hi; r += 8) {
            float4 v[8];
#pragma unroll
            for (int u = 0; u < 8; ++u)
                v[u] = (r + u < hi) ? ldg_feat4(frames + (base + r + u) * Dv + 4 * c) : make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
            for (int u = 0; u < 8; ++u) {
#pragma unroll
                for (int j = 0; j < NQ; ++j) {
                    if (r + u >= st[j] && r + u < en[j]) {
                        acc[j].x += v[u].x; acc[j].y += v[u].y; acc[j].z += v[u].z; acc[j].w += v[u].w;
                    }
                }
            }
        }
#pragma unroll
        for (int j = 0; j < NQ; ++j) {
            if (j < nq) {
                float4 o;
                if (cnt[j] > 0) {
                    const float fn = (float)cnt[j];
                    o = make_float4(acc[j].x / fn, acc[j].y / fn, acc[j].z / fn, acc[j].w / fn);
                } else {
                    o = make_float4(CUDART_NAN_F, CUDART_NAN_F, CUDART_NAN_F, CUDART_NAN_F);
                }
                reinterpret_cast<float4*>(pooled + (b * nq + j) * Dv)[c] = o;
            }
        }
    }
}

// out[p] = sum_d (x[p,d] / ||x[p]||) * t[qidx[b], d]     one warp per proposal
__global__ void norm_dot_kernel(const float* __restrict__ x, const float* __restrict__ t,
                                const int32_t* __restrict__ qidx, float* __restrict__ out, int64_t rows, int nq, int Dv) {
    const int lane = threadIdx.x & 31;
    const int64_t p = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (p >= rows) return;
    const float4* xr = reinterpret_cast<const float4*>(x + p * Dv);
    const float4* tr = reinterpret_cast<const float4*>(t + (int64_t)qidx[p / nq] * Dv);
    const int nv = Dv >> 2;
    float sq = 0.f;
    for (int i = lane; i < nv; i += 32) {
        const float4 v = xr[i];
        sq += (v.x * v.x + v.y * v.y) + (v.z * v.z + v.w * v.w);
    }
    const float nrm = sqrtf(warp_sum(sq));
    float dot = 0.f;
    for (int i = lane; i < nv; i += 32) {
        const float4 v = xr[i];
        const float4 u = __ldg(tr + i);
        dot += (v.x / nrm) * u.x + (v.y / nrm) * u.y + (v.z / nrm) * u.z + (v.w / nrm) * u.w;
    }
    dot = warp_sum(dot);
    if (lane == 0) out[p] = dot;
}

}  // namespace

int span_mean_pool(const void* frames_v, int frames_dtype, int64_t n_frames, const int64_t* vid_base, const int32_t* vlen,
                   const int32_t* pad_len, const float* spans, float* pooled, int64_t B, int nq, int Dv,
                   cudaStream_t s) {
    return dispatch_feature(frames_dtype, [&](auto tag) {
        using T = std::remove_const_t<std::remove_pointer_t<decltype(tag)>>;
        const T* frames = static_cast<const T*>(frames_v);
        if (B == 0) return CONE_OK;
        CONE_REQUIRE((Dv & 3) == 0, "span_mean_pool: Dv must be a multiple of 4");
        const int threads = (Dv / 4) >= 256 ? 256 : ((Dv / 4 + 31) / 32) * 32;
        ProfScope ps(s, P_POOL);
        if (nq <= 5) {
            span_mean_pool_window_kernel<5, T><<<(unsigned)B, threads, 0, s>>>(frames, n_frames, vid_base, vlen, pad_len,
                                                                            spans, pooled, nq, Dv);
        } else if (nq <= 8) {
            span_mean_pool_window_kernel<8, T><<<(unsigned)B, threads, 0, s>>>(frames, n_frames, vid_base, vlen, pad_len,
                                                                            spans, pooled, nq, Dv);
        } else {  // many proposals per window (cone_clip_matching allows up to 64): one CTA per proposal
            span_mean_pool_kernel<T><<<(unsigned)(B * nq), threads, 0, s>>>(frames, n_frames, vid_base, vlen, pad_len, spans,
                                                                          pooled, nq, Dv);
        }
        CONE_LAUNCH_CHECK("span_mean_pool");
        return CONE_OK;
    });
}

int norm_dot(const float* p, const float* t, const int32_t* qidx, float* out, int64_t B, int nq, int Dv,
             cudaStream_t s) {
    if (B == 0) return CONE_OK;
    const int warps = 8;
    ProfScope ps(s, P_POOL);
    norm_dot_kernel<<<(unsigned)cdiv64(B * nq, warps), warps * 32, 0, s>>>(p, t, qidx, out, B * nq, nq, Dv);
    CONE_LAUNCH_CHECK("norm_dot");
    return CONE_OK;
}

}  // namespace cone
