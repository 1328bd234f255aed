// Row-wise fp32 kernels: LayerNorm (+residual), L2 normalisation, sine position table, window row gather.
// All are HBM/L2-bound: one warp per row, float4 accesses, grid sized from the row count.
// LayerNorm and L2 normalisation also read raw feature rows stored as fp16 / bf16 (features.cuh): a lane then loads the
// same 4 elements per step with one 8-byte load, so its partial sums, and the result, are those of the fp32 kernel.
#include <cuda_fp16.h>

#include <type_traits>

#include "features.cuh"
#include "kernels.h"

namespace cone {

namespace {

constexpr int kWarpsPerBlock = 8;

// out = LayerNorm(x (+ residual)) * gamma + beta     (torch.nn.LayerNorm: biased variance, eps inside sqrt)
template <class T>
__global__ void layernorm_rows_kernel(const T* __restrict__ x, const float* __restrict__ res,
                                      const float* __restrict__ gamma, const float* __restrict__ beta,
                                      float* __restrict__ out, int64_t rows, int D, float eps) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
    if (row >= rows) return;
    const T* xr = x + row * D;
    const float4* rr = res ? reinterpret_cast<const float4*>(res + row * D) : nullptr;
    const int nv = D >> 2;
    float sum = 0.f;
    for (int i = lane; i < nv; i += 32) {
        float4 v = load_feat4(xr + 4 * i);
        if (rr) {
            const float4 r = rr[i];
            v.x += r.x; v.y += r.y; v.z += r.z; v.w += r.w;
        }
        sum += (v.x + v.y) + (v.z + v.w);
    }
    const float mean = warp_sum(sum) / (float)D;
    float sq = 0.f;
    for (int i = lane; i < nv; i += 32) {
        float4 v = load_feat4(xr + 4 * i);
        if (rr) {
            const float4 r = rr[i];
            v.x += r.x; v.y += r.y; v.z += r.z; v.w += r.w;
        }
        const float a = v.x - mean, b = v.y - mean, c = v.z - mean, d = v.w - mean;
        sq += (a * a + b * b) + (c * c + d * d);
    }
    const float rstd = rsqrtf(warp_sum(sq) / (float)D + eps);
    float4* orow = reinterpret_cast<float4*>(out + row * D);
    for (int i = lane; i < nv; i += 32) {
        float4 v = load_feat4(xr + 4 * i);
        if (rr) {
            const float4 r = rr[i];
            v.x += r.x; v.y += r.y; v.z += r.z; v.w += r.w;
        }
        const float4 g = __ldg(reinterpret_cast<const float4*>(gamma) + i);
        const float4 b = __ldg(reinterpret_cast<const float4*>(beta) + i);
        float4 o;
        o.x = (v.x - mean) * rstd * g.x + b.x;
        o.y = (v.y - mean) * rstd * g.y + b.y;
        o.z = (v.z - mean) * rstd * g.z + b.z;
        o.w = (v.w - mean) * rstd * g.w + b.w;
        orow[i] = o;
    }
}

// out = x / (||x||_2 + eps)
template <class T>
__global__ void l2norm_rows_kernel(const T* __restrict__ x, float* __restrict__ out, int64_t rows, int D, float eps) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * kWarpsPerBlock + (threadIdx.x >> 5);
    if (row >= rows) return;
    const T* xr = x + row * D;
    const int nv = D >> 2;
    float sq = 0.f;
    for (int i = lane; i < nv; i += 32) {
        const float4 v = load_feat4(xr + 4 * i);
        sq += (v.x * v.x + v.y * v.y) + (v.z * v.z + v.w * v.w);
    }
    // eps >= 0: x / (||x|| + eps) (utils/basic_utils.py:97-99); eps < 0: x / max(||x||, -eps) = torch F.normalize
    // (run_on_video/cone_localizator.py:127, 131)
    const float nrm = sqrtf(warp_sum(sq));
    const float denom = eps >= 0.f ? nrm + eps : fmaxf(nrm, -eps);
    float4* orow = reinterpret_cast<float4*>(out + row * D);
    for (int i = lane; i < nv; i += 32) {
        const float4 v = load_feat4(xr + 4 * i);
        orow[i] = make_float4(v.x / denom, v.y / denom, v.z / denom, v.w / denom);
    }
}

// PositionEmbeddingSine (cone/position_encoding.py:51-72) for every valid length 0..max_v_l.
// table[len][r][c]: x = min(r+1,len) / (len + 1e-6) * 2pi (fp32 ops as torch does), dim_t = 10000^(2*(c/2)/d),
// even c -> sin(x / dim_t), odd c -> cos.  pow/sin/cos are evaluated in fp64 and rounded once, i.e. the
// correctly rounded value of the fp32 expression the reference evaluates.
__global__ void pos_table_kernel(float* __restrict__ table, int max_v_l, int d) {
    const int64_t total = (int64_t)(max_v_l + 1) * max_v_l * d;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % d);
        const int r = (int)((i / d) % max_v_l);
        const int len = (int)(i / ((int64_t)d * max_v_l));
        const float cum = (float)min(r + 1, len);
        const float denom = __fadd_rn((float)len, 1e-6f);
        const float xe = __fmul_rn(__fdiv_rn(cum, denom), 6.283185307179586f);
        const float expo = __fdiv_rn((float)(2 * (c / 2)), (float)d);
        const float dim_t = (float)pow(10000.0, (double)expo);
        const float v = __fdiv_rn(xe, dim_t);
        table[i] = (c & 1) ? (float)cos((double)v) : (float)sin((double)v);
    }
}

__global__ void gather_window_rows_kernel(const float* __restrict__ vidproj, int64_t n_vid_rows,
                                          const int64_t* __restrict__ vid_base, const float* __restrict__ txtproj,
                                          const int64_t* __restrict__ txt_base, float* __restrict__ src, int64_t B,
                                          int Lv, int Lt, int d4) {
    const int S = Lv + Lt;
    const int64_t total = B * S * d4;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % d4);
        const int64_t row = i / d4;
        const int r = (int)(row % S);
        const int64_t b = row / S;
        const float4* from;
        if (r < Lv) {
            int64_t fr = vid_base[b] + r;
            fr = fr < n_vid_rows ? fr : n_vid_rows - 1;  // rows past the tensor end are masked; never read OOB
            from = reinterpret_cast<const float4*>(vidproj) + fr * d4 + c;
        } else {
            from = reinterpret_cast<const float4*>(txtproj) + (txt_base[b] + (r - Lv)) * d4 + c;
        }
        reinterpret_cast<float4*>(src)[i] = __ldg(from);
    }
}

__global__ void add_pos_rows_kernel(const float* __restrict__ src, const float* __restrict__ pos_table,
                                    const int32_t* __restrict__ vlen, float* __restrict__ out, int64_t B, int Lv, int Lt,
                                    int d4, int table_lv) {
    const int S = Lv + Lt;
    const int64_t total = B * S * d4;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % d4);
        const int64_t row = i / d4;
        const int r = (int)(row % S);
        const int64_t b = row / S;
        float4 v = reinterpret_cast<const float4*>(src)[i];
        if (r < Lv) {
            const float4 p = __ldg(reinterpret_cast<const float4*>(pos_table) +
                                   ((int64_t)vlen[b] * table_lv + r) * d4 + c);
            v.x += p.x; v.y += p.y; v.z += p.z; v.w += p.w;
        }
        reinterpret_cast<float4*>(out)[i] = v;
    }
}

// fp16 GEMM operands from the fp32 residual stream: plain16 = fp16(src), pos16 = fp16(src + pos) (either may be null)
__global__ void add_pos_rows_f16_kernel(const float* __restrict__ src, const float* __restrict__ pos_table,
                                        const int32_t* __restrict__ vlen, __half* __restrict__ plain16,
                                        __half* __restrict__ pos16, int64_t B, int Lv, int Lt, int d4, int table_lv) {
    const int S = Lv + Lt;
    const int64_t total = B * S * d4;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % d4);
        const int64_t row = i / d4;
        const int r = (int)(row % S);
        const int64_t b = row / S;
        float4 v = reinterpret_cast<const float4*>(src)[i];
        if (plain16) {
            __half2 h0 = __floats2half2_rn(v.x, v.y), h1 = __floats2half2_rn(v.z, v.w);
            uint2 u;
            u.x = *reinterpret_cast<uint32_t*>(&h0);
            u.y = *reinterpret_cast<uint32_t*>(&h1);
            reinterpret_cast<uint2*>(plain16)[i] = u;
        }
        if (pos16) {
            if (r < Lv) {
                const float4 p = __ldg(reinterpret_cast<const float4*>(pos_table) + ((int64_t)vlen[b] * table_lv + r) * d4 + c);
                v.x += p.x; v.y += p.y; v.z += p.z; v.w += p.w;
            }
            __half2 h0 = __floats2half2_rn(v.x, v.y), h1 = __floats2half2_rn(v.z, v.w);
            uint2 u;
            u.x = *reinterpret_cast<uint32_t*>(&h0);
            u.y = *reinterpret_cast<uint32_t*>(&h1);
            reinterpret_cast<uint2*>(pos16)[i] = u;
        }
    }
}

// gather straight into the fp16 operand of the first encoder layer: src16 = fp16(projected row)
__global__ void gather_window_rows_f16_kernel(const float* __restrict__ vidproj, int64_t n_vid_rows,
                                              const int64_t* __restrict__ vid_base, const float* __restrict__ txtproj,
                                              const int64_t* __restrict__ txt_base, __half* __restrict__ src16,
                                              __half* __restrict__ src16lo, int64_t B, int Lv, int Lt, int d4) {
    const int S = Lv + Lt;
    const int64_t total = B * S * d4;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % d4);
        const int64_t row = i / d4;
        const int r = (int)(row % S);
        const int64_t b = row / S;
        float4 v;
        if (r < Lv) {
            int64_t fr = vid_base[b] + r;
            fr = fr < n_vid_rows ? fr : n_vid_rows - 1;
            v = __ldg(reinterpret_cast<const float4*>(vidproj) + fr * d4 + c);
        } else {
            v = __ldg(reinterpret_cast<const float4*>(txtproj) + (txt_base[b] + (r - Lv)) * d4 + c);
        }
        __half2 h0 = __floats2half2_rn(v.x, v.y), h1 = __floats2half2_rn(v.z, v.w);
        uint2 u;
        u.x = *reinterpret_cast<uint32_t*>(&h0);
        u.y = *reinterpret_cast<uint32_t*>(&h1);
        reinterpret_cast<uint2*>(src16)[i] = u;
        if (src16lo) {  // lo = fp16(value - hi): the residual stream crosses HBM as hi + lo (enc_tail.cu)
            const float2 f0 = __half22float2(h0), f1 = __half22float2(h1);
            __half2 l0 = __floats2half2_rn(v.x - f0.x, v.y - f0.y), l1 = __floats2half2_rn(v.z - f1.x, v.w - f1.y);
            u.x = *reinterpret_cast<uint32_t*>(&l0);
            u.y = *reinterpret_cast<uint32_t*>(&l1);
            reinterpret_cast<uint2*>(src16lo)[i] = u;
        }
    }
}

// x fp32 -> hi = fp16(x), lo = fp16(x - hi); and back
__global__ void split_hilo_kernel(const float* __restrict__ x, __half* __restrict__ hi, __half* __restrict__ lo, int64_t n4) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (int64_t)gridDim.x * blockDim.x) {
        const float4 v = reinterpret_cast<const float4*>(x)[i];
        __half2 h0 = __floats2half2_rn(v.x, v.y), h1 = __floats2half2_rn(v.z, v.w);
        const float2 f0 = __half22float2(h0), f1 = __half22float2(h1);
        __half2 l0 = __floats2half2_rn(v.x - f0.x, v.y - f0.y), l1 = __floats2half2_rn(v.z - f1.x, v.w - f1.y);
        uint2 u;
        u.x = *reinterpret_cast<uint32_t*>(&h0);
        u.y = *reinterpret_cast<uint32_t*>(&h1);
        reinterpret_cast<uint2*>(hi)[i] = u;
        if (lo) {
            u.x = *reinterpret_cast<uint32_t*>(&l0);
            u.y = *reinterpret_cast<uint32_t*>(&l1);
            reinterpret_cast<uint2*>(lo)[i] = u;
        }
    }
}
__global__ void combine_hilo_kernel(const __half* __restrict__ hi, const __half* __restrict__ lo, float* __restrict__ out,
                                    int64_t n2) {
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n2; i += (int64_t)gridDim.x * blockDim.x) {
        float2 a = __half22float2(reinterpret_cast<const __half2*>(hi)[i]);
        if (lo) {
            const float2 b = __half22float2(reinterpret_cast<const __half2*>(lo)[i]);
            a.x += b.x;
            a.y += b.y;
        }
        reinterpret_cast<float2*>(out)[i] = a;
    }
}

// fp16 rows -> fp16 window rows, 16-byte chunks (the per-frame / per-token projections already exist in fp16)
__global__ void gather_window_rows_h2h_kernel(const uint4* __restrict__ vid16, int64_t n_vid_rows,
                                              const int64_t* __restrict__ vid_base, const uint4* __restrict__ txt16,
                                              const int64_t* __restrict__ txt_base, uint4* __restrict__ src16, int64_t B,
                                              int Lv, int Lt, int d8) {
    const int S = Lv + Lt;
    const int64_t total = B * S * d8;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % d8);
        const int64_t row = i / d8;
        const int r = (int)(row % S);
        const int64_t b = row / S;
        if (r < Lv) {
            int64_t fr = vid_base[b] + r;
            fr = fr < n_vid_rows ? fr : n_vid_rows - 1;
            src16[i] = __ldg(vid16 + fr * d8 + c);
        } else {
            src16[i] = __ldg(txt16 + (txt_base[b] + (r - Lv)) * d8 + c);
        }
    }
}

__global__ void add_row_table_kernel(const float* __restrict__ x, const float* __restrict__ table,
                                     float* __restrict__ out, int64_t rows, int period, int d4) {
    const int64_t total = rows * d4;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % d4);
        const int64_t row = i / d4;
        float4 v = x ? reinterpret_cast<const float4*>(x)[i] : make_float4(0.f, 0.f, 0.f, 0.f);
        const float4 t = __ldg(reinterpret_cast<const float4*>(table) + (row % period) * d4 + c);
        v.x += t.x; v.y += t.y; v.z += t.z; v.w += t.w;
        reinterpret_cast<float4*>(out)[i] = v;
    }
}

__global__ void add_row_table_f16_kernel(const float* __restrict__ x, const float* __restrict__ table,
                                         __half* __restrict__ out, int64_t rows, int period, int d4) {
    const int64_t total = rows * d4;
    for (int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (int64_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % d4);
        const int64_t row = i / d4;
        float4 v = x ? reinterpret_cast<const float4*>(x)[i] : make_float4(0.f, 0.f, 0.f, 0.f);
        const float4 t = __ldg(reinterpret_cast<const float4*>(table) + (row % period) * d4 + c);
        __half2 h0 = __floats2half2_rn(v.x + t.x, v.y + t.y), h1 = __floats2half2_rn(v.z + t.z, v.w + t.w);
        uint2 u;
        u.x = *reinterpret_cast<uint32_t*>(&h0);
        u.y = *reinterpret_cast<uint32_t*>(&h1);
        reinterpret_cast<uint2*>(out)[i] = u;
    }
}

__global__ void fill_window_desc_dense_kernel(int64_t* vid_base, int64_t* txt_base, int32_t* qidx, int64_t B, int Lv,
                                              int Lt) {
    const int64_t b = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (b >= B) return;
    vid_base[b] = b * Lv;
    txt_base[b] = b * Lt;
    qidx[b] = (int32_t)b;
}

__global__ void fill_i32_kernel(int32_t* p, int64_t n, int32_t value) {
    const int64_t i = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (i < n) p[i] = value;
}

inline unsigned grid_for(int64_t total, int block) {
    const int64_t want = cdiv64(total, block);
    const int64_t cap = (int64_t)kNumSMs * 16;  // grid-stride: a few waves of 148 SMs
    return (unsigned)(want < cap ? (want > 0 ? want : 1) : cap);
}

}  // namespace

int layernorm_rows(const void* x, int x_dtype, const float* residual, const float* gamma, const float* beta, float* out,
                   int64_t rows, int D, float eps, cudaStream_t s) {
    return dispatch_feature(x_dtype, [&](auto tag) {
        using T = std::remove_const_t<std::remove_pointer_t<decltype(tag)>>;
        if (rows == 0) return CONE_OK;
        CONE_REQUIRE((D & 3) == 0, "layernorm: D must be a multiple of 4");
        ProfScope ps(s, P_LAYERNORM, 0.0, ((residual ? 8.0 : 4.0) + sizeof(T)) * (double)rows * D);
        layernorm_rows_kernel<T><<<(unsigned)cdiv64(rows, kWarpsPerBlock), kWarpsPerBlock * 32, 0, s>>>(
            static_cast<const T*>(x), residual, gamma, beta, out, rows, D, eps);
        CONE_LAUNCH_CHECK("layernorm_rows");
        return CONE_OK;
    });
}

int l2norm_rows(const void* x, int x_dtype, float* out, int64_t rows, int D, float eps, cudaStream_t s) {
    return dispatch_feature(x_dtype, [&](auto tag) {
        using T = std::remove_const_t<std::remove_pointer_t<decltype(tag)>>;
        if (rows == 0) return CONE_OK;
        CONE_REQUIRE((D & 3) == 0, "l2norm: D must be a multiple of 4");
        ProfScope ps(s, P_LAYERNORM, 0.0, (4.0 + sizeof(T)) * (double)rows * D);
        l2norm_rows_kernel<T><<<(unsigned)cdiv64(rows, kWarpsPerBlock), kWarpsPerBlock * 32, 0, s>>>(
            static_cast<const T*>(x), out, rows, D, eps);
        CONE_LAUNCH_CHECK("l2norm_rows");
        return CONE_OK;
    });
}

int build_pos_table(float* table, int max_v_l, int d, cudaStream_t s) {
    const int64_t total = (int64_t)(max_v_l + 1) * max_v_l * d;
    pos_table_kernel<<<grid_for(total, 256), 256, 0, s>>>(table, max_v_l, d);
    CONE_LAUNCH_CHECK("pos_table");
    return CONE_OK;
}

int gather_window_rows(const float* vidproj, int64_t n_vid_rows, const int64_t* vid_base, const float* txtproj,
                       const int64_t* txt_base, float* src, int64_t B, int Lv, int Lt, int d, cudaStream_t s) {
    if (B == 0) return CONE_OK;
    ProfScope ps(s, P_ROWOPS, 0.0, 8.0 * (double)B * (Lv + Lt) * d);
    gather_window_rows_kernel<<<grid_for(B * (Lv + Lt) * (d / 4), 256), 256, 0, s>>>(vidproj, n_vid_rows, vid_base,
                                                                                   txtproj, txt_base, src, B, Lv, Lt,
                                                                                   d / 4);
    CONE_LAUNCH_CHECK("gather_window_rows");
    return CONE_OK;
}

int add_pos_rows(const float* src, const float* pos_table, const int32_t* vlen, float* out, int64_t B, int Lv, int Lt,
                 int d, int table_lv, cudaStream_t s) {
    if (B == 0) return CONE_OK;
    ProfScope ps(s, P_ROWOPS, 0.0, 8.0 * (double)B * (Lv + Lt) * d);
    add_pos_rows_kernel<<<grid_for(B * (Lv + Lt) * (d / 4), 256), 256, 0, s>>>(src, pos_table, vlen, out, B, Lv, Lt,
                                                                             d / 4, table_lv);
    CONE_LAUNCH_CHECK("add_pos_rows");
    return CONE_OK;
}

int add_pos_rows_f16(const float* src, const float* pos_table, const int32_t* vlen, uint16_t* plain16, uint16_t* pos16,
                     int64_t B, int Lv, int Lt, int d, int table_lv, cudaStream_t s) {
    if (B == 0) return CONE_OK;
    ProfScope ps(s, P_ROWOPS, 0.0, (4.0 + (plain16 ? 2.0 : 0.0) + (pos16 ? 2.0 : 0.0)) * (double)B * (Lv + Lt) * d);
    add_pos_rows_f16_kernel<<<grid_for(B * (Lv + Lt) * (d / 4), 256), 256, 0, s>>>(
        src, pos_table, vlen, reinterpret_cast<__half*>(plain16), reinterpret_cast<__half*>(pos16), B, Lv, Lt, d / 4, table_lv);
    CONE_LAUNCH_CHECK("add_pos_rows_f16");
    return CONE_OK;
}

int gather_window_rows_f16(const float* vidproj, int64_t n_vid_rows, const int64_t* vid_base, const float* txtproj,
                           const int64_t* txt_base, uint16_t* src16, int64_t B, int Lv, int Lt, int d, cudaStream_t s,
                           uint16_t* src16lo) {
    if (B == 0) return CONE_OK;
    ProfScope ps(s, P_ROWOPS, 0.0, (src16lo ? 8.0 : 6.0) * (double)B * (Lv + Lt) * d);
    gather_window_rows_f16_kernel<<<grid_for(B * (Lv + Lt) * (d / 4), 256), 256, 0, s>>>(
        vidproj, n_vid_rows, vid_base, txtproj, txt_base, reinterpret_cast<__half*>(src16),
        reinterpret_cast<__half*>(src16lo), B, Lv, Lt, d / 4);
    CONE_LAUNCH_CHECK("gather_window_rows_f16");
    return CONE_OK;
}

int split_hilo_rows(const float* x, uint16_t* hi, uint16_t* lo, int64_t n, cudaStream_t s) {
    if (n == 0) return CONE_OK;
    CONE_REQUIRE((n & 3) == 0, "split_hilo_rows: element count must be a multiple of 4");
    ProfScope ps(s, P_CONVERT, 0.0, 8.0 * (double)n);
    split_hilo_kernel<<<grid_for(n / 4, 256), 256, 0, s>>>(x, reinterpret_cast<__half*>(hi), reinterpret_cast<__half*>(lo), n / 4);
    CONE_LAUNCH_CHECK("split_hilo");
    return CONE_OK;
}

int combine_hilo_rows(const uint16_t* hi, const uint16_t* lo, float* out, int64_t n, cudaStream_t s) {
    if (n == 0) return CONE_OK;
    CONE_REQUIRE((n & 1) == 0, "combine_hilo_rows: element count must be even");
    ProfScope ps(s, P_CONVERT, 0.0, 8.0 * (double)n);
    combine_hilo_kernel<<<grid_for(n / 2, 256), 256, 0, s>>>(reinterpret_cast<const __half*>(hi),
                                                            reinterpret_cast<const __half*>(lo), out, n / 2);
    CONE_LAUNCH_CHECK("combine_hilo");
    return CONE_OK;
}

int gather_window_rows_h2h(const uint16_t* vid16, int64_t n_vid_rows, const int64_t* vid_base, const uint16_t* txt16,
                           const int64_t* txt_base, uint16_t* src16, int64_t B, int Lv, int Lt, int d, cudaStream_t s) {
    if (B == 0) return CONE_OK;
    CONE_REQUIRE((d & 7) == 0, "gather_window_rows_h2h: d must be a multiple of 8");
    ProfScope ps(s, P_ROWOPS, 0.0, 4.0 * (double)B * (Lv + Lt) * d);
    gather_window_rows_h2h_kernel<<<grid_for(B * (Lv + Lt) * (d / 8), 256), 256, 0, s>>>(
        reinterpret_cast<const uint4*>(vid16), n_vid_rows, vid_base, reinterpret_cast<const uint4*>(txt16), txt_base,
        reinterpret_cast<uint4*>(src16), B, Lv, Lt, d / 8);
    CONE_LAUNCH_CHECK("gather_window_rows_h2h");
    return CONE_OK;
}

int add_row_table(const float* x, const float* table, float* out, int64_t rows, int period, int d, cudaStream_t s) {
    if (rows == 0) return CONE_OK;
    ProfScope ps(s, P_ROWOPS, 0.0, 8.0 * (double)rows * d);
    add_row_table_kernel<<<grid_for(rows * (d / 4), 256), 256, 0, s>>>(x, table, out, rows, period, d / 4);
    CONE_LAUNCH_CHECK("add_row_table");
    return CONE_OK;
}

int add_row_table_f16(const float* x, const float* table, uint16_t* out16, int64_t rows, int period, int d, cudaStream_t s) {
    if (rows == 0) return CONE_OK;
    ProfScope ps(s, P_ROWOPS, 0.0, 6.0 * (double)rows * d);
    add_row_table_f16_kernel<<<grid_for(rows * (d / 4), 256), 256, 0, s>>>(x, table, reinterpret_cast<__half*>(out16), rows,
                                                                          period, d / 4);
    CONE_LAUNCH_CHECK("add_row_table_f16");
    return CONE_OK;
}

int fill_window_desc_dense(int64_t* vid_base, int64_t* txt_base, int32_t* qidx, int64_t B, int Lv, int Lt,
                           cudaStream_t s) {
    if (B == 0) return CONE_OK;
    fill_window_desc_dense_kernel<<<(unsigned)cdiv64(B, 256), 256, 0, s>>>(vid_base, txt_base, qidx, B, Lv, Lt);
    CONE_LAUNCH_CHECK("fill_window_desc_dense");
    return CONE_OK;
}

int fill_i32(int32_t* p, int64_t n, int32_t value, cudaStream_t s) {
    if (n == 0) return CONE_OK;
    fill_i32_kernel<<<(unsigned)cdiv64(n, 256), 256, 0, s>>>(p, n, value);
    CONE_LAUNCH_CHECK("fill_i32");
    return CONE_OK;
}

}  // namespace cone
