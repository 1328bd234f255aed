// fp32 CUDA-core GEMMs (parity mode, CONE_PREC_FP32): C = epi(A * W^T), A [M,K] and W [N,K] both K-major.
// 128x128x16 CTA tile, 256 threads, 8x8 register micro-tile split as 2x2 blocks of 4x4 so that shared-memory
// reads are conflict-free float4s; global loads are float4 along K; one __syncthreads per k-tile (register
// prefetch + double-buffered shared memory).
#include "kernels.h"

namespace cone {

namespace {

constexpr int BM = 128, BN = 128, BK = 16, NTHREADS = 256;

struct TileArgs {
    const float* A;
    int64_t lda;
    const float* W;
    int64_t ldw;
    float* C;
    int64_t ldc;
    const float* bias;
    const float* R;
    int64_t ldr;
    int64_t M;
    int N, K, relu;
};

// kRowOffsets = false: row m of C starts at C + m * ldc.  true: at C + row_off[m] (ldc unused), and each row takes the
// float4 epilogue only where its own start is 16-byte aligned.
template <bool kRowOffsets>
__device__ __forceinline__ void sgemm_tile(const TileArgs& p, int64_t m0, int n0, const int64_t* row_off = nullptr) {
    __shared__ __align__(16) float As[2][BK][BM + 4];
    __shared__ __align__(16) float Ws[2][BK][BN + 4];
    const int tid = threadIdx.x;
    const int tx = tid & 15, ty = tid >> 4;
    const int lrow = tid >> 2;       // 0..63
    const int lk = (tid & 3) * 4;    // 0,4,8,12

    float acc[8][8];
#pragma unroll
    for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;

    float4 ra[2], rw[2];
    auto gload = [&](int k0) {
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const int row = lrow + 64 * i;
            const int64_t gm = m0 + row;
            const int gn = n0 + row;
            const bool kin = (k0 + lk) < p.K;
            ra[i] = (gm < p.M && kin) ? __ldg(reinterpret_cast<const float4*>(p.A + gm * p.lda + k0 + lk))
                                      : make_float4(0.f, 0.f, 0.f, 0.f);
            rw[i] = (gn < p.N && kin) ? __ldg(reinterpret_cast<const float4*>(p.W + (int64_t)gn * p.ldw + k0 + lk))
                                      : make_float4(0.f, 0.f, 0.f, 0.f);
        }
    };
    auto sstore = [&](int buf) {
#pragma unroll
        for (int i = 0; i < 2; ++i) {
            const int row = lrow + 64 * i;
            As[buf][lk + 0][row] = ra[i].x;
            As[buf][lk + 1][row] = ra[i].y;
            As[buf][lk + 2][row] = ra[i].z;
            As[buf][lk + 3][row] = ra[i].w;
            Ws[buf][lk + 0][row] = rw[i].x;
            Ws[buf][lk + 1][row] = rw[i].y;
            Ws[buf][lk + 2][row] = rw[i].z;
            Ws[buf][lk + 3][row] = rw[i].w;
        }
    };

    const int nk = (p.K + BK - 1) / BK;
    gload(0);
    sstore(0);
    __syncthreads();
    for (int kt = 0; kt < nk; ++kt) {
        const int buf = kt & 1;
        if (kt + 1 < nk) gload((kt + 1) * BK);
#pragma unroll
        for (int k = 0; k < BK; ++k) {
            const float4 a0 = *reinterpret_cast<const float4*>(&As[buf][k][ty * 4]);
            const float4 a1 = *reinterpret_cast<const float4*>(&As[buf][k][64 + ty * 4]);
            const float4 w0 = *reinterpret_cast<const float4*>(&Ws[buf][k][tx * 4]);
            const float4 w1 = *reinterpret_cast<const float4*>(&Ws[buf][k][64 + tx * 4]);
            const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
            const float w[8] = {w0.x, w0.y, w0.z, w0.w, w1.x, w1.y, w1.z, w1.w};
#pragma unroll
            for (int i = 0; i < 8; ++i)
#pragma unroll
                for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], w[j], acc[i][j]);
        }
        if (kt + 1 < nk) sstore(buf ^ 1);
        __syncthreads();
    }

    // epilogue: bias -> residual -> relu
    const bool r_ok = p.R == nullptr || (((p.ldr & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.R) & 15) == 0));
    const bool vec_all = ((p.ldc & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.C) & 15) == 0) &&
                         (p.R == nullptr || (((p.ldr & 3) == 0) && ((reinterpret_cast<uintptr_t>(p.R) & 15) == 0)));
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        const int64_t m = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
        if (m >= p.M) continue;
        float* crow;
        bool vec_ok;
        if constexpr (kRowOffsets) {
            crow = p.C + row_off[m];
            vec_ok = ((reinterpret_cast<uintptr_t>(crow) & 15) == 0) && r_ok;
        } else {
            crow = p.C + m * p.ldc;
            vec_ok = vec_all;
        }
#pragma unroll
        for (int jb = 0; jb < 2; ++jb) {
            const int n = n0 + (jb == 0 ? tx * 4 : 64 + tx * 4);
            if (n >= p.N) continue;
            float v[4] = {acc[i][jb * 4 + 0], acc[i][jb * 4 + 1], acc[i][jb * 4 + 2], acc[i][jb * 4 + 3]};
            if (vec_ok && n + 3 < p.N) {
                if (p.bias) {
                    const float4 b = __ldg(reinterpret_cast<const float4*>(p.bias + n));
                    v[0] += b.x; v[1] += b.y; v[2] += b.z; v[3] += b.w;
                }
                if (p.R) {
                    const float4 r = *reinterpret_cast<const float4*>(p.R + m * p.ldr + n);
                    v[0] += r.x; v[1] += r.y; v[2] += r.z; v[3] += r.w;
                }
                if (p.relu) {
#pragma unroll
                    for (int t = 0; t < 4; ++t) v[t] = fmaxf(v[t], 0.f);
                }
                *reinterpret_cast<float4*>(crow + n) = make_float4(v[0], v[1], v[2], v[3]);
            } else {
#pragma unroll
                for (int t = 0; t < 4; ++t) {
                    if (n + t >= p.N) break;
                    float x = v[t];
                    if (p.bias) x += __ldg(p.bias + n + t);
                    if (p.R) x += p.R[m * p.ldr + n + t];
                    if (p.relu) x = fmaxf(x, 0.f);
                    crow[n + t] = x;
                }
            }
        }
    }
}

__global__ void __launch_bounds__(NTHREADS, 2) sgemm_nt_kernel(TileArgs p) {
    sgemm_tile<false>(p, (int64_t)blockIdx.x * BM, (int)blockIdx.y * BN);
}

// one z-slice per video: A = the video's query CLS rows, W = the video's context frames
__global__ void __launch_bounds__(NTHREADS, 2)
frame_scores_kernel(const float* __restrict__ ctx, const float* __restrict__ cls, int K,
                    const int64_t* __restrict__ video_offsets, const int32_t* __restrict__ q_first,
                    float* __restrict__ score, const int64_t* __restrict__ score_offsets) {
    const int v = blockIdx.z;
    const int q0 = q_first[v], q1 = q_first[v + 1];
    const int64_t f0 = video_offsets[v], f1 = video_offsets[v + 1];
    const int M = q1 - q0;
    const int N = (int)(f1 - f0);
    const int64_t m0 = (int64_t)blockIdx.y * BM;
    const int n0 = blockIdx.x * BN;
    if (m0 >= M || n0 >= N) return;
    TileArgs p;
    p.A = cls + (int64_t)q0 * K;
    p.lda = K;
    p.W = ctx + f0 * K;
    p.ldw = K;
    p.C = score;
    p.ldc = 0;
    p.bias = nullptr;
    p.R = nullptr;
    p.ldr = 0;
    p.M = M;
    p.N = N;
    p.K = K;
    p.relu = 0;
    sgemm_tile<true>(p, m0, n0, score_offsets + q0);  // query q's N scores start at score_offsets[q]
}

// tiny-N linear heads: one warp per row
template <int MAXN>
__global__ void rowdot_small_kernel(const float* __restrict__ x, int64_t ldx, const float* __restrict__ W,
                                    const float* __restrict__ bias, float* __restrict__ out, int64_t rows, int N, int K,
                                    int mode, int group_out, int group_in) {
    const int lane = threadIdx.x & 31;
    const int64_t row = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (row >= rows) return;
    // optional row remap: output row r reads input row (r / group_out) * group_in + r % group_out
    const int64_t xrow = group_out > 0 ? (row / group_out) * group_in + (row % group_out) : row;
    float acc[MAXN];
#pragma unroll
    for (int n = 0; n < MAXN; ++n) acc[n] = 0.f;
    const float* xr = x + xrow * ldx;
    for (int k = lane * 4; k < K; k += 128) {
        const float4 xv = *reinterpret_cast<const float4*>(xr + k);
#pragma unroll
        for (int n = 0; n < MAXN; ++n) {
            if (n < N) {
                const float4 wv = __ldg(reinterpret_cast<const float4*>(W + (int64_t)n * K + k));
                acc[n] = fmaf(xv.x, wv.x, acc[n]);
                acc[n] = fmaf(xv.y, wv.y, acc[n]);
                acc[n] = fmaf(xv.z, wv.z, acc[n]);
                acc[n] = fmaf(xv.w, wv.w, acc[n]);
            }
        }
    }
#pragma unroll
    for (int n = 0; n < MAXN; ++n) {
        acc[n] = warp_sum(acc[n]);
        if (bias != nullptr && n < N) acc[n] += __ldg(bias + n);
    }
    if (lane != 0) return;
    if (mode == 0) {
        for (int n = 0; n < N; ++n) out[row * N + n] = acc[n];
    } else if (mode == 1) {
        for (int n = 0; n < N; ++n) out[row * N + n] = 1.f / (1.f + expf(-acc[n]));
    } else {
        float mx = acc[0];
        for (int n = 1; n < N; ++n) mx = fmaxf(mx, acc[n]);
        float sum = 0.f;
        float e[MAXN];
        for (int n = 0; n < N; ++n) {
            e[n] = expf(acc[n] - mx);
            sum += e[n];
        }
        if (mode == 2) {
            out[row] = e[0] / sum;
        } else {
            for (int n = 0; n < N; ++n) out[row * N + n] = e[n] / sum;
        }
    }
}

}  // namespace

int sgemm_nt(const GemmParams& g, cudaStream_t s) {
    if (g.M == 0 || g.N == 0) return CONE_OK;
    CONE_REQUIRE((g.K & 3) == 0 && (g.lda & 3) == 0 && (g.ldw & 3) == 0, "sgemm_nt: K/lda/ldw must be multiples of 4");
    CONE_REQUIRE(((reinterpret_cast<uintptr_t>(g.A) | reinterpret_cast<uintptr_t>(g.W)) & 15) == 0,
                 "sgemm_nt: operands must be 16-byte aligned");
    TileArgs p{g.A, g.lda, g.W, g.ldw, g.C, g.ldc, g.bias, g.R, g.ldr, g.M, g.N, g.K, g.relu};
    dim3 grid((unsigned)cdiv64(g.M, BM), (unsigned)cdiv(g.N, BN), 1);
    ProfScope ps(s, P_GEMM_FP32, 2.0 * (double)g.M * g.N * g.K, 4.0 * ((double)g.M * g.K + (double)g.N * g.K + (double)g.M * g.N));
    sgemm_nt_kernel<<<grid, NTHREADS, 0, s>>>(p);
    CONE_LAUNCH_CHECK("sgemm_nt");
    return CONE_OK;
}

int sgemm_frame_scores(const float* ctx, const float* cls, int K, const int64_t* video_offsets, const int32_t* q_first,
                       int n_videos, int max_video_frames, int max_video_queries, float* score,
                       const int64_t* score_offsets, cudaStream_t s) {
    if (n_videos == 0 || max_video_frames == 0 || max_video_queries == 0) return CONE_OK;
    CONE_REQUIRE((K & 3) == 0, "frame_scores: feature dim must be a multiple of 4");
    CONE_REQUIRE(n_videos <= 65535, "frame_scores: at most 65535 videos per call");
    dim3 grid((unsigned)cdiv(max_video_frames, BN), (unsigned)cdiv(max_video_queries, BM), (unsigned)n_videos);
    ProfScope ps(s, P_SCORES);
    frame_scores_kernel<<<grid, NTHREADS, 0, s>>>(ctx, cls, K, video_offsets, q_first, score, score_offsets);
    CONE_LAUNCH_CHECK("frame_scores");
    return CONE_OK;
}

int rowdot_small(const float* x, int64_t ldx, const float* W, const float* bias, float* out, int64_t rows, int N, int K,
                 int mode, cudaStream_t s, int group_out, int group_in) {
    if (rows == 0) return CONE_OK;
    CONE_REQUIRE(N >= 1 && N <= 8 && (K & 3) == 0 && (ldx & 3) == 0, "rowdot_small: unsupported shape N=%d K=%d", N, K);
    const int warps = 8;
    ProfScope ps(s, P_ROWOPS);
    rowdot_small_kernel<8><<<(unsigned)cdiv64(rows, warps), warps * 32, 0, s>>>(x, ldx, W, bias, out, rows, N, K, mode,
                                                                                        group_out, group_in);
    CONE_LAUNCH_CHECK("rowdot_small");
    return CONE_OK;
}

}  // namespace cone
