// Small-sequence multi-head attention for Moment-DETR windows (S = Lv + Lt <= 512 rows, head_dim 32).  Windows of up
// to 256 rows run the kernels sized for them; longer windows (256 < S <= 512) run the long-window variants below.
// Math follows torch.nn.functional.multi_head_attention_forward as called at cone/transformer.py:239,
// 304, 308: q scaled by sqrt(1/head_dim) BEFORE the dot product, additive -inf key-padding mask,
// softmax over keys, then P.V.  One CTA per (window, head); K and V of the head live in shared memory.
#include <cuda_fp16.h>
#include <math_constants.h>

#include "kernels.h"

namespace cone {

namespace {

constexpr int HD = 32;            // head dim (hidden 256 / 8 heads)
constexpr int MAX_S = 256;        // max keys per window of the short-window kernels
constexpr int MAX_S_LONG = 512;   // max keys per window of the long-window variants
constexpr int ENC_WARPS = 4;

__device__ __forceinline__ float fast_exp2(float x) {
    float y;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
    return y;
}

__device__ __forceinline__ bool key_valid(int j, int Lv, int vl, int tl) { return j < Lv ? (j < vl) : ((j - Lv) < tl); }

// KPL = keys per lane: MAX_S / 32, or MAX_S_LONG / 32 for long windows
template <int KPL>
__global__ void __launch_bounds__(ENC_WARPS * 32)
enc_self_attention_kernel(const float* __restrict__ qk, int64_t ldqk, const float* __restrict__ v, int64_t ldv,
                          float* __restrict__ o, int64_t ldo, const int32_t* __restrict__ vlen,
                          const int32_t* __restrict__ tlen, int Lv, int Lt, int d_model) {
    extern __shared__ float smem[];
    const int S = Lv + Lt;
    float* Ks = smem;                        // [S][HD+1]
    float* Vs = Ks + S * (HD + 1);           // [S][HD]
    float* Qs = Vs + S * HD;                 // [ENC_WARPS][HD]
    float* Ps = Qs + ENC_WARPS * HD;         // [ENC_WARPS][S]
    const int64_t b = blockIdx.x;
    const int h = blockIdx.y;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int vl = vlen[b], tl = tlen[b];
    const int64_t row0 = b * S;
    const float scale = 0.17677669529663687f;  // sqrt(1/32), as torch scales q

    for (int i = threadIdx.x; i < S * HD; i += blockDim.x) {
        const int j = i / HD, c = i % HD;
        Ks[j * (HD + 1) + c] = qk[(row0 + j) * ldqk + d_model + h * HD + c];
        Vs[j * HD + c] = v[(row0 + j) * ldv + h * HD + c];
    }
    __syncthreads();

    for (int i = warp; i < S; i += ENC_WARPS) {
        Qs[warp * HD + lane] = qk[(row0 + i) * ldqk + h * HD + lane] * scale;
        __syncwarp();
        float sc[KPL];
        float mx = -CUDART_INF_F;
#pragma unroll
        for (int t = 0; t < KPL; ++t) {
            const int j = lane + 32 * t;
            float a = -CUDART_INF_F;
            if (j < S && key_valid(j, Lv, vl, tl)) {
                a = 0.f;
#pragma unroll
                for (int c = 0; c < HD; ++c) a = fmaf(Qs[warp * HD + c], Ks[j * (HD + 1) + c], a);
            }
            sc[t] = a;
            mx = fmaxf(mx, a);
        }
        mx = warp_max(mx);
        float sum = 0.f;
#pragma unroll
        for (int t = 0; t < KPL; ++t) {
            const int j = lane + 32 * t;
            const float e = (sc[t] == -CUDART_INF_F) ? 0.f : expf(sc[t] - mx);
            if (j < S) Ps[warp * S + j] = e;
            sum += e;
        }
        sum = warp_sum(sum);
        __syncwarp();
        float acc = 0.f;
        for (int j = 0; j < S; ++j) acc = fmaf(Ps[warp * S + j], Vs[j * HD + lane], acc);
        // all keys masked (cannot happen for real windows) -> 0/0 = NaN, like torch's softmax of all -inf
        o[(row0 + i) * ldo + h * HD + lane] = acc / sum;
        __syncwarp();
    }
}

// decoder self-attention: nq <= 8 slots, one warp per (window, head), lane = channel.  T = float (parity mode) or
// __half (tensor-core mode: q|k|v come from fp16 GEMM outputs and the result feeds an fp16 GEMM operand)
__device__ __forceinline__ float ld_f32(const float* p) { return *p; }
__device__ __forceinline__ float ld_f32(const __half* p) { return __half2float(*p); }
__device__ __forceinline__ void st_f32(float* p, float v) { *p = v; }
__device__ __forceinline__ void st_f32(__half* p, float v) { *p = __float2half_rn(v); }

template <typename T>
__global__ void dec_self_attention_kernel(const T* __restrict__ qk, int64_t ldqk, const T* __restrict__ v,
                                          int64_t ldv, T* __restrict__ o, int64_t ldo, int64_t B, int nq,
                                          int nheads, int d_model) {
    const int lane = threadIdx.x & 31;
    const int64_t wid = (int64_t)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
    if (wid >= B * nheads) return;
    const int64_t b = wid / nheads;
    const int h = (int)(wid % nheads);
    const float scale = 0.17677669529663687f;
    float q[8], k[8], vv[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        if (i < nq) {
            const int64_t row = b * nq + i;
            q[i] = ld_f32(qk + row * ldqk + h * HD + lane) * scale;
            k[i] = ld_f32(qk + row * ldqk + d_model + h * HD + lane);
            vv[i] = ld_f32(v + row * ldv + h * HD + lane);
        } else {
            q[i] = k[i] = vv[i] = 0.f;
        }
    }
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        if (i >= nq) break;
        float sc[8];
        float mx = -CUDART_INF_F;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            if (j < nq) {
                sc[j] = warp_sum(q[i] * k[j]);
                mx = fmaxf(mx, sc[j]);
            }
        }
        float sum = 0.f, acc = 0.f;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            if (j < nq) {
                const float e = expf(sc[j] - mx);
                sum += e;
                acc = fmaf(e, vv[j], acc);
            }
        }
        st_f32(o + (b * nq + i) * ldo + h * HD + lane, acc / sum);
    }
}

// decoder cross-attention: one warp per (window, head); nq <= 8 queries against S memory keys
__device__ __forceinline__ void load_head_row(const float* p, float* out) {
#pragma unroll
    for (int c = 0; c < HD / 4; ++c) {
        const float4 t = reinterpret_cast<const float4*>(p)[c];
        out[4 * c] = t.x; out[4 * c + 1] = t.y; out[4 * c + 2] = t.z; out[4 * c + 3] = t.w;
    }
}
__device__ __forceinline__ void load_head_row(const __half* p, float* out) {
#pragma unroll
    for (int c = 0; c < HD / 8; ++c) {
        const uint4 t = reinterpret_cast<const uint4*>(p)[c];
        const __half2* h = reinterpret_cast<const __half2*>(&t);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const float2 f = __half22float2(h[e]);
            out[8 * c + 2 * e] = f.x;
            out[8 * c + 2 * e + 1] = f.y;
        }
    }
}
__device__ __forceinline__ float to_f32(float x) { return x; }
__device__ __forceinline__ float to_f32(__half x) { return __half2float(x); }

// One CTA per window, 8 warps, K / V read straight from global memory with every load of a batch of rows in flight
// before the first is consumed (the earlier versions — one warp per (window, head), then one thread per (key, head) —
// waited for one memory round trip per row and ran at 5x their HBM time).
//   lane = (head h = lane / 4, part = lane % 4): the lane owns dims [8 part, 8 part + 8) of head h, so the 32 lanes of
//   a warp read one whole 256-wide K (or V) row per instruction, fully coalesced; warp w takes rows w, w + 8, ...
//   1. scores: the lane's slice of the nq scaled queries lives in registers; partial dot products are reduced over the
//      4 lanes of a head with two shuffles; rows are processed XB at a time
//   2. masked softmax per (head, slot) row: one warp per row of the score matrix in shared memory
//   3. P.V: each lane accumulates its 8 channels over its warp's rows (VB rows in flight), then the 8 warps' partial
//      sums are added through shared memory
template <typename KV>
struct XChunk;  // 8 consecutive elements of a K / V row
template <>
struct XChunk<__half> {
    uint4 v;
    __device__ __forceinline__ void load(const __half* p) { v = *reinterpret_cast<const uint4*>(p); }
    __device__ __forceinline__ void to_float(float* o) const {
        const __half2* h = reinterpret_cast<const __half2*>(&v);
#pragma unroll
        for (int e = 0; e < 4; ++e) {
            const float2 f = __half22float2(h[e]);
            o[2 * e] = f.x;
            o[2 * e + 1] = f.y;
        }
    }
};
template <>
struct XChunk<float> {
    float4 a, b;
    __device__ __forceinline__ void load(const float* p) {
        a = reinterpret_cast<const float4*>(p)[0];
        b = reinterpret_cast<const float4*>(p)[1];
    }
    __device__ __forceinline__ void to_float(float* o) const {
        o[0] = a.x; o[1] = a.y; o[2] = a.z; o[3] = a.w;
        o[4] = b.x; o[5] = b.y; o[6] = b.z; o[7] = b.w;
    }
};

// KPL = scores per lane in phase 2: MAX_S / 32, or MAX_S_LONG / 32 for long windows
template <typename KV, int NQ, int KPL>
__global__ void __launch_bounds__(256, 2)
dec_cross_attention_kernel(const float* __restrict__ q, int64_t ldq, const KV* __restrict__ k, int64_t ldk,
                           const KV* __restrict__ v, int64_t ldv, float* __restrict__ o, int64_t ldo,
                           const int32_t* __restrict__ vlen, const int32_t* __restrict__ tlen, int nq, int Lv,
                           int Lt, const float* __restrict__ posk, int64_t ldposk, int table_lv) {
    constexpr int H = 8;
    constexpr int XB = sizeof(KV) == 2 ? 6 : 3;  // rows in flight per warp, phase 1 (K chunk + 2 position float4 each)
    constexpr int VB = sizeof(KV) == 2 ? 10 : 5; // rows in flight per warp, phase 3
    extern __shared__ __align__(16) float xsmem[];
    const int S = Lv + Lt;
    const int Sp = (S + 3) & ~3;
    float* Ps = xsmem;                   // [H][NQ][Sp]
    float* inv = Ps + H * NQ * Sp;       // [H][NQ]
    float* red = inv + H * NQ;           // [8 warps][NQ * 8][32 lanes]
    const int64_t b = blockIdx.x;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const int h = lane >> 2, part = lane & 3;
    const int col = h * HD + part * 8;   // this lane's 8 columns of a 256-wide row
    const float scale = 0.17677669529663687f;
    float qv[NQ][8];
#pragma unroll
    for (int s = 0; s < NQ; ++s) {
        if (s < nq) {
            const float4 a = *reinterpret_cast<const float4*>(q + (b * nq + s) * ldq + col);
            const float4 c = *reinterpret_cast<const float4*>(q + (b * nq + s) * ldq + col + 4);
            qv[s][0] = a.x * scale; qv[s][1] = a.y * scale; qv[s][2] = a.z * scale; qv[s][3] = a.w * scale;
            qv[s][4] = c.x * scale; qv[s][5] = c.y * scale; qv[s][6] = c.z * scale; qv[s][7] = c.w * scale;
        } else {
#pragma unroll
            for (int e = 0; e < 8; ++e) qv[s][e] = 0.f;
        }
    }
    const int vl = vlen[b], tl = tlen[b];
    // phase 1
    for (int base = warp; base < S; base += 8 * XB) {
        XChunk<KV> kc[XB];
        float4 p0[XB], p1[XB];
#pragma unroll
        for (int r = 0; r < XB; ++r) {
            const int j = base + 8 * r;
            p0[r] = make_float4(0.f, 0.f, 0.f, 0.f);
            p1[r] = p0[r];
            if (j < S) {
                kc[r].load(k + (b * S + j) * ldk + col);
                if (posk != nullptr && j < Lv) {  // k = memory Wk^T + bk + pos Wk^T (table row of (valid length, j))
                    const float4* pr = reinterpret_cast<const float4*>(posk + ((int64_t)vl * table_lv + j) * ldposk + col);
                    p0[r] = __ldg(pr);
                    p1[r] = __ldg(pr + 1);
                }
            }
        }
#pragma unroll
        for (int r = 0; r < XB; ++r) {
            const int j = base + 8 * r;
            if (j < S) {  // warp-uniform
                float kr[8];
                kc[r].to_float(kr);
                kr[0] += p0[r].x; kr[1] += p0[r].y; kr[2] += p0[r].z; kr[3] += p0[r].w;
                kr[4] += p1[r].x; kr[5] += p1[r].y; kr[6] += p1[r].z; kr[7] += p1[r].w;
                const bool ok = key_valid(j, Lv, vl, tl);
#pragma unroll
                for (int s = 0; s < NQ; ++s) {
                    float a = 0.f;
#pragma unroll
                    for (int e = 0; e < 8; ++e) a = fmaf(qv[s][e], kr[e], a);
                    a += __shfl_xor_sync(0xffffffffu, a, 1);
                    a += __shfl_xor_sync(0xffffffffu, a, 2);
                    if ((s & 3) == part) Ps[(h * NQ + s) * Sp + j] = ok ? a : -CUDART_INF_F;
                }
            }
        }
    }
    __syncthreads();
    // phase 2: each lane keeps its (at most 8) scores of the row in registers
    for (int r = warp; r < H * NQ; r += 8) {
        float* row = Ps + r * Sp;
        float a[KPL];
        float mx = -CUDART_INF_F;
#pragma unroll
        for (int t = 0; t < KPL; ++t) {
            const int j = lane + 32 * t;
            a[t] = j < S ? row[j] : -CUDART_INF_F;
            mx = fmaxf(mx, a[t]);
        }
        mx = warp_max(mx);
        float sum = 0.f;
#pragma unroll
        for (int t = 0; t < KPL; ++t) {
            const int j = lane + 32 * t;
            float e;
            if (sizeof(KV) == 2) {  // reduced-precision mode: exp2 with the hardware approximation (2^-22 relative)
                e = fast_exp2((a[t] - mx) * 1.4426950408889634f);  // exp2(-inf) = 0 for masked keys
            } else {
                e = (a[t] == -CUDART_INF_F) ? 0.f : expf(a[t] - mx);
            }
            if (j < Sp) row[j] = e;  // columns S..Sp-1 become 0
            sum += e;
        }
        sum = warp_sum(sum);
        if (lane == 0) inv[r] = 1.f / sum;  // all keys masked -> NaN, like torch's softmax of all -inf
    }
    __syncthreads();
    // phase 3
    float acc[NQ][8];
#pragma unroll
    for (int s = 0; s < NQ; ++s)
#pragma unroll
        for (int e = 0; e < 8; ++e) acc[s][e] = 0.f;
    for (int base = warp; base < S; base += 8 * VB) {
        XChunk<KV> vc[VB];
#pragma unroll
        for (int r = 0; r < VB; ++r) {
            const int j = base + 8 * r;
            if (j < S) vc[r].load(v + (b * S + j) * ldv + col);
        }
#pragma unroll
        for (int r = 0; r < VB; ++r) {
            const int j = base + 8 * r;
            if (j < S) {
                float vr[8];
                vc[r].to_float(vr);
#pragma unroll
                for (int s = 0; s < NQ; ++s) {
                    const float p = Ps[(h * NQ + s) * Sp + j];
#pragma unroll
                    for (int e = 0; e < 8; ++e) acc[s][e] = fmaf(p, vr[e], acc[s][e]);
                }
            }
        }
    }
#pragma unroll
    for (int s = 0; s < NQ; ++s)
#pragma unroll
        for (int e = 0; e < 8; ++e) red[(warp * NQ * 8 + s * 8 + e) * 32 + lane] = acc[s][e];
    __syncthreads();
    // each warp finishes NQ of the NQ * 8 (slot, element) pairs: lane-contiguous reads, no bank conflicts
    for (int kk = warp * NQ; kk < (warp + 1) * NQ; ++kk) {
        float t = 0.f;
#pragma unroll
        for (int w = 0; w < 8; ++w) t += red[(w * NQ * 8 + kk) * 32 + lane];
        const int s = kk >> 3, e = kk & 7;
        if (s < nq) o[(b * nq + s) * ldo + col + e] = t * inv[h * NQ + s];
    }
}


// ------------------------------------------------------------------------------------------------
// Tensor-core encoder self-attention (CONE_PREC_TC): fp16 Q/K/V, fp32 scores and softmax, fp16 output.
// One CTA per (window, head); Q, K and V^T of the head in shared memory (padded rows: conflict-free fragment
// loads); each warp owns 16-query-row blocks and keeps the whole score row block (16 x S) in registers:
// S = Q.K^T with mma.sync.m16n8k16, masked softmax on the accumulator fragments, P re-used in place as the
// A operand of P.V (FlashAttention-2 register layout).  S <= 8*NB keys.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void mma_16816(float* c, const uint32_t* a, uint32_t b0, uint32_t b1) {
    asm volatile(
        "mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
        : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
        : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t pack_half2(float x, float y) {
    __half2 h = __floats2half2_rn(x, y);
    return *reinterpret_cast<uint32_t*>(&h);
}

constexpr int ATT_WARPS = 5;
constexpr int QK_PAD = 40;  // halves per Q/K/V row in smem (32 + 8): 80-byte stride -> conflict-free ldmatrix rows

__device__ __forceinline__ void ldsm_x4(uint32_t* r, const __half* p) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
                 : "r"((uint32_t)__cvta_generic_to_shared(p)));
}
__device__ __forceinline__ void ldsm_x2(uint32_t& r0, uint32_t& r1, const __half* p) {  // lanes 0-15 supply the row addresses
    asm volatile("ldmatrix.sync.aligned.m8n8.x2.shared.b16 {%0,%1}, [%2];"
                 : "=r"(r0), "=r"(r1)
                 : "r"((uint32_t)__cvta_generic_to_shared(p)));
}
__device__ __forceinline__ void ldsm_x4_trans(uint32_t* r, const __half* p) {
    asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3])
                 : "r"((uint32_t)__cvta_generic_to_shared(p)));
}

// Layer 0 reads q|k|v rows through the window descriptors (frame / token row tables) instead of a per-window copy:
// the projection of a frame or a token does not depend on the window it is sliced into (see api.cu).
struct EncRowSource {
    const __half* frames;      // [n_frames, 3 d] q|k|v of every frame, or null = dense per-window rows
    const __half* tokens;      // [n_tokens, 3 d]
    const int64_t* vid_base;   // [B] first frame row of each window
    const int64_t* txt_base;   // [B] first token row of each window
    int64_t n_frames;
};

// EXACT: the window has exactly NB key blocks (Sp == 8 NB), so none of the per-block range guards is compiled.
template <int NB, bool EXACT>
__global__ void __launch_bounds__(ATT_WARPS * 32, NB <= 20 ? 4 : 2)
enc_attention_f16_kernel(const __half* __restrict__ qk, int64_t ldqk, const __half* __restrict__ v, int64_t ldv,
                         __half* __restrict__ o, int64_t ldo, const int32_t* __restrict__ vlen,
                         const int32_t* __restrict__ tlen, int Lv, int Lt, int d_model,
                         const __half* __restrict__ posqk, int table_lv, EncRowSource src) {
    extern __shared__ __align__(16) unsigned char att_smem[];
    const int S = Lv + Lt;
    const int Sp = (S + 15) & ~15;
    __half* Qs = reinterpret_cast<__half*>(att_smem);  // [Sp][QK_PAD]
    __half* Ks = Qs + Sp * QK_PAD;                      // [Sp][QK_PAD]
    __half* Vs = Ks + Sp * QK_PAD;                      // [Sp][QK_PAD]  (row-major; P.V uses ldmatrix.trans)
    float* mbias = reinterpret_cast<float*>(Vs + Sp * QK_PAD);  // [Sp] additive key-padding mask: 0 or -inf
    // heads are the fast grid index: the 8 heads of a window run together, so both 64-byte halves of every
    // 128-byte line of its q|k|v rows are consumed while the line is in L2 (halves the DRAM reads, ncu-measured)
    const int nheads = d_model / HD;
    const int64_t b = blockIdx.x / nheads;
    const int h = blockIdx.x % nheads;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t row0 = b * S;

    // cooperative load: 4 x 16-byte chunks per row for each of Q, K, V.  The trip count is a compile-time constant
    // and the loads of ALL iterations are issued before anything is consumed, so one round of global-memory
    // latency covers the whole tile (the CTA is short-lived: ncu showed a third of its life in this phase when the
    // loads of each iteration waited for the previous one)
    constexpr int LOAD_ITERS = (NB * 8 * 4 + ATT_WARPS * 32 - 1) / (ATT_WARPS * 32);
    constexpr int ROWS_PER_IT = ATT_WARPS * 32 / 4;  // 4 threads per row: the row of iteration `it` is r0 + it * 40
    uint4 q4[LOAD_ITERS], k4[LOAD_ITERS], v4[LOAD_ITERS];
    const int r0 = threadIdx.x >> 2, c8 = (threadIdx.x & 3) * 8 + h * HD;
    // per-thread base pointers, advanced by a constant per iteration (the 64-bit row arithmetic of the first version
    // was a third of this phase's instructions)
    const bool indirect = src.frames != nullptr;
    const int64_t vbase = indirect ? src.vid_base[b] : 0;
    const int64_t tbase = indirect ? src.txt_base[b] : 0;
    const __half* qp = qk + (row0 + r0) * ldqk + c8;
    const __half* vp = v + (row0 + r0) * ldv + c8;
#pragma unroll
    for (int it = 0; it < LOAD_ITERS; ++it) {
        const int r = r0 + it * ROWS_PER_IT;
        q4[it] = make_uint4(0, 0, 0, 0);
        k4[it] = q4[it];
        v4[it] = q4[it];
        if (r < S) {
            if (indirect) {
                const __half* row;
                if (r < Lv) {
                    int64_t fr = vbase + r;  // rows past the tensor end belong to masked keys: never read out of bounds
                    fr = fr < src.n_frames ? fr : src.n_frames - 1;
                    row = src.frames + fr * (3 * d_model) + c8;
                } else {
                    row = src.tokens + (tbase + (r - Lv)) * (3 * d_model) + c8;
                }
                q4[it] = *reinterpret_cast<const uint4*>(row);
                k4[it] = *reinterpret_cast<const uint4*>(row + d_model);
                v4[it] = *reinterpret_cast<const uint4*>(row + 2 * d_model);
            } else {
                q4[it] = *reinterpret_cast<const uint4*>(qp + (int64_t)it * ROWS_PER_IT * ldqk);
                k4[it] = *reinterpret_cast<const uint4*>(qp + (int64_t)it * ROWS_PER_IT * ldqk + d_model);
                v4[it] = *reinterpret_cast<const uint4*>(vp + (int64_t)it * ROWS_PER_IT * ldv);
            }
        }
    }
    const int vl = vlen[b], tl = tlen[b];
    const __half* pp = posqk + ((int64_t)vl * table_lv + r0) * (2 * d_model) + c8;
    unsigned char* sbase = att_smem + (r0 * QK_PAD + (threadIdx.x & 3) * 8) * 2;  // this thread's chunk of row r0 in Qs
    const int mat_bytes = Sp * QK_PAD * 2;
#pragma unroll
    for (int it = 0; it < LOAD_ITERS; ++it) {
        const int r = r0 + it * ROWS_PER_IT;
        if (r < Sp) {
            if (posqk != nullptr && r < Lv) {
                // q = (src + pos) Wq^T + bq = (src Wq^T + bq) + pos Wq^T: the position term comes from a per-layer
                // table indexed by (valid length, row), so no position-added copy of the activations exists
                const __half* pr = pp + it * ROWS_PER_IT * 2 * d_model;
                const uint4 pq = __ldg(reinterpret_cast<const uint4*>(pr));
                const uint4 pk = __ldg(reinterpret_cast<const uint4*>(pr + d_model));
                __half2* qh = reinterpret_cast<__half2*>(&q4[it]);
                __half2* kh = reinterpret_cast<__half2*>(&k4[it]);
                const __half2* pqh = reinterpret_cast<const __half2*>(&pq);
                const __half2* pkh = reinterpret_cast<const __half2*>(&pk);
#pragma unroll
                for (int e = 0; e < 4; ++e) {  // exact sum of two fp16 values, one rounding
                    qh[e] = __hadd2(qh[e], pqh[e]);
                    kh[e] = __hadd2(kh[e], pkh[e]);
                }
            }
            unsigned char* sp = sbase + it * ROWS_PER_IT * QK_PAD * 2;
            *reinterpret_cast<uint4*>(sp) = q4[it];
            *reinterpret_cast<uint4*>(sp + mat_bytes) = k4[it];
            *reinterpret_cast<uint4*>(sp + 2 * mat_bytes) = v4[it];
        }
    }
    for (int key = threadIdx.x; key < Sp; key += blockDim.x)
        mbias[key] = (key < S && key_valid(key, Lv, vl, tl)) ? 0.f : -CUDART_INF_F;
    __syncthreads();

    const int nkb = Sp >> 3;  // key blocks of 8 (even)
    const int nrb = Sp >> 4;  // query row blocks of 16
    const int g = lane >> 2, t4 = lane & 3;
    const int l8 = lane & 7, lq = lane >> 3;  // ldmatrix: lane -> (row in 8x8 matrix, matrix id)
    const float sl2 = 0.17677669529663687f * 1.4426950408889634f;  // softmax scale * log2(e)
    // bit jb set = key block jb touches a padded key: only those blocks pay for the mask (one ballot per warp)
    uint32_t blkflags;
    {
        const int k0 = lane * 8, k1 = k0 + 8;
        const bool all_valid = (k1 <= vl) || (k1 <= Lv + tl && (vl == Lv || k0 >= Lv));
        blkflags = __ballot_sync(0xffffffffu, !all_valid);
    }
    // Rows from Lv + tl on are text padding: they are never valid keys and nobody reads their outputs, so a 16-row block
    // that holds only such rows is not computed (zeros are written: the rows stay finite for the GEMMs that follow).
    const int nrb_live = (Lv + tl + 15) >> 4;
    const int nkb_live = (Lv + tl + 7) >> 3;  // key blocks from here on hold only padding: their P is exactly 0
    for (int rb = warp; rb < nrb; rb += ATT_WARPS) {
        const int r_lo = rb * 16 + g, r_hi = r_lo + 8;
        if (rb >= nrb_live) {  // warp-uniform
#pragma unroll
            for (int nb = 0; nb < 4; ++nb) {
                if (r_lo < S) *reinterpret_cast<uint32_t*>(o + (row0 + r_lo) * ldo + h * HD + nb * 8 + t4 * 2) = 0u;
                if (r_hi < S) *reinterpret_cast<uint32_t*>(o + (row0 + r_hi) * ldo + h * HD + nb * 8 + t4 * 2) = 0u;
            }
            continue;
        }
        uint32_t aq[2][4];
        // A fragments of Q: matrices (rows 0-7 | 8-15) x (k 0-7 | 8-15) for each 16-wide k step
#pragma unroll
        for (int ks = 0; ks < 2; ++ks)
            ldsm_x4(aq[ks], Qs + (rb * 16 + l8 + (lq & 1) * 8) * QK_PAD + ks * 16 + (lq >> 1) * 8);
        // Keys are processed in two chunks of NB/2 blocks with a running (max, sum) per row (online softmax): only
        // half of the score row block lives in registers at a time, which is what lets 4 CTAs share an SM.
        constexpr int CH = NB / 2;  // key blocks per chunk (even: two blocks form one k-step of P.V)
        float m_lo = -CUDART_INF_F, m_hi = -CUDART_INF_F;
        float rs[4] = {0.f, 0.f, 0.f, 0.f};                // accumulator of the ones block (row sums)
        const uint32_t ones = g == 0 ? 0x3C003C00u : 0u;  // B fragment: B[k][n = g] = 1 for n = 0
        float out[4][4];
#pragma unroll
        for (int nb = 0; nb < 4; ++nb) out[nb][0] = out[nb][1] = out[nb][2] = out[nb][3] = 0.f;
#pragma unroll
        for (int ch = 0; ch < 2; ++ch) {
            if (EXACT || ch * CH < nkb) {  // warp-uniform
                float sc[CH][4];
                float c_lo = -CUDART_INF_F, c_hi = -CUDART_INF_F;
#pragma unroll
                for (int jj = 0; jj < CH; ++jj) {
                    const int jb = ch * CH + jj;
                    sc[jj][0] = sc[jj][1] = sc[jj][2] = sc[jj][3] = -CUDART_INF_F;
                    // the last 16 keys of the tile are often all text padding (see nkb_live): only these two key blocks
                    // carry the (warp-uniform) test, the others stay unconditional in the exact-size variant
                    const bool live = jb < NB - 2 || jb < nkb_live;
                    if ((EXACT || jb < nkb) && live) {
                        sc[jj][0] = sc[jj][1] = sc[jj][2] = sc[jj][3] = 0.f;
                        uint32_t bk[4];  // B fragments of K for keys jb*8..+7: dims 0-7, 8-15, 16-23, 24-31
                        ldsm_x4(bk, Ks + (jb * 8 + l8) * QK_PAD + lq * 8);
                        mma_16816(sc[jj], aq[0], bk[0], bk[1]);
                        mma_16816(sc[jj], aq[1], bk[2], bk[3]);
                        if (blkflags & (1u << jb)) {  // additive -inf for the padded keys of this block (warp-uniform)
                            const float2 mb = *reinterpret_cast<const float2*>(mbias + jb * 8 + t4 * 2);
                            sc[jj][0] += mb.x; sc[jj][1] += mb.y;
                            sc[jj][2] += mb.x; sc[jj][3] += mb.y;
                        }
                        c_lo = fmaxf(c_lo, fmaxf(sc[jj][0], sc[jj][1]));
                        c_hi = fmaxf(c_hi, fmaxf(sc[jj][2], sc[jj][3]));
                    }
                }
                c_lo = fmaxf(c_lo, __shfl_xor_sync(0xffffffffu, c_lo, 1));
                c_lo = fmaxf(c_lo, __shfl_xor_sync(0xffffffffu, c_lo, 2));
                c_hi = fmaxf(c_hi, __shfl_xor_sync(0xffffffffu, c_hi, 1));
                c_hi = fmaxf(c_hi, __shfl_xor_sync(0xffffffffu, c_hi, 2));
                const float n_lo = fmaxf(m_lo, c_lo), n_hi = fmaxf(m_hi, c_hi);
                // p = exp(scale * (s - max)) = exp2(s * sl2 - max * sl2): one FFMA + EX2 per score; exp2(-inf) = 0 for
                // masked keys.  A row whose keys are all masked so far keeps offset 0 (its p and its rescale factor are 0).
                const float o_lo = n_lo == -CUDART_INF_F ? 0.f : -n_lo * sl2;
                const float o_hi = n_hi == -CUDART_INF_F ? 0.f : -n_hi * sl2;
                if (ch > 0) {  // rescale what the previous chunk accumulated against its own maximum
                    const float f_lo = fast_exp2(fmaf(m_lo, sl2, o_lo)), f_hi = fast_exp2(fmaf(m_hi, sl2, o_hi));
                    rs[0] *= f_lo;
                    rs[2] *= f_hi;
#pragma unroll
                    for (int nb = 0; nb < 4; ++nb) {
                        out[nb][0] *= f_lo; out[nb][1] *= f_lo;
                        out[nb][2] *= f_hi; out[nb][3] *= f_hi;
                    }
                }
                m_lo = n_lo;
                m_hi = n_hi;
#pragma unroll
                for (int jj = 0; jj < CH; ++jj) {
#pragma unroll
                    for (int e = 0; e < 2; ++e) {
                        sc[jj][e] = fast_exp2(fmaf(sc[jj][e], sl2, o_lo));
                        sc[jj][2 + e] = fast_exp2(fmaf(sc[jj][2 + e], sl2, o_hi));
                    }
                }
#pragma unroll
                for (int kk = 0; kk < CH / 2; ++kk) {
                    const int kb = ch * (CH / 2) + kk;  // k-step of 16 keys
                    if ((EXACT || kb * 2 < nkb) && (kb < NB / 2 - 1 || kb * 2 < nkb_live)) {
                        uint32_t ap[4];
                        ap[0] = pack_half2(sc[2 * kk][0], sc[2 * kk][1]);
                        ap[1] = pack_half2(sc[2 * kk][2], sc[2 * kk][3]);
                        ap[2] = pack_half2(sc[2 * kk + 1][0], sc[2 * kk + 1][1]);
                        ap[3] = pack_half2(sc[2 * kk + 1][2], sc[2 * kk + 1][3]);
                        // B fragments of V (k = key, n = dim) from row-major V via transposing ldmatrix:
                        // matrices (keys 0-7 | 8-15) x (dims nb*8 | (nb+1)*8)
#pragma unroll
                        for (int np = 0; np < 2; ++np) {
                            uint32_t bv[4];
                            ldsm_x4_trans(bv, Vs + (kb * 16 + l8 + (lq & 1) * 8) * QK_PAD + (np * 2 + (lq >> 1)) * 8);
                            mma_16816(out[np * 2], ap, bv[0], bv[1]);
                            mma_16816(out[np * 2 + 1], ap, bv[2], bv[3]);
                        }
                        // row sums of P through the tensor pipe: a fifth n-block whose column 0 is all ones.  The sum
                        // is taken over the fp16 values that multiply V, so the normalisation is exact for them.
                        mma_16816(rs, ap, ones, ones);
                    }
                }
            }
        }
        // column 0 of the ones block lives in the t4 = 0 lane of each quad: rs[0] = row g, rs[2] = row g + 8
        const float s_lo = __shfl_sync(0xffffffffu, rs[0], lane & ~3), s_hi = __shfl_sync(0xffffffffu, rs[2], lane & ~3);
        const float i_lo = 1.f / s_lo, i_hi = 1.f / s_hi;
#pragma unroll
        for (int nb = 0; nb < 4; ++nb) {
            if (r_lo < S)
                *reinterpret_cast<uint32_t*>(o + (row0 + r_lo) * ldo + h * HD + nb * 8 + t4 * 2) =
                    pack_half2(out[nb][0] * i_lo, out[nb][1] * i_lo);
            if (r_hi < S)
                *reinterpret_cast<uint32_t*>(o + (row0 + r_hi) * ldo + h * HD + nb * 8 + t4 * 2) =
                    pack_half2(out[nb][2] * i_hi, out[nb][3] * i_hi);
        }
    }
}

// Long windows (256 < S <= 512 keys): the kernel above issues the loads of the whole tile before the first use and keeps
// half a score row block in registers, and neither fits at 64 key blocks.  Same inputs (dense rows or the layer-0 row
// tables, the per-layer position table) and the same arithmetic per key block; what changes:
//   - 16 warps, the tile loaded in rounds of LA_ROUND rows per thread (3 x LA_ROUND 16-byte loads in flight);
//   - online softmax over chunks of LA_CH key blocks (64 keys): a running (max, sum) per row, the accumulators of P.V and
//     of the row sums rescaled when the maximum grows;
//   - only the key blocks that hold a valid-length key are visited (the others are text padding: their P is exactly 0).
// Shared memory is the same [Sp][QK_PAD] x 3 tile (123 KB at S = 512): one CTA per SM at 512 rows.
constexpr int LA_WARPS = 16;
constexpr int LA_ROUND = 4;  // load iterations per round
constexpr int LA_CH = 8;     // key blocks per chunk of the online softmax

__global__ void __launch_bounds__(LA_WARPS * 32, 1)
enc_attention_f16_long_kernel(const __half* __restrict__ qk, int64_t ldqk, const __half* __restrict__ v, int64_t ldv,
                              __half* __restrict__ o, int64_t ldo, const int32_t* __restrict__ vlen,
                              const int32_t* __restrict__ tlen, int Lv, int Lt, int d_model,
                              const __half* __restrict__ posqk, int table_lv, EncRowSource src) {
    extern __shared__ __align__(16) unsigned char att_smem[];
    const int S = Lv + Lt;
    const int Sp = (S + 15) & ~15;
    __half* Qs = reinterpret_cast<__half*>(att_smem);  // [Sp][QK_PAD]
    __half* Ks = Qs + Sp * QK_PAD;                      // [Sp][QK_PAD]
    __half* Vs = Ks + Sp * QK_PAD;                      // [Sp][QK_PAD]
    float* mbias = reinterpret_cast<float*>(Vs + Sp * QK_PAD);  // [Sp]
    const int nheads = d_model / HD;
    const int64_t b = blockIdx.x / nheads;
    const int h = blockIdx.x % nheads;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int64_t row0 = b * S;
    const int vl = vlen[b], tl = tlen[b];

    constexpr int ROWS_PER_IT = LA_WARPS * 32 / 4;  // 4 threads per row
    const int r0 = threadIdx.x >> 2, c8 = (threadIdx.x & 3) * 8 + h * HD;
    const bool indirect = src.frames != nullptr;
    const int64_t vbase = indirect ? src.vid_base[b] : 0;
    const int64_t tbase = indirect ? src.txt_base[b] : 0;
    const __half* qp = qk + (row0 + r0) * ldqk + c8;
    const __half* vp = v + (row0 + r0) * ldv + c8;
    const __half* pp = posqk + ((int64_t)vl * table_lv + r0) * (2 * d_model) + c8;
    unsigned char* sbase = att_smem + (r0 * QK_PAD + (threadIdx.x & 3) * 8) * 2;
    const int mat_bytes = Sp * QK_PAD * 2;
    for (int it0 = 0; it0 * ROWS_PER_IT < Sp; it0 += LA_ROUND) {
        uint4 q4[LA_ROUND], k4[LA_ROUND], v4[LA_ROUND];
#pragma unroll
        for (int u = 0; u < LA_ROUND; ++u) {
            const int it = it0 + u;
            const int r = r0 + it * ROWS_PER_IT;
            q4[u] = make_uint4(0, 0, 0, 0);
            k4[u] = q4[u];
            v4[u] = q4[u];
            if (r < S) {
                if (indirect) {
                    const __half* row;
                    if (r < Lv) {
                        int64_t fr = vbase + r;  // rows past the tensor end belong to masked keys: never read out of bounds
                        fr = fr < src.n_frames ? fr : src.n_frames - 1;
                        row = src.frames + fr * (3 * d_model) + c8;
                    } else {
                        row = src.tokens + (tbase + (r - Lv)) * (3 * d_model) + c8;
                    }
                    q4[u] = *reinterpret_cast<const uint4*>(row);
                    k4[u] = *reinterpret_cast<const uint4*>(row + d_model);
                    v4[u] = *reinterpret_cast<const uint4*>(row + 2 * d_model);
                } else {
                    q4[u] = *reinterpret_cast<const uint4*>(qp + (int64_t)it * ROWS_PER_IT * ldqk);
                    k4[u] = *reinterpret_cast<const uint4*>(qp + (int64_t)it * ROWS_PER_IT * ldqk + d_model);
                    v4[u] = *reinterpret_cast<const uint4*>(vp + (int64_t)it * ROWS_PER_IT * ldv);
                }
            }
        }
#pragma unroll
        for (int u = 0; u < LA_ROUND; ++u) {
            const int it = it0 + u;
            const int r = r0 + it * ROWS_PER_IT;
            if (r < Sp) {
                if (posqk != nullptr && r < Lv) {  // q | k + pos . [Wq; Wk]^T, one fp16 rounding (as the kernel above)
                    const __half* pr = pp + (int64_t)it * ROWS_PER_IT * 2 * d_model;
                    const uint4 pq = __ldg(reinterpret_cast<const uint4*>(pr));
                    const uint4 pk = __ldg(reinterpret_cast<const uint4*>(pr + d_model));
                    __half2* qh = reinterpret_cast<__half2*>(&q4[u]);
                    __half2* kh = reinterpret_cast<__half2*>(&k4[u]);
                    const __half2* pqh = reinterpret_cast<const __half2*>(&pq);
                    const __half2* pkh = reinterpret_cast<const __half2*>(&pk);
#pragma unroll
                    for (int e = 0; e < 4; ++e) {
                        qh[e] = __hadd2(qh[e], pqh[e]);
                        kh[e] = __hadd2(kh[e], pkh[e]);
                    }
                }
                unsigned char* sp = sbase + it * ROWS_PER_IT * QK_PAD * 2;
                *reinterpret_cast<uint4*>(sp) = q4[u];
                *reinterpret_cast<uint4*>(sp + mat_bytes) = k4[u];
                *reinterpret_cast<uint4*>(sp + 2 * mat_bytes) = v4[u];
            }
        }
    }
    for (int key = threadIdx.x; key < Sp; key += blockDim.x)
        mbias[key] = (key < S && key_valid(key, Lv, vl, tl)) ? 0.f : -CUDART_INF_F;
    __syncthreads();

    const int nrb = Sp >> 4;
    const int g = lane >> 2, t4 = lane & 3;
    const int l8 = lane & 7, lq = lane >> 3;
    const float sl2 = 0.17677669529663687f * 1.4426950408889634f;
    // bit jb of word jb / 32 set = key block jb touches a padded key (64 blocks: two ballots)
    uint32_t blkflags[2];
#pragma unroll
    for (int w = 0; w < 2; ++w) {
        const int k0 = (w * 32 + lane) * 8, k1 = k0 + 8;
        const bool all_valid = (k1 <= vl) || (k1 <= Lv + tl && (vl == Lv || k0 >= Lv));
        blkflags[w] = __ballot_sync(0xffffffffu, !all_valid);
    }
    const int nrb_live = (Lv + tl + 15) >> 4;
    const int nkb_live = (Lv + tl + 7) >> 3;  // key blocks from here on hold only padding
    const int nch = (nkb_live + LA_CH - 1) / LA_CH;
    for (int rb = warp; rb < nrb; rb += LA_WARPS) {
        const int r_lo = rb * 16 + g, r_hi = r_lo + 8;
        if (rb >= nrb_live) {  // warp-uniform: text padding rows, zeros
#pragma unroll
            for (int nb = 0; nb < 4; ++nb) {
                if (r_lo < S) *reinterpret_cast<uint32_t*>(o + (row0 + r_lo) * ldo + h * HD + nb * 8 + t4 * 2) = 0u;
                if (r_hi < S) *reinterpret_cast<uint32_t*>(o + (row0 + r_hi) * ldo + h * HD + nb * 8 + t4 * 2) = 0u;
            }
            continue;
        }
        uint32_t aq[2][4];
#pragma unroll
        for (int ks = 0; ks < 2; ++ks)
            ldsm_x4(aq[ks], Qs + (rb * 16 + l8 + (lq & 1) * 8) * QK_PAD + ks * 16 + (lq >> 1) * 8);
        float m_lo = -CUDART_INF_F, m_hi = -CUDART_INF_F;
        float rs[4] = {0.f, 0.f, 0.f, 0.f};
        const uint32_t ones = g == 0 ? 0x3C003C00u : 0u;
        float out[4][4];
#pragma unroll
        for (int nb = 0; nb < 4; ++nb) out[nb][0] = out[nb][1] = out[nb][2] = out[nb][3] = 0.f;
        for (int ch = 0; ch < nch; ++ch) {
            const int jb0 = ch * LA_CH;
            const uint32_t fl = (jb0 < 32 ? blkflags[0] : blkflags[1]) >> (jb0 & 31);  // a chunk lies within one word
            float sc[LA_CH][4];
            float c_lo = -CUDART_INF_F, c_hi = -CUDART_INF_F;
#pragma unroll
            for (int jj = 0; jj < LA_CH; ++jj) {
                const int jb = jb0 + jj;
                sc[jj][0] = sc[jj][1] = sc[jj][2] = sc[jj][3] = -CUDART_INF_F;
                if (jb < nkb_live) {  // warp-uniform
                    sc[jj][0] = sc[jj][1] = sc[jj][2] = sc[jj][3] = 0.f;
                    uint32_t bk[4];
                    ldsm_x4(bk, Ks + (jb * 8 + l8) * QK_PAD + lq * 8);
                    mma_16816(sc[jj], aq[0], bk[0], bk[1]);
                    mma_16816(sc[jj], aq[1], bk[2], bk[3]);
                    if (fl & (1u << jj)) {
                        const float2 mb = *reinterpret_cast<const float2*>(mbias + jb * 8 + t4 * 2);
                        sc[jj][0] += mb.x; sc[jj][1] += mb.y;
                        sc[jj][2] += mb.x; sc[jj][3] += mb.y;
                    }
                    c_lo = fmaxf(c_lo, fmaxf(sc[jj][0], sc[jj][1]));
                    c_hi = fmaxf(c_hi, fmaxf(sc[jj][2], sc[jj][3]));
                }
            }
            c_lo = fmaxf(c_lo, __shfl_xor_sync(0xffffffffu, c_lo, 1));
            c_lo = fmaxf(c_lo, __shfl_xor_sync(0xffffffffu, c_lo, 2));
            c_hi = fmaxf(c_hi, __shfl_xor_sync(0xffffffffu, c_hi, 1));
            c_hi = fmaxf(c_hi, __shfl_xor_sync(0xffffffffu, c_hi, 2));
            const float n_lo = fmaxf(m_lo, c_lo), n_hi = fmaxf(m_hi, c_hi);
            const float o_lo = n_lo == -CUDART_INF_F ? 0.f : -n_lo * sl2;
            const float o_hi = n_hi == -CUDART_INF_F ? 0.f : -n_hi * sl2;
            if (ch > 0) {  // exp2(-inf) = 0: a row with no valid key so far has nothing to rescale
                const float f_lo = fast_exp2(fmaf(m_lo, sl2, o_lo)), f_hi = fast_exp2(fmaf(m_hi, sl2, o_hi));
                rs[0] *= f_lo;
                rs[2] *= f_hi;
#pragma unroll
                for (int nb = 0; nb < 4; ++nb) {
                    out[nb][0] *= f_lo; out[nb][1] *= f_lo;
                    out[nb][2] *= f_hi; out[nb][3] *= f_hi;
                }
            }
            m_lo = n_lo;
            m_hi = n_hi;
#pragma unroll
            for (int jj = 0; jj < LA_CH; ++jj) {
#pragma unroll
                for (int e = 0; e < 2; ++e) {
                    sc[jj][e] = fast_exp2(fmaf(sc[jj][e], sl2, o_lo));
                    sc[jj][2 + e] = fast_exp2(fmaf(sc[jj][2 + e], sl2, o_hi));
                }
            }
#pragma unroll
            for (int kk = 0; kk < LA_CH / 2; ++kk) {
                const int kb = jb0 / 2 + kk;  // k-step of 16 keys
                if (kb * 2 < nkb_live) {
                    uint32_t ap[4];
                    ap[0] = pack_half2(sc[2 * kk][0], sc[2 * kk][1]);
                    ap[1] = pack_half2(sc[2 * kk][2], sc[2 * kk][3]);
                    ap[2] = pack_half2(sc[2 * kk + 1][0], sc[2 * kk + 1][1]);
                    ap[3] = pack_half2(sc[2 * kk + 1][2], sc[2 * kk + 1][3]);
#pragma unroll
                    for (int np = 0; np < 2; ++np) {
                        uint32_t bv[4];
                        ldsm_x4_trans(bv, Vs + (kb * 16 + l8 + (lq & 1) * 8) * QK_PAD + (np * 2 + (lq >> 1)) * 8);
                        mma_16816(out[np * 2], ap, bv[0], bv[1]);
                        mma_16816(out[np * 2 + 1], ap, bv[2], bv[3]);
                    }
                    mma_16816(rs, ap, ones, ones);  // row sums over the fp16 values of P
                }
            }
        }
        const float s_lo = __shfl_sync(0xffffffffu, rs[0], lane & ~3), s_hi = __shfl_sync(0xffffffffu, rs[2], lane & ~3);
        const float i_lo = 1.f / s_lo, i_hi = 1.f / s_hi;
#pragma unroll
        for (int nb = 0; nb < 4; ++nb) {
            if (r_lo < S)
                *reinterpret_cast<uint32_t*>(o + (row0 + r_lo) * ldo + h * HD + nb * 8 + t4 * 2) =
                    pack_half2(out[nb][0] * i_lo, out[nb][1] * i_lo);
            if (r_hi < S)
                *reinterpret_cast<uint32_t*>(o + (row0 + r_hi) * ldo + h * HD + nb * 8 + t4 * 2) =
                    pack_half2(out[nb][2] * i_hi, out[nb][3] * i_hi);
        }
    }
}


// ------------------------------------------------------------------------------------------------
// Memory-direct decoder cross-attention (CONE_PREC_TC).  The K and V projections of the memory are never formed:
//   score(slot, h, key) = q_h . (Wk_h (m_key + pos_key) + bk_h)
//                       = (Wk_h^T q_h) . m_key + q_h . (Wk_h pos_key) + const(key)      [const cancels in the softmax]
//   out(slot, h)        = sum_key p_key (Wv_h m_key + bv_h) = Wv_h (sum_key p_key m_key) + bv_h     [sum p = 1]
// so the kernel works on the RAW encoder output m [S, 256] of the window: the queries arrive already pushed through
// Wk_h^T (qt [slot, h, 256], produced by the same GEMM that makes q), and what leaves is the attention-pooled memory
// pm [slot, h, 256]; Wv_h and the output projection are folded into the next GEMM (K = 8 x 256).  This removes the
// [R, 2 DL 256] K|V projection GEMM of the memory (the largest decoder launch) and its 2 x 1 KB per memory row and
// layer of HBM traffic; the window's memory is read once (512 B per row) into shared memory and feeds both products.
// One CTA per window, one warp per 16 rows of the (head, slot) x key score matrix (8 nq rows): S = Qt.M^T with
// mma.sync m16n8k16 (K = 256: A fragments of qt stay in registers, B fragments by ldmatrix), position term through
// the per-layer pos.Wk^T table (K = 32 per head, fragments straight from 16-byte global loads, contraction index
// permuted: lane (g, t4) puts channels [8 t4, 8 t4 + 8) of key 8 jb + g — one 16-byte load — into the B fragments
// of the head's two k-steps and the same channels of q into the A fragments), masked softmax on the accumulators, P.M with transposing ldmatrix.
// The softmax scale and log2(e) are folded into the weights that produce q and qt.
// ------------------------------------------------------------------------------------------------
constexpr int XM_PAD = 264;  // halves per shared-memory row (256 + 8): 528-byte stride -> conflict-free ldmatrix

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(smem_dst)),
                 "l"(gmem_src)
                 : "memory");
}

template <int NB, int MT>
__global__ void __launch_bounds__(MT * 64, NB <= 20 ? 2 : 1)
dec_cross_attention_mem_kernel(const __half* __restrict__ mem, int64_t ldm, const __half* __restrict__ qqt, int64_t ldq,
                               __half* __restrict__ pm, int64_t ldp, const int32_t* __restrict__ vlen,
                               const int32_t* __restrict__ tlen, int nq, int Lv, int Lt,
                               const __half* __restrict__ posk, int64_t ldposk, int table_lv, int q_bcast) {
    // Two warps per 16-row block of the score matrix (ncu on the one-warp-per-block version: 6 warps per SM, every stall
    // a fixed-latency dependency): for the scores they split the key blocks (even / odd), exchange row maxima and
    // sums through shared memory, publish their halves of P there, and for P.M they split the 256 channels.
    constexpr int D = 256;
    constexpr int NW = MT * 2;     // warps
    constexpr int NJ = NB / 2;     // key blocks per warp
    constexpr int PS_PAD = NB * 8 + 8;  // halves per row of P in shared memory (conflict-free 4-byte stores and ldmatrix)
    static_assert(PS_PAD <= XM_PAD, "P must fit the shared memory of the qt rows it replaces");
    extern __shared__ __align__(16) unsigned char xsm[];
    __half* Ms = reinterpret_cast<__half*>(xsm);   // [NB * 8][XM_PAD] memory rows of the window (rows >= S are zero)
    __half* Qt = Ms + NB * 8 * XM_PAD;             // [MT * 16][XM_PAD] qt rows, row = head * nq + slot
    __half* Ps = Qt;                               // [MT * 16][PS_PAD] P, once the qt fragments are in registers
    float* red = reinterpret_cast<float*>(Qt + MT * 16 * XM_PAD);  // [MT][2 halves][16 rows][max, sum]
    const int64_t b = blockIdx.x;
    const int S = Lv + Lt;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int mt = warp >> 1, half = warp & 1;
    const int64_t row0 = b * S;
    const int R = 8 * nq;  // valid score rows

    {   // memory rows: 32 chunks of 16 bytes per row, one row per warp and iteration (pointer increments only)
        const int c = lane * 8;
        const __half* src = mem + (row0 + warp) * ldm + c;
        __half* dst = Ms + warp * XM_PAD + c;
#pragma unroll 4
        for (int r = warp; r < NB * 8; r += NW) {
            if (r < S) cp_async16(dst, src);
            else *reinterpret_cast<uint4*>(dst) = make_uint4(0u, 0u, 0u, 0u);
            src += (int64_t)NW * ldm;
            dst += NW * XM_PAD;
        }
        for (int r = warp; r < MT * 16; r += NW) {
            __half* qd = Qt + r * XM_PAD + c;
            if (r < R) {
                const int hh = r / nq, slot = r - hh * nq;
                cp_async16(qd, qqt + ((q_bcast ? 0 : b * nq) + slot) * ldq + D + hh * D + c);
            } else {
                *reinterpret_cast<uint4*>(qd) = make_uint4(0u, 0u, 0u, 0u);
            }
        }
    }
    asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
    __syncthreads();

    const int vl = vlen[b], tl = tlen[b];
    const int g = lane >> 2, t4 = lane & 3;
    const int l8 = lane & 7, lq = lane >> 3;
    const int r_lo = mt * 16 + g, r_hi = r_lo + 8;           // this lane's two score rows
    const int h_lo = r_lo < R ? r_lo / nq : -1, h_hi = r_hi < R ? r_hi / nq : -1;
    // output rows; the query rows are the same unless the queries are shared by all windows (q_bcast: rows 0..nq-1)
    const int64_t q_lo = r_lo < R ? (b * nq + (r_lo - h_lo * nq)) : 0, q_hi = r_hi < R ? (b * nq + (r_hi - h_hi * nq)) : 0;
    const int64_t qs_lo = (q_bcast && r_lo < R) ? q_lo - b * nq : q_lo, qs_hi = (q_bcast && r_hi < R) ? q_hi - b * nq : q_hi;

    float sc[NJ][4];  // key block jb = 2 j + half
#pragma unroll
    for (int j = 0; j < NJ; ++j) sc[j][0] = sc[j][1] = sc[j][2] = sc[j][3] = 0.f;
    {   // content term: 16 k-steps over the 256 channels
        uint32_t aq[16][4];
#pragma unroll
        for (int ks = 0; ks < 16; ++ks)
            ldsm_x4(aq[ks], Qt + (mt * 16 + l8 + (lq & 1) * 8) * XM_PAD + ks * 16 + (lq >> 1) * 8);
        __syncthreads();  // every warp holds its qt fragments: the rows may now be overwritten by P
        // One k-step (16 channels) at a time over this warp's key blocks: back-to-back MMAs never share an accumulator.
        // All blocks are processed without range tests: rows past S are zero in shared memory (masked below).
#pragma unroll
        for (int ks = 0; ks < 16; ++ks) {
#pragma unroll
            for (int j = 0; j < NJ; ++j) {
                uint32_t b0, b1;  // keys jb*8..+7, channels ks*16 + (0-7 | 8-15)
                ldsm_x2(b0, b1, Ms + ((2 * j + half) * 8 + l8) * XM_PAD + ks * 16 + (lq & 1) * 8);
                mma_16816(sc[j], aq[ks], b0, b1);
            }
        }
    }
    if (posk != nullptr) {  // position term of the video keys, one head of this row block at a time
        const int h_first = (mt * 16) / nq;
        const int h_last = min(7, (mt * 16 + 15) / nq);
        // Two heads per pass: the table rows of all of this warp's key blocks for both heads are requested together
        // (ncu: one L2 round trip per (key block, head), 64 in a row, was 3/4 of the first version's time; one per head
        // was still a quarter of the second's).
        constexpr int HP = MT <= 3 ? 2 : 1;  // heads per pass (register budget: 170 at 6 warps per CTA, 128 at 8)
        for (int hh = h_first; hh <= h_last; hh += HP) {
            uint32_t a[HP][2][4];
            uint4 pf[HP][NJ];
#pragma unroll
            for (int u = 0; u < HP; ++u) {
                const int hu = hh + u;  // hu > h_last: no row of this block belongs to it, its A fragments are zero
                uint4 xl = make_uint4(0u, 0u, 0u, 0u), xh = xl;
                if (h_lo == hu) xl = *reinterpret_cast<const uint4*>(qqt + qs_lo * ldq + hu * HD + t4 * 8);
                if (h_hi == hu) xh = *reinterpret_cast<const uint4*>(qqt + qs_hi * ldq + hu * HD + t4 * 8);
                a[u][0][0] = xl.x; a[u][0][1] = xh.x; a[u][0][2] = xl.y; a[u][0][3] = xh.y;
                a[u][1][0] = xl.z; a[u][1][1] = xh.z; a[u][1][2] = xl.w; a[u][1][3] = xh.w;
                const __half* pbase = posk + ((int64_t)vl * table_lv + half * 8 + g) * ldposk + hu * HD + t4 * 8;
#pragma unroll
                for (int j = 0; j < NJ; ++j) {
                    pf[u][j] = make_uint4(0u, 0u, 0u, 0u);
                    if (hu <= h_last && (2 * j + half) * 8 + g < Lv)
                        pf[u][j] = __ldg(reinterpret_cast<const uint4*>(pbase + (int64_t)j * 16 * ldposk));
                }
            }
#pragma unroll
            for (int u = 0; u < HP; ++u) {
                if (hh + u <= h_last) {  // warp-uniform
#pragma unroll
                    for (int j = 0; j < NJ; ++j) mma_16816(sc[j], a[u][0], pf[u][j].x, pf[u][j].y);
#pragma unroll
                    for (int j = 0; j < NJ; ++j) mma_16816(sc[j], a[u][1], pf[u][j].z, pf[u][j].w);
                }
            }
        }
    }
    // masked softmax over the keys (exp2 domain), rows g and g + 8; the partner warp holds the other key blocks
    float m_lo = -CUDART_INF_F, m_hi = -CUDART_INF_F;
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
#pragma unroll
        for (int e = 0; e < 2; ++e) {
            const int key = (2 * j + half) * 8 + t4 * 2 + e;
            const bool ok = key < S && key_valid(key, Lv, vl, tl);
            sc[j][e] = ok ? sc[j][e] : -CUDART_INF_F;
            sc[j][2 + e] = ok ? sc[j][2 + e] : -CUDART_INF_F;
            m_lo = fmaxf(m_lo, sc[j][e]);
            m_hi = fmaxf(m_hi, sc[j][2 + e]);
        }
    }
    m_lo = fmaxf(m_lo, __shfl_xor_sync(0xffffffffu, m_lo, 1));
    m_lo = fmaxf(m_lo, __shfl_xor_sync(0xffffffffu, m_lo, 2));
    m_hi = fmaxf(m_hi, __shfl_xor_sync(0xffffffffu, m_hi, 1));
    m_hi = fmaxf(m_hi, __shfl_xor_sync(0xffffffffu, m_hi, 2));
    float* my_red = red + ((mt * 2 + half) * 16) * 2;
    const float* other_red = red + ((mt * 2 + (half ^ 1)) * 16) * 2;
    if (t4 == 0) {
        my_red[g * 2] = m_lo;
        my_red[(g + 8) * 2] = m_hi;
    }
    asm volatile("bar.sync %0, 64;" ::"r"(1 + mt) : "memory");  // the two warps of this row block
    m_lo = fmaxf(m_lo, other_red[g * 2]);
    m_hi = fmaxf(m_hi, other_red[(g + 8) * 2]);
    // a row whose keys are all masked keeps offset 0: exp2(-inf) = 0, sum 0 -> NaN, like torch's softmax of all -inf
    const float o_lo = m_lo == -CUDART_INF_F ? 0.f : m_lo, o_hi = m_hi == -CUDART_INF_F ? 0.f : m_hi;
    float s_lo = 0.f, s_hi = 0.f;
#pragma unroll
    for (int j = 0; j < NJ; ++j) {
        const uint32_t pl = pack_half2(fast_exp2(sc[j][0] - o_lo), fast_exp2(sc[j][1] - o_lo));
        const uint32_t ph = pack_half2(fast_exp2(sc[j][2] - o_hi), fast_exp2(sc[j][3] - o_hi));
        // the row sum is taken over the fp16 values that multiply M, so the normalisation is exact for them
        const float2 fl = __half22float2(*reinterpret_cast<const __half2*>(&pl));
        const float2 fh = __half22float2(*reinterpret_cast<const __half2*>(&ph));
        s_lo += fl.x + fl.y;
        s_hi += fh.x + fh.y;
        const int key = (2 * j + half) * 8 + t4 * 2;
        *reinterpret_cast<uint32_t*>(Ps + r_lo * PS_PAD + key) = pl;
        *reinterpret_cast<uint32_t*>(Ps + r_hi * PS_PAD + key) = ph;
    }
    s_lo += __shfl_xor_sync(0xffffffffu, s_lo, 1);
    s_lo += __shfl_xor_sync(0xffffffffu, s_lo, 2);
    s_hi += __shfl_xor_sync(0xffffffffu, s_hi, 1);
    s_hi += __shfl_xor_sync(0xffffffffu, s_hi, 2);
    if (t4 == 0) {
        my_red[g * 2 + 1] = s_lo;
        my_red[(g + 8) * 2 + 1] = s_hi;
    }
    asm volatile("bar.sync %0, 64;" ::"r"(1 + mt) : "memory");  // sums and both halves of P are visible
    const float i_lo = 1.f / (s_lo + other_red[g * 2 + 1]), i_hi = 1.f / (s_hi + other_red[(g + 8) * 2 + 1]);

    // pooled memory: out[16 rows x 128 channels of this warp] = P . M over all keys
    float out[16][4];
#pragma unroll
    for (int nt = 0; nt < 16; ++nt) out[nt][0] = out[nt][1] = out[nt][2] = out[nt][3] = 0.f;
#pragma unroll
    for (int kb = 0; kb < NJ; ++kb) {
        uint32_t ap[4];  // P rows (0-7 | 8-15) x keys kb*16 + (0-7 | 8-15)
        ldsm_x4(ap, Ps + (mt * 16 + l8 + (lq & 1) * 8) * PS_PAD + kb * 16 + (lq >> 1) * 8);
#pragma unroll
        for (int np = 0; np < 8; ++np) {
            uint32_t bv[4];  // keys kb*16 + (0-7 | 8-15) x channels half*128 + np*16 + (0-7 | 8-15)
            ldsm_x4_trans(bv, Ms + (kb * 16 + l8 + (lq & 1) * 8) * XM_PAD + half * 128 + (np * 2 + (lq >> 1)) * 8);
            mma_16816(out[np * 2], ap, bv[0], bv[1]);
            mma_16816(out[np * 2 + 1], ap, bv[2], bv[3]);
        }
    }
    __half* o_lo_p = pm + q_lo * ldp + (h_lo < 0 ? 0 : h_lo) * D + half * 128 + t4 * 2;
    __half* o_hi_p = pm + q_hi * ldp + (h_hi < 0 ? 0 : h_hi) * D + half * 128 + t4 * 2;
#pragma unroll
    for (int nt = 0; nt < 16; ++nt) {
        if (h_lo >= 0) *reinterpret_cast<uint32_t*>(o_lo_p + nt * 8) = pack_half2(out[nt][0] * i_lo, out[nt][1] * i_lo);
        if (h_hi >= 0) *reinterpret_cast<uint32_t*>(o_hi_p + nt * 8) = pack_half2(out[nt][2] * i_hi, out[nt][3] * i_hi);
    }
}

// Long windows (256 < S <= 512): 512 memory rows at 528 B would need 270 KB of shared memory.  This variant streams the
// memory through two buffers of XL_KC rows (cp.async: chunk c + 1 is in flight while chunk c is multiplied), with an
// online softmax across chunks: an fp32 running maximum per score row (shared by the two warps of a row block through
// shared memory), fp32 partial row sums and P.M accumulators rescaled whenever the maximum grows.  Per chunk the
// arithmetic is that of the kernel above: content term over the 256 channels, position term through the pos.Wk^T
// table, masked exp2 softmax with P rounded to fp16 and the row sums taken over the rounded values, P.M with
// transposing ldmatrix.  The qt rows stay in shared memory (their fragments are re-read per chunk) and P has its own
// buffer.  Shared memory at MT = 4: 2 x 66 KB (memory) + 33 KB (qt) + 17 KB (P) = 183 KB, one CTA per SM.
constexpr int XL_KC = 128;  // memory rows per chunk

template <int MT>
__global__ void __launch_bounds__(MT * 64, 1)
dec_cross_attention_mem_long_kernel(const __half* __restrict__ mem, int64_t ldm, const __half* __restrict__ qqt, int64_t ldq,
                                    __half* __restrict__ pm, int64_t ldp, const int32_t* __restrict__ vlen,
                                    const int32_t* __restrict__ tlen, int nq, int Lv, int Lt,
                                    const __half* __restrict__ posk, int64_t ldposk, int table_lv, int q_bcast) {
    constexpr int D = 256;
    constexpr int NW = MT * 2;         // warps
    constexpr int NJ = XL_KC / 16;     // key blocks of a chunk per warp (the two warps of a row block: even / odd)
    constexpr int PS_PAD = XL_KC + 8;  // halves per row of P (272-byte stride: conflict-free stores and ldmatrix)
    extern __shared__ __align__(16) unsigned char xsm[];
    __half* Ms = reinterpret_cast<__half*>(xsm);          // [2][XL_KC][XM_PAD] memory chunks (rows >= S are zero)
    __half* Qt = Ms + 2 * XL_KC * XM_PAD;                 // [MT * 16][XM_PAD] qt rows, row = head * nq + slot
    __half* Ps = Qt + MT * 16 * XM_PAD;                   // [MT * 16][PS_PAD] P of the current chunk
    float* red = reinterpret_cast<float*>(Ps + MT * 16 * PS_PAD);  // [MT][2 halves][16 rows][max, sum]
    const int64_t b = blockIdx.x;
    const int S = Lv + Lt;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const int mt = warp >> 1, half = warp & 1;
    const int64_t row0 = b * S;
    const int R = 8 * nq;
    const int nch = (S + XL_KC - 1) / XL_KC;

    auto load_chunk = [&](int c) {  // one row per warp and iteration, 32 chunks of 16 bytes per row
        const int k0 = c * XL_KC;
        const __half* src = mem + (row0 + k0 + warp) * ldm + lane * 8;
        __half* dst = Ms + (c & 1) * XL_KC * XM_PAD + warp * XM_PAD + lane * 8;
#pragma unroll 4
        for (int r = warp; r < XL_KC; r += NW) {
            if (k0 + r < S) cp_async16(dst, src);
            else *reinterpret_cast<uint4*>(dst) = make_uint4(0u, 0u, 0u, 0u);
            src += (int64_t)NW * ldm;
            dst += NW * XM_PAD;
        }
        asm volatile("cp.async.commit_group;" ::: "memory");
    };
    for (int r = warp; r < MT * 16; r += NW) {
        __half* qd = Qt + r * XM_PAD + lane * 8;
        if (r < R) {
            const int hh = r / nq, slot = r - hh * nq;
            cp_async16(qd, qqt + ((q_bcast ? 0 : b * nq) + slot) * ldq + D + hh * D + lane * 8);
        } else {
            *reinterpret_cast<uint4*>(qd) = make_uint4(0u, 0u, 0u, 0u);
        }
    }
    load_chunk(0);  // the same commit group as the qt rows

    const int vl = vlen[b], tl = tlen[b];
    const int g = lane >> 2, t4 = lane & 3;
    const int l8 = lane & 7, lq = lane >> 3;
    const int r_lo = mt * 16 + g, r_hi = r_lo + 8;
    const int h_lo = r_lo < R ? r_lo / nq : -1, h_hi = r_hi < R ? r_hi / nq : -1;
    const int64_t q_lo = r_lo < R ? (b * nq + (r_lo - h_lo * nq)) : 0, q_hi = r_hi < R ? (b * nq + (r_hi - h_hi * nq)) : 0;
    const int64_t qs_lo = (q_bcast && r_lo < R) ? q_lo - b * nq : q_lo, qs_hi = (q_bcast && r_hi < R) ? q_hi - b * nq : q_hi;
    const int h_first = (mt * 16) / nq;
    const int h_last = min(7, (mt * 16 + 15) / nq);
    float* my_red = red + ((mt * 2 + half) * 16) * 2;
    const float* other_red = red + ((mt * 2 + (half ^ 1)) * 16) * 2;

    float m_lo = -CUDART_INF_F, m_hi = -CUDART_INF_F;  // running maxima (the same in both warps of the row block)
    float s_lo = 0.f, s_hi = 0.f;                      // this lane's part of the row sums, against the running maxima
    float out[16][4];
#pragma unroll
    for (int nt = 0; nt < 16; ++nt) out[nt][0] = out[nt][1] = out[nt][2] = out[nt][3] = 0.f;
    for (int c = 0; c < nch; ++c) {
        asm volatile("cp.async.wait_group 0;" ::: "memory");
        __syncthreads();  // chunk c is in place; every warp is done with chunk c - 1 (its buffer, P and the maxima)
        if (c + 1 < nch) load_chunk(c + 1);
        const __half* Mc = Ms + (c & 1) * XL_KC * XM_PAD;
        const int k0 = c * XL_KC;
        float sc[NJ][4];  // key block jb = 2 j + half of the chunk
#pragma unroll
        for (int j = 0; j < NJ; ++j) sc[j][0] = sc[j][1] = sc[j][2] = sc[j][3] = 0.f;
#pragma unroll
        for (int ks = 0; ks < 16; ++ks) {  // content term: 16 k-steps over the 256 channels
            uint32_t aq[4];
            ldsm_x4(aq, Qt + (mt * 16 + l8 + (lq & 1) * 8) * XM_PAD + ks * 16 + (lq >> 1) * 8);
#pragma unroll
            for (int j = 0; j < NJ; ++j) {
                uint32_t b0, b1;
                ldsm_x2(b0, b1, Mc + ((2 * j + half) * 8 + l8) * XM_PAD + ks * 16 + (lq & 1) * 8);
                mma_16816(sc[j], aq, b0, b1);
            }
        }
        if (posk != nullptr && k0 < Lv) {  // position term of the video keys of this chunk, two heads per pass
            for (int hh = h_first; hh <= h_last; hh += 2) {
                uint32_t a[2][2][4];
                uint4 pf[2][NJ];
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    const int hu = hh + u;
                    uint4 xl = make_uint4(0u, 0u, 0u, 0u), xh = xl;
                    if (h_lo == hu) xl = *reinterpret_cast<const uint4*>(qqt + qs_lo * ldq + hu * HD + t4 * 8);
                    if (h_hi == hu) xh = *reinterpret_cast<const uint4*>(qqt + qs_hi * ldq + hu * HD + t4 * 8);
                    a[u][0][0] = xl.x; a[u][0][1] = xh.x; a[u][0][2] = xl.y; a[u][0][3] = xh.y;
                    a[u][1][0] = xl.z; a[u][1][1] = xh.z; a[u][1][2] = xl.w; a[u][1][3] = xh.w;
                    const __half* pbase = posk + ((int64_t)vl * table_lv + k0 + half * 8 + g) * ldposk + hu * HD + t4 * 8;
#pragma unroll
                    for (int j = 0; j < NJ; ++j) {
                        pf[u][j] = make_uint4(0u, 0u, 0u, 0u);
                        if (hu <= h_last && k0 + (2 * j + half) * 8 + g < Lv)
                            pf[u][j] = __ldg(reinterpret_cast<const uint4*>(pbase + (int64_t)j * 16 * ldposk));
                    }
                }
#pragma unroll
                for (int u = 0; u < 2; ++u) {
                    if (hh + u <= h_last) {  // warp-uniform
#pragma unroll
                        for (int j = 0; j < NJ; ++j) mma_16816(sc[j], a[u][0], pf[u][j].x, pf[u][j].y);
#pragma unroll
                        for (int j = 0; j < NJ; ++j) mma_16816(sc[j], a[u][1], pf[u][j].z, pf[u][j].w);
                    }
                }
            }
        }
        // mask, chunk maxima of rows g and g + 8 over both warps' key blocks
        float c_lo = -CUDART_INF_F, c_hi = -CUDART_INF_F;
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
#pragma unroll
            for (int e = 0; e < 2; ++e) {
                const int key = k0 + (2 * j + half) * 8 + t4 * 2 + e;
                const bool ok = key < S && key_valid(key, Lv, vl, tl);
                sc[j][e] = ok ? sc[j][e] : -CUDART_INF_F;
                sc[j][2 + e] = ok ? sc[j][2 + e] : -CUDART_INF_F;
                c_lo = fmaxf(c_lo, sc[j][e]);
                c_hi = fmaxf(c_hi, sc[j][2 + e]);
            }
        }
        c_lo = fmaxf(c_lo, __shfl_xor_sync(0xffffffffu, c_lo, 1));
        c_lo = fmaxf(c_lo, __shfl_xor_sync(0xffffffffu, c_lo, 2));
        c_hi = fmaxf(c_hi, __shfl_xor_sync(0xffffffffu, c_hi, 1));
        c_hi = fmaxf(c_hi, __shfl_xor_sync(0xffffffffu, c_hi, 2));
        if (t4 == 0) {
            my_red[g * 2] = c_lo;
            my_red[(g + 8) * 2] = c_hi;
        }
        asm volatile("bar.sync %0, 64;" ::"r"(1 + mt) : "memory");  // the two warps of this row block
        c_lo = fmaxf(c_lo, other_red[g * 2]);
        c_hi = fmaxf(c_hi, other_red[(g + 8) * 2]);
        const float n_lo = fmaxf(m_lo, c_lo), n_hi = fmaxf(m_hi, c_hi);
        // a row with no valid key so far keeps offset 0: exp2(-inf) = 0 for its P and its rescale factor
        const float o_lo = n_lo == -CUDART_INF_F ? 0.f : n_lo, o_hi = n_hi == -CUDART_INF_F ? 0.f : n_hi;
        if (c > 0) {
            const float f_lo = fast_exp2(m_lo - o_lo), f_hi = fast_exp2(m_hi - o_hi);
            s_lo *= f_lo;
            s_hi *= f_hi;
#pragma unroll
            for (int nt = 0; nt < 16; ++nt) {
                out[nt][0] *= f_lo; out[nt][1] *= f_lo;
                out[nt][2] *= f_hi; out[nt][3] *= f_hi;
            }
        }
        m_lo = n_lo;
        m_hi = n_hi;
#pragma unroll
        for (int j = 0; j < NJ; ++j) {
            const uint32_t pl = pack_half2(fast_exp2(sc[j][0] - o_lo), fast_exp2(sc[j][1] - o_lo));
            const uint32_t ph = pack_half2(fast_exp2(sc[j][2] - o_hi), fast_exp2(sc[j][3] - o_hi));
            const float2 fl = __half22float2(*reinterpret_cast<const __half2*>(&pl));
            const float2 fh = __half22float2(*reinterpret_cast<const __half2*>(&ph));
            s_lo += fl.x + fl.y;
            s_hi += fh.x + fh.y;
            const int key = (2 * j + half) * 8 + t4 * 2;
            *reinterpret_cast<uint32_t*>(Ps + r_lo * PS_PAD + key) = pl;
            *reinterpret_cast<uint32_t*>(Ps + r_hi * PS_PAD + key) = ph;
        }
        asm volatile("bar.sync %0, 64;" ::"r"(1 + mt) : "memory");  // both halves of P are visible
#pragma unroll
        for (int kb = 0; kb < NJ; ++kb) {  // out[16 rows x this warp's 128 channels] += P . M over the chunk
            uint32_t ap[4];
            ldsm_x4(ap, Ps + (mt * 16 + l8 + (lq & 1) * 8) * PS_PAD + kb * 16 + (lq >> 1) * 8);
#pragma unroll
            for (int np = 0; np < 8; ++np) {
                uint32_t bv[4];
                ldsm_x4_trans(bv, Mc + (kb * 16 + l8 + (lq & 1) * 8) * XM_PAD + half * 128 + (np * 2 + (lq >> 1)) * 8);
                mma_16816(out[np * 2], ap, bv[0], bv[1]);
                mma_16816(out[np * 2 + 1], ap, bv[2], bv[3]);
            }
        }
    }
    s_lo += __shfl_xor_sync(0xffffffffu, s_lo, 1);
    s_lo += __shfl_xor_sync(0xffffffffu, s_lo, 2);
    s_hi += __shfl_xor_sync(0xffffffffu, s_hi, 1);
    s_hi += __shfl_xor_sync(0xffffffffu, s_hi, 2);
    if (t4 == 0) {
        my_red[g * 2 + 1] = s_lo;
        my_red[(g + 8) * 2 + 1] = s_hi;
    }
    asm volatile("bar.sync %0, 64;" ::"r"(1 + mt) : "memory");
    // all keys masked -> sum 0 -> NaN, like torch's softmax of all -inf
    const float i_lo = 1.f / (s_lo + other_red[g * 2 + 1]), i_hi = 1.f / (s_hi + other_red[(g + 8) * 2 + 1]);
    __half* o_lo_p = pm + q_lo * ldp + (h_lo < 0 ? 0 : h_lo) * D + half * 128 + t4 * 2;
    __half* o_hi_p = pm + q_hi * ldp + (h_hi < 0 ? 0 : h_hi) * D + half * 128 + t4 * 2;
#pragma unroll
    for (int nt = 0; nt < 16; ++nt) {
        if (h_lo >= 0) *reinterpret_cast<uint32_t*>(o_lo_p + nt * 8) = pack_half2(out[nt][0] * i_lo, out[nt][1] * i_lo);
        if (h_hi >= 0) *reinterpret_cast<uint32_t*>(o_hi_p + nt * 8) = pack_half2(out[nt][2] * i_hi, out[nt][3] * i_hi);
    }
}

}  // namespace

int enc_self_attention(const float* qk, int64_t ldqk, const float* v, int64_t ldv, float* o, int64_t ldo,
                       const int32_t* vlen, const int32_t* tlen, int64_t B, int Lv, int Lt, int nheads,
                       cudaStream_t s) {
    if (B == 0) return CONE_OK;
    const int S = Lv + Lt;
    CONE_REQUIRE(S <= MAX_S_LONG, "enc_self_attention: window of %d rows exceeds %d", S, MAX_S_LONG);
    const size_t smem = sizeof(float) * ((size_t)S * (HD + 1) + (size_t)S * HD + ENC_WARPS * HD + (size_t)ENC_WARPS * S);
    dim3 grid((unsigned)B, (unsigned)nheads);
    ProfScope ps(s, P_ENC_ATTN, 4.0 * (double)B * nheads * S * S * HD, 16.0 * (double)B * S * nheads * HD);
    if (S <= MAX_S) {
        static bool attr_set = false;
        if (!attr_set) {
            CONE_CUDA(cudaFuncSetAttribute(enc_self_attention_kernel<MAX_S / 32>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                           100 * 1024));
            attr_set = true;
        }
        enc_self_attention_kernel<MAX_S / 32><<<grid, ENC_WARPS * 32, smem, s>>>(qk, ldqk, v, ldv, o, ldo, vlen, tlen, Lv, Lt,
                                                                                nheads * HD);
    } else {  // long windows: 16 keys per lane, up to 139 KB of shared memory at 512 rows
        static bool attr_set = false;
        if (!attr_set) {
            const size_t smem_max = sizeof(float) * ((size_t)MAX_S_LONG * (2 * HD + 1) + ENC_WARPS * HD + (size_t)ENC_WARPS * MAX_S_LONG);
            CONE_CUDA(cudaFuncSetAttribute(enc_self_attention_kernel<MAX_S_LONG / 32>,
                                           cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_max));
            attr_set = true;
        }
        enc_self_attention_kernel<MAX_S_LONG / 32><<<grid, ENC_WARPS * 32, smem, s>>>(qk, ldqk, v, ldv, o, ldo, vlen, tlen, Lv,
                                                                                     Lt, nheads * HD);
    }
    CONE_LAUNCH_CHECK("enc_self_attention");
    return CONE_OK;
}

int dec_self_attention(const void* qk, int64_t ldqk, const void* v, int64_t ldv, void* o, int64_t ldo, int64_t B,
                       int nq, int nheads, int f16, cudaStream_t s) {
    if (B == 0) return CONE_OK;
    CONE_REQUIRE(nq <= 8, "dec_self_attention: at most 8 moment slots");
    const int warps = 4;
    ProfScope ps(s, P_DEC_ATTN);
    const unsigned grid = (unsigned)cdiv64(B * nheads, warps);
    if (f16) {
        dec_self_attention_kernel<__half><<<grid, warps * 32, 0, s>>>(static_cast<const __half*>(qk), ldqk,
                                                                    static_cast<const __half*>(v), ldv,
                                                                    static_cast<__half*>(o), ldo, B, nq, nheads, nheads * HD);
    } else {
        dec_self_attention_kernel<float><<<grid, warps * 32, 0, s>>>(static_cast<const float*>(qk), ldqk,
                                                                   static_cast<const float*>(v), ldv,
                                                                   static_cast<float*>(o), ldo, B, nq, nheads, nheads * HD);
    }
    CONE_LAUNCH_CHECK("dec_self_attention");
    return CONE_OK;
}

int dec_cross_attention(const void* q_any, int64_t ldq, const void* k, int64_t ldk, const void* v, int64_t ldv,
                        void* o_any, int64_t ldo, const int32_t* vlen, const int32_t* tlen, int64_t B, int nq, int Lv,
                        int Lt, int nheads, int kv_f16, const void* posk_any, int64_t ldposk, int table_lv,
                        cudaStream_t s) {
    const float* posk = static_cast<const float*>(posk_any);
    const float* q = static_cast<const float*>(q_any);  // fp32 mode; in fp16 mode q and o are fp16 as well
    float* o = static_cast<float*>(o_any);
    if (B == 0) return CONE_OK;
    const int S = Lv + Lt;
    CONE_REQUIRE(nq >= 1 && nq <= 8 && S <= MAX_S_LONG && nheads == 8, "dec_cross_attention: unsupported nq=%d S=%d heads=%d",
                 nq, S, nheads);
    CONE_REQUIRE((ldk & 7) == 0, "dec_cross_attention: ldk must be a multiple of 8");
    const int NQ = nq <= 5 ? 5 : 8;
    const int Sp = (S + 3) & ~3;
    const size_t smem = sizeof(float) * ((size_t)8 * NQ * Sp + 8 * NQ + (size_t)8 * NQ * 8 * 32);
    ProfScope ps(s, P_DEC_ATTN, 4.0 * (double)B * nheads * nq * S * HD, (kv_f16 ? 4.0 : 8.0) * (double)B * S * nheads * HD);
    const unsigned grid = (unsigned)B;
    // long windows (S > 256): 16 scores per lane in the softmax phase, up to 192 KB of shared memory at 512 rows
#define CONE_XATT(KV, NQV, KPL, SMEM_MAX)                                                                               \
    do {                                                                                                                \
        static bool attr = false;                                                                                       \
        if (!attr) {                                                                                                    \
            CONE_CUDA(cudaFuncSetAttribute(dec_cross_attention_kernel<KV, NQV, KPL>,                                    \
                                           cudaFuncAttributeMaxDynamicSharedMemorySize, (int)(SMEM_MAX)));              \
            attr = true;                                                                                                \
        }                                                                                                               \
        dec_cross_attention_kernel<KV, NQV, KPL><<<grid, 256, smem, s>>>(q, ldq, static_cast<const KV*>(k), ldk,        \
                                                                         static_cast<const KV*>(v), ldv, o, ldo, vlen,  \
                                                                         tlen, nq, Lv, Lt, posk, ldposk, table_lv);     \
    } while (0)
    CONE_REQUIRE(!kv_f16, "dec_cross_attention: the tensor-core decoder uses dec_cross_attention_mem");
    const size_t smem_long = sizeof(float) * ((size_t)8 * NQ * MAX_S_LONG + 8 * NQ + (size_t)8 * NQ * 8 * 32);
    if (S <= MAX_S) {
        if (NQ == 5) CONE_XATT(float, 5, MAX_S / 32, 160 * 1024); else CONE_XATT(float, 8, MAX_S / 32, 160 * 1024);
    } else {
        if (NQ == 5) CONE_XATT(float, 5, MAX_S_LONG / 32, smem_long); else CONE_XATT(float, 8, MAX_S_LONG / 32, smem_long);
    }

#undef CONE_XATT
    CONE_LAUNCH_CHECK("dec_cross_attention");
    return CONE_OK;
}

int enc_self_attention_f16(const void* qk, int64_t ldqk, const void* v, int64_t ldv, void* o, int64_t ldo,
                           const int32_t* vlen, const int32_t* tlen, int64_t B, int Lv, int Lt, int nheads,
                           const void* posqk16, int table_lv, cudaStream_t s, const void* frame_qkv,
                           const void* token_qkv, const int64_t* vid_base, const int64_t* txt_base, int64_t n_frames) {
    if (B == 0) return CONE_OK;
    const int S = Lv + Lt;
    CONE_REQUIRE(S <= MAX_S_LONG, "enc_self_attention_f16: window of %d rows exceeds %d", S, MAX_S_LONG);
    CONE_REQUIRE((ldqk % 8) == 0 && (ldv % 8) == 0 && (ldo % 2) == 0, "enc_self_attention_f16: leading dims must keep 16-byte rows");
    const int Sp = (S + 15) & ~15;
    const size_t smem = sizeof(__half) * (size_t)3 * Sp * QK_PAD + sizeof(float) * Sp;
    dim3 grid((unsigned)(B * nheads));
    ProfScope ps(s, P_ENC_ATTN, 4.0 * (double)B * nheads * S * S * HD, 8.0 * (double)B * S * nheads * HD);
    const __half* qk16 = static_cast<const __half*>(qk);
    const __half* v16 = static_cast<const __half*>(v);
    __half* o16 = static_cast<__half*>(o);
#define CONE_ENC_ATT(NBV, EX)                                                                                      \
    enc_attention_f16_kernel<NBV, EX><<<grid, ATT_WARPS * 32, smem, s>>>(qk16, ldqk, v16, ldv, o16, ldo, vlen, tlen, Lv, Lt, \
                                                                       nheads * HD, static_cast<const __half*>(posqk16), table_lv, rs)
    EncRowSource rs{static_cast<const __half*>(frame_qkv), static_cast<const __half*>(token_qkv), vid_base, txt_base, n_frames};
    CONE_REQUIRE(frame_qkv == nullptr || (token_qkv && vid_base && txt_base && n_frames > 0),
                 "enc_self_attention_f16: incomplete row tables");
    if (Sp == 160) {  // MAD windows: 125 frames + 25 tokens
        CONE_ENC_ATT(20, true);
    } else if (Sp <= 160) {
        CONE_ENC_ATT(20, false);
    } else if (Sp <= MAX_S) {
        static bool attr = false;
        if (!attr) {
            CONE_CUDA(cudaFuncSetAttribute(enc_attention_f16_kernel<32, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024));
            attr = true;
        }
        CONE_ENC_ATT(32, false);
    } else {  // long windows: 16 warps, tile loaded in rounds, online softmax over 64-key chunks (123 KB at 512 rows)
        static bool attr = false;
        if (!attr) {
            const int smem_max = (int)(sizeof(__half) * (size_t)3 * MAX_S_LONG * QK_PAD + sizeof(float) * MAX_S_LONG);
            CONE_CUDA(cudaFuncSetAttribute(enc_attention_f16_long_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem_max));
            attr = true;
        }
        enc_attention_f16_long_kernel<<<grid, LA_WARPS * 32, smem, s>>>(qk16, ldqk, v16, ldv, o16, ldo, vlen, tlen, Lv, Lt,
                                                                        nheads * HD, static_cast<const __half*>(posqk16),
                                                                        table_lv, rs);
    }
#undef CONE_ENC_ATT
    CONE_LAUNCH_CHECK("enc_self_attention_f16");
    return CONE_OK;
}

// long windows (256 < S <= 512): the memory streamed in chunks of XL_KC rows (see the kernel's comment)
static int dec_cross_attention_mem_long(const void* mem, int64_t ldm, const void* qqt, int64_t ldq, void* pm, int64_t ldp,
                                        const int32_t* vlen, const int32_t* tlen, int64_t B, int nq, int Lv, int Lt,
                                        const void* posk, int64_t ldposk, int table_lv, cudaStream_t s, int q_bcast, int MT) {
    const int S = Lv + Lt;
    const size_t smem = ((size_t)(2 * XL_KC + MT * 16) * XM_PAD + (size_t)MT * 16 * (XL_KC + 8)) * sizeof(__half) +
                        (size_t)MT * 2 * 16 * 2 * sizeof(float);
    ProfScope ps(s, P_DEC_ATTN, 2.0 * 2.0 * (double)B * 8 * nq * S * 256, 2.0 * (double)B * S * 256 + 2.0 * 2.0 * (double)B * nq * 9 * 256);
#define CONE_XMEM_LONG(MTV)                                                                                             \
    do {                                                                                                                \
        static bool attr = false;                                                                                       \
        if (!attr) {                                                                                                    \
            CONE_CUDA(cudaFuncSetAttribute(dec_cross_attention_mem_long_kernel<MTV>,                                    \
                                           cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));                    \
            attr = true;                                                                                                \
        }                                                                                                               \
        dec_cross_attention_mem_long_kernel<MTV><<<(unsigned)B, MTV * 64, smem, s>>>(                                   \
            static_cast<const __half*>(mem), ldm, static_cast<const __half*>(qqt), ldq, static_cast<__half*>(pm), ldp,  \
            vlen, tlen, nq, Lv, Lt, static_cast<const __half*>(posk), ldposk, table_lv, q_bcast);                       \
    } while (0)
    if (MT == 3) CONE_XMEM_LONG(3);
    else CONE_XMEM_LONG(4);
#undef CONE_XMEM_LONG
    CONE_LAUNCH_CHECK("dec_cross_attention_mem");
    return CONE_OK;
}

// q | qt [B nq, 256 + 8 * 256] fp16 -> attention-pooled memory pm [B nq, 8 * 256] fp16 (see the kernel's comment)
int dec_cross_attention_mem(const void* mem, int64_t ldm, const void* qqt, int64_t ldq, void* pm, int64_t ldp,
                            const int32_t* vlen, const int32_t* tlen, int64_t B, int nq, int Lv, int Lt, const void* posk,
                            int64_t ldposk, int table_lv, cudaStream_t s, int q_bcast) {
    if (B == 0) return CONE_OK;
    const int S = Lv + Lt;
    CONE_REQUIRE(nq >= 1 && nq <= 8 && S <= MAX_S_LONG, "dec_cross_attention_mem: unsupported nq=%d S=%d", nq, S);
    CONE_REQUIRE((ldm & 7) == 0 && (ldq & 7) == 0 && (ldp & 1) == 0 && (ldposk & 7) == 0,
                 "dec_cross_attention_mem: rows must be 16-byte aligned");
    const int MT = nq <= 6 ? 3 : 4;  // warps = 16-row blocks of the 8 nq score rows (rows past 8 nq are zero)
    if (S > MAX_S) return dec_cross_attention_mem_long(mem, ldm, qqt, ldq, pm, ldp, vlen, tlen, B, nq, Lv, Lt, posk, ldposk,
                                                       table_lv, s, q_bcast, MT);
    const int NB = S <= 112 ? 14 : (S <= 160 ? 20 : (S <= 208 ? 26 : 32));  // key blocks of 8, all processed
    const size_t smem = (size_t)(NB * 8 + MT * 16) * XM_PAD * sizeof(__half) + (size_t)MT * 2 * 16 * 2 * sizeof(float);
    // algorithmic work: both products over the raw memory, which is read once
    ProfScope ps(s, P_DEC_ATTN, 2.0 * 2.0 * (double)B * 8 * nq * S * 256, 2.0 * (double)B * S * 256 + 2.0 * 2.0 * (double)B * nq * 9 * 256);
#define CONE_XMEM(NBV, MTV)                                                                                             \
    do {                                                                                                                \
        static bool attr = false;                                                                                       \
        if (!attr) {                                                                                                    \
            CONE_CUDA(cudaFuncSetAttribute(dec_cross_attention_mem_kernel<NBV, MTV>,                                    \
                                           cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));                    \
            attr = true;                                                                                                \
        }                                                                                                               \
        dec_cross_attention_mem_kernel<NBV, MTV><<<(unsigned)B, MTV * 64, smem, s>>>(                                   \
            static_cast<const __half*>(mem), ldm, static_cast<const __half*>(qqt), ldq, static_cast<__half*>(pm), ldp,  \
            vlen, tlen, nq, Lv, Lt, static_cast<const __half*>(posk), ldposk, table_lv, q_bcast);                       \
    } while (0)
#define CONE_XMEM_MT(NBV)            \
    do {                             \
        if (MT == 3) CONE_XMEM(NBV, 3); \
        else CONE_XMEM(NBV, 4);      \
    } while (0)
    if (NB == 14) CONE_XMEM_MT(14);
    else if (NB == 20) CONE_XMEM_MT(20);
    else if (NB == 26) CONE_XMEM_MT(26);
    else CONE_XMEM_MT(32);
#undef CONE_XMEM_MT
#undef CONE_XMEM
    CONE_LAUNCH_CHECK("dec_cross_attention_mem");
    return CONE_OK;
}

}  // namespace cone
