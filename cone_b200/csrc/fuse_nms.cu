// Stage 3 of the reference, one CTA per query (cone/inference.py:70-91, 103-127, 169-217;
// utils/temporal_nms.py:6-74).  Everything after the fp32 span arithmetic is fp64, as in the reference's
// Python floats; orderings are stable with the insertion ordinal (window rank, then within-window score
// rank) as the secondary key (SURVEY.md §7 H4).
#include <climits>

#include "kernels.h"

namespace cone {

namespace {

constexpr int NMS_THREADS = 128;
constexpr int MAX_NQ = 8;

// float(f"{x:.4f}") for a value that came from fp32: x*1e4 is exact in fp64 (24+10 significant bits),
// rint is round-half-even like Python's correctly rounded formatting, and n/1e4 is the correctly rounded
// quotient, i.e. the double nearest to the decimal string.
__device__ __forceinline__ double round4(float x) { return rint((double)x * 1e4) / 1e4; }

// A10 for window g = q * topk + j of a query: seconds in fp32 (no FMA contraction), stable sort by fp32 score within
// the window, 4-decimal rounding.  Writes rows j*nq .. j*nq+nq-1.  Both stage-3 kernels call this, so they give the
// same bits.
__device__ __forceinline__ void a10_window_rows(const float* __restrict__ pred_spans, const float* __restrict__ prob_fg,
                                                const float* __restrict__ match, const int32_t* __restrict__ win_start,
                                                const int32_t* __restrict__ win_len, int64_t g, int j, int nq,
                                                float clip_length, int fixed_duration, int sort_windows, double* st,
                                                double* ed, double* sc, double* mt) {
    // eval_epoch scales by the window's own length (inference.py:75-78), the demo by max_v_l (cone_localizator.py:188)
    const float dur = fixed_duration > 0 ? (float)fixed_duration : (float)win_len[g], vs = (float)win_start[g];
    int idx[MAX_NQ];
    float key[MAX_NQ];
    for (int a = 0; a < nq; ++a) {
        const float k = prob_fg[g * nq + a];
        int pos = a;
        // the demo keeps slot order (cone_localizator.py:186-197): no per-window sort
        while (sort_windows && pos > 0 && key[pos - 1] < k) {  // strict: equal scores keep slot order
            key[pos] = key[pos - 1];
            idx[pos] = idx[pos - 1];
            --pos;
        }
        key[pos] = k;
        idx[pos] = a;
    }
    for (int a = 0; a < nq; ++a) {
        const int64_t p = g * nq + idx[a];
        const float cx = pred_spans[p * 2], w = pred_spans[p * 2 + 1];
        const float hw = __fmul_rn(0.5f, w);
        const float x1 = __fsub_rn(cx, hw), x2 = __fadd_rn(cx, hw);
        const float s = __fmul_rn(__fadd_rn(__fmul_rn(x1, dur), vs), clip_length);
        const float e = __fmul_rn(__fadd_rn(__fmul_rn(x2, dur), vs), clip_length);
        const int r = j * nq + a;
        st[r] = round4(s);
        ed[r] = round4(e);
        sc[r] = round4(prob_fg[p]);
        mt[r] = round4(match[p]);
    }
}

// A11: min-max normalisation of both scores (identity when constant) and their sum
__device__ __forceinline__ double a11_fusion(double sc, double mt, double smin, double smax, double mmin, double mmax) {
    const double a = (smin == smax) ? sc : (sc - smin) / (smax - smin);
    const double b = (mmin == mmax) ? mt : (mt - mmin) / (mmax - mmin);
    return a + b;
}

// compute_temporal_iou (temporal_nms.py:6-22): intersection over the hull, 0 when the hull is empty
__device__ __forceinline__ double hull_iou(double s1, double e1, double s2, double e2) {
    const double inter = fmax(0.0, fmin(e1, e2) - fmax(s1, s2));
    const double hull = fmax(e1, e2) - fmin(s1, s2);
    return hull == 0.0 ? 0.0 : inter / hull;
}

// Greedy NMS over candidates order[0..P) (already sorted, best first).  Writes kept candidate ids.
// Equivalent to temporal_nms.py:45-71 including its "append the last survivor" tail.
__device__ int greedy_nms(const double* st, const double* ed, const int* order, int P, double thd, int max_after,
                          unsigned char* dead, int* kept, int* sh_head) {
    for (int i = threadIdx.x; i < P; i += blockDim.x) dead[i] = 0;
    __syncthreads();
    if (P == 1) {  // `if len(predictions) == 1: return predictions`
        if (threadIdx.x == 0) kept[0] = order[0];
        __syncthreads();
        return max_after >= 0 ? 1 : 0;
    }
    int nkept = 0;
    int head = 0;
    while (nkept < max_after) {
        if (threadIdx.x == 0) {
            int h = head;
            while (h < P && dead[h]) ++h;
            *sh_head = h;
        }
        __syncthreads();
        head = *sh_head;
        if (head >= P) break;
        const int c = order[head];
        const double s1 = st[c], e1 = ed[c];
        for (int t = head + 1 + threadIdx.x; t < P; t += blockDim.x) {
            if (!dead[t]) {
                const int o = order[t];
                if (hull_iou(s1, e1, st[o], ed[o]) > thd) dead[t] = 1;
            }
        }
        if (threadIdx.x == 0) kept[nkept] = c;
        ++nkept;
        ++head;
        __syncthreads();
    }
    __syncthreads();
    return nkept;
}

// stable descending rank by value: position of i = #{j : v[j] > v[i] or (v[j] == v[i] and j < i)}.
// NaN (undefined order in the reference's Python sort) is ranked last so that `order` is always a permutation.
__device__ void stable_rank_desc(const double* v, int M, int* order) {
    for (int i = threadIdx.x; i < M; i += blockDim.x) {
        const double vi = v[i];
        const bool ni = vi != vi;
        int r = 0;
        for (int j = 0; j < M; ++j) {
            const double vj = v[j];
            const bool nj = vj != vj;
            r += (ni || nj) ? ((ni && !nj) || (ni && nj && j < i)) : ((vj > vi) || (vj == vi && j < i));
        }
        order[r] = i;
    }
    __syncthreads();
}

struct Smem {
    double *st, *ed, *sc, *mt, *fu;      // N rows in insertion order
    double *ust, *ued, *usc, *umt, *ufu;  // M unique (st,ed) entries: first position, last value
    int *last, *order, *kept;
    unsigned char* dead;
};

__device__ Smem carve(unsigned char* base, int N) {
    Smem s;
    double* d = reinterpret_cast<double*>(base);
    s.st = d; s.ed = d + N; s.sc = d + 2 * N; s.mt = d + 3 * N; s.fu = d + 4 * N;
    s.ust = d + 5 * N; s.ued = d + 6 * N; s.usc = d + 7 * N; s.umt = d + 8 * N; s.ufu = d + 9 * N;
    int* i = reinterpret_cast<int*>(d + 10 * N);
    s.last = i; s.order = i + N; s.kept = i + 2 * N;
    s.dead = reinterpret_cast<unsigned char*>(i + 3 * N);
    return s;
}

__host__ __device__ constexpr size_t smem_bytes(int N) { return (size_t)N * (10 * 8 + 3 * 4 + 1) + 64; }

__global__ void __launch_bounds__(NMS_THREADS)
fuse_nms_kernel(const float* __restrict__ pred_spans, const float* __restrict__ prob_fg, const float* __restrict__ match,
                const int32_t* __restrict__ win_start, const int32_t* __restrict__ win_len, int topk, int nq,
                float clip_length, double nms_thd, int max_before, int max_after, int fixed_duration, int sort_windows,
                double* __restrict__ out, int32_t* __restrict__ out_count, double* __restrict__ rows_out,
                int32_t* __restrict__ rows_count) {
    extern __shared__ __align__(16) unsigned char raw[];
    __shared__ int sh_head, sh_M, sh_cnt;
    __shared__ double sh_mm[4];
    const int q = blockIdx.x;
    const int Nmax = topk * nq;
    Smem s = carve(raw, Nmax);

    // present windows form a prefix of the top-k list (absent ones have len 0)
    if (threadIdx.x == 0) {
        int c = 0;
        while (c < topk && win_len[(int64_t)q * topk + c] > 0) ++c;
        sh_cnt = c;
    }
    __syncthreads();
    const int cnt = sh_cnt;
    const int N = cnt * nq;

    for (int j = threadIdx.x; j < cnt; j += blockDim.x)
        a10_window_rows(pred_spans, prob_fg, match, win_start, win_len, (int64_t)q * topk + j, j, nq, clip_length,
                        fixed_duration, sort_windows, s.st, s.ed, s.sc, s.mt);
    __syncthreads();
    if (rows_out) {
        for (int r = threadIdx.x; r < N; r += blockDim.x) {
            double* o = rows_out + ((int64_t)q * Nmax + r) * 4;
            o[0] = s.st[r]; o[1] = s.ed[r]; o[2] = s.sc[r]; o[3] = s.mt[r];
        }
        if (threadIdx.x == 0 && rows_count) rows_count[q] = N;
    }
    if (N == 0) {
        if (threadIdx.x < 3) out_count[q * 3 + threadIdx.x] = 0;
        return;
    }

    // A11: min-max over all N rows, before de-duplication
    if (threadIdx.x < 4) {
        const double* v = (threadIdx.x < 2) ? s.sc : s.mt;
        const bool want_max = threadIdx.x & 1;
        double m = v[0];
        for (int r = 1; r < N; ++r) m = want_max ? (v[r] > m ? v[r] : m) : (v[r] < m ? v[r] : m);
        sh_mm[threadIdx.x] = m;
    }
    __syncthreads();
    {
        const double smin = sh_mm[0], smax = sh_mm[1], mmin = sh_mm[2], mmax = sh_mm[3];
        for (int r = threadIdx.x; r < N; r += blockDim.x) {
            s.fu[r] = a11_fusion(s.sc[r], s.mt[r], smin, smax, mmin, mmax);
        }
    }
    __syncthreads();
    // dict keyed by (st, ed): first position, last value
    for (int r = threadIdx.x; r < N; r += blockDim.x) {
        const double a = s.st[r], b = s.ed[r];
        int first = r, last = r;
        for (int t = 0; t < N; ++t) {
            if (s.st[t] == a && s.ed[t] == b) {
                if (t < first) first = t;
                if (t > last) last = t;
            }
        }
        s.last[r] = (first == r) ? last : -1;
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        int m = 0;
        for (int r = 0; r < N; ++r) {
            const int l = s.last[r];
            if (l >= 0) {
                s.ust[m] = s.st[r]; s.ued[m] = s.ed[r];
                s.usc[m] = s.sc[l]; s.umt[m] = s.mt[l]; s.ufu[m] = s.fu[l];
                ++m;
            }
        }
        sh_M = m;
    }
    __syncthreads();
    const int M = sh_M;

    // A12/A13: three rankings — 0 fusion (idx 2), 1 proposal (idx 0), 2 matching (idx 1)
    for (int mode = 0; mode < 3; ++mode) {
        const double* val = mode == 0 ? s.ufu : (mode == 1 ? s.usc : s.umt);
        stable_rank_desc(val, M, s.order);
        int nk;
        if (nms_thd != -1.0) {
            const int P = M < max_before ? M : max_before;
            nk = greedy_nms(s.ust, s.ued, s.order, P, nms_thd, max_after, s.dead, s.kept, &sh_head);
        } else {
            nk = M < max_after ? M : max_after;
            for (int i = threadIdx.x; i < nk; i += blockDim.x) s.kept[i] = s.order[i];
            __syncthreads();
        }
        for (int i = threadIdx.x; i < nk; i += blockDim.x) {
            const int c = s.kept[i];
            double* o = out + (((int64_t)q * 3 + mode) * max_after + i) * 5;
            o[0] = s.ust[c]; o[1] = s.ued[c]; o[2] = s.usc[c]; o[3] = s.umt[c]; o[4] = s.ufu[c];
        }
        if (threadIdx.x == 0) out_count[q * 3 + mode] = nk;
        __syncthreads();
    }
}

__global__ void __launch_bounds__(NMS_THREADS)
temporal_nms_single_kernel(const double* __restrict__ st, const double* __restrict__ ed,
                           const double* __restrict__ score, int n, double thd, int max_after,
                           int32_t* __restrict__ keep_out, int32_t* __restrict__ n_keep_out) {
    extern __shared__ __align__(16) unsigned char raw[];
    __shared__ int sh_head;
    int* order = reinterpret_cast<int*>(raw);
    int* kept = order + n;
    unsigned char* dead = reinterpret_cast<unsigned char*>(kept + n);
    if (n == 0) {
        if (threadIdx.x == 0) n_keep_out[0] = 0;
        return;
    }
    stable_rank_desc(score, n, order);
    const int nk = greedy_nms(st, ed, order, n, thd, max_after, dead, kept, &sh_head);
    for (int i = threadIdx.x; i < nk; i += blockDim.x) keep_out[i] = kept[i];
    if (threadIdx.x == 0) n_keep_out[0] = nk;
}


// ---- the workspace path: any number of candidates up to FUSE_WS_MAX_N, O(N log N) per query -------------------------
// One CTA per query, every per-row array in the workspace.  Orderings are LSD radix sorts (8-bit digits, stable) of an
// index array on 64-bit keys computed from the fp64 values, so ties keep index order exactly as stable_rank_desc does.

constexpr int WS_THREADS = 512;
constexpr int WS_WARPS = WS_THREADS / 32;
constexpr int FUSE_WS_MAX_N = CONE_FUSE_NMS_MAX_CANDIDATES;
static_assert(FUSE_WS_MAX_N == 16384 * MAX_NQ, "the longest rank-list times the most slots");
static_assert(smem_bytes(CONE_FUSE_NMS_MAX_SHARED_CANDIDATES) <= 200 * 1024 &&
              smem_bytes(CONE_FUSE_NMS_MAX_SHARED_CANDIDATES + 1) > 200 * 1024, "the documented limit of fuse_nms_kernel");

// ascending order of doubles as unsigned integers; -0.0 and +0.0 share a key, every NaN maps past +inf
__device__ __forceinline__ uint64_t key_asc(double x) {
    if (x != x) return ~0ull;
    const uint64_t u = (uint64_t)__double_as_longlong(x == 0.0 ? 0.0 : x);
    return (u >> 63) ? ~u : (u | (1ull << 63));
}
// descending order, NaN last
__device__ __forceinline__ uint64_t key_desc(double x) { return x != x ? ~0ull : ~key_asc(x); }

struct __align__(16) WsSmem {
    int hist[256];
    int warp_hist[WS_WARPS][256];
    int warp_tot[WS_WARPS];
    int flag;
};

// inclusive block-wide sum (max_op = 0) or max (max_op = 1) of one value per thread; *total gets the block's result
__device__ int block_scan(int v, bool max_op, WsSmem& sm, int* total) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int o = 1; o < 32; o <<= 1) {
        const int t = __shfl_up_sync(0xffffffffu, v, o);
        if (lane >= o) v = max_op ? max(v, t) : v + t;
    }
    if (lane == 31) sm.warp_tot[warp] = v;
    __syncthreads();
    if (warp == 0) {
        int t = lane < WS_WARPS ? sm.warp_tot[lane] : (max_op ? INT_MIN : 0);
        for (int o = 1; o < 32; o <<= 1) {
            const int u = __shfl_up_sync(0xffffffffu, t, o);
            if (lane >= o) t = max_op ? max(t, u) : t + u;
        }
        if (lane < WS_WARPS) sm.warp_tot[lane] = t;
    }
    __syncthreads();
    if (warp > 0) v = max_op ? max(v, sm.warp_tot[warp - 1]) : v + sm.warp_tot[warp - 1];
    *total = sm.warp_tot[WS_WARPS - 1];
    __syncthreads();
    return v;
}

// one stable counting pass on digit `shift` of key(idx); returns false (and leaves `out` untouched) when every element
// has the same digit, i.e. the pass would not move anything
template <class KeyFn>
__device__ bool radix_pass(const int* in, int* out, int n, int shift, KeyFn key, WsSmem& sm) {
    for (int b = threadIdx.x; b < 256; b += blockDim.x) sm.hist[b] = 0;
    if (threadIdx.x == 0) sm.flag = 0;
    __syncthreads();
    for (int i = threadIdx.x; i < n; i += blockDim.x) atomicAdd(&sm.hist[(key(in[i]) >> shift) & 255], 1);
    __syncthreads();
    for (int b = threadIdx.x; b < 256; b += blockDim.x)
        if (sm.hist[b] == n) sm.flag = 1;
    __syncthreads();
    const bool skip = sm.flag;
    __syncthreads();  // every thread has read the flag before the next pass resets it
    if (skip) return false;
    if (threadIdx.x < 32) {  // exclusive scan of the 256 bins: 8 consecutive bins per lane
        const int lane = threadIdx.x;
        int c[8], sum = 0;
        for (int k = 0; k < 8; ++k) { c[k] = sm.hist[lane * 8 + k]; sum += c[k]; }
        int incl = sum;
        for (int o = 1; o < 32; o <<= 1) {
            const int t = __shfl_up_sync(0xffffffffu, incl, o);
            if (lane >= o) incl += t;
        }
        int run = incl - sum;
        for (int k = 0; k < 8; ++k) { sm.hist[lane * 8 + k] = run; run += c[k]; }
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    for (int base = 0; base < n; base += blockDim.x) {
        for (int t = threadIdx.x; t < WS_WARPS * 256; t += blockDim.x) (&sm.warp_hist[0][0])[t] = 0;
        __syncthreads();
        const int i = base + threadIdx.x;
        const int e = i < n ? in[i] : 0;
        const int d = i < n ? (int)((key(e) >> shift) & 255) : 256;
        const unsigned peers = __match_any_sync(0xffffffffu, d);
        const int rank = __popc(peers & ((1u << lane) - 1));
        if (d < 256 && rank == 0) sm.warp_hist[warp][d] = __popc(peers);
        __syncthreads();
        for (int b = threadIdx.x; b < 256; b += blockDim.x) {  // warp offsets within the bin, in warp order
            int run = sm.hist[b];
            for (int w = 0; w < WS_WARPS; ++w) {
                const int c = sm.warp_hist[w][b];
                sm.warp_hist[w][b] = run;
                run += c;
            }
            sm.hist[b] = run;
        }
        __syncthreads();
        if (d < 256) out[sm.warp_hist[warp][d] + rank] = e;
        __syncthreads();
    }
    return true;
}

// stable ascending sort of the index array *a (scratch *b) on a 64-bit key; returns the buffer holding the result
template <class KeyFn>
__device__ int* radix_sort64(int* a, int* b, int n, KeyFn key, WsSmem& sm) {
    for (int shift = 0; shift < 64; shift += 8) {
        if (radix_pass(a, b, n, shift, key, sm)) {
            int* t = a; a = b; b = t;
        }
    }
    return a;
}

// first-occurrence min / max as the sequential scans of fuse_nms_kernel give them: NaN never wins a comparison, equal
// values keep the earlier row
__device__ __forceinline__ bool wins(double v, int i, double u, int j, bool want_max) {
    if (v != v) return u != u && i < j;
    if (u != u) return true;
    return (want_max ? v > u : v < u) || (v == u && i < j);
}

struct WsQuery {
    double *st, *ed, *sc, *mt, *fu;
    double *ust, *ued, *usc, *umt, *ufu;
    int *ia, *ib, *last, *epos;
    unsigned char* dead;
};

__host__ __device__ inline size_t ws_query_bytes(int N) { return ((size_t)N * (10 * 8 + 4 * 4 + 1) + 255) / 256 * 256; }

__device__ WsQuery carve_ws(unsigned char* base, int N) {
    WsQuery s;
    double* d = reinterpret_cast<double*>(base);
    s.st = d; s.ed = d + N; s.sc = d + 2 * N; s.mt = d + 3 * N; s.fu = d + 4 * N;
    s.ust = d + 5 * N; s.ued = d + 6 * N; s.usc = d + 7 * N; s.umt = d + 8 * N; s.ufu = d + 9 * N;
    int* i = reinterpret_cast<int*>(d + 10 * N);
    s.ia = i; s.ib = i + N; s.last = i + 2 * N; s.epos = i + 3 * N;
    s.dead = reinterpret_cast<unsigned char*>(i + 4 * N);
    return s;
}

__global__ void __launch_bounds__(WS_THREADS)
fuse_nms_ws_kernel(const float* __restrict__ pred_spans, const float* __restrict__ prob_fg, const float* __restrict__ match,
                   const int32_t* __restrict__ win_start, const int32_t* __restrict__ win_len, int q0, int topk, int nq,
                   float clip_length, double nms_thd, int max_before, int max_after, int fixed_duration, int sort_windows,
                   double* __restrict__ out, int32_t* __restrict__ out_count, double* __restrict__ rows_out,
                   int32_t* __restrict__ rows_count, unsigned char* __restrict__ workspace) {
    __shared__ WsSmem sm;
    __shared__ int sh_head, sh_cnt;
    __shared__ double sh_mm[4];
    const int q = q0 + blockIdx.x;
    const int Nmax = topk * nq;
    const WsQuery s = carve_ws(workspace + ws_query_bytes(Nmax) * blockIdx.x, Nmax);

    // present windows form a prefix of the top-k list (absent ones have len 0)
    if (threadIdx.x == 0) {
        int c = 0;
        while (c < topk && win_len[(int64_t)q * topk + c] > 0) ++c;
        sh_cnt = c;
    }
    __syncthreads();
    const int cnt = sh_cnt;
    const int N = cnt * nq;
    for (int j = threadIdx.x; j < cnt; j += blockDim.x)
        a10_window_rows(pred_spans, prob_fg, match, win_start, win_len, (int64_t)q * topk + j, j, nq, clip_length,
                        fixed_duration, sort_windows, s.st, s.ed, s.sc, s.mt);
    __syncthreads();
    if (rows_out) {
        for (int r = threadIdx.x; r < N; r += blockDim.x) {
            double* o = rows_out + ((int64_t)q * Nmax + r) * 4;
            o[0] = s.st[r]; o[1] = s.ed[r]; o[2] = s.sc[r]; o[3] = s.mt[r];
        }
        if (threadIdx.x == 0 && rows_count) rows_count[q] = N;
    }
    if (N == 0) {
        if (threadIdx.x < 3) out_count[q * 3 + threadIdx.x] = 0;
        return;
    }

    // A11: min / max of score and match over all N rows: per thread, then per warp, then across warps
    {
        double v[4];
        int vi[4];
        for (int k = 0; k < 4; ++k) { v[k] = __longlong_as_double(0x7ff8000000000000ll); vi[k] = INT_MAX; }
        for (int r = threadIdx.x; r < N; r += blockDim.x) {
            for (int k = 0; k < 4; ++k) {
                const double x = k < 2 ? s.sc[r] : s.mt[r];
                if (wins(x, r, v[k], vi[k], k & 1)) { v[k] = x; vi[k] = r; }
            }
        }
        for (int k = 0; k < 4; ++k) {
            for (int o = 16; o > 0; o >>= 1) {
                const double u = __shfl_down_sync(0xffffffffu, v[k], o);
                const int j = __shfl_down_sync(0xffffffffu, vi[k], o);
                if (wins(u, j, v[k], vi[k], k & 1)) { v[k] = u; vi[k] = j; }
            }
        }
        double* wv = reinterpret_cast<double*>(&sm.warp_hist[0][0]);  // [4][WS_WARPS] doubles, then [4][WS_WARPS] ints
        int* wi = reinterpret_cast<int*>(wv + 4 * WS_WARPS);
        if ((threadIdx.x & 31) == 0)
            for (int k = 0; k < 4; ++k) { wv[k * WS_WARPS + (threadIdx.x >> 5)] = v[k]; wi[k * WS_WARPS + (threadIdx.x >> 5)] = vi[k]; }
        __syncthreads();
        if (threadIdx.x < 4) {
            const int k = threadIdx.x;
            double b = wv[k * WS_WARPS];
            int bi = wi[k * WS_WARPS];
            for (int w = 1; w < WS_WARPS; ++w)
                if (wins(wv[k * WS_WARPS + w], wi[k * WS_WARPS + w], b, bi, k & 1)) { b = wv[k * WS_WARPS + w]; bi = wi[k * WS_WARPS + w]; }
            const double first = k < 2 ? s.sc[0] : s.mt[0];
            sh_mm[k] = first != first ? first : b;  // a NaN first row stays the running extreme of the sequential scan
        }
        __syncthreads();
    }
    {
        const double smin = sh_mm[0], smax = sh_mm[1], mmin = sh_mm[2], mmax = sh_mm[3];
        for (int r = threadIdx.x; r < N; r += blockDim.x) s.fu[r] = a11_fusion(s.sc[r], s.mt[r], smin, smax, mmin, mmax);
    }

    // dict keyed by (st, ed): sort the rows on (st, ed, row), then every run of equal keys is one entry
    for (int r = threadIdx.x; r < N; r += blockDim.x) { s.ia[r] = r; s.last[r] = -1; }
    __syncthreads();
    const double* st = s.st;
    const double* ed = s.ed;
    int* perm = radix_sort64(s.ia, s.ib, N, [ed](int r) { return key_asc(ed[r]); }, sm);
    perm = radix_sort64(perm, perm == s.ia ? s.ib : s.ia, N, [st](int r) { return key_asc(st[r]); }, sm);
    int* gstart = perm == s.ia ? s.ib : s.ia;
    // position of each row's run start (inclusive max-scan of the start positions)
    int carry = 0;
    for (int base = 0; base < N; base += blockDim.x) {
        const int i = base + threadIdx.x;
        int v = 0;
        if (i < N && i > 0) {
            const int a = perm[i], b = perm[i - 1];
            v = (st[a] == st[b] && ed[a] == ed[b]) ? 0 : i;
        }
        int tot;
        const int incl = max(carry, block_scan(v, true, sm, &tot));
        if (i < N) gstart[i] = incl;
        carry = max(carry, tot);
    }
    __syncthreads();
    // the first row of a run (its smallest row index) points to the last one
    for (int i = threadIdx.x; i < N; i += blockDim.x) {
        const bool end = i == N - 1 || gstart[i + 1] != gstart[i];
        if (end) s.last[perm[gstart[i]]] = perm[i];
    }
    __syncthreads();
    // entries in first-occurrence order: exclusive count of run starts over the rows
    carry = 0;
    for (int base = 0; base < N; base += blockDim.x) {
        const int r = base + threadIdx.x;
        const int v = (r < N && s.last[r] >= 0) ? 1 : 0;
        int tot;
        const int incl = block_scan(v, false, sm, &tot);
        if (r < N) s.epos[r] = carry + incl - v;
        carry += tot;
    }
    const int M = carry;
    for (int r = threadIdx.x; r < N; r += blockDim.x) {
        const int l = s.last[r];
        if (l >= 0) {
            const int m = s.epos[r];
            s.ust[m] = s.st[r]; s.ued[m] = s.ed[r];
            s.usc[m] = s.sc[l]; s.umt[m] = s.mt[l]; s.ufu[m] = s.fu[l];
        }
    }
    __syncthreads();

    // A12/A13: three rankings — 0 fusion (idx 2), 1 proposal (idx 0), 2 matching (idx 1)
    int* kept = s.last;
    for (int mode = 0; mode < 3; ++mode) {
        const double* val = mode == 0 ? s.ufu : (mode == 1 ? s.usc : s.umt);
        for (int i = threadIdx.x; i < M; i += blockDim.x) s.ia[i] = i;
        __syncthreads();
        const int* order = radix_sort64(s.ia, s.ib, M, [val](int e) { return key_desc(val[e]); }, sm);
        int nk;
        if (nms_thd != -1.0) {
            const int P = M < max_before ? M : max_before;
            nk = greedy_nms(s.ust, s.ued, order, P, nms_thd, max_after, s.dead, kept, &sh_head);
        } else {
            nk = M < max_after ? M : max_after;
            for (int i = threadIdx.x; i < nk; i += blockDim.x) kept[i] = order[i];
            __syncthreads();
        }
        for (int i = threadIdx.x; i < nk; i += blockDim.x) {
            const int c = kept[i];
            double* o = out + (((int64_t)q * 3 + mode) * max_after + i) * 5;
            o[0] = s.ust[c]; o[1] = s.ued[c]; o[2] = s.usc[c]; o[3] = s.umt[c]; o[4] = s.ufu[c];
        }
        if (threadIdx.x == 0) out_count[q * 3 + mode] = nk;
        __syncthreads();
    }
}
}  // namespace

int fuse_nms(const float* pred_spans, const float* prob_fg, const float* match, const int32_t* win_start,
             const int32_t* win_len, int n_queries, int topk, int nq, float clip_length, double nms_thd,
             int max_before_nms, int max_after_nms, double* out, int32_t* out_count, double* rows_out,
             int32_t* rows_count, cudaStream_t s, int fixed_duration, int sort_windows) {
    if (n_queries == 0) return CONE_OK;
    CONE_REQUIRE(nq >= 1 && nq <= MAX_NQ, "fuse_nms: 1..%d moment slots supported", MAX_NQ);
    CONE_REQUIRE(max_after_nms >= 1 && max_before_nms >= 1, "fuse_nms: max_before/after_nms must be >= 1");
    const size_t smem = smem_bytes(topk * nq);
    CONE_REQUIRE(smem <= 200 * 1024, "fuse_nms: %d candidates per query exceed shared memory", topk * nq);
    if (smem > 48 * 1024)
        CONE_CUDA(cudaFuncSetAttribute(fuse_nms_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    ProfScope ps(s, P_NMS);
    fuse_nms_kernel<<<n_queries, NMS_THREADS, smem, s>>>(pred_spans, prob_fg, match, win_start, win_len, topk, nq,
                                                         clip_length, nms_thd, max_before_nms, max_after_nms,
                                                         fixed_duration, sort_windows, out, out_count, rows_out,
                                                         rows_count);
    CONE_LAUNCH_CHECK("fuse_nms");
    return CONE_OK;
}

size_t fuse_nms_workspace_bytes(int n_queries, int topk, int nq) {
    if (n_queries < 0 || topk < 1 || nq < 1 || nq > MAX_NQ) {
        set_error("fuse_nms_workspace_bytes: n_queries=%d topk=%d nq=%d (1..%d slots)", n_queries, topk, nq, MAX_NQ);
        return 0;
    }
    if ((int64_t)topk * nq > FUSE_WS_MAX_N) {
        set_error("fuse_nms_ws: %lld candidates per query exceed the limit of %d", (long long)topk * nq, FUSE_WS_MAX_N);
        return 0;
    }
    return ws_query_bytes(topk * nq) * (size_t)(n_queries > 1 ? n_queries : 1);
}

int fuse_nms_ws(const float* pred_spans, const float* prob_fg, const float* match, const int32_t* win_start,
                const int32_t* win_len, int n_queries, int topk, int nq, float clip_length, double nms_thd,
                int max_before_nms, int max_after_nms, double* out, int32_t* out_count, double* rows_out,
                int32_t* rows_count, void* workspace, size_t workspace_bytes, cudaStream_t s, int fixed_duration,
                int sort_windows) {
    CONE_REQUIRE(nq >= 1 && nq <= MAX_NQ, "fuse_nms_ws: 1..%d moment slots supported", MAX_NQ);
    CONE_REQUIRE(topk >= 1 && n_queries >= 0, "fuse_nms_ws: topk=%d n_queries=%d", topk, n_queries);
    CONE_REQUIRE(max_after_nms >= 1 && max_before_nms >= 1, "fuse_nms_ws: max_before/after_nms must be >= 1");
    CONE_REQUIRE((int64_t)topk * nq <= FUSE_WS_MAX_N, "fuse_nms_ws: %lld candidates per query exceed the limit of %d",
                 (long long)topk * nq, FUSE_WS_MAX_N);
    if (n_queries == 0) return CONE_OK;
    const size_t per_query = ws_query_bytes(topk * nq);
    if (!workspace || workspace_bytes < per_query) {
        set_error("fuse_nms_ws: workspace of %zu bytes cannot hold one query (%zu needed)", workspace_bytes, per_query);
        return CONE_ERR_WORKSPACE;
    }
    const int chunk = (int)(workspace_bytes / per_query < (size_t)n_queries ? workspace_bytes / per_query : n_queries);
    ProfScope ps(s, P_NMS);
    for (int q0 = 0; q0 < n_queries; q0 += chunk) {
        const int n = n_queries - q0 < chunk ? n_queries - q0 : chunk;
        fuse_nms_ws_kernel<<<n, WS_THREADS, 0, s>>>(pred_spans, prob_fg, match, win_start, win_len, q0, topk, nq,
                                                    clip_length, nms_thd, max_before_nms, max_after_nms, fixed_duration,
                                                    sort_windows, out, out_count, rows_out, rows_count,
                                                    static_cast<unsigned char*>(workspace));
        CONE_LAUNCH_CHECK("fuse_nms_ws");
    }
    return CONE_OK;
}

int temporal_nms_single(const double* st, const double* ed, const double* score, int n, double nms_thd,
                        int max_after_nms, int32_t* keep_out, int32_t* n_keep_out, cudaStream_t s) {
    CONE_REQUIRE(n >= 0 && max_after_nms >= 0, "temporal_nms: negative sizes");
    const size_t smem = (size_t)n * 9 + 64;
    CONE_REQUIRE(smem <= 200 * 1024, "temporal_nms: %d predictions exceed shared memory", n);
    if (smem > 48 * 1024)
        CONE_CUDA(cudaFuncSetAttribute(temporal_nms_single_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    temporal_nms_single_kernel<<<1, NMS_THREADS, smem, s>>>(st, ed, score, n, nms_thd, max_after_nms, keep_out,
                                                           n_keep_out);
    CONE_LAUNCH_CHECK("temporal_nms_single");
    return CONE_OK;
}

}  // namespace cone
