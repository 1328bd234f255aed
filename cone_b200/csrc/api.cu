// extern "C" entry points of libcone_b200 (include/cone_b200.h): weights handle, workspace planning and the
// launch sequences of the coarse-to-fine path.  No hidden allocation outside the weights handle.
#include <math.h>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <map>
#include <string>
#include <vector>

#include "kernels.h"
#include "tc_gemm.h"

namespace cone {

static thread_local char g_err[512] = "";
static thread_local int64_t g_launches = 0;

void set_error(const char* fmt, ...) {
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(g_err, sizeof(g_err), fmt, ap);
    va_end(ap);
}
void count_launch(int n) { g_launches += n; }

// ---- per-kernel profile -------------------------------------------------------------------------
namespace {
struct ProfRec {
    cudaEvent_t a, b;
    int cat;
    double flops, bytes;
};
thread_local bool g_prof_on = false;
thread_local std::vector<ProfRec> g_prof;
thread_local std::vector<cudaEvent_t> g_event_pool;
cudaEvent_t take_event() {
    if (!g_event_pool.empty()) {
        cudaEvent_t e = g_event_pool.back();
        g_event_pool.pop_back();
        return e;
    }
    cudaEvent_t e;
    cudaEventCreate(&e);
    return e;
}
}  // namespace

ProfScope::ProfScope(cudaStream_t s, ProfCat cat, double flops, double bytes) : slot(-1), stream(s) {
    if (!g_prof_on) return;
    ProfRec r{take_event(), take_event(), (int)cat, flops, bytes};
    cudaEventRecord(r.a, s);
    slot = (int)g_prof.size();
    g_prof.push_back(r);
}
ProfScope::~ProfScope() {
    if (slot >= 0) cudaEventRecord(g_prof[slot].b, stream);
}

}  // namespace cone

static const char* kProfNames[cone::P_COUNT] = {"gemm_fp32", "gemm_tc", "enc_attention", "dec_attention", "layernorm",
                                                "rowops", "frame_scores", "window_ranklist", "span_pool", "fuse_nms",
                                                "convert", "enc_tail", "enc_tail_gather"};
extern "C" void cone_profile_enable(int on) {
    cone::g_prof_on = on != 0;
    // events are created here, not at the first profiled launches: event creation inside a timed region showed up as
    // host-side gaps between launches
    if (on) {
        while (cone::g_event_pool.size() < 4096) {
            cudaEvent_t e;
            if (cudaEventCreate(&e) != cudaSuccess) break;
            cone::g_event_pool.push_back(e);
        }
    }
}
extern "C" int cone_profile_categories(void) { return cone::P_COUNT; }
extern "C" const char* cone_profile_name(int cat) { return (cat >= 0 && cat < cone::P_COUNT) ? kProfNames[cat] : ""; }
// Waits for the recorded events, adds them up per category and clears the log.
extern "C" int cone_profile_read(double* ms, int64_t* launches, double* flops, double* bytes, int ncat) {
    for (int i = 0; i < ncat; ++i) {
        ms[i] = 0; launches[i] = 0; flops[i] = 0; bytes[i] = 0;
    }
    for (auto& r : cone::g_prof) {
        float t = 0.f;
        cudaEventSynchronize(r.b);
        cudaEventElapsedTime(&t, r.a, r.b);
        if (r.cat < ncat) {
            ms[r.cat] += t; launches[r.cat] += 1; flops[r.cat] += r.flops; bytes[r.cat] += r.bytes;
        }
        cone::g_event_pool.push_back(r.a);
        cone::g_event_pool.push_back(r.b);
    }
    cone::g_prof.clear();
    return CONE_OK;
}

using namespace cone;

// ------------------------------------------------------------------------------------------------
// weights
// ------------------------------------------------------------------------------------------------
struct cone_weights {
    cone_dims dims;
    float* blob = nullptr;  // the state dict, canonical order, device
    size_t n_floats = 0;
    std::map<std::string, size_t> off;
    float* derived = nullptr;  // dec_kw | dec_kb | dec_vw | dec_vb | pos_table
    float *dec_kw = nullptr, *dec_kb = nullptr, *dec_vw = nullptr, *dec_vb = nullptr, *pos_table = nullptr;
    TcWeights* tc = nullptr;  // fp16 copies + TMA descriptors for the tensor-core path (lazy)
    // tensor-core path only (lazy): position embedding pushed through the q|k projections of every encoder layer
    // [enc_layers][(max_v_l+1)*max_v_l][2d] and through the decoder cross-attention K projections [..][DL*d]
    float* pos_proj = nullptr;
    std::vector<float*> pos_qk;
    float* pos_kdec = nullptr;
    uint16_t* pos_kdec16 = nullptr;  // fp16 copy for the mma.sync cross-attention
    uint16_t* pos_qk16 = nullptr;    // fp16 copy of pos_qk [enc_layers][rows][2d] for the tcgen05 attention (TMA boxes)
    // memory-direct cross-attention of the tensor-core decoder (attention.cu): per decoder layer
    //   xq_w [9 d, d], xq_b [9 d]: rows [0, d) = c Wq, rows d + h d + j = c Wk_h^T Wq_h (c = softmax scale * log2 e)
    //   xo_w [d, 8 d], xo_b [d]:   columns h d + j = Wo[:, head h] Wv_h;  xo_b = Wo bv + bo
    float* xattn = nullptr;
    std::vector<float*> xq_w, xq_b, xo_w, xo_b;
    const float* p(const std::string& name) const { return blob + off.at(name); }
};

// input width of input_vid_proj: the motion feature dim, which defaults to the appearance dim
static int motion_dim(const cone_dims& c) { return c.m_dim > 0 ? c.m_dim : c.v_dim; }

// the canonical order of cone_b200/weights.py::state_dict_shapes
static void layout(const cone_dims& c, std::vector<std::pair<std::string, size_t>>& out) {
    const size_t d = c.hidden, ff = c.ffn, dv = c.v_dim, dt = c.t_dim, dm = motion_dim(c);
    auto attn = [&](const std::string& p) {
        out.push_back({p + ".in_proj_weight", 3 * d * d});
        out.push_back({p + ".in_proj_bias", 3 * d});
        out.push_back({p + ".out_proj.weight", d * d});
        out.push_back({p + ".out_proj.bias", d});
    };
    auto ffn_norms = [&](const std::string& p, int n_norm) {
        out.push_back({p + ".linear1.weight", ff * d});
        out.push_back({p + ".linear1.bias", ff});
        out.push_back({p + ".linear2.weight", d * ff});
        out.push_back({p + ".linear2.bias", d});
        for (int i = 1; i <= n_norm; ++i) {
            out.push_back({p + ".norm" + std::to_string(i) + ".weight", d});
            out.push_back({p + ".norm" + std::to_string(i) + ".bias", d});
        }
    };
    for (int i = 0; i < c.enc_layers; ++i) {
        const std::string p = "transformer.encoder.layers." + std::to_string(i);
        attn(p + ".self_attn");
        ffn_norms(p, 2);
    }
    for (int i = 0; i < c.dec_layers; ++i) {
        const std::string p = "transformer.decoder.layers." + std::to_string(i);
        attn(p + ".self_attn");
        attn(p + ".multihead_attn");
        ffn_norms(p, 3);
    }
    out.push_back({"transformer.decoder.norm.weight", d});
    out.push_back({"transformer.decoder.norm.bias", d});
    out.push_back({"txt_position_embed.position_embeddings.weight", (size_t)c.max_q_l * d});
    out.push_back({"txt_position_embed.LayerNorm.weight", d});
    out.push_back({"txt_position_embed.LayerNorm.bias", d});
    const size_t span_out[3] = {d, d, 2};
    for (int i = 0; i < 3; ++i) {
        out.push_back({"span_embed.layers." + std::to_string(i) + ".weight", span_out[i] * d});
        out.push_back({"span_embed.layers." + std::to_string(i) + ".bias", span_out[i]});
    }
    out.push_back({"class_embed.weight", 2 * d});
    out.push_back({"class_embed.bias", 2});
    out.push_back({"query_embed.weight", (size_t)c.num_queries * d});
    const char* names[2] = {"input_txt_proj", "input_vid_proj"};
    const size_t din[2] = {dt, dm};
    for (int t = 0; t < 2; ++t) {
        for (int i = 0; i < 2; ++i) {
            const size_t k = i == 0 ? din[t] : d;
            const std::string p = std::string(names[t]) + "." + std::to_string(i);
            out.push_back({p + ".LayerNorm.weight", k});
            out.push_back({p + ".LayerNorm.bias", k});
            out.push_back({p + ".net.1.weight", d * k});
            out.push_back({p + ".net.1.bias", d});
        }
    }
    out.push_back({"saliency_proj.weight", d});
    out.push_back({"saliency_proj.bias", 1});
    out.push_back({"adapter_layer.layers.0.weight", d * dv});
    out.push_back({"adapter_layer.layers.0.bias", d});
    out.push_back({"adapter_layer.layers.1.weight", dv * d});
    out.push_back({"adapter_layer.layers.1.bias", dv});
}

static int check_dims(const cone_dims* c) {
    CONE_REQUIRE(c != nullptr, "dims is null");
    CONE_REQUIRE(c->hidden == 256 && c->nheads == 8, "only hidden_dim 256 with 8 heads (head_dim 32) is built");
    CONE_REQUIRE(c->v_dim > 0 && c->v_dim % 16 == 0 && c->t_dim > 0 && c->t_dim % 16 == 0,
                 "feature dims must be positive multiples of 16");
    CONE_REQUIRE(c->m_dim >= 0 && c->m_dim % 16 == 0, "motion feature dim must be 0 (= v_dim) or a positive multiple of 16");
    CONE_REQUIRE(c->ffn > 0 && c->ffn % 16 == 0, "dim_feedforward must be a multiple of 16");
    CONE_REQUIRE(c->enc_layers >= 1 && c->dec_layers >= 1 && c->enc_layers <= 8 && c->dec_layers <= 8, "1..8 layers");
    CONE_REQUIRE(c->num_queries >= 1 && c->num_queries <= 8, "1..8 moment slots");
    // windows of up to 256 rows run the short-window attention kernels, 257..512 rows their long-window variants
    CONE_REQUIRE(c->max_v_l >= 2 && c->max_q_l >= 1 && c->max_v_l + c->max_q_l <= CONE_MAX_WINDOW_ROWS,
                 "window (max_v_l + max_q_l = %d) must fit %d rows", c->max_v_l + c->max_q_l, CONE_MAX_WINDOW_ROWS);
    return CONE_OK;
}

extern "C" const char* cone_last_error(void) { return g_err; }
extern "C" int cone_version(void) { return 4; }
extern "C" int64_t cone_launch_count(void) { return g_launches; }
extern "C" void cone_launch_count_reset(void) { g_launches = 0; }

extern "C" size_t cone_weights_expected_floats(const cone_dims* dims) {
    if (check_dims(dims) != CONE_OK) return 0;
    std::vector<std::pair<std::string, size_t>> l;
    layout(*dims, l);
    size_t n = 0;
    for (auto& e : l) n += e.second;
    return n;
}

extern "C" void cone_weights_destroy(cone_weights* w) {
    if (!w) return;
    if (w->tc) tc_weights_destroy(w->tc);
    if (w->pos_proj) cudaFree(w->pos_proj);
    if (w->pos_kdec16) cudaFree(w->pos_kdec16);
    if (w->pos_qk16) cudaFree(w->pos_qk16);
    if (w->xattn) cudaFree(w->xattn);
    if (w->blob) cudaFree(w->blob);
    if (w->derived) cudaFree(w->derived);
    delete w;
}

// Host staging shared by create / update: the state dict padded per tensor to a multiple of 4 floats (float4 loads are
// always aligned) and the derived [K-proj rows; V-proj rows] cross-attention weights of all decoder layers.
static int stage_blob(cone_weights* w, const float* blob_host, size_t n_floats, std::vector<float>& staged,
                      std::vector<float>& der) {
    const cone_dims* dims = &w->dims;
    std::vector<std::pair<std::string, size_t>> l;
    layout(*dims, l);
    size_t n = 0;
    for (auto& e : l) n += e.second;
    if (n != n_floats) {
        set_error("state dict has %zu floats, expected %zu for these dims", n_floats, n);
        return CONE_ERR_INVALID;
    }
    staged.clear();
    staged.reserve(n + 4 * l.size());
    size_t src = 0;
    for (auto& e : l) {
        w->off[e.first] = staged.size();
        staged.insert(staged.end(), blob_host + src, blob_host + src + e.second);
        while (staged.size() & 3) staged.push_back(0.f);
        src += e.second;
    }
    const size_t d = dims->hidden;
    const int DL = dims->dec_layers;
    // derived: concatenated cross-attention K / V projections of all decoder layers (memory is shared)
    der.assign((size_t)DL * d * d * 2 + (size_t)DL * d * 2, 0.f);
    float* kw = der.data();  // layout kw | vw | kb | vb: [K-proj rows; V-proj rows] form one [2*DL*d, d] weight
    float* vw = kw + (size_t)DL * d * d;
    float* kb = vw + (size_t)DL * d * d;
    float* vb = kb + (size_t)DL * d;
    for (int i = 0; i < DL; ++i) {
        const std::string p = "transformer.decoder.layers." + std::to_string(i) + ".multihead_attn";
        const float* inw = staged.data() + w->off.at(p + ".in_proj_weight");
        const float* inb = staged.data() + w->off.at(p + ".in_proj_bias");
        memcpy(kw + (size_t)i * d * d, inw + d * d, sizeof(float) * d * d);
        memcpy(vw + (size_t)i * d * d, inw + 2 * d * d, sizeof(float) * d * d);
        memcpy(kb + (size_t)i * d, inb + d, sizeof(float) * d);
        memcpy(vb + (size_t)i * d, inb + 2 * d, sizeof(float) * d);
    }
    return CONE_OK;
}

// Folded cross-attention weights (see cone_weights::xattn), computed in fp64 on the host from the staged state dict.
static size_t xattn_floats_per_layer(size_t d) { return 9 * d * d + 9 * d + 8 * d * d + d; }
static void build_xattn(const cone_weights* w, const std::vector<float>& staged, std::vector<float>& out) {
    const size_t d = w->dims.hidden, H = w->dims.nheads, hd = d / H;
    const int DL = w->dims.dec_layers;
    const double c = (1.0 / sqrt((double)hd)) * 1.4426950408889634;
    out.assign(xattn_floats_per_layer(d) * DL, 0.f);
    std::vector<double> acc(d);
    for (int l = 0; l < DL; ++l) {
        const std::string p = "transformer.decoder.layers." + std::to_string(l) + ".multihead_attn";
        const float* inw = staged.data() + w->off.at(p + ".in_proj_weight");
        const float* inb = staged.data() + w->off.at(p + ".in_proj_bias");
        const float* ow = staged.data() + w->off.at(p + ".out_proj.weight");
        const float* ob = staged.data() + w->off.at(p + ".out_proj.bias");
        const float *Wq = inw, *Wk = inw + d * d, *Wv = inw + 2 * d * d;
        const float *bq = inb, *bv = inb + 2 * d;
        float* xq_w = out.data() + xattn_floats_per_layer(d) * l;
        float* xq_b = xq_w + 9 * d * d;
        float* xo_w = xq_b + 9 * d;
        float* xo_b = xo_w + 8 * d * d;
        for (size_t i = 0; i < d * d; ++i) xq_w[i] = (float)(c * Wq[i]);
        for (size_t i = 0; i < d; ++i) xq_b[i] = (float)(c * bq[i]);
        for (size_t h = 0; h < H; ++h) {
            for (size_t j = 0; j < d; ++j) {  // row d + h d + j = c * sum_e Wk[h hd + e, j] * Wq[h hd + e, :]
                std::fill(acc.begin(), acc.end(), 0.0);
                double bacc = 0.0;
                for (size_t e = 0; e < hd; ++e) {
                    const double wk = Wk[(h * hd + e) * d + j];
                    const float* wq = Wq + (h * hd + e) * d;
                    for (size_t i = 0; i < d; ++i) acc[i] += wk * wq[i];
                    bacc += wk * bq[h * hd + e];
                }
                float* row = xq_w + (d + h * d + j) * d;
                for (size_t i = 0; i < d; ++i) row[i] = (float)(c * acc[i]);
                xq_b[d + h * d + j] = (float)(c * bacc);
            }
            for (size_t o = 0; o < d; ++o) {  // xo_w[o, h d + j] = sum_e Wo[o, h hd + e] * Wv[h hd + e, j]
                std::fill(acc.begin(), acc.end(), 0.0);
                for (size_t e = 0; e < hd; ++e) {
                    const double wo = ow[o * d + h * hd + e];
                    const float* wv = Wv + (h * hd + e) * d;
                    for (size_t j = 0; j < d; ++j) acc[j] += wo * wv[j];
                }
                float* row = xo_w + o * 8 * d + h * d;
                for (size_t j = 0; j < d; ++j) row[j] = (float)acc[j];
            }
        }
        for (size_t o = 0; o < d; ++o) {
            double a = ob[o];
            for (size_t e = 0; e < d; ++e) a += (double)ow[o * d + e] * bv[e];
            xo_b[o] = (float)a;
        }
    }
}
static int upload_xattn(cone_weights* w, const std::vector<float>& staged, cudaStream_t s) {
    std::vector<float> x;
    build_xattn(w, staged, x);
    const size_t d = w->dims.hidden;
    if (w->xattn == nullptr) CONE_CUDA(cudaMalloc(&w->xattn, sizeof(float) * x.size()));
    CONE_CUDA(cudaMemcpyAsync(w->xattn, x.data(), sizeof(float) * x.size(), cudaMemcpyHostToDevice, s));
    CONE_CUDA(cudaStreamSynchronize(s));  // the staging vector dies at return
    w->xq_w.clear(); w->xq_b.clear(); w->xo_w.clear(); w->xo_b.clear();
    for (int l = 0; l < w->dims.dec_layers; ++l) {
        float* base = w->xattn + xattn_floats_per_layer(d) * l;
        w->xq_w.push_back(base);
        w->xq_b.push_back(base + 9 * d * d);
        w->xo_w.push_back(base + 9 * d * d + 9 * d);
        w->xo_b.push_back(base + 9 * d * d + 9 * d + 8 * d * d);
    }
    return CONE_OK;
}

extern "C" int cone_weights_create(const float* blob_host, size_t n_floats, const cone_dims* dims, void* stream,
                                   cone_weights** out) {
    CONE_TRY(check_dims(dims));
    CONE_REQUIRE(blob_host != nullptr && out != nullptr, "null argument");
    cudaStream_t s = (cudaStream_t)stream;
    cone_weights* w = new cone_weights();
    w->dims = *dims;
    std::vector<float> staged, der;
    int r = stage_blob(w, blob_host, n_floats, staged, der);
    if (r != CONE_OK) {
        delete w;
        return r;
    }
    w->n_floats = staged.size();
    const size_t d = dims->hidden;
    const int DL = dims->dec_layers;
    const size_t pos_floats = (size_t)(dims->max_v_l + 1) * dims->max_v_l * d;
    cudaError_t e = cudaMalloc(&w->blob, sizeof(float) * w->n_floats);
    if (e == cudaSuccess) e = cudaMalloc(&w->derived, sizeof(float) * (der.size() + pos_floats));
    if (e == cudaSuccess) e = cudaMemcpyAsync(w->blob, staged.data(), sizeof(float) * w->n_floats, cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = cudaMemcpyAsync(w->derived, der.data(), sizeof(float) * der.size(), cudaMemcpyHostToDevice, s);
    if (e == cudaSuccess) e = cudaStreamSynchronize(s);  // staging vectors die at return
    if (e != cudaSuccess) {
        set_error("cone_weights_create: %s", cudaGetErrorString(e));
        cone_weights_destroy(w);
        return CONE_ERR_CUDA;
    }
    w->dec_kw = w->derived;
    w->dec_vw = w->dec_kw + (size_t)DL * d * d;
    w->dec_kb = w->dec_vw + (size_t)DL * d * d;
    w->dec_vb = w->dec_kb + (size_t)DL * d;
    w->pos_table = w->derived + der.size();
    r = build_pos_table(w->pos_table, dims->max_v_l, (int)d, s);
    if (r == CONE_OK) r = upload_xattn(w, staged, s);
    if (r != CONE_OK) {
        cone_weights_destroy(w);
        return r;
    }
    *out = w;
    return CONE_OK;
}

// Forward declaration: defined with the tensor-core helpers below.
namespace { int fill_pos_proj(cone_weights* mw, cudaStream_t s); }

// Live weights (SURVEY.md §8(f)4: cone/train.py:164-168 evaluates every few epochs on the weights being trained): the
// new state dict is written INTO the existing device buffers and every derived tensor (decoder K|V concatenation, fp16
// copies, position-projection tables) is recomputed in place, so the handle, all device pointers, TMA descriptors and
// captured CUDA graphs stay valid.  Ordered on `stream` after the work already queued there.
extern "C" int cone_weights_update(cone_weights* w, const float* blob_host, size_t n_floats, void* stream) {
    CONE_REQUIRE(w != nullptr && blob_host != nullptr, "null argument");
    cudaStream_t s = (cudaStream_t)stream;
    std::vector<float> staged, der;
    CONE_TRY(stage_blob(w, blob_host, n_floats, staged, der));
    CONE_REQUIRE(staged.size() == w->n_floats, "cone_weights_update: layout changed");
    CONE_CUDA(cudaMemcpyAsync(w->blob, staged.data(), sizeof(float) * w->n_floats, cudaMemcpyHostToDevice, s));
    CONE_CUDA(cudaMemcpyAsync(w->derived, der.data(), sizeof(float) * der.size(), cudaMemcpyHostToDevice, s));
    CONE_CUDA(cudaStreamSynchronize(s));  // staging vectors die at return
    CONE_TRY(upload_xattn(w, staged, s));
    CONE_TRY(tc_weights_refresh(w->tc, s));
    if (w->pos_proj) CONE_TRY(fill_pos_proj(w, s));
    return CONE_OK;
}

// ------------------------------------------------------------------------------------------------
// workspace arena
// ------------------------------------------------------------------------------------------------
namespace {

struct Arena {
    char* base;
    size_t cap;
    size_t used = 0;
    Arena(void* b, size_t c) : base((char*)b), cap(c) {}
    template <class T>
    T* get(size_t n) {
        const size_t bytes = (n * sizeof(T) + 255) & ~(size_t)255;
        T* p = base ? (T*)(base + used) : nullptr;
        used += bytes;
        return p;
    }
    bool fits() const { return base == nullptr || used <= cap; }
};

struct Linear {
    const float* W;
    const float* b;
    int N, K;
    const char* name;  // state-dict key of W (tensor-core weight cache lookup)
};

struct Ctx {
    const cone_weights* w;
    int prec;
    cudaStream_t s;
    uint16_t* split_scratch = nullptr;  // [M, 3 K] fp16 operand staging of the 3-product GEMM (CONE_PREC_TC_SPLIT)
};

// y = epi(x W^T + b (+R)) with fp32-class accuracy on the fp16 tensor pipe: x and W are split into fp16 hi + lo parts and
// the three significant products are accumulated in fp32 by one GEMM over 3 K columns (tc_gemm.cu, split3).
// Used in tensor-core mode for the projections whose accuracy must not enter the fp16 error budget (input projections,
// span head); the window-ranking GEMMs stay on the fp32 pipe so that rank-lists do not depend on the precision mode.
int split_linear(const Ctx& c, const float* x, int64_t ldx, int64_t M, const float* W, const float* b, int N, int K,
                 float* y, int64_t ldy, int relu, const float* R, int64_t ldr, uint16_t* scratch16) {
    CONE_TRY(split3_f16_rows(x, ldx, scratch16, M, K, c.s));
    TcGemmArgs g;
    g.A16 = scratch16; g.lda = 3 * (int64_t)K; g.M = M; g.W = W; g.bias = b; g.N = N; g.K = K; g.split3 = 1;
    g.C32 = y; g.ldc32 = ldy; g.relu = relu; g.R32 = R; g.ldr32 = ldr;
    return tc_gemm_run(c.w->tc, g, c.s);
}

// y[M,N] = epi(x[M,K] * W^T + b (+R)) in the requested precision
int linear(const Ctx& c, const float* x, int64_t ldx, int64_t M, const float* W, const float* b, int N, int K, float* y,
           int64_t ldy, int relu, const float* R = nullptr, int64_t ldr = 0) {
    if (c.prec == CONE_PREC_TC && tc_gemm_supported(M, N, K)) {
        return tc_gemm(c.w->tc, x, ldx, M, W, b, N, K, y, ldy, relu, R, ldr, c.s);
    }
    if (c.prec == CONE_PREC_TC_SPLIT) {
        CONE_REQUIRE(tc_gemm_supported(M, N, 3 * K) && (K & 3) == 0, "split GEMM: unsupported shape M=%lld N=%d K=%d", (long long)M, N, K);
        CONE_REQUIRE(c.split_scratch != nullptr, "split GEMM: no operand scratch");
        return split_linear(c, x, ldx, M, W, b, N, K, y, ldy, relu, R, ldr, c.split_scratch);
    }
    GemmParams g;
    g.A = x; g.lda = ldx; g.W = W; g.ldw = K; g.C = y; g.ldc = ldy; g.bias = b; g.R = R; g.ldr = ldr;
    g.M = M; g.N = N; g.K = K; g.relu = relu;
    return sgemm_nt(g, c.s);
}

int linear_named(const Ctx& c, const float* x, int64_t ldx, int64_t M, const std::string& prefix, int N, int K, float* y,
                 int64_t ldy, int relu, const float* R = nullptr, int64_t ldr = 0) {
    return linear(c, x, ldx, M, c.w->p(prefix + ".weight"), c.w->p(prefix + ".bias"), N, K, y, ldy, relu, R, ldr);
}

// LinearLayer x2 (cone/model.py:443-465, 55-72): LN -> Linear -> ReLU -> LN -> Linear
struct ProjBuffers {
    float *ln_in, *h1, *ln_h1;
    uint16_t* a3;  // split fp16 operand staging (tensor-core mode)
};
ProjBuffers plan_proj(Arena& a, int64_t rows, int din, int d) {
    ProjBuffers b;
    b.ln_in = a.get<float>(rows * din);
    b.h1 = a.get<float>(rows * d);
    b.ln_h1 = a.get<float>(rows * d);
    b.a3 = a.get<uint16_t>(rows * 3 * (din > d ? din : d));
    return b;
}
// x: raw rows of storage type x_dtype (CONE_DTYPE_*), read only by the first LayerNorm
int input_proj(const Ctx& cin, const char* name, const void* x, int x_dtype, int64_t rows, int din, float* out,
               ProjBuffers& b) {
    // per-frame / per-query work, a few GFLOP per movie: kept in fp32 in every mode (error budget, DESIGN.md)
    // (measured: plain fp16-operand tensor-core GEMMs here save 0.9 ms per step but raise the end-to-end error by 13-20 %
    // rms and push 0.27 % of the values past 1e-3: profiles/r01_notes.md — hence the split GEMM in tensor-core mode)
    const bool split = cin.prec == CONE_PREC_TC && (din % 64) == 0 && cin.w->tc != nullptr;
    const Ctx c{cin.w, split ? CONE_PREC_TC_SPLIT : CONE_PREC_FP32, cin.s, b.a3};
    const int d = c.w->dims.hidden;
    const std::string p0 = std::string(name) + ".0", p1 = std::string(name) + ".1";
    CONE_TRY(layernorm_rows(x, x_dtype, nullptr, c.w->p(p0 + ".LayerNorm.weight"), c.w->p(p0 + ".LayerNorm.bias"), b.ln_in,
                            rows, din, 1e-5f, c.s));
    CONE_TRY(linear_named(c, b.ln_in, din, rows, p0 + ".net.1", d, din, b.h1, d, 1));
    CONE_TRY(layernorm_rows(b.h1, nullptr, c.w->p(p1 + ".LayerNorm.weight"), c.w->p(p1 + ".LayerNorm.bias"), b.ln_h1,
                            rows, d, 1e-5f, c.s));
    CONE_TRY(linear_named(c, b.ln_h1, d, rows, p1 + ".net.1", d, d, out, d, 0));
    return CONE_OK;
}
int input_proj(const Ctx& c, const char* name, const float* x, int64_t rows, int din, float* out, ProjBuffers& b) {
    return input_proj(c, name, x, CONE_DTYPE_F32, rows, din, out, b);
}

// adapter_layer(x) (+ x): MLP(Dv, 256, Dv, 2) (cone/model.py:80, 428-440)
int adapter_rows(const Ctx& c, const float* x, int64_t rows, float* hid, float* out, int residual) {
    const int d = c.w->dims.hidden, dv = c.w->dims.v_dim;
    CONE_TRY(linear_named(c, x, dv, rows, "adapter_layer.layers.0", d, dv, hid, d, 1));
    CONE_TRY(linear_named(c, hid, d, rows, "adapter_layer.layers.1", dv, d, out, dv, 0, residual ? x : nullptr, dv));
    return CONE_OK;
}

// ---- the Moment-DETR core over B windows of S = Lv + Lt rows -------------------------------------
struct CoreBuffers {
    int64_t B;
    int Lv, Lt, hw;
    float *src, *srcpos, *qk, *v, *att, *tmp, *h;                      // [R, .] fp32 (srcpos..h: fp32 mode only)
    uint16_t *src16, *qkv16, *att16, *h16;                             // [R, .] fp16 (tensor-core mode only)
    uint16_t* src16lo = nullptr;                                       // [R, d] fp16 low part of the residual stream
    float *tgt, *t2, *dqkin, *dqk, *dv, *datt, *dq, *dh, *hs, *hid1, *hid2;  // [B*nq, .]
    uint16_t *dqt16, *dpm16, *dh16;                                          // [B*nq, .] fp16 (tensor-core mode only)
    uint16_t* hs3 = nullptr;                                                 // [B*nq, 3 d] split operand of the span head
    uint16_t* dsplit16 = nullptr;                                            // [B*nq, 3 ffn] split operand staging of the decoder
    int64_t *vid_base, *txt_base;
    int32_t *vlen, *tlen, *pad_len, *qidx;
    // tensor-core mode, optional: q|k|v of encoder layer 0 per FRAME and per TOKEN (the projection of a row does not
    // depend on the window it is sliced into); when set, layer 0 runs no per-window QKV GEMM
    const uint16_t* frame_qkv = nullptr;
    const uint16_t* token_qkv = nullptr;
    int64_t n_frames = 0, n_tokens = 0;
    // ... and the hi / lo fp16 tables [n_frames + n_tokens, d] of the projected frame and token rows: when set, the fused tail
    // of layer 0 fetches its residual rows from them by TMA gather4 and no per-window copy of the inputs is made
    const uint16_t* g_src_hi = nullptr;
    const uint16_t* g_src_lo = nullptr;
};

// The fused encoder tail (enc_tail.cu) replaces out_proj + norm1 + linear1 + linear2 + norm2 of the tensor-core mode;
// CONE_FUSED_TAIL=0 in the environment selects the unfused three-GEMM chain (A/B measurements, fall-back).
// CONE_TAIL_GATHER=0: materialise the window rows with the gather kernel instead (A/B measurements, fall-back)
bool tail_gather_enabled() {
    static int env = -1;
    if (env < 0) {
        const char* e = getenv("CONE_TAIL_GATHER");
        env = (e && e[0] == '0') ? 0 : 1;
    }
    return env == 1;
}

bool fused_tail_enabled(const cone_dims& c) {
    static int env = -1;
    if (env < 0) {
        const char* e = getenv("CONE_FUSED_TAIL");
        env = (e && e[0] == '0') ? 0 : 1;
    }
    return env == 1 && enc_tail_supported(c.hidden, c.ffn);
}

CoreBuffers plan_core(Arena& a, const cone_dims& c, int64_t B, int Lv, int Lt, int prec) {
    CoreBuffers b{};
    b.B = B; b.Lv = Lv; b.Lt = Lt;
    const int64_t R = B * (Lv + Lt), Q = B * c.num_queries;
    const int d = c.hidden;
    b.hw = c.ffn > 2 * d * c.dec_layers ? c.ffn : 2 * d * c.dec_layers;
    b.src = a.get<float>(R * d);
    if (prec == CONE_PREC_TC) {
        b.src16 = a.get<uint16_t>(R * d);
        b.src16lo = a.get<uint16_t>(R * d);
        b.qkv16 = a.get<uint16_t>(R * 3 * d);
        b.att16 = a.get<uint16_t>(R * d);
        // the [R, ffn] hidden activations only exist in the unfused chain (enc_tail.cu keeps them on chip)
        b.h16 = fused_tail_enabled(c) ? nullptr : a.get<uint16_t>(R * b.hw);
    } else {
        b.srcpos = a.get<float>(R * d);
        b.qk = a.get<float>(R * 2 * d);
        b.v = a.get<float>(R * d);
        b.att = a.get<float>(R * d);
        b.tmp = a.get<float>(R * d);
        b.h = a.get<float>(R * b.hw);
    }
    b.tgt = a.get<float>(Q * d);
    b.dqkin = a.get<float>(Q * d);
    b.dqk = a.get<float>(Q * 2 * d);
    b.dv = a.get<float>(Q * d);
    b.datt = a.get<float>(Q * d);
    if (prec == CONE_PREC_TC) {  // the decoder chain is fp32 between kernels; its GEMMs are 3-product split GEMMs
        b.dqt16 = a.get<uint16_t>(Q * 9 * d);  // q | q pushed through Wk_h^T per head
        b.dpm16 = a.get<uint16_t>(Q * 8 * d);  // attention-pooled memory per head
        b.dh16 = a.get<uint16_t>(Q * c.ffn);   // FFN hidden
        b.hs3 = a.get<uint16_t>(Q * 3 * d);
        b.dsplit16 = a.get<uint16_t>(Q * 3 * d);
    } else {
        b.dh = a.get<float>(Q * c.ffn);
        b.t2 = a.get<float>(Q * d);
        b.dq = a.get<float>(Q * d);
    }
    b.hs = a.get<float>(Q * d);
    b.hid1 = a.get<float>(Q * d);
    b.hid2 = a.get<float>(Q * d);
    b.vid_base = a.get<int64_t>(B);
    b.txt_base = a.get<int64_t>(B);
    b.vlen = a.get<int32_t>(B);
    b.tlen = a.get<int32_t>(B);
    b.pad_len = a.get<int32_t>(B);
    b.qidx = a.get<int32_t>(B);
    return b;
}

// heads on hs [Q, d]: class logits / foreground probability and sigmoid spans (cone/model.py:112-115,
// cone/inference.py:47,52)
int heads(const Ctx& cin, CoreBuffers& b, const float* hs, int64_t Q, float* logits, float* prob_fg, float* spans) {
    // 5 rows per window: fp32 accuracy in every mode (split GEMM on the tensor pipe in tensor-core mode)
    const bool split = cin.prec == CONE_PREC_TC && b.hs3 != nullptr && cin.w->tc != nullptr;
    const Ctx c{cin.w, split ? CONE_PREC_TC_SPLIT : CONE_PREC_FP32, cin.s, b.hs3};
    const int d = c.w->dims.hidden;
    if (logits) CONE_TRY(rowdot_small(hs, d, c.w->p("class_embed.weight"), c.w->p("class_embed.bias"), logits, Q, 2, d, 0, c.s));
    if (prob_fg) CONE_TRY(rowdot_small(hs, d, c.w->p("class_embed.weight"), c.w->p("class_embed.bias"), prob_fg, Q, 2, d, 2, c.s));
    if (spans) {
        CONE_TRY(linear_named(c, hs, d, Q, "span_embed.layers.0", d, d, b.hid1, d, 1));
        CONE_TRY(linear_named(c, b.hid1, d, Q, "span_embed.layers.1", d, d, b.hid2, d, 1));
        CONE_TRY(rowdot_small(b.hid2, d, c.w->p("span_embed.layers.2.weight"), c.w->p("span_embed.layers.2.bias"), spans, Q,
                              2, d, 1, c.s));
    }
    return CONE_OK;
}

// b.src must hold the projected window rows; vlen / tlen the valid lengths.
int transformer_core(const Ctx& c, CoreBuffers& b, float* logits, float* prob_fg, float* spans, float* saliency,
                     float* aux_logits, float* aux_spans) {
    const cone_dims& dm = c.w->dims;
    const int d = dm.hidden, ff = dm.ffn, nq = dm.num_queries, H = dm.nheads;
    const int S = b.Lv + b.Lt;
    const int64_t R = b.B * S, Q = b.B * nq;
    const int DL = dm.dec_layers;
    const bool tc = (c.prec == CONE_PREC_TC);
    if (!tc) {
        // encoder (cone/transformer.py:233-246), fp32
        for (int l = 0; l < dm.enc_layers; ++l) {
            const std::string p = "transformer.encoder.layers." + std::to_string(l);
            const float* inw = c.w->p(p + ".self_attn.in_proj_weight");
            const float* inb = c.w->p(p + ".self_attn.in_proj_bias");
            CONE_TRY(add_pos_rows(b.src, c.w->pos_table, b.vlen, b.srcpos, b.B, b.Lv, b.Lt, d, dm.max_v_l, c.s));
            CONE_TRY(linear(c, b.srcpos, d, R, inw, inb, 2 * d, d, b.qk, 2 * d, 0));                 // q | k
            CONE_TRY(linear(c, b.src, d, R, inw + (size_t)2 * d * d, inb + 2 * d, d, d, b.v, d, 0));  // v
            CONE_TRY(enc_self_attention(b.qk, 2 * d, b.v, d, b.att, d, b.vlen, b.tlen, b.B, b.Lv, b.Lt, H, c.s));
            CONE_TRY(linear_named(c, b.att, d, R, p + ".self_attn.out_proj", d, d, b.tmp, d, 0, b.src, d));
            CONE_TRY(layernorm_rows(b.tmp, nullptr, c.w->p(p + ".norm1.weight"), c.w->p(p + ".norm1.bias"), b.src, R, d, 1e-5f, c.s));
            CONE_TRY(linear_named(c, b.src, d, R, p + ".linear1", ff, d, b.h, b.hw, 1));
            CONE_TRY(linear_named(c, b.h, b.hw, R, p + ".linear2", d, ff, b.tmp, d, 0, b.src, d));
            CONE_TRY(layernorm_rows(b.tmp, nullptr, c.w->p(p + ".norm2.weight"), c.w->p(p + ".norm2.bias"), b.src, R, d, 1e-5f, c.s));
        }
    } else {
        // encoder on the tensor cores.  Everything between two GEMMs is fp16 and is produced by the previous
        // kernel's epilogue: b.src16 was filled by the fp16 gather; the residual stream is the fp16 LayerNorm
        // output (no accuracy cost, DESIGN.md); LayerNorm is fused into the out_proj / linear2 epilogues (N = 256
        // = one accumulator row per thread); q, k and v come from ONE GEMM over the packed in_proj (N = 768)
        // because the position term of q and k is added inside the attention kernel from a per-layer table.
        TcWeights* t = c.w->tc;
        auto G = [&](const uint16_t* A, int64_t lda, const float* W, const float* bias, int N, int K) {
            TcGemmArgs g;
            g.A16 = A; g.lda = lda; g.M = R; g.W = W; g.bias = bias; g.N = N; g.K = K;
            return g;
        };
        for (int l = 0; l < dm.enc_layers; ++l) {
            const std::string p = "transformer.encoder.layers." + std::to_string(l);
            TcGemmArgs g;
            // attention on tcgen05 (enc_attn_tc.cu) where the window fits its TMEM / shared-memory plan, else mma.sync
            const bool attn_tc = enc_attn_tc_supported(b.Lv, b.Lt, d, H);
            const size_t pos_rows = (size_t)(dm.max_v_l + 1) * dm.max_v_l;
            const uint16_t* pos16 = c.w->pos_qk16 + (size_t)l * pos_rows * 2 * d;
            if (l == 0 && b.frame_qkv != nullptr) {
                if (attn_tc) {
                    CONE_TRY(enc_attn_tc_run(b.frame_qkv, b.n_frames, b.att16, d, b.vlen, b.tlen, b.B, b.Lv, b.Lt, pos16, dm.max_v_l,
                                             b.token_qkv, b.n_tokens, b.vid_base, b.txt_base, tc_num_sms(t), c.s));
                } else {
                    CONE_TRY(enc_self_attention_f16(nullptr, 3 * d, nullptr, 3 * d, b.att16, d, b.vlen, b.tlen, b.B, b.Lv, b.Lt, H,
                                                    pos16, dm.max_v_l, c.s, b.frame_qkv, b.token_qkv, b.vid_base,
                                                    b.txt_base, b.n_frames));
                }
            } else {
                g = G(b.src16, d, c.w->p(p + ".self_attn.in_proj_weight"), c.w->p(p + ".self_attn.in_proj_bias"), 3 * d, d);
                g.C16 = b.qkv16; g.ldc16 = 3 * d;
                CONE_TRY(tc_gemm_run(t, g, c.s));
                if (attn_tc) {
                    CONE_TRY(enc_attn_tc_run(b.qkv16, R, b.att16, d, b.vlen, b.tlen, b.B, b.Lv, b.Lt, pos16, dm.max_v_l, nullptr, 0,
                                             nullptr, nullptr, tc_num_sms(t), c.s));
                } else {
                    CONE_TRY(enc_self_attention_f16(b.qkv16, 3 * d, b.qkv16 + 2 * d, 3 * d, b.att16, d, b.vlen, b.tlen, b.B,
                                                    b.Lv, b.Lt, H, pos16, dm.max_v_l, c.s));
                }
            }
            const bool last_enc = (l == dm.enc_layers - 1);
            if (fused_tail_enabled(dm)) {
                // out_proj + norm1 + linear1 + relu + linear2 + norm2 in ONE kernel (enc_tail.cu): the residual stream is
                // fp32-accurate (hi + lo fp16 across HBM, fp32 inside the kernel), the [R, ffn] hidden stays on chip
                EncTailArgs e;
                e.att16 = b.att16; e.lda = d;
                e.res_hi = b.src16; e.res_lo = b.src16lo; e.ldr = d;
                if (l == 0 && b.g_src_hi != nullptr) {  // window slicing fused into the tail: residual rows by TMA gather4
                    e.res_hi = b.g_src_hi; e.res_lo = b.g_src_lo;
                    e.g_vid_base = b.vid_base; e.g_txt_base = b.txt_base;
                    e.g_S = b.Lv + b.Lt; e.g_Lv = b.Lv;
                    e.g_nvid = b.n_frames; e.g_nsrc = b.n_frames + b.n_tokens;
                }
                e.out_hi = b.src16; e.out_lo = last_enc ? nullptr : b.src16lo; e.ldo = d;  // the memory is read as fp16
                if (saliency && last_enc) { e.C32 = b.src; e.ldc32 = d; }
                e.M = R; e.d = d; e.ffn = ff;
                e.Wo = c.w->p(p + ".self_attn.out_proj.weight"); e.bo = c.w->p(p + ".self_attn.out_proj.bias");
                e.ln1_g = c.w->p(p + ".norm1.weight"); e.ln1_b = c.w->p(p + ".norm1.bias");
                e.W1 = c.w->p(p + ".linear1.weight"); e.b1 = c.w->p(p + ".linear1.bias");
                e.W2 = c.w->p(p + ".linear2.weight"); e.b2 = c.w->p(p + ".linear2.bias");
                e.ln2_g = c.w->p(p + ".norm2.weight"); e.ln2_b = c.w->p(p + ".norm2.bias");
                CONE_TRY(enc_tail_run(t, e, c.s));
                continue;
            }
            g = G(b.att16, d, c.w->p(p + ".self_attn.out_proj.weight"), c.w->p(p + ".self_attn.out_proj.bias"), d, d);
            g.R16 = b.src16; g.ldr16 = d;
            g.ln_g = c.w->p(p + ".norm1.weight"); g.ln_b = c.w->p(p + ".norm1.bias");
            g.C16 = b.src16; g.ldc16 = d;
            CONE_TRY(tc_gemm_run(t, g, c.s));
            g = G(b.src16, d, c.w->p(p + ".linear1.weight"), c.w->p(p + ".linear1.bias"), ff, d);
            g.relu = 1; g.C16 = b.h16; g.ldc16 = b.hw;
            CONE_TRY(tc_gemm_run(t, g, c.s));
            g = G(b.h16, b.hw, c.w->p(p + ".linear2.weight"), c.w->p(p + ".linear2.bias"), d, ff);
            g.R16 = b.src16; g.ldr16 = d;
            g.ln_g = c.w->p(p + ".norm2.weight"); g.ln_b = c.w->p(p + ".norm2.bias");
            g.C16 = b.src16; g.ldc16 = d;
            if (saliency && last_enc) { g.C32 = b.src; g.ldc32 = d; }  // fp32 memory for saliency_proj
            CONE_TRY(tc_gemm_run(t, g, c.s));
        }
    }
    if (saliency) {  // saliency_proj(vid_mem) (cone/model.py:119-122), video rows only
        CONE_TRY(rowdot_small(b.src, d, c.w->p("saliency_proj.weight"), c.w->p("saliency_proj.bias"), saliency, b.B * b.Lv,
                              1, d, 0, c.s, b.Lv, S));
    }
    // decoder (cone/transformer.py:296-317, 117-146): the memory K and V projections of ALL layers in one GEMM
    // (weights concatenated at load time: columns [0, DL*d) = K of layer 0.., [DL*d, 2*DL*d) = V of layer 0..)
    float* kdec = b.h;
    float* vdec = b.h ? b.h + (size_t)DL * d : nullptr;
    if (!tc) {
        CONE_TRY(add_pos_rows(b.src, c.w->pos_table, b.vlen, b.srcpos, b.B, b.Lv, b.Lt, d, dm.max_v_l, c.s));
        CONE_TRY(linear(c, b.srcpos, d, R, c.w->dec_kw, c.w->dec_kb, DL * d, d, kdec, b.hw, 0));
        CONE_TRY(linear(c, b.src, d, R, c.w->dec_vw, c.w->dec_vb, DL * d, d, vdec, b.hw, 0));
    }
    // tensor-core mode: no K / V projection of the memory at all — the cross-attention works on the raw encoder output
    // (dec_cross_attention_mem, attention.cu)
    // The decoder starts from tgt = 0 (transformer.py:61), so everything up to the first cross-attention — self-attention
    // block, norm1, and the cross-attention queries — is the same for every window: in tensor-core mode it is computed
    // for ONE window (nq rows) and broadcast (identical bits: every row of these kernels is computed independently).
    CONE_CUDA(cudaMemsetAsync(b.tgt, 0, sizeof(float) * (tc ? nq : Q) * d, c.s));
    const float* qpos = c.w->p("query_embed.weight");
    for (int l = 0; l < DL; ++l) {
        const std::string p = "transformer.decoder.layers." + std::to_string(l);
        const float* inw = c.w->p(p + ".self_attn.in_proj_weight");
        const float* inb = c.w->p(p + ".self_attn.in_proj_bias");
        const float* cw = c.w->p(p + ".multihead_attn.in_proj_weight");
        const float* cb = c.w->p(p + ".multihead_attn.in_proj_bias");
        if (!tc) {
            CONE_TRY(add_row_table(b.tgt, qpos, b.dqkin, Q, nq, d, c.s));
            CONE_TRY(linear(c, b.dqkin, d, Q, inw, inb, 2 * d, d, b.dqk, 2 * d, 0));
            CONE_TRY(linear(c, b.tgt, d, Q, inw + (size_t)2 * d * d, inb + 2 * d, d, d, b.dv, d, 0));
            CONE_TRY(dec_self_attention(b.dqk, 2 * d, b.dv, d, b.datt, d, b.B, nq, H, 0, c.s));
            CONE_TRY(linear_named(c, b.datt, d, Q, p + ".self_attn.out_proj", d, d, b.t2, d, 0, b.tgt, d));
            CONE_TRY(layernorm_rows(b.t2, nullptr, c.w->p(p + ".norm1.weight"), c.w->p(p + ".norm1.bias"), b.tgt, Q, d, 1e-5f, c.s));
            CONE_TRY(add_row_table(b.tgt, qpos, b.dqkin, Q, nq, d, c.s));
            CONE_TRY(linear(c, b.dqkin, d, Q, cw, cb, d, d, b.dq, d, 0));
            CONE_TRY(dec_cross_attention(b.dq, d, kdec + (size_t)l * d, b.hw, vdec + (size_t)l * d, b.hw, b.datt, d, b.vlen,
                                         b.tlen, b.B, nq, b.Lv, b.Lt, H, 0, nullptr, 0, 0, c.s));
            CONE_TRY(linear_named(c, b.datt, d, Q, p + ".multihead_attn.out_proj", d, d, b.t2, d, 0, b.tgt, d));
            CONE_TRY(layernorm_rows(b.t2, nullptr, c.w->p(p + ".norm2.weight"), c.w->p(p + ".norm2.bias"), b.tgt, Q, d, 1e-5f, c.s));
            CONE_TRY(linear_named(c, b.tgt, d, Q, p + ".linear1", ff, d, b.dh, ff, 1));
            CONE_TRY(linear_named(c, b.dh, ff, Q, p + ".linear2", d, ff, b.t2, d, 0, b.tgt, d));
            CONE_TRY(layernorm_rows(b.t2, nullptr, c.w->p(p + ".norm3.weight"), c.w->p(p + ".norm3.bias"), b.tgt, Q, d, 1e-5f, c.s));
        } else {
            // Tensor-core decoder chain.  5 rows per window against 150 in the encoder: the decoder is cheap, and its
            // roundings reach the span / class heads without being averaged over keys, so it keeps fp32-class accuracy:
            // fp32 activations between kernels, every GEMM a 3-product split-fp16 GEMM on tcgen05 (operands AND weights
            // as fp16 hi + lo, tc_gemm.cu), LayerNorm + fp32 residual in the epilogues.  Only the cross-attention kernel
            // itself works on fp16 (queries pushed through Wk^T, raw encoder memory, pooled memory).  Measured by
            // emulation (profiles/tc_emulate.py): with fp16 decoder operands the end-to-end error of spans / probabilities
            // is 1.8e-4 rms with a tail past 1e-3; with this chain 1.3e-4 rms and max 7-8e-4.
            TcWeights* t = c.w->tc;
            const bool shared = (l == 0);           // window-independent prefix of layer 0: one window's rows
            const int64_t Qs = shared ? nq : Q;
            // y = epi(x W^T + b): x fp32 [M, K] -> [hi | hi | lo] staging -> split GEMM; the caller fills the epilogue
            auto SG = [&](const float* x, int64_t ldx, int64_t M, const float* W, const float* bias, int N, int K,
                          TcGemmArgs& g) -> int {
                CONE_TRY(split3_f16_rows(x, ldx, b.dsplit16, M, K, c.s));
                g = TcGemmArgs();
                g.A16 = b.dsplit16; g.lda = 3 * (int64_t)K; g.M = M; g.W = W; g.bias = bias; g.N = N; g.K = K; g.split3 = 1;
                return CONE_OK;
            };
            auto LN = [&](TcGemmArgs& g, const std::string& norm) {  // + fp32 residual, LayerNorm, fp32 stream out
                g.R32 = b.tgt; g.ldr32 = d;
                g.ln_g = c.w->p(norm + ".weight"); g.ln_b = c.w->p(norm + ".bias");
                g.C32 = b.tgt; g.ldc32 = d;
            };
            TcGemmArgs g;
            CONE_TRY(add_row_table(b.tgt, qpos, b.dqkin, Qs, nq, d, c.s));
            CONE_TRY(SG(b.dqkin, d, Qs, inw, inb, 2 * d, d, g));  // q | k of the self-attention
            g.C32 = b.dqk; g.ldc32 = 2 * d;
            CONE_TRY(tc_gemm_run(t, g, c.s));
            CONE_TRY(SG(b.tgt, d, Qs, inw + (size_t)2 * d * d, inb + 2 * d, d, d, g));  // v
            g.C32 = b.dv; g.ldc32 = d;
            CONE_TRY(tc_gemm_run(t, g, c.s));
            CONE_TRY(dec_self_attention(b.dqk, 2 * d, b.dv, d, b.datt, d, shared ? 1 : b.B, nq, H, 0, c.s));
            CONE_TRY(SG(b.datt, d, Qs, c.w->p(p + ".self_attn.out_proj.weight"), c.w->p(p + ".self_attn.out_proj.bias"), d, d, g));
            LN(g, p + ".norm1");
            CONE_TRY(tc_gemm_run(t, g, c.s));
            CONE_TRY(add_row_table(b.tgt, qpos, b.dqkin, Qs, nq, d, c.s));
            // cross-attention on the raw memory: q | Wk_h^T q_h in one GEMM (N = 9 d), pooled memory per head out of the
            // attention kernel, Wv_h and the output projection folded into the next GEMM (K = 8 d)
            CONE_TRY(SG(b.dqkin, d, Qs, c.w->xq_w[l], c.w->xq_b[l], 9 * d, d, g));
            g.C16 = b.dqt16; g.ldc16 = 9 * d;
            CONE_TRY(tc_gemm_run(t, g, c.s));
            if (shared) {  // the fp32 residual of every window = the shared rows (staged in b.hs, free until the heads)
                CONE_CUDA(cudaMemcpyAsync(b.hs, b.tgt, sizeof(float) * nq * d, cudaMemcpyDeviceToDevice, c.s));
                CONE_TRY(add_row_table(nullptr, b.hs, b.tgt, Q, nq, d, c.s));
            }
            CONE_TRY(dec_cross_attention_mem(b.src16, d, b.dqt16, 9 * d, b.dpm16, 8 * d, b.vlen, b.tlen, b.B, nq, b.Lv, b.Lt,
                                             c.w->pos_kdec16 + (size_t)l * d, (int64_t)DL * d, dm.max_v_l, c.s, shared ? 1 : 0));
            // the pooled memory only exists in fp16: 2-product GEMM (weights hi + lo)
            g = TcGemmArgs();
            g.A16 = b.dpm16; g.lda = 8 * d; g.M = Q; g.W = c.w->xo_w[l]; g.bias = c.w->xo_b[l]; g.N = d; g.K = 8 * d; g.wsplit = 1;
            LN(g, p + ".norm2");
            CONE_TRY(tc_gemm_run(t, g, c.s));
            // FFN: linear1 as a split GEMM writing the hidden activations straight to fp16 (their rounding is the one
            // decoder rounding the emulation shows to be harmless: 1.47e-4 -> 1.50e-4 rms), linear2 as a 2-product GEMM
            // (fp16 hidden x weights hi + lo)
            CONE_TRY(SG(b.tgt, d, Q, c.w->p(p + ".linear1.weight"), c.w->p(p + ".linear1.bias"), ff, d, g));
            g.relu = 1; g.C16 = b.dh16; g.ldc16 = ff;
            CONE_TRY(tc_gemm_run(t, g, c.s));
            g = TcGemmArgs();
            g.A16 = b.dh16; g.lda = ff; g.M = Q; g.W = c.w->p(p + ".linear2.weight"); g.bias = c.w->p(p + ".linear2.bias");
            g.N = d; g.K = ff; g.wsplit = 1;
            LN(g, p + ".norm3");
            CONE_TRY(tc_gemm_run(t, g, c.s));
        }
        const bool last = (l == DL - 1);
        if (last || aux_logits || aux_spans) {
            CONE_TRY(layernorm_rows(b.tgt, nullptr, c.w->p("transformer.decoder.norm.weight"),
                                    c.w->p("transformer.decoder.norm.bias"), b.hs, Q, d, 1e-5f, c.s));
            if (last) {
                CONE_TRY(heads(c, b, b.hs, Q, logits, prob_fg, spans));
            } else {
                CONE_TRY(heads(c, b, b.hs, Q, aux_logits ? aux_logits + (size_t)l * Q * 2 : nullptr, nullptr,
                               aux_spans ? aux_spans + (size_t)l * Q * 2 : nullptr));
            }
        }
    }
    return CONE_OK;
}

// A9 after pooling: adapter + residual, normalise, dot with the normalised CLS
struct MatchBuffers {
    float *pooled, *hid, *adapted, *tnorm;
};
MatchBuffers plan_match(Arena& a, const cone_dims& c, int64_t B, int64_t n_cls) {
    MatchBuffers m;
    const int64_t Q = B * c.num_queries;
    m.pooled = a.get<float>(Q * c.v_dim);
    m.hid = a.get<float>(Q * c.hidden);
    m.adapted = a.get<float>(Q * c.v_dim);
    m.tnorm = a.get<float>(n_cls * c.v_dim);
    return m;
}
int match_core(const Ctx& c, const void* frames, int frames_dtype, int64_t n_frames, const CoreBuffers& b,
               const float* spans, const float* cls, int64_t n_cls, MatchBuffers& m, float* out, int nq) {
    const int dv = c.w->dims.v_dim;
    CONE_TRY(span_mean_pool(frames, frames_dtype, n_frames, b.vid_base, b.vlen, b.pad_len, spans, m.pooled, b.B, nq, dv, c.s));
    CONE_TRY(adapter_rows(c, m.pooled, b.B * nq, m.hid, m.adapted, 1));
    CONE_TRY(l2norm_rows(cls, m.tnorm, n_cls, dv, 0.f, c.s));  // text_cls / ||text_cls|| (model.py:142)
    CONE_TRY(norm_dot(m.adapted, m.tnorm, b.qidx, out, b.B, nq, dv, c.s));
    return CONE_OK;
}

// pos . [Wq; Wk]^T per encoder layer and pos . Wk^T per decoder layer, for every (valid length, row): fp32 tables (and
// the fp16 copy the mma.sync cross-attention reads), recomputed whenever the weights change
int fill_pos_proj(cone_weights* mw, cudaStream_t s) {
    const cone_dims& dm = mw->dims;
    const size_t d = dm.hidden, rows = (size_t)(dm.max_v_l + 1) * dm.max_v_l;
    const size_t per_enc = rows * 2 * d, dec = rows * dm.dec_layers * d;
    mw->pos_qk.clear();
    for (int l = 0; l < dm.enc_layers; ++l) {
        float* out = mw->pos_proj + per_enc * l;
        GemmParams g;
        g.A = mw->pos_table; g.lda = d;
        g.W = mw->p("transformer.encoder.layers." + std::to_string(l) + ".self_attn.in_proj_weight"); g.ldw = d;
        g.C = out; g.ldc = 2 * d; g.M = rows; g.N = 2 * d; g.K = d;
        CONE_TRY(sgemm_nt(g, s));
        mw->pos_qk.push_back(out);
    }
    mw->pos_kdec = mw->pos_proj + per_enc * dm.enc_layers;
    GemmParams g;
    g.A = mw->pos_table; g.lda = d; g.W = mw->dec_kw; g.ldw = d;
    g.C = mw->pos_kdec; g.ldc = dm.dec_layers * d; g.M = rows; g.N = dm.dec_layers * d; g.K = d;
    CONE_TRY(sgemm_nt(g, s));
    CONE_TRY(f32_to_f16_rows(mw->pos_kdec, dm.dec_layers * d, mw->pos_kdec16, rows, (int)(dm.dec_layers * d), s));
    CONE_TRY(f32_to_f16_rows(mw->pos_proj, 2 * d, mw->pos_qk16, rows * dm.enc_layers, (int)(2 * d), s));
    (void)dec;
    return CONE_OK;
}

int ensure_tc(const cone_weights* w, int prec, cudaStream_t s) {
    if (prec != CONE_PREC_TC) return CONE_OK;
    cone_weights* mw = const_cast<cone_weights*>(w);
    if (mw->tc == nullptr) CONE_TRY(tc_weights_create(&mw->tc, s));
    if (mw->pos_proj == nullptr) {
        const cone_dims& dm = w->dims;
        const size_t d = dm.hidden, rows = (size_t)(dm.max_v_l + 1) * dm.max_v_l;
        CONE_CUDA(cudaMalloc(&mw->pos_proj, sizeof(float) * (rows * 2 * d * dm.enc_layers + rows * dm.dec_layers * d)));
        CONE_CUDA(cudaMalloc(&mw->pos_kdec16, sizeof(uint16_t) * rows * dm.dec_layers * d));
        CONE_CUDA(cudaMalloc(&mw->pos_qk16, sizeof(uint16_t) * rows * 2 * d * dm.enc_layers));
        CONE_TRY(fill_pos_proj(mw, s));
    }
    return CONE_OK;
}

int check_prec(int prec) {
    CONE_REQUIRE(prec == CONE_PREC_FP32 || prec == CONE_PREC_TC, "unknown precision %d", prec);
    return CONE_OK;
}

// a raw feature tensor of an _ex entry point: known storage type; 16-bit rows are read 4 elements (8 bytes) at a time,
// and a sliced view can start at any element
int check_feature(const char* who, const char* name, const void* p, int32_t dtype) {
    CONE_REQUIRE(feature_elem_bytes(dtype) != 0, "%s: unknown dtype %d for %s", who, dtype, name);
    CONE_REQUIRE(dtype == CONE_DTYPE_F32 || ((uintptr_t)p & 7) == 0,
                 "%s: %s is a 16-bit feature tensor at %p, which is not 8-byte aligned", who, name, p);
    return CONE_OK;
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// entry points
// ------------------------------------------------------------------------------------------------
extern "C" int cone_l2_normalize(const float* x, float* out, int64_t rows, int32_t dim, float eps, void* stream) {
    return cone_l2_normalize_ex(x, CONE_DTYPE_F32, out, rows, dim, eps, stream);
}

extern "C" int cone_l2_normalize_ex(const void* x, int32_t x_dtype, float* out, int64_t rows, int32_t dim, float eps,
                                    void* stream) {
    CONE_TRY(check_feature("cone_l2_normalize_ex", "x", x, x_dtype));
    CONE_REQUIRE(x_dtype == CONE_DTYPE_F32 || x != out, "cone_l2_normalize_ex: in place needs fp32 x");
    return l2norm_rows(x, x_dtype, out, rows, dim, eps, (cudaStream_t)stream);
}

extern "C" size_t cone_prepare_workspace_bytes(const cone_dims* dims, int64_t n_frames) {
    if (check_dims(dims) != CONE_OK) return 0;
    Arena a(nullptr, 0);
    const int dm = motion_dim(*dims), dx = dims->v_dim > dm ? dims->v_dim : dm;
    a.get<float>(n_frames * dx);           // xn: normalised appearance or motion rows
    a.get<float>(n_frames * dims->hidden); // adapter hidden
    a.get<float>(n_frames * dims->v_dim);  // adapted
    plan_proj(a, n_frames, dm, dims->hidden);
    return a.used + tc_scratch_bytes(n_frames, dx > dims->ffn ? dx : dims->ffn);
}

// rows per slab of the frame stage: n_frames halved until the slab's buffers fit the workspace
static int64_t prepare_slab(const cone_dims& dm, int64_t n_frames, size_t workspace_bytes, const char* who) {
    int64_t slab = n_frames;
    while (slab > 1 && cone_prepare_workspace_bytes(&dm, slab) > workspace_bytes) slab = (slab + 1) / 2;
    if (cone_prepare_workspace_bytes(&dm, slab) > workspace_bytes) {
        set_error("%s: workspace of %zu bytes cannot hold one frame", who, workspace_bytes);
        return -1;
    }
    return slab;
}

extern "C" int cone_video_prepare(const cone_weights* w, const float* frames_raw, int64_t n_frames, float* ctx_out,
                                  float* vidproj_out, void* workspace, size_t workspace_bytes, int precision,
                                  void* stream) {
    return cone_video_prepare_ex(w, frames_raw, CONE_DTYPE_F32, n_frames, ctx_out, vidproj_out, workspace, workspace_bytes,
                                 precision, stream);
}

extern "C" int cone_video_prepare_ex(const cone_weights* w, const void* frames_raw, int32_t frames_dtype, int64_t n_frames,
                                     float* ctx_out, float* vidproj_out, void* workspace, size_t workspace_bytes,
                                     int precision, void* stream) {
    CONE_REQUIRE(w && frames_raw, "null argument");
    CONE_TRY(check_feature("cone_video_prepare", "frames_raw", frames_raw, frames_dtype));
    CONE_TRY(check_prec(precision));
    const cone_dims& dm = w->dims;
    CONE_REQUIRE(vidproj_out == nullptr || motion_dim(dm) == dm.v_dim,
                 "cone_video_prepare: the handle reads %d-d motion features: project them with cone_video_prepare_motion",
                 motion_dim(dm));
    Ctx c{w, precision, (cudaStream_t)stream};
    CONE_TRY(ensure_tc(w, precision, c.s));
    // frames are processed in slabs sized to the workspace
    const int64_t slab = prepare_slab(dm, n_frames, workspace_bytes, "cone_video_prepare");
    if (slab < 0) return CONE_ERR_WORKSPACE;
    for (int64_t f0 = 0; f0 < n_frames; f0 += slab) {
        const int64_t n = (n_frames - f0) < slab ? (n_frames - f0) : slab;
        Arena a(workspace, workspace_bytes);
        float* xn = a.get<float>(n * dm.v_dim);
        float* hid = a.get<float>(n * dm.hidden);
        float* ad = a.get<float>(n * dm.v_dim);
        ProjBuffers pb = plan_proj(a, n, dm.v_dim, dm.hidden);
        tc_set_scratch(w->tc, a.base ? a.base + a.used : nullptr, workspace_bytes > a.used ? workspace_bytes - a.used : 0);
        const void* x = static_cast<const char*>(frames_raw) + f0 * dm.v_dim * feature_elem_bytes(frames_dtype);
        if (ctx_out) {
            // host-side L2 norm of the dataset (dataloader:459), adapter + residual, no-eps norm (inference.py:255-257)
            CONE_TRY(l2norm_rows(x, frames_dtype, xn, n, dm.v_dim, 1e-5f, c.s));
            const Ctx c32{w, CONE_PREC_FP32, c.s};  // the window ranking must be bit-stable across precisions
            CONE_TRY(adapter_rows(c32, xn, n, hid, ad, 1));
            CONE_TRY(l2norm_rows(ad, ctx_out + f0 * dm.v_dim, n, dm.v_dim, 0.f, c.s));
        }
        if (vidproj_out)
            CONE_TRY(input_proj(c, "input_vid_proj", x, frames_dtype, n, dm.v_dim, vidproj_out + f0 * dm.hidden, pb));
    }
    return CONE_OK;
}

extern "C" int cone_video_prepare_motion(const cone_weights* w, const float* motion_raw, int64_t n_frames,
                                         float* vidproj_out, void* workspace, size_t workspace_bytes, int precision,
                                         void* stream) {
    return cone_video_prepare_motion_ex(w, motion_raw, CONE_DTYPE_F32, n_frames, vidproj_out, workspace, workspace_bytes,
                                        precision, stream);
}

extern "C" int cone_video_prepare_motion_ex(const cone_weights* w, const void* motion_raw, int32_t motion_dtype,
                                            int64_t n_frames, float* vidproj_out, void* workspace, size_t workspace_bytes,
                                            int precision, void* stream) {
    CONE_REQUIRE(w && motion_raw && vidproj_out, "null argument");
    CONE_TRY(check_feature("cone_video_prepare_motion", "motion_raw", motion_raw, motion_dtype));
    CONE_REQUIRE(n_frames >= 0, "cone_video_prepare_motion: n_frames=%lld", (long long)n_frames);
    CONE_TRY(check_prec(precision));
    Ctx c{w, precision, (cudaStream_t)stream};
    CONE_TRY(ensure_tc(w, precision, c.s));
    const cone_dims& dm = w->dims;
    const int dmot = motion_dim(dm);
    const int64_t slab = prepare_slab(dm, n_frames, workspace_bytes, "cone_video_prepare_motion");
    if (slab < 0) return CONE_ERR_WORKSPACE;
    for (int64_t f0 = 0; f0 < n_frames; f0 += slab) {
        const int64_t n = (n_frames - f0) < slab ? (n_frames - f0) : slab;
        Arena a(workspace, workspace_bytes);
        float* xn = a.get<float>(n * dmot);
        ProjBuffers pb = plan_proj(a, n, dmot, dm.hidden);
        tc_set_scratch(w->tc, a.base ? a.base + a.used : nullptr, workspace_bytes > a.used ? workspace_bytes - a.used : 0);
        // the dataloader normalises motion rows on the host (ego4d_mad_dataloader.py:284-292) before input_vid_proj
        CONE_TRY(l2norm_rows(static_cast<const char*>(motion_raw) + f0 * dmot * feature_elem_bytes(motion_dtype), motion_dtype,
                             xn, n, dmot, 1e-5f, c.s));
        CONE_TRY(input_proj(c, "input_vid_proj", xn, n, dmot, vidproj_out + f0 * dm.hidden, pb));
    }
    return CONE_OK;
}

extern "C" int cone_adapter(const cone_weights* w, const float* x, float* out, int64_t rows, int residual,
                            void* workspace, size_t workspace_bytes, int precision, void* stream) {
    CONE_REQUIRE(w && x && out, "null argument");
    CONE_TRY(check_prec(precision));
    Ctx c{w, precision, (cudaStream_t)stream};
    CONE_TRY(ensure_tc(w, precision, c.s));
    Arena a(workspace, workspace_bytes);
    float* hid = a.get<float>(rows * w->dims.hidden);
    if (!a.fits()) {
        set_error("cone_adapter: workspace needs %zu bytes", a.used);
        return CONE_ERR_WORKSPACE;
    }
    tc_set_scratch(w->tc, a.base + a.used, workspace_bytes - a.used);
    return adapter_rows(c, x, rows, hid, out, residual);
}

extern "C" int cone_linear(const cone_weights* w, const float* x, const float* W, const float* bias, int64_t M, int32_t N,
                           int32_t K, int relu, const float* residual, float* y, void* workspace, size_t workspace_bytes,
                           int precision, void* stream) {
    CONE_REQUIRE(w && x && W && y, "null argument");
    if (precision == CONE_PREC_TC_SPLIT) {  // operator-level access to the 3-product GEMM (tests)
        CONE_REQUIRE(workspace && workspace_bytes >= (size_t)M * 3 * K * 2, "cone_linear: split GEMM needs %zu bytes of workspace",
                     (size_t)M * 3 * K * 2);
        Ctx c{w, precision, (cudaStream_t)stream, static_cast<uint16_t*>(workspace)};
        CONE_TRY(ensure_tc(w, CONE_PREC_TC, c.s));
        return linear(c, x, K, M, W, bias, N, K, y, N, relu, residual, N);
    }
    CONE_TRY(check_prec(precision));
    Ctx c{w, precision, (cudaStream_t)stream};
    CONE_TRY(ensure_tc(w, precision, c.s));
    tc_set_scratch(w->tc, workspace, workspace_bytes);
    return linear(c, x, K, M, W, bias, N, K, y, N, relu, residual, N);
}

extern "C" int cone_encoder_tail(const cone_weights* w, int32_t layer, const float* att, const float* res, int64_t M,
                                 float* out, int32_t cta_group, void* workspace, size_t workspace_bytes, void* stream) {
    CONE_REQUIRE(w && att && res && out && workspace, "null argument");
    const cone_dims& dm = w->dims;
    CONE_REQUIRE(layer >= 0 && layer < dm.enc_layers, "cone_encoder_tail: layer %d out of range", layer);
    CONE_REQUIRE(enc_tail_supported(dm.hidden, dm.ffn), "cone_encoder_tail: unsupported width");
    CONE_REQUIRE(M >= 1, "cone_encoder_tail: no rows");
    cudaStream_t s = (cudaStream_t)stream;
    CONE_TRY(ensure_tc(w, CONE_PREC_TC, s));
    const int d = dm.hidden;
    Arena a(workspace, workspace_bytes);
    uint16_t* att16 = a.get<uint16_t>(M * d);
    uint16_t* rhi = a.get<uint16_t>(M * d);
    uint16_t* rlo = a.get<uint16_t>(M * d);
    uint16_t* ohi = a.get<uint16_t>(M * d);
    uint16_t* olo = a.get<uint16_t>(M * d);
    if (!a.fits()) {
        set_error("cone_encoder_tail: workspace needs %zu bytes, got %zu", a.used, workspace_bytes);
        return CONE_ERR_WORKSPACE;
    }
    CONE_TRY(f32_to_f16_rows(att, d, att16, M, d, s));
    CONE_TRY(split_hilo_rows(res, rhi, rlo, M * d, s));
    const std::string p = "transformer.encoder.layers." + std::to_string(layer);
    EncTailArgs e;
    e.att16 = att16; e.lda = d;
    e.res_hi = rhi; e.res_lo = rlo; e.ldr = d;
    e.out_hi = ohi; e.out_lo = olo; e.ldo = d;
    e.M = M; e.d = d; e.ffn = dm.ffn;
    e.Wo = w->p(p + ".self_attn.out_proj.weight"); e.bo = w->p(p + ".self_attn.out_proj.bias");
    e.ln1_g = w->p(p + ".norm1.weight"); e.ln1_b = w->p(p + ".norm1.bias");
    e.W1 = w->p(p + ".linear1.weight"); e.b1 = w->p(p + ".linear1.bias");
    e.W2 = w->p(p + ".linear2.weight"); e.b2 = w->p(p + ".linear2.bias");
    e.ln2_g = w->p(p + ".norm2.weight"); e.ln2_b = w->p(p + ".norm2.bias");
    e.cta_group = cta_group;
    CONE_TRY(enc_tail_run(w->tc, e, s));
    return combine_hilo_rows(ohi, olo, out, M * d, s);
}

extern "C" int cone_frame_scores(const float* ctx, int32_t v_dim, const int64_t* video_offsets, const int32_t* q_first,
                                 int32_t n_videos, int32_t max_video_frames, int32_t max_video_queries,
                                 const float* cls_norm, float* score_out, const int64_t* score_offsets, int precision,
                                 void* stream) {
    CONE_REQUIRE(ctx && video_offsets && q_first && cls_norm && score_out && score_offsets, "null argument");
    CONE_TRY(check_prec(precision));
    // The window ranking must be bit-stable (SURVEY.md §7 H1): scores are always computed in fp32.
    return sgemm_frame_scores(ctx, cls_norm, v_dim, video_offsets, q_first, n_videos, max_video_frames,
                              max_video_queries, score_out, score_offsets, (cudaStream_t)stream);
}

extern "C" int cone_window_ranklist(const float* frame_score, const int64_t* score_offsets, const int32_t* frame_count,
                                    int32_t n_queries, int32_t max_v_l, int32_t* ranklist_out, float* winscore_out,
                                    int32_t ranklist_stride, void* stream) {
    CONE_REQUIRE(frame_score && score_offsets && frame_count && ranklist_out, "null argument");
    return window_ranklist(frame_score, score_offsets, frame_count, n_queries, max_v_l, ranklist_out, winscore_out,
                           ranklist_stride, (cudaStream_t)stream);
}

// ---- A1-A3 for one video in one call (SURVEY.md §8b `cone_prefilter`)
static int prefilter_windows(const cone_dims& dm, int64_t L) { return (int)((L + dm.max_v_l / 2 - 1) / (dm.max_v_l / 2)) + 1; }

extern "C" size_t cone_prefilter_workspace_bytes(const cone_dims* dims, int64_t L, int32_t n_queries) {
    if (check_dims(dims) != CONE_OK || L <= 0 || n_queries < 0) return 0;
    Arena a(nullptr, 0);
    const int nw = prefilter_windows(*dims, L);
    a.get<float>(L * dims->v_dim);                    // ctx
    a.get<float>((int64_t)n_queries * dims->v_dim);   // normalised CLS
    a.get<float>((int64_t)n_queries * L);             // frame scores
    a.get<int64_t>(2); a.get<int32_t>(2); a.get<int64_t>(n_queries); a.get<int32_t>(n_queries);
    a.get<int32_t>((int64_t)n_queries * nw);          // rank-lists
    a.get<float>((int64_t)n_queries * nw);            // window scores
    // the frame stage works in slabs sized to what is left: ask for enough to take a 4096-frame slab in one piece
    return a.used + cone_prepare_workspace_bytes(dims, L < 4096 ? L : 4096);
}

extern "C" int cone_prefilter(const cone_weights* w, const float* frames_raw, int64_t L, const float* cls_raw,
                              int32_t n_queries, int32_t topk, int32_t* win_idx, float* win_score, void* workspace,
                              size_t workspace_bytes, void* stream) {
    return cone_prefilter_ex(w, frames_raw, CONE_DTYPE_F32, L, cls_raw, CONE_DTYPE_F32, n_queries, topk, win_idx, win_score,
                             workspace, workspace_bytes, stream);
}

extern "C" int cone_prefilter_ex(const cone_weights* w, const void* frames_raw, int32_t frames_dtype, int64_t L,
                                 const void* cls_raw, int32_t cls_dtype, int32_t n_queries, int32_t topk, int32_t* win_idx,
                                 float* win_score, void* workspace, size_t workspace_bytes, void* stream) {
    CONE_REQUIRE(w && frames_raw && win_idx && (cls_raw || n_queries == 0), "null argument");
    CONE_TRY(check_feature("cone_prefilter", "frames_raw", frames_raw, frames_dtype));
    CONE_TRY(check_feature("cone_prefilter", "cls_raw", cls_raw, cls_dtype));
    CONE_REQUIRE(L > 0 && n_queries >= 0 && topk > 0, "cone_prefilter: L=%lld n_queries=%d topk=%d", (long long)L, n_queries, topk);
    if (n_queries == 0) return CONE_OK;
    const cone_dims& dm = w->dims;
    cudaStream_t s = (cudaStream_t)stream;
    const int nw = prefilter_windows(dm, L);
    Arena a(workspace, workspace_bytes);
    float* ctx = a.get<float>(L * dm.v_dim);
    float* cls_n = a.get<float>((int64_t)n_queries * dm.v_dim);
    float* scores = a.get<float>((int64_t)n_queries * L);
    int64_t* video_offsets = a.get<int64_t>(2);
    int32_t* q_first = a.get<int32_t>(2);
    int64_t* score_offsets = a.get<int64_t>(n_queries);
    int32_t* frame_count = a.get<int32_t>(n_queries);
    int32_t* ranklist = a.get<int32_t>((int64_t)n_queries * nw);
    float* winscore = a.get<float>((int64_t)n_queries * nw);
    if (!workspace || a.used >= workspace_bytes || cone_prepare_workspace_bytes(&dm, 1) > workspace_bytes - a.used) {
        set_error("cone_prefilter: workspace of %zu bytes, cone_prefilter_workspace_bytes() asks for %zu", workspace_bytes,
                  cone_prefilter_workspace_bytes(&dm, L, n_queries));
        return CONE_ERR_WORKSPACE;
    }
    // A1 + A2: normalised, adapted context features of every frame (always fp32: the ranking must be bit-stable)
    CONE_TRY(cone_video_prepare_ex(w, frames_raw, frames_dtype, L, ctx, nullptr, a.base + a.used, workspace_bytes - a.used,
                                   CONE_PREC_FP32, stream));
    CONE_TRY(l2norm_rows(cls_raw, cls_dtype, cls_n, n_queries, dm.v_dim, 1e-5f, s));  // dataloader:472
    // A3: frame scores, window maxima, full rank-list; the first topk entries leave
    CONE_TRY(prefilter_desc(video_offsets, q_first, score_offsets, frame_count, L, n_queries, s));
    CONE_REQUIRE(L <= INT32_MAX, "cone_prefilter: video too long");
    CONE_TRY(sgemm_frame_scores(ctx, cls_n, dm.v_dim, video_offsets, q_first, 1, (int)L, n_queries, scores, score_offsets, s));
    CONE_TRY(window_ranklist(scores, score_offsets, frame_count, n_queries, dm.max_v_l, ranklist, winscore, nw, s));
    return take_topk(ranklist, winscore, nw, n_queries, topk, win_idx, win_score, s);
}

namespace {
size_t ground_chunk_bytes(const cone_dims& dm, int64_t nqc, int topk, int Lv, int Lt, int prec) {
    Arena a(nullptr, 0);
    const int64_t B = nqc * topk;
    plan_core(a, dm, B, Lv, Lt, prec);
    plan_match(a, dm, B, nqc);
    a.get<float>(nqc * Lt * dm.hidden);  // txtproj
    plan_proj(a, nqc * Lt, dm.t_dim, dm.hidden);
    if (prec == CONE_PREC_TC) {
        a.get<uint16_t>(nqc * Lt * dm.hidden);      // txtproj16
        a.get<uint16_t>(nqc * Lt * 3 * dm.hidden);  // token q|k|v of encoder layer 0
    }
    return a.used + tc_scratch_bytes(B * (Lv + Lt), dm.ffn);
}
}  // namespace

extern "C" size_t cone_workspace_bytes(const cone_dims* dims, int64_t n_windows, int32_t lv, int32_t lt) {
    if (check_dims(dims) != CONE_OK) return 0;
    // dense forward: vid/txt projections of every row + core + matching
    Arena a(nullptr, 0);
    plan_core(a, *dims, n_windows, lv, lt, CONE_PREC_FP32);  // the fp32 plan is the larger one
    plan_match(a, *dims, n_windows, n_windows);
    a.get<float>(n_windows * lv * dims->hidden);
    a.get<float>(n_windows * lt * dims->hidden);
    plan_proj(a, n_windows * lv, motion_dim(*dims), dims->hidden);
    plan_proj(a, n_windows * lt, dims->t_dim, dims->hidden);
    return a.used + tc_scratch_bytes(n_windows * (lv + lt), dims->ffn) + 4096;
}

extern "C" int cone_ground_windows(const cone_weights* w, const float* frames_raw, int64_t n_frames,
                                   const float* vidproj, const int64_t* q_video_start, const int32_t* q_video_len,
                                   const int32_t* ranklist, int32_t ranklist_stride, const float* tok,
                                   const int32_t* tok_len, const float* cls_norm, const int32_t* q_batch,
                                   int32_t n_batches, int32_t n_queries, int32_t topk, float* pred_spans,
                                   float* prob_fg, float* match, int32_t* win_start, int32_t* win_len, void* workspace,
                                   size_t workspace_bytes, int precision, void* stream) {
    return cone_ground_windows_ex(w, frames_raw, CONE_DTYPE_F32, n_frames, vidproj, q_video_start, q_video_len, ranklist,
                                  ranklist_stride, tok, tok_len, cls_norm, q_batch, n_batches, n_queries, topk, pred_spans,
                                  prob_fg, match, win_start, win_len, workspace, workspace_bytes, precision, stream);
}

extern "C" int cone_ground_windows_ex(const cone_weights* w, const void* frames_raw, int32_t frames_dtype, int64_t n_frames,
                                      const float* vidproj, const int64_t* q_video_start, const int32_t* q_video_len,
                                      const int32_t* ranklist, int32_t ranklist_stride, const float* tok,
                                      const int32_t* tok_len, const float* cls_norm, const int32_t* q_batch,
                                      int32_t n_batches, int32_t n_queries, int32_t topk, float* pred_spans,
                                      float* prob_fg, float* match, int32_t* win_start, int32_t* win_len, void* workspace,
                                      size_t workspace_bytes, int precision, void* stream) {
    CONE_REQUIRE(w && frames_raw && vidproj && q_video_start && q_video_len && ranklist && tok && tok_len && cls_norm &&
                     pred_spans && prob_fg && match && win_start && win_len && workspace,
                 "null argument");
    CONE_TRY(check_feature("cone_ground_windows", "frames_raw", frames_raw, frames_dtype));
    CONE_REQUIRE(topk >= 1 && n_batches >= 1 && n_queries >= 0, "bad sizes");
    CONE_TRY(check_prec(precision));
    Ctx c{w, precision, (cudaStream_t)stream};
    CONE_TRY(ensure_tc(w, precision, c.s));
    const cone_dims& dm = w->dims;
    const int Lv = dm.max_v_l, Lt = dm.max_q_l, nq = dm.num_queries;
    if (n_queries == 0) return CONE_OK;

    // window descriptors of every query, and the per-eval-batch padded length the reference pools over
    CONE_TRY(build_windows(ranklist, ranklist_stride, q_video_len, n_queries, topk, Lv, win_start, win_len, c.s));
    Arena head(workspace, workspace_bytes);
    int32_t* batch_max = head.get<int32_t>(n_batches);
    if (!head.fits()) {
        set_error("cone_ground_windows: workspace too small");
        return CONE_ERR_WORKSPACE;
    }
    if (q_batch) CONE_TRY(batch_max_len(win_len, q_batch, n_queries, topk, batch_max, n_batches, c.s));
    // tensor-core mode: q|k|v of encoder layer 0 once per frame (the reference, and a per-window GEMM, compute the
    // same row once for every window that contains the frame: k * Nq * Lv rows against n_frames)
    uint16_t* frame_qkv = nullptr;
    uint16_t* vidproj16 = nullptr;
    uint16_t* vidproj16lo = nullptr;
    const int d = dm.hidden;
    const std::string l0 = "transformer.encoder.layers.0.self_attn";
    // window slicing fused into the encoder tail (TMA gather4 from the per-frame / per-token tables) instead of a gathered copy
    const bool tail_gather = precision == CONE_PREC_TC && fused_tail_enabled(dm) && tail_gather_enabled() &&
                             n_frames + (int64_t)n_queries * Lt < ((int64_t)1 << 31);
    if (precision == CONE_PREC_TC) {
        // [frames | tokens of the current chunk]: the fp16 (= hi) rows, and with tail_gather their lo parts
        vidproj16 = head.get<uint16_t>((n_frames + (tail_gather ? (int64_t)n_queries * Lt : 0)) * d);
        if (tail_gather) vidproj16lo = head.get<uint16_t>((n_frames + (int64_t)n_queries * Lt) * d);
        frame_qkv = head.get<uint16_t>(n_frames * 3 * d);
        if (!head.fits()) {
            set_error("cone_ground_windows: workspace too small for the per-frame projections");
            return CONE_ERR_WORKSPACE;
        }
        if (tail_gather) CONE_TRY(split_hilo_rows(vidproj, vidproj16, vidproj16lo, n_frames * d, c.s));
        else CONE_TRY(f32_to_f16_rows(vidproj, d, vidproj16, n_frames, d, c.s));
        TcGemmArgs g;
        g.A16 = vidproj16; g.lda = d; g.M = n_frames; g.W = w->p(l0 + ".in_proj_weight"); g.bias = w->p(l0 + ".in_proj_bias");
        g.N = 3 * d; g.K = d; g.C16 = frame_qkv; g.ldc16 = 3 * d;
        CONE_TRY(tc_gemm_run(w->tc, g, c.s));
    }

    const size_t avail = workspace_bytes - head.used;
    int64_t nqc = n_queries;
    while (nqc > 1 && ground_chunk_bytes(dm, nqc, topk, Lv, Lt, precision) > avail) nqc = (nqc + 1) / 2;
    if (ground_chunk_bytes(dm, nqc, topk, Lv, Lt, precision) > avail) {
        set_error("cone_ground_windows: workspace of %zu bytes cannot hold one query (%zu needed)", workspace_bytes,
                  ground_chunk_bytes(dm, 1, topk, Lv, Lt, precision) + head.used);
        return CONE_ERR_WORKSPACE;
    }
    for (int64_t q0 = 0; q0 < n_queries; q0 += nqc) {
        const int64_t n = (n_queries - q0) < nqc ? (n_queries - q0) : nqc;
        const int64_t B = n * topk;
        Arena a((char*)workspace + head.used, avail);
        CoreBuffers cb = plan_core(a, dm, B, Lv, Lt, precision);
        MatchBuffers mb = plan_match(a, dm, B, n);
        float* txtproj = a.get<float>(n * Lt * dm.hidden);
        ProjBuffers pb = plan_proj(a, n * Lt, dm.t_dim, dm.hidden);
        tc_set_scratch(w->tc, a.base + a.used, avail > a.used ? avail - a.used : 0);
        // text projection once per query (the reference recomputes it for each of the k windows)
        CONE_TRY(input_proj(c, "input_txt_proj", tok + q0 * Lt * dm.t_dim, n * Lt, dm.t_dim, txtproj, pb));
        uint16_t* txtproj16 = nullptr;
        if (precision == CONE_PREC_TC) {  // token q|k|v of encoder layer 0, once per query token
            txtproj16 = tail_gather ? vidproj16 + n_frames * d : a.get<uint16_t>(n * Lt * d);
            uint16_t* token_qkv = a.get<uint16_t>(n * Lt * 3 * d);
            tc_set_scratch(w->tc, a.base + a.used, avail > a.used ? avail - a.used : 0);
            if (tail_gather) CONE_TRY(split_hilo_rows(txtproj, txtproj16, vidproj16lo + n_frames * d, n * Lt * d, c.s));
            else CONE_TRY(f32_to_f16_rows(txtproj, d, txtproj16, n * Lt, d, c.s));
            TcGemmArgs g;
            g.A16 = txtproj16; g.lda = d; g.M = n * Lt; g.W = w->p(l0 + ".in_proj_weight"); g.bias = w->p(l0 + ".in_proj_bias");
            g.N = 3 * d; g.K = d; g.C16 = token_qkv; g.ldc16 = 3 * d;
            CONE_TRY(tc_gemm_run(w->tc, g, c.s));
            cb.frame_qkv = frame_qkv;
            cb.token_qkv = token_qkv;
            cb.n_frames = n_frames;
            cb.n_tokens = n * Lt;
            if (tail_gather) {
                cb.g_src_hi = vidproj16;
                cb.g_src_lo = vidproj16lo;
            }
        }
        CONE_TRY(fill_window_desc_chunk(q_video_start, win_start, win_len, tok_len, q_batch, batch_max, (int)q0, (int)n,
                                        topk, Lt, Lv, cb.vid_base, cb.vlen, cb.txt_base, cb.tlen, cb.pad_len, cb.qidx, c.s));
        if (tail_gather) {
            // nothing to copy: layer 0 reads q|k|v and its residual rows through the window descriptors
        } else if (precision == CONE_PREC_TC && fused_tail_enabled(dm)) {  // hi + lo of the projected rows (fp32-accurate residual)
            CONE_TRY(gather_window_rows_f16(vidproj, n_frames, cb.vid_base, txtproj, cb.txt_base, cb.src16, B, Lv, Lt, dm.hidden,
                                            c.s, cb.src16lo));
        } else if (precision == CONE_PREC_TC) {
            CONE_TRY(gather_window_rows_h2h(vidproj16, n_frames, cb.vid_base, txtproj16, cb.txt_base, cb.src16, B, Lv, Lt,
                                            dm.hidden, c.s));
        } else {
            CONE_TRY(gather_window_rows(vidproj, n_frames, cb.vid_base, txtproj, cb.txt_base, cb.src, B, Lv, Lt, dm.hidden, c.s));
        }
        float* spans_c = pred_spans + q0 * topk * nq * 2;
        CONE_TRY(transformer_core(c, cb, nullptr, prob_fg + q0 * topk * nq, spans_c, nullptr, nullptr, nullptr));
        CONE_TRY(match_core(c, frames_raw, frames_dtype, n_frames, cb, spans_c, cls_norm + q0 * dm.v_dim, n, mb, match + q0 * topk * nq, nq));
    }
    return CONE_OK;
}

extern "C" int cone_forward(const cone_weights* w, const float* src_txt, const int32_t* txt_len, const float* src_vid,
                            const int32_t* vid_len, int32_t B, int32_t Lt, int32_t Lv, float* pred_logits,
                            float* pred_spans, float* saliency, float* aux_logits, float* aux_spans, void* workspace,
                            size_t workspace_bytes, int precision, void* stream) {
    CONE_REQUIRE(w && src_txt && txt_len && src_vid && vid_len && pred_logits && pred_spans && workspace, "null argument");
    CONE_TRY(check_prec(precision));
    const cone_dims& dm = w->dims;
    CONE_REQUIRE(Lv >= 1 && Lv <= dm.max_v_l, "cone_forward: L_vid=%d exceeds max_v_l=%d of the weights handle", Lv, dm.max_v_l);
    CONE_REQUIRE(Lt >= 1 && Lv + Lt <= CONE_MAX_WINDOW_ROWS, "cone_forward: window of %d rows exceeds %d", Lv + Lt,
                 CONE_MAX_WINDOW_ROWS);
    if (B == 0) return CONE_OK;
    Ctx c{w, precision, (cudaStream_t)stream};
    CONE_TRY(ensure_tc(w, precision, c.s));
    Arena a(workspace, workspace_bytes);
    CoreBuffers cb = plan_core(a, dm, B, Lv, Lt, precision);
    float* vidproj = a.get<float>((int64_t)B * Lv * dm.hidden);
    float* txtproj = a.get<float>((int64_t)B * Lt * dm.hidden);
    ProjBuffers pv = plan_proj(a, (int64_t)B * Lv, motion_dim(dm), dm.hidden);
    ProjBuffers pt = plan_proj(a, (int64_t)B * Lt, dm.t_dim, dm.hidden);
    if (!a.fits()) {
        set_error("cone_forward: workspace needs %zu bytes, got %zu", a.used, workspace_bytes);
        return CONE_ERR_WORKSPACE;
    }
    tc_set_scratch(w->tc, a.base + a.used, workspace_bytes - a.used);
    CONE_TRY(input_proj(c, "input_vid_proj", src_vid, (int64_t)B * Lv, motion_dim(dm), vidproj, pv));
    CONE_TRY(input_proj(c, "input_txt_proj", src_txt, (int64_t)B * Lt, dm.t_dim, txtproj, pt));
    CONE_TRY(fill_window_desc_dense(cb.vid_base, cb.txt_base, cb.qidx, B, Lv, Lt, c.s));
    CONE_CUDA(cudaMemcpyAsync(cb.vlen, vid_len, sizeof(int32_t) * B, cudaMemcpyDeviceToDevice, c.s));
    CONE_CUDA(cudaMemcpyAsync(cb.tlen, txt_len, sizeof(int32_t) * B, cudaMemcpyDeviceToDevice, c.s));
    if (precision == CONE_PREC_TC) {
        CONE_TRY(gather_window_rows_f16(vidproj, (int64_t)B * Lv, cb.vid_base, txtproj, cb.txt_base, cb.src16, B, Lv, Lt,
                                        dm.hidden, c.s, fused_tail_enabled(dm) ? cb.src16lo : nullptr));
    } else {
        CONE_TRY(gather_window_rows(vidproj, (int64_t)B * Lv, cb.vid_base, txtproj, cb.txt_base, cb.src, B, Lv, Lt, dm.hidden, c.s));
    }
    return transformer_core(c, cb, pred_logits, nullptr, pred_spans, saliency, aux_logits, aux_spans);
}

extern "C" int cone_clip_matching(const cone_weights* w, const float* src_cls_txt, const float* src_vid_appear,
                                  const int32_t* vid_len, const float* spans, int32_t B, int32_t Lv, int32_t nq,
                                  float* out, void* workspace, size_t workspace_bytes, int precision, void* stream) {
    CONE_REQUIRE(w && src_cls_txt && src_vid_appear && vid_len && spans && out && workspace, "null argument");
    CONE_TRY(check_prec(precision));
    CONE_REQUIRE(nq >= 1 && nq <= 64, "cone_clip_matching: bad number of proposals");
    if (B == 0) return CONE_OK;
    const cone_dims& dm = w->dims;
    Ctx c{w, precision, (cudaStream_t)stream};
    CONE_TRY(ensure_tc(w, precision, c.s));
    Arena a(workspace, workspace_bytes);
    CoreBuffers cb{};
    cb.B = B;
    cb.vid_base = a.get<int64_t>(B);
    cb.txt_base = a.get<int64_t>(B);
    cb.vlen = a.get<int32_t>(B);
    cb.pad_len = a.get<int32_t>(B);
    cb.qidx = a.get<int32_t>(B);
    MatchBuffers mb;
    const int64_t Q = (int64_t)B * nq;
    mb.pooled = a.get<float>(Q * dm.v_dim);
    mb.hid = a.get<float>(Q * dm.hidden);
    mb.adapted = a.get<float>(Q * dm.v_dim);
    mb.tnorm = a.get<float>((int64_t)B * dm.v_dim);
    if (!a.fits()) {
        set_error("cone_clip_matching: workspace needs %zu bytes, got %zu", a.used, workspace_bytes);
        return CONE_ERR_WORKSPACE;
    }
    tc_set_scratch(w->tc, a.base + a.used, workspace_bytes - a.used);
    CONE_TRY(fill_window_desc_dense(cb.vid_base, cb.txt_base, cb.qidx, B, Lv, 0, c.s));
    CONE_CUDA(cudaMemcpyAsync(cb.vlen, vid_len, sizeof(int32_t) * B, cudaMemcpyDeviceToDevice, c.s));
    CONE_TRY(fill_i32(cb.pad_len, B, Lv, c.s));  // the dense tensor is already padded to Lv rows
    return match_core(c, src_vid_appear, CONE_DTYPE_F32, (int64_t)B * Lv, cb, spans, src_cls_txt, B, mb, out, nq);
}

extern "C" int cone_fuse_nms(const float* pred_spans, const float* prob_fg, const float* match, const int32_t* win_start,
                             const int32_t* win_len, int32_t n_queries, int32_t topk, int32_t nq, float clip_length,
                             double nms_thd, int32_t max_before_nms, int32_t max_after_nms, double* out,
                             int32_t* out_count, double* rows_out, int32_t* rows_count, void* stream) {
    CONE_REQUIRE(pred_spans && prob_fg && match && win_start && win_len && out && out_count, "null argument");
    return fuse_nms(pred_spans, prob_fg, match, win_start, win_len, n_queries, topk, nq, clip_length, nms_thd,
                    max_before_nms, max_after_nms, out, out_count, rows_out, rows_count, (cudaStream_t)stream);
}

extern "C" int cone_fuse_nms_ex(const float* pred_spans, const float* prob_fg, const float* match,
                                const int32_t* win_start, const int32_t* win_len, int32_t n_queries, int32_t topk, int32_t nq,
                                float clip_length, double nms_thd, int32_t max_before_nms, int32_t max_after_nms,
                                int32_t fixed_duration, int32_t sort_within_window, double* out, int32_t* out_count,
                                double* rows_out, int32_t* rows_count, void* stream) {
    CONE_REQUIRE(pred_spans && prob_fg && match && win_start && win_len && out && out_count, "null argument");
    CONE_REQUIRE(fixed_duration >= 0, "cone_fuse_nms_ex: fixed_duration must be >= 0");
    return fuse_nms(pred_spans, prob_fg, match, win_start, win_len, n_queries, topk, nq, clip_length, nms_thd,
                    max_before_nms, max_after_nms, out, out_count, rows_out, rows_count, (cudaStream_t)stream,
                    fixed_duration, sort_within_window != 0);
}

extern "C" int cone_temporal_nms(const double* st, const double* ed, const double* score, int32_t n, double nms_thd,
                                 int32_t max_after_nms, int32_t* keep_out, int32_t* n_keep_out, void* stream) {
    CONE_REQUIRE(keep_out && n_keep_out && (n == 0 || (st && ed && score)), "null argument");
    return temporal_nms_single(st, ed, score, n, nms_thd, max_after_nms, keep_out, n_keep_out, (cudaStream_t)stream);
}

extern "C" int cone_eval_recall(const double* nms, const int32_t* nms_count, const double* gt, int32_t n_queries,
                                int32_t max_after_nms, const int32_t* topk_host, int32_t n_topk,
                                const double* thresholds_host, int32_t n_thresholds, int32_t flavour, int64_t* hits,
                                double* top1_iou, void* stream) {
    CONE_REQUIRE(n_queries == 0 || (nms && nms_count && gt), "null argument");
    CONE_REQUIRE(hits && topk_host && thresholds_host && max_after_nms >= 1, "null argument");
    return eval_recall(nms, nms_count, gt, n_queries, max_after_nms, topk_host, n_topk, thresholds_host, n_thresholds,
                       flavour, hits, top1_iou, (cudaStream_t)stream);
}

extern "C" int cone_eval_window_recall(const int32_t* ranklist, int32_t ranklist_stride, const double* gt,
                                       int32_t n_queries, double clip_length, int32_t max_v_l, const int32_t* topk_host,
                                       int32_t n_topk, int64_t* hits, void* stream) {
    CONE_REQUIRE(n_queries == 0 || (ranklist && gt), "null argument");
    CONE_REQUIRE(hits && topk_host && ranklist_stride >= 1, "null argument");
    return eval_window_recall(ranklist, ranklist_stride, gt, n_queries, clip_length, max_v_l, topk_host, n_topk, hits,
                              (cudaStream_t)stream);
}
