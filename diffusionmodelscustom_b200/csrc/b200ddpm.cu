// b200ddpm: C-ABI implementation (include/b200ddpm.h) — handle, weight re-packing, the per-step kernel program for
// Family R (DiffusionNet) and the CUDA-graph sampling loop.  Host orchestration only; all arithmetic is in the kernels.
#include "../../include/b200ddpm.h"

#include <chrono>
#include <cmath>
#include <cstring>
#include <functional>
#include <map>
#include <memory>
#include <vector>

#include "attention.cuh"
#include "attention_tc.cuh"
#include "attention_tc2.cuh"
#include "attention_tc3.cuh"
#include "attention_tc3d32.cuh"
#include "attention_tc6.cuh"
#include "attention_tc8.cuh"
#include "attn_block.cuh"
#include "common.cuh"
#include "conv.cuh"
#include "conv_persist.cuh"
#include "elementwise.cuh"
#include "evalops.cuh"
#include "gemm_stream.cuh"
#include "norm_fused.cuh"
#include "tail_tc.cuh"

namespace b2d {
thread_local Status g_status;
int g_pdl_enabled = getenv("B2D_NO_PDL") ? 0 : 1;

static inline cudaStream_t as_stream(void* s) { return reinterpret_cast<cudaStream_t>(s); }

struct HostTensor {
    std::vector<float> v;
    std::vector<int64_t> shape;
    size_t numel() const { return v.size(); }
};

static inline uint16_t f2h(float f) {   // host fp32 -> fp16 bits (round to nearest even, saturating)
    const float c = f > 65504.0f ? 65504.0f : (f < -65504.0f ? -65504.0f : f);
    const __half h = __float2half_rn(c);
    uint16_t u;
    memcpy(&u, &h, 2);
    return u;
}

typedef std::function<int(cudaStream_t)> OpFn;
// One kernel launch of the per-step program, with the algorithmic work it represents (for roofline reporting).
struct Op {
    std::string name;   // layer, e.g. "l2b0.c1"
    std::string klass;  // kernel class, e.g. "conv_tc", "flash_attn"
    double flops = 0;   // algorithmic FLOPs of this launch (2*M*N*K; attention 4*L^2*C per sample)
    double bytes = 0;   // algorithmic HBM bytes of this launch (activations read + written, weights once)
    OpFn fn;
    bool side = false;  // independent of the next op(s): launched on the handle's side stream (a concurrent graph branch)
    bool join = false;  // first op that consumes the side branch's result: waits for it
    int operator()(cudaStream_t st) const { return fn(st); }
};
struct OpList {
    std::vector<Op> v;
    Op pending;
    void meta(const std::string& name, const std::string& klass, double flops, double bytes) {
        pending.name = name; pending.klass = klass; pending.flops = flops; pending.bytes = bytes;
    }
    void push_back(OpFn f) {
        pending.fn = std::move(f);
        v.push_back(pending);
        pending = Op();
    }
};

struct EnsembleRes;
void ensemble_release(EnsembleRes* r);
struct Handle {
    b2d_config cfg{};
    int num_sms = 148;
    std::vector<void*> allocs;       // live for the life of the handle
    std::vector<void*> prog_allocs;  // activations/workspaces of the current per-batch program
    bool in_prog = false;
    std::map<std::string, HostTensor> sd;
    std::map<std::string, void*> dev;  // packed device weights by role name
    bool weights_loaded = false;

    // schedule
    int T = 0;
    float *d_betas = nullptr, *d_alphas = nullptr, *d_alpha_hat = nullptr;

    // per-batch program
    int prog_B = 0;
    std::vector<Op> step_ops;    // one eps evaluation (reads cur_x, writes cur_eps)
    size_t stats_floats = 0;
    float* d_stats = nullptr;
    const float* cur_x = nullptr;
    float* cur_eps = nullptr;
    float* d_eps = nullptr;  // internal eps buffer for sampling
    int *d_t = nullptr, *d_step = nullptr, *d_y = nullptr;
    bool has_y = false, has_cond_set = false;
    float* d_cond_stack = nullptr;  // [B][Ccond][H][H] fp32 (lsm, topo, cond...)
    float* d_cond_pre = nullptr;    // [B][H/2][H/2][64] fp32 : conv1 contribution of the conditioning channels
    float* d_temb = nullptr;        // [B][n_temb]
    int n_temb = 0;
    float* d_noise_stage = nullptr;
    size_t noise_stage_elems = 0;

    // Sampling graphs.  Everything a sampling job can change between calls (the state pointer, host-injected noise, seed, sample
    // offset, noise scale) lives in the device-resident SampleJob block that posterior_update_kernel reads, and the state itself
    // is the handle's own d_x_work buffer, so the graphs depend on (program, schedule tables, has_y) only and are captured ONCE:
    // graph_multi holds `graph_steps` consecutive reverse steps (PDL overlap spans the step boundaries), graph_one a single
    // step for the remainder of (T-1) / graph_steps.
    cudaGraphExec_t graph_multi = nullptr, graph_one = nullptr;
    int graph_steps = 0, graph_nodes_multi = 0, graph_nodes_one = 0;
    // DDIM sampler (b2d_set_timesteps): the sequence tau, its per-step coefficients and the step index k are device-resident, so
    // its own graph pair depends on (program, schedule tables, has_y) like the DDPM pair and not on S; the two pairs coexist.
    bool ddim = false;                 // sampler mode of sample_core: false = the reference DDPM loop
    std::vector<int> ddim_tau;         // tau_0 > ... > tau_{S-1}
    float ddim_eta = 0.f;
    bool ddim_dirty = true;            // sequence, eta or schedule changed since the tables were uploaded
    int ddim_cap = 0;                  // entries of d_ddim_tau (T + 1: S <= T-1 plus two trailing zeros)
    int* d_ddim_tau = nullptr;
    float4* d_ddim_coef = nullptr;     // [S] {cx, ce, sigma, 0} from ddim_coefficients()
    int* d_t_next = nullptr;           // [max_batch] tau_{k+1}: the timestep the DDIM side branch embeds
    cudaGraphExec_t graph_multi_ddim = nullptr, graph_one_ddim = nullptr;
    int graph_nodes_multi_ddim = 0, graph_nodes_one_ddim = 0;
    std::vector<float> h_alpha_hat;    // host copy of the schedule's alpha_hat (the DDIM coefficients are computed from it)
    SampleJob* d_job = nullptr;
    float* d_x_work = nullptr;       // [max_batch][c_hr][H][H] fp32: the diffusion state of the running job
    // host-entry staging (allocated once with the handle: no cudaMalloc/cudaFree inside b2d_sample_host)
    float *d_lsm_stage = nullptr, *d_topo_stage = nullptr, *d_cond_stage = nullptr;
    size_t cond_stage_elems = 0;
    int* h_y_pinned = nullptr;       // pinned int32 labels for the host entry
    struct EnsembleRes* ens = nullptr;   // double-buffered staging of the ensemble driver (ensemble.cuh), created on first use
    int64_t last_launches = 0;
    cudaStream_t own_stream = nullptr;
    // Time-embedding pipelining inside the reverse loop: d_temb depends on the step index only, so the projections for
    // step i-1 are launched on a side stream as soon as step i's last reader of d_temb has been enqueued, and overlap the
    // final layer + posterior update (a concurrent branch of the captured step graph).
    // stand-alone Encoder.forward / Decoder.forward (Family R): op range of the decoder and the five feature maps
    int dec_begin_op = -1;
    struct Fmap { f16* p; int C, hw; } fmaps[5] = {};
    int temb_free_op = -1;   // index of the first step op after the last reader of d_temb (set by the program builders)
    int* temb_t = nullptr;   // timesteps the next temb launch reads: d_t, or d_t_next on the DDIM side branch
    int temb_t_off = 0;      // added to *temb_t by the next temb launch (-1 on the DDPM side branch)
    cudaStream_t side_stream = nullptr;
    cudaEvent_t ev_side_fork = nullptr, ev_side_join = nullptr;
    cudaEvent_t ev_br_fork = nullptr, ev_br_join = nullptr;   // Op::side / Op::join branches
    struct Tap { const f16* p; int C, hw; };
    std::map<std::string, Tap> taps;  // named activations (NHWC f16) readable through b2d_debug_read

    template <typename T>
    int alloc(T** p, size_t count) {
        void* q = nullptr;
        B2D_CUDA(cudaMalloc(&q, count * sizeof(T) + 256));
        (in_prog ? prog_allocs : allocs).push_back(q);
        *p = reinterpret_cast<T*>(q);
        return 0;
    }
    void free_program() {
        for (void* p : prog_allocs) cudaFree(p);
        prog_allocs.clear();
        step_ops.clear();
        taps.clear();
        prog_B = 0;
    }
    void drop_ddim_graphs() {
        if (graph_multi_ddim) cudaGraphExecDestroy(graph_multi_ddim);
        if (graph_one_ddim) cudaGraphExecDestroy(graph_one_ddim);
        graph_multi_ddim = graph_one_ddim = nullptr;
    }
    void drop_graphs() {
        if (graph_multi) cudaGraphExecDestroy(graph_multi);
        if (graph_one) cudaGraphExecDestroy(graph_one);
        graph_multi = graph_one = nullptr;
        drop_ddim_graphs();
    }
    // cudaFree of one long-lived allocation (schedule tables / noise staging that are re-sized)
    void release(void* p) {
        if (!p) return;
        for (auto it = allocs.begin(); it != allocs.end(); ++it)
            if (*it == p) { allocs.erase(it); break; }
        cudaFree(p);
    }
    ~Handle() {
        drop_graphs();
        ensemble_release(ens);
        if (h_y_pinned) cudaFreeHost(h_y_pinned);
        free_program();
        for (void* p : allocs) cudaFree(p);
        if (own_stream) cudaStreamDestroy(own_stream);
        if (side_stream) cudaStreamDestroy(side_stream);
        if (ev_side_fork) cudaEventDestroy(ev_side_fork);
        if (ev_side_join) cudaEventDestroy(ev_side_join);
        if (ev_br_fork) cudaEventDestroy(ev_br_fork);
        if (ev_br_join) cudaEventDestroy(ev_br_join);
    }
};

}  // namespace b2d
struct b2d_handle : public b2d::Handle {};
namespace b2d {

// ------------------------------------------------------------------------------------------------ weight packing
static const HostTensor* find(Handle* h, const std::string& k) {
    auto it = h->sd.find(k);
    return it == h->sd.end() ? nullptr : &it->second;
}

#define NEED(var, key)                                             \
    const HostTensor* var = find(h, key);                          \
    if (!var) return fail(-3, std::string("missing tensor ") + (key));

static int upload_f32(Handle* h, const std::string& role, const std::vector<float>& v) {
    float* d;
    B2D_TRY(h->alloc(&d, v.size()));
    B2D_CUDA(cudaMemcpy(d, v.data(), v.size() * 4, cudaMemcpyHostToDevice));
    h->dev[role] = d;
    return 0;
}
static int upload_f16(Handle* h, const std::string& role, const std::vector<uint16_t>& v) {
    f16* d;
    B2D_TRY(h->alloc(&d, v.size()));
    B2D_CUDA(cudaMemcpy(d, v.data(), v.size() * 2, cudaMemcpyHostToDevice));
    h->dev[role] = d;
    return 0;
}

// Conv2d weight [Cout][Cin][R][S] (+ optional eval-BatchNorm folding) -> f16 [Cout][(r*S+s)*Cin+ci], fp32 bias.
// BN fold (SURVEY.md App. A): s = gamma/sqrt(running_var+1e-5); W' = W*s[co]; b' = beta - running_mean*s (+ conv bias*s).
static int pack_conv(Handle* h, const std::string& role, const std::string& wkey, const std::string& bias_key,
                     const std::string& bn_prefix) {
    NEED(w, wkey);
    if (w->shape.size() != 4) return fail(-3, wkey + ": expected 4-d weight");
    const int Cout = (int)w->shape[0], Cin = (int)w->shape[1], R = (int)w->shape[2], S = (int)w->shape[3];
    std::vector<float> scale(Cout, 1.0f), bias(Cout, 0.0f);
    if (!bias_key.empty()) {
        NEED(b, bias_key);
        for (int i = 0; i < Cout; ++i) bias[i] = b->v[i];
    }
    if (!bn_prefix.empty()) {
        NEED(g, bn_prefix + ".weight");
        NEED(be, bn_prefix + ".bias");
        NEED(mu, bn_prefix + ".running_mean");
        NEED(var, bn_prefix + ".running_var");
        for (int i = 0; i < Cout; ++i) {
            const float s = g->v[i] / std::sqrt(var->v[i] + 1e-5f);
            scale[i] = s;
            bias[i] = be->v[i] + (bias[i] - mu->v[i]) * s;
        }
    }
    std::vector<uint16_t> p((size_t)Cout * R * S * Cin);
    for (int co = 0; co < Cout; ++co)
        for (int ci = 0; ci < Cin; ++ci)
            for (int r = 0; r < R; ++r)
                for (int s = 0; s < S; ++s)
                    p[((size_t)co * R * S + (r * S + s)) * Cin + ci] =
                        f2h(w->v[(((size_t)co * Cin + ci) * R + r) * S + s] * scale[co]);
    B2D_TRY(upload_f16(h, role + ".w", p));
    B2D_TRY(upload_f32(h, role + ".b", bias));
    return 0;
}
// ConvTranspose2d weight [Cin][Cout][2][2] -> f16 [(a*2+b)*Cout+co][ci]; bias [Cout].
static int pack_convt(Handle* h, const std::string& role, const std::string& prefix) {
    NEED(w, prefix + ".weight");
    NEED(b, prefix + ".bias");
    const int Cin = (int)w->shape[0], Cout = (int)w->shape[1];
    if (w->shape[2] != 2 || w->shape[3] != 2) return fail(-3, prefix + ": ConvTranspose2d must be k=2");
    std::vector<uint16_t> p((size_t)4 * Cout * Cin);
    for (int ci = 0; ci < Cin; ++ci)
        for (int co = 0; co < Cout; ++co)
            for (int a = 0; a < 2; ++a)
                for (int bb = 0; bb < 2; ++bb)
                    p[((size_t)(a * 2 + bb) * Cout + co) * Cin + ci] = f2h(w->v[(((size_t)ci * Cout + co) * 2 + a) * 2 + bb]);
    B2D_TRY(upload_f16(h, role + ".w", p));
    B2D_TRY(upload_f32(h, role + ".b", b->v));
    return 0;
}
static int pack_linear(Handle* h, const std::string& role, const std::string& wkey, const std::string& bkey) {
    NEED(w, wkey);
    NEED(b, bkey);
    std::vector<uint16_t> p(w->numel());
    for (size_t i = 0; i < p.size(); ++i) p[i] = f2h(w->v[i]);
    B2D_TRY(upload_f16(h, role + ".w", p));
    B2D_TRY(upload_f32(h, role + ".b", b->v));
    return 0;
}
// LayerNorm folded into the following Linear: W' = W * gamma (fp16), c1[n] = sum_k W'[n][k] (of the ROUNDED weights, so the
// mean correction cancels exactly what the MMA accumulates), c2[n] = sum_k W[n][k] * beta[k] + b[n].
static int pack_ln_linear(Handle* h, const std::string& role, const std::string& wkey, const std::string& bkey,
                          const HostTensor* g, const HostTensor* be) {
    NEED(w, wkey);
    NEED(b, bkey);
    const int N = (int)w->shape[0], K = (int)w->shape[1];
    std::vector<uint16_t> p((size_t)N * K);
    std::vector<float> c1(N), c2(N);
    for (int n = 0; n < N; ++n) {
        double s1 = 0.0, s2 = 0.0;
        for (int k = 0; k < K; ++k) {
            const uint16_t hv = f2h(w->v[(size_t)n * K + k] * g->v[k]);
            p[(size_t)n * K + k] = hv;
            __half hh;
            memcpy(&hh, &hv, 2);
            s1 += (double)__half2float(hh);
            s2 += (double)w->v[(size_t)n * K + k] * (double)be->v[k];
        }
        c1[n] = (float)s1;
        c2[n] = (float)(s2 + (double)b->v[n]);
    }
    B2D_TRY(upload_f16(h, role + ".w", p));
    B2D_TRY(upload_f32(h, role + ".c1", c1));
    B2D_TRY(upload_f32(h, role + ".b", c2));
    return 0;
}

static int pack_attention(Handle* h, const std::string& role, const std::string& prefix, const char* ln, const char* mha,
                          const char* ffp = "ff_self") {
    NEED(g, prefix + "." + ln + ".weight");
    NEED(b, prefix + "." + ln + ".bias");
    B2D_TRY(upload_f32(h, role + ".ln.g", g->v));
    B2D_TRY(upload_f32(h, role + ".ln.b", b->v));
    B2D_TRY(pack_linear(h, role + ".qkv", prefix + "." + mha + ".in_proj_weight", prefix + "." + mha + ".in_proj_bias"));
    B2D_TRY(pack_ln_linear(h, role + ".qkvln", prefix + "." + mha + ".in_proj_weight", prefix + "." + mha + ".in_proj_bias", g, b));
    B2D_TRY(pack_linear(h, role + ".out", prefix + "." + mha + ".out_proj.weight", prefix + "." + mha + ".out_proj.bias"));
    if (h->cfg.attn_ff) {
        const std::string fp = prefix + "." + ffp;
        NEED(g2, fp + ".0.weight");
        NEED(b2, fp + ".0.bias");
        B2D_TRY(upload_f32(h, role + ".ffln.g", g2->v));
        B2D_TRY(upload_f32(h, role + ".ffln.b", b2->v));
        B2D_TRY(pack_linear(h, role + ".ff1", fp + ".1.weight", fp + ".1.bias"));
        if (g2->v.size() <= 128) B2D_TRY(pack_ln_linear(h, role + ".ff1ln", fp + ".1.weight", fp + ".1.bias", g2, b2));
        B2D_TRY(pack_linear(h, role + ".ff2", fp + ".3.weight", fp + ".3.bias"));
    }
    return 0;
}

static const int ENC_CH[5] = {64, 64, 128, 256, 512};
static const int DEC_IN[4] = {512, 256, 128, 64};
static const int DEC_OUT[4] = {256, 128, 64, 64};
static const int TEMB_ENC_OFF[5] = {0, 64, 128, 256, 512};
static const int TEMB_DEC_OFF[4] = {1024, 1280, 1408, 1472};
static const int TEMB_R_TOTAL = 1536;

static int pack_family_r(Handle* h) {
    const std::string E = "encoder.", D = "decoder.";
    {   // stem: fp32 [64][Cin_total][8][8]
        NEED(w, E + "conv1.weight");
        const int cin_total = h->cfg.c_hr + h->cfg.has_lsm + h->cfg.has_topo + h->cfg.cond_channels;
        if (w->shape[0] != 64 || w->shape[1] != cin_total || w->shape[2] != 8 || w->shape[3] != 8)
            return fail(-3, "encoder.conv1.weight shape does not match the configured input channels");
        // transpose to [Cin_total][64 taps][64 couts] so the stem kernel stages one channel's weights with 16-byte loads
        std::vector<float> wt((size_t)cin_total * 64 * 64);
        for (int co = 0; co < 64; ++co)
            for (int ci = 0; ci < cin_total; ++ci)
                for (int tap = 0; tap < 64; ++tap) wt[((size_t)ci * 64 + tap) * 64 + co] = w->v[((size_t)co * cin_total + ci) * 64 + tap];
        B2D_TRY(upload_f32(h, "stem.w", wt));
    }
    B2D_TRY(pack_conv(h, "conv2", E + "conv2.weight", "", E + "bn1"));
    for (int li = 1; li <= 4; ++li)
        for (int bi = 0; bi < 2; ++bi) {
            const std::string p = E + "layer" + std::to_string(li) + "." + std::to_string(bi) + ".";
            const std::string r = "l" + std::to_string(li) + "b" + std::to_string(bi);
            B2D_TRY(pack_conv(h, r + ".c1", p + "conv1.weight", "", p + "bn1"));
            B2D_TRY(pack_conv(h, r + ".c2", p + "conv2.weight", "", p + "bn2"));
            if (li > 1 && bi == 0) B2D_TRY(pack_conv(h, r + ".ds", p + "downsample.0.weight", "", p + "downsample.1"));
        }
    // time projections: one [1536][256] fp32 matrix (5 encoder + 4 decoder blocks), consumed by temb_project_kernel
    std::vector<float> W((size_t)TEMB_R_TOTAL * 256), Bv(TEMB_R_TOTAL);
    for (int i = 0; i < 5; ++i) {
        NEED(w, E + "time_projection_layers." + std::to_string(i) + ".1.weight");
        NEED(b, E + "time_projection_layers." + std::to_string(i) + ".1.bias");
        memcpy(&W[(size_t)TEMB_ENC_OFF[i] * 256], w->v.data(), w->v.size() * 4);
        memcpy(&Bv[TEMB_ENC_OFF[i]], b->v.data(), b->v.size() * 4);
    }
    for (int i = 0; i < 4; ++i) {
        NEED(w, D + "residual_layers." + std::to_string(i) + ".time_projection_layer.1.weight");
        NEED(b, D + "residual_layers." + std::to_string(i) + ".time_projection_layer.1.bias");
        memcpy(&W[(size_t)TEMB_DEC_OFF[i] * 256], w->v.data(), w->v.size() * 4);
        memcpy(&Bv[TEMB_DEC_OFF[i]], b->v.data(), b->v.size() * 4);
    }
    B2D_TRY(upload_f32(h, "temb.w", W));
    B2D_TRY(upload_f32(h, "temb.b", Bv));
    if (h->cfg.num_classes > 0) {
        NEED(le, E + "label_emb.weight");
        B2D_TRY(upload_f32(h, "label_emb", le->v));
    }
    // frequency tables (double pow, rounded once — within 1 ulp of torch's fp32 pow)
    std::vector<float> enc_inv(128), dec_div(128);
    for (int j = 0; j < 128; ++j) {
        enc_inv[j] = (float)(1.0 / (double)(float)std::pow(1000.0, (double)(float)((float)(2 * j) / 256.0f)));
        dec_div[j] = (float)std::pow(10000.0, (2.0 * j) / 256.0);
    }
    B2D_TRY(upload_f32(h, "enc_inv", enc_inv));
    B2D_TRY(upload_f32(h, "dec_div", dec_div));
    // two generations of ImageSelfAttention: modules_DANRA_conditional.py (keys attention.*, no FF) and
    // DDPM_clean_application/src/unet.py (keys mha.*, ff.{0,1,3}.*); told apart by the keys present
    const bool clean = find(h, E + "attention_layers.0.mha.in_proj_weight") != nullptr;
    if (clean != (h->cfg.attn_ff != 0)) return fail(-3, "attn_ff of the config does not match the attention keys of the state_dict");
    const char* mha = clean ? "mha" : "attention";
    for (int i = 0; i < 5; ++i)
        B2D_TRY(pack_attention(h, "ea" + std::to_string(i), E + "attention_layers." + std::to_string(i), "layernorm", mha, "ff"));
    for (int i = 0; i < 4; ++i) {
        const std::string p = D + "residual_layers." + std::to_string(i);
        B2D_TRY(pack_attention(h, "da" + std::to_string(i), p + ".attention", "layernorm", mha, "ff"));
        B2D_TRY(pack_convt(h, "d" + std::to_string(i) + ".up", p + ".transpose"));
        B2D_TRY(pack_conv(h, "d" + std::to_string(i) + ".conv", p + ".conv.weight", p + ".conv.bias", ""));
    }
    B2D_TRY(pack_convt(h, "final.up", D + "final_layer.transpose"));
    {
        NEED(w, D + "final_layer.conv.weight");
        NEED(b, D + "final_layer.conv.bias");
        if (w->shape[0] != h->cfg.c_out || w->shape[1] != 64) return fail(-3, "final_layer.conv.weight shape mismatch");
        B2D_TRY(upload_f32(h, "tail.w", w->v));
        B2D_TRY(upload_f32(h, "tail.b", b->v));
        // K-major copy for the tensor-core tail: [n][tap * 64 + c]
        std::vector<float> wk((size_t)h->cfg.c_out * 576);
        for (int n = 0; n < h->cfg.c_out; ++n)
            for (int c = 0; c < 64; ++c)
                for (int tap = 0; tap < 9; ++tap) wk[(size_t)n * 576 + tap * 64 + c] = w->v[((size_t)n * 64 + c) * 9 + tap];
        B2D_TRY(upload_f32(h, "tail.wk", wk));
    }
    return 0;
}

// ------------------------------------------------------------------------------------------------ program building
struct Builder {
    Handle* h;
    int B;
    int err = 0;
    OpList& ops;
    Builder(Handle* hh, int b, OpList& o) : h(hh), B(b), ops(o) {}

    f16* act(size_t elems) {
        f16* p = nullptr;
        if (h->alloc(&p, elems) != 0) err = -2;
        return p;
    }
    template <typename T>
    T* W(const std::string& role) {
        auto it = h->dev.find(role);
        if (it == h->dev.end()) {
            err = fail(-3, "internal: missing packed weight " + role);
            return nullptr;
        }
        return reinterpret_cast<T*>(it->second);
    }

    // GEMM-shaped op through the tcgen05 kernel (or the SIMT cross-check when cfg.debug_simt_conv)
    const float* next_ln_c1 = nullptr;   // set right before conv(): fold a LayerNorm into this GEMM (stream path only)
    bool want_gn_partial = false;        // set right before conv(): emit per-tile GroupNorm partial sums if the plan allows
    const float* last_gn_partial = nullptr;   // result of that request, consumed by BuilderD::gn()
    int last_gn_tps = 0, last_gn_ntiles = 0, last_gn_mtiles = 0;
    void conv(const f16* in, int Hi, int Wi, int Cin, f16* out, int Cout, int R, int stride, int pad, bool convt,
              const std::string& role, const f16* residual, const float* post_add, int post_stride, int act) {
        auto pl = std::make_shared<ConvPlan>();
        ConvParams& p = pl->p;
        memset(&p, 0, sizeof(p));
        p.B = B; p.Hi = Hi; p.Wi = Wi; p.Cin = Cin;
        p.R = R; p.S = R; p.stride = stride; p.pad = pad;
        p.convt = convt ? 1 : 0;
        if (convt) {
            p.Ho = Hi; p.Wo = Wi; p.Cout = 4 * Cout; p.CoutT = Cout;
        } else {
            p.Ho = (Hi + 2 * pad - R) / stride + 1;
            p.Wo = (Wi + 2 * pad - R) / stride + 1;
            p.Cout = Cout; p.CoutT = Cout;
        }
        p.in = in;
        p.w = W<f16>(role + ".w");
        p.bias = W<float>(role + ".b");
        p.residual = residual;
        p.post_add = post_add;
        p.post_stride = post_stride;
        p.act = act;
        p.out = out;
        p.ln_c1 = next_ln_c1;
        next_ln_c1 = nullptr;
        const bool want_gn = want_gn_partial;
        want_gn_partial = false;
        last_gn_partial = nullptr;
        if (err) return;
        if (p.ln_c1 && (h->cfg.debug_simt_conv || !gemm_stream_supported(p))) {
            err = fail(-1, "internal: LayerNorm-folded GEMM requested for a shape the streaming GEMM does not take");
            return;
        }
        {
            const double M = (double)B * p.Ho * p.Wo, Nn = p.Cout, K = (double)R * R * Cin;
            ops.meta(role, h->cfg.debug_simt_conv ? "conv_simt" : "conv_tc", 2.0 * M * Nn * K,
                     2.0 * ((double)B * Hi * Wi * Cin + M * Nn * (residual ? 2 : 1) + Nn * K));
        }
        static const bool no_stream = getenv("B2D_NO_STREAM_GEMM") != nullptr;
        if (h->cfg.debug_simt_conv) {
            ops.push_back([pl](cudaStream_t st) { return conv_launch_simt(pl->p, st); });
        } else if (!no_stream && gemm_stream_supported(p)) {
            auto gp = std::make_shared<GemmStreamPlan>();
            gp->p = p;
            if (gemm_stream_plan_build(*gp, h->num_sms) != 0) { err = -1; return; }
            ops.pending.klass = "gemm_stream";
            ops.push_back([gp](cudaStream_t st) { return gemm_stream_launch(*gp, st); });
        } else {
            if (conv_plan_build(*pl, h->num_sms) != 0) { err = -1; return; }
            static const bool no_gn_epi = getenv("B2D_NO_GN_EPILOGUE") != nullptr;
            const int hw_out = pl->p.Ho * pl->p.Wo;
            const bool gn_whole = pl->p.TN == 1;                                   // a tile lies inside one sample
            const bool gn_quarter = pl->p.TN > 1 && hw_out % 32 == 0;              // several samples per tile, 32-row quarters do not straddle
            if (want_gn && !no_gn_epi && pl->p.splits == 1 && (gn_whole || gn_quarter) && !convt) {
                const int sub = gn_whole ? 1 : 4;
                const int mtiles = (int)pl->grid.x * sub, ntiles = (int)pl->grid.y;
                float* part = nullptr;
                if (h->alloc(&part, (size_t)mtiles * ntiles * 2) != 0) { err = -2; return; }
                pl->p.gn_partial = part;
                pl->p.gn_sub = sub;
                last_gn_partial = part;
                last_gn_tps = gn_whole ? pl->p.tiles_w * pl->p.tiles_h : hw_out / 32;
                last_gn_ntiles = ntiles;
                last_gn_mtiles = mtiles;
            }
            if (pl->ws_floats) {
                if (h->alloc(&pl->p.ws, pl->ws_floats) != 0) { err = -2; return; }
            }
            if (conv_tcp_eligible(*pl, h->num_sms)) {      // large layers: persistent two-accumulator kernel (conv_persist.cuh)
                const int sms = h->num_sms;
                ops.pending.klass = "conv_tc";
                ops.push_back([pl, sms](cudaStream_t st) { return conv_launch_tcp(*pl, sms, st); });
            } else {
                ops.push_back([pl](cudaStream_t st) { return conv_launch_tc(*pl, st); });
            }
        }
    }

    // scratch shared by all attention blocks (they run one after another)
    f16 *s_xn = nullptr, *s_qkv = nullptr, *s_ao = nullptr, *s_h1 = nullptr, *s_mid = nullptr;

    // ImageSelfAttention (+ optional FF tail) on tokens x [B, hw*hw, C]; final_act applies to the block output.
    void attention(const f16* x, int hw, int C, const std::string& role, f16* out, int final_act) {
        const int rows = B * hw * hw, L = hw * hw, heads = h->cfg.n_heads;
        const float* g = W<float>(role + ".ln.g");
        const float* b = W<float>(role + ".ln.b");
        f16 *xn = s_xn, *qkv = s_qkv, *ao = s_ao;
        const int Bc = B;
        // LayerNorm folded into the QKV / FF1 GEMM whenever that GEMM runs on the streaming kernel (C <= 128, enough rows)
        static const bool no_ln_fold = getenv("B2D_NO_LN_FOLD") != nullptr;
        const bool fold = !no_ln_fold && !h->cfg.debug_simt_conv && !getenv("B2D_NO_STREAM_GEMM") && C <= 128 && rows >= GS_MIN_ROWS;
        // low-resolution levels (L <= 64 tokens): LayerNorm + QKV + attention in ONE launch
        static const bool no_attn_block = getenv("B2D_NO_ATTN_BLOCK") != nullptr;
        const bool fused_block = !no_attn_block && !h->cfg.debug_simt_conv && attn_block_supported(L, C, heads);
        bool fused_out = false;
        if (fused_block) {
            auto pl = std::make_shared<AttnBlockPlan>();
            if (attn_block_plan_build(*pl, x, W<f16>(role + ".qkvln.w"), W<float>(role + ".qkvln.c1"), W<float>(role + ".qkvln.b"), ao,
                                      rows, C, L, heads) != 0) { err = -1; return; }
            static const bool no_out_fuse = getenv("B2D_NO_ATTN_OUT_FUSE") != nullptr;
            static const int out_fuse_maxc = getenv("B2D_ATTN_OUT_FUSE_MAXC") ? atoi(getenv("B2D_ATTN_OUT_FUSE_MAXC")) : 128;
            // gather mode (fp16 head outputs exchanged through DSMEM, out-projection for every C inside the block): measured 1 %
            // SLOWER per step than the separate conv_tc out-projection (the block only has heads x tiles CTAs) -> opt-in
            static const bool want_gather = getenv("B2D_ATTN_GATHER") != nullptr;
            const bool gather = !no_out_fuse && want_gather && attn_block_gather_supported(C, heads);
            fused_out = gather || (!no_out_fuse && attn_block_out_supported(C, heads) && C <= out_fuse_maxc);
            double fl = 6.0 * rows * C * C + 4.0 * (double)L * L * C * B, by = 4.0 * rows * C + 6.0 * C * C;
            if (fused_out) {   // + out-projection, bias, residual (and the decoder's ReLU): the whole block is one launch
                float* ws = nullptr;
                if (!gather && h->alloc(&ws, attn_block_ws_floats(rows, C, heads)) != 0) { err = -2; return; }
                if (attn_block_plan_fuse_out(*pl, W<f16>(role + ".out.w"), W<float>(role + ".out.b"), x,
                                             h->cfg.attn_ff ? s_mid : out, ws, h->cfg.attn_ff ? 0 : final_act, gather ? 2 : 1) != 0) { err = -1; return; }
                fl += 2.0 * rows * C * C;
                by += 4.0 * rows * C + 2.0 * C * C;
            }
            ops.meta(role + ".attn", "attn_block", fl, by);
            ops.push_back([=](cudaStream_t st) { return attn_block_launch(*pl, st); });
        } else if (fold) {
            next_ln_c1 = W<float>(role + ".qkvln.c1");
            conv(x, hw, hw, C, qkv, 3 * C, 1, 1, 0, false, role + ".qkvln", nullptr, nullptr, 0, 0);
        } else {
            ops.meta(role + ".ln", "layernorm", 0, 4.0 * rows * C);
            ops.push_back([=](cudaStream_t st) { return layernorm_launch(x, g, b, xn, rows, C, st); });
            conv(xn, hw, hw, C, qkv, 3 * C, 1, 1, 0, false, role + ".qkv", nullptr, nullptr, 0, 0);
        }
        static const bool no_tc_attn = getenv("B2D_NO_TC_ATTN") != nullptr;
        if (fused_block) {
            // attention output already in `ao`
        } else if (attn_tc_supported(L, C, heads) && !no_tc_attn) {
            auto tmq = std::make_shared<AttnTcMaps>();
            if (attn_tc_make_map(tmq.get(), qkv, B, L, C) != 0) { err = -1; return; }
            ops.meta(role + ".sdpa", "attn_tc", 4.0 * (double)L * L * C * B, 8.0 * rows * C);
            // B2D_ATTN_V=1: round-1 kernel (3 CTAs/SM); 2: persistent two-tile kernel; 3: four CTAs per SM, optimistic maximum; 4: 32-key
            // blocks; 6 / 7: self-issuing / named-barrier-issuer variants; default 8: attention_tc8.cuh — A/B switches, all parity-tested
            static const int attn_v = getenv("B2D_ATTN_V") ? atoi(getenv("B2D_ATTN_V")) : 8;
            const int sms = h->num_sms;
            if (attn_v == 2 && attn_tc2_supported(L, C, heads))
                ops.push_back([=](cudaStream_t st) { return attn_tc2_launch(*tmq, ao, Bc, L, C, heads, sms, st); });
            else if (attn_v == 1)
                ops.push_back([=](cudaStream_t st) { return attn_tc_launch(*tmq, ao, Bc, L, C, heads, st); });
            else if (attn_v == 4) {
                auto tm4 = std::make_shared<AttnTcMaps>();
                if (attn_tc4_make_map(tm4.get(), qkv, B, L, C) != 0) { err = -1; return; }
                ops.push_back([=](cudaStream_t st) { return attn_tc4_launch(*tm4, ao, Bc, L, C, heads, st); });
            } else if (attn_v == 6)
                ops.push_back([=](cudaStream_t st) { return attn_tc6_launch<0>(*tmq, ao, Bc, L, C, heads, st); });
            else if (attn_v == 7)
                ops.push_back([=](cudaStream_t st) { return attn_tc6_launch<1>(*tmq, ao, Bc, L, C, heads, st); });
            else if (attn_v == 8)
                ops.push_back([=](cudaStream_t st) { return attn_tc8_launch(*tmq, ao, Bc, L, C, heads, st); });
            else
                ops.push_back([=](cudaStream_t st) { return attn_tc3_launch(*tmq, ao, Bc, L, C, heads, st); });
        } else if (attn_tc5_supported(L, C, heads) && !no_tc_attn) {     // head_dim 32 on tcgen05 (attention_tc3d32.cuh)
            auto tm5 = std::make_shared<AttnTcMaps>();
            if (attn_tc5_make_map(tm5.get(), qkv, B, L, C) != 0) { err = -1; return; }
            ops.meta(role + ".sdpa", "attn_tc32", 4.0 * (double)L * L * C * B, 8.0 * rows * C);
            ops.push_back([=](cudaStream_t st) { return attn_tc5_launch(*tm5, ao, Bc, L, C, heads, st); });
        } else {
            ops.meta(role + ".sdpa", "flash_attn", 4.0 * (double)L * L * C * B, 8.0 * rows * C);
            ops.push_back([=](cudaStream_t st) { return flash_attn_launch(qkv, ao, Bc, L, C, heads, st); });
        }
        if (!h->cfg.attn_ff) {
            if (!fused_out) conv(ao, hw, hw, C, out, C, 1, 1, 0, false, role + ".out", x, nullptr, 0, final_act);
        } else {
            f16* mid = s_mid;
            f16* h1 = s_h1;
            if (!fused_out) conv(ao, hw, hw, C, mid, C, 1, 1, 0, false, role + ".out", x, nullptr, 0, 0);
            const float* g2 = W<float>(role + ".ffln.g");
            const float* b2 = W<float>(role + ".ffln.b");
            if (fold) {
                next_ln_c1 = W<float>(role + ".ff1ln.c1");
                conv(mid, hw, hw, C, h1, C, 1, 1, 0, false, role + ".ff1ln", nullptr, nullptr, 0, 2);
            } else {
                ops.meta(role + ".ffln", "layernorm", 0, 4.0 * rows * C);
                ops.push_back([=](cudaStream_t st) { return layernorm_launch(mid, g2, b2, xn, rows, C, st); });
                conv(xn, hw, hw, C, h1, C, 1, 1, 0, false, role + ".ff1", nullptr, nullptr, 0, 2);
            }
            conv(h1, hw, hw, C, out, C, 1, 1, 0, false, role + ".ff2", mid, nullptr, 0, final_act);
        }
    }

    float* stats_slice(int C) {
        float* p = h->d_stats + h->stats_floats;
        h->stats_floats += (size_t)B * C * 2;
        return p;
    }
    void plane_stats(const f16* x, int hw, int C, float* st) {
        const int HW = hw * hw, Bc = B;
        const int ppc = 256;  // pixels per CTA
        const int nslab = (HW + ppc - 1) / ppc, ngrp = C / 64;
        float* partial = nullptr;
        unsigned int* counters = nullptr;
        if (h->alloc(&partial, (size_t)B * ngrp * nslab * 128) != 0 || h->alloc(&counters, (size_t)B * ngrp) != 0) {
            err = -2;
            return;
        }
        if (cudaMemset(counters, 0, (size_t)B * ngrp * sizeof(unsigned int)) != cudaSuccess) err = -2;
        ops.meta("in_stats", "plane_stats", 0, 2.0 * B * HW * C);
        ops.push_back([=](cudaStream_t s) {
            dim3 grid(nslab, ngrp, Bc);
            B2D_CUDA(launch_k(plane_stats_kernel, dim3(grid), dim3(256), 0, s, x, partial, counters, st, HW, C, ppc));
            B2D_CUDA(cudaGetLastError());
            return 0;
        });
    }
    // InstanceNorm (+skip +vec) in ONE launch when the (sample, 64-channel) slab fits a cluster's shared memory
    bool instnorm_fused(const f16* x, const f16* skip, const float* vec, int vec_stride, f16* y, int hw, int C) {
        static const bool off = getenv("B2D_NO_FUSED_NORM") != nullptr;
        const int HW = hw * hw;
        if (off || norm_fused_cluster(HW) == 0) return false;
        NormParams np{};
        np.x = x; np.y = y; np.add = skip; np.vec = vec; np.vec_stride = vec_stride; np.C = C; np.rows = HW;
        np.slab_stride = (long long)HW * C;
        const int Bc = B, groups = C / 64;
        ops.meta("in_fused", "norm_fused", 0, 2.0 * B * HW * C * (skip ? 3 : 2));
        ops.push_back([=](cudaStream_t s) { return norm_fused_launch<0>(np, Bc, groups, s); });
        return true;
    }
    void instnorm_apply(const f16* x, const float* st, const f16* skip, const float* vec, int vec_stride, f16* y, int hw,
                        int C) {
        const int HW = hw * hw;
        const size_t total8 = (size_t)B * HW * C / 8;
        ops.meta("in_apply", "instnorm_apply", 0, 2.0 * B * HW * C * (skip ? 3 : 2));
        ops.push_back([=](cudaStream_t s) {
            int blocks = (int)std::min<size_t>((total8 + 255) / 256, (size_t)148 * 16);
            B2D_CUDA(launch_k(instnorm_apply_kernel, dim3(blocks), dim3(256), 0, s, x, st, skip, vec, vec_stride, y, HW, C, total8));
            B2D_CUDA(cudaGetLastError());
            return 0;
        });
    }
};

}  // namespace b2d
#include "family_d.cuh"
namespace b2d {

static const size_t STATS_CAPACITY_PER_SAMPLE = 2 * (512 + 256 + 256 + 128 + 128 + 64 + 64 + 64 + 64) + 4096;

static int build_program_r(Handle* h, int B) {
    const b2d_config& c = h->cfg;
    const int H = c.img_size;
    const int s[6] = {H, H / 2, H / 4, H / 8, H / 16, H / 32};
    OpList ops;
    Builder bd(h, B, ops);
    h->stats_floats = 0;
    // scratch for attention (largest layer: fmap1 / dec3, rows = B*s1^2, C = 64; deeper layers are never larger)
    size_t max_rc = 0;
    for (int i = 0; i < 5; ++i) max_rc = std::max(max_rc, (size_t)B * s[i + 1] * s[i + 1] * ENC_CH[i]);
    bd.s_xn = bd.act(max_rc);
    bd.s_qkv = bd.act(max_rc * 3);
    bd.s_ao = bd.act(max_rc);
    if (c.attn_ff) {
        bd.s_h1 = bd.act(max_rc);
        bd.s_mid = bd.act(max_rc);
    }
    float* temb = h->d_temb;
    const int TS = TEMB_R_TOTAL;

    // ---- time embeddings + all nine projections (one launch)
    {
        Handle* hh = h;
        const float* label = c.num_classes > 0 ? bd.W<float>("label_emb") : nullptr;
        const float* ei = bd.W<float>("enc_inv");
        const float* dd = bd.W<float>("dec_div");
        const float* tw = bd.W<float>("temb.w");
        const float* tb = bd.W<float>("temb.b");
        ops.meta("temb", "temb_project", 2.0 * B * TS * 256, 4.0 * TS * 256);
        ops.push_back([=](cudaStream_t st) {
            dim3 grid((TS + TEMB_OC - 1) / TEMB_OC, (B + TEMB_SB - 1) / TEMB_SB);
            B2D_CUDA(launch_k(temb_project_kernel, dim3(grid), dim3(256), 0, st, hh->temb_t, hh->has_y ? hh->d_y : nullptr, label, ei, dd, tw, tb, temb, 1024,
                                                      TS, B, hh->temb_t_off, hh->cfg.stem_embedding));
            B2D_CUDA(cudaGetLastError());
            return 0;
        });
    }
    // ---- Encoder.forward (modules_DANRA_conditional.py:213-312)
    f16* f1_pre = bd.act((size_t)B * s[1] * s[1] * 64);
    {
        Handle* hh = h;
        const float* sw = bd.W<float>("stem.w");
        const int cin_total = c.c_hr + c.has_lsm + c.has_topo + c.cond_channels;
        const int chr = c.c_hr, Hh = H, ho = s[1];
        ops.meta("conv1", "stem_conv", 2.0 * B * ho * ho * 64 * 64 * chr,
                 (double)B * (4.0 * chr * Hh * Hh + ho * ho * 64 * (2 + 4)));
        ops.push_back([=](cudaStream_t st) {
            const bool have_cond = (cin_total > chr);
            const float* addp = have_cond ? hh->d_cond_pre : nullptr;
            if (ho % 16 == 0) {   // tensor-core stem (hi/lo split operands, fp32-equivalent)
                dim3 grid(ho / 16, ho / 16, B);
                B2D_CUDA(launch_k(stem_mma_kernel, dim3(grid), dim3(256), STEM_MMA_SMEM, st, hh->cur_x, chr, Hh, Hh, sw, addp,
                                  temb + TEMB_ENC_OFF[0], TS, f1_pre, ho, ho));
            } else {
                dim3 grid((ho + 15) / 16, (ho + 15) / 16, B);
                B2D_CUDA(launch_k(stem_conv_kernel<8, 2>, dim3(grid), dim3(256), 0, st, hh->cur_x, chr, Hh, Hh, sw, cin_total, 0, addp,
                                  temb + TEMB_ENC_OFF[0], TS, f1_pre, nullptr, ho, ho, 3));
            }
            B2D_CUDA(cudaGetLastError());
            return 0;
        });
    }
    f16* fmap[5];
    fmap[0] = bd.act((size_t)B * s[1] * s[1] * 64);
    bd.attention(f1_pre, s[1], 64, "ea0", fmap[0], 0);
    h->taps["f1_pre"] = {f1_pre, 64, s[1]};
    h->taps["fmap1"] = {fmap[0], 64, s[1]};
    // conv2 -> bn1 -> relu (:269-273)
    f16* cur = bd.act((size_t)B * s[2] * s[2] * 64);
    bd.conv(fmap[0], s[1], s[1], 64, cur, 64, 8, 2, 3, false, "conv2", nullptr, nullptr, 0, 1);
    int cin = 64;
    for (int li = 1; li <= 4; ++li) {
        const int cout = ENC_CH[li];
        const int hin = (li == 1) ? s[2] : s[li];  // input extent of this layer
        const int hout = s[li + 1];
        const size_t n_out = (size_t)B * hout * hout * cout;
        const std::string r0 = "l" + std::to_string(li) + "b0", r1 = "l" + std::to_string(li) + "b1";
        f16* t1 = bd.act(n_out);
        f16* b0 = bd.act(n_out);
        f16* pre = bd.act(n_out);
        const f16* identity = cur;
        const int stride = (li > 1) ? 2 : 1;
        if (li > 1) {   // the 1x1/s2 downsample only depends on the block input: a side branch next to c1
            f16* ds = bd.act(n_out);
            ops.pending.side = true;
            bd.conv(cur, hin, hin, cin, ds, cout, 1, 2, 0, false, r0 + ".ds", nullptr, nullptr, 0, 0);
            identity = ds;
        }
        bd.conv(cur, hin, hin, cin, t1, cout, 3, stride, 1, false, r0 + ".c1", nullptr, nullptr, 0, 1);
        ops.pending.join = (li > 1);
        bd.conv(t1, hout, hout, cout, b0, cout, 3, 1, 1, false, r0 + ".c2", identity, nullptr, 0, 1);
        bd.conv(b0, hout, hout, cout, t1, cout, 3, 1, 1, false, r1 + ".c1", nullptr, nullptr, 0, 1);
        // last conv of the stage: + identity, ReLU, then + time projection (fmap = layer(x) + t_emb, :276-280)
        bd.conv(t1, hout, hout, cout, pre, cout, 3, 1, 1, false, r1 + ".c2", b0, temb + TEMB_ENC_OFF[li], TS, 1);
        fmap[li] = bd.act(n_out);
        bd.attention(pre, hout, cout, "ea" + std::to_string(li), fmap[li], 0);
        h->taps["pre" + std::to_string(li + 1)] = {pre, cout, hout};
        h->taps["fmap" + std::to_string(li + 1)] = {fmap[li], cout, hout};
        cur = fmap[li];
        cin = cout;
    }
    // ---- Decoder.forward (:512-536), DecoderBlock.forward (:425-460)
    h->dec_begin_op = (int)ops.v.size();
    for (int i = 0; i < 5; ++i) h->fmaps[i] = {fmap[i], ENC_CH[i], s[i + 1]};
    const f16* dcur = fmap[4];
    for (int i = 0; i < 4; ++i) {
        const int ci = DEC_IN[i], co = DEC_OUT[i];
        const int hin = s[5 - i], hout = s[4 - i];
        const std::string r = "d" + std::to_string(i);
        f16* up = bd.act((size_t)B * hout * hout * ci);
        bd.conv(dcur, hin, hin, ci, up, ci, 1, 1, 0, true, r + ".up", nullptr, nullptr, 0, 0);
        if (!bd.instnorm_fused(up, nullptr, nullptr, 0, up, hout, ci)) {
            float* st1 = bd.stats_slice(ci);
            bd.plane_stats(up, hout, ci, st1);
            bd.instnorm_apply(up, st1, nullptr, nullptr, 0, up, hout, ci);
        }
        f16* cv = bd.act((size_t)B * hout * hout * co);
        bd.conv(up, hout, hout, ci, cv, co, 3, 1, 1, false, r + ".conv", nullptr, nullptr, 0, 0);
        f16* pre = bd.act((size_t)B * hout * hout * co);
        if (!bd.instnorm_fused(cv, fmap[3 - i], temb + TEMB_DEC_OFF[i], TS, pre, hout, co)) {
            float* st2 = bd.stats_slice(co);
            bd.plane_stats(cv, hout, co, st2);
            bd.instnorm_apply(cv, st2, fmap[3 - i], temb + TEMB_DEC_OFF[i], TS, pre, hout, co);
        }
        f16* dout = bd.act((size_t)B * hout * hout * co);
        bd.attention(pre, hout, co, "da" + std::to_string(i), dout, 1 /*ReLU after attention, :459*/);
        h->taps["dec" + std::to_string(i) + "_pre"] = {pre, co, hout};
        h->taps["dec" + std::to_string(i)] = {dout, co, hout};
        dcur = dout;
    }
    h->temb_free_op = (int)ops.v.size();   // nothing below reads d_temb
    // ---- final_layer: ConvT -> IN -> Conv3x3(64->c_out), no skip/time/attention/activation (:503-509, :535)
    {
        f16* up = bd.act((size_t)B * H * H * 64);
        bd.conv(dcur, s[1], s[1], 64, up, 64, 1, 1, 0, true, "final.up", nullptr, nullptr, 0, 0);
        float* st = bd.stats_slice(64);
        bd.plane_stats(up, H, 64, st);
        Handle* hh = h;
        const float* tw = bd.W<float>("tail.w");
        const float* tb = bd.W<float>("tail.b");
        const float* twk = bd.W<float>("tail.wk");
        const int cout = c.c_out, Hh = H;
        ops.meta("final.conv", "tail_conv", 2.0 * B * Hh * Hh * 576 * cout, (double)B * Hh * Hh * (64 * 2 + 4 * cout));
        static const bool no_tc_tail = getenv("B2D_NO_TC_TAIL") != nullptr;
        auto ttp = std::make_shared<TailTcPlan>();
        const bool tc_tail = tail_tc_supported(Hh, Hh, cout) && !no_tc_tail;
        if (tc_tail && tail_tc_plan_build(*ttp, up, B, Hh, Hh) != 0) return g_status.code ? g_status.code : fail(-1, "tail plan failed");
        ops.push_back([=](cudaStream_t s2) {
            dim3 grid((Hh + 31) / 32, (Hh + 7) / 8, B);
            static const bool simt_tail = getenv("B2D_SIMT_TAIL") != nullptr;
            if (tc_tail)
                return tail_tc_launch(*ttp, st, twk, tb, hh->cur_eps, Hh, Hh, s2);
            if (cout <= 8 && !simt_tail)
                B2D_CUDA(launch_k(tail_mma_kernel, dim3(grid), dim3(256), TAILM_SMEM, s2, up, st, twk, tb, hh->cur_eps, Hh, Hh, cout));
            else
                B2D_CUDA(launch_k(tail_conv_kernel, dim3(grid), dim3(256), TAIL_SMEM, s2, up, st, tw, tb, hh->cur_eps, Hh, Hh, cout));
            B2D_CUDA(cudaGetLastError());
            return 0;
        });
    }
    if (bd.err) return g_status.code ? g_status.code : fail(-1, "program build failed");
    if (h->stats_floats > STATS_CAPACITY_PER_SAMPLE * (size_t)c.max_batch) return fail(-1, "internal: stats buffer too small");
    h->step_ops.swap(ops.v);
    h->prog_B = B;
    return 0;
}

// Every kernel of the step asks for the same (maximum) shared-memory carve-out: consecutive kernels with different
// L1/shared splits force the SMs to drain and reconfigure between launches, which costs microseconds per launch.
template <typename K>
static int set_carveout(K kern) {
    B2D_CUDA(cudaFuncSetAttribute(kern, cudaFuncAttributePreferredSharedMemoryCarveout, cudaSharedmemCarveoutMaxShared));
    return 0;
}
static int init_uniform_carveout() {
    static bool done = false;
    if (done || getenv("B2D_NO_CARVEOUT")) return 0;
    B2D_TRY(set_carveout(conv_tc_kernel<64, 4>));
    B2D_TRY(set_carveout(conv_tc_kernel<64, 8>));
    B2D_TRY(set_carveout(conv_tc_kernel<128, 3>));
    B2D_TRY(set_carveout(conv_tc_kernel<128, 6>));
    B2D_TRY(set_carveout(conv_simt_kernel));
    B2D_TRY(set_carveout(layernorm_rows_kernel<64>));
    B2D_TRY(set_carveout(layernorm_rows_kernel<128>));
    B2D_TRY(set_carveout(layernorm_rows_kernel<256>));
    B2D_TRY(set_carveout(layernorm_rows_kernel<512>));
    B2D_TRY(set_carveout(flash_attn_kernel<16>));
    B2D_TRY(set_carveout(flash_attn_kernel<32>));
    B2D_TRY(set_carveout(flash_attn_kernel<64>));
    B2D_TRY(set_carveout(flash_attn_kernel<128>));
    B2D_TRY(set_carveout(attn_small_d_kernel<2>));
    B2D_TRY(set_carveout(attn_small_d_kernel<4>));
    B2D_TRY(set_carveout(attn_small_d_kernel<8>));
    B2D_TRY(set_carveout(attn_tc_kernel));
    B2D_TRY(set_carveout(attn_tc2_kernel<0>));
    B2D_TRY(set_carveout(attn_tc2_kernel<1>));
    B2D_TRY(set_carveout(attn_tc2_kernel<2>));
    B2D_TRY(set_carveout(attn_tc2_kernel<3>));
    B2D_TRY(set_carveout(attn_tc2_kernel<4>));
    B2D_TRY(set_carveout(temb_project_kernel));
    B2D_TRY(set_carveout(stem_conv_kernel<8, 2>));
    B2D_CUDA(cudaFuncSetAttribute(stem_mma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, STEM_MMA_SMEM));
    B2D_CUDA(cudaFuncSetAttribute(tail_mma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TAILM_SMEM));
    B2D_TRY(set_carveout(stem_conv_kernel<3, 1>));
    B2D_TRY(set_carveout(plane_stats_kernel));
    B2D_TRY(set_carveout(instnorm_apply_kernel));
    B2D_TRY(set_carveout(tail_conv_kernel));
    B2D_TRY(set_carveout(posterior_update_kernel));
    B2D_TRY(set_carveout(ddim_update_kernel));
    B2D_TRY(set_carveout(fill_int_kernel));
    B2D_TRY(set_carveout(bicubic_resize_kernel));
    B2D_TRY(set_carveout(linear_nearest_resize_kernel));
    B2D_TRY(set_carveout(sample_stats_kernel));
    B2D_TRY(set_carveout(groupnorm_apply_kernel));
    B2D_TRY(set_carveout(maxpool2_kernel));
    B2D_TRY(set_carveout(upsample_cat_kernel));
    B2D_TRY(set_carveout(outc_kernel));
    B2D_TRY(set_carveout(norm_fused_kernel<0>));
    B2D_TRY(set_carveout(norm_fused_kernel<1>));
    B2D_TRY(set_carveout(gemm_stream_kernel<1>));
    B2D_TRY(set_carveout(gemm_stream_kernel<2>));
    done = true;
    return 0;
}

// Per-batch device buffers of a handle (parent or kid).
static int init_batch_buffers(Handle* h) {
    const b2d_config& c = h->cfg;
    const int B = c.max_batch, H = c.img_size;
    B2D_TRY(h->alloc(&h->d_t, B));
    B2D_TRY(h->alloc(&h->d_t_next, B));
    h->temb_t = h->d_t;
    B2D_TRY(h->alloc(&h->d_y, B));
    B2D_TRY(h->alloc(&h->d_step, 4));   // [0] step index i, [1] arrival counter of the posterior update (self-resetting)
    B2D_CUDA(cudaMemset(h->d_step, 0, 16));
    B2D_TRY(h->alloc(&h->d_eps, (size_t)B * c.c_out * H * H));
    B2D_TRY(h->alloc(&h->d_stats, STATS_CAPACITY_PER_SAMPLE * (size_t)B));
    h->n_temb = TEMB_R_TOTAL;
    B2D_TRY(h->alloc(&h->d_temb, (size_t)B * 2048));
    const int ccond = c.has_lsm + c.has_topo + c.cond_channels;
    B2D_TRY(h->alloc(&h->d_cond_stack, (size_t)B * std::max(ccond, 1) * H * H));
    const size_t pre_px = (c.family == B2D_FAMILY_D) ? (size_t)H * H : (size_t)(H / 2) * (H / 2);
    B2D_TRY(h->alloc(&h->d_cond_pre, (size_t)B * pre_px * 64));
    if (cudaStreamCreateWithFlags(&h->own_stream, cudaStreamNonBlocking) != cudaSuccess) return fail(-2, "stream create failed");
    return 0;
}

static int ensure_program(Handle* h, int B) {
    B2D_CHECK(h->weights_loaded, "b2d_load_weights has not been called");
    B2D_CHECK(B >= 1 && B <= h->cfg.max_batch, "batch exceeds max_batch of the handle");
    if (h->prog_B == B) return 0;
    h->drop_graphs();
    h->free_program();
    h->in_prog = true;
    const int rc = (h->cfg.family == B2D_FAMILY_R) ? build_program_r(h, B) : build_program_d(h, B);
    h->in_prog = false;
    if (rc) h->free_program();
    return rc;
}

// pipelined = inside the reverse loop: op 0 (time embeddings) of this step was produced by the previous step's side branch
// (or by the loop prologue), and the embeddings of the NEXT step are launched on the side stream at temb_free_op.  The
// caller joins the side branch (join_temb_side) before it advances the step counter.  The side branch runs before the update
// that advances t, so it cannot read the next t from d_t: the DDPM loop embeds d_t - 1, the DDIM loop (ddim = true) embeds
// d_t_next, which holds tau_{k+1} (a stride of more than one step).
static int run_step_ops(Handle* h, cudaStream_t st, bool pipelined = false, int first = 0, int last = -1, bool ddim = false) {
    static const bool dbg = getenv("B2D_DEBUG_SYNC") != nullptr;
    static const bool no_pipe = getenv("B2D_NO_TEMB_PIPE") != nullptr;
    static const bool no_branch = getenv("B2D_NO_BRANCH") != nullptr;
    const bool pipe = pipelined && !no_pipe && h->temb_free_op > 0;
    if (!h->side_stream) {
        B2D_CUDA(cudaStreamCreateWithFlags(&h->side_stream, cudaStreamNonBlocking));
        B2D_CUDA(cudaEventCreateWithFlags(&h->ev_side_fork, cudaEventDisableTiming));
        B2D_CUDA(cudaEventCreateWithFlags(&h->ev_side_join, cudaEventDisableTiming));
        B2D_CUDA(cudaEventCreateWithFlags(&h->ev_br_fork, cudaEventDisableTiming));
        B2D_CUDA(cudaEventCreateWithFlags(&h->ev_br_join, cudaEventDisableTiming));
    }
    int idx = 0;
    bool branch_open = false;
    if (last < 0) last = (int)h->step_ops.size();
    for (auto& op : h->step_ops) {
        if (idx < first || idx >= last) { ++idx; continue; }     // partial programs (stand-alone Encoder / Decoder)
        if (pipe && idx == 0) { ++idx; continue; }
        if (op.side && !no_branch && !dbg) {
            B2D_CUDA(cudaEventRecord(h->ev_br_fork, st));
            B2D_CUDA(cudaStreamWaitEvent(h->side_stream, h->ev_br_fork, 0));
            B2D_TRY(op(h->side_stream));
            B2D_CUDA(cudaEventRecord(h->ev_br_join, h->side_stream));
            branch_open = true;
            ++idx;
            continue;
        }
        if (op.join && branch_open) {
            B2D_CUDA(cudaStreamWaitEvent(st, h->ev_br_join, 0));
            branch_open = false;
        }
        if (pipe && idx == h->temb_free_op) {
            B2D_CUDA(cudaEventRecord(h->ev_side_fork, st));
            B2D_CUDA(cudaStreamWaitEvent(h->side_stream, h->ev_side_fork, 0));
            if (ddim) h->temb_t = h->d_t_next;
            else h->temb_t_off = -1;
            const int rc = h->step_ops[0](h->side_stream);
            h->temb_t = h->d_t;
            h->temb_t_off = 0;
            if (rc) return rc;
            B2D_CUDA(cudaEventRecord(h->ev_side_join, h->side_stream));
        }
        B2D_TRY(op(st));
        if (dbg) {
            cudaError_t e = cudaStreamSynchronize(st);
            if (e != cudaSuccess)
                return fail(-2, "step op #" + std::to_string(idx) + " failed: " + cudaGetErrorString(e));
        }
        ++idx;
    }
    return 0;
}

static bool temb_pipelined(const Handle* h) {
    static const bool no_pipe = getenv("B2D_NO_TEMB_PIPE") != nullptr;
    return !no_pipe && h->temb_free_op > 0;
}
static int join_temb_side(Handle* h, cudaStream_t st) {
    if (temb_pipelined(h)) B2D_CUDA(cudaStreamWaitEvent(st, h->ev_side_join, 0));
    return 0;
}

// Device tables of the DDIM loop for the current (schedule, sequence, eta): re-validated against T, re-computed and uploaded only
// when one of them changed (this synchronises the device: queued work may still read the old tables).
static int ddim_prepare(Handle* h) {
    const int T = h->T, S = (int)h->ddim_tau.size();
    B2D_CHECK(S >= 1 && h->ddim_tau[0] <= T - 1, "DDIM timesteps exceed T-1 of the current schedule");
    B2D_CHECK((int)h->h_alpha_hat.size() == T, "internal: host alpha_hat out of date");
    if (!h->ddim_dirty && h->ddim_cap >= T + 1) return 0;
    B2D_CUDA(cudaDeviceSynchronize());
    if (h->ddim_cap < T + 1) {
        h->drop_ddim_graphs();   // they hold the table pointers
        h->release(h->d_ddim_tau);
        h->release(h->d_ddim_coef);
        h->d_ddim_tau = nullptr;
        h->d_ddim_coef = nullptr;
        h->ddim_cap = 0;
        B2D_TRY(h->alloc(&h->d_ddim_tau, T + 1));
        B2D_TRY(h->alloc(&h->d_ddim_coef, T + 1));
        h->ddim_cap = T + 1;
    }
    std::vector<int> tau(h->ddim_tau);
    tau.resize(S + 2, 0);
    std::vector<float4> coef(S);
    for (int k = 0; k < S; ++k)
        coef[k] = ddim_coefficients(h->h_alpha_hat[tau[k]], k + 1 < S ? h->h_alpha_hat[tau[k + 1]] : 1.0f, h->ddim_eta);
    B2D_CUDA(cudaMemcpy(h->d_ddim_tau, tau.data(), tau.size() * sizeof(int), cudaMemcpyHostToDevice));
    B2D_CUDA(cudaMemcpy(h->d_ddim_coef, coef.data(), coef.size() * sizeof(float4), cudaMemcpyHostToDevice));
    h->ddim_dirty = false;
    return 0;
}

}  // namespace b2d

using namespace b2d;

// ================================================================================================= C ABI
extern "C" {

const char* b2d_last_error(void) { return g_status.msg.c_str(); }
int b2d_abi_version(void) { return B2D_ABI_VERSION; }

int b2d_create(const b2d_config* cfg, b2d_handle** out) {
    B2D_CHECK(cfg && out, "null argument");
    B2D_CHECK(cfg->family == B2D_FAMILY_R || cfg->family == B2D_FAMILY_D, "unknown family");
    B2D_CHECK(is_pow2(cfg->img_size) && cfg->img_size >= 32 && cfg->img_size <= 128, "img_size must be 32, 64 or 128");
    B2D_CHECK(cfg->max_batch >= 1, "max_batch must be positive");
    B2D_CHECK(cfg->c_hr >= 1 && cfg->c_out >= 1, "channel counts must be positive");
    int dev = 0, ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0)
        return fail(-2, "no CUDA device: this library has no CPU fallback (" + std::string(cudaGetErrorString(e)) + ")");
    B2D_CUDA(cudaGetDevice(&dev));
    cudaDeviceProp prop;
    B2D_CUDA(cudaGetDeviceProperties(&prop, dev));
    B2D_CHECK(prop.major == 10, "b200ddpm kernels are compiled for sm_100a only");
    auto* h = new b2d_handle();
    h->cfg = *cfg;
    if (h->cfg.n_heads <= 0) h->cfg.n_heads = 4;
    h->num_sms = prop.multiProcessorCount;
    int rc = 0;
    do {
        if ((rc = conv_tc_init_attrs())) break;
        if ((rc = conv_tcp_init_attrs())) break;
        if ((rc = flash_attn_init_attrs())) break;
        if ((rc = attn_tc_init_attrs())) break;
        if ((rc = attn_tc2_init_attrs())) break;
        if ((rc = attn_tc3_init_attrs())) break;
        if ((rc = attn_tc5_init_attrs())) break;
        if ((rc = attn_tc6_init_attrs())) break;
        if ((rc = attn_tc8_init_attrs())) break;
        if ((rc = tail_tc_init_attrs())) break;
        if ((rc = gemm_stream_init_attrs())) break;
        if ((rc = attn_block_init_attrs())) break;
        if ((rc = norm_fused_init_attrs())) break;
        if ((rc = init_uniform_carveout())) break;
        const int B = cfg->max_batch, H = cfg->img_size;
        const size_t n = (size_t)B * cfg->c_hr * H * H, plane = (size_t)H * H;
        if ((rc = init_batch_buffers(h))) break;
        if ((rc = h->alloc(&h->d_x_work, n))) break;
        if ((rc = h->alloc(&h->d_job, 1))) break;
        // staging of the host entry point (b2d_sample_host): sized once, never re-allocated per call
        if (cfg->family == B2D_FAMILY_R) {
            if (cfg->has_lsm && (rc = h->alloc(&h->d_lsm_stage, (size_t)B * plane))) break;
            if (cfg->has_topo && (rc = h->alloc(&h->d_topo_stage, (size_t)B * plane))) break;
        }
        h->cond_stage_elems = (size_t)B * std::max(cfg->cond_channels, 1) * plane;   // Family D low-res fields are smaller
        if ((rc = h->alloc(&h->d_cond_stage, h->cond_stage_elems))) break;
        if (cudaMallocHost(reinterpret_cast<void**>(&h->h_y_pinned), (size_t)B * sizeof(int)) != cudaSuccess) {
            rc = fail(-2, "pinned label staging allocation failed");
            break;
        }
    } while (0);
    if (rc) {
        delete h;
        return rc;
    }
    *out = h;
    return 0;
}

void b2d_destroy(b2d_handle* h) { delete h; }

int b2d_load_weights(b2d_handle* h, const b2d_tensor* tensors, int32_t n) {
    B2D_CHECK(h && tensors && n > 0, "null argument");
    B2D_CHECK(!h->weights_loaded, "weights already loaded on this handle (create a new handle to reload)");
    h->sd.clear();
    for (int i = 0; i < n; ++i) {
        const b2d_tensor& t = tensors[i];
        B2D_CHECK(t.name && t.data && t.ndim >= 0 && t.ndim <= 4, "malformed tensor entry");
        HostTensor ht;
        size_t numel = 1;
        for (int d = 0; d < t.ndim; ++d) {
            ht.shape.push_back(t.shape[d]);
            numel *= (size_t)t.shape[d];
        }
        ht.v.assign(t.data, t.data + numel);
        h->sd[t.name] = std::move(ht);
    }
    int rc = (h->cfg.family == B2D_FAMILY_R) ? pack_family_r(h) : pack_family_d(h);
    h->sd.clear();
    if (rc) return rc;
    h->weights_loaded = true;
    return 0;
}

int b2d_set_schedule(b2d_handle* h, const float* betas, const float* alphas, const float* alpha_hat, int32_t T) {
    B2D_CHECK(h && betas && alphas && alpha_hat && T >= 2, "bad schedule");
    // the tables may still be read by work queued earlier on any stream of this device
    B2D_CUDA(cudaDeviceSynchronize());
    if (T != h->T) {
        // the captured step graphs hold the table pointers: drop them together with the old tables
        h->drop_graphs();
        h->release(h->d_betas);
        h->release(h->d_alphas);
        h->release(h->d_alpha_hat);
        h->d_betas = h->d_alphas = h->d_alpha_hat = nullptr;
        h->T = 0;
        B2D_TRY(h->alloc(&h->d_betas, T));
        B2D_TRY(h->alloc(&h->d_alphas, T));
        B2D_TRY(h->alloc(&h->d_alpha_hat, T));
        h->T = T;
    }
    B2D_CUDA(cudaMemcpy(h->d_betas, betas, T * 4, cudaMemcpyHostToDevice));
    B2D_CUDA(cudaMemcpy(h->d_alphas, alphas, T * 4, cudaMemcpyHostToDevice));
    B2D_CUDA(cudaMemcpy(h->d_alpha_hat, alpha_hat, T * 4, cudaMemcpyHostToDevice));
    h->h_alpha_hat.assign(alpha_hat, alpha_hat + T);
    h->ddim_dirty = true;
    return 0;
}

int b2d_set_timesteps(b2d_handle* h, const int32_t* timesteps_host, int32_t n, float eta) {
    B2D_CHECK(h, "null handle");
    if (n == 0) {
        B2D_CHECK(timesteps_host == nullptr, "n == 0 restores the DDPM loop and takes no timesteps");
        h->ddim = false;
        return 0;
    }
    B2D_CHECK(timesteps_host && n >= 1, "timesteps: NULL or negative length");
    B2D_CHECK(eta >= 0.f && eta <= 1.f, "eta must lie in [0, 1]");
    for (int k = 0; k < n; ++k) {
        B2D_CHECK(timesteps_host[k] >= 1, "timesteps must be >= 1");
        B2D_CHECK(k == 0 || timesteps_host[k] < timesteps_host[k - 1], "timesteps must be strictly decreasing");
    }
    B2D_CHECK(h->T < 2 || timesteps_host[0] <= h->T - 1, "timesteps must be <= T-1 of the current schedule");
    std::vector<int> tau(timesteps_host, timesteps_host + n);
    if (tau != h->ddim_tau || eta != h->ddim_eta) {
        h->ddim_tau.swap(tau);
        h->ddim_eta = eta;
        h->ddim_dirty = true;
    }
    h->ddim = true;
    return 0;
}


// y_dev: int64 labels in device memory (synchronises once to range-check them, as nn.Embedding would raise);
// y_host: the same in host memory (no device round trip).  At most one of them is non-null.
static int set_conditioning_impl(b2d_handle* h, const float* lsm, const float* topo, const float* cond, int32_t cond_h,
                                 int32_t cond_w, const int64_t* y_dev, const int64_t* y_host, int32_t B, cudaStream_t st,
                                 const int* y_dev_i32 = nullptr /* already range-checked int32 labels in device memory */) {
    B2D_CHECK(h, "null handle");
    B2D_TRY(ensure_program(h, B));
    const b2d_config& c = h->cfg;
    const int H = c.img_size;
    const bool has_y = (y_dev != nullptr || y_host != nullptr || y_dev_i32 != nullptr);
    if (y_dev_i32) {
        B2D_CHECK(c.num_classes > 0, "y given but the model has no label embedding");
        B2D_CUDA(cudaMemcpyAsync(h->d_y, y_dev_i32, B * 4, cudaMemcpyDeviceToDevice, st));
    } else if (has_y) {
        B2D_CHECK(c.num_classes > 0, "y given but the model has no label embedding");
        std::vector<int64_t> tmp;
        if (y_dev) {
            tmp.resize(B);
            B2D_CUDA(cudaMemcpyAsync(tmp.data(), y_dev, B * 8, cudaMemcpyDeviceToHost, st));
            B2D_CUDA(cudaStreamSynchronize(st));
            y_host = tmp.data();
        } else {
            B2D_CUDA(cudaStreamSynchronize(st));   // h_y_pinned may still be the source of an earlier upload
        }
        for (int i = 0; i < B; ++i) {
            B2D_CHECK(y_host[i] >= 0 && y_host[i] < c.num_classes, "class label out of range");
            h->h_y_pinned[i] = (int)y_host[i];
        }
        B2D_CUDA(cudaMemcpyAsync(h->d_y, h->h_y_pinned, B * 4, cudaMemcpyHostToDevice, st));
    }
    if (has_y != h->has_y) h->drop_graphs();   // the time-embedding launch of a captured graph holds (has_y ? d_y : null)
    h->has_y = has_y;
    if (c.family == B2D_FAMILY_D) return set_conditioning_d(h, cond, cond_h, cond_w, B, st);
    // Family R: stack [lsm, topo, cond] (concat order of Encoder.forward :228-238) per sample, then conv1's share of it
    B2D_CHECK(!c.has_lsm || lsm, "model was built with lsm_tensor: lsm_cond is required");
    B2D_CHECK(!c.has_topo || topo, "model was built with topo_tensor: topo_cond is required");
    B2D_CHECK((c.cond_channels > 0) == (cond != nullptr), "cond_img presence must match cond_on_img of the model");
    const int ccond = c.has_lsm + c.has_topo + c.cond_channels;
    if (ccond == 0) return 0;
    const size_t plane = (size_t)H * H;
    int ch = 0;
    auto put = [&](const float* src, int nch) -> int {
        B2D_CUDA(cudaMemcpy2DAsync(h->d_cond_stack + (size_t)ch * plane, (size_t)ccond * plane * 4, src, (size_t)nch * plane * 4,
                                   (size_t)nch * plane * 4, B, cudaMemcpyDeviceToDevice, st));
        ch += nch;
        return 0;
    };
    if (c.has_lsm) B2D_TRY(put(lsm, 1));
    if (c.has_topo) B2D_TRY(put(topo, 1));
    if (c.cond_channels) B2D_TRY(put(cond, c.cond_channels));
    const int cin_total = c.c_hr + ccond;
    dim3 grid(H / 2 / 16, H / 2 / 16, B);
    B2D_CUDA(launch_k(stem_conv_kernel<8, 2>, dim3(grid), dim3(256), 0, st, h->d_cond_stack, ccond, H, H, reinterpret_cast<float*>(h->dev["stem.w"]),
                                                 cin_total, c.c_hr, nullptr, nullptr, 0, nullptr, h->d_cond_pre, H / 2, H / 2,
                                                 3));
    B2D_CUDA(cudaGetLastError());
    return 0;
}

int b2d_set_conditioning(b2d_handle* h, const float* lsm, const float* topo, const float* cond, int32_t cond_h,
                         int32_t cond_w, const int64_t* y, int32_t B, void* stream) {
    return set_conditioning_impl(h, lsm, topo, cond, cond_h, cond_w, y, nullptr, B, as_stream(stream));
}

int b2d_forward(b2d_handle* h, const float* x, const int64_t* t_host, float* eps_out, int32_t B, void* stream) {
    B2D_CHECK(h && x && t_host && eps_out, "null argument");
    B2D_TRY(ensure_program(h, B));
    cudaStream_t st = as_stream(stream);
    std::vector<int> ti(B);
    for (int i = 0; i < B; ++i) ti[i] = (int)t_host[i];
    B2D_CUDA(cudaMemcpyAsync(h->d_t, ti.data(), B * 4, cudaMemcpyHostToDevice, st));
    B2D_CUDA(cudaStreamSynchronize(st));  // ti is a stack-lifetime staging buffer
    h->cur_x = x;
    h->cur_eps = eps_out;
    B2D_TRY(run_step_ops(h, st));
    h->last_launches = (int64_t)h->step_ops.size();
    return 0;
}

// NHWC f16 <-> NCHW f32 (stand-alone Encoder / Decoder boundaries: the reference hands feature maps around as NCHW fp32)
__global__ void nhwc_f16_to_nchw_f32_kernel(const f16* __restrict__ in, float* __restrict__ out, int C, int HW, size_t total) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int p = (int)(i % HW);
        const int c = (int)((i / HW) % C);
        const size_t b = i / ((size_t)HW * C);
        out[i] = __half2float(in[(b * HW + p) * C + c]);
    }
}
__global__ void nchw_f32_to_nhwc_f16_kernel(const float* __restrict__ in, f16* __restrict__ out, int C, int HW, size_t total) {
    for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
        const int c = (int)(i % C);
        const int p = (int)((i / C) % HW);
        const size_t b = i / ((size_t)HW * C);
        const float v = in[(b * C + c) * HW + p];
        if (fabsf(v) > F16_MAX) atomicAdd(&g_sat_count, 1u);
        out[i] = __float2half_rn(sat_h(v));
    }
}

static int upload_t(b2d_handle* h, const int64_t* t_host, int B, cudaStream_t st) {
    std::vector<int> ti(B);
    for (int i = 0; i < B; ++i) ti[i] = (int)t_host[i];
    B2D_CUDA(cudaMemcpyAsync(h->d_t, ti.data(), B * 4, cudaMemcpyHostToDevice, st));
    B2D_CUDA(cudaStreamSynchronize(st));  // ti is a stack-lifetime staging buffer
    return 0;
}

int b2d_encoder_forward(b2d_handle* h, const float* x, const int64_t* t_host, float* const* fmaps_out, int32_t B, void* stream) {
    B2D_CHECK(h && x && t_host && fmaps_out, "null argument");
    B2D_CHECK(h->cfg.family == B2D_FAMILY_R, "stand-alone Encoder.forward exists for Family R only");
    B2D_TRY(ensure_program(h, B));
    cudaStream_t st = as_stream(stream);
    B2D_TRY(upload_t(h, t_host, B, st));
    h->cur_x = x;
    h->cur_eps = h->d_eps;
    B2D_TRY(run_step_ops(h, st, false, 0, h->dec_begin_op));
    for (int i = 0; i < 5; ++i) {
        const Handle::Fmap& f = h->fmaps[i];
        const size_t total = (size_t)B * f.C * f.hw * f.hw;
        const int blocks = (int)std::min<size_t>((total + 255) / 256, (size_t)148 * 16);
        nhwc_f16_to_nchw_f32_kernel<<<blocks, 256, 0, st>>>(f.p, fmaps_out[i], f.C, f.hw * f.hw, total);
    }
    B2D_CUDA(cudaGetLastError());
    h->last_launches = h->dec_begin_op + 5;
    return 0;
}

int b2d_decoder_forward(b2d_handle* h, const float* const* fmaps_in, const int64_t* t_host, float* out, int32_t B, void* stream) {
    B2D_CHECK(h && fmaps_in && t_host && out, "null argument");
    B2D_CHECK(h->cfg.family == B2D_FAMILY_R, "stand-alone Decoder.forward exists for Family R only");
    B2D_TRY(ensure_program(h, B));
    cudaStream_t st = as_stream(stream);
    B2D_TRY(upload_t(h, t_host, B, st));
    for (int i = 0; i < 5; ++i) {
        const Handle::Fmap& f = h->fmaps[i];
        const size_t total = (size_t)B * f.C * f.hw * f.hw;
        const int blocks = (int)std::min<size_t>((total + 255) / 256, (size_t)148 * 16);
        nchw_f32_to_nhwc_f16_kernel<<<blocks, 256, 0, st>>>(fmaps_in[i], f.p, f.C, f.hw * f.hw, total);
    }
    B2D_CUDA(cudaGetLastError());
    h->cur_x = h->d_x_work;
    h->cur_eps = out;
    B2D_TRY(run_step_ops(h, st, false, 0, 1));                                   // time embeddings + projections
    B2D_TRY(run_step_ops(h, st, false, h->dec_begin_op, (int)h->step_ops.size()));
    h->last_launches = (int64_t)h->step_ops.size() - h->dec_begin_op + 6;
    return 0;
}

// One reverse step on stream `st`: the eps program on d_x_work, then the posterior update (whose last block advances i and t),
// or in DDIM mode the DDIM update (whose last block advances k, t and t_next).
static int enqueue_reverse_step(b2d_handle* h, int B, cudaStream_t st, bool ddim) {
    const b2d_config& c = h->cfg;
    const size_t per_sample = (size_t)c.c_hr * c.img_size * c.img_size;
    const size_t n = per_sample * B;
    h->cur_x = h->d_x_work;
    h->cur_eps = h->d_eps;
    B2D_TRY(run_step_ops(h, st, true, 0, -1, ddim));
    const int blocks = (int)std::min<size_t>((n / 4 + 255) / 256, (size_t)h->num_sms * 8);
    B2D_TRY(join_temb_side(h, st));   // the update's last block advances d_t / d_t_next, which the side branch reads
    if (ddim)
        B2D_CUDA(launch_k(ddim_update_kernel, dim3(blocks), dim3(256), 0, st, h->d_x_work, h->d_eps, h->d_job, h->d_ddim_tau,
                          h->d_ddim_coef, h->d_step, h->d_t, h->d_t_next, B, n, per_sample));
    else
        B2D_CUDA(launch_k(posterior_update_kernel, dim3(blocks), dim3(256), 0, st, h->d_x_work, h->d_eps, h->d_job, h->d_alphas,
                          h->d_betas, h->d_alpha_hat, h->d_step, h->d_t, B, n, per_sample));
    return 0;
}

static int capture_steps(b2d_handle* h, int B, int nsteps, bool ddim, cudaGraphExec_t* out, int* nodes_out) {
    cudaStream_t cs = h->own_stream;
    B2D_CUDA(cudaStreamBeginCapture(cs, cudaStreamCaptureModeThreadLocal));
    int rc = 0;
    for (int s = 0; s < nsteps && rc == 0; ++s) rc = enqueue_reverse_step(h, B, cs, ddim);
    cudaGraph_t graph = nullptr;
    cudaError_t ce = cudaStreamEndCapture(cs, &graph);
    if (rc) {
        if (graph) cudaGraphDestroy(graph);
        return rc;
    }
    B2D_CUDA(ce);
    size_t nn = 0;
    cudaGraphGetNodes(graph, nullptr, &nn);
    *nodes_out = (int)nn;
    cudaError_t ie = cudaGraphInstantiate(out, graph, 0);
    cudaGraphDestroy(graph);
    B2D_CUDA(ie);
    return 0;
}

// The loop on the handle's own state buffer d_x_work (already filled by the caller, on `st`).
static int sample_core(b2d_handle* h, const float* noise, uint64_t seed, uint64_t sample_offset, float noise_scale, int32_t B,
                       cudaStream_t st) {
    B2D_CHECK(h->T >= 2, "b2d_set_schedule has not been called");
    const b2d_config& c = h->cfg;
    B2D_CHECK(c.c_hr == c.c_out, "sampling needs c_out == c_hr");
    const size_t per_sample = (size_t)c.c_hr * c.img_size * c.img_size;
    const int T = h->T;
    SampleJob job{};
    job.noise = noise;
    job.seed = seed;
    job.sample_offset = sample_offset;
    job.noise_stride = per_sample * B;
    job.noise_scale = noise_scale;
    const bool ddim = h->ddim;
    int n_evals = T - 1;   // model evaluations of the loop
    if (ddim) {
        B2D_TRY(ddim_prepare(h));
        n_evals = (int)h->ddim_tau.size();
        B2D_CUDA(launch_k(set_job_ddim_kernel, dim3(1), dim3(256), 0, st, h->d_job, job, h->d_ddim_tau, h->d_t, h->d_t_next,
                          h->d_step, B));
    } else {
        B2D_CUDA(launch_k(set_job_kernel, dim3(1), dim3(256), 0, st, h->d_job, job, h->d_t, h->d_step, T - 1, B));
    }
    static const bool no_graph = getenv("B2D_NO_GRAPH") != nullptr;   // A/B: plain stream launches (PDL) instead of graphs
    if (temb_pipelined(h)) B2D_TRY(h->step_ops[0](st));   // embeddings of the first step; later ones come from the side branch
    if (no_graph) {
        for (int i = 0; i < n_evals; ++i) B2D_TRY(enqueue_reverse_step(h, B, st, ddim));
        h->last_launches = ((int64_t)h->step_ops.size() + 1) * n_evals + 2;
        return 0;
    }
    static const int env_steps = getenv("B2D_GRAPH_STEPS") ? atoi(getenv("B2D_GRAPH_STEPS")) : 8;
    const int gs = std::max(1, std::min(env_steps, T - 1));
    if (h->graph_steps != gs) {
        h->drop_graphs();
        h->graph_steps = gs;
    }
    // each mode replays its own pair; capturing one pair leaves the other untouched
    cudaGraphExec_t& g_one = ddim ? h->graph_one_ddim : h->graph_one;
    cudaGraphExec_t& g_multi = ddim ? h->graph_multi_ddim : h->graph_multi;
    int& nodes_one = ddim ? h->graph_nodes_one_ddim : h->graph_nodes_one;
    int& nodes_multi = ddim ? h->graph_nodes_multi_ddim : h->graph_nodes_multi;
    if (!g_one) B2D_TRY(capture_steps(h, B, 1, ddim, &g_one, &nodes_one));
    if (gs > 1 && !g_multi) B2D_TRY(capture_steps(h, B, gs, ddim, &g_multi, &nodes_multi));
    const int n_multi = gs > 1 ? n_evals / gs : 0, n_one = n_evals - n_multi * gs;
    for (int k = 0; k < n_multi; ++k) B2D_CUDA(cudaGraphLaunch(g_multi, st));
    for (int k = 0; k < n_one; ++k) B2D_CUDA(cudaGraphLaunch(g_one, st));
    h->last_launches = (int64_t)nodes_multi * n_multi + (int64_t)nodes_one * n_one + 2;
    return 0;
}

int b2d_sample(b2d_handle* h, float* x_inout, const float* noise, uint64_t seed, uint64_t sample_offset,
               float noise_scale, int32_t B, void* stream) {
    B2D_CHECK(h && x_inout, "null argument");
    B2D_TRY(ensure_program(h, B));
    cudaStream_t st = as_stream(stream);
    const size_t n = (size_t)h->cfg.c_hr * h->cfg.img_size * h->cfg.img_size * B;
    B2D_CUDA(cudaMemcpyAsync(h->d_x_work, x_inout, n * 4, cudaMemcpyDeviceToDevice, st));
    B2D_TRY(sample_core(h, noise, seed, sample_offset, noise_scale, B, st));
    B2D_CUDA(cudaMemcpyAsync(x_inout, h->d_x_work, n * 4, cudaMemcpyDeviceToDevice, st));
    return 0;
}

// Host entry: enqueue only (uploads, loop, download into x_inout_host); b2d_sample_host adds the final synchronise, the
// ensemble driver overlaps the next job's host work with it.
static int sample_host_enqueue(b2d_handle* h, float* x_inout_host, const float* lsm_host, const float* topo_host,
                               const float* cond_host, int32_t cond_h, int32_t cond_w, const int64_t* y_host,
                               const float* noise_host, uint64_t seed, uint64_t sample_offset, float noise_scale, int32_t B,
                               cudaStream_t st) {
    B2D_CHECK(h && x_inout_host, "null argument");
    B2D_CHECK(B >= 1 && B <= h->cfg.max_batch, "batch exceeds max_batch of the handle");
    const b2d_config& c = h->cfg;
    const int H = c.img_size;
    const size_t plane = (size_t)H * H;
    const size_t n = (size_t)B * c.c_hr * plane;
    B2D_CHECK(!lsm_host || h->d_lsm_stage, "lsm given but the model was built without lsm conditioning");
    B2D_CHECK(!topo_host || h->d_topo_stage, "topo given but the model was built without topography conditioning");
    const size_t cond_elems = !cond_host ? 0
                              : (c.family == B2D_FAMILY_D) ? (size_t)B * c.cond_channels * cond_h * cond_w
                                                           : (size_t)B * c.cond_channels * plane;
    B2D_CHECK(cond_elems <= h->cond_stage_elems, "conditioning field larger than the handle's staging buffer");
    B2D_CUDA(cudaMemcpyAsync(h->d_x_work, x_inout_host, n * 4, cudaMemcpyHostToDevice, st));
    if (lsm_host) B2D_CUDA(cudaMemcpyAsync(h->d_lsm_stage, lsm_host, (size_t)B * plane * 4, cudaMemcpyHostToDevice, st));
    if (topo_host) B2D_CUDA(cudaMemcpyAsync(h->d_topo_stage, topo_host, (size_t)B * plane * 4, cudaMemcpyHostToDevice, st));
    if (cond_host) B2D_CUDA(cudaMemcpyAsync(h->d_cond_stage, cond_host, cond_elems * 4, cudaMemcpyHostToDevice, st));
    if (noise_host) {
        // [T][n] indexed by i for the DDPM loop, [S][n] indexed by k for the DDIM loop (S <= T-1 fits the same staging)
        const size_t ne = (h->ddim ? h->ddim_tau.size() : (size_t)h->T) * n;
        if (ne > h->noise_stage_elems) {
            B2D_CUDA(cudaStreamSynchronize(st));
            h->release(h->d_noise_stage);
            h->d_noise_stage = nullptr;
            h->noise_stage_elems = 0;
            B2D_TRY(h->alloc(&h->d_noise_stage, ne));
            h->noise_stage_elems = ne;
        }
        B2D_CUDA(cudaMemcpyAsync(h->d_noise_stage, noise_host, ne * 4, cudaMemcpyHostToDevice, st));
    }
    B2D_TRY(set_conditioning_impl(h, lsm_host ? h->d_lsm_stage : nullptr, topo_host ? h->d_topo_stage : nullptr,
                                  cond_host ? h->d_cond_stage : nullptr, cond_h, cond_w, nullptr, y_host, B, st));
    B2D_TRY(sample_core(h, noise_host ? h->d_noise_stage : nullptr, seed, sample_offset, noise_scale, B, st));
    B2D_CUDA(cudaMemcpyAsync(x_inout_host, h->d_x_work, n * 4, cudaMemcpyDeviceToHost, st));
    return 0;
}

int b2d_sample_host(b2d_handle* h, float* x_inout_host, const float* lsm_host, const float* topo_host,
                    const float* cond_host, int32_t cond_h, int32_t cond_w, const int64_t* y_host,
                    const float* noise_host, uint64_t seed, uint64_t sample_offset, float noise_scale, int32_t B) {
    B2D_CHECK(h, "null handle");
    cudaStream_t st = h->own_stream;
    const int rc = sample_host_enqueue(h, x_inout_host, lsm_host, topo_host, cond_host, cond_h, cond_w, y_host, noise_host, seed,
                                       sample_offset, noise_scale, B, st);
    cudaError_t se = cudaStreamSynchronize(st);
    if (rc) return rc;
    B2D_CUDA(se);
    return 0;
}

#include "ensemble.cuh"

int64_t b2d_last_launch_count(const b2d_handle* h) { return h ? h->last_launches : 0; }

int b2d_profile_step(b2d_handle* h, const float* x, const int64_t* t_host, int32_t B, int32_t reps, b2d_op_profile* out,
                     int32_t max_ops, int32_t* n_ops) {
    B2D_CHECK(h && x && t_host && out && n_ops && reps >= 1, "bad argument");
    B2D_TRY(ensure_program(h, B));
    cudaStream_t st = h->own_stream;
    std::vector<int> ti(B);
    for (int i = 0; i < B; ++i) ti[i] = (int)t_host[i];
    B2D_CUDA(cudaMemcpy(h->d_t, ti.data(), B * 4, cudaMemcpyHostToDevice));
    h->cur_x = x;
    h->cur_eps = h->d_eps;
    const int n = (int)h->step_ops.size();
    B2D_CHECK(n <= max_ops, "profile buffer too small");
    std::vector<cudaEvent_t> ev(n + 1);
    for (auto& e : ev) B2D_CUDA(cudaEventCreate(&e));
    std::vector<double> ms(n, 0.0);
    for (int r = 0; r < reps + 1; ++r) {   // first repetition is a warm-up
        B2D_CUDA(cudaEventRecord(ev[0], st));
        for (int i = 0; i < n; ++i) {
            B2D_TRY(h->step_ops[i](st));
            B2D_CUDA(cudaEventRecord(ev[i + 1], st));
        }
        B2D_CUDA(cudaStreamSynchronize(st));
        if (r == 0) continue;
        for (int i = 0; i < n; ++i) {
            float m = 0;
            cudaEventElapsedTime(&m, ev[i], ev[i + 1]);
            ms[i] += m;
        }
    }
    for (auto& e : ev) cudaEventDestroy(e);
    for (int i = 0; i < n; ++i) {
        const Op& op = h->step_ops[i];
        memset(&out[i], 0, sizeof(out[i]));
        strncpy(out[i].name, op.name.c_str(), sizeof(out[i].name) - 1);
        strncpy(out[i].klass, op.klass.c_str(), sizeof(out[i].klass) - 1);
        out[i].flops = op.flops;
        out[i].bytes = op.bytes;
        out[i].ms = ms[i] / reps;
    }
    *n_ops = n;
    return 0;
}

int b2d_debug_read(b2d_handle* h, const char* name, float* out_host, int64_t max_elems, int32_t* C_out, int32_t* hw_out) {
    B2D_CHECK(h && name && out_host, "null argument");
    auto it = h->taps.find(name);
    if (it == h->taps.end()) return fail(-3, std::string("no such tap: ") + name);
    const size_t n = (size_t)h->prog_B * it->second.hw * it->second.hw * it->second.C;
    B2D_CHECK((int64_t)n <= max_elems, "output buffer too small");
    std::vector<uint16_t> tmp(n);
    B2D_CUDA(cudaDeviceSynchronize());
    B2D_CUDA(cudaMemcpy(tmp.data(), it->second.p, n * 2, cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < n; ++i) {
        __half hv;
        memcpy(&hv, &tmp[i], 2);
        out_host[i] = __half2float(hv);
    }
    if (C_out) *C_out = it->second.C;
    if (hw_out) *hw_out = it->second.hw;
    return 0;
}

// ------------------------------------------------------------------------------------------------ single operators
int b2d_op_conv2d(const void* in, const void* w, const float* bias, const void* residual, const float* post_add,
                  int32_t post_stride, void* out, int32_t B, int32_t Hi, int32_t Wi, int32_t Cin, int32_t Cout, int32_t R,
                  int32_t S, int32_t stride, int32_t pad, int32_t convt, int32_t act, int32_t impl, void* stream) {
    B2D_CHECK(in && w && out, "null argument");
    B2D_CHECK(R == S, "square filters only");
    ConvPlan pl;
    ConvParams& p = pl.p;
    memset(&p, 0, sizeof(p));
    p.B = B; p.Hi = Hi; p.Wi = Wi; p.Cin = Cin; p.R = R; p.S = S; p.stride = stride; p.pad = pad; p.convt = convt;
    if (convt) {
        p.Ho = Hi; p.Wo = Wi; p.Cout = 4 * Cout; p.CoutT = Cout;
    } else {
        p.Ho = (Hi + 2 * pad - R) / stride + 1;
        p.Wo = (Wi + 2 * pad - S) / stride + 1;
        p.Cout = Cout; p.CoutT = Cout;
    }
    p.in = (const f16*)in; p.w = (const f16*)w; p.bias = bias; p.residual = (const f16*)residual;
    p.post_add = post_add; p.post_stride = post_stride; p.act = act; p.out = (f16*)out;
    if (impl == 1) return conv_launch_simt(p, as_stream(stream));
    int dev = 0, sms = 148;
    cudaGetDevice(&dev);
    cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
    if (impl == 2 || (impl == 0 && gemm_stream_supported(p) && getenv("B2D_NO_STREAM_GEMM") == nullptr)) {
        B2D_CHECK(gemm_stream_supported(p, impl == 2 ? 0 : GS_MIN_ROWS), "shape not eligible for the streaming GEMM");
        B2D_TRY(gemm_stream_init_attrs());
        GemmStreamPlan gp;
        gp.p = p;
        B2D_TRY(gemm_stream_plan_build(gp, sms));
        return gemm_stream_launch(gp, as_stream(stream));
    }
    B2D_TRY(conv_tc_init_attrs());
    B2D_TRY(conv_plan_build(pl, sms, impl != 4 && impl != 5));      // impl 5: persistent kernel without the slab tiling
    if (impl == 5) impl = 3;
    if (impl == 3 || (impl == 0 && conv_tcp_eligible(pl, sms))) {      // impl 3: force the persistent kernel, 4: the one-tile kernel
        B2D_CHECK(pl.p.splits == 1, "shape not eligible for the persistent convolution (split-K plan)");
        B2D_TRY(conv_tcp_init_attrs());
        return conv_launch_tcp(pl, sms, as_stream(stream));
    }
    float* ws = nullptr;
    if (pl.ws_floats) {
        B2D_CUDA(cudaMalloc(&ws, pl.ws_floats * sizeof(float)));
        pl.p.ws = ws;
    }
    int rc = conv_launch_tc(pl, as_stream(stream));
    if (ws) {
        cudaStreamSynchronize(as_stream(stream));
        cudaFree(ws);
    }
    return rc;
}

int b2d_op_layernorm(const void* x, const float* gamma, const float* beta, void* y, int32_t rows, int32_t C, void* stream) {
    return layernorm_launch((const f16*)x, gamma, beta, (f16*)y, rows, C, as_stream(stream));
}

int b2d_op_attention(const void* qkv, void* o, int32_t B, int32_t L, int32_t C, int32_t heads, void* stream) {
    B2D_TRY(flash_attn_init_attrs());
    if (attn_tc_supported(L, C, heads) && getenv("B2D_NO_TC_ATTN") == nullptr) {
        B2D_TRY(attn_tc_init_attrs());
        AttnTcMaps tm;
        B2D_TRY(attn_tc_make_map(&tm, (const f16*)qkv, B, L, C));
        const int attn_v = getenv("B2D_ATTN_V") ? atoi(getenv("B2D_ATTN_V")) : 8;
        if (attn_v == 3) {
            B2D_TRY(attn_tc3_init_attrs());
            return attn_tc3_launch(tm, (f16*)o, B, L, C, heads, as_stream(stream));
        }
        if (attn_v == 8) {
            B2D_TRY(attn_tc8_init_attrs());
            return attn_tc8_launch(tm, (f16*)o, B, L, C, heads, as_stream(stream));
        }
        if (attn_v == 6 || attn_v == 7) {
            B2D_TRY(attn_tc6_init_attrs());
            return attn_v == 6 ? attn_tc6_launch<0>(tm, (f16*)o, B, L, C, heads, as_stream(stream))
                               : attn_tc6_launch<1>(tm, (f16*)o, B, L, C, heads, as_stream(stream));
        }
        if (attn_v == 4) {
            B2D_TRY(attn_tc3_init_attrs());
            B2D_TRY(attn_tc4_make_map(&tm, (const f16*)qkv, B, L, C));
            return attn_tc4_launch(tm, (f16*)o, B, L, C, heads, as_stream(stream));
        }
        if (attn_v == 2 && attn_tc2_supported(L, C, heads)) {
            B2D_TRY(attn_tc2_init_attrs());
            int dev = 0, sms = 148;
            cudaGetDevice(&dev);
            cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev);
            return attn_tc2_launch(tm, (f16*)o, B, L, C, heads, sms, as_stream(stream));
        }
        return attn_tc_launch(tm, (f16*)o, B, L, C, heads, as_stream(stream));
    }
    if (attn_tc5_supported(L, C, heads) && getenv("B2D_NO_TC_ATTN") == nullptr) {
        B2D_TRY(attn_tc5_init_attrs());
        AttnTcMaps tm5;
        B2D_TRY(attn_tc5_make_map(&tm5, (const f16*)qkv, B, L, C));
        return attn_tc5_launch(tm5, (f16*)o, B, L, C, heads, as_stream(stream));
    }
    return flash_attn_launch((const f16*)qkv, (f16*)o, B, L, C, heads, as_stream(stream));
}

int b2d_op_attn_block(const void* x, const void* w_folded, const float* c1, const float* bias, void* o, int32_t B, int32_t L,
                      int32_t C, int32_t heads, void* stream) {
    B2D_CHECK(attn_block_supported(L, C, heads), "shape not eligible for the fused low-resolution attention");
    B2D_TRY(attn_block_init_attrs());
    AttnBlockPlan pl;
    B2D_TRY(attn_block_plan_build(pl, (const f16*)x, (const f16*)w_folded, c1, bias, (f16*)o, B * L, C, L, heads));
    return attn_block_launch(pl, as_stream(stream));
}

int b2d_op_attn_block_out(const void* x, const void* w_folded, const float* c1, const float* bias, const void* wo,
                          const float* out_bias, void* y, int32_t B, int32_t L, int32_t C, int32_t heads, int32_t final_act,
                          void* stream) {
    B2D_CHECK(attn_block_supported(L, C, heads) && attn_block_out_supported(C, heads), "shape not eligible for the fused attention block");
    B2D_TRY(attn_block_init_attrs());
    AttnBlockPlan pl;
    B2D_TRY(attn_block_plan_build(pl, (const f16*)x, (const f16*)w_folded, c1, bias, nullptr, B * L, C, L, heads));
    float* ws = nullptr;
    B2D_CUDA(cudaMalloc(&ws, attn_block_ws_floats(B * L, C, heads) * sizeof(float)));
    // same polarity as the model program: the DSMEM-gather variant is opt-in (measured slower; B2D_ATTN_GATHER=1 selects it)
    const bool gather = getenv("B2D_ATTN_GATHER") != nullptr && attn_block_gather_supported(C, heads);
    int rc = attn_block_plan_fuse_out(pl, (const f16*)wo, out_bias, (const f16*)x, (f16*)y, ws, final_act, gather ? 2 : 1);
    if (rc == 0) rc = attn_block_launch(pl, as_stream(stream));
    cudaStreamSynchronize(as_stream(stream));
    cudaFree(ws);
    return rc;
}

int b2d_op_instnorm(const void* x, const void* skip, const float* vec, int32_t vec_stride, void* y, float* stats_ws,
                    int32_t B, int32_t HW, int32_t C, void* stream) {
    cudaStream_t st = as_stream(stream);
    (void)stats_ws;  // kept for ABI stability; the operator owns its scratch
    B2D_CHECK(C % 64 == 0, "C must be a multiple of 64");
    const int nslab = (HW + 255) / 256, ngrp = C / 64;
    float* ws = nullptr;
    const size_t n_stats = (size_t)B * C * 2, n_part = (size_t)B * ngrp * nslab * 128, n_cnt = (size_t)B * ngrp;
    B2D_CUDA(cudaMalloc(&ws, (n_stats + n_part + n_cnt) * 4));
    float* stats = ws;
    float* partial = ws + n_stats;
    unsigned int* counters = reinterpret_cast<unsigned int*>(ws + n_stats + n_part);
    cudaMemsetAsync(counters, 0, n_cnt * 4, st);
    dim3 grid(nslab, ngrp, B);
    B2D_CUDA(launch_k(plane_stats_kernel, dim3(grid), dim3(256), 0, st, (const f16*)x, partial, counters, stats, HW, C, 256));
    const size_t total8 = (size_t)B * HW * C / 8;
    const int blocks = (int)std::min<size_t>((total8 + 255) / 256, (size_t)148 * 16);
    B2D_CUDA(launch_k(instnorm_apply_kernel, dim3(blocks), dim3(256), 0, st, (const f16*)x, stats, (const f16*)skip, vec, vec_stride, (f16*)y, HW, C,
                                                  total8));
    cudaError_t e = cudaGetLastError();
    cudaStreamSynchronize(st);
    cudaFree(ws);
    B2D_CUDA(e);
    return 0;
}

int b2d_op_final_layer(const void* x, const float* w, const float* bias, float* out, int32_t B, int32_t H, int32_t W,
                       int32_t use_mma_sync, void* stream) {
    cudaStream_t st = as_stream(stream);
    B2D_CHECK(x && w && bias && out && B >= 1 && H >= 1 && W >= 1, "bad argument");
    const int HW = H * W, C = 64;
    const int nslab = (HW + 255) / 256;
    float* ws = nullptr;
    const size_t n_stats = (size_t)B * C * 2, n_part = (size_t)B * nslab * 128, n_cnt = (size_t)B;
    B2D_CUDA(cudaMalloc(&ws, (n_stats + n_part + n_cnt) * 4));
    float* stats = ws;
    float* partial = ws + n_stats;
    unsigned int* counters = reinterpret_cast<unsigned int*>(ws + n_stats + n_part);
    cudaMemsetAsync(counters, 0, n_cnt * 4, st);
    int rc = 0;
    do {
        cudaError_t e = launch_k(plane_stats_kernel, dim3(nslab, 1, B), dim3(256), 0, st, (const f16*)x, partial, counters, stats, HW, C, 256);
        if (e != cudaSuccess) { rc = fail(-2, cudaGetErrorString(e)); break; }
        if (!use_mma_sync && tail_tc_supported(H, W, 1)) {
            if ((rc = tail_tc_init_attrs())) break;
            TailTcPlan pl;
            if ((rc = tail_tc_plan_build(pl, (const f16*)x, B, H, W))) break;
            rc = tail_tc_launch(pl, stats, w, bias, out, H, W, st);
        } else {
            e = cudaFuncSetAttribute(tail_mma_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, TAILM_SMEM);
            if (e == cudaSuccess)
                e = launch_k(tail_mma_kernel, dim3((W + 31) / 32, (H + 7) / 8, B), dim3(256), TAILM_SMEM, st, (const f16*)x, stats, w, bias, out, H, W, 1);
            if (e != cudaSuccess) rc = fail(-2, cudaGetErrorString(e));
        }
    } while (0);
    cudaError_t e2 = cudaStreamSynchronize(st);
    cudaFree(ws);
    if (rc) return rc;
    B2D_CUDA(e2);
    return 0;
}

int b2d_op_posterior_update(float* x, const float* eps, const float* z, const float* betas, const float* alphas,
                            const float* alpha_hat, int32_t i, int32_t B, int64_t per_sample, uint64_t seed,
                            uint64_t sample_offset, float noise_scale, void* stream) {
    B2D_CHECK(x && eps && betas && alphas && alpha_hat && B >= 1 && per_sample >= 1, "bad argument");
    B2D_CHECK(per_sample % 4 == 0, "per-sample element count must be a multiple of 4 (vectorised update)");
    cudaStream_t st = as_stream(stream);
    // persistent scratch of this entry point (step index + job block): no allocation or synchronisation per call
    struct Scratch { int* step = nullptr; SampleJob* job = nullptr; };
    static thread_local Scratch sc;
    if (!sc.step) {
        B2D_CUDA(cudaMalloc(&sc.step, 16));
        B2D_CUDA(cudaMalloc(&sc.job, sizeof(SampleJob)));
    }
    const size_t n = (size_t)B * per_sample;
    SampleJob job{};
    // z (if given) is the noise of THIS step: bias the pointer so that noise + i*n lands on it
    job.noise = z ? z - (size_t)i * n : nullptr;
    job.seed = seed;
    job.sample_offset = sample_offset;
    job.noise_stride = n;
    job.noise_scale = noise_scale;
    B2D_CUDA(launch_k(set_job_kernel, dim3(1), dim3(32), 0, st, sc.job, job, sc.step + 2, sc.step, (int)i, 0));
    const int blocks = (int)std::min<size_t>((n / 4 + 255) / 256, (size_t)148 * 8);
    B2D_CUDA(launch_k(posterior_update_kernel, dim3(blocks), dim3(256), 0, st, x, eps, sc.job, alphas, betas, alpha_hat, sc.step, nullptr, B, n,
                      (size_t)per_sample));
    B2D_CUDA(cudaGetLastError());
    return 0;
}

int b2d_op_ddim_update(float* x, const float* eps, const float* z_or_null, const float* alpha_hat, int32_t T, int32_t t,
                       int32_t t_prev, float eta, int32_t B, int64_t per_sample, uint64_t seed, uint64_t sample_offset,
                       float noise_scale, void* stream) {
    B2D_CHECK(x && eps && alpha_hat && B >= 1 && per_sample >= 1 && T >= 2, "bad argument");
    B2D_CHECK(per_sample % 4 == 0, "per-sample element count must be a multiple of 4 (vectorised update)");
    B2D_CHECK(t >= 1 && t <= T - 1, "t must lie in [1, T-1]");
    B2D_CHECK(t_prev == -1 || (t_prev >= 1 && t_prev < t), "t_prev must be -1 (final step) or lie in [1, t-1]");
    B2D_CHECK(eta >= 0.f && eta <= 1.f, "eta must lie in [0, 1]");
    cudaStream_t st = as_stream(stream);
    // the coefficients come from the fp32 alpha_hat values the caller's table holds, through the same host function as the
    // handle's per-step table
    float ah[2] = {0.f, 1.f};
    B2D_CUDA(cudaMemcpyAsync(&ah[0], alpha_hat + t, 4, cudaMemcpyDeviceToHost, st));
    if (t_prev >= 1) B2D_CUDA(cudaMemcpyAsync(&ah[1], alpha_hat + t_prev, 4, cudaMemcpyDeviceToHost, st));
    B2D_CUDA(cudaStreamSynchronize(st));
    const float4 c = ddim_coefficients(ah[0], ah[1], eta);
    // persistent scratch of this entry point (step index, job block, one-row tables), written in stream order
    struct Scratch { int* step = nullptr; SampleJob* job = nullptr; int* tau = nullptr; float4* coef = nullptr; };
    static thread_local Scratch sc;
    if (!sc.step) {
        B2D_CUDA(cudaMalloc(&sc.step, 16));
        B2D_CUDA(cudaMalloc(&sc.job, sizeof(SampleJob)));
        B2D_CUDA(cudaMalloc(&sc.tau, 16));
        B2D_CUDA(cudaMalloc(&sc.coef, sizeof(float4)));
    }
    const size_t n = (size_t)B * per_sample;
    SampleJob job{};
    job.noise = z_or_null;   // the noise of THIS step: k = 0
    job.seed = seed;
    job.sample_offset = sample_offset;
    job.noise_stride = n;
    job.noise_scale = noise_scale;
    ddim_op_setup_kernel<<<1, 32, 0, st>>>(sc.job, job, sc.step, sc.tau, sc.coef, (int)t, c);
    B2D_CUDA(cudaGetLastError());
    const int blocks = (int)std::min<size_t>((n / 4 + 255) / 256, (size_t)148 * 8);
    B2D_CUDA(launch_k(ddim_update_kernel, dim3(blocks), dim3(256), 0, st, x, eps, sc.job, sc.tau, sc.coef, sc.step, nullptr, nullptr, B,
                      n, (size_t)per_sample));
    B2D_CUDA(cudaGetLastError());
    return 0;
}

// ------------------------------------------------------------------------------------------------ forward process / loss / evaluation
int b2d_op_noise_image(const float* x0, const int64_t* t_dev, const float* alpha_hat, const float* noise_or_null, float* x_t,
                       float* noise_out, int32_t B, int64_t per_sample, uint64_t seed, uint64_t sample_offset, float noise_scale,
                       void* stream) {
    B2D_CHECK(x0 && t_dev && alpha_hat && x_t && noise_out && B >= 1 && per_sample >= 1, "bad argument");
    B2D_CHECK(per_sample % 4 == 0, "per-sample element count must be a multiple of 4 (vectorised pass)");
    const size_t n = (size_t)B * per_sample;
    const int blocks = (int)std::min<size_t>((n / 4 + 255) / 256, (size_t)148 * 8);
    noise_image_kernel<<<blocks, 256, 0, as_stream(stream)>>>(x0, reinterpret_cast<const long long*>(t_dev), alpha_hat, noise_or_null, x_t,
                                                               noise_out, n, (size_t)per_sample, seed, sample_offset, noise_scale);
    B2D_CUDA(cudaGetLastError());
    return 0;
}

int b2d_op_weighted_mse(const float* input, const float* target, const float* sdf_or_null, float max_land_weight,
                        float min_sea_weight, float* out_scalar_dev, int64_t n, void* stream) {
    B2D_CHECK(input && target && out_scalar_dev && n >= 1, "bad argument");
    static thread_local double* partial = nullptr;       // persistent scratch: no allocation per call
    if (!partial) B2D_CUDA(cudaMalloc(&partial, WMSE_BLOCKS * sizeof(double)));
    const int blocks = (int)std::min<int64_t>((n + 255) / 256, WMSE_BLOCKS);
    cudaStream_t st = as_stream(stream);
    weighted_mse_partial_kernel<<<blocks, 256, 0, st>>>(input, target, sdf_or_null, max_land_weight - min_sea_weight, min_sea_weight,
                                                         partial, (size_t)n);
    weighted_mse_final_kernel<<<1, 256, 0, st>>>(partial, blocks, 1.0 / (double)n, out_scalar_dev);
    B2D_CUDA(cudaGetLastError());
    return 0;
}

int b2d_op_eval_daily(const float* gen, const float* eval, float* mae_out, float* rmse_out, int32_t n_samples, int64_t hw,
                      void* stream) {
    B2D_CHECK(gen && eval && mae_out && rmse_out && n_samples >= 1 && hw >= 1, "bad argument");
    eval_daily_kernel<<<n_samples, 256, 0, as_stream(stream)>>>(gen, eval, mae_out, rmse_out, (size_t)hw);
    B2D_CUDA(cudaGetLastError());
    return 0;
}

int b2d_op_eval_pixel(const float* gen, const float* eval, float* mae_out, float* rmse_out, float* bias_out, int32_t n_samples,
                      int64_t hw, void* stream) {
    B2D_CHECK(gen && eval && mae_out && rmse_out && bias_out && n_samples >= 1 && hw >= 1, "bad argument");
    eval_pixel_kernel<<<(unsigned)((hw + 255) / 256), 256, 0, as_stream(stream)>>>(gen, eval, mae_out, rmse_out, bias_out, n_samples, (size_t)hw);
    B2D_CUDA(cudaGetLastError());
    return 0;
}

int b2d_op_histogram(const float* x, int64_t n, float lo, float hi, int32_t bins, unsigned long long* counts_dev, void* stream) {
    B2D_CHECK(x && counts_dev && n >= 0 && bins >= 1 && bins <= HIST_MAX_BINS && hi > lo, "bad argument");
    cudaStream_t st = as_stream(stream);
    B2D_CUDA(cudaMemsetAsync(counts_dev, 0, (size_t)bins * 8, st));
    if (n == 0) return 0;
    const int blocks = (int)std::min<int64_t>((n + 255) / 256, 148 * 4);
    histogram_kernel<<<blocks, 256, (size_t)bins * 4, st>>>(x, (size_t)n, lo, hi, bins, counts_dev);
    B2D_CUDA(cudaGetLastError());
    return 0;
}

int b2d_debug_attn_trace(long long* out_host, int32_t max_elems) {
    B2D_CHECK(out_host && max_elems >= AT2_TRACE_BLOCKS * 12, "trace buffer too small");
    B2D_CUDA(cudaDeviceSynchronize());
    B2D_CUDA(cudaMemcpyFromSymbol(out_host, g_at2_trace, sizeof(long long) * AT2_TRACE_BLOCKS * 12));
    return AT2_TRACE_BLOCKS;
}

unsigned int b2d_saturation_count(int32_t reset) {
    unsigned int v = 0;
    if (cudaMemcpyFromSymbol(&v, g_sat_count, sizeof(v)) != cudaSuccess) return 0xFFFFFFFFu;
    if (reset) {
        const unsigned int z = 0;
        cudaMemcpyToSymbol(g_sat_count, &z, sizeof(z));
    }
    return v;
}

}  // extern "C"
