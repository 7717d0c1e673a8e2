// C ABI of flocoder_b200 (include/flocoder_b200.h): parameter manifest, weight packing, the
// static op program of the U-Net forward (unet.py:289-372), per-batch plans (workspace, TMA
// tensor maps, CUDA graph) and the device-side integrators (sampling.py:36-122).
#include <cuda_fp16.h>
#include <math.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <algorithm>
#include <chrono>
#include <float.h>
#include <map>
#include <memory>
#include <string>
#include <vector>

#include "flo_internal.h"

namespace flo {

int conv_umma_smem_bytes(const ConvUmmaParams& p);

// ------------------------------------------------------------------------------------------------
// errors
// ------------------------------------------------------------------------------------------------
static thread_local std::string g_last_error;
void set_error(const char* fmt, ...) {
    char buf[1024];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof(buf), fmt, ap);
    va_end(ap);
    g_last_error = buf;
}
#define CUDA_TRY(expr)                                                                       \
    do {                                                                                     \
        cudaError_t _e = (expr);                                                             \
        if (_e != cudaSuccess) {                                                             \
            set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
            return FLO_ERR_CUDA;                                                             \
        }                                                                                    \
    } while (0)

EncodeTiledFn get_encode_tiled() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* sym = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(sym);
    }
    return fn;
}

// ------------------------------------------------------------------------------------------------
// spec + parameter manifest (reference state_dict order, SURVEY.md section 8a)
// ------------------------------------------------------------------------------------------------
struct Spec {
    int dim, channels, n_levels, groups, n_classes, H, W;
    bool bf16;                 // 16-bit tensor-core operand path (bf16 or fp16)
    bool f16;                  // operands are fp16 instead of bf16 (fused path only)
    bool fused;                // fused stage kernels (default for the 16-bit paths)
    bool mask_cond;            // inpainting U-Net: mask-fusion branches (unet.py:214-235), fp32 path only
    int flags, device;
    std::vector<int> dims;     // [dim, dim*m0, dim*m1, ...]   (unet.py:189)
    int time_dim;              // dim*8                         (unet.py:197)
};

struct ParamInfo {
    std::string name;
    std::vector<int64_t> shape;
    int64_t numel() const {
        int64_t n = 1;
        for (auto s : shape) n *= s;
        return n;
    }
};

static int make_spec(const flo_unet_cfg* c, Spec& s) {
    if (!c) { set_error("cfg is NULL"); return FLO_ERR_INVALID; }
    if (c->mask_cond && c->compute_dtype != FLO_F32) {
        set_error("mask_cond=1 (inpainting U-Net, unet.py:214-235) runs on the fp32 path only: its 5x5 / (dim+channels)-input "
                  "fusion convolutions have no tcgen05 stage kernels; use compute_dtype fp32");
        return FLO_ERR_UNSUPPORTED;
    }
    if (c->n_mults < 1 || c->n_mults > 8) { set_error("n_mults must be in 1..8"); return FLO_ERR_INVALID; }
    if (c->dim <= 0 || c->dim % 8) { set_error("dim must be a positive multiple of 8, got %d", c->dim); return FLO_ERR_UNSUPPORTED; }
    if (c->compute_dtype != FLO_F32 && c->compute_dtype != FLO_BF16 && c->compute_dtype != FLO_F16) { set_error("bad compute_dtype"); return FLO_ERR_INVALID; }
    if (c->compute_dtype == FLO_F16 && (c->flags & FLO_FLAG_LAYERWISE)) { set_error("fp16 operands are only available on the fused path"); return FLO_ERR_UNSUPPORTED; }
    if (c->compute_dtype != FLO_F32 && c->dim % 16) {
        set_error("the bf16 tcgen05 path needs dim %% 16 == 0 (K slices of 16 channels), got %d", c->dim);
        return FLO_ERR_UNSUPPORTED;
    }
    if (c->mask_cond && c->channels > 8) { set_error("mask_cond needs channels <= 8"); return FLO_ERR_UNSUPPORTED; }
    if (c->channels < 1 || c->channels > 16) { set_error("channels must be in 1..16"); return FLO_ERR_UNSUPPORTED; }
    if (c->dim > 64) { set_error("dim > 64 is not supported by the final-conv kernel"); return FLO_ERR_UNSUPPORTED; }
    if (c->n_classes < 0) { set_error("n_classes < 0"); return FLO_ERR_INVALID; }
    s.dim = c->dim; s.channels = c->channels; s.n_levels = c->n_mults; s.groups = c->groups;
    s.n_classes = c->n_classes; s.H = c->height; s.W = c->width; s.bf16 = c->compute_dtype != FLO_F32;
    s.f16 = c->compute_dtype == FLO_F16;
    s.mask_cond = c->mask_cond != 0;
    // fused stage kernels: latent channels <= 4 (registers of the final epilogue); otherwise the layer-wise tcgen05 path
    s.fused = s.bf16 && !(c->flags & FLO_FLAG_LAYERWISE) && c->channels <= 4;
    s.flags = c->flags; s.device = c->device;
    s.dims.clear();
    s.dims.push_back(c->dim);
    for (int i = 0; i < c->n_mults; ++i) {
        if (c->mults[i] < 1) { set_error("dim_mults must be >= 1"); return FLO_ERR_INVALID; }
        s.dims.push_back(c->dim * c->mults[i]);
    }
    s.time_dim = c->dim * 8;
    const int div = 1 << (c->n_mults - 1);
    if (s.H <= 0 || s.W <= 0 || s.H % div || s.W % div) {
        set_error("latent %dx%d is not divisible by 2^(levels-1)=%d", s.H, s.W, div);
        return FLO_ERR_INVALID;
    }
    if (s.H * s.W > 256 && (s.bf16 || (s.H * s.W) % 256 || s.H * s.W > 4096)) {
        set_error("latents larger than 256 pixels run on the fp32 path only (tiled linear attention), with H*W a multiple of 256 up to 4096");
        return FLO_ERR_UNSUPPORTED;
    }
    if (s.groups < 1) { set_error("groups < 1"); return FLO_ERR_INVALID; }
    for (size_t i = 0; i < s.dims.size(); ++i) {
        const int C = s.dims[i];
        if (C % s.groups) { set_error("channels %d not divisible by groups %d", C, s.groups); return FLO_ERR_INVALID; }
        const int cpg = C / s.groups;
        // the fp32 path has a generic GroupNorm kernel (k_gn_any); the 16-bit paths pack whole sectors per group
        if (s.bf16 && cpg != 4 && cpg % 8) { set_error("channels per group must be 4 or a multiple of 8 on the 16-bit paths, got %d", cpg); return FLO_ERR_UNSUPPORTED; }
    }
    return FLO_OK;
}

static void add_conv(std::vector<ParamInfo>& v, const std::string& p, int co, int ci, int k, bool bias = true) {
    v.push_back({p + ".weight", {co, ci, k, k}});
    if (bias) v.push_back({p + ".bias", {co}});
}
static void add_linear(std::vector<ParamInfo>& v, const std::string& p, int out, int in) {
    v.push_back({p + ".weight", {out, in}});
    v.push_back({p + ".bias", {out}});
}
static void add_norm(std::vector<ParamInfo>& v, const std::string& p, int c) {
    v.push_back({p + ".weight", {c}});
    v.push_back({p + ".bias", {c}});
}
static void add_resnet(std::vector<ParamInfo>& v, const std::string& p, int din, int dout, int tdim) {
    add_linear(v, p + ".mlp.1", 2 * dout, tdim);
    add_conv(v, p + ".block1.proj", dout, din, 3);
    add_norm(v, p + ".block1.norm", dout);
    add_conv(v, p + ".block2.proj", dout, dout, 3);
    add_norm(v, p + ".block2.norm", dout);
    if (din != dout) add_conv(v, p + ".res_conv", dout, din, 1);
}
static void add_attn(std::vector<ParamInfo>& v, const std::string& p, int dim, bool linear) {
    add_conv(v, p + ".fn.fn.to_qkv", 384, dim, 1, false);
    if (linear) {
        add_conv(v, p + ".fn.fn.to_out.0", dim, 128, 1);
        add_norm(v, p + ".fn.fn.to_out.1", dim);
    } else {
        add_conv(v, p + ".fn.fn.to_out", dim, 128, 1);
    }
    add_norm(v, p + ".fn.norm", dim);
}
static std::vector<ParamInfo> manifest(const Spec& s) {
    std::vector<ParamInfo> v;
    const int n = s.n_levels, td = s.time_dim;
    add_conv(v, "init_conv", s.dim, s.channels, 1);
    add_linear(v, "time_mlp.1", td, s.dim);
    add_linear(v, "time_mlp.3", td, td);
    if (s.n_classes > 0) {
        v.push_back({"class_cond_mlp.0.weight", {s.n_classes, td}});
        add_linear(v, "class_cond_mlp.1", td, td);
        add_linear(v, "class_cond_mlp.3", td, td);
    }
    if (s.mask_cond) {                      // unet.py:214-235 (registered before downs / ups)
        add_conv(v, "mask_fusion_conv.0", 2 * s.dim, s.dim + s.channels, 5);
        add_conv(v, "mask_fusion_conv.2", 2 * s.dim, 2 * s.dim, 3);
        add_conv(v, "mask_fusion_conv.4", s.dim, 2 * s.dim, 3);
        for (int i = 0; i < std::min(2, n); ++i) add_conv(v, "down_mask_fusions." + std::to_string(i) + ".0", s.dims[i], s.dims[i] + s.channels, 3);
        for (int i = 0; i < std::min(2, n); ++i) add_conv(v, "up_mask_fusions." + std::to_string(i) + ".0", s.dims[n - i], s.dims[n - i] + s.channels, 3);
    }
    for (int l = 0; l < n; ++l) {
        const int din = s.dims[l], dout = s.dims[l + 1];
        const std::string p = "downs." + std::to_string(l);
        add_resnet(v, p + ".0", din, din, td);
        add_resnet(v, p + ".1", din, din, td);
        add_attn(v, p + ".2", din, true);
        if (l < n - 1) add_conv(v, p + ".3.1", dout, din * 4, 1);
        else add_conv(v, p + ".3", dout, din, 3);
    }
    for (int i = 0; i < n; ++i) {
        const int l = n - 1 - i, din = s.dims[l], dout = s.dims[l + 1];
        const std::string p = "ups." + std::to_string(i);
        add_resnet(v, p + ".0", dout + din, dout, td);
        add_resnet(v, p + ".1", dout + din, dout, td);
        add_attn(v, p + ".2", dout, true);
        if (i < n - 1) add_conv(v, p + ".3.1", din, dout, 3);
        else add_conv(v, p + ".3", din, dout, 3);
    }
    const int mid = s.dims[n];
    add_resnet(v, "mid_block1", mid, mid, td);
    add_attn(v, "mid_attn", mid, false);
    add_resnet(v, "mid_block2", mid, mid, td);
    add_resnet(v, "final_res_block", 2 * s.dim, s.dim, td);
    add_conv(v, "final_conv", s.channels, s.dim, 1);
    return v;
}

// ------------------------------------------------------------------------------------------------
// program: buffers + ops
// ------------------------------------------------------------------------------------------------
struct Buf {
    std::string name;
    int C, H, W;
    bool bf16;
    size_t bytes_ps;     // bytes per sample
    int def = -1, last = -1;
    size_t off_ps = 0;   // offset (bytes per sample) inside the activation arena
};
struct Val {             // a logical tensor: fp32 master and/or operand copy (same buffer in fp32 mode)
    int m = -1, o = -1, un = -1, up = -1;
    int C = 0, H = 0, W = 0;
};
enum OpKind { OP_INIT, OP_CONV, OP_GN, OP_LINATTN, OP_MIDATTN, OP_FINAL };
static const size_t NONE = (size_t)-1;
struct Op {
    int kind;
    std::string name;
    std::string pname;        // parameter prefix of a conv ('<pname>.weight')
    bool unshuf_in = false;   // conv input is the pixel-unshuffled tensor in (p1 p2 c) channel order
    // conv
    int in0 = -1, in1 = -1, ncb0 = 0, ncb1 = 0, cout = 0, ksize = 0, H = 0, W = 0;
    size_t w_simt = NONE, w_umma = NONE, bias = NONE;
    int n_tile = 0;
    int res = -1, out_m = -1, out_o = -1;
    int act_silu = 0, need_mode = 0, bypass = -1;   // mask-fusion convs (fp32 path)
    // gn
    int gn_in = -1, C = 0, groups = 0, film_off = -1, silu = 0, out_un = -1, out_up = -1;
    size_t gamma = NONE, beta = NONE;
    // attention
    int qkv = -1, attn_out = -1, n = 0;
};

// ---- fused path (fused_plan.inc)
struct FTensor {
    std::string name;
    int C, H, W;
    size_t bytes_ps, off_ps;
};
struct FStage {
    int kind;                 // 0 = k_chain, 1 = k_attn
    std::string name;
    ChainParams cp;
    AttnFusedParams ap;
    int nb;
    int n_maps;
    int map_tensor[CH_MAX_LOADS];   // tensors loaded by TMA (chain: padded box, attn: plain box)
    int gt_tensor[CH_MAX_GT];       // chain: global tensor table -> tensor ids (-1 unused)
    int x2_t, out_t, out_un_t, out_up_t;   // attn
};

struct Handle;
struct Plan {
    int B = 0;
    uint8_t* arena = nullptr;          // activations
    size_t arena_bytes = 0;
    float *y = nullptr, *acc = nullptr, *xs = nullptr, *vcond = nullptr, *film_ps = nullptr;
    int64_t* cls = nullptr;
    Ctrl* ctrl = nullptr;
    int* pair_flags = nullptr;         // [B] arrival counters of the single-pass CFG combine (SF_CFG_2B; this plan's batch = 2 x caller's)
    cudaGraphExec_t graph_c = nullptr, graph_c4 = nullptr;   // k_temb (stage time from the control block) + one / four forwards
    int graph_c_cond = -1;             // conditional rows the captured k_temb node was built for
    int* mask_mode = nullptr;          // 0 no mask (default), 1 mask of all ones, 2 mask in use (flo_unet_set_mask)
    std::vector<void*> buf_ptr;
    std::vector<ConvUmmaParams> umma;   // per op (valid for conv ops on the bf16 path)
    std::vector<CUtensorMap> tmA0, tmA1;
    cudaGraphExec_t graph = nullptr;        // one forward
    cudaGraphExec_t graph4 = nullptr;       // four forwards back to back (one RK4 interval): the dependent-launch chain then
                                            // also covers final stage -> first stage of the next evaluation
    size_t total_bytes = 0;
    uint8_t* base = nullptr;
    // fused path
    uint8_t* farena = nullptr;
    std::vector<CUtensorMap> fstage_maps;
    int fvar = 0;                           // which Handle::stages() variant this plan runs
    std::vector<ChainParams> fchain;
    std::vector<AttnFusedParams> fattn;
    long long* dbg = nullptr;
    uint64_t last_use = 0;                  // LRU stamp (Handle::use_ctr)
    // RK45 (flo_integrate_rk45), allocated on first use: K [7][n] | y, y_new [2][n] | controller | partial sums
    float* rk_buf = nullptr;
    Rk45Ctl* rk_ctl = nullptr;
    double* rk_part = nullptr;
    cudaGraphExec_t graph_rk = nullptr;     // one attempt: [k_rk45_stage -> k_temb -> forward] x 6 -> k_rk45_end
    int64_t graph_rk_key = -1;
    Plan() = default;
    Plan(const Plan&) = delete;
    Plan& operator=(const Plan&) = delete;
    ~Plan() {                               // every exit path of get_plan releases what it has allocated so far
        if (graph) cudaGraphExecDestroy(graph);
        if (graph4) cudaGraphExecDestroy(graph4);
        if (graph_c) cudaGraphExecDestroy(graph_c);
        if (graph_c4) cudaGraphExecDestroy(graph_c4);
        if (graph_rk) cudaGraphExecDestroy(graph_rk);
        if (rk_buf) cudaFree(rk_buf);
        if (base) cudaFree(base);
        if (dbg) cudaFree(dbg);
    }
};
constexpr size_t MAX_PLANS = 8;             // per-batch-size plans kept per handle (least recently used one is evicted)

struct Handle {
    Spec spec;
    std::vector<ParamInfo> params;
    std::map<std::string, std::vector<float>> host;     // fp32 parameters on the host (packing source)
    std::vector<float> blob_f32;                        // packed fp32 constants
    std::vector<__nv_bfloat16> blob_bf16;               // packed tcgen05 weight streams
    float* d_f32 = nullptr;
    __nv_bfloat16* d_bf16 = nullptr;
    std::vector<Buf> bufs;
    std::vector<Op> ops;
    int film_dim = 0;
    size_t arena_ps = 0;                                // activation arena bytes per sample
    // temb constants (offsets into blob_f32)
    size_t o_freqs, o_w1t, o_b1, o_w2t, o_b2, o_emb = NONE, o_wc1t = NONE, o_bc1 = NONE, o_wc3t = NONE, o_bc3 = NONE,
           o_wft, o_bf, o_init_w, o_init_b, o_final_w, o_final_b;
    std::map<int, std::unique_ptr<Plan>> plans;
    uint64_t use_ctr = 0;
    cudaStream_t last_stream = nullptr;     // a handle serves one stream at a time: calls on another stream first wait for this one
    bool has_last_stream = false;
    // stage tables
    Stage* d_stages = nullptr; float* d_stage_t = nullptr; float* d_film_u = nullptr;
    int stage_cap = 0;
    Stage* h_stages[4] = {nullptr, nullptr, nullptr, nullptr}; float* h_stage_t[4] = {nullptr, nullptr, nullptr, nullptr};
    cudaEvent_t h_ev[4] = {nullptr, nullptr, nullptr, nullptr};
    int h_cap = 0, h_next = 0;
    cudaStream_t capture_stream = nullptr;
    int64_t launches = 0;
    Val r_val;
    int mask_buf[8] = {-1, -1, -1, -1, -1, -1, -1, -1};   // per-level blocked mask tensors (mask_cond)
    std::vector<FTensor> ftensors;
    std::vector<FStage> fstages;            // variant 0: N-split of the low-resolution chain stages up to 4 CTAs
    std::vector<FStage> fstages_alt[2];     // variants 1, 2: N-split capped at 2 / none (picked per batch size so the
                                            // split stages still fit the GPU in one wave)
    const std::vector<FStage>& stages(int variant) const { return variant == 0 ? fstages : fstages_alt[variant - 1]; }
    size_t farena_ps = 0;
    // RK45 host side: pinned status record, events around every attempt, timing of the last call
    Rk45Status* h_rk = nullptr;
    cudaEvent_t rk_ev[3] = {nullptr, nullptr, nullptr};
    double rk_timing[3] = {0, 0, 0};        // attempts, host wall ms, graph ms (CUDA events)
    Handle() = default;
    Handle(const Handle&) = delete;
    Handle& operator=(const Handle&) = delete;
    ~Handle() {                   // also runs on every early return of flo_unet_create (the handle lives in a unique_ptr there)
        plans.clear();
        if (d_f32) cudaFree(d_f32);
        if (d_bf16) cudaFree(d_bf16);
        if (d_stages) { cudaFree(d_stages); cudaFree(d_stage_t); cudaFree(d_film_u); }
        for (int i = 0; i < 4; ++i) {
            if (h_stages[i]) { cudaFreeHost(h_stages[i]); cudaFreeHost(h_stage_t[i]); }
            if (h_ev[i]) cudaEventDestroy(h_ev[i]);
        }
        if (h_rk) cudaFreeHost(h_rk);
        for (auto& e : rk_ev) if (e) cudaEventDestroy(e);
        if (capture_stream) cudaStreamDestroy(capture_stream);
    }
};

// ---- program builder ---------------------------------------------------------------------------
struct Builder {
    Handle& h;
    const Spec& s;
    int film_dim = 0;
    explicit Builder(Handle& hh) : h(hh), s(hh.spec) {}

    int newbuf(const std::string& name, int C, int H, int W, bool bf16) {
        Buf b;
        b.name = name; b.C = C; b.H = H; b.W = W; b.bf16 = bf16;
        b.bytes_ps = (size_t)C * H * W * (bf16 ? 2 : 4);
        h.bufs.push_back(b);
        return (int)h.bufs.size() - 1;
    }
    Val newval(const std::string& name, int C, int H, int W, bool need_m, bool need_o) {
        Val v; v.C = C; v.H = H; v.W = W;
        if (!s.bf16) { v.m = v.o = newbuf(name, C, H, W, false); }
        else {
            if (need_m) v.m = newbuf(name + ":m", C, H, W, false);
            if (need_o) v.o = newbuf(name + ":o", C, H, W, true);
        }
        return v;
    }
    void def(int b) { if (b >= 0 && h.bufs[b].def < 0) h.bufs[b].def = (int)h.ops.size(); if (b >= 0) h.bufs[b].last = std::max(h.bufs[b].last, (int)h.ops.size()); }
    void use(int b) { if (b >= 0) h.bufs[b].last = std::max(h.bufs[b].last, (int)h.ops.size()); }

    size_t put_f32(const float* src, size_t n) {
        size_t off = (h.blob_f32.size() + 7) & ~(size_t)7;
        h.blob_f32.resize(off + n);
        memcpy(h.blob_f32.data() + off, src, n * sizeof(float));
        return off;
    }
    const std::vector<float>& P(const std::string& name) { return h.host.at(name); }
    size_t put_param(const std::string& name) { const auto& v = P(name); return put_f32(v.data(), v.size()); }
    // [out][in] -> [in][out]
    size_t put_transposed(const std::string& name, int out, int in) {
        const auto& w = P(name);
        std::vector<float> t((size_t)out * in);
        for (int o = 0; o < out; ++o) for (int i = 0; i < in; ++i) t[(size_t)i * out + o] = w[(size_t)o * in + i];
        return put_f32(t.data(), t.size());
    }

    // conv with optional second (concatenated) source; perm maps OUR input-channel order to the reference's
    struct ConvExtra {          // mask-fusion convs: C1 holds c1_real reference channels (the rest of the block is padding)
        int c1_real = -1; bool silu = false; int need_mode = 0; int bypass = -1; bool want_un = false, want_up = false;
    };
    Val conv(const std::string& pname, const std::string& vname, int in0, int C0, int in1, int C1, int H, int W,
             int cout, int ksize, bool bias, bool need_m, bool need_o, int res_m = -1, const std::vector<int>* perm = nullptr,
             const ConvExtra* ex = nullptr) {
        Op op; op.kind = OP_CONV; op.name = vname; op.pname = pname; op.unshuf_in = perm != nullptr;
        const int c1_real = (ex && ex->c1_real >= 0) ? ex->c1_real : C1, cin_ref = C0 + c1_real;
        if (ex) { op.act_silu = ex->silu; op.need_mode = ex->need_mode; op.bypass = ex->bypass; }
        op.in0 = in0; op.in1 = in1; op.ncb0 = C0 / 8; op.ncb1 = C1 / 8; op.cout = cout; op.ksize = ksize; op.H = H; op.W = W;
        const int cin = C0 + C1, taps = ksize * ksize;
        const auto& w = P(pname + ".weight");
        {   // SIMT layout [tap][cin][cout]; always packed (fp32 path, and the self-test reference)
            std::vector<float> t((size_t)taps * cin * cout);
            for (int co = 0; co < cout; ++co)
                for (int ci = 0; ci < cin; ++ci) {
                    const int cref = perm ? (*perm)[ci] : ci;
                    if (cref >= cin_ref) continue;                    // padding channels of the mask block: zero weights
                    for (int tp = 0; tp < taps; ++tp)
                        t[((size_t)tp * cin + ci) * cout + co] = w[((size_t)co * cin_ref + cref) * taps + tp];
                }
            op.w_simt = put_f32(t.data(), t.size());
        }
        if (s.bf16) {
            int n_tile = cout;
            if (cout > 256) n_tile = 128;
            if (cout % n_tile || n_tile % 16 || cin % 16) { /* falls back to an explicit error at plan time */ n_tile = 0; }
            op.n_tile = n_tile;
            if (n_tile) {
                size_t off = (h.blob_bf16.size() + 63) & ~(size_t)63;     // 128-byte aligned streams
                h.blob_bf16.resize(off);
                pack_umma_weights(w.data(), cout, cin, ksize, perm ? perm->data() : nullptr, n_tile, s.f16, h.blob_bf16);
                op.w_umma = off;
            }
        }
        if (bias) op.bias = put_param(pname + ".bias");
        Val out = newval(vname, cout, H, W, need_m, need_o);
        if (ex && ex->want_un) out.un = newbuf(vname + ":unshuf", cout * 4, H / 2, W / 2, s.bf16);
        if (ex && ex->want_up) out.up = newbuf(vname + ":up", cout, H * 2, W * 2, s.bf16);
        use(in0); use(in1); use(res_m); use(op.bypass);
        op.res = res_m; op.out_m = out.m; op.out_o = (out.o != out.m) ? out.o : -1;
        op.out_un = out.un; op.out_up = out.up;
        def(out.m); def(out.o); def(out.un); def(out.up);
        h.ops.push_back(op);
        return out;
    }
    Val gn(const std::string& pname, const std::string& vname, const Val& in, int groups, int film_off, bool silu,
           int res_m, bool need_m, bool need_o, bool want_un = false, bool want_up = false) {
        Op op; op.kind = OP_GN; op.name = vname;
        op.gn_in = in.m; op.C = in.C; op.H = in.H; op.W = in.W; op.groups = groups; op.film_off = film_off; op.silu = silu;
        op.gamma = put_param(pname + ".weight"); op.beta = put_param(pname + ".bias");
        Val out = newval(vname, in.C, in.H, in.W, need_m, need_o);
        if (want_un) out.un = newbuf(vname + ":unshuf", in.C * 4, in.H / 2, in.W / 2, s.bf16);
        if (want_up) out.up = newbuf(vname + ":up", in.C, in.H * 2, in.W * 2, s.bf16);
        use(in.m); use(res_m);
        op.res = res_m;
        if (!s.bf16) { op.out_m = -1; op.out_o = out.o; }
        else { op.out_m = out.m; op.out_o = out.o; }
        op.out_un = out.un; op.out_up = out.up;
        def(out.m); def(out.o); def(out.un); def(out.up);
        h.ops.push_back(op);
        return out;
    }
    // ResnetBlock (unet.py:88-96); x1 = second concat source or empty Val
    Val resblock(const std::string& p, const Val& x0, const Val& x1, int dout, bool out_m, bool out_o,
                 std::vector<std::pair<std::string, int>>& film_layout) {
        const int C1 = x1.o >= 0 ? x1.C : 0, cin = x0.C + C1, H = x0.H, W = x0.W;
        const int foff = film_dim;
        film_dim += 2 * dout;
        film_layout.push_back({p + ".mlp.1", dout});
        Val c1 = conv(p + ".block1.proj", p + ".block1.proj", x0.o, x0.C, C1 ? x1.o : -1, C1, H, W, dout, 3, true, true, false);
        Val g1 = gn(p + ".block1.norm", p + ".block1", c1, s.groups, foff, true, -1, false, true);
        Val c2 = conv(p + ".block2.proj", p + ".block2.proj", g1.o, dout, -1, 0, H, W, dout, 3, true, true, false);
        int res_m;
        if (cin != dout) {
            Val rc = conv(p + ".res_conv", p + ".res_conv", x0.o, x0.C, C1 ? x1.o : -1, C1, H, W, dout, 1, true, true, false);
            res_m = rc.m;
        } else {
            res_m = x0.m;     // identity residual needs the fp32 master copy of the block input
        }
        return gn(p + ".block2.norm", p, c2, s.groups, -1, true, res_m, out_m, out_o);
    }
    Val attn_core(const std::string& vname, const Val& qkv, bool linear) {
        Op op; op.kind = linear ? OP_LINATTN : OP_MIDATTN; op.name = vname;
        op.qkv = qkv.o; op.n = qkv.H * qkv.W; op.H = qkv.H; op.W = qkv.W;
        Val out = newval(vname, 128, qkv.H, qkv.W, false, true);
        use(qkv.o);
        op.attn_out = out.o;
        def(out.o);
        h.ops.push_back(op);
        return out;
    }
    // Residual(PreNorm(dim, LinearAttention(dim)))   (unet.py:33-39,135-161)
    Val linattn(const std::string& p, const Val& x, bool out_m, bool out_o, bool want_un, bool want_up) {
        Val n1 = gn(p + ".fn.norm", p + ".fn.norm", x, 1, -1, false, -1, false, true);
        Val qkv = conv(p + ".fn.fn.to_qkv", p + ".fn.fn.to_qkv", n1.o, x.C, -1, 0, x.H, x.W, 384, 1, false, false, true);
        Val a = attn_core(p + ".fn.fn.attn", qkv, true);
        Val po = conv(p + ".fn.fn.to_out.0", p + ".fn.fn.to_out.0", a.o, 128, -1, 0, x.H, x.W, x.C, 1, true, true, false);
        return gn(p + ".fn.fn.to_out.1", p, po, 1, -1, false, x.m, out_m, out_o, want_un, want_up);
    }
    // Residual(PreNorm(dim, Attention(dim)))   (unet.py:108-122)
    Val midattn(const std::string& p, const Val& x, bool out_m, bool out_o) {
        Val n1 = gn(p + ".fn.norm", p + ".fn.norm", x, 1, -1, false, -1, false, true);
        Val qkv = conv(p + ".fn.fn.to_qkv", p + ".fn.fn.to_qkv", n1.o, x.C, -1, 0, x.H, x.W, 384, 1, false, false, true);
        Val a = attn_core(p + ".fn.fn.attn", qkv, false);
        return conv(p + ".fn.fn.to_out", p, a.o, 128, -1, 0, x.H, x.W, x.C, 1, true, out_m, out_o, x.m);
    }

    int build() {
        const int n = s.n_levels;
        std::vector<std::pair<std::string, int>> film_layout;
        // ---- init conv
        Val x;
        {
            Op op; op.kind = OP_INIT; op.name = "init_conv"; op.H = s.H; op.W = s.W;
            h.o_init_w = put_param("init_conv.weight");
            h.o_init_b = put_param("init_conv.bias");
            x = newval("init_conv", s.dim, s.H, s.W, true, true);
            op.out_m = s.bf16 ? x.m : -1; op.out_o = x.o;
            def(x.m); def(x.o);
            h.ops.push_back(op);
        }
        const int n_mask = s.mask_cond ? std::min(2, n) : 0;      // levels with a down / up mask fusion (unet.py:225,232)
        if (s.mask_cond) {
            // per-level blocked copies of cond['mask_cond'] (8-channel block, zero padded), filled by flo_unet_set_mask;
            // never (re)defined by an op, so the arena keeps them for the whole program
            for (int l = 0; l < n; ++l) h.mask_buf[l] = newbuf("mask_cond:" + std::to_string(l), 8, s.H >> l, s.W >> l, false);
            // x = mask_fusion_conv(cat(x, mask))   (unet.py:298-305; no residual; skipped when the mask is all ones)
            ConvExtra e0; e0.c1_real = s.channels; e0.silu = true; e0.need_mode = 2;
            Val f0 = conv("mask_fusion_conv.0", "mask_fusion_conv.0", x.o, s.dim, h.mask_buf[0], 8, s.H, s.W, 2 * s.dim, 5, true, true, true, -1, nullptr, &e0);
            ConvExtra e1; e1.silu = true; e1.need_mode = 2;
            Val f1 = conv("mask_fusion_conv.2", "mask_fusion_conv.2", f0.o, 2 * s.dim, -1, 0, s.H, s.W, 2 * s.dim, 3, true, true, true, -1, nullptr, &e1);
            ConvExtra e2; e2.need_mode = 2; e2.bypass = x.m;
            x = conv("mask_fusion_conv.4", "mask_fusion_conv", f1.o, 2 * s.dim, -1, 0, s.H, s.W, s.dim, 3, true, true, true, -1, nullptr, &e2);
        }
        Val r = x;
        Val none;
        std::vector<Val> skips;
        int H = s.H, W = s.W;
        for (int l = 0; l < n; ++l) {
            const int din = s.dims[l], dout = s.dims[l + 1];
            const std::string p = "downs." + std::to_string(l);
            const bool last = l == n - 1;
            Val x1 = resblock(p + ".0", x, none, din, true, true, film_layout);
            skips.push_back(x1);
            Val x2 = resblock(p + ".1", x1, none, din, true, false, film_layout);
            const bool fuse = l < n_mask;
            Val x3 = linattn(p + ".2", x2, fuse, true, !last && !fuse, false);
            skips.push_back(x3);
            if (fuse) {
                // x = x + SiLU(conv3x3(cat(x, resize(mask))))   (unet.py:336-340); the skip above keeps the un-fused x
                ConvExtra e; e.c1_real = s.channels; e.silu = true; e.need_mode = 1; e.bypass = x3.m; e.want_un = !last;
                const std::string mp = "down_mask_fusions." + std::to_string(l) + ".0";
                x3 = conv(mp, mp, x3.o, din, h.mask_buf[l], 8, H, W, din, 3, true, true, true, x3.m, nullptr, &e);
            }
            if (!last) {
                // our unshuffled channel order is (p1 p2 c); the reference's is (c p1 p2)  (unet.py:52)
                std::vector<int> perm(din * 4);
                for (int q = 0; q < 4; ++q) for (int c = 0; c < din; ++c) perm[q * din + c] = c * 4 + q;
                x = conv(p + ".3.1", p + ".3", x3.un, din * 4, -1, 0, H / 2, W / 2, dout, 1, true, true, true, -1, &perm);
                H /= 2; W /= 2;
            } else {
                x = conv(p + ".3", p + ".3", x3.o, din, -1, 0, H, W, dout, 3, true, true, true);
            }
        }
        const int mid = s.dims[n];
        x = resblock("mid_block1", x, none, mid, true, false, film_layout);
        x = midattn("mid_attn", x, true, true);
        x = resblock("mid_block2", x, none, mid, false, true, film_layout);
        for (int i = 0; i < n; ++i) {
            const int l = n - 1 - i, din = s.dims[l], dout = s.dims[l + 1];
            const std::string p = "ups." + std::to_string(i);
            const bool last = i == n - 1;
            Val sk = skips.back(); skips.pop_back();
            x = resblock(p + ".0", x, sk, dout, false, true, film_layout);
            sk = skips.back(); skips.pop_back();
            x = resblock(p + ".1", x, sk, dout, true, false, film_layout);
            const bool fuse = i < n_mask;
            x = linattn(p + ".2", x, fuse, last || fuse, false, !last && !fuse);
            if (fuse) {
                // unet.py:360-364, at the resolution of this up level (mask level l)
                ConvExtra e; e.c1_real = s.channels; e.silu = true; e.need_mode = 1; e.bypass = x.m; e.want_up = !last;
                const std::string mp = "up_mask_fusions." + std::to_string(i) + ".0";
                x = conv(mp, mp, x.o, dout, h.mask_buf[l], 8, H, W, dout, 3, true, true, true, x.m, nullptr, &e);
            }
            if (!last) {
                x = conv(p + ".3.1", p + ".3", x.up, dout, -1, 0, H * 2, W * 2, din, 3, true, false, true);
                H *= 2; W *= 2;
            } else {
                x = conv(p + ".3", p + ".3", x.o, dout, -1, 0, H, W, din, 3, true, false, true);
            }
        }
        x = resblock("final_res_block", x, r, s.dim, true, false, film_layout);
        {
            Op op; op.kind = OP_FINAL; op.name = "final_conv"; op.H = s.H; op.W = s.W;
            op.gn_in = x.m;
            use(x.m);
            h.o_final_w = put_param("final_conv.weight");
            h.o_final_b = put_param("final_conv.bias");
            h.ops.push_back(op);
        }
        h.film_dim = film_dim;
        h.r_val = r;

        // ---- time-embedding constants
        {
            const int half = s.dim / 2, td = s.time_dim;
            std::vector<float> f(half);
            const double c = log(10000.0) / (half - 1);
            for (int j = 0; j < half; ++j) f[j] = (float)exp((double)((float)j * (float)(-c)));   // unet.py:26-27
            h.o_freqs = put_f32(f.data(), f.size());
            h.o_w1t = put_transposed("time_mlp.1.weight", td, s.dim); h.o_b1 = put_param("time_mlp.1.bias");
            h.o_w2t = put_transposed("time_mlp.3.weight", td, td);    h.o_b2 = put_param("time_mlp.3.bias");
            if (s.n_classes > 0) {
                h.o_emb = put_param("class_cond_mlp.0.weight");
                h.o_wc1t = put_transposed("class_cond_mlp.1.weight", td, td); h.o_bc1 = put_param("class_cond_mlp.1.bias");
                h.o_wc3t = put_transposed("class_cond_mlp.3.weight", td, td); h.o_bc3 = put_param("class_cond_mlp.3.bias");
            }
            std::vector<float> wft((size_t)td * film_dim), bf(film_dim);
            int off = 0;
            for (auto& fl : film_layout) {
                const auto& w = P(fl.first + ".weight");     // [2*dout][td]
                const auto& b = P(fl.first + ".bias");
                const int rows = 2 * fl.second;
                for (int o = 0; o < rows; ++o) {
                    bf[off + o] = b[o];
                    for (int i = 0; i < td; ++i) wft[(size_t)i * film_dim + off + o] = w[(size_t)o * td + i];
                }
                off += rows;
            }
            h.o_wft = put_f32(wft.data(), wft.size());
            h.o_bf = put_f32(bf.data(), bf.size());
        }
        return FLO_OK;
    }
};

// ---- kernels of the layer-by-layer program ----------------------------------------------------
// launch_op runs each op with one kernel, chosen from the op's shape alone: refuse at plan time an op no kernel can run, so
// that a forward never starts on it.  The fused path runs its own stage kernels; its planner (fused_plan.inc) checks them.
static int check_op_kernels(const Handle& h) {
    const Spec& s = h.spec;
    if (s.fused) return FLO_OK;
    const char* path = s.bf16 ? "the layer-wise 16-bit path" : "the fp32 path";
    for (const Op& op : h.ops) {
        if (op.kind == OP_GN && gn_variant(op.C, op.H, op.W, op.groups, s.bf16) == GN_NONE) {
            set_error("GroupNorm '%s' (C=%d, %dx%d, groups=%d) has no kernel on %s: its 16-bit kernels need W, H*W and the "
                      "groups (or channel-block pairs of 4-channel groups) per sample to be powers of two, and at most 8192 "
                      "elements per group", op.name.c_str(), op.C, op.H, op.W, op.groups, path);
            return FLO_ERR_UNSUPPORTED;
        }
        if (op.kind == OP_MIDATTN && !midattn_supported(op.n)) {
            set_error("mid attention '%s' at %dx%d (n=%d) has no kernel on %s: it holds at most 64 pixels", op.name.c_str(), op.H,
                      op.W, op.n, path);
            return FLO_ERR_UNSUPPORTED;
        }
        if (op.kind == OP_LINATTN && !linattn_supported(op.n, s.bf16)) {
            set_error("linear attention '%s' at %dx%d (n=%d) has no kernel on %s: more than 256 pixels need fp32 and a multiple "
                      "of 256", op.name.c_str(), op.H, op.W, op.n, path);
            return FLO_ERR_UNSUPPORTED;
        }
    }
    return FLO_OK;
}

// ---- activation arena: linear-scan allocation over buffer live ranges ---------------------------
static void allocate_arena(Handle& h) {
    const bool reuse = !(h.spec.flags & FLO_FLAG_NO_BUFFER_REUSE);
    struct Free { size_t off, size; };
    std::vector<Free> free_list;
    size_t top = 0;
    auto align = [](size_t x) { return (x + 255) & ~(size_t)255; };
    const int n_ops = (int)h.ops.size();
    // skip/long-lived buffers keep their space until their last use; process in op order
    std::vector<std::vector<int>> def_at(n_ops + 1), die_at(n_ops + 1);
    for (int i = 0; i < (int)h.bufs.size(); ++i) {
        Buf& b = h.bufs[i];
        if (b.def < 0) { b.def = 0; b.last = n_ops; }
        def_at[b.def].push_back(i);
        die_at[std::min(b.last, n_ops)].push_back(i);
    }
    for (int op = 0; op <= n_ops; ++op) {
        for (int i : def_at[op]) {
            Buf& b = h.bufs[i];
            const size_t need = align(b.bytes_ps);
            bool placed = false;
            if (reuse) {
                int best = -1;
                for (int f = 0; f < (int)free_list.size(); ++f)
                    if (free_list[f].size >= need && (best < 0 || free_list[f].size < free_list[best].size)) best = f;
                if (best >= 0) {
                    b.off_ps = free_list[best].off;
                    free_list[best].off += need; free_list[best].size -= need;
                    if (free_list[best].size == 0) free_list.erase(free_list.begin() + best);
                    placed = true;
                }
            }
            if (!placed) { b.off_ps = top; top += need; }
        }
        if (reuse) {
            for (int i : die_at[op]) {
                Buf& b = h.bufs[i];
                if (b.last >= n_ops) continue;
                free_list.push_back({b.off_ps, align(b.bytes_ps)});
                std::sort(free_list.begin(), free_list.end(), [](const Free& a, const Free& c) { return a.off < c.off; });
                for (size_t f = 0; f + 1 < free_list.size();) {
                    if (free_list[f].off + free_list[f].size == free_list[f + 1].off) {
                        free_list[f].size += free_list[f + 1].size;
                        free_list.erase(free_list.begin() + f + 1);
                    } else ++f;
                }
            }
        }
    }
    h.arena_ps = top;
}

// ---- tcgen05 conv tiling -----------------------------------------------------------------------
int plan_umma(const ConvShape& op, int B, ConvUmmaParams& p) {
    memset(&p, 0, sizeof(p));
    const int H = op.H, W = op.W, pad = op.ksize / 2, Wp = W + 2 * pad, Hp = H + 2 * pad, PP = Wp * Hp;
    const int ncbT = op.ncb0 + op.ncb1, taps = op.ksize * op.ksize;
    if (!op.n_tile || ncbT % 2) { set_error("conv '%s': channel counts not supported by the tcgen05 kernel", op.name); return FLO_ERR_UNSUPPORTED; }
    p.B = B; p.H = H; p.W = W; p.ncb0 = op.ncb0; p.ncb1 = op.ncb1; p.cout = op.cout; p.n_tile = op.n_tile; p.ksize = op.ksize;
    const bool strips = pad && (W % 8 == 0) && (H % 16 == 0) && (H / 16) * (W / 8) * op.n_tile <= 512;
    if (strips) {
        p.nb = 1; p.n_mtiles = (H / 16) * (W / 8); p.sbo_px = Wp; p.row0 = 0; p.tile_stride = 0;
    } else {
        // flattened padded pixels; choose samples per CTA: enough CTAs to fill the GPU, then fewer junk rows
        const int max_mt = std::max(1, std::min(4, 256 / op.n_tile));   // <= 256 TMEM columns: two CTAs per SM
        int best_nb = 1; double best_cost = 1e30;
        for (int nb = 1; nb <= 64; ++nb) {
            const int rows = nb * PP - 2 * (pad ? Wp + 1 : 0);
            const int mt = (rows + 127) / 128;
            if (mt > max_mt) break;
            const size_t a_bytes = (size_t)ncbT * nb * PP * 16;
            if (a_bytes > 120 * 1024) break;
            const int ctas = ((B + nb - 1) / nb) * (op.cout / op.n_tile);
            const int waves = (ctas + 148 * 2 - 1) / (148 * 2);
            const double cost = waves * (2.0 + mt);
            if (cost <= best_cost + 1e-9) { best_cost = cost; best_nb = nb; }   // ties: more samples per weight fetch
        }
        p.nb = best_nb;
        const int rows = p.nb * PP - 2 * (pad ? Wp + 1 : 0);
        p.n_mtiles = (rows + 127) / 128;
        p.sbo_px = 8; p.row0 = pad ? Wp + 1 : 0; p.tile_stride = 128;
    }
    p.plane_px = p.nb * PP;
    const int total_slices = taps * (ncbT / 2);
    int S = std::max(1, std::min(total_slices, 16384 / (op.n_tile * 32)));
    while (total_slices % S) --S;
    p.slices_per_stage = S;
    p.n_wstages = std::min(4, total_slices / S);
    int cols = 32;
    while (cols < p.n_mtiles * op.n_tile) cols <<= 1;
    p.tmem_cols = cols;
    p.smem_bytes = conv_umma_smem_bytes(p);
    if (p.smem_bytes > 227 * 1024 || cols > 512) { set_error("conv '%s': tile does not fit (smem %d, tmem %d)", op.name, p.smem_bytes, cols); return FLO_ERR_UNSUPPORTED; }
    return FLO_OK;
}

int make_tmap(CUtensorMap* tm, void* base, int ncb, int B, int H, int W, int pad, int nb) {
    EncodeTiledFn enc = get_encode_tiled();
    if (!enc) { set_error("cuTensorMapEncodeTiled is not available from the driver"); return FLO_ERR_CUDA; }
    cuuint64_t gdim[5] = {8, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)B, (cuuint64_t)ncb};
    cuuint64_t gstr[4] = {16, (cuuint64_t)W * 16, (cuuint64_t)H * W * 16, (cuuint64_t)B * H * W * 16};
    cuuint32_t box[5] = {8, (cuuint32_t)(W + 2 * pad), (cuuint32_t)(H + 2 * pad), (cuuint32_t)nb, (cuuint32_t)ncb};
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    CUresult r = enc(tm, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 5, base, gdim, gstr, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
                     CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { set_error("cuTensorMapEncodeTiled failed (%d) for [%d][%d][%d][%d][8] box nb=%d pad=%d", (int)r, ncb, B, H, W, nb, pad); return FLO_ERR_CUDA; }
    return FLO_OK;
}

// ---- op launch ---------------------------------------------------------------------------------
static int launch_op(Handle& h, Plan& pl, int i, cudaStream_t st) {
    const Op& op = h.ops[i];
    const Spec& s = h.spec;
    auto ptr = [&](int b) -> void* { return b >= 0 ? pl.buf_ptr[b] : nullptr; };
    auto f32c = [&](size_t off) -> const float* { return off == NONE ? nullptr : h.d_f32 + off; };
    cudaError_t e = cudaSuccess;
    switch (op.kind) {
        case OP_INIT: {
            InitConvParams p{};
            p.ctrl = pl.ctrl; p.w = f32c(h.o_init_w); p.bias = f32c(h.o_init_b);
            p.out_m = (float*)ptr(op.out_m); p.out_o = ptr(op.out_o);
            p.B = pl.B; p.HW = s.H * s.W; p.cin = s.channels; p.dim = s.dim; p.o_is_bf16 = s.bf16;
            e = launch_init_conv(p, st);
        } break;
        case OP_CONV: {
            if (s.bf16) {
                ConvUmmaParams p = pl.umma[i];
                p.w = h.d_bf16 + op.w_umma; p.bias = f32c(op.bias); p.res = (const float*)ptr(op.res);
                p.out_m = (float*)ptr(op.out_m); p.out_o = (__nv_bfloat16*)ptr(op.out_o);
                e = launch_conv_umma(p, pl.tmA0[i], pl.tmA1[i], st);
            } else {
                ConvSimtParams p{};
                p.in0 = ptr(op.in0); p.in1 = ptr(op.in1); p.ncb0 = op.ncb0; p.ncb1 = op.ncb1; p.in_is_bf16 = 0;
                p.w = f32c(op.w_simt); p.bias = f32c(op.bias); p.res = (const float*)ptr(op.res);
                p.out_m = (float*)ptr(op.out_m); p.out_o = nullptr; p.o_is_bf16 = 0;
                p.B = pl.B; p.H = op.H; p.W = op.W; p.cout = op.cout; p.ksize = op.ksize;
                p.act_silu = op.act_silu; p.out_unshuf = ptr(op.out_un); p.out_up = ptr(op.out_up);
                if (op.need_mode) { p.mask_mode = pl.mask_mode; p.need_mode = op.need_mode; p.bypass = (const float*)ptr(op.bypass); }
                e = launch_conv_simt(p, st);
            }
        } break;
        case OP_GN: {
            GnParams p{};
            p.ctrl = pl.ctrl; p.in = (const float*)ptr(op.gn_in); p.res = (const float*)ptr(op.res);
            p.gamma = f32c(op.gamma); p.beta = f32c(op.beta);
            p.out_m = (float*)ptr(op.out_m); p.out_o = ptr(op.out_o); p.out_unshuf = ptr(op.out_un); p.out_up = ptr(op.out_up);
            p.o_is_bf16 = s.bf16; p.B = pl.B; p.C = op.C; p.H = op.H; p.W = op.W; p.groups = op.groups;
            p.film_off = op.film_off; p.film_dim = h.film_dim; p.silu = op.silu;
            e = launch_gn(p, st);
        } break;
        case OP_LINATTN:
        case OP_MIDATTN: {
            AttnParams p{};
            p.qkv = ptr(op.qkv); p.out = ptr(op.attn_out); p.is_bf16 = s.bf16; p.B = pl.B; p.n = op.n;
            e = op.kind == OP_LINATTN ? launch_linattn(p, st) : launch_midattn(p, st);
        } break;
        case OP_FINAL: {
            FinalParams p{};
            p.ctrl = pl.ctrl; p.in = (const float*)ptr(op.gn_in); p.w = f32c(h.o_final_w); p.bias = f32c(h.o_final_b);
            p.B = pl.B; p.HW = s.H * s.W; p.dim = s.dim; p.channels = s.channels;
            e = launch_final(p, st);
        } break;
    }
    if (e != cudaSuccess) { set_error("launch of op %d '%s' failed: %s", i, op.name.c_str(), cudaGetErrorString(e)); return FLO_ERR_CUDA; }
    return FLO_OK;
}

static int finalize_fused(Handle& h, Plan& pl);
static int launch_fused_stage(Handle& h, Plan& pl, int i, cudaStream_t st);
static int n_units(const Handle& h) { return h.spec.fused ? (int)h.fstages.size() : (int)h.ops.size(); }
static int launch_unit(Handle& h, Plan& pl, int i, cudaStream_t st) {
    return h.spec.fused ? launch_fused_stage(h, pl, i, st) : launch_op(h, pl, i, st);
}

static void destroy_plan(Plan&) {}          // resources are released by ~Plan when the owning unique_ptr goes away

// One stream at a time per handle (the stage table, the control block and the workspaces are per handle / per plan):
// a call on a different stream than the previous one first waits for that stream's work.
static int enter_stream(Handle& h, cudaStream_t st) {
    if (h.has_last_stream && h.last_stream != st) CUDA_TRY(cudaStreamSynchronize(h.last_stream));
    h.last_stream = st; h.has_last_stream = true;
    return FLO_OK;
}

static int get_plan(Handle& h, int B, Plan** out, cudaStream_t st) {
    auto it = h.plans.find(B);
    if (it != h.plans.end()) { it->second->last_use = ++h.use_ctr; *out = it->second.get(); return FLO_OK; }
    if (B <= 0) { set_error("batch size must be positive, got %d", B); return FLO_ERR_INVALID; }
    if (h.plans.size() >= MAX_PLANS) {
        // ragged last batches / uneven shards would otherwise grow the cache without bound: drop the least recently used plan
        // (its workspace may still be in use by enqueued work: wait for the device first; plan creation is a slow path anyway)
        auto lru = h.plans.begin();
        for (auto jt = h.plans.begin(); jt != h.plans.end(); ++jt)
            if (jt->second->last_use < lru->second->last_use) lru = jt;
        CUDA_TRY(cudaDeviceSynchronize());
        h.plans.erase(lru);
    }
    const Spec& s = h.spec;
    std::unique_ptr<Plan> pl(new Plan());
    pl->B = B;
    auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
    const size_t state_bytes = al((size_t)B * s.channels * s.H * s.W * 4);
    const size_t film_bytes = al((size_t)B * h.film_dim * 4);
    const size_t cls_bytes = al((size_t)B * 8);
    pl->arena_bytes = s.fused ? 256 : al(h.arena_ps * (size_t)B);     // layer-by-layer activations
    const size_t farena_bytes = s.fused ? al(h.farena_ps * (size_t)B) : 0;   // stage-boundary tensors of the fused path
    const size_t flag_bytes = al((size_t)B * 4);
    pl->total_bytes = pl->arena_bytes + farena_bytes + 4 * state_bytes + film_bytes + cls_bytes + flag_bytes + 512;
    cudaError_t e = cudaMalloc((void**)&pl->base, pl->total_bytes);
    if (e != cudaSuccess) { set_error("cudaMalloc of %zu workspace bytes for B=%d failed: %s", pl->total_bytes, B, cudaGetErrorString(e)); cudaGetLastError(); return FLO_ERR_NOMEM; }
    uint8_t* q = pl->base;
    pl->arena = q; q += pl->arena_bytes;
    pl->farena = q; q += farena_bytes;
    pl->y = (float*)q; q += state_bytes;
    pl->acc = (float*)q; q += state_bytes;
    pl->xs = (float*)q; q += state_bytes;
    pl->vcond = (float*)q; q += state_bytes;
    pl->film_ps = (float*)q; q += film_bytes;
    pl->cls = (int64_t*)q; q += cls_bytes;
    pl->pair_flags = (int*)q; q += flag_bytes;
    pl->ctrl = (Ctrl*)q; q += 256;
    pl->mask_mode = (int*)q;
    pl->buf_ptr.resize(h.bufs.size());
    for (size_t i = 0; i < h.bufs.size(); ++i) pl->buf_ptr[i] = s.fused ? nullptr : pl->arena + h.bufs[i].off_ps * (size_t)B;
    // halo / padding rows of the arena are never read as data, but keep everything finite.  On the CALLER's stream: the
    // first kernels of this plan are enqueued there right after this call, and a non-blocking stream is not ordered after
    // the legacy default stream.
    CUDA_TRY(cudaMemsetAsync(pl->base, 0, pl->total_bytes, st));

    const int n_ops = (int)h.ops.size();
    pl->umma.resize(n_ops); pl->tmA0.resize(n_ops); pl->tmA1.resize(n_ops);
    if (s.fused) {
        int rc = finalize_fused(h, *pl);
        if (rc) { destroy_plan(*pl); return rc; }
    } else if (s.bf16) {
        for (int i = 0; i < n_ops; ++i) {
            const Op& op = h.ops[i];
            if (op.kind != OP_CONV) continue;
            ConvShape cs{op.name.c_str(), op.H, op.W, op.ksize, op.ncb0, op.ncb1, op.cout, op.n_tile};
            int rc = plan_umma(cs, B, pl->umma[i]);
            if (rc) { destroy_plan(*pl); return rc; }
            const int pad = op.ksize / 2;
            rc = make_tmap(&pl->tmA0[i], pl->buf_ptr[op.in0], op.ncb0, B, op.H, op.W, pad, pl->umma[i].nb);
            if (rc) { destroy_plan(*pl); return rc; }
            if (op.in1 >= 0) rc = make_tmap(&pl->tmA1[i], pl->buf_ptr[op.in1], op.ncb1, B, op.H, op.W, pad, pl->umma[i].nb);
            else pl->tmA1[i] = pl->tmA0[i];
            if (rc) { destroy_plan(*pl); return rc; }
        }
    }
    if (!(s.flags & FLO_FLAG_NO_GRAPH)) {
        cudaGraph_t g = nullptr;
        CUDA_TRY(cudaStreamBeginCapture(h.capture_stream, cudaStreamCaptureModeThreadLocal));
        int rc = FLO_OK;
        for (int i = 0; i < n_units(h) && rc == FLO_OK; ++i) rc = launch_unit(h, *pl, i, h.capture_stream);
        cudaError_t ce = cudaStreamEndCapture(h.capture_stream, &g);
        if (rc) { if (g) cudaGraphDestroy(g); destroy_plan(*pl); return rc; }
        if (ce != cudaSuccess) { set_error("graph capture failed: %s", cudaGetErrorString(ce)); destroy_plan(*pl); return FLO_ERR_CUDA; }
        ce = cudaGraphInstantiate(&pl->graph, g, 0);
        cudaGraphDestroy(g);
        if (ce != cudaSuccess) { set_error("graph instantiate failed: %s", cudaGetErrorString(ce)); destroy_plan(*pl); return FLO_ERR_CUDA; }
        if (s.fused) {     // the stage kernels find their ODE stage in the device-side control block
            g = nullptr;
            CUDA_TRY(cudaStreamBeginCapture(h.capture_stream, cudaStreamCaptureModeThreadLocal));
            for (int k = 0; k < 4 && rc == FLO_OK; ++k)
                for (int i = 0; i < n_units(h) && rc == FLO_OK; ++i) rc = launch_unit(h, *pl, i, h.capture_stream);
            ce = cudaStreamEndCapture(h.capture_stream, &g);
            if (rc == FLO_OK && ce == cudaSuccess) ce = cudaGraphInstantiate(&pl->graph4, g, 0);
            if (g) cudaGraphDestroy(g);
            if (rc || ce != cudaSuccess) { set_error("graph capture (x4) failed"); destroy_plan(*pl); return rc ? rc : FLO_ERR_CUDA; }
        }
    }
    pl->last_use = ++h.use_ctr;
    *out = pl.get();
    h.plans[B] = std::move(pl);
    return FLO_OK;
}

static int run_forward(Handle& h, Plan& pl, cudaStream_t st) {
    if (pl.graph) {
        CUDA_TRY(cudaGraphLaunch(pl.graph, st));
    } else {
        for (int i = 0; i < n_units(h); ++i) {
            int rc = launch_unit(h, pl, i, st);
            if (rc) return rc;
        }
    }
    h.launches += (int64_t)n_units(h);
    return FLO_OK;
}

static TembParams temb_params(Handle& h) {
    const Spec& s = h.spec;
    TembParams p{};
    p.dim = s.dim; p.time_dim = s.time_dim; p.film_dim = h.film_dim; p.n_classes = s.n_classes;
    p.freqs = h.d_f32 + h.o_freqs;
    p.w1t = h.d_f32 + h.o_w1t; p.b1 = h.d_f32 + h.o_b1; p.w2t = h.d_f32 + h.o_w2t; p.b2 = h.d_f32 + h.o_b2;
    if (s.n_classes > 0) {
        p.emb = h.d_f32 + h.o_emb; p.wc1t = h.d_f32 + h.o_wc1t; p.bc1 = h.d_f32 + h.o_bc1;
        p.wc3t = h.d_f32 + h.o_wc3t; p.bc3 = h.d_f32 + h.o_bc3;
    }
    p.wft = h.d_f32 + h.o_wft; p.bf = h.d_f32 + h.o_bf;
    p.n_cond = -1;
    return p;
}

static int ensure_stage_capacity(Handle& h, int n) {
    if (n <= h.stage_cap) return FLO_OK;
    int cap = std::max(n, 1024);
    if (h.d_stages) { cudaFree(h.d_stages); cudaFree(h.d_stage_t); cudaFree(h.d_film_u); }
    CUDA_TRY(cudaMalloc((void**)&h.d_stages, (size_t)cap * sizeof(Stage)));
    CUDA_TRY(cudaMalloc((void**)&h.d_stage_t, (size_t)cap * sizeof(float)));
    CUDA_TRY(cudaMalloc((void**)&h.d_film_u, (size_t)cap * h.film_dim * sizeof(float)));
    h.stage_cap = cap;
    return FLO_OK;
}
static int ensure_host_staging(Handle& h, int n) {
    if (n <= h.h_cap) return FLO_OK;
    int cap = std::max(n, 1024);
    for (int i = 0; i < 4; ++i) {
        if (h.h_stages[i]) { cudaEventSynchronize(h.h_ev[i]); cudaFreeHost(h.h_stages[i]); cudaFreeHost(h.h_stage_t[i]); }
        CUDA_TRY(cudaMallocHost((void**)&h.h_stages[i], (size_t)cap * sizeof(Stage)));
        CUDA_TRY(cudaMallocHost((void**)&h.h_stage_t[i], (size_t)cap * sizeof(float)));
        if (!h.h_ev[i]) CUDA_TRY(cudaEventCreateWithFlags(&h.h_ev[i], cudaEventDisableTiming));
    }
    h.h_cap = cap;
    return FLO_OK;
}

#include "fused_plan.inc"

}  // namespace flo

using namespace flo;

// =================================================================================================
// C ABI
// =================================================================================================
extern "C" {

int flo_version(void) { return FLO_VERSION; }
const char* flo_last_error(void) { return g_last_error.c_str(); }

int flo_param_count(const flo_unet_cfg* cfg) {
    Spec s;
    int rc = make_spec(cfg, s);
    if (rc) return rc;
    return (int)manifest(s).size();
}

int flo_param_info(const flo_unet_cfg* cfg, int index, char* name, int name_cap, int64_t shape[4], int* ndim) {
    Spec s;
    int rc = make_spec(cfg, s);
    if (rc) return rc;
    auto m = manifest(s);
    if (index < 0 || index >= (int)m.size()) { set_error("parameter index %d out of range", index); return FLO_ERR_INVALID; }
    if (name && name_cap > 0) snprintf(name, name_cap, "%s", m[index].name.c_str());
    for (int i = 0; i < 4; ++i) shape[i] = i < (int)m[index].shape.size() ? m[index].shape[i] : 1;
    if (ndim) *ndim = (int)m[index].shape.size();
    return FLO_OK;
}

int flo_unet_destroy(flo_unet_t* hh) {
    Handle* h = reinterpret_cast<Handle*>(hh);
    if (!h) return FLO_OK;
    cudaSetDevice(h->spec.device);
    cudaDeviceSynchronize();
    delete h;                     // ~Handle releases the plans, the packed weights, the stage tables and the capture stream
    return FLO_OK;
}

int flo_unet_create(flo_unet_t** out, const flo_unet_cfg* cfg, const void* const* params, int n_params, void* stream) {
    if (!out) { set_error("out is NULL"); return FLO_ERR_INVALID; }
    *out = nullptr;
    std::unique_ptr<Handle> h(new Handle());
    int rc = make_spec(cfg, h->spec);
    if (rc) return rc;
    h->params = manifest(h->spec);
    if (n_params != (int)h->params.size()) {
        set_error("expected %d parameter tensors, got %d", (int)h->params.size(), n_params);
        return FLO_ERR_INVALID;
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        set_error("no CUDA device: flocoder_b200 has no CPU fallback");
        return FLO_ERR_CUDA;
    }
    CUDA_TRY(cudaSetDevice(h->spec.device));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, h->spec.device));
    if (prop.major != 10) {
        set_error("device %d is sm_%d%d; this library is built for sm_100a (B200) only", h->spec.device, prop.major, prop.minor);
        return FLO_ERR_UNSUPPORTED;
    }
    cudaStream_t st = (cudaStream_t)stream;
    CUDA_TRY(cudaStreamSynchronize(st));
    for (int i = 0; i < n_params; ++i) {
        if (!params[i]) { set_error("parameter %d ('%s') is NULL", i, h->params[i].name.c_str()); return FLO_ERR_INVALID; }
        std::vector<float>& v = h->host[h->params[i].name];
        v.resize((size_t)h->params[i].numel());
        CUDA_TRY(cudaMemcpy(v.data(), params[i], v.size() * sizeof(float), cudaMemcpyDeviceToHost));
    }
    Builder b(*h);
    rc = b.build();
    if (rc) return rc;
    rc = check_op_kernels(*h);
    if (rc) return rc;
    allocate_arena(*h);
    if (h->spec.fused) {
        FusedBuilder fb(*h, h->ftensors, h->fstages, 4);
        rc = fb.build();
        if (rc) return rc;
        for (int v = 0; v < 2; ++v) {
            std::vector<FTensor> scratch;              // same tensors in the same order as variant 0
            FusedBuilder fa(*h, scratch, h->fstages_alt[v], v == 0 ? 2 : 1);
            rc = fa.build();
            if (rc) return rc;
        }
    }
    h->host.clear();
    CUDA_TRY(cudaMalloc((void**)&h->d_f32, h->blob_f32.size() * sizeof(float)));
    CUDA_TRY(cudaMemcpy(h->d_f32, h->blob_f32.data(), h->blob_f32.size() * sizeof(float), cudaMemcpyHostToDevice));
    if (!h->blob_bf16.empty()) {
        CUDA_TRY(cudaMalloc((void**)&h->d_bf16, h->blob_bf16.size() * sizeof(__nv_bfloat16)));
        CUDA_TRY(cudaMemcpy(h->d_bf16, h->blob_bf16.data(), h->blob_bf16.size() * sizeof(__nv_bfloat16), cudaMemcpyHostToDevice));
        CUDA_TRY(conv_umma_configure());
    }
    CUDA_TRY(simt_configure());
    if (h->spec.fused) CUDA_TRY(fused_configure());
    CUDA_TRY(cudaStreamCreateWithFlags(&h->capture_stream, cudaStreamNonBlocking));
    *out = reinterpret_cast<flo_unet_t*>(h.release());
    return FLO_OK;
}

size_t flo_workspace_bytes(flo_unet_t* hh, int B) {
    Handle* h = reinterpret_cast<Handle*>(hh);
    if (!h) return 0;
    cudaSetDevice(h->spec.device);
    Plan* pl = nullptr;
    if (get_plan(*h, B, &pl, nullptr)) return 0;
    cudaStreamSynchronize(nullptr);
    return pl->total_bytes;
}

int flo_unet_forward(flo_unet_t* hh, const float* x, const float* time, const int64_t* class_ids, float* v, int B,
                     void* stream) {
    Handle* h = reinterpret_cast<Handle*>(hh);
    if (!h || !x || !time || !v) { set_error("NULL argument"); return FLO_ERR_INVALID; }
    CUDA_TRY(cudaSetDevice(h->spec.device));
    cudaStream_t st = (cudaStream_t)stream;
    int rc = enter_stream(*h, st);
    if (rc) return rc;
    Plan* pl = nullptr;
    rc = get_plan(*h, B, &pl, st);
    if (rc) return rc;
    const Spec& s = h->spec;
    const size_t n = (size_t)B * s.channels * s.H * s.W;
    CUDA_TRY(cudaMemcpyAsync(pl->xs, x, n * sizeof(float), cudaMemcpyDeviceToDevice, st));
    TembParams tp = temb_params(*h);
    tp.t = time; tp.t_stride = 1; tp.cls = (s.n_classes > 0) ? class_ids : nullptr; tp.n_rows = B; tp.film = pl->film_ps;
    CUDA_TRY(launch_temb(tp, st));
    rc = ensure_stage_capacity(*h, 1);
    if (rc) return rc;
    Ctrl c{};
    c.step = 0; c.done_ctr = 0; c.film_per_sample = 1; c.n_stages = 1; c.cfg = 0.f;
    c.y = pl->y; c.acc = pl->acc; c.xs = pl->xs; c.vcond = pl->vcond; c.vout = v; c.vtrace = nullptr;
    c.film = pl->film_ps; c.stages = h->d_stages;
    Stage s0{};
    s0.kind = ST_PLAIN; s0.eval_idx = -1;
    CUDA_TRY(launch_setup_ctrl(pl->ctrl, c, h->d_stages, &s0, st));
    h->launches += 2;
    return run_forward(*h, *pl, st);
}

int flo_unet_set_mask(flo_unet_t* hh, const float* mask, int B, void* stream) {
    Handle* h = reinterpret_cast<Handle*>(hh);
    if (!h) { set_error("NULL handle"); return FLO_ERR_INVALID; }
    const Spec& s = h->spec;
    if (!s.mask_cond) {
        if (!mask) return FLO_OK;           // unet.py:298: hasattr(self, 'mask_fusion_conv') is False -> cond['mask_cond'] is ignored
        set_error("this U-Net was built with mask_cond=0: it has no mask-fusion branches");
        return FLO_ERR_INVALID;
    }
    CUDA_TRY(cudaSetDevice(s.device));
    cudaStream_t st = (cudaStream_t)stream;
    int rc = enter_stream(*h, st);
    if (rc) return rc;
    Plan* pl = nullptr;
    rc = get_plan(*h, B, &pl, st);
    if (rc) return rc;
    MaskPrepParams mp{};
    mp.mask = mask; mp.n_levels = s.n_levels; mp.B = B; mp.ch = s.channels; mp.H = s.H; mp.W = s.W; mp.mode = pl->mask_mode;
    for (int l = 0; l < s.n_levels; ++l) mp.out[l] = (float*)pl->buf_ptr[h->mask_buf[l]];
    CUDA_TRY(launch_mask_prep(mp, st));
    h->launches += mask ? 2 : 1;
    return FLO_OK;
}

int flo_integrate_nfe(int method, int n_ts) {
    if (n_ts < 1) return 0;
    switch (method) {
        case FLO_RK4: return 4 * (n_ts - 1);
        case FLO_EULER_LEGACY: return n_ts;
        case FLO_EULER_GRID: return n_ts - 1;
        default: return -1;
    }
}

static int integrate_impl(Handle* h, Plan* pl, float* y, const float* ts, int n_ts, int method, float dt_arg,
                          float t_scale, const int64_t* class_ids, float cfg_strength, float* v_trace,
                          cudaStream_t st) {
    const Spec& s = h->spec;
    const int B = pl->B;
    if (method != FLO_RK4 && method != FLO_EULER_LEGACY && method != FLO_EULER_GRID) { set_error("unknown method %d", method); return FLO_ERR_INVALID; }
    if (n_ts < 1 || !ts) { set_error("need at least one time point"); return FLO_ERR_INVALID; }
    if (s.n_classes == 0) class_ids = nullptr;              // unet.py:315: no class_cond_mlp -> cond ignored
    const bool use_cls = class_ids != nullptr;
    const bool use_cfg = use_cls && cfg_strength != 0.0f;   // sampling.py:69
    // ---- stage list (fp32 arithmetic exactly as the reference's 0-d tensors, sampling.py:44-47,117)
    struct Ev { float t; float dt; float dt6; int kind; };
    std::vector<Ev> evs;
    if (method == FLO_RK4) {
        for (int i = 0; i + 1 < n_ts; ++i) {
            const float t = ts[i];
            const float dt = ts[i + 1] - ts[i];
            const float half = dt / 2.0f;
            const float th = t + half;
            const float te = t + dt;
            const float dt6 = dt / 6.0f;
            evs.push_back({t, dt, dt6, ST_RK1});
            evs.push_back({th, dt, dt6, ST_RK2});
            evs.push_back({th, dt, dt6, ST_RK3});
            evs.push_back({te, dt, dt6, ST_RK4});
        }
    } else if (method == FLO_EULER_LEGACY) {
        for (int i = 0; i < n_ts; ++i) evs.push_back({ts[i], dt_arg, 0.f, ST_EULER});
    } else {
        for (int i = 0; i + 1 < n_ts; ++i) evs.push_back({ts[i], ts[i + 1] - ts[i], 0.f, ST_EULER});
    }
    const int n_eval = (int)evs.size();
    if (n_eval == 0) return FLO_OK;
    // ---- classifier-free guidance as ONE forward over 2B samples per evaluation (fused path): rows [0,B) carry the class FiLM,
    // rows [B,2B) the unconditional one; the final epilogue combines the halves (SF_CFG_2B).  Twice the CTAs per launch, half
    // the launches, and the time embedding becomes a node of the replayed graph (it reads the stage time on the device).
    // Class conditioning WITHOUT guidance takes the same route with B rows: its per-sample FiLM table is then also built by
    // the in-graph k_temb, so the four-pass graph is kept (the host-launched k_temb per pass is what broke it).
    if (use_cls && s.fused && !getenv("FLO_CFG_TWO_PASS")) {
        Plan* p2 = nullptr;
        const int Bf = use_cfg ? 2 * B : B;
        int rc2 = get_plan(*h, Bf, &p2, st);
        if (rc2) return rc2;
        const FStage& last = h->stages(p2->fvar).back();
        if (last.kind == 0 && (last.cp.nsplit == 1 || !use_cfg)) {
            rc2 = ensure_stage_capacity(*h, n_eval);
            if (rc2) return rc2;
            rc2 = ensure_host_staging(*h, n_eval);
            if (rc2) return rc2;
            const int slot = h->h_next;
            h->h_next = (h->h_next + 1) & 3;
            CUDA_TRY(cudaEventSynchronize(h->h_ev[slot]));
            Stage* hs = h->h_stages[slot];
            for (int e = 0; e < n_eval; ++e) {
                Stage a{};
                a.t_scaled = evs[e].t * t_scale; a.dt = evs[e].dt; a.dt6 = evs[e].dt6; a.kind = evs[e].kind; a.film_row = 0;
                a.flags = use_cfg ? SF_CFG_2B : 0; a.eval_idx = e;
                hs[e] = a;
            }
            CUDA_TRY(cudaMemcpyAsync(h->d_stages, hs, (size_t)n_eval * sizeof(Stage), cudaMemcpyHostToDevice, st));
            CUDA_TRY(cudaEventRecord(h->h_ev[slot], st));
            const size_t n = (size_t)B * s.channels * s.H * s.W;
            CUDA_TRY(cudaMemcpyAsync(p2->xs, y, n * sizeof(float), cudaMemcpyDeviceToDevice, st));
            if (use_cfg) CUDA_TRY(cudaMemcpyAsync(p2->xs + n, y, n * sizeof(float), cudaMemcpyDeviceToDevice, st));
            CUDA_TRY(cudaMemcpyAsync(p2->cls, class_ids, (size_t)B * sizeof(int64_t), cudaMemcpyDeviceToDevice, st));
            Ctrl c{};
            c.step = 0; c.done_ctr = 0; c.film_per_sample = 1; c.n_stages = n_eval; c.cfg = cfg_strength; c.cfg_half = use_cfg ? B : 0;
            c.y = y; c.acc = p2->acc; c.xs = p2->xs; c.vcond = p2->vcond; c.vout = nullptr; c.vtrace = v_trace;
            c.film = p2->film_ps; c.stages = h->d_stages; c.pair_flags = p2->pair_flags;
            CUDA_TRY(launch_setup_ctrl(p2->ctrl, c, nullptr, nullptr, st));
            h->launches += 1;
            TembParams tp = temb_params(*h);
            tp.ctrl = p2->ctrl; tp.t = nullptr; tp.t_stride = 0; tp.cls = p2->cls; tp.n_cond = B; tp.n_rows = Bf; tp.film = p2->film_ps;
            auto one_pass = [&](cudaStream_t ss) -> int {
                if (launch_temb(tp, ss) != cudaSuccess) { set_error("k_temb launch failed"); return FLO_ERR_CUDA; }
                for (int i = 0; i < n_units(*h); ++i) {
                    int r = launch_unit(*h, *p2, i, ss);
                    if (r) return r;
                }
                return FLO_OK;
            };
            const bool graphs = !(s.flags & FLO_FLAG_NO_GRAPH);
            if (graphs && (!p2->graph_c || p2->graph_c_cond != B)) {
                if (p2->graph_c) { cudaGraphExecDestroy(p2->graph_c); p2->graph_c = nullptr; }
                if (p2->graph_c4) { cudaGraphExecDestroy(p2->graph_c4); p2->graph_c4 = nullptr; }
                for (int reps = 1; reps <= 4; reps += 3) {
                    cudaGraph_t g = nullptr;
                    CUDA_TRY(cudaStreamBeginCapture(h->capture_stream, cudaStreamCaptureModeThreadLocal));
                    int r = FLO_OK;
                    for (int k = 0; k < reps && r == FLO_OK; ++k) r = one_pass(h->capture_stream);
                    cudaError_t ce = cudaStreamEndCapture(h->capture_stream, &g);
                    if (r == FLO_OK && ce == cudaSuccess) ce = cudaGraphInstantiate(reps == 1 ? &p2->graph_c : &p2->graph_c4, g, 0);
                    if (g) cudaGraphDestroy(g);
                    if (r || ce != cudaSuccess) { if (!r) set_error("graph capture (CFG) failed: %s", cudaGetErrorString(ce)); return r ? r : FLO_ERR_CUDA; }
                }
                p2->graph_c_cond = B;
            }
            for (int e = 0; e < n_eval; ++e) {
                if (graphs && e + 3 < n_eval) { CUDA_TRY(cudaGraphLaunch(p2->graph_c4, st)); e += 3; h->launches += 4 * (int64_t)(n_units(*h) + 1); continue; }
                if (graphs) { CUDA_TRY(cudaGraphLaunch(p2->graph_c, st)); }
                else { rc2 = one_pass(st); if (rc2) return rc2; }
                h->launches += (int64_t)(n_units(*h) + 1);
            }
            return FLO_OK;
        }
    }
    const int n_pass = use_cfg ? 2 * n_eval : n_eval;
    int rc = ensure_stage_capacity(*h, n_pass);
    if (rc) return rc;
    rc = ensure_host_staging(*h, n_pass);
    if (rc) return rc;
    const int slot = h->h_next;
    h->h_next = (h->h_next + 1) & 3;
    CUDA_TRY(cudaEventSynchronize(h->h_ev[slot]));
    Stage* hs = h->h_stages[slot];
    float* ht = h->h_stage_t[slot];
    // FiLM rows: conditional passes use the per-sample table; unconditional passes the uniform table
    std::vector<int> pass_per_sample(n_pass);
    int pi = 0;
    for (int e = 0; e < n_eval; ++e) {
        const float t_scaled = evs[e].t * t_scale;
        if (use_cfg) {
            Stage a{}; a.t_scaled = t_scaled; a.dt = evs[e].dt; a.dt6 = evs[e].dt6; a.kind = ST_CFG_COND; a.film_row = 0; a.flags = 0; a.eval_idx = -1;
            hs[pi] = a; ht[pi] = t_scaled; pass_per_sample[pi] = 1; ++pi;
            Stage b2{}; b2.t_scaled = t_scaled; b2.dt = evs[e].dt; b2.dt6 = evs[e].dt6; b2.kind = evs[e].kind; b2.film_row = pi; b2.flags = SF_CFG_COMBINE; b2.eval_idx = e;
            hs[pi] = b2; ht[pi] = t_scaled; pass_per_sample[pi] = 0; ++pi;
        } else {
            Stage a{}; a.t_scaled = t_scaled; a.dt = evs[e].dt; a.dt6 = evs[e].dt6; a.kind = evs[e].kind; a.film_row = pi; a.flags = 0; a.eval_idx = e;
            hs[pi] = a; ht[pi] = t_scaled; pass_per_sample[pi] = use_cls ? 1 : 0; ++pi;
        }
    }
    CUDA_TRY(cudaMemcpyAsync(h->d_stages, hs, (size_t)n_pass * sizeof(Stage), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaMemcpyAsync(h->d_stage_t, ht, (size_t)n_pass * sizeof(float), cudaMemcpyHostToDevice, st));
    CUDA_TRY(cudaEventRecord(h->h_ev[slot], st));
    // uniform FiLM table for every pass that needs it (one launch for the whole trajectory)
    TembParams tp = temb_params(*h);
    if (!use_cls || use_cfg) {
        tp.t = h->d_stage_t; tp.t_stride = 1; tp.cls = nullptr; tp.n_rows = n_pass; tp.film = h->d_film_u;
        CUDA_TRY(launch_temb(tp, st));
        h->launches += 1;
    }
    const size_t n = (size_t)B * s.channels * s.H * s.W;
    CUDA_TRY(cudaMemcpyAsync(pl->xs, y, n * sizeof(float), cudaMemcpyDeviceToDevice, st));
    Ctrl c{};
    c.step = 0; c.done_ctr = 0; c.film_per_sample = 0; c.n_stages = n_pass; c.cfg = cfg_strength;
    c.y = y; c.acc = pl->acc; c.xs = pl->xs; c.vcond = pl->vcond; c.vout = nullptr; c.vtrace = v_trace;
    c.film = h->d_film_u; c.stages = h->d_stages;
    // film_per_sample is a per-pass property: encode it by pointing ctrl at the right table per pass
    for (int p = 0; p < n_pass; ++p) {
        if (pass_per_sample[p]) {
            tp.t = h->d_stage_t + p; tp.t_stride = 0; tp.cls = class_ids; tp.n_rows = B; tp.film = pl->film_ps;
            CUDA_TRY(launch_temb(tp, st));
            h->launches += 1;
        }
        if (p == 0 || pass_per_sample[p] != pass_per_sample[p - 1] || p == 0) {
            Ctrl cc = c;
            cc.step = p;
            cc.film_per_sample = pass_per_sample[p];
            cc.film = pass_per_sample[p] ? pl->film_ps : h->d_film_u;
            CUDA_TRY(launch_setup_ctrl(pl->ctrl, cc, nullptr, nullptr, st));
            h->launches += 1;
        }
        // four consecutive passes with nothing to launch in between go out as one graph
        if (pl->graph4 && p + 3 < n_pass && !pass_per_sample[p] && !pass_per_sample[p + 1] && !pass_per_sample[p + 2] &&
            !pass_per_sample[p + 3]) {
            CUDA_TRY(cudaGraphLaunch(pl->graph4, st));
            h->launches += 4 * (int64_t)n_units(*h);
            p += 3;
            continue;
        }
        rc = run_forward(*h, *pl, st);
        if (rc) return rc;
    }
    return FLO_OK;
}

int flo_integrate(flo_unet_t* hh, float* y, const float* ts, int n_ts, int method, float dt, float t_scale,
                  const int64_t* class_ids, float cfg_strength, float* v_trace, int B, void* stream) {
    Handle* h = reinterpret_cast<Handle*>(hh);
    if (!h || !y) { set_error("NULL argument"); return FLO_ERR_INVALID; }
    CUDA_TRY(cudaSetDevice(h->spec.device));
    int rc = enter_stream(*h, (cudaStream_t)stream);
    if (rc) return rc;
    Plan* pl = nullptr;
    rc = get_plan(*h, B, &pl, (cudaStream_t)stream);
    if (rc) return rc;
    return integrate_impl(h, pl, y, ts, n_ts, method, dt, t_scale, class_ids, cfg_strength, v_trace, (cudaStream_t)stream);
}

int flo_integrate_host(flo_unet_t* hh, const float* x0, float* x1, const float* ts, int n_ts, int method, float dt,
                       float t_scale, const int64_t* class_ids, float cfg_strength, int B, void* stream) {
    Handle* h = reinterpret_cast<Handle*>(hh);
    if (!h || !x0 || !x1) { set_error("NULL argument"); return FLO_ERR_INVALID; }
    CUDA_TRY(cudaSetDevice(h->spec.device));
    cudaStream_t st = (cudaStream_t)stream;
    int rc = enter_stream(*h, st);
    if (rc) return rc;
    Plan* pl = nullptr;
    rc = get_plan(*h, B, &pl, st);
    if (rc) return rc;
    const Spec& s = h->spec;
    const size_t bytes = (size_t)B * s.channels * s.H * s.W * sizeof(float);
    CUDA_TRY(cudaMemcpyAsync(pl->y, x0, bytes, cudaMemcpyHostToDevice, st));
    const int64_t* cls_dev = nullptr;
    if (class_ids && s.n_classes > 0) {
        CUDA_TRY(cudaMemcpyAsync(pl->cls, class_ids, (size_t)B * sizeof(int64_t), cudaMemcpyHostToDevice, st));
        cls_dev = pl->cls;
    }
    rc = integrate_impl(h, pl, pl->y, ts, n_ts, method, dt, t_scale, cls_dev, cfg_strength, nullptr, st);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(x1, pl->y, bytes, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return FLO_OK;
}

// ---- adaptive Dormand-Prince 5(4) (rk45.cu): stage times, step control and stage inputs on the device; the host waits once
// per attempt for a 40-byte status record.
static int ensure_rk45(Handle& h, Plan& fp, cudaStream_t st) {
    if (!fp.rk_buf) {
        auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
        const size_t nmax = (size_t)fp.B * h.spec.channels * h.spec.H * h.spec.W;     // >= n on every route
        const size_t fbytes = al(9 * nmax * sizeof(float)), cbytes = al(sizeof(Rk45Ctl));
        const size_t bytes = fbytes + cbytes + 2 * 1024 * sizeof(double);
        cudaError_t e = cudaMalloc((void**)&fp.rk_buf, bytes);
        if (e != cudaSuccess) { cudaGetLastError(); fp.rk_buf = nullptr; set_error("cudaMalloc of %zu RK45 bytes failed", bytes); return FLO_ERR_NOMEM; }
        fp.rk_ctl = (Rk45Ctl*)((uint8_t*)fp.rk_buf + fbytes);
        fp.rk_part = (double*)((uint8_t*)fp.rk_ctl + cbytes);
        CUDA_TRY(cudaMemsetAsync(fp.rk_buf, 0, bytes, st));
    }
    if (!h.h_rk) {
        CUDA_TRY(cudaMallocHost((void**)&h.h_rk, sizeof(Rk45Status)));
        for (auto& e : h.rk_ev) CUDA_TRY(cudaEventCreate(&e));
    }
    return FLO_OK;
}

int flo_integrate_rk45(flo_unet_t* hh, float* y, double t0, double t1, double rtol, double atol, float t_scale,
                       const int64_t* class_ids, float cfg_strength, int max_steps, int counts[3], int B, void* stream) {
    // argument checks first: they need neither a handle nor a device
    if (!(rtol > 0)) { set_error("rtol must be > 0, got %g", rtol); return FLO_ERR_INVALID; }
    if (!(atol >= 0)) { set_error("atol must be >= 0, got %g", atol); return FLO_ERR_INVALID; }
    if (!(t1 > t0) || !isfinite(t0) || !isfinite(t1)) { set_error("need finite t0 < t1, got t0=%g t1=%g", t0, t1); return FLO_ERR_INVALID; }
    if (max_steps < 1) { set_error("max_steps must be >= 1, got %d", max_steps); return FLO_ERR_INVALID; }
    Handle* h = reinterpret_cast<Handle*>(hh);
    if (!h || !y || !counts) { set_error("NULL argument"); return FLO_ERR_INVALID; }
    rtol = std::max(rtol, 100 * DBL_EPSILON);             // scipy's validate_tol raises a too small rtol to 100 eps
    counts[0] = counts[1] = counts[2] = 0;
    CUDA_TRY(cudaSetDevice(h->spec.device));
    cudaStream_t st = (cudaStream_t)stream;
    int rc = enter_stream(*h, st);
    if (rc) return rc;
    Plan* pl = nullptr;
    rc = get_plan(*h, B, &pl, st);
    if (rc) return rc;
    const Spec& s = h->spec;
    if (s.n_classes == 0) class_ids = nullptr;              // unet.py:315: no class_cond_mlp -> cond ignored
    const bool use_cls = class_ids != nullptr;
    const bool use_cfg = use_cls && cfg_strength != 0.0f;   // sampling.py:69
    // route: as flo_integrate -- guidance as one 2B-sample forward on the fused path when its last stage is not N-split, else a
    // conditional and a combining pass per evaluation
    Plan* fp = pl;
    int flags = 0, two_pass = use_cfg ? 1 : 0;
    if (use_cfg && s.fused && !getenv("FLO_CFG_TWO_PASS")) {
        Plan* p2 = nullptr;
        rc = get_plan(*h, 2 * B, &p2, st);
        if (rc) return rc;
        const FStage& last = h->stages(p2->fvar).back();
        if (last.kind == 0 && last.cp.nsplit == 1) { fp = p2; flags = SF_CFG_2B; two_pass = 0; }
    }
    const size_t n = (size_t)B * s.channels * s.H * s.W;
    rc = ensure_stage_capacity(*h, 12);
    if (rc) return rc;
    rc = ensure_rk45(*h, *fp, st);
    if (rc) return rc;
    Rk45Params rp{};
    rp.rc = fp->rk_ctl; rp.ctrl = fp->ctrl; rp.k = fp->rk_buf; rp.ybuf = fp->rk_buf + 7 * n;
    rp.xs = fp->xs; rp.xs2 = (flags & SF_CFG_2B) ? fp->xs + n : nullptr; rp.part = fp->rk_part; rp.n = (int)n;
    CUDA_TRY(cudaMemcpyAsync(rp.ybuf, y, n * sizeof(float), cudaMemcpyDeviceToDevice, st));
    if (use_cls) CUDA_TRY(cudaMemcpyAsync(fp->cls, class_ids, (size_t)B * sizeof(int64_t), cudaMemcpyDeviceToDevice, st));
    Ctrl c{};
    c.step = 0; c.done_ctr = 0; c.film_per_sample = use_cls ? 1 : 0; c.n_stages = two_pass ? 12 : 6; c.cfg = cfg_strength;
    c.cfg_half = (flags & SF_CFG_2B) ? B : 0;
    c.y = rp.ybuf;          // read (and ignored) by the ST_STORE epilogues
    c.acc = fp->acc; c.xs = fp->xs; c.vcond = fp->vcond; c.vout = nullptr; c.vtrace = rp.k;
    c.film = fp->film_ps; c.stages = h->d_stages; c.pair_flags = fp->pair_flags;
    CUDA_TRY(launch_setup_ctrl(fp->ctrl, c, nullptr, nullptr, st));
    Rk45Ctl r{};
    r.t = t0; r.t_new = t0; r.t1 = t1; r.rtol = rtol; r.atol = atol; r.max_step = INFINITY; r.interval = fabs(t1 - t0);
    r.t_scale = t_scale; r.max_steps = max_steps; r.k0 = 0; r.two_pass = two_pass; r.flags = flags;
    r.status.state = RK_RUNNING; r.status.t = t0;
    CUDA_TRY(launch_rk45_setup(fp->rk_ctl, r, fp->ctrl, st));
    h->launches += 2;
    // time embedding inside the evaluation: the stage time comes from the stage table the controller wrote.  Unconditional:
    // one batch-uniform FiLM row; class conditioning: one row per sample (per half on the 2B route).
    TembParams tp = temb_params(*h);
    tp.ctrl = fp->ctrl; tp.t = nullptr; tp.t_stride = 0; tp.film = fp->film_ps;
    tp.cls = use_cls ? fp->cls : nullptr; tp.n_cond = use_cls ? B : -1;
    tp.n_rows = !use_cls ? 1 : ((flags & SF_CFG_2B) ? 2 * B : B);
    TembParams tp_nc = tp;                                  // the unconditional pass of the two-pass route
    tp_nc.n_cond = 0;
    auto evaluate = [&](cudaStream_t ss) -> int {
        for (int pass = 0; pass < (two_pass ? 2 : 1); ++pass) {
            if (launch_temb(pass ? tp_nc : tp, ss) != cudaSuccess) { set_error("k_temb launch failed"); return FLO_ERR_CUDA; }
            for (int i = 0; i < n_units(*h); ++i) {
                int r2 = launch_unit(*h, *fp, i, ss);
                if (r2) return r2;
            }
        }
        return FLO_OK;
    };
    auto attempt = [&](cudaStream_t ss) -> int {
        for (int e = 1; e <= 6; ++e) {
            if (launch_rk45_stage(rp, e, ss) != cudaSuccess) { set_error("k_rk45_stage launch failed"); return FLO_ERR_CUDA; }
            int r2 = evaluate(ss);
            if (r2) return r2;
        }
        if (launch_rk45_end(rp, RK_END_STEP, ss) != cudaSuccess) { set_error("k_rk45_end launch failed"); return FLO_ERR_CUDA; }
        return FLO_OK;
    };
    const int64_t per_eval = (int64_t)(two_pass ? 2 : 1) * (n_units(*h) + 1);
    // select_initial_step: f0 = fun(t0, y0), the norms d0 / d1, a trial evaluation at t0 + h0, d2 -> first step
    CUDA_TRY(launch_rk45_stage(rp, 0, st));
    if ((rc = evaluate(st))) return rc;
    CUDA_TRY(launch_rk45_end(rp, RK_END_NORM0, st));
    CUDA_TRY(launch_rk45_stage(rp, -1, st));
    if ((rc = evaluate(st))) return rc;
    CUDA_TRY(launch_rk45_end(rp, RK_END_NORM1, st));
    h->launches += 2 * per_eval + 4;
    const bool graphs = !(s.flags & FLO_FLAG_NO_GRAPH);
    const int64_t key = (int64_t)B * 8 + (use_cls ? 4 : 0) + (flags ? 2 : 0) + two_pass;
    if (graphs && (!fp->graph_rk || fp->graph_rk_key != key)) {
        if (fp->graph_rk) { cudaGraphExecDestroy(fp->graph_rk); fp->graph_rk = nullptr; }
        cudaGraph_t g = nullptr;
        CUDA_TRY(cudaStreamBeginCapture(h->capture_stream, cudaStreamCaptureModeThreadLocal));
        int r2 = attempt(h->capture_stream);
        cudaError_t ce = cudaStreamEndCapture(h->capture_stream, &g);
        if (r2 == FLO_OK && ce == cudaSuccess) ce = cudaGraphInstantiate(&fp->graph_rk, g, 0);
        if (g) cudaGraphDestroy(g);
        if (r2 || ce != cudaSuccess) { if (!r2) set_error("graph capture (RK45) failed: %s", cudaGetErrorString(ce)); return r2 ? r2 : FLO_ERR_CUDA; }
        fp->graph_rk_key = key;
    }
    Rk45Status* hs = h->h_rk;
    auto read_status = [&]() -> int {
        CUDA_TRY(cudaMemcpyAsync(hs, &fp->rk_ctl->status, sizeof(Rk45Status), cudaMemcpyDeviceToHost, st));
        CUDA_TRY(cudaEventRecord(h->rk_ev[2], st));
        CUDA_TRY(cudaEventSynchronize(h->rk_ev[2]));
        return FLO_OK;
    };
    if ((rc = read_status())) return rc;
    double wall_ms = 0, graph_ms = 0;
    int attempts = 0;
    while (hs->state == RK_RUNNING) {
        const auto w0 = std::chrono::steady_clock::now();
        CUDA_TRY(cudaEventRecord(h->rk_ev[0], st));
        if (graphs) CUDA_TRY(cudaGraphLaunch(fp->graph_rk, st));
        else if ((rc = attempt(st))) return rc;
        CUDA_TRY(cudaEventRecord(h->rk_ev[1], st));
        if ((rc = read_status())) return rc;
        const auto w1 = std::chrono::steady_clock::now();
        float ms = 0.f;
        CUDA_TRY(cudaEventElapsedTime(&ms, h->rk_ev[0], h->rk_ev[1]));
        wall_ms += std::chrono::duration<double, std::milli>(w1 - w0).count();
        graph_ms += ms;
        ++attempts;
        h->launches += 6 * (per_eval + 1) + 1;
    }
    h->rk_timing[0] = attempts; h->rk_timing[1] = wall_ms; h->rk_timing[2] = graph_ms;
    counts[0] = hs->nfev; counts[1] = hs->accepted; counts[2] = hs->rejected;
    if (hs->state == RK_TOO_SMALL) {
        set_error("RK45 step size fell below the minimum step at t=%.17g after %d accepted and %d rejected steps "
                  "(scipy: 'Required step size is less than spacing between numbers.')", hs->t, hs->accepted, hs->rejected);
        return FLO_ERR_STEP;
    }
    if (hs->state != RK_DONE) {
        set_error("RK45 used max_steps=%d attempts and stopped at t=%.17g (%d accepted, %d rejected)", max_steps, hs->t,
                  hs->accepted, hs->rejected);
        return FLO_ERR_STEP;
    }
    CUDA_TRY(cudaMemcpyAsync(y, rp.ybuf + (size_t)hs->y_idx * n, n * sizeof(float), cudaMemcpyDeviceToDevice, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    return FLO_OK;
}

int flo_integrate_rk45_timing(flo_unet_t* hh, double out[3]) {
    Handle* h = reinterpret_cast<Handle*>(hh);
    if (!h || !out) { set_error("NULL argument"); return FLO_ERR_INVALID; }
    for (int i = 0; i < 3; ++i) out[i] = h->rk_timing[i];
    return FLO_OK;
}

int flo_unet_set_time_freqs(flo_unet_t* hh, const float* freqs, int n) {
    Handle* h = reinterpret_cast<Handle*>(hh);
    if (!h || !freqs) { set_error("NULL argument"); return FLO_ERR_INVALID; }
    if (n != h->spec.dim / 2) { set_error("expected %d frequencies, got %d", h->spec.dim / 2, n); return FLO_ERR_INVALID; }
    CUDA_TRY(cudaSetDevice(h->spec.device));
    CUDA_TRY(cudaDeviceSynchronize());
    CUDA_TRY(cudaMemcpy(h->d_f32 + h->o_freqs, freqs, (size_t)n * sizeof(float), cudaMemcpyHostToDevice));
    return FLO_OK;
}

// Host-only: build the op program for `cfg` (zero weights) and describe ops, buffers and tcgen05 tilings.
int flo_describe_plan(const flo_unet_cfg* cfg, int B, char* out, int cap) {
    Handle h;
    int rc = make_spec(cfg, h.spec);
    if (rc) return rc;
    h.params = manifest(h.spec);
    for (auto& pi : h.params) h.host[pi.name].assign((size_t)pi.numel(), 0.f);
    Builder b(h);
    rc = b.build();
    if (rc) return rc;
    rc = check_op_kernels(h);
    if (rc) return rc;
    allocate_arena(h);
    std::string t;
    char line[512];
    snprintf(line, sizeof(line), "ops=%d bufs=%d film_dim=%d arena_bytes_per_sample=%zu f32_blob=%zu bf16_blob=%zu\n",
             (int)h.ops.size(), (int)h.bufs.size(), h.film_dim, h.arena_ps, h.blob_f32.size(), h.blob_bf16.size());
    t += line;
    static const char* kinds[] = {"init", "conv", "gn", "linattn", "midattn", "final"};
    auto bn = [&](int id) { return id >= 0 ? h.bufs[id].name.c_str() : "-"; };
    for (size_t i = 0; i < h.ops.size(); ++i) {
        const Op& op = h.ops[i];
        if (op.kind == OP_CONV) {
            snprintf(line, sizeof(line), "%3zu conv    %-28s %dx%d k=%d cin=%d+%d cout=%d in0=%s in1=%s res=%s out_m=%s out_o=%s", i,
                     op.name.c_str(), op.H, op.W, op.ksize, op.ncb0 * 8, op.ncb1 * 8, op.cout, bn(op.in0), bn(op.in1), bn(op.res),
                     bn(op.out_m), bn(op.out_o));
            t += line;
            if (h.spec.bf16) {
                ConvUmmaParams up;
                ConvShape cs{op.name.c_str(), op.H, op.W, op.ksize, op.ncb0, op.ncb1, op.cout, op.n_tile};
                if (plan_umma(cs, B, up) == FLO_OK) {
                    snprintf(line, sizeof(line), " | nb=%d mt=%d n_tile=%d sbo=%d S=%d stages=%d smem=%d tmem=%d ctas=%d", up.nb,
                             up.n_mtiles, up.n_tile, up.sbo_px, up.slices_per_stage, up.n_wstages, up.smem_bytes, up.tmem_cols,
                             ((B + up.nb - 1) / up.nb) * (op.cout / up.n_tile));
                    t += line;
                } else {
                    t += " | UNSUPPORTED: " + g_last_error;
                }
            }
            t += "\n";
        } else if (op.kind == OP_GN) {
            snprintf(line, sizeof(line), "%3zu gn      %-28s C=%d %dx%d groups=%d film=%d silu=%d in=%s res=%s out_m=%s out_o=%s un=%s up=%s", i,
                     op.name.c_str(), op.C, op.H, op.W, op.groups, op.film_off, op.silu, bn(op.gn_in), bn(op.res), bn(op.out_m),
                     bn(op.out_o), bn(op.out_un), bn(op.out_up));
            t += line;
            // the kernel launch_gn runs; the fused stage kernels normalise in their own epilogues and never launch it
            if (!h.spec.fused) t += std::string(" gn=") + gn_variant_name(gn_variant(op.C, op.H, op.W, op.groups, h.spec.bf16));
            t += "\n";
        } else if (op.kind == OP_LINATTN || op.kind == OP_MIDATTN) {
            snprintf(line, sizeof(line), "%3zu %-7s %-28s n=%d qkv=%s out=%s\n", i, kinds[op.kind], op.name.c_str(), op.n, bn(op.qkv),
                     bn(op.attn_out));
            t += line;
        } else {
            snprintf(line, sizeof(line), "%3zu %-7s %-28s in=%s out_m=%s out_o=%s\n", i, kinds[op.kind], op.name.c_str(), bn(op.gn_in),
                     bn(op.out_m), bn(op.out_o));
            t += line;
        }
    }
    for (size_t i = 0; i < h.bufs.size(); ++i) {
        const Buf& bf = h.bufs[i];
        snprintf(line, sizeof(line), "buf %3zu %-34s C=%d %dx%d %s bytes_ps=%zu live=[%d,%d] off_ps=%zu\n", i, bf.name.c_str(), bf.C, bf.H,
                 bf.W, bf.bf16 ? "bf16" : "f32 ", bf.bytes_ps, bf.def, bf.last, bf.off_ps);
        t += line;
    }
    if (h.spec.fused) {
        FusedBuilder fb(h, h.ftensors, h.fstages, 4);
        rc = fb.build();
        if (rc) return rc;
        snprintf(line, sizeof(line), "fused: %d stages, %d boundary tensors, %zu bytes/sample\n", (int)h.fstages.size(),
                 (int)h.ftensors.size(), h.farena_ps);
        t += line;
        for (size_t i = 0; i < h.fstages.size(); ++i) {
            const FStage& st = h.fstages[i];
            if (st.kind == 0) {
                const ChainParams& c = st.cp;
                snprintf(line, sizeof(line), "stage %2zu chain %-12s %dx%d nb=%d mt=%d strips=%d steps=%d loads=%d smem=%d (slots %d, ring %dx%d) tmem=%d nsplit=%d ctas=%d\n",
                         i, st.name.c_str(), c.H, c.W, c.nb, c.n_mtiles, c.strips, c.n_steps, c.n_loads, c.smem_bytes, c.ring_off,
                         c.n_ring, c.ring_slot_bytes, c.tmem_cols, c.nsplit, c.nsplit * ((B + c.nb - 1) / c.nb));
                t += line;
                for (int k = 0; k < c.n_steps; ++k) {
                    const ChainStep& cs = c.st[k];
                    snprintf(line, sizeof(line), "      step %d: conv=%d k=%d cin=%d+%d n=%d chunks=%dx%d res=%d(%dx%d) epi=%d C=%d G=%d film=%d resmode=%d out_slot=%d out_g=%d un=%d up=%d pn=%d final=%d a0=%d a1=%d\n",
                             k, cs.has_conv, cs.ksize, cs.a0_ncb * 8, cs.a1_ncb * 8, cs.n, cs.slices, cs.slices_per_chunk, cs.has_res,
                             cs.res_slices, cs.res_slices_per_chunk, cs.epi, cs.C, cs.groups, cs.film_off, cs.res_mode, cs.out_slot_off,
                             cs.out_g, cs.out_un_g, cs.out_up_g, cs.pn_g, cs.final, cs.a0_off, cs.a1_off);
                    t += line;
                }
            } else {
                const AttnFusedParams& a = st.ap;
                snprintf(line, sizeof(line), "stage %2zu attn  %-12s %dx%d C=%d nb=%d n=%d n_pad=%d mt=%d full=%d smem=%d plane=%d tmem=%d cols(k=%d v=%d ctx=%d q=%d out=%d proj=%d) ctas=%d\n",
                         i, st.name.c_str(), a.H, a.W, a.C, a.nb, a.n, a.n_pad, a.n_mtiles, a.full, a.smem_bytes, a.plane_bytes, a.tmem_cols,
                         a.col_k, a.col_v, a.col_ctx, a.col_q, a.col_out, a.col_proj, (B + a.nb - 1) / a.nb);
                t += line;
            }
        }
        for (size_t i = 0; i < h.ftensors.size(); ++i) {
            snprintf(line, sizeof(line), "ftensor %2zu %-24s C=%d %dx%d off_ps=%zu\n", i, h.ftensors[i].name.c_str(), h.ftensors[i].C,
                     h.ftensors[i].H, h.ftensors[i].W, h.ftensors[i].off_ps);
            t += line;
        }
    }
    if (out && cap > 0) snprintf(out, cap, "%s", t.c_str());
    return (int)t.size();
}

// algorithmic flops / bytes of one layer-by-layer op (per sample)
static void op_cost(const Handle& h, const Op& op, double& fl, double& by) {
    const Spec& s = h.spec;
    const double ob = s.bf16 ? 2.0 : 4.0;      // operand bytes
    fl = 0; by = 0;
    const double hw = (double)op.H * op.W;
    switch (op.kind) {
        case OP_INIT:
            fl = 2.0 * hw * s.dim * s.channels;
            by = hw * (s.channels * 4.0 + s.dim * (ob + (s.bf16 ? 4.0 : 0.0)));
            break;
        case OP_CONV: {
            const double cin = (op.ncb0 + op.ncb1) * 8.0;
            fl = 2.0 * hw * op.cout * cin * op.ksize * op.ksize;
            by = hw * cin * ob + hw * op.cout * ((op.out_m >= 0 ? 4.0 : 0.0) + (op.out_o >= 0 ? ob : 0.0) + (op.res >= 0 ? 4.0 : 0.0));
        } break;
        case OP_GN:
            by = hw * op.C * (4.0 + (op.res >= 0 ? 4.0 : 0.0) + (op.out_m >= 0 ? 4.0 : 0.0) + (op.out_o >= 0 ? ob : 0.0) +
                              (op.out_un >= 0 ? ob : 0.0) + (op.out_up >= 0 ? 4.0 * ob : 0.0));
            fl = 10.0 * hw * op.C;
            break;
        case OP_LINATTN:
            fl = 4.0 * 2.0 * 2.0 * 32.0 * 32.0 * op.n;        // 4 heads x (context + output) einsums (unet.py:146,148)
            by = op.n * (384.0 + 128.0) * ob;
            break;
        case OP_MIDATTN:
            fl = 4.0 * 2.0 * 2.0 * 32.0 * op.n * op.n;
            by = op.n * (384.0 + 128.0) * ob;
            break;
        case OP_FINAL:
            fl = 2.0 * hw * s.dim * s.channels;
            by = hw * (s.dim * 4.0 + s.channels * 16.0);
            break;
    }
}

// Launch units of the active path: layer-by-layer ops, or fused stages.
// kind: 0 init conv, 1 conv, 2 GroupNorm pass, 3 linear attention core, 4 mid attention core, 5 final conv + integrator
//       epilogue, 6 fused conv-chain stage (k_chain), 7 fused attention stage (k_attn).
// flops = algorithmic CONV flops inside the unit (2*M*N*K, SURVEY.md 8d); bytes = algorithmic global-memory bytes.
int flo_unet_op_info(flo_unet_t* hh, int index, int* kind, double* flops_per_sample, double* bytes_per_sample) {
    Handle* h = reinterpret_cast<Handle*>(hh);
    if (!h || index < 0 || index >= n_units(*h)) { set_error("op index out of range"); return FLO_ERR_INVALID; }
    double fl = 0, by = 0;
    int k = 0;
    if (!h->spec.fused) {
        const Op& op = h->ops[index];
        op_cost(*h, op, fl, by);
        k = op.kind;
    } else {
        const FStage& st = h->fstages[index];
        auto tbytes = [&](int t) { return t >= 0 ? (double)h->ftensors[t].C * h->ftensors[t].H * h->ftensors[t].W * 2.0 : 0.0; };
        if (st.kind == 0) {
            k = 6;
            const ChainParams& c = st.cp;
            const double hw = (double)c.H * c.W;
            for (int i = 0; i < c.n_steps; ++i) {
                const ChainStep& cs = c.st[i];
                if (cs.epi == CE_INIT) fl += 2.0 * hw * h->spec.dim * h->spec.channels;
                if (!cs.has_conv) continue;
                const double cin = (cs.a0_ncb + cs.a1_ncb) * 8.0;
                // cs.C = all output channels of the step (cs.n is the per-CTA slice of an N-split stage)
                fl += 2.0 * hw * cs.C * cin * cs.ksize * cs.ksize;
                if (cs.has_res) fl += 2.0 * hw * cs.C * cin;
                if (cs.final) fl += 2.0 * hw * h->spec.dim * h->spec.channels;
            }
            for (int m = 0; m < st.n_maps; ++m) by += tbytes(st.map_tensor[m]);
            for (int g = 0; g < CH_MAX_GT; ++g) by += tbytes(st.gt_tensor[g]);
        } else {
            k = 7;
            const AttnFusedParams& a = st.ap;
            fl = 2.0 * a.n * a.C * 384.0 + 2.0 * a.n * 128.0 * a.C;          // to_qkv + to_out 1x1 convs
            by = tbytes(st.map_tensor[0]) + tbytes(st.x2_t) + tbytes(st.out_t) + tbytes(st.out_un_t) + tbytes(st.out_up_t);
        }
    }
    if (kind) *kind = k;
    if (flops_per_sample) *flops_per_sample = fl;
    if (bytes_per_sample) *bytes_per_sample = by;
    return FLO_OK;
}

int flo_unet_profile_ops(flo_unet_t* hh, int B, int reps, float* ms_per_op, void* stream) {
    Handle* h = reinterpret_cast<Handle*>(hh);
    if (!h || !ms_per_op || reps < 1) { set_error("bad argument"); return FLO_ERR_INVALID; }
    CUDA_TRY(cudaSetDevice(h->spec.device));
    cudaStream_t st = (cudaStream_t)stream;
    int rc = enter_stream(*h, st);
    if (rc) return rc;
    Plan* pl = nullptr;
    rc = get_plan(*h, B, &pl, st);
    if (rc) return rc;
    const int n_ops = n_units(*h);
    rc = ensure_stage_capacity(*h, 1);
    if (rc) return rc;
    // a plain forward on the current contents of the state buffers, FiLM rows for t = 500
    std::vector<float> tvals(B, 500.0f);
    float* d_t = nullptr;
    CUDA_TRY(cudaMalloc((void**)&d_t, (size_t)B * sizeof(float)));
    CUDA_TRY(cudaMemcpy(d_t, tvals.data(), (size_t)B * sizeof(float), cudaMemcpyHostToDevice));
    TembParams tp = temb_params(*h);
    tp.t = d_t; tp.t_stride = 1; tp.cls = nullptr; tp.n_rows = B; tp.film = pl->film_ps;
    CUDA_TRY(launch_temb(tp, st));
    Ctrl c{};
    c.film_per_sample = 1; c.n_stages = 1;
    c.y = pl->y; c.acc = pl->acc; c.xs = pl->xs; c.vcond = pl->vcond; c.vout = pl->vcond; c.film = pl->film_ps; c.stages = h->d_stages;
    Stage s0{};
    s0.kind = ST_PLAIN; s0.eval_idx = -1;
    std::vector<cudaEvent_t> ev(n_ops + 1);
    for (auto& e : ev) CUDA_TRY(cudaEventCreate(&e));
    std::vector<float> best(n_ops, 1e30f);
    for (int r = 0; r < reps + 1; ++r) {
        CUDA_TRY(launch_setup_ctrl(pl->ctrl, c, h->d_stages, &s0, st));
        for (int i = 0; i < n_ops; ++i) {
            CUDA_TRY(cudaEventRecord(ev[i], st));
            rc = launch_unit(*h, *pl, i, st);
            if (rc) return rc;
        }
        CUDA_TRY(cudaEventRecord(ev[n_ops], st));
        CUDA_TRY(cudaStreamSynchronize(st));
        if (r == 0) continue;      // warm-up
        for (int i = 0; i < n_ops; ++i) {
            float ms = 0.f;
            CUDA_TRY(cudaEventElapsedTime(&ms, ev[i], ev[i + 1]));
            best[i] = std::min(best[i], ms);
        }
    }
    for (int i = 0; i < n_ops; ++i) ms_per_op[i] = best[i];
    for (auto& e : ev) cudaEventDestroy(e);
    cudaFree(d_t);
    h->launches += (int64_t)(reps + 1) * (n_ops + 1) + 1;
    return FLO_OK;
}

// debug: clock64 timeline of CTA 0 of fused chain stage `stage` (needs env FLO_TIMELINE=1 at plan creation)
int flo_unet_read_timeline(flo_unet_t* hh, int B, int stage, long long* out128) {
    Handle* h = reinterpret_cast<Handle*>(hh);
    if (!h || !out128) { set_error("NULL argument"); return FLO_ERR_INVALID; }
    auto it = h->plans.find(B);
    if (it == h->plans.end() || !it->second->dbg || stage < 0 || stage >= (int)h->fstages.size()) { set_error("no timeline"); return FLO_ERR_INVALID; }
    CUDA_TRY(cudaSetDevice(h->spec.device));
    CUDA_TRY(cudaDeviceSynchronize());
    CUDA_TRY(cudaMemcpy(out128, it->second->dbg + stage * 128, 128 * sizeof(long long), cudaMemcpyDeviceToHost));
    return FLO_OK;
}

int flo_unet_num_ops(flo_unet_t* hh) {
    Handle* h = reinterpret_cast<Handle*>(hh);
    return h ? n_units(*h) : 0;
}
int flo_unet_op_name(flo_unet_t* hh, int index, char* name, int name_cap) {
    Handle* h = reinterpret_cast<Handle*>(hh);
    if (!h || index < 0 || index >= n_units(*h)) { set_error("op index out of range"); return FLO_ERR_INVALID; }
    snprintf(name, name_cap, "%s", h->spec.fused ? h->fstages[index].name.c_str() : h->ops[index].name.c_str());
    return FLO_OK;
}
int flo_unet_launches_per_forward(flo_unet_t* hh, int B) {
    Handle* h = reinterpret_cast<Handle*>(hh);
    (void)B;
    return h ? n_units(*h) : 0;
}
int64_t flo_unet_launch_count(flo_unet_t* hh) {
    Handle* h = reinterpret_cast<Handle*>(hh);
    return h ? h->launches : 0;
}

int flo_unet_read_activation(flo_unet_t* hh, const char* name, int B, float* out, int64_t cap, int64_t shape[4],
                             void* stream) {
    Handle* h = reinterpret_cast<Handle*>(hh);
    if (!h || !name || !out) { set_error("NULL argument"); return FLO_ERR_INVALID; }
    if (!(h->spec.flags & FLO_FLAG_NO_BUFFER_REUSE)) { set_error("read_activation needs FLO_FLAG_NO_BUFFER_REUSE"); return FLO_ERR_INVALID; }
    CUDA_TRY(cudaSetDevice(h->spec.device));
    auto it = h->plans.find(B);
    if (it == h->plans.end()) { set_error("no forward has run at B=%d", B); return FLO_ERR_INVALID; }
    Plan& pl = *it->second;
    const std::string n(name);
    int C = 0, H = 0, W = 0, elem = 0;      // elem: 0 fp32, 1 bf16, 2 fp16
    const void* src_ptr = nullptr;
    if (h->spec.fused) {
        for (size_t i = 0; i < h->ftensors.size(); ++i)
            if (h->ftensors[i].name == n) {
                const FTensor& t = h->ftensors[i];
                C = t.C; H = t.H; W = t.W; elem = h->spec.f16 ? 2 : 1;
                src_ptr = pl.farena + t.off_ps * (size_t)B;
                break;
            }
    } else {
        int id = -1;
        for (const char* suffix : {"", ":m", ":o"}) {
            for (size_t i = 0; i < h->bufs.size(); ++i)
                if (h->bufs[i].name == n + suffix) { id = (int)i; break; }
            if (id >= 0) break;
        }
        if (id >= 0) {
            const Buf& b = h->bufs[id];
            C = b.C; H = b.H; W = b.W; elem = b.bf16 ? 1 : 0;
            src_ptr = pl.buf_ptr[id];
        }
    }
    if (!src_ptr) { set_error("no activation named '%s'", name); return FLO_ERR_INVALID; }
    const int64_t numel = (int64_t)B * C * H * W;
    if (numel > cap) { set_error("output buffer too small"); return FLO_ERR_INVALID; }
    CUDA_TRY(cudaStreamSynchronize((cudaStream_t)stream));
    std::vector<uint8_t> raw((size_t)numel * (elem ? 2 : 4));
    CUDA_TRY(cudaMemcpy(raw.data(), src_ptr, raw.size(), cudaMemcpyDeviceToHost));
    const int HW = H * W;
    for (int cb = 0; cb < C / 8; ++cb)
        for (int bb = 0; bb < B; ++bb)
            for (int px = 0; px < HW; ++px)
                for (int j = 0; j < 8; ++j) {
                    const size_t src = (((size_t)cb * B + bb) * HW + px) * 8 + j;
                    float v;
                    if (elem == 1) v = __bfloat162float(reinterpret_cast<const __nv_bfloat16*>(raw.data())[src]);
                    else if (elem == 2) v = __half2float(reinterpret_cast<const __half*>(raw.data())[src]);
                    else v = reinterpret_cast<const float*>(raw.data())[src];
                    out[((size_t)bb * C + cb * 8 + j) * HW + px] = v;
                }
    shape[0] = B; shape[1] = C; shape[2] = H; shape[3] = W;
    return FLO_OK;
}

}  // extern "C"
