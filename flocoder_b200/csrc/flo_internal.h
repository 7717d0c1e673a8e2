// Internal declarations shared by the flocoder_b200 translation units (not part of the C ABI).
//
// Activation layout ("blocked"): a tensor with C channels (C % 8 == 0) at H x W for B samples is
// stored as [C/8][B][H][W][8] -- channel-blocks outermost, 8 channels innermost.  One 8-channel
// pixel is 16 B in bf16 / 32 B in fp32, which is (a) the 16-byte row of a tcgen05 no-swizzle
// K-major core matrix, so a TMA box of the padded image is directly a UMMA A operand whose 3x3
// taps are shifted start addresses, and (b) a full vector load for the elementwise kernels.
#pragma once
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#include <cuda.h>
#include <stdint.h>
#include <string>
#include <vector>

#include "../../include/flocoder_b200.h"

namespace flo {

// ---------------------------------------------------------------------------------------------
// device-resident control block: everything that changes between replays of the forward graph
// ---------------------------------------------------------------------------------------------
enum StageKind : int {
    ST_PLAIN = 0,     // write v to ctrl.vout                              (Unet.forward)
    ST_RK1 = 1,       // acc = k;        xs = y + (dt*k)/2                 (sampling.py:43,45)
    ST_RK2 = 2,       // acc += 2k;      xs = y + (dt*k)/2                 (sampling.py:45,46)
    ST_RK3 = 3,       // acc += 2k;      xs = y + dt*k                     (sampling.py:46,47)
    ST_RK4 = 4,       // acc += k;       y += (dt/6)*acc; xs = y           (sampling.py:48)
    ST_EULER = 5,     // y = y + k*dt;   xs = y                            (legacy/train_sd_flowers.py:64)
    ST_CFG_COND = 6,  // vcond = k (conditional pass of classifier-free guidance, sampling.py:63)
    ST_STORE = 7      // only vtrace[eval_idx] = k: the RK45 stage slot; k_rk45_stage forms the next input (rk45.cu)
};
enum StageFlags : int {
    SF_CFG_COMBINE = 1,  // this pass is the unconditional one: k = k + cfg*(vcond - k)  (sampling.py:74)
    SF_CFG_2B = 2        // ONE pass over 2B samples: [0,B) conditional, [B,2B) unconditional (ctrl.cfg_half = B); the later of
                         // the two CTAs holding a sample's halves combines them and does the integrator update
};

struct Stage {
    float t_scaled;   // fl32(t) * t_scale, the value fed to the U-Net (sampling.py:63)
    float dt;
    float dt6;        // dt / 6 in fp32 (sampling.py:48)
    int kind;
    int film_row;     // row of the FiLM table for a batch-uniform time
    int flags;
    int eval_idx;     // index of this velocity evaluation in ctrl.vtrace, or -1
    int pad;
};

struct Ctrl {
    int step;             // index of the current stage; advanced by the last CTA of the final kernel
    int done_ctr;
    int film_per_sample;  // 1: FiLM row = sample index (per-sample time / class conditioning)
    int n_stages;
    float cfg;
    int cfg_half;         // SF_CFG_2B: B (the forward runs on 2B samples); else 0
    float* y;             // [B,C,H,W] integrator state
    float* acc;           // [B,C,H,W] running k1+2k2+2k3+k4
    float* xs;            // [B,C,H,W] input of the current U-Net evaluation
    float* vcond;         // [B,C,H,W] conditional velocity (CFG)
    float* vout;          // ST_PLAIN destination
    float* vtrace;        // optional [n_eval,B,C,H,W]
    const float* film;    // FiLM table [rows][film_dim]
    const Stage* stages;
    int* pair_flags;      // SF_CFG_2B: [B] arrival counters of the sample halves (zero between passes)
};

// ---------------------------------------------------------------------------------------------
// kernel parameter blocks
// ---------------------------------------------------------------------------------------------
struct InitConvParams {
    const Ctrl* ctrl;
    const float* w;       // [dim][cin]
    const float* bias;    // [dim]
    float* out_m;         // fp32 blocked or null
    void* out_o;          // operand blocked (bf16 or fp32) or null
    int B, HW, cin, dim, o_is_bf16;
};

struct ConvSimtParams {
    const void* in0; const void* in1;   // blocked sources (operand dtype), in1 may be null
    int ncb0, ncb1;                     // channel blocks per source
    int in_is_bf16;
    const float* w;                     // [taps][cin][cout]
    const float* bias;                  // [cout] or null
    const float* res;                   // fp32 blocked residual or null
    float* out_m; void* out_o;          // fp32 blocked / operand blocked (either may be null)
    int o_is_bf16;
    int B, H, W, cout, ksize;
    // inpainting mask branches (unet.py:298-305,336-340,360-364): out = res + SiLU(conv + bias), the pixel-unshuffled /
    // nearest-x2 copies the following Downsample / Upsample conv reads, and the run-time bypass
    int act_silu;                       // SiLU on (conv + bias) before the residual is added
    void* out_unshuf; void* out_up;     // operand copies as in GnParams, or null
    const int* mask_mode;               // device flag (0 no mask, 1 mask all ones, 2 mask in use), or null
    int need_mode;                      // the op runs when *mask_mode >= need_mode ...
    const float* bypass;                // ... else out = bypass (fp32 blocked, same shape), or nothing is written if null
};

// cond['mask_cond'] [B,ch,H,W] (NCHW fp32) -> one blocked 8-channel fp32 tensor per resolution level (bilinear,
// F.interpolate(..., mode='bilinear'), unet.py:338,362) + the "mask in use" flag (unet.py:301 torch.allclose)
struct MaskPrepParams {
    const float* mask;
    float* out[8];
    int n_levels, B, ch, H, W;
    int* mode;
};

struct GnParams {
    const Ctrl* ctrl;
    const float* in;      // fp32 blocked [C/8][B][HW][8]
    const float* res;     // fp32 blocked residual or null
    const float* gamma; const float* beta;
    float* out_m;         // fp32 blocked or null
    void* out_o;          // operand blocked or null
    void* out_unshuf;     // operand [4*C/8][B][H/2][W/2][8] or null  (pixel-unshuffle, unet.py:52)
    void* out_up;         // operand [C/8][B][2H][2W][8] or null      (nearest x2, unet.py:44)
    int o_is_bf16;
    int B, C, H, W, groups;
    int film_off;         // offset of this block's (scale|shift) in a FiLM row, or -1
    int film_dim;
    int silu;
};

struct AttnParams {
    const void* qkv;      // operand blocked [48][B][n][8]   (q | k | v, 4 heads x 32)
    void* out;            // operand blocked [16][B][n][8]
    int is_bf16;
    int B, n;
};

struct TembParams {
    const Ctrl* ctrl;                    // non-null: every row's time is the current ODE stage's (ctrl->stages[ctrl->step].t_scaled),
                                         // so the launch can sit inside the replayed forward graph
    int n_cond;                          // rows [0, n_cond) use their class id, the rest are unconditional (< 0: all rows)
    const float* t; int t_stride;        // time per row (already scaled); stride 0 = same for all rows
    const int64_t* cls;                  // class id per row or null
    int n_rows;
    float* film;                         // [n_rows][film_dim]
    int dim, time_dim, film_dim, n_classes;
    const float* freqs;                  // [dim/2]
    const float* w1t; const float* b1;   // [dim][time_dim]
    const float* w2t; const float* b2;   // [time_dim][time_dim]
    const float* emb;                    // [n_classes][time_dim]
    const float* wc1t; const float* bc1;
    const float* wc3t; const float* bc3;
    const float* wft; const float* bf;   // [time_dim][film_dim]
};

struct FinalParams {
    Ctrl* ctrl;
    const float* in;      // fp32 blocked [dim/8][B][HW][8]
    const float* w;       // [channels][dim]
    const float* bias;
    int B, HW, dim, channels;
};

// tcgen05 convolution (conv_umma.cu)
struct ConvUmmaParams {
    const __nv_bfloat16* w;      // packed weight stream for this layer (see pack_umma_weights)
    const float* bias;           // [cout] or null
    const float* res;            // fp32 blocked residual or null
    float* out_m;                // fp32 blocked or null
    __nv_bfloat16* out_o;        // bf16 blocked or null
    int B, H, W;
    int ncb0, ncb1;              // channel blocks of the two (concatenated) sources
    int cout;                    // total output channels
    int n_tile;                  // output channels per CTA (multiple of 16, <= 256)
    int ksize;                   // 1 or 3
    int nb;                      // samples per CTA
    int n_mtiles;                // 128-row M tiles per CTA
    int row0;                    // flattened (padded) pixel index of row 0 of M tile 0
    int tile_stride;             // pixel distance between consecutive M tiles
    int sbo_px;                  // pixel distance between consecutive 8-row groups (8 = flattened)
    int plane_px;                // pixels per channel-block plane in shared memory (nb * Hp * Wp)
    int slices_per_stage;        // K16 slices per weight pipeline stage
    int n_wstages;               // ring depth
    int smem_bytes;
    int tmem_cols;
};

// ---------------------------------------------------------------------------------------------
// launchers (each returns cudaGetLastError())
// ---------------------------------------------------------------------------------------------
cudaError_t launch_setup_ctrl(Ctrl* ctrl_dev, const Ctrl& value, Stage* stage0_dev, const Stage* stage0_value,
                              cudaStream_t s);
cudaError_t launch_init_conv(const InitConvParams& p, cudaStream_t s);
cudaError_t launch_conv_simt(const ConvSimtParams& p, cudaStream_t s);
cudaError_t launch_gn(const GnParams& p, cudaStream_t s);
cudaError_t launch_linattn(const AttnParams& p, cudaStream_t s);
cudaError_t launch_midattn(const AttnParams& p, cudaStream_t s);
cudaError_t launch_temb(const TembParams& p, cudaStream_t s);
cudaError_t launch_final(const FinalParams& p, cudaStream_t s);
cudaError_t launch_mask_prep(const MaskPrepParams& p, cudaStream_t s);   // p.mask == null: *mode = 0 only
cudaError_t launch_gn_any(const GnParams& p, cudaStream_t s);            // any channels-per-group (fp32 path)

// Host-side kernel choices of the layer-by-layer program: the launchers above follow them, and the planner refuses an op
// they give no kernel for before anything is launched.
enum GnVariant { GN_TMA, GN_WARP, GN_CTA, GN_ANY, GN_NONE };
GnVariant gn_variant(int C, int H, int W, int groups, bool bf16);       // the GroupNorm kernel launch_gn runs
const char* gn_variant_name(GnVariant v);                               // "tma", "warp", "cta", "any", "none"
bool linattn_supported(int n, bool bf16);                               // launch_linattn has a kernel for n pixels
bool midattn_supported(int n);                                          // launch_midattn has a kernel for n pixels
cudaError_t launch_conv_umma(const ConvUmmaParams& p, const CUtensorMap& a0, const CUtensorMap& a1,
                             cudaStream_t s);
cudaError_t conv_umma_configure();   // one-time cudaFuncSetAttribute calls
cudaError_t simt_configure();
cudaError_t launch_umma_micro(const __nv_bfloat16* a, const __nv_bfloat16* b, float* d, int N, int K, int a_lbo,
                              int a_sbo, int a_shift, int b_lbo, int b_sbo, cudaStream_t s);

cudaError_t launch_umma_rate(long long* cycles, int N, int n_mma, int n_acc, cudaStream_t s, int a_mode = 0, int a_shift = 0);
cudaError_t launch_stream_rate(const void* src, long long* cycles, int grid, int total_bytes, int chunk_bytes, int n_ring, int pieces,
                               int same_src, cudaStream_t s);
cudaError_t launch_umma_micro2(const __nv_bfloat16* a, const __nv_bfloat16* b, float* d, long long* cycles, int N, int K, int layout,
                               int row_bytes, int a_sbo, int a_shift, int a_lbo, int use_base_offset, int reps, cudaStream_t s);

// tiling of one convolution for the tcgen05 kernel, and the TMA map of a blocked bf16 tensor
struct ConvShape { const char* name; int H, W, ksize, ncb0, ncb1, cout, n_tile; };
int plan_umma(const ConvShape& shape, int B, ConvUmmaParams& p);
int make_tmap(CUtensorMap* tm, void* base, int ncb, int B, int H, int W, int pad, int nb);

// host-side packing of OIHW fp32 weights (with input-channel permutation `perm`, or null) into the
// bf16 stream the tcgen05 kernel consumes; returns elements written.
size_t pack_umma_weights(const float* w_oihw, int cout, int cin, int ksize, const int* perm, int n_tile, bool f16,
                         std::vector<__nv_bfloat16>& out);   // f16: the 16-bit container holds IEEE half bits

// TMA tensor-map encoder obtained through the runtime (no link-time libcuda dependency)
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn get_encode_tiled();

void set_error(const char* fmt, ...);

// ---------------------------------------------------------------------------------------------
// fused stage kernels (fused.cu): a CTA owns `nb` whole samples and runs a chain of convolutions with
// GroupNorm/FiLM/SiLU/residual epilogues entirely on-chip (activations in shared memory, accumulators
// in TMEM, weights streamed by bulk TMA); see DESIGN.md "Fused stage kernels".
// ---------------------------------------------------------------------------------------------
constexpr int MAX_WSTAGES = 8;          // largest depth of the shared-memory weight ring
constexpr int CH_MAX_STEPS = 8;
constexpr int CH_MAX_LOADS = 4;
constexpr int CH_MAX_GT = 10;
enum ChainEpi : int { CE_GN = 1, CE_BIAS = 2, CE_INIT = 3 };

struct ChainStep {
    // ---- MMA part (has_conv == 0: none)
    int has_conv;
    int a0_off, a0_ncb, a1_off, a1_ncb;     // A operand slots: byte offset in smem, channel blocks (a1_ncb = 0: none)
    int ksize, n;                           // kernel size, output channels
    int acc_col;                            // TMEM column of tile 0 (tile t at acc_col + t*n)
    unsigned w_off; int slices, slices_per_chunk;              // weight stream (16-bit elements into wblob): K16 slices
                                                               // incl. the trailing bias slice, slices per ring chunk
    int has_res, res_col; unsigned wres_off; int res_slices, res_slices_per_chunk;   // 1x1 res_conv on the same A
    int tab_idx, res_tab_idx;               // first entry of this conv's A-address table (ChainParams::tab_off)
    int chunk0, res_chunk0;                 // first weight-ring chunk of the conv / res_conv in the stage's chunk list
    // ---- epilogue part
    int epi;                                // ChainEpi
    int C, groups, silu, film_off;          // film_off < 0: no FiLM
    int bias_off, gamma_off, beta_off;      // offsets into fblob (< 0: none)
    int res_mode;                           // 0 none, 1 TMEM (res_col) + res_bias_off, 2 shared-memory slot (16-bit)
    int res_slot_off, res_bias_off;
    int out_slot_off;                       // < 0: none
    int out_g, out_un_g, out_up_g;          // global tensor table indices (< 0: none)
    int pn_g, pn_gamma_off, pn_beta_off;    // fused PreNorm (GroupNorm(1,C) of the result) -> global tensor
    int final;                              // 1: final 1x1 conv + integrator stage update instead of tensor outputs
};

struct ChainParams {
    int n_steps;
    ChainStep st[CH_MAX_STEPS];
    int B, H, W, nb, n_mtiles, strips, plane_px;
    int n_loads, load_off[CH_MAX_LOADS], load_ncb[CH_MAX_LOADS];
    int zero_off, zero_bytes;               // shared-memory range to clear at start (epilogue-written slots)
    int ones_off;                           // 4 KB constant A tile [1,0,...] that multiplies the bias slice
    int fast;                               // 1: the stage runs the warp-shuffle GroupNorm variant of k_chain (one sample per CTA, one
                                            // accumulator chunk per thread in every step)
    int max_c;                              // largest per-step channel count (sizes gpar and the tables of the warp-shuffle GroupNorm path)
    int g_max, coef_n, cpar_n;              // stats region layout: rowstat[rows*g_max] | coef[coef_n] (float2) | cpar[cpar_n] (float) |
                                            // gpar[C] (float2)
    int wide;                               // 1: the grid leaves at most one CTA per SM: launch the instance without the register cap
    int ring_off, ring_slot_bytes, n_ring, n_ring_deep;   // n_ring_deep: depth when one CTA owns the SM (chosen per plan)
    int stats_off, bar_off, smem_bytes, tmem_cols;
    int tab_off, tab_n;                     // per-K16-slice A operand start addresses (>>4), built at kernel start
    int wtab_off, n_chunks;                 // weight chunk list (byte offset into wblob, bytes)
    int tabs_off;                           // both tables, host-built, in fblob: int32 atab[tab_n], then uint2 wtab[nsplit][n_chunks]
    int nsplit;                             // output channels split over this many CTAs of a cluster (1 = none)
    int xpart_off;                          // [nsplit][nb] float2 partial PreNorm statistics exchanged through DSMEM
    int fmt;                                // 16-bit operand format: 1 = bf16, 0 = fp16
    int film_dim;
    int cin0, dim, channels;                // init conv / final conv shapes
    int init_w_off, init_b_off, final_w_off, final_b_off;
    const uint16_t* wblob;
    const float* fblob;
    void* gt[CH_MAX_GT];
    Ctrl* ctrl;
    long long* dbg;                         // optional clock64 timeline of CTA 0: [step][8] (null in production)
};

// linear-attention block  Residual(PreNorm(dim, LinearAttention(dim)))  (unet.py:33-39,125-161) and the
// mid-block full attention (unet.py:99-122), one kernel, `nb` samples per CTA
struct AttnFusedParams {
    int epi_warps;                          // 4 for mid attention; linear attention: 8 for one M tile, 16 for two (a sample spans two tiles)
    int B, H, W, C, nb, n, n_pad, n_mtiles; // n = H*W; n_pad = max(n,16) rows per sample in the P/V/Q slots;
                                            // n_mtiles = 128-row tiles of the dense rows (s*n + p)
    int full;                               // 1: softmax(QK^T)V mid attention (no GroupNorm after to_out)
    int ktrans;                             // 1: K and V are projected TRANSPOSED (weights as the A operand, the CTA's pixels as N): tensor-
                                            // memory lanes = channels, columns = pixels, so the softmax over pixels is a loop per thread
    int small;                              // 1: k_attn_small (n = 4 or 16 pixels: 128 / n samples per CTA, attention core on CUDA cores)
    int fmt;
    unsigned wq_off, wk_off, wv_off, wo_off; // 16-bit weight streams in wblob (N = 128,128,128,C)
    int qkv_chunks, qkv_S, o_chunks, o_S;   // ring chunking of those streams
    int bo_off, gamma_off, beta_off;        // to_out bias, to_out.1 GroupNorm affine (fblob)
    int xh_off, p_off, v_off, ct_off, kmax_off, stats_off;   // shared-memory regions
    int plane_bytes;                        // plane stride of the P/Q and V/O slots
    int ring_off, ring_slot_bytes, n_ring, bar_off, smem_bytes, tmem_cols;
    int zero_off, zero_bytes;
    int col_k, col_v, col_ctx, col_q, col_out, col_proj;     // TMEM column plan
    const uint16_t* wblob;
    const float* fblob;
    const void* x2;                         // residual input (16-bit blocked, global)
    void* out; void* out_un; void* out_up;  // outputs (16-bit blocked); un/up may be null
    long long* dbg;                         // optional clock64 timeline of CTA 0 (null in production)
};

// ---------------------------------------------------------------------------------------------
// adaptive Dormand-Prince 5(4) with scipy's step-size control (rk45.cu, flo_integrate_rk45)
// ---------------------------------------------------------------------------------------------
enum Rk45State : int { RK_RUNNING = 0, RK_DONE = 1, RK_TOO_SMALL = 2, RK_TOO_MANY = 3 };
enum Rk45EndMode : int { RK_END_NORM0 = 0, RK_END_NORM1 = 1, RK_END_STEP = 2 };

struct Rk45Status {           // what the host reads back after every attempt
    double t, h_abs;
    int accepted, rejected, nfev, state;
    int y_idx, pad;           // which half of Rk45Params::ybuf holds the current y
};

struct Rk45Ctl {              // device-resident controller state (scipy RungeKutta._step_impl, fp64)
    double t, t_new, t1, h, h_abs, min_step, max_step, rtol, atol, h0, d1, interval;
    float t_scale;
    int max_steps, attempts, step_rejected;
    int k0;                   // physical K slot holding K[0] (0 or 6); K[6] is in 6 - k0
    int two_pass;             // 1: conditional + combining pass per evaluation (12 stage entries per attempt)
    int flags;                // Stage::flags of the evaluation's (last) pass: 0, SF_CFG_2B or SF_CFG_COMBINE
    unsigned arrive;          // k_rk45_end arrival counter (zero between launches)
    Rk45Status status;
};

struct Rk45Params {
    Rk45Ctl* rc;
    Ctrl* ctrl;
    float* k;                 // [7][n] stage velocities (Ctrl::vtrace of the attempt)
    float* ybuf;              // [2][n] y | y_new, swapped by index on accept
    float* xs;                // forward input [n] ...
    float* xs2;               // ... and its unconditional half on the 2B route, or null
    double* part;             // [rk45_end_grid(n)][2] per-CTA partial sums
    int n;                    // B*C*H*W
};

int rk45_end_grid(int n);
cudaError_t launch_rk45_setup(Rk45Ctl* dst, const Rk45Ctl& value, Ctrl* ctrl, cudaStream_t s);   // + stage entry of f0
cudaError_t launch_rk45_stage(const Rk45Params& p, int stage, cudaStream_t s);   // 0: xs = y; -1: first-step trial; 1..6
cudaError_t launch_rk45_end(const Rk45Params& p, int mode, cudaStream_t s);

cudaError_t fused_configure();
int fused_max_active_clusters(int nsplit, int smem_bytes);
cudaError_t launch_chain(const ChainParams& p, const CUtensorMap* maps, int grid, cudaStream_t s);
cudaError_t launch_attn_fused(const AttnFusedParams& p, const CUtensorMap& xh_map, int grid, cudaStream_t s);


}  // namespace flo
