// CUDA-core kernels of the flocoder_b200 sampling path (sm_100a).
//
//   k_init_conv   init_conv 1x1 (unet.py:295) reading the NCHW fp32 integrator state
//   k_conv_simt   fp32 direct convolution on blocked tensors (the FLO_F32 path, <=1e-5 parity)
//   k_gn_tma /    GroupNorm + timestep-FiLM + SiLU + residual in ONE pass (unet.py:64-73,96,133,157), HBM-bound:
//   k_gn_warp /   each value is read once and written once; k_gn_tma stages (sample, group) units through shared memory
//   k_gn          with 1-D bulk copies and warp teams, k_gn_warp holds small units in registers (shuffle-only
//                 reductions), k_gn is the one-CTA-per-unit fallback
//   k_linattn     LinearAttention core (unet.py:142-149), one CTA per (sample, head)
//   k_midattn     mid-block Attention core (unet.py:114-121), one CTA per (sample, head)
//   k_temb        sinusoidal embedding + time/class MLPs + all ResnetBlock FiLM projections
//                 (unet.py:23-30,199-212,79-82,90-92) -> one FiLM row per distinct time / sample
//   k_final       final_conv 1x1 (unet.py:372) with the RK4 / Euler / CFG stage update fused as its
//                 epilogue (sampling.py:43-48,69-74)
//
// All tensors other than the NCHW latents use the blocked layout of flo_internal.h.
#include <type_traits>

#include <algorithm>

#include "umma_common.cuh"

namespace flo {

// ------------------------------------------------------------------------------------------------
// small helpers
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void load8(const float* src, float v[8]) {
    float4 a = *reinterpret_cast<const float4*>(src);
    float4 b = *reinterpret_cast<const float4*>(src + 4);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ void load8(const __nv_bfloat16* src, float v[8]) {
    uint4 u = *reinterpret_cast<const uint4*>(src);
    const __nv_bfloat162* h = reinterpret_cast<const __nv_bfloat162*>(&u);
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        float2 f = __bfloat1622float2(h[i]);
        v[2 * i] = f.x; v[2 * i + 1] = f.y;
    }
}
__device__ __forceinline__ void store8(float* dst, const float v[8]) {
    *reinterpret_cast<float4*>(dst) = make_float4(v[0], v[1], v[2], v[3]);
    *reinterpret_cast<float4*>(dst + 4) = make_float4(v[4], v[5], v[6], v[7]);
}
__device__ __forceinline__ void store8(__nv_bfloat16* dst, const float v[8]) {
    uint4 u;
    __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&u);
#pragma unroll
    for (int i = 0; i < 4; ++i) h[i] = __floats2bfloat162_rn(v[2 * i], v[2 * i + 1]);
    *reinterpret_cast<uint4*>(dst) = u;
}
__device__ __forceinline__ void store4(float* dst, float4 v) { *reinterpret_cast<float4*>(dst) = v; }
__device__ __forceinline__ void store4(__nv_bfloat16* dst, float4 v) {
    uint2 u;
    __nv_bfloat162* h = reinterpret_cast<__nv_bfloat162*>(&u);
    h[0] = __floats2bfloat162_rn(v.x, v.y);
    h[1] = __floats2bfloat162_rn(v.z, v.w);
    *reinterpret_cast<uint2*>(dst) = u;
}

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float warp_max(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
// block-wide sum; `red` is >= 32 floats of shared memory; every thread gets the result
__device__ __forceinline__ float block_sum(float v, float* red) {
    v = warp_sum(v);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    if (nw == 1) return v;
    __syncthreads();                 // protect `red` from the previous use
    if (lane == 0) red[warp] = v;
    __syncthreads();
    float t = (lane < nw) ? red[lane] : 0.f;
    return warp_sum(t);
}

// ------------------------------------------------------------------------------------------------
// control block setup (by-value launch arguments -> device memory; fully stream-ordered)
// ------------------------------------------------------------------------------------------------
__global__ void k_setup_ctrl(Ctrl* dst, Ctrl value, Stage* stage0_dst, Stage stage0, int write_stage) {
    if (threadIdx.x == 0 && blockIdx.x == 0) {
        *dst = value;
        if (write_stage) *stage0_dst = stage0;
    }
}
cudaError_t launch_setup_ctrl(Ctrl* ctrl_dev, const Ctrl& value, Stage* stage0_dev, const Stage* stage0_value,
                              cudaStream_t s) {
    Stage st = {};
    if (stage0_value) st = *stage0_value;
    k_setup_ctrl<<<1, 32, 0, s>>>(ctrl_dev, value, stage0_dev, st, stage0_value != nullptr);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// init_conv: NCHW fp32 latents -> blocked activations (fp32 master and/or operand copy)
// ------------------------------------------------------------------------------------------------
template <typename TO>
__global__ void __launch_bounds__(128) k_init_conv(InitConvParams p) {
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= p.B * p.HW) return;
    const int b = idx / p.HW, px = idx % p.HW;
    const float* x = p.ctrl->xs;
    float xin[16];
#pragma unroll 4
    for (int ci = 0; ci < p.cin; ++ci) xin[ci] = x[((size_t)b * p.cin + ci) * p.HW + px];
    const int ncb = p.dim >> 3;
    const bool bias = !p.n_bias_rows || b < p.n_bias_rows;
    for (int cb = 0; cb < ncb; ++cb) {
        float o[8];
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            const int co = cb * 8 + j;
            float a = 0.f;
            for (int ci = 0; ci < p.cin; ++ci) a = fmaf(xin[ci], p.w[co * p.cin + ci], a);
            o[j] = bias ? a + p.bias[co] : a;
        }
        const size_t off = ((size_t)(cb * p.B + b) * p.HW + px) * 8;
        if (p.out_m) store8(p.out_m + off, o);
        if (p.out_o) store8(reinterpret_cast<TO*>(p.out_o) + off, o);
    }
}
cudaError_t launch_init_conv(const InitConvParams& p, cudaStream_t s) {
    const int n = p.B * p.HW;
    if (p.o_is_bf16) k_init_conv<__nv_bfloat16><<<(n + 127) / 128, 128, 0, s>>>(p);
    else k_init_conv<float><<<(n + 127) / 128, 128, 0, s>>>(p);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// fp32 direct convolution (1x1 or 3x3 pad 1, stride 1) over up to two concatenated sources
// ------------------------------------------------------------------------------------------------
template <typename TI, typename TO>
__global__ void __launch_bounds__(128) k_conv_simt(ConvSimtParams p) {
    const int HW = p.H * p.W;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= p.B * HW) return;
    const int b = idx / HW, px = idx % HW, h = px / p.W, w = px % p.W;
    const int co0 = blockIdx.y * 8;
    const int cin = (p.ncb0 + p.ncb1) * 8;
    const size_t off = ((size_t)(blockIdx.y * p.B + b) * HW + px) * 8;
    float acc[8];
    // mask branches that are switched off at run time (no mask / all-ones mask): pass the bypass tensor through
    const bool live = !p.mask_mode || *p.mask_mode >= p.need_mode;
    if (!live && !p.bypass) return;
    if (live) {
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[j] = 0.f;
        const int taps = p.ksize * p.ksize, r = p.ksize >> 1;
        for (int t = 0; t < taps; ++t) {
            const int hh = h + t / p.ksize - r, ww = w + t % p.ksize - r;
            if (hh < 0 || hh >= p.H || ww < 0 || ww >= p.W) continue;
            const int q = hh * p.W + ww;
            const float* wt = p.w + (size_t)t * cin * p.cout + co0;
            for (int src = 0; src < 2; ++src) {
                const TI* in = reinterpret_cast<const TI*>(src ? p.in1 : p.in0);
                const int ncb = src ? p.ncb1 : p.ncb0;
                const int cbase = src ? p.ncb0 * 8 : 0;
                for (int cb = 0; cb < ncb; ++cb) {
                    float xv[8];
                    load8(in + ((size_t)(cb * p.B + b) * HW + q) * 8, xv);
#pragma unroll
                    for (int c8 = 0; c8 < 8; ++c8) {
                        float wv[8];
                        load8(wt + (size_t)(cbase + cb * 8 + c8) * p.cout, wv);
#pragma unroll
                        for (int j = 0; j < 8; ++j) acc[j] = fmaf(xv[c8], wv[j], acc[j]);
                    }
                }
            }
        }
        if (p.bias && (!p.n_bias_rows || b < p.n_bias_rows)) {
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[j] += p.bias[co0 + j];
        }
        if (p.act_silu) {                                  // nn.SiLU of the mask-fusion convs (unet.py:217-235)
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[j] = acc[j] / (1.0f + expf(-acc[j]));
        }
        if (p.res) {
            float rv[8];
            load8(p.res + off, rv);
#pragma unroll
            for (int j = 0; j < 8; ++j) acc[j] += rv[j];
        }
    } else {
        load8(p.bypass + off, acc);
    }
    if (p.out_m) store8(p.out_m + off, acc);
    if (p.out_o) store8(reinterpret_cast<TO*>(p.out_o) + off, acc);
    if (p.out_unshuf) {      // 'b c (h p1) (w p2) -> b (c p1 p2) h w' in our (p1 p2 c) channel order, as k_gn writes it
        const int ncb = p.cout >> 3;
        const int plane = ((h & 1) * 2 + (w & 1)) * ncb + (int)blockIdx.y;
        const int q = (h >> 1) * (p.W >> 1) + (w >> 1);
        store8(reinterpret_cast<TO*>(p.out_unshuf) + ((size_t)(plane * p.B + b) * (HW >> 2) + q) * 8, acc);
    }
    if (p.out_up) {          // nearest x2
        const int W2 = p.W * 2;
#pragma unroll
        for (int d = 0; d < 4; ++d) {
            const int q = (2 * h + (d >> 1)) * W2 + 2 * w + (d & 1);
            store8(reinterpret_cast<TO*>(p.out_up) + ((size_t)(blockIdx.y * p.B + b) * (HW * 4) + q) * 8, acc);
        }
    }
}
cudaError_t launch_conv_simt(const ConvSimtParams& p, cudaStream_t s) {
    dim3 grid((p.B * p.H * p.W + 127) / 128, p.cout / 8);
    if (p.in_is_bf16) {
        if (p.o_is_bf16) k_conv_simt<__nv_bfloat16, __nv_bfloat16><<<grid, 128, 0, s>>>(p);
        else k_conv_simt<__nv_bfloat16, float><<<grid, 128, 0, s>>>(p);
    } else {
        if (p.o_is_bf16) k_conv_simt<float, __nv_bfloat16><<<grid, 128, 0, s>>>(p);
        else k_conv_simt<float, float><<<grid, 128, 0, s>>>(p);
    }
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// GroupNorm + FiLM + SiLU + residual, one pass.  One CTA per (sample, group).
// ------------------------------------------------------------------------------------------------
constexpr int GN_VPT = 8;   // float4 vectors held per thread

template <typename TO>
__global__ void __launch_bounds__(256) k_gn(GnParams p) {
    __shared__ float red[32];
    const int G = p.groups, cpg = p.C / G, HW = p.H * p.W;
    // shifts, not integer divisions: gn_variant picks this kernel only when W, H*W and groups are powers of two
    const int lgG = 31 - __clz(G), lgW = 31 - __clz(p.W), lgPC = 31 - __clz(HW * 2);
    const int b = blockIdx.x >> lgG, g = blockIdx.x & (G - 1);
    const int nvec = cpg * HW / 4;
    const int NT = blockDim.x, tid = threadIdx.x;
    const int ncb = p.C >> 3;

    float4 v[GN_VPT];
    size_t offs[GN_VPT];
    int chan[GN_VPT], pix[GN_VPT];
    float sum = 0.f;
#pragma unroll
    for (int k = 0; k < GN_VPT; ++k) {
        const int i = tid + k * NT;
        v[k] = make_float4(0.f, 0.f, 0.f, 0.f);
        offs[k] = 0; chan[k] = 0; pix[k] = 0;
        if (i < nvec) {
            int cb, sub, px;
            if (cpg >= 8) {                 // the group spans whole channel blocks
                cb = g * (cpg >> 3) + (i >> lgPC);
                const int r = i & (HW * 2 - 1);
                px = r >> 1; sub = (r & 1) * 4;
            } else {                        // cpg == 4: half a channel block
                cb = (g * 4) >> 3; sub = (g & 1) * 4; px = i;
            }
            offs[k] = ((size_t)(cb * p.B + b) * HW + px) * 8 + sub;
            chan[k] = cb * 8 + sub; pix[k] = px;
            v[k] = *reinterpret_cast<const float4*>(p.in + offs[k]);
            sum += (v[k].x + v[k].y) + (v[k].z + v[k].w);
        }
    }
    const float inv_n = 1.f / (float)(cpg * HW);
    const float mean = block_sum(sum, red) * inv_n;
    float sq = 0.f;
#pragma unroll
    for (int k = 0; k < GN_VPT; ++k) {
        if (tid + k * NT < nvec) {
            const float a = v[k].x - mean, b2 = v[k].y - mean, c = v[k].z - mean, d = v[k].w - mean;
            sq += (a * a + b2 * b2) + (c * c + d * d);
        }
    }
    const float var = block_sum(sq, red) * inv_n;          // biased variance (nn.GroupNorm)
    const float rstd = 1.0f / sqrtf(var + 1e-5f);

    const float* film = nullptr;
    if (p.film_off >= 0) {
        const Ctrl* c = p.ctrl;
        const int row = c->film_per_sample ? b : c->stages[c->step].film_row;
        film = c->film + (size_t)row * p.film_dim + p.film_off;
    }
    TO* out_o = reinterpret_cast<TO*>(p.out_o);
    TO* out_un = reinterpret_cast<TO*>(p.out_unshuf);
    TO* out_up = reinterpret_cast<TO*>(p.out_up);
#pragma unroll
    for (int k = 0; k < GN_VPT; ++k) {
        if (tid + k * NT >= nvec) continue;
        const int c0 = chan[k];
        float x[4] = {v[k].x, v[k].y, v[k].z, v[k].w};
        const float4 ga = *reinterpret_cast<const float4*>(p.gamma + c0);
        const float4 be = *reinterpret_cast<const float4*>(p.beta + c0);
        const float gam[4] = {ga.x, ga.y, ga.z, ga.w}, bet[4] = {be.x, be.y, be.z, be.w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float y = (x[j] - mean) * rstd * gam[j] + bet[j];
            if (film) y = y * (film[c0 + j] + 1.0f) + film[p.C + c0 + j];     // unet.py:70
            if (p.silu) y = y / (1.0f + expf(-y));                            // x*sigmoid(x)
            x[j] = y;
        }
        if (p.res) {
            const float4 r = *reinterpret_cast<const float4*>(p.res + offs[k]);
            x[0] += r.x; x[1] += r.y; x[2] += r.z; x[3] += r.w;
        }
        const float4 o = make_float4(x[0], x[1], x[2], x[3]);
        if (p.out_m) store4(p.out_m + offs[k], o);
        if (out_o) store4(out_o + offs[k], o);
        if (out_un || out_up) {
            const int h = pix[k] >> lgW, w = pix[k] & (p.W - 1), cb = c0 >> 3, sub = c0 & 7;
            if (out_un) {   // 'b c (h p1) (w p2) -> b (c p1 p2) h w' with our channel order (p1 p2 c)
                const int plane = ((h & 1) * 2 + (w & 1)) * ncb + cb;
                const int q = (h >> 1) * (p.W >> 1) + (w >> 1);
                store4(out_un + ((size_t)(plane * p.B + b) * (HW >> 2) + q) * 8 + sub, o);
            }
            if (out_up) {   // nearest x2: dst(2h+dy, 2w+dx) = src(h, w)
                const int W2 = p.W * 2;
#pragma unroll
                for (int d = 0; d < 4; ++d) {
                    const int q = (2 * h + (d >> 1)) * W2 + 2 * w + (d & 1);
                    store4(out_up + ((size_t)(cb * p.B + b) * (HW * 4) + q) * 8 + sub, o);
                }
            }
        }
    }
}
// Warp-team variant for units of <= 1024 float4 (every GroupNorm of the BASELINE U-Nets):
// a team of T <= 32 lanes owns one unit, holds it in registers (V float4 per lane), reduces with xor-shuffles only
// (no shared memory, no __syncthreads) and reads / writes whole 32-byte pixel rows.  When a group is half a channel
// block (cpg == 4) the team takes the PAIR of groups sharing that block, so that consecutive lanes touch consecutive
// 16 bytes (full sectors both ways); lane parity = group, and the reduction skips the xor-1 step.
// MUFU forms for the 16-bit variant (the fp32 variant keeps expf / IEEE division).  With h = y/2,
// SiLU(y) = y * sigmoid(y) = h + h * tanh(h): one MUFU and one FMA per element once the affine is folded to produce h
// directly.  tanh.approx.f32 is accurate to ~2^-11, a quarter of the bf16 output rounding that follows.
__device__ __forceinline__ float gn_fast_silu(float y) {
    float e, r;
    asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(-1.4426950408889634f * y));
    asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(r) : "f"(1.0f + e));
    return y * r;
}
__device__ __forceinline__ float gn_silu_from_half(float h) {
    float t;
    asm("tanh.approx.f32 %0, %1;" : "=f"(t) : "f"(h));
    return fmaf(h, t, h);
}
constexpr int GNW_THREADS = 64;
template <typename TO, int V>
__global__ void __launch_bounds__(GNW_THREADS) k_gn_warp(GnParams p, int T, int pair, int n_units) {
    constexpr bool kFast = !std::is_same<TO, float>::value;              // 16-bit outputs: folded affine + MUFU SiLU
    const int G = p.groups, cpg = p.C / G, HW = p.H * p.W;
    const int lgW = 31 - __clz(p.W), lgPC = 31 - __clz(HW * 2), lgT = 31 - __clz(T);
    const int lane = threadIdx.x & 31, lt = lane & (T - 1);
    const int unit = ((blockIdx.x * (GNW_THREADS / 32) + (threadIdx.x >> 5)) << (5 - lgT)) + (lane >> lgT);
    const bool live = unit < n_units;
    const int upb = pair ? (p.C >> 3) : G, lgU = 31 - __clz(upb);       // units per sample (power of two)
    const int b = unit >> lgU, j = unit & (upb - 1);
    const int cb0 = pair ? j : j * (cpg >> 3);
    const int ncb = p.C >> 3;

    float4 v[V];
    float sum = 0.f;
#pragma unroll
    for (int k = 0; k < V; ++k) {
        const int i = lt + k * T;
        v[k] = make_float4(0.f, 0.f, 0.f, 0.f);
        if (live) {
            const size_t off = ((size_t)((cb0 + (i >> lgPC)) * p.B + b) * HW) * 8 + (size_t)(i & (HW * 2 - 1)) * 4;
            v[k] = __ldcs(reinterpret_cast<const float4*>(p.in + off));
        }
        sum += (v[k].x + v[k].y) + (v[k].z + v[k].w);
    }
    const int o_min = pair ? 2 : 1;
    for (int o = T >> 1; o >= o_min; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    const float inv_n = 1.f / (float)(cpg * HW);
    const float mean = sum * inv_n;
    float sq = 0.f;
#pragma unroll
    for (int k = 0; k < V; ++k) {
        const float a = v[k].x - mean, b2 = v[k].y - mean, c = v[k].z - mean, d = v[k].w - mean;
        sq += (a * a + b2 * b2) + (c * c + d * d);
    }
    for (int o = T >> 1; o >= o_min; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
    if (!live) return;
    const float rstd = 1.0f / sqrtf(sq * inv_n + 1e-5f);                // biased variance (nn.GroupNorm)

    const float* film = nullptr;
    if (p.film_off >= 0) {
        const Ctrl* c = p.ctrl;
        const int row = c->film_per_sample ? b : c->stages[c->step].film_row;
        film = c->film + (size_t)row * p.film_dim + p.film_off;
    }
    TO* out_o = reinterpret_cast<TO*>(p.out_o);
    TO* out_un = reinterpret_cast<TO*>(p.out_unshuf);
    TO* out_up = reinterpret_cast<TO*>(p.out_up);
    // per-channel coefficients, reloaded only when the lane moves to another channel quad (never, when the unit is one
    // channel block): exact variant keeps (gamma, beta, scale+1, shift) and the reference's operation order
    // (unet.py:64-70); fast variant folds them into y = x * ca + cb.
    int c_prev = -1;
    float ca[4] = {0.f, 0.f, 0.f, 0.f}, cb_[4] = {0.f, 0.f, 0.f, 0.f}, cs[4] = {1.f, 1.f, 1.f, 1.f}, ch[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
    for (int k = 0; k < V; ++k) {
        const int i = lt + k * T, r = i & (HW * 2 - 1);
        const int cb = cb0 + (i >> lgPC), sub = (r & 1) * 4, c0 = cb * 8 + sub, px = r >> 1;
        const size_t off = ((size_t)(cb * p.B + b) * HW) * 8 + (size_t)r * 4;
        if (c0 != c_prev) {
            c_prev = c0;
            const float4 ga = *reinterpret_cast<const float4*>(p.gamma + c0);
            const float4 be = *reinterpret_cast<const float4*>(p.beta + c0);
            ca[0] = ga.x; ca[1] = ga.y; ca[2] = ga.z; ca[3] = ga.w;
            cb_[0] = be.x; cb_[1] = be.y; cb_[2] = be.z; cb_[3] = be.w;
            if (film) {
#pragma unroll
                for (int q = 0; q < 4; ++q) { cs[q] = film[c0 + q] + 1.0f; ch[q] = film[p.C + c0 + q]; }
            }
            if (kFast) {
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    const float g2 = rstd * ca[q];
                    ca[q] = g2 * cs[q];
                    cb_[q] = fmaf(fmaf(-mean, g2, cb_[q]), cs[q], ch[q]);
                }
            }
        }
        float x[4] = {v[k].x, v[k].y, v[k].z, v[k].w};
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            float y;
            if (kFast) {
                y = fmaf(x[q], ca[q], cb_[q]);
                if (p.silu) y = gn_fast_silu(y);
            } else {
                y = (x[q] - mean) * rstd * ca[q] + cb_[q];
                if (film) y = y * cs[q] + ch[q];                              // unet.py:70
                if (p.silu) y = y / (1.0f + expf(-y));                        // x*sigmoid(x)
            }
            x[q] = y;
        }
        if (p.res) {
            const float4 rr = __ldcs(reinterpret_cast<const float4*>(p.res + off));
            x[0] += rr.x; x[1] += rr.y; x[2] += rr.z; x[3] += rr.w;
        }
        const float4 o = make_float4(x[0], x[1], x[2], x[3]);
        if (p.out_m) store4(p.out_m + off, o);
        if (out_o) store4(out_o + off, o);
        if (out_un || out_up) {
            const int h = px >> lgW, w = px & (p.W - 1);
            if (out_un) {   // 'b c (h p1) (w p2) -> b (c p1 p2) h w' with our channel order (p1 p2 c)
                const int plane = ((h & 1) * 2 + (w & 1)) * ncb + cb;
                const int q2 = (h >> 1) * (p.W >> 1) + (w >> 1);
                store4(out_un + ((size_t)(plane * p.B + b) * (HW >> 2) + q2) * 8 + sub, o);
            }
            if (out_up) {   // nearest x2: dst(2h+dy, 2w+dx) = src(h, w)
                const int W2 = p.W * 2;
#pragma unroll
                for (int d = 0; d < 4; ++d) {
                    const int q2 = (2 * h + (d >> 1)) * W2 + 2 * w + (d & 1);
                    store4(out_up + ((size_t)(cb * p.B + b) * (HW * 4) + q2) * 8 + sub, o);
                }
            }
        }
    }
}
// Staged variant for units of >= 2 KB: the pass is HBM-bound, so what matters is bytes in flight.  A TEAM of TW warps
// (1, 2 or 4) owns a two-deep ring of unit-sized shared-memory stages filled by 1-D bulk copies (cp.async.bulk + mbarrier
// complete_tx; a unit is cpg/8 contiguous runs of HW*32 bytes in the blocked layout, plus the same runs of the residual)
// and strides over the units persistently: while it normalises unit k out of one stage, unit k+1 is landing in the
// other, and the refill for k+2 is issued as soon as the team has finished reading.  The three passes (sum, centred
// squares, normalise) re-read shared memory with conflict-free 16-byte accesses, so the register footprint is small;
// reductions are xor-shuffles inside a warp and a fixed-order sum of TW partials across the team (named barrier of
// TW*32 threads; nothing CTA-wide after the prologue).  Teams of more than one warp keep 24 warps per SM busy on the
// 8-32 KB stages that would otherwise leave 3-12.
constexpr int GNT_STAGES = 2;
constexpr int GNT_MAX_WARPS = 8;
template <typename TO>
__global__ void __launch_bounds__(GNT_MAX_WARPS * 32) k_gn_tma(GnParams p, int pair, int n_units, int n_chunks, int total_teams, int TW) {
    extern __shared__ __align__(128) uint8_t gn_smem[];
    constexpr bool kFast = !std::is_same<TO, float>::value;
    const int G = p.groups, cpg = p.C / G, HW = p.H * p.W;
    const int lgW = 31 - __clz(p.W), lgTW = 31 - __clz(TW);
    const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, tpb = (blockDim.x >> 5) >> lgTW;
    const int team = w >> lgTW, wt = w & (TW - 1);
    const int VCw = (HW >> 4) >> lgTW;                                   // float4 per lane per chunk (HW * 2 / 32 / TW)
    const int chunk_bytes = HW * 32, unit_bytes = n_chunks * chunk_bytes;
    const int stage_bytes = unit_bytes * (p.res ? 2 : 1);
    const int Vw = (unit_bytes >> 9) >> lgTW;                            // float4 per lane per unit
    const int upb = pair ? (p.C >> 3) : G, lgU = 31 - __clz(upb);
    const int ncb = p.C >> 3, sub = (lane & 1) * 4;
    const int step = TW * 32;                                            // float4 between a lane's consecutive vectors
    uint8_t* my = gn_smem + (size_t)team * GNT_STAGES * stage_bytes;
    uint8_t* tail = gn_smem + (size_t)tpb * GNT_STAGES * stage_bytes;
    const uint32_t bar0 = smem_u32(tail) + team * GNT_STAGES * 8;
    float* red = reinterpret_cast<float*>(tail + GNT_MAX_WARPS * GNT_STAGES * 8) + team * 16;     // [2 (sum|sq)][TW <= 4][2 groups]
    const int gteam = blockIdx.x * tpb + team;

    auto issue = [&](int k) {          // one lane of the team
        const int unit = gteam + k * total_teams;
        if (unit >= n_units) return;
        const int s = k & 1, b = unit >> lgU, j = unit & (upb - 1);
        const int cb0 = pair ? j : j * (cpg >> 3);
        const uint32_t bar = bar0 + s * 8, dst = smem_u32(my + (size_t)s * stage_bytes);
        mbar_expect_tx(bar, (uint32_t)stage_bytes);
        for (int c = 0; c < n_chunks; ++c) {
            const size_t off = ((size_t)((cb0 + c) * p.B + b) * HW) * 8;
            bulk_load_1d(dst + c * chunk_bytes, p.in + off, (uint32_t)chunk_bytes, bar);
            if (p.res) bulk_load_1d(dst + unit_bytes + c * chunk_bytes, p.res + off, (uint32_t)chunk_bytes, bar);
        }
    };
    auto team_sync = [&]() {
        if (TW == 1) __syncwarp();
        else named_bar_sync(1 + team, TW * 32);
    };
    // warp partial -> team total, per group (lane parity = group when two groups share the channel block)
    auto team_sum = [&](float v, int which, int o_min) -> float {
        for (int o = 16; o >= o_min; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
        if (TW == 1) return v;
        if (lane < 2) red[which * 8 + wt * 2 + lane] = v;
        named_bar_sync(1 + team, TW * 32);
        float t = 0.f;
        for (int q = 0; q < TW; ++q) t += red[which * 8 + q * 2 + (lane & 1)];
        return t;
    };
    if (wt == 0 && lane == 0) {
        mbar_init(bar0, 1); mbar_init(bar0 + 8, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        fence_proxy_async();
        issue(0); issue(1);
    }
    __syncthreads();

    const float inv_n = 1.f / (float)(cpg * HW);
    const int o_min = pair ? 2 : 1;
    TO* out_o = reinterpret_cast<TO*>(p.out_o);
    TO* out_un = reinterpret_cast<TO*>(p.out_unshuf);
    TO* out_up = reinterpret_cast<TO*>(p.out_up);
    for (int k = 0;; ++k) {
        const int unit = gteam + k * total_teams;
        if (unit >= n_units) break;
        const int s = k & 1, b = unit >> lgU, j = unit & (upb - 1);
        const int cb0 = pair ? j : j * (cpg >> 3);
        mbar_wait(bar0 + s * 8, (uint32_t)((k >> 1) & 1));
        const float4* xs = reinterpret_cast<const float4*>(my + (size_t)s * stage_bytes) + wt * 32 + lane;
        const float4* rs = reinterpret_cast<const float4*>(my + (size_t)s * stage_bytes + unit_bytes) + wt * 32 + lane;
        float mean, rstd;
        if (kFast) {                       // one pass: sum and sum of squares (fp32, <= 4096 values of O(1) magnitude)
            float sum = 0.f, sq = 0.f;
#pragma unroll 4
            for (int i = 0; i < Vw; ++i) {
                const float4 v = xs[i * step];
                sum += (v.x + v.y) + (v.z + v.w);
                sq = fmaf(v.x, v.x, fmaf(v.y, v.y, fmaf(v.z, v.z, fmaf(v.w, v.w, sq))));
            }
            mean = team_sum(sum, 0, o_min) * inv_n;
            const float var = fmaxf(team_sum(sq, 1, o_min) * inv_n - mean * mean, 0.f);
            rstd = rsqrtf(var + 1e-5f);
        } else {                           // two passes, the reference's formula (biased variance of nn.GroupNorm)
            float sum = 0.f;
#pragma unroll 4
            for (int i = 0; i < Vw; ++i) { const float4 v = xs[i * step]; sum += (v.x + v.y) + (v.z + v.w); }
            mean = team_sum(sum, 0, o_min) * inv_n;
            float sq = 0.f;
#pragma unroll 4
            for (int i = 0; i < Vw; ++i) {
                const float4 v = xs[i * step];
                const float a = v.x - mean, b2 = v.y - mean, c = v.z - mean, d = v.w - mean;
                sq += (a * a + b2 * b2) + (c * c + d * d);
            }
            rstd = 1.0f / sqrtf(team_sum(sq, 1, o_min) * inv_n + 1e-5f);
        }
        const float* film = nullptr;
        if (p.film_off >= 0) {
            const Ctrl* c = p.ctrl;
            const int row = c->film_per_sample ? b : c->stages[c->step].film_row;
            film = c->film + (size_t)row * p.film_dim + p.film_off;
        }
        for (int c = 0; c < n_chunks; ++c) {
            // per-channel coefficients of this channel block (lane parity = channel quad): the exact variant keeps
            // (gamma, beta, scale+1, shift) and the reference's operation order (unet.py:64-70); the 16-bit variant
            // folds them into y = x * ca + cb.
            const int cb = cb0 + c, c0 = cb * 8 + sub;
            float ca[4], cb_[4], cs[4] = {1.f, 1.f, 1.f, 1.f}, ch[4] = {0.f, 0.f, 0.f, 0.f};
            {
                const float4 ga = *reinterpret_cast<const float4*>(p.gamma + c0);
                const float4 be = *reinterpret_cast<const float4*>(p.beta + c0);
                ca[0] = ga.x; ca[1] = ga.y; ca[2] = ga.z; ca[3] = ga.w;
                cb_[0] = be.x; cb_[1] = be.y; cb_[2] = be.z; cb_[3] = be.w;
                if (film) {
#pragma unroll
                    for (int q = 0; q < 4; ++q) { cs[q] = film[c0 + q] + 1.0f; ch[q] = film[p.C + c0 + q]; }
                }
                if (kFast) {
#pragma unroll
                    for (int q = 0; q < 4; ++q) {
                        const float g2 = rstd * ca[q];
                        ca[q] = g2 * cs[q];
                        cb_[q] = fmaf(fmaf(-mean, g2, cb_[q]), cs[q], ch[q]);
                        if (p.silu) { ca[q] *= 0.5f; cb_[q] *= 0.5f; }       // the loop below then yields h = y / 2
                    }
                }
            }
            const size_t base = ((size_t)(cb * p.B + b) * HW) * 8 + (size_t)(wt * 32 + lane) * 4;
            float* om = p.out_m ? p.out_m + base : nullptr;
            TO* oo = out_o ? out_o + base : nullptr;
            const float4* xc = xs + c * (HW * 2);
            const float4* rc = rs + c * (HW * 2);
#pragma unroll 4
            for (int it = 0; it < VCw; ++it) {
                const float4 v = xc[it * step];
                float x[4] = {v.x, v.y, v.z, v.w};
#pragma unroll
                for (int q = 0; q < 4; ++q) {
                    float y;
                    if (kFast) {
                        y = fmaf(x[q], ca[q], cb_[q]);
                        if (p.silu) y = gn_silu_from_half(y);
                    } else {
                        y = (x[q] - mean) * rstd * ca[q] + cb_[q];
                        if (film) y = y * cs[q] + ch[q];                      // unet.py:70
                        if (p.silu) y = y / (1.0f + expf(-y));                // x*sigmoid(x)
                    }
                    x[q] = y;
                }
                if (p.res) {
                    const float4 rr = rc[it * step];
                    x[0] += rr.x; x[1] += rr.y; x[2] += rr.z; x[3] += rr.w;
                }
                const float4 o = make_float4(x[0], x[1], x[2], x[3]);
                if (om) store4(om + it * step * 4, o);
                if (oo) store4(oo + it * step * 4, o);
                if (out_un || out_up) {
                    const int px = (it * step + wt * 32 + lane) >> 1;
                    const int h = px >> lgW, ww = px & (p.W - 1);
                    if (out_un) {   // 'b c (h p1) (w p2) -> b (c p1 p2) h w' with our channel order (p1 p2 c)
                        const int plane = ((h & 1) * 2 + (ww & 1)) * ncb + cb;
                        const int q2 = (h >> 1) * (p.W >> 1) + (ww >> 1);
                        store4(out_un + ((size_t)(plane * p.B + b) * (HW >> 2) + q2) * 8 + sub, o);
                    }
                    if (out_up) {   // nearest x2: dst(2h+dy, 2w+dx) = src(h, w)
                        const int W2 = p.W * 2;
#pragma unroll
                        for (int d = 0; d < 4; ++d) {
                            const int q2 = (2 * h + (d >> 1)) * W2 + 2 * ww + (d & 1);
                            store4(out_up + ((size_t)(cb * p.B + b) * (HW * 4) + q2) * 8 + sub, o);
                        }
                    }
                }
            }
        }
        team_sync();                       // every lane of the team has finished reading this stage
        if (wt == 0 && lane == 0) issue(k + 2);
    }
}
static int gn_num_sms() {
    static int n = 0;
    if (!n) {
        int dev = 0;
        if (cudaGetDevice(&dev) != cudaSuccess || cudaDeviceGetAttribute(&n, cudaDevAttrMultiProcessorCount, dev) != cudaSuccess || n <= 0) n = 148;
    }
    return n;
}
constexpr int GNT_MAX_SMEM = 72 * 1024;
template <typename TO>
static void launch_gn_tma(const GnParams& p, int pair, int n_chunks, cudaStream_t s) {
    const int HW = p.H * p.W, unit_bytes = n_chunks * HW * 32, stage_bytes = unit_bytes * (p.res ? 2 : 1);
    const int n_units = p.B * (pair ? p.C / 8 : p.groups);
    int TW = 1;                                                          // warps per unit: ~4 KB of stage per warp
    while (TW < 4 && TW * 2 <= HW / 16 && stage_bytes / (TW * 2) >= 4096) TW *= 2;
    int tpb = GNT_MAX_SMEM / (GNT_STAGES * stage_bytes);
    tpb = std::max(1, std::min(tpb, GNT_MAX_WARPS / TW));
    const int smem = tpb * GNT_STAGES * stage_bytes + GNT_MAX_WARPS * GNT_STAGES * 8 + GNT_MAX_WARPS * 16 * 4;
    const int per_sm = std::max(1, std::min(16, (220 * 1024) / (smem + 1024)));
    const int grid = std::min((n_units + tpb - 1) / tpb, gn_num_sms() * per_sm);
    k_gn_tma<TO><<<grid, tpb * TW * 32, smem, s>>>(p, pair, n_units, n_chunks, grid * tpb, TW);
}
template <typename TO>
static void launch_gn_warp(const GnParams& p, int nvec, int pair, cudaStream_t s) {
    const int T = nvec < 32 ? nvec : 32, V = nvec / T;
    const int n_units = p.B * (pair ? p.C / 8 : p.groups);
    const int warps = (n_units + 32 / T - 1) / (32 / T), wpb = GNW_THREADS / 32, grid = (warps + wpb - 1) / wpb;
    switch (V) {
        case 1:  k_gn_warp<TO, 1><<<grid, GNW_THREADS, 0, s>>>(p, T, pair, n_units); break;
        case 2:  k_gn_warp<TO, 2><<<grid, GNW_THREADS, 0, s>>>(p, T, pair, n_units); break;
        case 4:  k_gn_warp<TO, 4><<<grid, GNW_THREADS, 0, s>>>(p, T, pair, n_units); break;
        case 8:  k_gn_warp<TO, 8><<<grid, GNW_THREADS, 0, s>>>(p, T, pair, n_units); break;
        case 16: k_gn_warp<TO, 16><<<grid, GNW_THREADS, 0, s>>>(p, T, pair, n_units); break;
        default: k_gn_warp<TO, 32><<<grid, GNW_THREADS, 0, s>>>(p, T, pair, n_units); break;
    }
}
static bool is_pow2(int x) { return x > 0 && (x & (x - 1)) == 0; }
constexpr int GN_CTA_THREADS = 256;
// k_gn_tma, k_gn_warp and k_gn locate pixels, channel blocks and samples with shifts and masks: each runs only where W, H*W
// and its units per sample are powers of two.  A unit is one (sample, group), or for 4-channel groups (pair) the two groups
// that share a channel block in k_gn_tma / k_gn_warp; k_gn always takes one group.  The order tma > warp > cta is the
// fastest first; FLO_GN_NO_TMA skips k_gn_tma and FLO_GN_CTA both, so that tests can compare the kernels on one input.
// Every other shape runs k_gn_any on the fp32 path and has no kernel on the 16-bit layer-wise path.
GnVariant gn_variant(int C, int H, int W, int groups, bool bf16) {
    const GnVariant generic = bf16 ? GN_NONE : GN_ANY;
    if (groups < 1 || C % groups) return GN_NONE;
    const int cpg = C / groups, HW = H * W;
    if (cpg != 4 && (cpg & 7)) return generic;                           // the three fast kernels read whole channel quads
    const bool pair = cpg == 4, shifts = is_pow2(W) && is_pow2(HW);
    const int upb = pair ? C / 8 : groups;                               // k_gn_tma / k_gn_warp units per sample
    const int nvec_w = pair ? HW * 2 : cpg * HW / 4;                     // float4 per warp-team unit
    const int unit_bytes = (pair ? 1 : cpg / 8) * HW * 32;
    const bool cta_only = getenv("FLO_GN_CTA") != nullptr;
    if (!cta_only && !getenv("FLO_GN_NO_TMA") && shifts && is_pow2(upb) && HW >= 16 && unit_bytes >= 2048 &&
        unit_bytes <= 16384 && is_pow2(unit_bytes))
        return GN_TMA;
    if (!cta_only && shifts && is_pow2(upb) && nvec_w >= 2 && nvec_w <= 1024 && is_pow2(nvec_w)) return GN_WARP;
    if (shifts && is_pow2(groups) && cpg * HW / 4 <= GN_CTA_THREADS * GN_VPT) return GN_CTA;   // the unit fits a CTA's registers
    return generic;
}
const char* gn_variant_name(GnVariant v) {
    switch (v) {
        case GN_TMA: return "tma";
        case GN_WARP: return "warp";
        case GN_CTA: return "cta";
        case GN_ANY: return "any";
        default: return "none";
    }
}
cudaError_t launch_gn(const GnParams& p, cudaStream_t s) {
    const int cpg = p.C / p.groups, HW = p.H * p.W, pair = cpg == 4 ? 1 : 0;
    switch (gn_variant(p.C, p.H, p.W, p.groups, p.o_is_bf16)) {
        case GN_TMA: {
            const int n_chunks = pair ? 1 : cpg / 8;
            if (p.o_is_bf16) launch_gn_tma<__nv_bfloat16>(p, pair, n_chunks, s);
            else launch_gn_tma<float>(p, pair, n_chunks, s);
        } break;
        case GN_WARP: {
            const int nvec_w = pair ? HW * 2 : cpg * HW / 4;
            if (p.o_is_bf16) launch_gn_warp<__nv_bfloat16>(p, nvec_w, pair, s);
            else launch_gn_warp<float>(p, nvec_w, pair, s);
        } break;
        case GN_CTA: {
            const int nvec = cpg * HW / 4;
            int nt = 32;
            while (nt < GN_CTA_THREADS && nt * GN_VPT < nvec) nt <<= 1;
            // prefer ~4 vectors per thread when the unit is big enough to fill more warps
            while (nt < GN_CTA_THREADS && nvec / nt > 4) nt <<= 1;
            const int grid = p.B * p.groups;
            if (p.o_is_bf16) k_gn<__nv_bfloat16><<<grid, nt, 0, s>>>(p);
            else k_gn<float><<<grid, nt, 0, s>>>(p);
        } break;
        case GN_ANY: return launch_gn_any(p, s);
        default: return cudaErrorInvalidValue;
    }
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// GroupNorm + FiLM + SiLU + residual for ANY channels-per-group (fp32 path; e.g. dim = 8 with 4 groups: 2 channels
// per group, the midi_inpainting U-Net).  One CTA per (sample, group), two-pass statistics, scalar accesses.
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_gn_any(GnParams p) {
    __shared__ float red[32];
    const int G = p.groups, cpg = p.C / G, HW = p.H * p.W, n = cpg * HW;
    const int b = blockIdx.x / G, g = blockIdx.x % G;
    auto addr = [&](int e) -> size_t {
        const int c = g * cpg + e / HW, px = e % HW;
        return ((size_t)((c >> 3) * p.B + b) * HW + px) * 8 + (c & 7);
    };
    float sum = 0.f;
    for (int e = threadIdx.x; e < n; e += blockDim.x) sum += p.in[addr(e)];
    const float mean = block_sum(sum, red) / (float)n;
    float sq = 0.f;
    for (int e = threadIdx.x; e < n; e += blockDim.x) { const float d = p.in[addr(e)] - mean; sq += d * d; }
    const float var = block_sum(sq, red) / (float)n;
    const float rstd = 1.0f / sqrtf(var + 1e-5f);
    const float* film = nullptr;
    if (p.film_off >= 0) {
        const Ctrl* c = p.ctrl;
        const int row = c->film_per_sample ? b : c->stages[c->step].film_row;
        film = c->film + (size_t)row * p.film_dim + p.film_off;
    }
    float* out_o = reinterpret_cast<float*>(p.out_o);
    float* out_un = reinterpret_cast<float*>(p.out_unshuf);
    float* out_up = reinterpret_cast<float*>(p.out_up);
    const int ncb = p.C >> 3;
    for (int e = threadIdx.x; e < n; e += blockDim.x) {
        const int c = g * cpg + e / HW, px = e % HW;
        const size_t o = addr(e);
        float y = (p.in[o] - mean) * rstd * p.gamma[c] + p.beta[c];
        if (film) y = y * (film[c] + 1.0f) + film[p.C + c];
        if (p.silu) y = y / (1.0f + expf(-y));
        if (p.res) y += p.res[o];
        if (p.out_m) p.out_m[o] = y;
        if (out_o) out_o[o] = y;
        const int h = px / p.W, w = px % p.W, cb = c >> 3, sub = c & 7;
        if (out_un) {
            const int plane = ((h & 1) * 2 + (w & 1)) * ncb + cb;
            const int q = (h >> 1) * (p.W >> 1) + (w >> 1);
            out_un[((size_t)(plane * p.B + b) * (HW >> 2) + q) * 8 + sub] = y;
        }
        if (out_up) {
            const int W2 = p.W * 2;
            for (int d = 0; d < 4; ++d) {
                const int q = (2 * h + (d >> 1)) * W2 + 2 * w + (d & 1);
                out_up[((size_t)(cb * p.B + b) * (HW * 4) + q) * 8 + sub] = y;
            }
        }
    }
}
cudaError_t launch_gn_any(const GnParams& p, cudaStream_t s) {
    if (p.o_is_bf16) return cudaErrorInvalidValue;
    k_gn_any<<<p.B * p.groups, 128, 0, s>>>(p);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// inpainting mask: NCHW fp32 [B,ch,H,W] -> per-level blocked tensors (channels >= ch are zero): 8 fp32 channels, or on the
// 16-bit path 16 bf16 channels (the second 8-channel block all zero), rounded only at the store.  Bilinear rule of F.interpolate(mask, size=(h,w), mode='bilinear') (align_corners=False, no antialias; unet.py:338,362):
// src = (dst + 0.5) * in/out - 0.5 clamped at 0, i1 = min(i0 + 1, in - 1).  Level 0 is a copy and also evaluates the
// reference's bypass test torch.allclose(mask, 1) (unet.py:301: |m - 1| <= 1e-8 + 1e-5): *mode = 2 if any element fails.
// ------------------------------------------------------------------------------------------------
__global__ void k_mask_mode(int* mode, int value) { if (threadIdx.x == 0 && blockIdx.x == 0) *mode = value; }
template <typename TO>
__global__ void __launch_bounds__(128) k_mask_prep(MaskPrepParams p) {
    const int lvl = blockIdx.y, h = p.H >> lvl, w = p.W >> lvl, hw = h * w;
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    if (idx >= p.B * hw) return;
    const int b = idx / hw, px = idx % hw, oy = px / w, ox = px % w;
    const float sy = (float)p.H / (float)h, sx = (float)p.W / (float)w;
    float fy = sy * ((float)oy + 0.5f) - 0.5f, fx = sx * ((float)ox + 0.5f) - 0.5f;
    if (fy < 0.f) fy = 0.f;
    if (fx < 0.f) fx = 0.f;
    const int y0 = (int)fy, x0 = (int)fx;
    const int y1 = y0 + (y0 < p.H - 1 ? 1 : 0), x1 = x0 + (x0 < p.W - 1 ? 1 : 0);
    const float ly1 = fy - (float)y0, ly0 = 1.0f - ly1, lx1 = fx - (float)x0, lx0 = 1.0f - lx1;
    float o[8];
    bool not_ones = false;
#pragma unroll
    for (int c = 0; c < 8; ++c) {
        o[c] = 0.f;
        if (c < p.ch) {
            const float* m = p.mask + ((size_t)b * p.ch + c) * p.H * p.W;
            if (lvl == 0) {
                o[c] = m[px];
                if (!(fabsf(o[c] - 1.0f) <= 1e-8f + 1e-5f)) not_ones = true;
            } else {
                const float t0 = __fadd_rn(__fmul_rn(lx0, m[y0 * p.W + x0]), __fmul_rn(lx1, m[y0 * p.W + x1]));
                const float t1 = __fadd_rn(__fmul_rn(lx0, m[y1 * p.W + x0]), __fmul_rn(lx1, m[y1 * p.W + x1]));
                o[c] = __fadd_rn(__fmul_rn(ly0, t0), __fmul_rn(ly1, t1));
            }
        }
    }
    TO* out = reinterpret_cast<TO*>(p.out[lvl]);
    store8(out + ((size_t)b * hw + px) * 8, o);
    if (std::is_same<TO, __nv_bfloat16>::value) {            // zero block: channels 8..15 of the K16 slice
#pragma unroll
        for (int c = 0; c < 8; ++c) o[c] = 0.f;
        store8(out + ((size_t)(p.B + b) * hw + px) * 8, o);
    }
    if (not_ones) atomicMax(p.mode, 2);
}
cudaError_t launch_mask_prep(const MaskPrepParams& p, cudaStream_t s) {
    k_mask_mode<<<1, 32, 0, s>>>(p.mode, p.mask ? 1 : 0);
    if (p.mask) {
        dim3 grid((p.B * p.H * p.W + 127) / 128, p.n_levels);
        if (p.out_bf16) k_mask_prep<__nv_bfloat16><<<grid, 128, 0, s>>>(p);
        else k_mask_prep<float><<<grid, 128, 0, s>>>(p);
    }
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// LinearAttention core (unet.py:142-149).  One CTA (256 threads) per (sample, head); n <= 256.
// q: softmax over the 32 head channels per pixel, then * 32^-0.5;  k: softmax over pixels per
// channel;  ctx[d][e] = sum_n k[d,n] v[e,n];  out[e][n] = sum_d ctx[d][e] q[d,n].
// ------------------------------------------------------------------------------------------------
constexpr int LA_THREADS = 256;
template <typename T>
__global__ void __launch_bounds__(LA_THREADS) k_linattn(AttnParams p) {
    extern __shared__ float sm[];
    const int n = p.n, ld = n + 1;
    float* sq = sm;                 // [32][ld]
    float* sk = sq + 32 * ld;       // [32][ld]
    float* sv = sk + 32 * ld;       // [32][ld]
    float* ctx = sv + 32 * ld;      // [32][33]
    const int b = blockIdx.x >> 2, head = blockIdx.x & 3;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const T* qkv = reinterpret_cast<const T*>(p.qkv);

    // load q, k, v: 3 tensors x 4 channel blocks x n pixels, 8 channels per item
    for (int it = tid; it < 12 * n; it += LA_THREADS) {
        const int which = it / (4 * n), rem = it % (4 * n), cbl = rem / n, px = rem % n;
        const int plane = which * 16 + head * 4 + cbl;
        float x[8];
        load8(qkv + ((size_t)(plane * p.B + b) * n + px) * 8, x);
        float* dst = (which == 0 ? sq : which == 1 ? sk : sv) + (cbl * 8) * ld + px;
#pragma unroll
        for (int j = 0; j < 8; ++j) dst[j * ld] = x[j];
    }
    __syncthreads();
    // q: softmax over d for each pixel
    for (int px = tid; px < n; px += LA_THREADS) {
        float m = -INFINITY;
#pragma unroll 8
        for (int d = 0; d < 32; ++d) m = fmaxf(m, sq[d * ld + px]);
        float s = 0.f;
#pragma unroll 8
        for (int d = 0; d < 32; ++d) { const float e = expf(sq[d * ld + px] - m); sq[d * ld + px] = e; s += e; }
        const float scale = 0.17677669529663687f;      // 32^-0.5
#pragma unroll 8
        for (int d = 0; d < 32; ++d) sq[d * ld + px] = (sq[d * ld + px] / s) * scale;
    }
    // k: softmax over pixels for each channel (one warp per channel)
    for (int d = warp; d < 32; d += LA_THREADS / 32) {
        float m = -INFINITY;
        for (int px = lane; px < n; px += 32) m = fmaxf(m, sk[d * ld + px]);
        m = warp_max(m);
        float s = 0.f;
        for (int px = lane; px < n; px += 32) { const float e = expf(sk[d * ld + px] - m); sk[d * ld + px] = e; s += e; }
        s = warp_sum(s);
        for (int px = lane; px < n; px += 32) sk[d * ld + px] = sk[d * ld + px] / s;
    }
    __syncthreads();
    // ctx[d][e]: warp w owns d = 4w..4w+3, lane = e
    {
        float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
        const float* k0 = sk + (warp * 4) * ld;
        const float* vv = sv + lane * ld;
        for (int px = 0; px < n; ++px) {
            const float x = vv[px];
            a0 = fmaf(k0[px], x, a0);
            a1 = fmaf(k0[ld + px], x, a1);
            a2 = fmaf(k0[2 * ld + px], x, a2);
            a3 = fmaf(k0[3 * ld + px], x, a3);
        }
        ctx[(warp * 4 + 0) * 33 + lane] = a0;
        ctx[(warp * 4 + 1) * 33 + lane] = a1;
        ctx[(warp * 4 + 2) * 33 + lane] = a2;
        ctx[(warp * 4 + 3) * 33 + lane] = a3;
    }
    __syncthreads();
    // out[e][px] = sum_d ctx[d][e] q[d][px]; thread = pixel
    T* out = reinterpret_cast<T*>(p.out);
    for (int px = tid; px < n; px += LA_THREADS) {
        float qv[32];
#pragma unroll
        for (int d = 0; d < 32; ++d) qv[d] = sq[d * ld + px];
#pragma unroll 1
        for (int cbl = 0; cbl < 4; ++cbl) {
            float o[8];
#pragma unroll
            for (int j = 0; j < 8; ++j) {
                const int e = cbl * 8 + j;
                float a = 0.f;
#pragma unroll
                for (int d = 0; d < 32; ++d) a = fmaf(ctx[d * 33 + e], qv[d], a);
                o[j] = a;
            }
            store8(out + ((size_t)((head * 4 + cbl) * p.B + b) * n + px) * 8, o);
        }
    }
}
// Same block for n > 256 pixels (fp32 path; e.g. the 32x32 "latents" of configs/flowers_resize.yaml): the sample does not fit in
// shared memory, so the pixels stream through in tiles of 256.  Pass 1: per-channel max of k over all pixels; pass 2: per tile
// exp(k - max) and the running sums  ksum[d] += sum_n e,  ctx[d][e] += sum_n e v[e,n]  (ctx / ksum == softmax_n(k) v^T, unet.py:142-146);
// pass 3: per tile softmax_d(q) * 32^-0.5 and out[e][n] = sum_d ctx[d][e] q[d,n]  (unet.py:141,143,148).
constexpr int LA_TILE = 256;
__global__ void __launch_bounds__(LA_THREADS) k_linattn_big(AttnParams p) {
    extern __shared__ float sm[];
    const int n = p.n, ld = LA_TILE + 1;
    float* sq = sm;                 // [32][ld]  (k tile in pass 2, q tile in pass 3)
    float* sv = sq + 32 * ld;       // [32][ld]
    float* ctx = sv + 32 * ld;      // [32][33]
    float* kmax = ctx + 32 * 33;    // [32]
    float* ksum = kmax + 32;        // [32]
    float* red = ksum + 32;         // [8][32]
    const int b = blockIdx.x >> 2, head = blockIdx.x & 3;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const float* qkv = reinterpret_cast<const float*>(p.qkv);
    auto src = [&](int which, int cbl, int px) { return qkv + ((size_t)((which * 16 + head * 4 + cbl) * p.B + b) * n + px) * 8; };
    // ---- pass 1: kmax[d]
    {
        float m[32];
#pragma unroll
        for (int d = 0; d < 32; ++d) m[d] = -INFINITY;
        for (int px = tid; px < n; px += LA_THREADS)
#pragma unroll
            for (int cbl = 0; cbl < 4; ++cbl) {
                float x[8];
                load8(src(1, cbl, px), x);
#pragma unroll
                for (int j = 0; j < 8; ++j) m[cbl * 8 + j] = fmaxf(m[cbl * 8 + j], x[j]);
            }
#pragma unroll
        for (int d = 0; d < 32; ++d) {
            const float w = warp_max(m[d]);
            if (lane == 0) red[warp * 32 + d] = w;
        }
        __syncthreads();
        if (tid < 32) {
            float w = red[tid];
            for (int k = 1; k < LA_THREADS / 32; ++k) w = fmaxf(w, red[k * 32 + tid]);
            kmax[tid] = w;
        }
        __syncthreads();
    }
    // ---- pass 2: ksum, ctx over the tiles; warp w owns d = 4w..4w+3, lane = e
    float a[4] = {0.f, 0.f, 0.f, 0.f}, ks[4] = {0.f, 0.f, 0.f, 0.f};
    for (int t0 = 0; t0 < n; t0 += LA_TILE) {
        for (int it = tid; it < 8 * LA_TILE; it += LA_THREADS) {
            const int which = 1 + it / (4 * LA_TILE), rem = it % (4 * LA_TILE), cbl = rem / LA_TILE, px = rem % LA_TILE;
            float x[8];
            load8(src(which, cbl, t0 + px), x);
            float* dst = (which == 1 ? sq : sv) + (cbl * 8) * ld + px;
#pragma unroll
            for (int j = 0; j < 8; ++j) dst[j * ld] = which == 1 ? expf(x[j] - kmax[cbl * 8 + j]) : x[j];
        }
        __syncthreads();
        const float* k0 = sq + (warp * 4) * ld;
        const float* vv = sv + lane * ld;
        for (int px = 0; px < LA_TILE; ++px) {
            const float x = vv[px];
#pragma unroll
            for (int j = 0; j < 4; ++j) a[j] = fmaf(k0[j * ld + px], x, a[j]);
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            float sacc = 0.f;
            for (int px = lane; px < LA_TILE; px += 32) sacc += k0[j * ld + px];
            ks[j] += warp_sum(sacc);
        }
        __syncthreads();
    }
#pragma unroll
    for (int j = 0; j < 4; ++j) ctx[(warp * 4 + j) * 33 + lane] = a[j] / ks[j];
    __syncthreads();
    // ---- pass 3: q softmax over d, out
    float* out = reinterpret_cast<float*>(p.out);
    for (int t0 = 0; t0 < n; t0 += LA_TILE) {
        for (int it = tid; it < 4 * LA_TILE; it += LA_THREADS) {
            const int cbl = it / LA_TILE, px = it % LA_TILE;
            float x[8];
            load8(src(0, cbl, t0 + px), x);
#pragma unroll
            for (int j = 0; j < 8; ++j) sq[(cbl * 8 + j) * ld + px] = x[j];
        }
        __syncthreads();
        {
            const int px = tid;                                   // LA_TILE == LA_THREADS
            float qv[32], m = -INFINITY, ssum = 0.f;
#pragma unroll
            for (int d = 0; d < 32; ++d) { qv[d] = sq[d * ld + px]; m = fmaxf(m, qv[d]); }
#pragma unroll
            for (int d = 0; d < 32; ++d) { qv[d] = expf(qv[d] - m); ssum += qv[d]; }
#pragma unroll
            for (int d = 0; d < 32; ++d) qv[d] = (qv[d] / ssum) * 0.17677669529663687f;
#pragma unroll 1
            for (int cbl = 0; cbl < 4; ++cbl) {
                float o[8];
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int e = cbl * 8 + j;
                    float acc = 0.f;
#pragma unroll
                    for (int d = 0; d < 32; ++d) acc = fmaf(ctx[d * 33 + e], qv[d], acc);
                    o[j] = acc;
                }
                store8(out + ((size_t)((head * 4 + cbl) * p.B + b) * n + t0 + px) * 8, o);
            }
        }
        __syncthreads();
    }
}
static size_t linattn_big_smem() { return (size_t)(2 * 32 * (LA_TILE + 1) + 32 * 33 + 64 + 8 * 32) * sizeof(float); }
static size_t linattn_smem(int n) { return (size_t)(3 * 32 * (n + 1) + 32 * 33) * sizeof(float); }
cudaError_t simt_configure() {
    cudaError_t e = cudaFuncSetAttribute(k_gn_tma<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, GNT_MAX_SMEM + 1024);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_gn_tma<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize, GNT_MAX_SMEM + 1024);
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(k_linattn_big, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)linattn_big_smem());
    if (e != cudaSuccess) return e;
    e = cudaFuncSetAttribute(k_linattn<float>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)linattn_smem(256));
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(k_linattn<__nv_bfloat16>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                (int)linattn_smem(256));
}
// up to 256 pixels: one CTA holds q, k, v of a (sample, head); beyond, the fp32 tiled kernel takes whole LA_TILE tiles
bool linattn_supported(int n, bool bf16) { return n >= 1 && (n <= 256 || (!bf16 && n % LA_TILE == 0)); }
cudaError_t launch_linattn(const AttnParams& p, cudaStream_t s) {
    if (!linattn_supported(p.n, p.is_bf16)) return cudaErrorInvalidValue;
    if (p.n > 256) {
        k_linattn_big<<<p.B * 4, LA_THREADS, linattn_big_smem(), s>>>(p);
        return cudaGetLastError();
    }
    const size_t smem = linattn_smem(p.n);
    if (p.is_bf16) k_linattn<__nv_bfloat16><<<p.B * 4, LA_THREADS, smem, s>>>(p);
    else k_linattn<float><<<p.B * 4, LA_THREADS, smem, s>>>(p);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// mid-block Attention core (unet.py:114-121), n = H*W <= 64.  One CTA (64 threads) per (sample, head).
// ------------------------------------------------------------------------------------------------
constexpr int MA_MAXN = 64;
template <typename T>
__global__ void __launch_bounds__(64) k_midattn(AttnParams p) {
    __shared__ float sq[32][MA_MAXN + 1], sk[32][MA_MAXN + 1], sv[32][MA_MAXN + 1];
    __shared__ float sim[MA_MAXN][MA_MAXN + 1];
    const int n = p.n;
    const int b = blockIdx.x >> 2, head = blockIdx.x & 3, tid = threadIdx.x;
    const T* qkv = reinterpret_cast<const T*>(p.qkv);
    for (int it = tid; it < 12 * n; it += 64) {
        const int which = it / (4 * n), rem = it % (4 * n), cbl = rem / n, px = rem % n;
        const int plane = which * 16 + head * 4 + cbl;
        float x[8];
        load8(qkv + ((size_t)(plane * p.B + b) * n + px) * 8, x);
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            if (which == 0) sq[cbl * 8 + j][px] = x[j] * 0.17677669529663687f;   // q * scale (unet.py:114)
            else if (which == 1) sk[cbl * 8 + j][px] = x[j];
            else sv[cbl * 8 + j][px] = x[j];
        }
    }
    __syncthreads();
    for (int ij = tid; ij < n * n; ij += 64) {
        const int i = ij / n, j = ij % n;
        float a = 0.f;
#pragma unroll 8
        for (int d = 0; d < 32; ++d) a = fmaf(sq[d][i], sk[d][j], a);
        sim[i][j] = a;
    }
    __syncthreads();
    for (int i = tid; i < n; i += 64) {          // softmax over j (the amax subtraction of unet.py:117 included)
        float m = -INFINITY;
        for (int j = 0; j < n; ++j) m = fmaxf(m, sim[i][j]);
        float s = 0.f;
        for (int j = 0; j < n; ++j) { const float e = expf(sim[i][j] - m); sim[i][j] = e; s += e; }
        for (int j = 0; j < n; ++j) sim[i][j] = sim[i][j] / s;
    }
    __syncthreads();
    // out[i][d] = sum_j attn[i][j] v[d][j] -> channel head*32+d at pixel i  ('b h (x y) d -> b (h d) x y')
    T* out = reinterpret_cast<T*>(p.out);
    for (int it = tid; it < 4 * n; it += 64) {
        const int cbl = it / n, i = it % n;
        float o[8];
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) {
            const int d = cbl * 8 + jj;
            float a = 0.f;
            for (int j = 0; j < n; ++j) a = fmaf(sim[i][j], sv[d][j], a);
            o[jj] = a;
        }
        store8(out + ((size_t)((head * 4 + cbl) * p.B + b) * n + i) * 8, o);
    }
}
bool midattn_supported(int n) { return n >= 1 && n <= MA_MAXN; }
cudaError_t launch_midattn(const AttnParams& p, cudaStream_t s) {
    if (!midattn_supported(p.n)) return cudaErrorInvalidValue;
    if (p.is_bf16) k_midattn<__nv_bfloat16><<<p.B * 4, 64, 0, s>>>(p);
    else k_midattn<float><<<p.B * 4, 64, 0, s>>>(p);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// time embedding -> FiLM rows.  grid (n_rows, splits); each CTA recomputes the small MLP and
// produces a slice of the row's film_dim outputs.
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ float gelu_erf(float x) { return x * 0.5f * (1.0f + erff(x * 0.70710678118654752440f)); }

__global__ void __launch_bounds__(128) k_temb(TembParams p) {
    extern __shared__ float sm[];
    float* e = sm;                       // [dim]
    float* h = e + p.dim;                // [time_dim]
    float* t = h + p.time_dim;           // [time_dim]
    float* c = t + p.time_dim;           // [time_dim]
    const int row = blockIdx.x, tid = threadIdx.x, NT = blockDim.x;
    const float tv = p.ctrl ? p.ctrl->stages[p.ctrl->step].t_scaled : p.t[(size_t)row * p.t_stride];
    const int half = p.dim >> 1;
    for (int j = tid; j < half; j += NT) {           // unet.py:28-29: [sin | cos]
        const float a = tv * p.freqs[j];
        e[j] = sinf(a);
        e[half + j] = cosf(a);
    }
    __syncthreads();
    for (int j = tid; j < p.time_dim; j += NT) {     // Linear(dim, time_dim) -> GELU
        float a = p.b1[j];
        for (int i = 0; i < p.dim; ++i) a = fmaf(e[i], p.w1t[i * p.time_dim + j], a);
        h[j] = gelu_erf(a);
    }
    __syncthreads();
    for (int j = tid; j < p.time_dim; j += NT) {     // Linear(time_dim, time_dim)
        float a = p.b2[j];
        for (int i = 0; i < p.time_dim; ++i) a = fmaf(h[i], p.w2t[i * p.time_dim + j], a);
        t[j] = a;
    }
    if (p.cls != nullptr && p.n_classes > 0 && (p.n_cond < 0 || row < p.n_cond)) {       // class_cond_mlp (unet.py:207-212,316)
        __syncthreads();
        long long id = p.cls[row];
        if (id < 0) id = 0;
        if (id >= p.n_classes) id = p.n_classes - 1;
        const float* emb = p.emb + (size_t)id * p.time_dim;
        for (int j = tid; j < p.time_dim; j += NT) {
            float a = p.bc1[j];
            for (int i = 0; i < p.time_dim; ++i) a = fmaf(emb[i], p.wc1t[i * p.time_dim + j], a);
            c[j] = gelu_erf(a);
        }
        __syncthreads();
        for (int j = tid; j < p.time_dim; j += NT) {
            float a = p.bc3[j];
            for (int i = 0; i < p.time_dim; ++i) a = fmaf(c[i], p.wc3t[i * p.time_dim + j], a);
            t[j] += a;
        }
    }
    __syncthreads();
    for (int j = tid; j < p.time_dim; j += NT) {     // ResnetBlock.mlp[0] = SiLU (unet.py:80)
        const float x = t[j];
        h[j] = x / (1.0f + expf(-x));
    }
    __syncthreads();
    const int per = (p.film_dim + gridDim.y - 1) / gridDim.y;
    const int o0 = blockIdx.y * per, o1 = min(p.film_dim, o0 + per);
    for (int o = o0 + tid; o < o1; o += NT) {        // all ResnetBlock Linear(time_dim, 2*dim_out) at once
        float a = p.bf[o];
        for (int i = 0; i < p.time_dim; ++i) a = fmaf(h[i], p.wft[(size_t)i * p.film_dim + o], a);
        p.film[(size_t)row * p.film_dim + o] = a;
    }
}
cudaError_t launch_temb(const TembParams& p, cudaStream_t s) {
    if (p.n_rows <= 0) return cudaSuccess;
    const size_t smem = (size_t)(p.dim + 3 * p.time_dim) * sizeof(float);
    int splits = p.n_rows >= 256 ? 2 : 16;
    dim3 grid(p.n_rows, splits);
    k_temb<<<grid, 128, smem, s>>>(p);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// final_conv 1x1 + integrator stage epilogue
// ------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(128) k_final(FinalParams p) {
    Ctrl* c = p.ctrl;
    const int step = c->step;
    const Stage st = c->stages[step];
    const int idx = blockIdx.x * blockDim.x + threadIdx.x;
    const int ns = p.n_bias_rows ? p.n_bias_rows : p.B;      // samples; rows from ns on are JVP tangents
    if (idx < p.B * p.HW) {
        const int b = idx / p.HW, px = idx % p.HW;
        float x[64];
        const int ncb = p.dim >> 3;
        for (int cb = 0; cb < ncb; ++cb) load8(p.in + ((size_t)(cb * p.B + b) * p.HW + px) * 8, x + cb * 8);
        const size_t plane = (size_t)ns * p.channels * p.HW;
        for (int co = 0; co < p.channels; ++co) {
            float k = 0.f;
            for (int i = 0; i < p.dim; ++i) k = fmaf(x[i], p.w[co * p.dim + i], k);
            const size_t o = ((size_t)b * p.channels + co) * p.HW + px;
            if (b >= ns) {                          // tangent row: dv, or eps * dv with the probe eps held in xs
                c->vtan[o - plane] = st.kind == ST_PLAIN ? k : k * c->xs[o];
                continue;
            }
            k += p.bias[co];
            if (st.flags & SF_CFG_COMBINE) {        // v = v_nc + cfg*(v_c - v_nc)   (sampling.py:74)
                const float vc = c->vcond[o];
                k = __fadd_rn(k, __fmul_rn(c->cfg, __fsub_rn(vc, k)));
            }
            if (c->vtrace && st.eval_idx >= 0) c->vtrace[(size_t)st.eval_idx * plane + o] = k;
            switch (st.kind) {
                case ST_PLAIN: c->vout[o] = k; break;
                case ST_CFG_COND: c->vcond[o] = k; break;
                case ST_RK1: {
                    c->acc[o] = k;
                    c->xs[o] = __fadd_rn(c->y[o], __fmul_rn(__fmul_rn(st.dt, k), 0.5f));
                } break;
                case ST_RK2: {
                    c->acc[o] = __fadd_rn(c->acc[o], __fmul_rn(2.0f, k));
                    c->xs[o] = __fadd_rn(c->y[o], __fmul_rn(__fmul_rn(st.dt, k), 0.5f));
                } break;
                case ST_RK3: {
                    c->acc[o] = __fadd_rn(c->acc[o], __fmul_rn(2.0f, k));
                    c->xs[o] = __fadd_rn(c->y[o], __fmul_rn(st.dt, k));
                } break;
                case ST_RK4: {
                    const float a = __fadd_rn(c->acc[o], k);
                    const float yn = __fadd_rn(c->y[o], __fmul_rn(st.dt6, a));
                    c->y[o] = yn; c->xs[o] = yn;
                } break;
                case ST_EULER: {
                    const float yn = __fadd_rn(c->y[o], __fmul_rn(k, st.dt));
                    c->y[o] = yn; c->xs[o] = yn;
                } break;
                default: break;
            }
        }
    }
    // the last CTA to finish advances the stage counter: every CTA has read `step` before it arrives here
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        const int done = atomicAdd(&c->done_ctr, 1);
        if (done == (int)gridDim.x - 1) {
            c->done_ctr = 0;
            c->step = step + 1;
            __threadfence();
        }
    }
}
cudaError_t launch_final(const FinalParams& p, cudaStream_t s) {
    const int n = p.B * p.HW;
    k_final<<<(n + 127) / 128, 128, 0, s>>>(p);
    return cudaGetLastError();
}

}  // namespace flo
