// Forward-mode Jacobian-vector products of the fp32 layer-by-layer program (sm_100a), for flo_unet_jvp and
// flo_integrate_divergence.
//
// A JVP plan runs the fp32 op program over R = (1+P)*B rows of the blocked layout: rows [0, B) are the samples (primal),
// row B*(1+p) + b is tangent p of sample b.  Every linear op (init conv, convolutions with their residual adds and the
// pixel-unshuffle / nearest-x2 copies, the final conv) computes its tangent rows as the same op without bias, in the same
// launch.  The three nonlinear op kinds have the kernels below; each takes the sample count B (GnParams::B, AttnParams::B)
// and the row stride R separately, and writes the primal rows exactly as the fp32 forward does.
//
//   k_gn_jvp        GroupNorm + FiLM + SiLU + residual, any channels per group.  x^ = (x - mu) r,
//                   dx^ = r (dx - mean(dx) - x^ mean(x^ dx)), dh = dx^ gamma (scale + 1), SiLU: dy = s(h) (1 + h (1 - s(h))) dh
//   k_linattn_jvp   LinearAttention core (n <= 256): q~ = softmax_d(q) 32^-1/2, k~ = softmax_n(k), ctx = k~ v^T, out = ctx^T q~;
//                   dq~ = q~ (dq - sum_d q' dq), dk~ = k~ (dk - sum_n k~ dk), dctx = dk~ v^T + k~ dv^T, dout = dctx^T q~ + ctx^T dq~
//   k_midattn_jvp   mid-block Attention core (n <= 64): P = softmax(s q k^T); dS = s (dq k^T + q dk^T),
//                   dP = P (dS - rowsum(P dS)), dout = dP v + P dv
//   k_div_reduce    div[b] += dt/6 w (1/P) sum_p sum_chw eps_p dv_p (the products k_final wrote), fp64, fixed order
#include <math.h>

#include "flo_internal.h"

namespace flo {

namespace {

__device__ __forceinline__ void ld8(const float* src, float v[8]) {
    const float4 a = *reinterpret_cast<const float4*>(src);
    const float4 b = *reinterpret_cast<const float4*>(src + 4);
    v[0] = a.x; v[1] = a.y; v[2] = a.z; v[3] = a.w; v[4] = b.x; v[5] = b.y; v[6] = b.z; v[7] = b.w;
}
__device__ __forceinline__ void st8(float* dst, const float v[8]) {
    *reinterpret_cast<float4*>(dst) = make_float4(v[0], v[1], v[2], v[3]);
    *reinterpret_cast<float4*>(dst + 4) = make_float4(v[4], v[5], v[6], v[7]);
}
__device__ __forceinline__ float wsum(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ float wmax(float v) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
    return v;
}
// block-wide sum (every thread gets it); red holds >= 32 floats
__device__ __forceinline__ float bsum(float v, float* red) {
    v = wsum(v);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5, nw = (blockDim.x + 31) >> 5;
    if (nw == 1) return v;
    __syncthreads();
    if (lane == 0) red[warp] = v;
    __syncthreads();
    return wsum(lane < nw ? red[lane] : 0.f);
}

constexpr float ATTN_SCALE = 0.17677669529663687f;     // 32^-0.5

}  // namespace

// ------------------------------------------------------------------------------------------------
// GroupNorm JVP.  Grid (B * groups, 1 + P): y = 0 writes the primal rows, y = 1 + p tangent p.  Every CTA computes the
// primal statistics of its (sample, group) with the two passes of the fp32 GroupNorm kernels.  The group's elements are
// walked in memory order over the channel blocks it touches (coalesced for any channels per group, lanes outside the
// group idle).
// ------------------------------------------------------------------------------------------------
constexpr int GNJ_THREADS = 256;
__global__ void __launch_bounds__(GNJ_THREADS) k_gn_jvp(GnParams p, int R) {
    __shared__ float red[32];
    const int G = p.groups, cpg = p.C / G, HW = p.H * p.W, n = cpg * HW, blk = HW * 8;
    const int b = blockIdx.x / G, g = blockIdx.x % G, t = blockIdx.y;
    const int c0 = g * cpg, cb0 = c0 >> 3, span = (((c0 + cpg - 1) >> 3) - cb0 + 1) * blk;
    auto chan = [&](int i) { return cb0 * 8 + (i / blk) * 8 + (i & 7); };
    auto off = [&](int row, int i) { return ((size_t)((cb0 + i / blk) * R + row) * HW) * 8 + (i % blk); };
    auto mine = [&](int c) { return c >= c0 && c < c0 + cpg; };

    float s = 0.f;
    for (int i = threadIdx.x; i < span; i += blockDim.x)
        if (mine(chan(i))) s += p.in[off(b, i)];
    const float mean = bsum(s, red) / (float)n;
    float q = 0.f;
    for (int i = threadIdx.x; i < span; i += blockDim.x)
        if (mine(chan(i))) { const float d = p.in[off(b, i)] - mean; q += d * d; }
    const float rstd = 1.0f / sqrtf(bsum(q, red) / (float)n + 1e-5f);     // biased variance (nn.GroupNorm)

    const float* film = nullptr;
    if (p.film_off >= 0) {
        const Ctrl* c = p.ctrl;
        const int frow = c->film_per_sample ? b : c->stages[c->step].film_row;
        film = c->film + (size_t)frow * p.film_dim + p.film_off;
    }
    float* out_o = reinterpret_cast<float*>(p.out_o);
    float* out_un = reinterpret_cast<float*>(p.out_unshuf);
    float* out_up = reinterpret_cast<float*>(p.out_up);
    const int ncb = p.C >> 3;
    auto put = [&](int row, int i, float y) {
        const size_t o = off(row, i);
        if (p.out_m) p.out_m[o] = y;
        if (out_o) out_o[o] = y;
        if (out_un || out_up) {
            const int c = chan(i), px = (i % blk) >> 3, h = px / p.W, w = px % p.W, cb = c >> 3, sub = c & 7;
            if (out_un) {   // 'b c (h p1) (w p2) -> b (c p1 p2) h w' in our (p1 p2 c) channel order
                const int plane = ((h & 1) * 2 + (w & 1)) * ncb + cb;
                const int q2 = (h >> 1) * (p.W >> 1) + (w >> 1);
                out_un[((size_t)(plane * R + row) * (HW >> 2) + q2) * 8 + sub] = y;
            }
            if (out_up) {   // nearest x2
                const int W2 = p.W * 2;
                for (int d = 0; d < 4; ++d) {
                    const int q2 = (2 * h + (d >> 1)) * W2 + 2 * w + (d & 1);
                    out_up[((size_t)(cb * R + row) * (HW * 4) + q2) * 8 + sub] = y;
                }
            }
        }
    };

    if (t == 0) {                      // primal rows: the fp32 GroupNorm epilogue (unet.py:64-73)
        for (int i = threadIdx.x; i < span; i += blockDim.x) {
            const int c = chan(i);
            if (!mine(c)) continue;
            float y = (p.in[off(b, i)] - mean) * rstd * p.gamma[c] + p.beta[c];
            if (film) y = y * (film[c] + 1.0f) + film[p.C + c];
            if (p.silu) y = y / (1.0f + expf(-y));
            if (p.res) y += p.res[off(b, i)];
            put(b, i, y);
        }
        return;
    }
    const int row = p.B * t + b;
    float sd = 0.f, sxd = 0.f;
    for (int i = threadIdx.x; i < span; i += blockDim.x) {
        if (!mine(chan(i))) continue;
        const float xh = (p.in[off(b, i)] - mean) * rstd, d = p.in[off(row, i)];
        sd += d;
        sxd = fmaf(xh, d, sxd);
    }
    const float md = bsum(sd, red) / (float)n;
    const float mxd = bsum(sxd, red) / (float)n;
    for (int i = threadIdx.x; i < span; i += blockDim.x) {
        const int c = chan(i);
        if (!mine(c)) continue;
        const float xh = (p.in[off(b, i)] - mean) * rstd, d = p.in[off(row, i)];
        const float sc = film ? film[c] + 1.0f : 1.0f;
        float dy = rstd * (d - md - xh * mxd) * p.gamma[c] * sc;
        if (p.silu) {
            float h = xh * p.gamma[c] + p.beta[c];
            if (film) h = h * sc + film[p.C + c];
            const float sg = 1.0f / (1.0f + expf(-h));
            dy *= sg * (1.0f + h * (1.0f - sg));
        }
        if (p.res) dy += p.res[off(row, i)];
        put(row, i, dy);
    }
}
cudaError_t launch_gn_jvp(const GnParams& p, int R, cudaStream_t s) {
    if (p.o_is_bf16 || p.groups < 1 || p.C % p.groups || R % p.B) return cudaErrorInvalidValue;
    k_gn_jvp<<<dim3(p.B * p.groups, R / p.B), GNJ_THREADS, 0, s>>>(p, R);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// LinearAttention JVP, n <= 256.  Grid (B * 4 heads, P): CTA (sample, head, p) recomputes the primal block exactly as
// k_linattn and forms tangent p; the CTAs of p = 0 also write the primal output.  Four [32][n+1] planes: k~ | v | dk~ | dv
// for the contexts, then q | dq in the first and third.
// ------------------------------------------------------------------------------------------------
constexpr int LAJ_THREADS = 256;
static size_t linattn_jvp_smem(int n) { return (size_t)(4 * 32 * (n + 1) + 2 * 32 * 33) * sizeof(float); }
__global__ void __launch_bounds__(LAJ_THREADS) k_linattn_jvp(AttnParams p, int R) {
    extern __shared__ float sm[];
    const int n = p.n, ld = n + 1;
    float* sa = sm;                 // k~, then q
    float* sb = sa + 32 * ld;       // v
    float* sc = sb + 32 * ld;       // dk~, then dq
    float* sd = sc + 32 * ld;       // dv
    float* ctx = sd + 32 * ld;      // [32][33]
    float* dctx = ctx + 32 * 33;    // [32][33]
    const int b = blockIdx.x >> 2, head = blockIdx.x & 3, row = p.B * (1 + blockIdx.y) + b;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const float* qkv = reinterpret_cast<const float*>(p.qkv);
    auto load = [&](int which, int r, float* dst) {     // which: 0 q, 1 k, 2 v (4 channel blocks of this head)
        for (int it = tid; it < 4 * n; it += LAJ_THREADS) {
            const int cbl = it / n, px = it % n;
            float x[8];
            ld8(qkv + ((size_t)((which * 16 + head * 4 + cbl) * R + r) * n + px) * 8, x);
#pragma unroll
            for (int j = 0; j < 8; ++j) dst[(cbl * 8 + j) * ld + px] = x[j];
        }
    };
    load(1, b, sa); load(2, b, sb); load(1, row, sc); load(2, row, sd);
    __syncthreads();
    // k~ = softmax over pixels per channel (k_linattn's operation order), dk~ = k~ (dk - sum_n k~ dk)
    for (int d = warp; d < 32; d += LAJ_THREADS / 32) {
        float* k = sa + d * ld;
        float* dk = sc + d * ld;
        float m = -INFINITY;
        for (int px = lane; px < n; px += 32) m = fmaxf(m, k[px]);
        m = wmax(m);
        float s = 0.f;
        for (int px = lane; px < n; px += 32) { const float e = expf(k[px] - m); k[px] = e; s += e; }
        s = wsum(s);
        float dot = 0.f;
        for (int px = lane; px < n; px += 32) { k[px] = k[px] / s; dot = fmaf(k[px], dk[px], dot); }
        dot = wsum(dot);
        for (int px = lane; px < n; px += 32) dk[px] = k[px] * (dk[px] - dot);
    }
    __syncthreads();
    // ctx[d][e] = sum_n k~[d,n] v[e,n] and its tangent; warp w owns d = 4w..4w+3, lane = e
    {
        float a[4] = {0.f, 0.f, 0.f, 0.f}, da[4] = {0.f, 0.f, 0.f, 0.f};
        const float* k0 = sa + (warp * 4) * ld;
        const float* dk0 = sc + (warp * 4) * ld;
        const float* vv = sb + lane * ld;
        const float* dvv = sd + lane * ld;
        for (int px = 0; px < n; ++px) {
            const float x = vv[px], dx = dvv[px];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                a[j] = fmaf(k0[j * ld + px], x, a[j]);
                da[j] = fmaf(dk0[j * ld + px], x, fmaf(k0[j * ld + px], dx, da[j]));
            }
        }
#pragma unroll
        for (int j = 0; j < 4; ++j) { ctx[(warp * 4 + j) * 33 + lane] = a[j]; dctx[(warp * 4 + j) * 33 + lane] = da[j]; }
    }
    __syncthreads();
    load(0, b, sa); load(0, row, sc);
    __syncthreads();
    // per pixel: q~ = softmax_d(q) * 32^-1/2 (k_linattn's order) in registers, and with dq~ = q~ (dq - sum_d q' dq) back into
    // the pixel's own columns of the q and dq planes; out and dout
    float* out = reinterpret_cast<float*>(p.out);
    for (int px = tid; px < n; px += LAJ_THREADS) {
        float qv[32], m = -INFINITY, s = 0.f, dot = 0.f;
        float* dqc = sc + px;
#pragma unroll
        for (int d = 0; d < 32; ++d) { qv[d] = sa[d * ld + px]; m = fmaxf(m, qv[d]); }
#pragma unroll
        for (int d = 0; d < 32; ++d) { qv[d] = expf(qv[d] - m); s += qv[d]; }
#pragma unroll
        for (int d = 0; d < 32; ++d) {
            const float qu = qv[d] / s;             // q' (unscaled softmax)
            dot = fmaf(qu, dqc[d * ld], dot);
            qv[d] = qu * ATTN_SCALE;
        }
#pragma unroll
        for (int d = 0; d < 32; ++d) { dqc[d * ld] = qv[d] * (dqc[d * ld] - dot); sa[d * ld + px] = qv[d]; }
#pragma unroll 1
        for (int cbl = 0; cbl < 4; ++cbl) {
            const int plane = head * 4 + cbl;
            float o[8];
            if (blockIdx.y == 0) {
#pragma unroll
                for (int j = 0; j < 8; ++j) {
                    const int e = cbl * 8 + j;
                    float acc = 0.f;
#pragma unroll
                    for (int d = 0; d < 32; ++d) acc = fmaf(ctx[d * 33 + e], qv[d], acc);
                    o[j] = acc;
                }
                st8(out + ((size_t)(plane * R + b) * n + px) * 8, o);
            }
#pragma unroll
            for (int j = 0; j < 8; ++j) o[j] = 0.f;
#pragma unroll 1
            for (int d = 0; d < 32; ++d) {
                const float qd = sa[d * ld + px], dqd = dqc[d * ld];
#pragma unroll
                for (int j = 0; j < 8; ++j) o[j] = fmaf(dctx[d * 33 + cbl * 8 + j], qd, fmaf(ctx[d * 33 + cbl * 8 + j], dqd, o[j]));
            }
            st8(out + ((size_t)(plane * R + row) * n + px) * 8, o);
        }
    }
}
cudaError_t launch_linattn_jvp(const AttnParams& p, int R, cudaStream_t s) {
    if (p.is_bf16 || p.n < 1 || p.n > LINATTN_JVP_MAX_N || R % p.B || R / p.B < 2) return cudaErrorInvalidValue;
    k_linattn_jvp<<<dim3(p.B * 4, R / p.B - 1), LAJ_THREADS, linattn_jvp_smem(p.n), s>>>(p, R);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// mid-block Attention JVP, n <= 64.  Grid (B * 4 heads, P), 64 threads; the primal as k_midattn, written by the CTAs of
// p = 0.  Shared memory: q*s | k | v | dq*s | dk | dv as [32][65], the attention matrix and its tangent as [64][65].
// ------------------------------------------------------------------------------------------------
constexpr int MAJ_N = 64, MAJ_LD = MAJ_N + 1;
static size_t midattn_jvp_smem() { return (size_t)(6 * 32 * MAJ_LD + 2 * MAJ_N * MAJ_LD) * sizeof(float); }
__global__ void __launch_bounds__(64) k_midattn_jvp(AttnParams p, int R) {
    extern __shared__ float sm[];
    float* sim = sm + 6 * 32 * MAJ_LD;          // [64][65]
    float* dsim = sim + MAJ_N * MAJ_LD;         // [64][65]
    const int n = p.n;
    const int b = blockIdx.x >> 2, head = blockIdx.x & 3, tid = threadIdx.x, row = p.B * (1 + blockIdx.y) + b;
    const float* qkv = reinterpret_cast<const float*>(p.qkv);
    for (int it = tid; it < 24 * n; it += 64) {
        const int tg = it / (12 * n), rem = it % (12 * n), which = rem / (4 * n), cbl = (rem % (4 * n)) / n, px = rem % n;
        float x[8];
        ld8(qkv + ((size_t)((which * 16 + head * 4 + cbl) * R + (tg ? row : b)) * n + px) * 8, x);
        float* dst = sm + (tg * 3 + which) * 32 * MAJ_LD;        // q*s, k, v, dq*s, dk, dv
#pragma unroll
        for (int j = 0; j < 8; ++j) dst[(cbl * 8 + j) * MAJ_LD + px] = which == 0 ? x[j] * ATTN_SCALE : x[j];   // q * scale (unet.py:114)
    }
    __syncthreads();
    const float *sq = sm, *sk = sq + 32 * MAJ_LD, *sv = sk + 32 * MAJ_LD, *dq = sv + 32 * MAJ_LD, *dk = dq + 32 * MAJ_LD,
                *dv = dk + 32 * MAJ_LD;
    for (int ij = tid; ij < n * n; ij += 64) {
        const int i = ij / n, j = ij % n;
        float a = 0.f, da = 0.f;
#pragma unroll 8
        for (int d = 0; d < 32; ++d) {
            a = fmaf(sq[d * MAJ_LD + i], sk[d * MAJ_LD + j], a);
            da = fmaf(dq[d * MAJ_LD + i], sk[d * MAJ_LD + j], fmaf(sq[d * MAJ_LD + i], dk[d * MAJ_LD + j], da));
        }
        sim[i * MAJ_LD + j] = a;
        dsim[i * MAJ_LD + j] = da;
    }
    __syncthreads();
    for (int i = tid; i < n; i += 64) {        // softmax over j as k_midattn, then dP = P (dS - rowsum(P dS))
        float* srow = sim + i * MAJ_LD;
        float* drow = dsim + i * MAJ_LD;
        float m = -INFINITY;
        for (int j = 0; j < n; ++j) m = fmaxf(m, srow[j]);
        float s = 0.f;
        for (int j = 0; j < n; ++j) { const float e = expf(srow[j] - m); srow[j] = e; s += e; }
        float r = 0.f;
        for (int j = 0; j < n; ++j) { srow[j] = srow[j] / s; r = fmaf(srow[j], drow[j], r); }
        for (int j = 0; j < n; ++j) drow[j] = srow[j] * (drow[j] - r);
    }
    __syncthreads();
    float* out = reinterpret_cast<float*>(p.out);
    for (int it = tid; it < 4 * n; it += 64) {
        const int cbl = it / n, i = it % n;
        float o[8], dout[8];
#pragma unroll
        for (int jj = 0; jj < 8; ++jj) {
            const int d = cbl * 8 + jj;
            float a = 0.f, da = 0.f;
            for (int j = 0; j < n; ++j) {
                a = fmaf(sim[i * MAJ_LD + j], sv[d * MAJ_LD + j], a);
                da = fmaf(dsim[i * MAJ_LD + j], sv[d * MAJ_LD + j], fmaf(sim[i * MAJ_LD + j], dv[d * MAJ_LD + j], da));
            }
            o[jj] = a; dout[jj] = da;
        }
        const int plane = head * 4 + cbl;
        if (blockIdx.y == 0) st8(out + ((size_t)(plane * R + b) * n + i) * 8, o);
        st8(out + ((size_t)(plane * R + row) * n + i) * 8, dout);
    }
}
cudaError_t launch_midattn_jvp(const AttnParams& p, int R, cudaStream_t s) {
    if (p.is_bf16 || p.n < 1 || p.n > MAJ_N || R % p.B || R / p.B < 2) return cudaErrorInvalidValue;
    k_midattn_jvp<<<dim3(p.B * 4, R / p.B - 1), 64, midattn_jvp_smem(), s>>>(p, R);
    return cudaGetLastError();
}

// ------------------------------------------------------------------------------------------------
// Hutchinson divergence of one RK4 stage.  One CTA per sample; thread i sums elements i, i + 256, ... of every probe in
// order, then a fixed tree: the result depends on C*H*W and P only, never on the batch.
// ------------------------------------------------------------------------------------------------
constexpr int DIV_THREADS = 256;
__global__ void __launch_bounds__(DIV_THREADS) k_div_reduce(const Ctrl* c, double* div, int B, int P, int chw) {
    __shared__ double red[DIV_THREADS];
    const Stage st = c->stages[c->step - 1];        // k_final has advanced the counter past the stage reduced here
    const double w = (st.kind == ST_RK1 || st.kind == ST_RK4) ? 1.0 : (st.kind == ST_RK2 || st.kind == ST_RK3) ? 2.0 : 0.0;
    if (w == 0.0) return;                           // a plain JVP: ctrl.vtan holds dv, nothing to integrate
    const int b = blockIdx.x, tid = threadIdx.x;
    double s = 0.0;
    for (int q = 0; q < P; ++q) {
        const float* src = c->vtan + ((size_t)q * B + b) * chw;
        for (int i = tid; i < chw; i += DIV_THREADS) s += (double)src[i];
    }
    red[tid] = s;
    __syncthreads();
    for (int o = DIV_THREADS / 2; o > 0; o >>= 1) {
        if (tid < o) red[tid] += red[tid + o];
        __syncthreads();
    }
    if (tid == 0) div[b] += (double)st.dt / 6.0 * w * (red[0] / (double)P);
}
cudaError_t launch_div_reduce(const Ctrl* ctrl, double* div, int B, int P, int chw, cudaStream_t s) {
    k_div_reduce<<<B, DIV_THREADS, 0, s>>>(ctrl, div, B, P, chw);
    return cudaGetLastError();
}

cudaError_t jvp_configure() {
    cudaError_t e = cudaFuncSetAttribute(k_linattn_jvp, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                         (int)linattn_jvp_smem(LINATTN_JVP_MAX_N));
    if (e != cudaSuccess) return e;
    return cudaFuncSetAttribute(k_midattn_jvp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)midattn_jvp_smem());
}

}  // namespace flo
