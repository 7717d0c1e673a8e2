// k_attn: one attention block of the U-Net in one kernel (sm_100a).
//
// Linear attention  Residual(PreNorm(dim, LinearAttention(dim)))  (unet.py:33-39,125-161):
//   input  xhat = GroupNorm(1,C)(x2)   (written by the preceding k_chain epilogue) and x2 (residual)
//   K,V = to_qkv 1x1 convs (tcgen05, N=128 each)            -> TMEM
//   P = exp(k - max_n k) (column softmax numerator, per sample and channel), V  -> 16-bit shared memory
//   ctx[(h,d)][(h,e)] = sum_n P[n][(h,d)] V[n][(h,e)]  : ONE tcgen05.mma chain per sample with BOTH operands
//        MN-major -- the blocked [C/8][pixel][8] layout is the canonical MN-major operand with K = pixels, so no
//        transposes; a column of ones appended to V yields the softmax denominators sum_n P for free
//   Q = softmax_d(q) (per pixel and head, thread-local)      -> shared memory (reuses P)
//   out[n][(h,e)] = sum_d Q[n][(h,d)] * ctx[d][e]/sum * 32^-0.5  : tcgen05.mma per (sample, head), N=32
//   y = to_out conv (tcgen05) + bias -> GroupNorm(1,C) -> + x2   -> global (normal / unshuffled / upsampled)
// Mid-block attention (unet.py:99-122), n = H*W <= 16: K,V,Q convs on tcgen05, softmax(QK^T)V per row on CUDA
// cores out of shared memory, to_out conv on tcgen05, + bias + x2.
//
// Rows: "dense" row = s*n + p for the convolutions and the final epilogue; the P/V/Q operand slots use
// s*n_pad + p (n_pad = max(n,16)) so every sample's pixel range is a whole number of K=16 slices.
#include "flo_internal.h"
#include "fused_common.cuh"

namespace flo {

struct RingA { int cc; };
__device__ __forceinline__ uint64_t desc64(uint32_t lo, uint32_t hi) {
    uint64_t d;
    asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "r"(lo), "r"(hi));
    return d;
}
constexpr int ATTN_RING = 4;       // weight ring depth of k_attn (the planner sets n_ring to it): masks, not divisions

// weight chunk g of the stage: K, V, Q projections (qkv_chunks each), then to_out (o_chunks)
__device__ __forceinline__ void attn_issue_chunk(const AttnFusedParams& p, uint32_t smem_base, uint32_t bar_full, uint32_t bar_empty,
                                                 int g, int qkv_bytes, int o_bytes) {
    const int qc = p.qkv_chunks;
    const uint16_t* w; int ci, bytes;
    if (g < qc) { w = p.wblob + p.wk_off; ci = g; bytes = qkv_bytes; }
    else if (g < 2 * qc) { w = p.wblob + p.wv_off; ci = g - qc; bytes = qkv_bytes; }
    else if (g < 3 * qc) { w = p.wblob + p.wq_off; ci = g - 2 * qc; bytes = qkv_bytes; }
    else { w = p.wblob + p.wo_off; ci = g - 3 * qc; bytes = o_bytes; }
    const int slot = g & (ATTN_RING - 1);
    if (g >= ATTN_RING) mbar_wait(bar_empty + 8 * slot, ((g / ATTN_RING) - 1) & 1);
    mbar_expect_tx(bar_full + 8 * slot, (uint32_t)bytes);
    bulk_load_1d(smem_base + p.ring_off + slot * p.ring_slot_bytes, reinterpret_cast<const uint8_t*>(w) + (size_t)ci * bytes,
                 (uint32_t)bytes, bar_full + 8 * slot);
}
// 1x1 conv over a K-major operand slot: A rows = tile t rows [128t, 128t+128), planes at `a_plane` stride.
// The weight stream holds tiles of `n_tile` output channels per K16 slice; the MMA uses the first `n` of them.
__device__ __forceinline__ void attn_conv(const AttnFusedParams& p, uint32_t smem_base, uint32_t tmem_base, uint32_t bar_full,
                                          uint32_t bar_empty, RingA& rs, uint32_t a_off, uint32_t a_plane, int n, int n_tile,
                                          int col, int n_chunks, int S) {
    const uint32_t idesc = make_idesc16(128, n, p.fmt, 0, 0);
    const int n_mtiles = p.n_mtiles;
    const uint32_t ring_off = p.ring_off, ring_slot_bytes = p.ring_slot_bytes;
    // descriptor words built once, then advanced by constant increments (address field = 14 bits of addr >> 4)
    const uint32_t hi = (128u >> 4) | (1u << 14);                                       // SBO = 128 B, descriptor version 1
    const uint32_t a_lo0 = (((smem_base + a_off) >> 4) & 0x3FFFu) | (((a_plane >> 4) & 0x3FFFu) << 16);
    const uint32_t a_step = (2u * a_plane) >> 4;                                         // two channel-block planes per K16 slice
    const uint32_t b_lbo = (((uint32_t)n_tile * 16u >> 4) & 0x3FFFu) << 16, b_step = (uint32_t)n_tile * 32u >> 4;
    for (int ci = 0; ci < n_chunks; ++ci) {
        const int slot = rs.cc & (ATTN_RING - 1);
        mbar_wait(bar_full + 8 * slot, (rs.cc / ATTN_RING) & 1);
        tc_fence_after();
        if (elect_one()) {
            uint32_t b_lo = (((smem_base + ring_off + slot * ring_slot_bytes) >> 4) & 0x3FFFu) | b_lbo;
            uint32_t a_lo = a_lo0 + (uint32_t)(ci * S) * a_step;
            for (int s = 0; s < S; ++s) {
                const uint64_t bdesc = desc64(b_lo, hi);
                const uint32_t acc = (ci * S + s) > 0 ? 1u : 0u;
                for (int t = 0; t < n_mtiles; ++t)
                    umma_bf16(tmem_base + (uint32_t)(col + t * n), desc64(a_lo + (uint32_t)t * 128u, hi), bdesc, idesc, acc);
                a_lo += a_step; b_lo += b_step;
            }
            umma_commit(bar_empty + 8 * slot);
        }
        __syncwarp();
        ++rs.cc;
    }
}

__device__ __forceinline__ void attn_write_out(const AttnFusedParams& p, int b, int px, int c16, const float* v, int fmt) {
    const int ncb = p.C >> 3;
    const int lgW = 31 - __clz(p.W);
    const int h = px >> lgW, w = px & (p.W - 1);
#pragma unroll
    for (int hb = 0; hb < 2; ++hb) {
        const int cb = (c16 >> 3) + hb;
        const uint4 u = pack8(v + hb * 8, fmt);
        if (p.out) reinterpret_cast<uint4*>(p.out)[(size_t)(cb * p.B + b) * p.n + px] = u;
        if (p.out_un) {
            const int plane = ((h & 1) * 2 + (w & 1)) * ncb + cb;
            const int q = (h >> 1) * (p.W >> 1) + (w >> 1);
            reinterpret_cast<uint4*>(p.out_un)[(size_t)(plane * p.B + b) * (p.n >> 2) + q] = u;
        }
        if (p.out_up) {
            const int W2 = p.W * 2;
            uint4* dst = reinterpret_cast<uint4*>(p.out_up) + (size_t)(cb * p.B + b) * (p.n * 4);
#pragma unroll
            for (int d = 0; d < 4; ++d) dst[(2 * h + (d >> 1)) * W2 + 2 * w + (d & 1)] = u;
        }
    }
}


// Warp-uniform variant (every lane of the warp calls it; `valid` predicates the stores).  The lanes of one image row are W
// consecutive lanes (px = row index & (n - 1), rows = TMEM lanes), so for the nearest-x2 copy each lane fetches, by shuffle, the
// blocks of the two source pixels whose copies land at output columns w and w + W: the W lanes of a row then write W * 16
// CONTIGUOUS bytes per store (whole 32-byte sectors) instead of four half-filled sectors per lane -- the scattered form ran at
// one sector per cycle and cost 9.5k cycles for the C = 128 output of the 2x2 level (profiles/r02_attn_small_timeline.txt).
__device__ __forceinline__ void attn_write_out_w(const AttnFusedParams& p, int b, int px, int c16, const float* v, bool valid, int fmt) {
    if (!p.out_up || p.W < 2) {
        if (valid) attn_write_out(p, b, px, c16, v, fmt);
        return;
    }
    const int ncb = p.C >> 3;
    const int lgW = 31 - __clz(p.W), W = p.W, W2 = 2 * W;
    const int h = px >> lgW, w = px & (W - 1);
    const int lane = (int)(threadIdx.x & 31), base = lane - w;
    const int src0 = base + (w >> 1), src1 = base + ((w + W) >> 1);
#pragma unroll
    for (int hb = 0; hb < 2; ++hb) {
        const int cb = (c16 >> 3) + hb;
        const uint4 u = pack8(v + hb * 8, fmt);
        uint4 a, c;
        a.x = __shfl_sync(0xffffffffu, u.x, src0); a.y = __shfl_sync(0xffffffffu, u.y, src0);
        a.z = __shfl_sync(0xffffffffu, u.z, src0); a.w = __shfl_sync(0xffffffffu, u.w, src0);
        c.x = __shfl_sync(0xffffffffu, u.x, src1); c.y = __shfl_sync(0xffffffffu, u.y, src1);
        c.z = __shfl_sync(0xffffffffu, u.z, src1); c.w = __shfl_sync(0xffffffffu, u.w, src1);
        if (!valid) continue;
        if (p.out) reinterpret_cast<uint4*>(p.out)[(size_t)(cb * p.B + b) * p.n + px] = u;
        if (p.out_un) {
            const int plane = ((h & 1) * 2 + (w & 1)) * ncb + cb;
            const int q = (h >> 1) * (W >> 1) + (w >> 1);
            reinterpret_cast<uint4*>(p.out_un)[(size_t)(plane * p.B + b) * (p.n >> 2) + q] = u;
        }
        uint4* dst = reinterpret_cast<uint4*>(p.out_up) + (size_t)(cb * p.B + b) * (p.n * 4) + (2 * h) * W2;
        dst[w] = a; dst[w + W] = c; dst[W2 + w] = a; dst[W2 + w + W] = c;
    }
}

// Column maximum over the lanes of a segment for 16 channels held per lane.  A butterfly would move all 16 values at
// every step (16 shuffles x log2(seg)); here every step also halves the channels a lane is responsible for, so the
// exchange costs 8 + 4 + 2 + 1 (+1) shuffles.  On return lane L holds `CNT` channels starting at channel `chan`.
template <int M>
__device__ __forceinline__ void colmax_halve(float (&v)[16], bool upper, int o) {
#pragma unroll
    for (int j = 0; j < M / 2; ++j) {
        const float send = upper ? v[j] : v[j + M / 2];
        const float keep = upper ? v[j + M / 2] : v[j];
        v[j] = fmaxf(keep, __shfl_xor_sync(0xffffffffu, send, o));
    }
}
template <int SEG>
__device__ __forceinline__ int colmax16(float (&v)[16], int lane) {
    int chan = 0;
    if (SEG == 32) {
        colmax_halve<16>(v, lane & 16, 16); chan += (lane & 16) ? 8 : 0;
        colmax_halve<8>(v, lane & 8, 8);    chan += (lane & 8) ? 4 : 0;
        colmax_halve<4>(v, lane & 4, 4);    chan += (lane & 4) ? 2 : 0;
        colmax_halve<2>(v, lane & 2, 2);    chan += (lane & 2) ? 1 : 0;
        v[0] = fmaxf(v[0], __shfl_xor_sync(0xffffffffu, v[0], 1));
    } else if (SEG == 16) {
        colmax_halve<16>(v, lane & 8, 8); chan += (lane & 8) ? 8 : 0;
        colmax_halve<8>(v, lane & 4, 4);  chan += (lane & 4) ? 4 : 0;
        colmax_halve<4>(v, lane & 2, 2);  chan += (lane & 2) ? 2 : 0;
        colmax_halve<2>(v, lane & 1, 1);  chan += (lane & 1) ? 1 : 0;
    } else {   // SEG == 4: four channels per lane remain
        colmax_halve<16>(v, lane & 2, 2); chan += (lane & 2) ? 8 : 0;
        colmax_halve<8>(v, lane & 1, 1);  chan += (lane & 1) ? 4 : 0;
    }
    return chan;
}

// NT: M tiles per CTA as a compile-time constant (1: the 8x8 level with 8 epilogue warps, 2: 16x16 with 16; 0: run time)
// NT > 0 is the LEAN instance the default plan launches (linear attention, transposed K / V projections): `full` and `ktrans` are
// compile-time there, so the mid-attention path, the row-form first epilogue and their helpers are not part of its code
// (200 KB -> the kernels are latency chains that stall on instruction fetch as much as on memory).  NT = 0 is the generic
// instance: full attention, and linear attention with the row-form projections.
// FMTK: the 16-bit operand format as a compile-time constant (0 fp16, 1 bf16; -1: run time)
template <int NT = 0, int FMTK = -1>
__global__ void __launch_bounds__(ATTN_MAX_THREADS) k_attn(const __grid_constant__ CUtensorMap tm_xh,
                                                        const __grid_constant__ AttnFusedParams p) {
    extern __shared__ __align__(128) uint8_t smem[];
    constexpr bool LEAN = NT > 0;
    const int fmt_k = FMTK >= 0 ? FMTK : p.fmt;
    const bool is_full = LEAN ? false : (p.full != 0);
    const bool is_kt = LEAN;                            // the generic instance is launched only for the row-form projections
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, tid = threadIdx.x;
    // Warp roles: [0, EW) epilogue (EW = 4 for mid attention, 8 for one M tile, 16 for two; the warp groups share the TMEM
    // lane quadrants), EW = TMA producer, EW + 1 = MMA issuer.
    const int EW = NT == 2 ? 16 : (NT == 1 ? 8 : p.epi_warps), n_epi = EW * 32, n_thr = (int)blockDim.x;
    const int n_mtiles_k = NT ? NT : p.n_mtiles;
    const bool n_ge32 = LEAN ? true : (p.n >= 32);
    const int w_prod = EW, w_mma = EW + 1;
    const uint32_t smem_base = smem_u32(smem);
    const uint32_t bar_full = smem_base + p.bar_off;
    const uint32_t bar_empty = bar_full + 8 * MAX_WSTAGES;
    const uint32_t bar_load = bar_empty + 8 * MAX_WSTAGES;
    const uint32_t bar_mma = bar_load + 8;
    const uint32_t bar_epi = bar_mma + 8;
    const uint32_t tmem_slot = bar_epi + 8;
    volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem + p.bar_off + 16 * MAX_WSTAGES + 24);
    constexpr int NCH = 128;                            // q / k / v channels: 4 heads x 32
    const int b0 = (int)blockIdx.x * p.nb;
    if (p.dbg && tid == 0 && blockIdx.x == 0) p.dbg[100] = global_ns();
    const int n = p.n, n_pad = p.n_pad, C = p.C;
    const uint32_t plane = (uint32_t)p.plane_bytes;
    const uint32_t xh_plane = (uint32_t)(p.nb * n) * 16u;
    const int lgn = 31 - __clz(n);                      // n = H*W is a power of two (planner): shifts, not divisions
    const int mtS = (n + 127) >> 7;                    // 128-row tiles per sample in the out contraction

    if (warp == w_prod && lane == 0) {
        for (int i = 0; i < p.n_ring; ++i) { mbar_init(bar_full + 8 * i, 1); mbar_init(bar_empty + 8 * i, 1); }
        mbar_init(bar_load, 1);
        mbar_init(bar_mma, 1);
        mbar_init(bar_epi, n_epi);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == w_mma) tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols);
    // The P / V / context slots must read as zero wherever no epilogue writes them: padding rows (n < 16), rows of samples past the
    // end of the batch, rows past the last sample of a partly filled M tile.  A CTA whose rows are all live skips the clear
    // (152 KB of shared-memory stores at the 16x16 level, on the critical path of every CTA that is not in the first wave):
    // every contraction runs over the rows of ONE sample, and what the unwritten planes feed are accumulator columns nobody loads.
    const bool all_live = !is_full && p.n_pad == p.n && ((p.nb * p.n) & 127) == 0 && b0 + p.nb <= p.B;
    if (!all_live)
        for (int i = tid * 16; i < p.zero_bytes; i += n_thr * 16)
            *reinterpret_cast<uint4*>(smem + p.zero_off + i) = make_uint4(0, 0, 0, 0);
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_ptr;
    long long* dbg = (blockIdx.x == 0) ? p.dbg : nullptr;
    if (dbg && tid == 0) dbg[64] = clock64();
    if (dbg && tid == 0) dbg[101] = global_ns();
    const int qkv_bytes = p.qkv_S * 128 * 32, o_bytes = p.o_S * C * 32;

    if (warp == w_prod) {
        if (lane == 0) {
            const int total = 3 * p.qkv_chunks + p.o_chunks, pre = min(ATTN_RING, total);
            for (int g = 0; g < pre; ++g) attn_issue_chunk(p, smem_base, bar_full, bar_empty, g, qkv_bytes, o_bytes);
            griddep_wait();          // weights are constants; the activations come from the previous kernel
            mbar_expect_tx(bar_load, (uint32_t)(C >> 3) * xh_plane);
            tma_load_5d(smem_base + p.xh_off, &tm_xh, bar_load, 0, 0, 0, b0, 0);
            for (int g = pre; g < total; ++g) attn_issue_chunk(p, smem_base, bar_full, bar_empty, g, qkv_bytes, o_bytes);
        }
    } else if (warp == w_mma) {
        {   // whole warp, warp-uniform; one elected lane issues the tcgen05 instructions
            RingA rs{0};
            mbar_wait(bar_load, 0);
            tc_fence_after();
            if (dbg && lane == 0) dbg[0] = clock64();
            // ---- phase 0: K and V convolutions (and Q for the mid attention)
            const bool tr = is_kt != 0;
            // transposed projection D[channel lanes][pixel columns] = W (A operand: the K-major weight tile, 128 rows x 16 B per K half)
            // x x^ (B operand: the CTA's nb * n pixel rows of the input tile, planes of 8 channels)
            auto conv_T = [&](int col) {
                const uint32_t idesc = make_idesc16(128, p.nb * n, fmt_k, 0, 0);
                for (int ci = 0; ci < p.qkv_chunks; ++ci) {
                    const int slot = rs.cc & (ATTN_RING - 1);
                    mbar_wait(bar_full + 8 * slot, (rs.cc / ATTN_RING) & 1);
                    tc_fence_after();
                    if (elect_one()) {
                        for (int sl = 0; sl < p.qkv_S; ++sl) {
                            const uint32_t a_addr = smem_base + p.ring_off + (uint32_t)slot * (uint32_t)p.ring_slot_bytes + (uint32_t)sl * 4096u;
                            const uint32_t b_addr = smem_base + p.xh_off + (uint32_t)(ci * p.qkv_S + sl) * 2u * xh_plane;
                            umma_bf16(tmem_base + (uint32_t)col, make_smem_desc(a_addr, 2048u, 128u), make_smem_desc(b_addr, xh_plane, 128u), idesc,
                                      (ci * p.qkv_S + sl) > 0 ? 1u : 0u);
                        }
                        umma_commit(bar_empty + 8 * slot);
                    }
                    __syncwarp();
                    ++rs.cc;
                }
            };
            if (tr) {
                conv_T(p.col_k);
                conv_T(p.col_v);
            } else {
            attn_conv(p, smem_base, tmem_base, bar_full, bar_empty, rs, p.xh_off, xh_plane, NCH, 128, p.col_k, p.qkv_chunks, p.qkv_S);
            attn_conv(p, smem_base, tmem_base, bar_full, bar_empty, rs, p.xh_off, xh_plane, NCH, 128, p.col_v, p.qkv_chunks, p.qkv_S);
            }
            if (is_full) attn_conv(p, smem_base, tmem_base, bar_full, bar_empty, rs, p.xh_off, xh_plane, NCH, 128, p.col_q, p.qkv_chunks, p.qkv_S);
            if (dbg && lane == 0) dbg[1] = clock64();
            if (elect_one()) umma_commit(bar_mma);
            __syncwarp();
            int ph = 0;
            if (!is_full) {
                // ---- phase 1: context per sample (both operands MN-major, K = pixels), then the Q convolution
                named_bar_sync(2, n_epi + 32); ++ph;
                tc_fence_after();
                if (dbg && lane == 0) dbg[8] = clock64();
                // M = the 128 (h, d) channel rows, N = the 128 (h, e) channels + the ones block
                const uint32_t idesc_ctx = make_idesc16(128, NCH + 16, fmt_k, 1, 1);
                {
                    const int nb = p.nb, col_ctx = p.col_ctx;
                    const uint32_t p_off = p.p_off, v_off = p.v_off;
                    if (tr) {
                        // k~ [128 channel rows][pixels] and v [144 rows: channels, then the ones row][pixels], both K-major: planes of
                        // eight pixels, 2048 / 2304 bytes each
                        const uint32_t idesc_t = make_idesc16(128, NCH + 16, fmt_k, 0, 0);
                        if (elect_one())
                            for (int s = 0; s < nb; ++s)
                                for (int ks = 0; ks < n / 16; ++ks) {
                                    const uint32_t pl = (uint32_t)(s * (n >> 3) + 2 * ks);
                                    umma_bf16(tmem_base + (uint32_t)(col_ctx + s * (NCH + 16)), make_smem_desc(smem_base + p_off + pl * 2048u, 2048u, 128u),
                                              make_smem_desc(smem_base + v_off + pl * 2304u, 2304u, 128u), idesc_t, ks > 0 ? 1u : 0u);
                                }
                    } else if (elect_one())
                        for (int s = 0; s < nb; ++s)
                            for (int ks = 0; ks < n_pad / 16; ++ks) {
                                const uint32_t roff = (uint32_t)(s * n_pad + ks * 16) * 16u;
                                umma_bf16(tmem_base + (uint32_t)(col_ctx + s * (NCH + 16)), make_smem_desc(smem_base + p_off + roff, 128u, plane),
                                          make_smem_desc(smem_base + v_off + roff, 128u, plane), idesc_ctx, ks > 0 ? 1u : 0u);
                            }
                    __syncwarp();
                }
                attn_conv(p, smem_base, tmem_base, bar_full, bar_empty, rs, p.xh_off, xh_plane, NCH, 128, p.col_q, p.qkv_chunks, p.qkv_S);
                if (dbg && lane == 0) dbg[9] = clock64();
                if (elect_one()) umma_commit(bar_mma);
                __syncwarp();
                // ---- phase 2: out[n][(h,e)] per (sample, tile, head)
                named_bar_sync(2, n_epi + 32); ++ph;
                tc_fence_after();
                if (dbg && lane == 0) dbg[16] = clock64();
                const uint32_t idesc_out = make_idesc16(128, 32, fmt_k, 0, 0);
                {
                    const int nb = p.nb, col_out = p.col_out;
                    const uint32_t p_off = p.p_off, ct_off = p.ct_off;
                    if (elect_one()) {
                        for (int s = 0; s < nb; ++s)
                            for (int t = 0; t < mtS; ++t)
                                for (int h = 0; h < 4; ++h)
                                    for (int k = 0; k < 2; ++k) {
                                        const uint32_t a_addr = smem_base + p_off + (uint32_t)(4 * h + 2 * k) * plane +
                                                                (uint32_t)(s * n_pad + t * 128) * 16u;
                                        const uint32_t b_addr = smem_base + ct_off + (uint32_t)(s * 4 + h) * 2048u + (uint32_t)k * 1024u;
                                        umma_bf16(tmem_base + (uint32_t)(col_out + (s * mtS + t) * NCH + h * 32),
                                                  make_smem_desc(a_addr, plane, 128u), make_smem_desc(b_addr, 512u, 128u), idesc_out,
                                                  k > 0 ? 1u : 0u);
                                    }
                        umma_commit(bar_mma);
                    }
                    __syncwarp();
                }
            }
            // ---- last phase: to_out convolution over the O slot
            named_bar_sync(2, n_epi + 32); ++ph;
            tc_fence_after();
            if (dbg && lane == 0) dbg[24] = clock64();
            attn_conv(p, smem_base, tmem_base, bar_full, bar_empty, rs, is_full ? p.p_off : p.v_off, plane, C, C, p.col_proj,
                      p.o_chunks, p.o_S);
            if (elect_one()) umma_commit(bar_mma);
            __syncwarp();
        }
    } else {
        const int quad = warp & 3, grp = warp >> 2;            // TMEM lane quadrant; which warp group
        const int r = quad * 32 + lane;                        // row inside an M tile == TMEM lane
        const int et = grp * 128 + r;                          // epilogue thread index
        // EW = 4 (mid attention): one warp group does everything; EW = 16 (a sample spans two M tiles): tile = grp & 1 and the two
        // groups of a tile split the q/k/v channels (cpart = grp >> 1) -- the softmax epilogues are chains of TMEM loads, shuffles
        // and MUFU ops, and four warps per scheduler hide what two cannot
        // EW = 8 (one M tile per CTA, 8x8 level, two samples): both groups work on tile 0 and split the channels the same way
        // (four warps per SM left every scheduler idle most of the time: 6 k-cycle softmax epilogues on 16 k exponentials).
        const int half = EW == 16 ? (grp & 1) : 0;
        const int t0 = half, tstep = EW == 16 ? 2 : 1;
        const int cpart = EW == 16 ? (grp >> 1) : (EW == 8 ? grp : 0), ncp = EW >= 8 ? 2 : 1;
        const int ch_lo = cpart * (NCH / ncp), ch_hi = ch_lo + NCH / ncp;      // this thread's q/k/v channels in the softmax epilogues
        const uint32_t tlane = tmem_base + ((uint32_t)(quad * 32) << 16);
        auto esync = [&]() { named_bar_sync(1, n_epi); };
        float* kmax = reinterpret_cast<float*>(smem + p.kmax_off);          // [nb][128]
        float* kpart = kmax + p.nb * 128;                                   // [n_mtiles*4][128]
        float2* rowstat = reinterpret_cast<float2*>(smem + p.stats_off);    // [n_mtiles*128]
        float2* partial = rowstat + n_mtiles_k * 128;
        float2* stat = partial + 256;
        int ph = 0;
        // to_out bias and GroupNorm affine into shared memory while the first MMAs run (they are read per channel chunk
        // in the last epilogue, where a cold global line per chunk was 1k cycles on the critical path)
        float* par = reinterpret_cast<float*>(stat + 128);                  // [3][128]: bias, gamma, beta
        for (int c = et; c < C; c += n_epi) {
            par[c] = p.fblob[p.bo_off + c];
            par[128 + c] = is_full ? 1.0f : p.fblob[p.gamma_off + c];
            par[256 + c] = is_full ? 0.0f : p.fblob[p.beta_off + c];
        }
        esync();
        griddep_wait();
        mbar_wait(bar_load, 0);
        mbar_wait(bar_mma, ph & 1); ++ph;
        tc_fence_after();
        if (dbg && r == 0) dbg[2] = clock64();
        if (!is_full) {
          if (is_kt) {
            // ================= EPI 0, transposed: tensor-memory lane = channel, columns = the CTA's pixels =================
            // A warp group owns 64 pixel columns of one sample; the softmax over pixels is a loop per thread (no shuffles), the
            // groups of a sample exchange one maximum per channel through shared memory, and k~ / v go to the operand slots K-major
            // (planes of eight pixels: a thread's eight consecutive pixels are one 16-byte row).
            const int d = r;                                  // channel (h, d') = TMEM lane
            const int col0 = grp * 64, s = col0 >> lgn, gps = n >> 6;      // this group's columns, their sample, groups per sample
            float mx = -INFINITY;
#pragma unroll
            for (int c = 0; c < 64; c += 32) {
                uint32_t ua[16], ub[16];
                tmem_ld16_issue(tlane + (uint32_t)(p.col_k + col0 + c), ua);
                tmem_ld16_issue(tlane + (uint32_t)(p.col_k + col0 + c + 16), ub);
                tmem_ld_wait();
                float m4[4] = {mx, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
                for (int j = 0; j < 16; ++j) { m4[j & 3] = fmaxf(m4[j & 3], __uint_as_float(ua[j])); m4[j & 3] = fmaxf(m4[j & 3], __uint_as_float(ub[j])); }
                mx = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));
            }
            kpart[grp * 128 + d] = mx;
            // the ones row of the V operand (row 128 of every plane; rows 129..143 feed context columns nobody loads)
            for (int pl = et; pl < (p.nb * n) >> 3; pl += n_epi) {
                const float ones[8] = {1.f, 1.f, 1.f, 1.f, 1.f, 1.f, 1.f, 1.f};
                *reinterpret_cast<uint4*>(smem + p.v_off + (uint32_t)pl * 2304u + 128u * 16u) = pack8(ones, fmt_k);
            }
            if (dbg && r == 0) dbg[3] = clock64();
            esync();
            for (int g = 0; g < gps; ++g) mx = fmaxf(mx, kpart[(s * gps + g) * 128 + d]);
#pragma unroll 2
            for (int c = 0; c < 64; c += 16) {
                uint32_t ku[16], vu[16];
                tmem_ld16_issue(tlane + (uint32_t)(p.col_k + col0 + c), ku);
                tmem_ld16_issue(tlane + (uint32_t)(p.col_v + col0 + c), vu);
                tmem_ld_wait();
                float kv[16], vv[16];
#pragma unroll
                for (int j = 0; j < 16; ++j) { kv[j] = fast_exp(__uint_as_float(ku[j]) - mx); vv[j] = __uint_as_float(vu[j]); }
                const uint32_t pl = (uint32_t)(col0 + c) >> 3;
                uint8_t* pd = smem + p.p_off + pl * 2048u + (uint32_t)d * 16u;
                uint8_t* vd = smem + p.v_off + pl * 2304u + (uint32_t)d * 16u;
                *reinterpret_cast<uint4*>(pd) = pack8(kv, fmt_k);
                *reinterpret_cast<uint4*>(pd + 2048u) = pack8(kv + 8, fmt_k);
                *reinterpret_cast<uint4*>(vd) = pack8(vv, fmt_k);
                *reinterpret_cast<uint4*>(vd + 2304u) = pack8(vv + 8, fmt_k);
            }
            if (dbg && r == 0) dbg[4] = clock64();
            fence_proxy_async();
            tc_fence_before();
            named_bar_arrive(2, n_epi + 32);
          } else {
            // ================= EPI 0: column softmax numerators of K, V to shared memory =================
            const int seg = n < 32 ? n : 32;                 // lanes per sample inside one warp
            // two 16-channel chunks per iteration: both TMEM loads are in flight together and the two shuffle
            // reductions are independent, so their latencies overlap
            for (int t = t0; t < n_mtiles_k; t += tstep) {
                const int rd = t * 128 + r, s = rd >> lgn;
                const bool valid = s < p.nb && b0 + s < p.B;
                for (int c32 = ch_lo; c32 < ch_hi; c32 += 32) {
                    uint32_t ua[16], ub[16];
                    tmem_ld16_issue(tlane + (uint32_t)(p.col_k + t * NCH + c32), ua);
                    tmem_ld16_issue(tlane + (uint32_t)(p.col_k + t * NCH + c32 + 16), ub);
                    tmem_ld_wait();
                    float va[16], vb[16];
#pragma unroll
                    for (int j = 0; j < 16; ++j) {
                        va[j] = valid ? __uint_as_float(ua[j]) : -INFINITY;
                        vb[j] = valid ? __uint_as_float(ub[j]) : -INFINITY;
                    }
                    if (seg == 32) {
                        const int ca = colmax16<32>(va, lane);
                        const int cb = colmax16<32>(vb, lane);
                        if ((lane & 1) == 0) {
                            kpart[(t * 4 + quad) * 128 + c32 + ca] = va[0];
                            kpart[(t * 4 + quad) * 128 + c32 + 16 + cb] = vb[0];
                        }
                    } else if (seg == 16) {
                        const int ca = colmax16<16>(va, lane);
                        const int cb = colmax16<16>(vb, lane);
                        if (s < p.nb) { kmax[s * 128 + c32 + ca] = va[0]; kmax[s * 128 + c32 + 16 + cb] = vb[0]; }
                    } else if (seg == 4) {
                        const int ca = colmax16<4>(va, lane);
                        const int cb = colmax16<4>(vb, lane);
                        if (s < p.nb) {
#pragma unroll
                            for (int j = 0; j < 4; ++j) { kmax[s * 128 + c32 + ca + j] = va[j]; kmax[s * 128 + c32 + 16 + cb + j] = vb[j]; }
                        }
                    } else {
                        // generic butterfly over the lanes of one sample
                        for (int o = seg >> 1; o > 0; o >>= 1) {
#pragma unroll
                            for (int j = 0; j < 16; ++j) {
                                va[j] = fmaxf(va[j], __shfl_xor_sync(0xffffffffu, va[j], o));
                                vb[j] = fmaxf(vb[j], __shfl_xor_sync(0xffffffffu, vb[j], o));
                            }
                        }
                        if ((lane & (seg - 1)) == 0 && s < p.nb) {
#pragma unroll
                            for (int j = 0; j < 16; ++j) { kmax[s * 128 + c32 + j] = va[j]; kmax[s * 128 + c32 + 16 + j] = vb[j]; }
                        }
                    }
                }
            }
            if (dbg && r == 0) dbg[3] = clock64();
            esync();
            if (n_ge32) {
                const int wps = n >> 5;                      // warp-rows per sample
                for (int idx = et; idx < p.nb * 128; idx += n_epi) {
                    const int s = idx >> 7, c = idx & 127;
                    if (c >= NCH) continue;
                    float m = -INFINITY;
                    for (int w = 0; w < wps; ++w) m = fmaxf(m, kpart[(s * wps + w) * 128 + c]);
                    kmax[idx] = m;
                }
                esync();
            }
            for (int t = t0; t < n_mtiles_k; t += tstep) {
                const int rd = t * 128 + r, s = rd >> lgn, px = rd & (n - 1);
                const bool valid = s < p.nb && b0 + s < p.B;
                const uint32_t row_off = (uint32_t)(s * n_pad + px) * 16u;
                for (int c16 = ch_lo; c16 < ch_hi; c16 += 16) {
                    uint32_t ku[16], vu[16];
                    tmem_ld16_issue(tlane + (uint32_t)(p.col_k + t * NCH + c16), ku);
                    tmem_ld16_issue(tlane + (uint32_t)(p.col_v + t * NCH + c16), vu);
                    tmem_ld_wait();
                    if (!valid) continue;
                    float kv[16], vv[16];
#pragma unroll
                    for (int j = 0; j < 16; ++j) { kv[j] = __uint_as_float(ku[j]); vv[j] = __uint_as_float(vu[j]); }
                    const float4* km4 = reinterpret_cast<const float4*>(kmax + s * 128 + c16);
#pragma unroll
                    for (int k4 = 0; k4 < 4; ++k4) {
                        const float4 m4 = km4[k4];
                        kv[4 * k4] = fast_exp(kv[4 * k4] - m4.x); kv[4 * k4 + 1] = fast_exp(kv[4 * k4 + 1] - m4.y);
                        kv[4 * k4 + 2] = fast_exp(kv[4 * k4 + 2] - m4.z); kv[4 * k4 + 3] = fast_exp(kv[4 * k4 + 3] - m4.w);
                    }
                    uint8_t* pd = smem + p.p_off + (uint32_t)(c16 >> 3) * plane + row_off;
                    uint8_t* vd = smem + p.v_off + (uint32_t)(c16 >> 3) * plane + row_off;
                    *reinterpret_cast<uint4*>(pd) = pack8(kv, fmt_k);
                    *reinterpret_cast<uint4*>(pd + plane) = pack8(kv + 8, fmt_k);
                    *reinterpret_cast<uint4*>(vd) = pack8(vv, fmt_k);
                    *reinterpret_cast<uint4*>(vd + plane) = pack8(vv + 8, fmt_k);
                }
                if (valid && cpart == 0) {
                    const float ones[8] = {1.f, 1.f, 1.f, 1.f, 1.f, 1.f, 1.f, 1.f};
                    *reinterpret_cast<uint4*>(smem + p.v_off + (uint32_t)(NCH >> 3) * plane + row_off) = pack8(ones, fmt_k);
                }
            }
            if (dbg && r == 0) dbg[4] = clock64();
            fence_proxy_async();
            tc_fence_before();
            named_bar_arrive(2, n_epi + 32);
          }
            // ================= EPI 1: context normalisation -> B operand; softmax_d(q) -> A operand =================
            mbar_wait(bar_mma, ph & 1); ++ph;
            tc_fence_after();
            if (dbg && r == 0) dbg[10] = clock64();
            {
                const int h = quad, d = lane;                // TMEM row r = (h, d)
                for (int s = t0; s < p.nb; s += tstep) {
                    uint32_t u0[16], u1[16], us[16];
                    // (with two channel groups per tile each takes 16 of the row's 32 context columns)
                    tmem_ld16_issue(tlane + (uint32_t)(p.col_ctx + s * (NCH + 16) + h * 32), u0);
                    tmem_ld16_issue(tlane + (uint32_t)(p.col_ctx + s * (NCH + 16) + h * 32 + 16), u1);
                    tmem_ld16_issue(tlane + (uint32_t)(p.col_ctx + s * (NCH + 16) + NCH), us);
                    tmem_ld_wait();
                    const int e_lo = cpart * (32 / ncp), e_hi = e_lo + 32 / ncp;
                    float c0[16], c1[16];
#pragma unroll
                    for (int j = 0; j < 16; ++j) { c0[j] = __uint_as_float(u0[j]); c1[j] = __uint_as_float(u1[j]); }
                    const float inv = 0.17677669529663687f * fast_rcp(__uint_as_float(us[0]));      // 32^-0.5 / sum_n exp(k - max)
                    uint8_t* base = smem + p.ct_off + (uint32_t)(s * 4 + h) * 2048u + (uint32_t)(d >> 3) * 512u + (uint32_t)(d & 7) * 2u;
#pragma unroll
                    for (int e = 0; e < 32; ++e) {
                        if (e < e_lo || e >= e_hi) continue;
                        const float val = (e < 16 ? c0[e] : c1[e - 16]) * inv;
                        const uint32_t u = pack2(val, 0.f, fmt_k);
                        *reinterpret_cast<uint16_t*>(base + (uint32_t)(e >> 3) * 128u + (uint32_t)(e & 7) * 16u) = (uint16_t)(u & 0xFFFFu);
                    }
                }
            }
            for (int t = t0; t < n_mtiles_k; t += tstep) {
                const int rd = t * 128 + r, s = rd >> lgn, px = rd & (n - 1);
                const bool valid = s < p.nb && b0 + s < p.B;
                const uint32_t row_off = (uint32_t)(s * n_pad + px) * 16u;
                // two heads per iteration (four TMEM loads in flight, two independent softmax chains); max and sum as
                // 4-way trees instead of 32-long dependent chains
                for (int h2 = cpart * (4 / ncp); h2 < (cpart + 1) * (4 / ncp); h2 += 2) {
                    uint32_t qu[2][32];
#pragma unroll
                    for (int k = 0; k < 2; ++k) {
                        tmem_ld16_issue(tlane + (uint32_t)(p.col_q + t * NCH + (h2 + k) * 32), *reinterpret_cast<uint32_t(*)[16]>(&qu[k][0]));
                        tmem_ld16_issue(tlane + (uint32_t)(p.col_q + t * NCH + (h2 + k) * 32 + 16), *reinterpret_cast<uint32_t(*)[16]>(&qu[k][16]));
                    }
                    tmem_ld_wait();
                    if (!valid) continue;
#pragma unroll
                    for (int k = 0; k < 2; ++k) {
                        float q[32];
#pragma unroll
                        for (int j = 0; j < 32; ++j) q[j] = __uint_as_float(qu[k][j]);
                        float m4[4] = {q[0], q[1], q[2], q[3]};
#pragma unroll
                        for (int j = 4; j < 32; ++j) m4[j & 3] = fmaxf(m4[j & 3], q[j]);
                        const float m = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));
                        float s4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                        for (int j = 0; j < 32; ++j) { q[j] = fast_exp(q[j] - m); s4[j & 3] += q[j]; }
                        const float inv = fast_rcp((s4[0] + s4[1]) + (s4[2] + s4[3]));
#pragma unroll
                        for (int j = 0; j < 32; ++j) q[j] *= inv;
                        uint8_t* qd = smem + p.p_off + (uint32_t)(4 * (h2 + k)) * plane + row_off;
#pragma unroll
                        for (int cb = 0; cb < 4; ++cb) *reinterpret_cast<uint4*>(qd + (uint32_t)cb * plane) = pack8(q + cb * 8, fmt_k);
                    }
                }
            }
            if (dbg && r == 0) dbg[11] = clock64();
            fence_proxy_async();
            tc_fence_before();
            named_bar_arrive(2, n_epi + 32);
            // ================= EPI 2: attention output -> O slot (dense rows), reuses the V slot =================
            mbar_wait(bar_mma, ph & 1); ++ph;
            tc_fence_after();
            if (dbg && r == 0) dbg[18] = clock64();
            for (int s = 0; s < p.nb; ++s)
                for (int t = (mtS > 1 ? t0 : 0); t < mtS; t += (mtS > 1 ? tstep : 1)) {
                    const int px = t * 128 + r;
                    const bool valid = px < n && b0 + s < p.B;
                    const uint32_t row_off = (uint32_t)(s * n + px) * 16u;
                    for (int c32 = ch_lo; c32 < ch_hi; c32 += 32) {
                        uint32_t ua[16], ub[16];
                        tmem_ld16_issue(tlane + (uint32_t)(p.col_out + (s * mtS + t) * NCH + c32), ua);
                        tmem_ld16_issue(tlane + (uint32_t)(p.col_out + (s * mtS + t) * NCH + c32 + 16), ub);
                        tmem_ld_wait();
                        if (!valid) continue;
                        float v[32];
#pragma unroll
                        for (int j = 0; j < 16; ++j) { v[j] = __uint_as_float(ua[j]); v[16 + j] = __uint_as_float(ub[j]); }
                        uint8_t* od = smem + p.v_off + (uint32_t)(c32 >> 3) * plane + row_off;
#pragma unroll
                        for (int k8 = 0; k8 < 4; ++k8) *reinterpret_cast<uint4*>(od + (uint32_t)k8 * plane) = pack8(v + 8 * k8, fmt_k);
                    }
                }
            fence_proxy_async();
            tc_fence_before();
            named_bar_arrive(2, n_epi + 32);
        } else {
            // ================= mid attention: softmax(q k^T) v on CUDA cores (unet.py:99-122) =================
            // A CTA owns nb = 32/n samples = 32 rows (TMEM lane quadrant 0).  Warp 0 moves K, V (16-bit) and Q (fp32)
            // from TMEM to shared memory; then thread (row = lane, head = warp) does one head of one query row.
            // Bank-conflict-free strides: K/V rows are stored key-pixel-major (index j*nb + s) with a 272-byte pitch, so the
            // 8 samples a warp reads for one key pixel j are 272 bytes apart; Q rows have a 528-byte pitch.
            constexpr uint32_t KP = 272u;
            constexpr int QP = 132;
            uint8_t* kbuf = smem + p.v_off;                    // [n][nb] rows of 128 16-bit values
            uint8_t* vbuf = kbuf + 32 * KP;
            float* qbuf = reinterpret_cast<float*>(vbuf + 32 * KP);      // [32] rows of 128 fp32
            if (warp == 0) {
                for (int c16 = 0; c16 < 128; c16 += 16) {
                    uint32_t ku[16], vu[16], qu[16];
                    tmem_ld16_issue(tlane + (uint32_t)(p.col_k + c16), ku);
                    tmem_ld16_issue(tlane + (uint32_t)(p.col_v + c16), vu);
                    tmem_ld16_issue(tlane + (uint32_t)(p.col_q + c16), qu);
                    tmem_ld_wait();
                    float kv[16], vv[16], qv[16];
#pragma unroll
                    for (int j = 0; j < 16; ++j) { kv[j] = __uint_as_float(ku[j]); vv[j] = __uint_as_float(vu[j]); qv[j] = __uint_as_float(qu[j]); }
                    const uint32_t kvrow = (uint32_t)((lane & (n - 1)) * p.nb + (lane >> lgn));
                    uint8_t* kd = kbuf + kvrow * KP + (uint32_t)c16 * 2u;
                    uint8_t* vd = vbuf + kvrow * KP + (uint32_t)c16 * 2u;
                    *reinterpret_cast<uint4*>(kd) = pack8(kv, fmt_k);
                    *reinterpret_cast<uint4*>(kd + 16) = pack8(kv + 8, fmt_k);
                    *reinterpret_cast<uint4*>(vd) = pack8(vv, fmt_k);
                    *reinterpret_cast<uint4*>(vd + 16) = pack8(vv + 8, fmt_k);
                    float4* qd = reinterpret_cast<float4*>(qbuf + lane * QP + c16);
#pragma unroll
                    for (int k4 = 0; k4 < 4; ++k4) qd[k4] = make_float4(qv[4 * k4], qv[4 * k4 + 1], qv[4 * k4 + 2], qv[4 * k4 + 3]);
                }
            }
            esync();
            {
                const int row = lane, h = warp;
                const int s = row >> lgn;
                const bool valid = b0 + s < p.B;
                float q[32];
                const float4* qs = reinterpret_cast<const float4*>(qbuf + row * QP + h * 32);
#pragma unroll
                for (int k4 = 0; k4 < 8; ++k4) {
                    const float4 t4 = qs[k4];
                    q[4 * k4] = t4.x * 0.17677669529663687f; q[4 * k4 + 1] = t4.y * 0.17677669529663687f;
                    q[4 * k4 + 2] = t4.z * 0.17677669529663687f; q[4 * k4 + 3] = t4.w * 0.17677669529663687f;
                }
                float sim[16];
                float m = -INFINITY;
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    sim[j] = -INFINITY;
                    if (j < n) {
                        const uint8_t* kr = kbuf + (uint32_t)(j * p.nb + s) * KP + (uint32_t)h * 64u;
                        float a = 0.f;
#pragma unroll
                        for (int cb = 0; cb < 4; ++cb) {
                            float kk[8];
                            unpack8(*reinterpret_cast<const uint4*>(kr + cb * 16), kk, fmt_k);
#pragma unroll
                            for (int e = 0; e < 8; ++e) a = fmaf(q[cb * 8 + e], kk[e], a);
                        }
                        sim[j] = a;
                        m = fmaxf(m, a);
                    }
                }
                float sum = 0.f;
#pragma unroll
                for (int j = 0; j < 16; ++j) { sim[j] = (j < n) ? fast_exp(sim[j] - m) : 0.f; sum += sim[j]; }
                const float inv = fast_rcp(sum);
                float o[32];
#pragma unroll
                for (int e = 0; e < 32; ++e) o[e] = 0.f;
#pragma unroll
                for (int j = 0; j < 16; ++j) {
                    if (j < n) {
                        const uint8_t* vr = vbuf + (uint32_t)(j * p.nb + s) * KP + (uint32_t)h * 64u;
                        const float a = sim[j] * inv;
#pragma unroll
                        for (int cb = 0; cb < 4; ++cb) {
                            float vv[8];
                            unpack8(*reinterpret_cast<const uint4*>(vr + cb * 16), vv, fmt_k);
#pragma unroll
                            for (int e = 0; e < 8; ++e) o[cb * 8 + e] = fmaf(a, vv[e], o[cb * 8 + e]);
                        }
                    }
                }
                if (!valid) {
#pragma unroll
                    for (int e = 0; e < 32; ++e) o[e] = 0.f;
                }
                // 'b h (x y) d -> b (h d) x y' (unet.py:121): channel = h*32 + d, as the A operand of the to_out conv
#pragma unroll
                for (int cb = 0; cb < 4; ++cb)
                    *reinterpret_cast<uint4*>(smem + p.p_off + (uint32_t)(4 * h + cb) * plane + (uint32_t)row * 16u) = pack8(o + cb * 8, fmt_k);
            }
            fence_proxy_async();
            tc_fence_before();
            named_bar_arrive(2, n_epi + 32);
        }
        if (dbg && r == 0) dbg[19] = clock64();
        // ================= last EPI: to_out bias -> GroupNorm(1,C) -> + x2 -> global =================
        // the residual rows of this thread's first tile are requested BEFORE waiting for the to_out MMAs: their L2 round trip
        // (~800 cycles) otherwise sits on the critical path between the statistics barrier and the stores
        uint4 pre_xa = make_uint4(0, 0, 0, 0), pre_xb = pre_xa;
        if (!is_full && t0 < n_mtiles_k && cpart == 0) {
            const int rd = t0 * 128 + r, s = rd >> lgn, px = rd & (n - 1);
            if (s < p.nb && b0 + s < p.B) {
                const uint4* xsrc = reinterpret_cast<const uint4*>(p.x2);
                pre_xa = xsrc[(size_t)(0 * p.B + b0 + s) * n + px];
                pre_xb = xsrc[(size_t)(1 * p.B + b0 + s) * n + px];
            }
        }
        mbar_wait(bar_mma, ph & 1); ++ph;
        tc_fence_after();
        if (dbg && r == 0) dbg[26] = clock64();
        griddep_launch();            // PDL: the next stage kernel may become resident during the last epilogue
        const float* bias = par;
        if (!is_full) {
            // (the C output channels are not split: with 16 epilogue warps the second channel group only keeps the barriers)
            for (int t = t0; t < n_mtiles_k && cpart == 0; t += tstep) {
                const int rd = t * 128 + r, s = rd >> lgn;
                const bool valid = s < p.nb && b0 + s < p.B;
                float sx = 0.f, sq = 0.f;
                float sx2 = 0.f, sq2 = 0.f;
                for (int c16 = 0; c16 < C; c16 += 32) {
                    uint32_t ua[16], ub[16];
                    const bool two = c16 + 16 < C;
                    tmem_ld16_issue(tlane + (uint32_t)(p.col_proj + t * C + c16), ua);
                    if (two) tmem_ld16_issue(tlane + (uint32_t)(p.col_proj + t * C + c16 + 16), ub);
                    tmem_ld_wait();
#pragma unroll
                    for (int j = 0; j < 16; ++j) { const float x = __uint_as_float(ua[j]) + bias[c16 + j]; sx += x; sq += x * x; }
                    if (two) {
#pragma unroll
                        for (int j = 0; j < 16; ++j) { const float x = __uint_as_float(ub[j]) + bias[c16 + 16 + j]; sx2 += x; sq2 += x * x; }
                    }
                }
                sx += sx2; sq += sq2;
                if (n_ge32) {
                    // a warp's 32 rows lie in one sample: reduce with shuffles, one partial per 32-row block, ONE barrier;
                    // every thread then adds its sample's n/32 block sums itself (fixed order: deterministic)
                    if (!valid) { sx = 0.f; sq = 0.f; }
                    for (int o = 16; o > 0; o >>= 1) { sx += __shfl_xor_sync(0xffffffffu, sx, o); sq += __shfl_xor_sync(0xffffffffu, sq, o); }
                    if (lane == 0) partial[rd >> 5] = make_float2(sx, sq);
                } else {
                    rowstat[rd] = valid ? make_float2(sx, sq) : make_float2(0.f, 0.f);
                }
            }
            // per-sample totals in a fixed order (deterministic)
            int parts = 1;
            while (parts * 2 * p.nb <= 128 && parts < 16) parts *= 2;
            if (dbg && et == 0) dbg[27] = clock64();
            esync();
            if (dbg && et == 0) dbg[28] = clock64();
            if (n_ge32) {
                // one thread per sample adds the n / 32 block sums (fixed order) and publishes mean / rstd; a second barrier is cheaper
                // than the same eight loads, sixteen adds, rcp and rsqrt in every thread on the tail of the kernel
                if (et < p.nb) {
                    const int bps = n >> 5;
                    float tx = 0.f, tq = 0.f;
#pragma unroll
                    for (int k = 0; k < 8; ++k)
                        if (k < bps) { const float2 a = partial[et * bps + k]; tx += a.x; tq += a.y; }
                    const float icnt = fast_rcp((float)(C * n));
                    const float mean = tx * icnt;
                    stat[et] = make_float2(mean, rsqrtf(fmaxf(tq * icnt - mean * mean, 0.f) + 1e-5f));
                }
                esync();
            } else {
            if (et < p.nb * parts) {
                const int lgp = 31 - __clz(parts);
                const int part = et & (parts - 1), s = et >> lgp;
                const int per = (n + parts - 1) >> lgp;
                const int a = s * n + part * per, bnd = min((s + 1) * n, a + per);
                float sx = 0.f, sq = 0.f;
                for (int k = a; k < bnd; ++k) { sx += rowstat[k].x; sq += rowstat[k].y; }
                partial[et] = make_float2(sx, sq);
            }
            esync();
            if (et < p.nb) {
                float sx = 0.f, sq = 0.f;
                for (int k = 0; k < parts; ++k) { sx += partial[et * parts + k].x; sq += partial[et * parts + k].y; }
                const float icnt = fast_rcp((float)(C * n));
                const float mean = sx * icnt;
                const float var = fmaxf(sq * icnt - mean * mean, 0.f);
                stat[et] = make_float2(mean, rsqrtf(var + 1e-5f));
            }
            esync();
            }
        }
        const float* gamma = par + 128;
        const float* beta = par + 256;
        if (is_full) {
            // 32 valid rows (TMEM quadrant 0): warp 0 moves the projection to shared memory, then every warp finishes a
            // quarter of the channels: + bias + x (unet.py:122, Residual)
            constexpr int QP = 132;
            float* ybuf = reinterpret_cast<float*>(smem + p.v_off);          // the K/V/Q staging is dead by now
            if (warp == 0) {
                for (int c16 = 0; c16 < C; c16 += 16) {
                    float v[16];
                    tmem_ld16(tlane + (uint32_t)(p.col_proj + c16), v);
                    float4* yd = reinterpret_cast<float4*>(ybuf + lane * QP + c16);
#pragma unroll
                    for (int k4 = 0; k4 < 4; ++k4) yd[k4] = make_float4(v[4 * k4], v[4 * k4 + 1], v[4 * k4 + 2], v[4 * k4 + 3]);
                }
            }
            esync();
            const int row = lane, s = row >> lgn, px = row & (n - 1), b = b0 + s;
            if (b < p.B) {
                const uint4* xsrc = reinterpret_cast<const uint4*>(p.x2);
                for (int c16 = warp * 16; c16 < C; c16 += 64) {              // 16-channel chunks round-robin over the warps
                    const uint4 xa = xsrc[(size_t)((c16 >> 3) * p.B + b) * n + px];
                    const uint4 xb = xsrc[(size_t)(((c16 >> 3) + 1) * p.B + b) * n + px];
                    float v[16], x2[16];
                    const float4* ys = reinterpret_cast<const float4*>(ybuf + row * QP + c16);
#pragma unroll
                    for (int k4 = 0; k4 < 4; ++k4) { const float4 t4 = ys[k4]; v[4 * k4] = t4.x; v[4 * k4 + 1] = t4.y; v[4 * k4 + 2] = t4.z; v[4 * k4 + 3] = t4.w; }
                    unpack8(xa, x2, fmt_k);
                    unpack8(xb, x2 + 8, fmt_k);
#pragma unroll
                    for (int j = 0; j < 16; ++j) v[j] = v[j] + bias[c16 + j] + x2[j];
                    attn_write_out(p, b, px, c16, v, fmt_k);
                }
            }
        } else {
            for (int t = t0; t < n_mtiles_k && cpart == 0; t += tstep) {
                const int rd = t * 128 + r, s = rd >> lgn, px = rd & (n - 1);
                const bool valid = s < p.nb && b0 + s < p.B;
                const int b = b0 + s;
                float2 ms = make_float2(0.f, 1.f);
                if (s < p.nb) ms = stat[s];
                if (dbg && et == 0) dbg[30] = clock64();
                const uint4* xsrc = reinterpret_cast<const uint4*>(p.x2);
                // the residual rows of the NEXT channel chunk are requested before this chunk is processed
                uint4 xa = pre_xa, xb = pre_xb;
                if (valid && t != t0) { xa = xsrc[(size_t)(0 * p.B + b) * n + px]; xb = xsrc[(size_t)(1 * p.B + b) * n + px]; }
                for (int c16 = 0; c16 < C; c16 += 16) {
                    uint4 na = make_uint4(0, 0, 0, 0), nb4 = na;
                    if (valid && c16 + 16 < C) {
                        na = xsrc[(size_t)(((c16 >> 3) + 2) * p.B + b) * n + px];
                        nb4 = xsrc[(size_t)(((c16 >> 3) + 3) * p.B + b) * n + px];
                    }
                    float v[16], x2[16];
                    tmem_ld16(tlane + (uint32_t)(p.col_proj + t * C + c16), v);
                    if (valid) {
                        unpack8(xa, x2, fmt_k);
                        unpack8(xb, x2 + 8, fmt_k);
#pragma unroll
                        for (int j = 0; j < 16; ++j) {
                            const float y = (v[j] + bias[c16 + j] - ms.x) * ms.y * gamma[c16 + j] + beta[c16 + j];
                            v[j] = y + x2[j];
                        }
                    }
                    attn_write_out_w(p, b, px, c16, v, valid, fmt_k);
                    xa = na; xb = nb4;
                }
            }
        }
        if (dbg && et == 0) dbg[29] = clock64();
    }
    tc_fence_before();
    __syncthreads();
    if (dbg && tid == 0) dbg[65] = clock64();
    if (p.dbg && tid == 0) { if (blockIdx.x == 0) p.dbg[102] = global_ns(); atomicMax(reinterpret_cast<unsigned long long*>(p.dbg + 103), (unsigned long long)global_ns()); }
    if (warp == w_mma) tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
}

// ------------------------------------------------------------------------------------------------------------------
// k_attn_small: the attention blocks of the 4x4 and 2x2 levels (n = H*W = 16 or 4 pixels per sample), linear
// (unet.py:125-150) and full (unet.py:99-122).  A sample's n x n interaction is tiny, so only the four 1x1 projections run on
// the tensor cores and a CTA owns 128 / n SAMPLES (128 dense rows: the M tile is full):
//   MMA   K, V, Q = to_qkv 1x1 convs (N = 128 each)                                        -> TMEM [0, 384)
//   EPI-A row r, channel half: k~ = softmax_n(k) (segmented halving shuffles over the n lanes of a sample) and V -> 16-bit
//         shared-memory rows                                                                  (linear; full: raw k, v)
//   EPI-B row r = (sample s, pixel i), two heads per thread, on CUDA cores out of shared memory:
//         linear: q~ = softmax_d(q) * 32^-.5;  S[m] = sum_d q~[d] k~[m][d];  out[e] = sum_m S[m] v[m][e]
//                 (== sum_d ctx[d][e] q~[d] with ctx = k~ v^T: the same contraction, reassociated)
//         full:   S[m] = sum_d 32^-.5 q[d] k[m][d];  softmax_m;  out[e] = sum_m S[m] v[m][e]
//         out -> 16-bit K-major operand slot
//   MMA   to_out 1x1 conv                                                                      -> TMEM [384, 384 + C)
//   EPI-C + bias [-> GroupNorm(1, C) per sample] + x2 -> global (normal / unshuffled / upsampled)
// Two MMA phases instead of four, no context / output MMAs, and 8x (n = 16) / 16x (n = 4) fewer CTAs than two samples per CTA.
// ------------------------------------------------------------------------------------------------------------------
constexpr uint32_t SM_KP = 528u;          // row pitch of the fp32 k~ / v staging (128 floats + 16 bytes: conflict-free rows)
constexpr int SMALL_EW = 16;              // epilogue warps of k_attn_small: one (row, head) task per thread in the attention core
constexpr int SMALL_THREADS = (SMALL_EW + 2) * 32;
template <int SEG, bool IS_MAX>
__device__ __forceinline__ int segred16(float (&v)[16], int lane) {
    // reduction over the SEG lanes of a segment for 16 values per lane; every level also halves the values a lane keeps
    // (colmax16's pattern).  Returns the first channel this lane ends up owning; it owns 16 / SEG... see callers.
    int chan = 0;
    auto halve = [&](int m, bool upper, int o) {
#pragma unroll
        for (int j = 0; j < 8; ++j) {
            if (j < m / 2) {
                const float send = upper ? v[j] : v[j + m / 2];
                const float keep = upper ? v[j + m / 2] : v[j];
                const float got = __shfl_xor_sync(0xffffffffu, send, o);
                v[j] = IS_MAX ? fmaxf(keep, got) : keep + got;
            }
        }
    };
    if (SEG == 16) {
        halve(16, lane & 8, 8); chan += (lane & 8) ? 8 : 0;
        halve(8, lane & 4, 4);  chan += (lane & 4) ? 4 : 0;
        halve(4, lane & 2, 2);  chan += (lane & 2) ? 2 : 0;
        halve(2, lane & 1, 1);  chan += (lane & 1) ? 1 : 0;
    } else {   // SEG == 4: four channels per lane remain
        halve(16, lane & 2, 2); chan += (lane & 2) ? 8 : 0;
        halve(8, lane & 1, 1);  chan += (lane & 1) ? 4 : 0;
    }
    return chan;
}

// QT: the quarter-tile instance (32 live rows, small-batch plan) -- `quarter` is a compile-time constant there and the full-tile
// forms of the first epilogue and of the attention core are not part of its code (and vice versa)
template <int NPX, bool LINEAR, bool QT = false>
__global__ void __launch_bounds__(SMALL_THREADS, 1) k_attn_small(const __grid_constant__ CUtensorMap tm_xh,
                                                                   const __grid_constant__ AttnFusedParams p) {
    extern __shared__ __align__(128) uint8_t smem[];
    constexpr int LGN = NPX == 16 ? 4 : 2;
    constexpr int SPW = 32 / NPX;                      // samples per warp
    constexpr int CNT = 16 / NPX;                      // channels a lane owns after a segmented reduction of 16 (1 or 4)
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, tid = threadIdx.x;
    constexpr int EW = SMALL_EW, n_epi = EW * 32, w_prod = EW, w_mma = EW + 1;
    const uint32_t smem_base = smem_u32(smem);
    const uint32_t bar_full = smem_base + p.bar_off;
    const uint32_t bar_empty = bar_full + 8 * MAX_WSTAGES;
    const uint32_t bar_load = bar_empty + 8 * MAX_WSTAGES;
    const uint32_t bar_mma = bar_load + 8;
    const uint32_t tmem_slot = bar_mma + 16;
    volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem + p.bar_off + 16 * MAX_WSTAGES + 24);
    const int b0 = (int)blockIdx.x * p.nb;
    const int C = p.C;
    const uint32_t plane = 2048u;                      // 128 rows x 16 bytes (operand slot of the attention output)
    // Small batches run FEWER samples per CTA than the 128 / NPX that fill the M tile (planner): the kernel is a latency chain
    // whose CUDA-core core, staging traffic and global stores are per-SM throughput, so half-empty tiles on four times the SMs
    // finish sooner.  The input tile is then nb * NPX rows per plane; accumulator rows past it are junk that nobody reads.
    const uint32_t in_plane = (uint32_t)(p.nb * NPX) * 16u;
    const int live_rows = p.nb * NPX;
    long long* dbg = (blockIdx.x == 0) ? p.dbg : nullptr;
    if (dbg && tid == 0) dbg[100] = global_ns();
    if (warp == w_prod && lane == 0) {
        for (int i = 0; i < p.n_ring; ++i) { mbar_init(bar_full + 8 * i, 1); mbar_init(bar_empty + 8 * i, 1); }
        mbar_init(bar_load, 1);
        mbar_init(bar_mma, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == w_mma) tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols);
    fence_proxy_async();
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_ptr;
    const int qkv_bytes = p.qkv_S * 128 * 32, o_bytes = p.o_S * C * 32;
    if (dbg && tid == 0) { dbg[64] = clock64(); dbg[101] = global_ns(); }

    // All weights are resident (no ring): the k / v / q streams (C/16 K16 slices x 4 KB each) land in the k~ / v staging area,
    // which is dead until the projections have completed, the to_out stream in its own 32 KB; four bulk copies from four lanes
    // at kernel start, i.e. under the previous kernel's tail (programmatic launch).  Streaming them through an 8 KB ring ran
    // at ~13 B/clk AFTER the input tile had arrived: 7.4k of a 22k-cycle kernel at C = 128 (profiles/r02_attn_small_timeline.txt).
    const uint32_t qkv_stream = (uint32_t)(p.qkv_chunks * qkv_bytes), o_stream = (uint32_t)(p.o_chunks * o_bytes);
    const uint32_t wk_smem = smem_base + p.p_off, wv_smem = wk_smem + qkv_stream, wq_smem = wv_smem + qkv_stream;
    const uint32_t wo_smem = smem_base + p.ring_off;
    if (warp == w_prod) {
        if (lane < 4) {
            const uint16_t* src = lane == 0 ? p.wblob + p.wk_off : lane == 1 ? p.wblob + p.wv_off : lane == 2 ? p.wblob + p.wq_off : p.wblob + p.wo_off;
            const uint32_t dst = lane == 0 ? wk_smem : lane == 1 ? wv_smem : lane == 2 ? wq_smem : wo_smem;
            const uint32_t bytes = lane == 3 ? o_stream : qkv_stream;
            mbar_expect_tx(bar_full + 8 * lane, bytes);
            bulk_load_1d(dst, reinterpret_cast<const uint8_t*>(src), bytes, bar_full + 8 * lane);
        }
        griddep_wait();              // weights are constants; the activations come from the previous kernel
        if (lane == 0) {
            mbar_expect_tx(bar_load, (uint32_t)(C >> 3) * in_plane);
            tma_load_5d(smem_base + p.xh_off, &tm_xh, bar_load, 0, 0, 0, b0, 0);
        }
    } else if (warp == w_mma) {
        // 1x1 conv over the K-major operand slot at xh_off (128 rows, planes of 2 KB) with a resident weight stream
        auto conv = [&](uint32_t w_smem, uint32_t bar, int n, int slices, int col, uint32_t a_plane) {
            const uint32_t idesc = make_idesc16(128, n, p.fmt, 0, 0);
            const uint32_t hi = (128u >> 4) | (1u << 14);
            uint32_t a_lo = (((smem_base + p.xh_off) >> 4) & 0x3FFFu) | (((a_plane >> 4) & 0x3FFFu) << 16);
            uint32_t b_lo = ((w_smem >> 4) & 0x3FFFu) | ((((uint32_t)n * 16u >> 4) & 0x3FFFu) << 16);
            const uint32_t a_step = (2u * a_plane) >> 4, b_step = (uint32_t)n * 32u >> 4;
            mbar_wait(bar, 0);
            tc_fence_after();
            if (elect_one()) {
                for (int sl = 0; sl < slices; ++sl) {
                    umma_bf16(tmem_base + (uint32_t)col, desc64(a_lo, hi), desc64(b_lo, hi), idesc, sl > 0 ? 1u : 0u);
                    a_lo += a_step; b_lo += b_step;
                }
            }
            __syncwarp();
        };
        mbar_wait(bar_load, 0);
        tc_fence_after();
        if (dbg && lane == 0) dbg[0] = clock64();
        conv(wk_smem, bar_full, 128, C >> 4, p.col_k, in_plane);
        conv(wv_smem, bar_full + 8, 128, C >> 4, p.col_v, in_plane);
        conv(wq_smem, bar_full + 16, 128, C >> 4, p.col_q, in_plane);
        if (dbg && lane == 0) dbg[1] = clock64();
        if (elect_one()) umma_commit(bar_mma);
        __syncwarp();
        named_bar_sync(2, n_epi + 32);       // the attention output is in the operand slot (which reuses the input tile: every
        tc_fence_after();                    // projection that read it has completed, the epilogue waited for bar_mma)
        if (dbg && lane == 0) dbg[24] = clock64();
        conv(wo_smem, bar_full + 24, C, 8, p.col_proj, plane);
        if (dbg && lane == 0) dbg[25] = clock64();
        if (elect_one()) umma_commit(bar_mma);
        __syncwarp();
    } else {
        const int quad = warp & 3, part = warp >> 2;           // TMEM lane quadrant; which quarter of the channels / which head
        const int r = quad * 32 + lane;                        // dense row = s * NPX + pixel == TMEM lane
        const int et = tid;
        const int s_loc = r >> LGN, px = r & (NPX - 1);        // sample within the CTA, pixel
        const int b = b0 + s_loc;
        const bool wact = quad * 32 < live_rows;               // warp-uniform: this warp's rows hold samples
        const bool valid = r < live_rows && b < p.B;
        const uint32_t tlane = tmem_base + ((uint32_t)(quad * 32) << 16);
        auto esync = [&]() { named_bar_sync(1, n_epi); };
        uint8_t* kst = smem + p.p_off;                         // k~ (linear) / k (full): [128 rows][SM_KP]
        uint8_t* vst = smem + p.v_off;
        // 16-byte column swizzle of the staging rows: EPI-B reads ONE row per sample at a time (the lanes of a sample broadcast),
        // and the rows of the 32 / NPX samples of a warp are NPX * 528 bytes apart = the same banks (2112 = 64 mod 128 at NPX = 4,
        // 8448 = 0 at NPX = 16: a 4- / 2-way conflict on every load).  XOR-ing the float4 index with a per-sample code (NPX = 4:
        // bits 1-2 of the sample index -- odd / even samples already sit 64 bytes apart; NPX = 16: bit 0) puts the samples of a
        // warp in distinct 16-byte bank groups; the row writes of EPI-A stay conflict-free (four wavefronts per 512-byte store).
        const uint32_t swz = NPX == 4 ? (uint32_t)((s_loc >> 1) & 3) : (uint32_t)(s_loc & 1);
        float* scr = reinterpret_cast<float*>(smem + p.kmax_off) + warp * (2 * SPW * 16);      // per warp: max[SPW][16], sum[SPW][16]
        float2* hstat = reinterpret_cast<float2*>(smem + p.stats_off);                          // [4 channel groups][32]: per-sample partial statistics of the last epilogue
        float* par = reinterpret_cast<float*>(hstat + 2 * 64);                                  // [3][128]: bias, gamma, beta
        for (int c = et; c < C; c += n_epi) {
            par[c] = p.fblob[p.bo_off + c];
            par[128 + c] = LINEAR ? p.fblob[p.gamma_off + c] : 1.0f;
            par[256 + c] = LINEAR ? p.fblob[p.beta_off + c] : 0.0f;
        }
        griddep_wait();
        if (dbg && et == 0) dbg[5] = clock64();
        // the residual rows are requested now: an exposed L2 round trip in the last epilogue otherwise
        const uint4* xsrc = reinterpret_cast<const uint4*>(p.x2);
        mbar_wait(bar_load, 0);
        if (dbg && et == 0) dbg[6] = clock64();
        mbar_wait(bar_mma, 0);
        tc_fence_after();
        if (dbg && et == 0) dbg[2] = clock64();
        // ================= EPI-A: this thread's 32 channels of row r: k (column softmax over the sample's pixels) and v =================
        // Both 16-channel chunks go through the segmented reductions together (independent shuffle chains in flight; the second
        // chunk's scratch rows live in the input tile, which is dead once the projections have completed).
        // quarter tile (32 live rows): twelve of the sixteen warps own no rows.  The four that do only MOVE k and v to the staging rows
        // and then turn to q; the column softmax of k runs out of shared memory on the others meanwhile (see below)
        const bool quarter = QT;
        const bool qsm = quarter && LINEAR;
        if (wact) {
            const int cA = part * 32;
            float kv[2][16];
            {
                uint32_t ku[2][16];
                tmem_ld16_issue(tlane + (uint32_t)(p.col_k + cA), ku[0]);
                tmem_ld16_issue(tlane + (uint32_t)(p.col_k + cA + 16), ku[1]);
                tmem_ld_wait();
#pragma unroll
                for (int h2 = 0; h2 < 2; ++h2)
#pragma unroll
                    for (int j = 0; j < 16; ++j) kv[h2][j] = __uint_as_float(ku[h2][j]);
            }
            if (LINEAR && !qsm) {
                float* const scr2[2] = {scr, reinterpret_cast<float*>(smem + p.xh_off) + warp * (2 * SPW * 16)};
                float red[2][16];
                int ch[2];
#pragma unroll
                for (int h2 = 0; h2 < 2; ++h2) {
#pragma unroll
                    for (int j = 0; j < 16; ++j) red[h2][j] = kv[h2][j];
                    ch[h2] = segred16<NPX, true>(red[h2], lane);
                    float* mx = scr2[h2] + (lane >> LGN) * 16;
#pragma unroll
                    for (int j = 0; j < CNT; ++j) mx[ch[h2] + j] = red[h2][j];
                }
                __syncwarp();
#pragma unroll
                for (int h2 = 0; h2 < 2; ++h2) {
                    const float4* mx = reinterpret_cast<const float4*>(scr2[h2] + (lane >> LGN) * 16);
#pragma unroll
                    for (int k4 = 0; k4 < 4; ++k4) {
                        const float4 m4 = mx[k4];
                        kv[h2][4 * k4] = fast_exp(kv[h2][4 * k4] - m4.x); kv[h2][4 * k4 + 1] = fast_exp(kv[h2][4 * k4 + 1] - m4.y);
                        kv[h2][4 * k4 + 2] = fast_exp(kv[h2][4 * k4 + 2] - m4.z); kv[h2][4 * k4 + 3] = fast_exp(kv[h2][4 * k4 + 3] - m4.w);
                    }
#pragma unroll
                    for (int j = 0; j < 16; ++j) red[h2][j] = kv[h2][j];
                    ch[h2] = segred16<NPX, false>(red[h2], lane);
                    float* sm = scr2[h2] + SPW * 16 + (lane >> LGN) * 16;
#pragma unroll
                    for (int j = 0; j < CNT; ++j) sm[ch[h2] + j] = red[h2][j];
                }
                __syncwarp();
#pragma unroll
                for (int h2 = 0; h2 < 2; ++h2) {
                    const float4* sm = reinterpret_cast<const float4*>(scr2[h2] + SPW * 16 + (lane >> LGN) * 16);
#pragma unroll
                    for (int k4 = 0; k4 < 4; ++k4) {
                        const float4 s4 = sm[k4];
                        kv[h2][4 * k4] *= fast_rcp(s4.x); kv[h2][4 * k4 + 1] *= fast_rcp(s4.y);
                        kv[h2][4 * k4 + 2] *= fast_rcp(s4.z); kv[h2][4 * k4 + 3] *= fast_rcp(s4.w);
                    }
                }
            }
            float4* kd = reinterpret_cast<float4*>(kst + (uint32_t)r * SM_KP);
            float4* vd = reinterpret_cast<float4*>(vst + (uint32_t)r * SM_KP);
#pragma unroll
            for (int h2 = 0; h2 < 2; ++h2)
#pragma unroll
                for (int k4 = 0; k4 < 4; ++k4)
                    kd[(uint32_t)(((cA + 16 * h2) >> 2) + k4) ^ swz] =
                        make_float4(kv[h2][4 * k4], kv[h2][4 * k4 + 1], kv[h2][4 * k4 + 2], kv[h2][4 * k4 + 3]);
            {
                uint32_t vu[2][16];
                tmem_ld16_issue(tlane + (uint32_t)(p.col_v + cA), vu[0]);
                tmem_ld16_issue(tlane + (uint32_t)(p.col_v + cA + 16), vu[1]);
                tmem_ld_wait();
#pragma unroll
                for (int h2 = 0; h2 < 2; ++h2)
#pragma unroll
                    for (int k4 = 0; k4 < 4; ++k4)
                        vd[(uint32_t)(((cA + 16 * h2) >> 2) + k4) ^ swz] =
                            make_float4(__uint_as_float(vu[h2][4 * k4]), __uint_as_float(vu[h2][4 * k4 + 1]),
                                        __uint_as_float(vu[h2][4 * k4 + 2]), __uint_as_float(vu[h2][4 * k4 + 3]));
            }
        }
        // q of (row r, head `part`) out of tensor memory: softmax over the 32 head channels, then * 32^-0.5 (unet.py:141-143), or
        // q * scale for the mid attention (unet.py:113)
        auto load_q = [&](float (&q)[32]) {
            uint32_t qa[16], qb[16];
            tmem_ld16_issue(tlane + (uint32_t)(p.col_q + part * 32), qa);
            tmem_ld16_issue(tlane + (uint32_t)(p.col_q + part * 32 + 16), qb);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 16; ++j) { q[j] = __uint_as_float(qa[j]); q[16 + j] = __uint_as_float(qb[j]); }
            if (LINEAR) {
                float m4[4] = {q[0], q[1], q[2], q[3]};
#pragma unroll
                for (int j = 4; j < 32; ++j) m4[j & 3] = fmaxf(m4[j & 3], q[j]);
                const float m = fmaxf(fmaxf(m4[0], m4[1]), fmaxf(m4[2], m4[3]));
                float s4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
                for (int j = 0; j < 32; ++j) { q[j] = fast_exp(q[j] - m); s4[j & 3] += q[j]; }
                const float inv = 0.17677669529663687f * fast_rcp((s4[0] + s4[1]) + (s4[2] + s4[3]));
#pragma unroll
                for (int j = 0; j < 32; ++j) q[j] *= inv;
            } else {
#pragma unroll
                for (int j = 0; j < 32; ++j) q[j] *= 0.17677669529663687f;
            }
        };
        // Quarter tile (32 live rows, the small-batch plan): twelve of the sixteen epilogue warps have no rows, and the attention
        // core of one (row, head) per thread is a serial chain of 64 (2x2) / 256 (4x4) 16-byte shared-memory loads that the register
        // budget keeps from overlapping (9k cycles at 4x4 with ONE warp per scheduler).  There the q~ rows go through shared memory
        // too (staging rows 32.., free in this mode) and FOUR threads share a (row, head): each takes a quarter of the key pixels
        // for S = q~ . k~, the four exchange S by shuffles, and each produces 8 of the head's 32 output channels.
        uint8_t* qst = kst + 32u * SM_KP;
        if (qsm) esync();                                       // the raw k rows are in the staging area
        if (quarter && wact) {
            float q[32];
            load_q(q);
            float4* qd = reinterpret_cast<float4*>(qst + (uint32_t)r * SM_KP);
#pragma unroll
            for (int k4 = 0; k4 < 8; ++k4)
                qd[(uint32_t)(part * 8 + k4) ^ swz] = make_float4(q[4 * k4], q[4 * k4 + 1], q[4 * k4 + 2], q[4 * k4 + 3]);
        } else if (qsm) {
            // k~ = softmax over the sample's pixels, in place: thread (sample s, float4 column f, row quarter rq) of the first 256
            // threads of the row-less warps.  The rows a thread takes and the order of the additions reproduce the halving
            // exchange of the full-tile path -- pixel i pairs with i ^ (NPX/2), then i ^ (NPX/4), ... -- so k~ is bit-identical
            // whichever plan runs: a thread owns pixels {rq, rq ^ 8, rq ^ 4, rq ^ 12} (NPX = 16; the xor-2 and xor-1 levels are two
            // shuffles over the four rq lanes) or {0, 2, 1, 3} (NPX = 4).
            constexpr int RQ = NPX / 4;
            const int u = ((warp >> 2) * 3 + (warp & 3) - 1) * 32 + lane;          // dense index over the twelve row-less warps
            if (u < 256) {
                const int rq = u % RQ, f = (u / RQ) & 31, s2 = u / (RQ * 32);
                const uint32_t sw = NPX == 4 ? (uint32_t)((s2 >> 1) & 3) : (uint32_t)(s2 & 1);
                const uint32_t col = ((uint32_t)f ^ sw) * 16u;
                const int px[4] = {rq, rq ^ (NPX / 2), rq ^ (NPX / 4), rq ^ (NPX / 2) ^ (NPX / 4)};
                float4* rows[4];
                float4 x[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    rows[k] = reinterpret_cast<float4*>(kst + (uint32_t)(s2 * NPX + px[k]) * SM_KP + col);
                    x[k] = *rows[k];
                }
                float4 m = make_float4(fmaxf(fmaxf(x[0].x, x[1].x), fmaxf(x[2].x, x[3].x)), fmaxf(fmaxf(x[0].y, x[1].y), fmaxf(x[2].y, x[3].y)),
                                       fmaxf(fmaxf(x[0].z, x[1].z), fmaxf(x[2].z, x[3].z)), fmaxf(fmaxf(x[0].w, x[1].w), fmaxf(x[2].w, x[3].w)));
#pragma unroll
                for (int o = RQ >> 1; o > 0; o >>= 1) {
                    m.x = fmaxf(m.x, __shfl_xor_sync(0xffffffffu, m.x, o)); m.y = fmaxf(m.y, __shfl_xor_sync(0xffffffffu, m.y, o));
                    m.z = fmaxf(m.z, __shfl_xor_sync(0xffffffffu, m.z, o)); m.w = fmaxf(m.w, __shfl_xor_sync(0xffffffffu, m.w, o));
                }
#pragma unroll
                for (int k = 0; k < 4; ++k) {
                    x[k].x = fast_exp(x[k].x - m.x); x[k].y = fast_exp(x[k].y - m.y); x[k].z = fast_exp(x[k].z - m.z); x[k].w = fast_exp(x[k].w - m.w);
                }
                float4 sum = make_float4((x[0].x + x[1].x) + (x[2].x + x[3].x), (x[0].y + x[1].y) + (x[2].y + x[3].y),
                                         (x[0].z + x[1].z) + (x[2].z + x[3].z), (x[0].w + x[1].w) + (x[2].w + x[3].w));
#pragma unroll
                for (int o = RQ >> 1; o > 0; o >>= 1) {
                    sum.x += __shfl_xor_sync(0xffffffffu, sum.x, o); sum.y += __shfl_xor_sync(0xffffffffu, sum.y, o);
                    sum.z += __shfl_xor_sync(0xffffffffu, sum.z, o); sum.w += __shfl_xor_sync(0xffffffffu, sum.w, o);
                }
                const float4 inv = make_float4(fast_rcp(sum.x), fast_rcp(sum.y), fast_rcp(sum.z), fast_rcp(sum.w));
#pragma unroll
                for (int k = 0; k < 4; ++k) *rows[k] = make_float4(x[k].x * inv.x, x[k].y * inv.y, x[k].z * inv.z, x[k].w * inv.w);
            }
        }
        if (dbg && et == 0) dbg[4] = clock64();
        esync();
        if (dbg && et == 0) dbg[10] = clock64();
        // ================= EPI-B: the attention core =================
        const int row_s0 = s_loc << LGN;                        // first row of this row's sample
        if (quarter) {
            constexpr int MPT = NPX / 4;                        // key pixels per thread in the S phase: m = j, j + 4, ...
            const int j = et & 3, row = (et >> 2) & 31, h = et >> 7;
            const int s2 = row >> LGN, rs0 = s2 << LGN;
            const uint32_t sw = NPX == 4 ? (uint32_t)((s2 >> 1) & 3) : (uint32_t)(s2 & 1);
            float q[32];
            {
                const float4* qr = reinterpret_cast<const float4*>(qst + (uint32_t)row * SM_KP + (uint32_t)h * 128u);
#pragma unroll
                for (int c4 = 0; c4 < 8; ++c4) {
                    const float4 t4 = qr[(uint32_t)c4 ^ sw];
                    q[4 * c4] = t4.x; q[4 * c4 + 1] = t4.y; q[4 * c4 + 2] = t4.z; q[4 * c4 + 3] = t4.w;
                }
            }
            float Sp[MPT];
#pragma unroll
            for (int i = 0; i < MPT; ++i) {
                const float4* kr = reinterpret_cast<const float4*>(kst + (uint32_t)(rs0 + j + 4 * i) * SM_KP + (uint32_t)h * 128u);
                float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;
#pragma unroll
                for (int c4 = 0; c4 < 8; ++c4) {
                    const float4 kk = kr[(uint32_t)c4 ^ sw];
                    a0 = fmaf(q[c4 * 4], kk.x, a0); a1 = fmaf(q[c4 * 4 + 1], kk.y, a1);
                    a2 = fmaf(q[c4 * 4 + 2], kk.z, a2); a3 = fmaf(q[c4 * 4 + 3], kk.w, a3);
                }
                Sp[i] = (a0 + a1) + (a2 + a3);
            }
            float S[NPX];
#pragma unroll
            for (int i = 0; i < MPT; ++i)
#pragma unroll
                for (int jj = 0; jj < 4; ++jj) S[jj + 4 * i] = __shfl_sync(0xffffffffu, Sp[i], (lane & ~3) | jj);
            if (!LINEAR) {                                      // softmax over the key pixels (unet.py:116-118)
                float m = S[0];
#pragma unroll
                for (int k = 1; k < NPX; ++k) m = fmaxf(m, S[k]);
                float sum = 0.f;
#pragma unroll
                for (int k = 0; k < NPX; ++k) { S[k] = fast_exp(S[k] - m); sum += S[k]; }
                const float inv = fast_rcp(sum);
#pragma unroll
                for (int k = 0; k < NPX; ++k) S[k] *= inv;
            }
            float o[8];
#pragma unroll
            for (int e = 0; e < 8; ++e) o[e] = 0.f;
#pragma unroll
            for (int m = 0; m < NPX; ++m) {
                const float4* vr = reinterpret_cast<const float4*>(vst + (uint32_t)(rs0 + m) * SM_KP + (uint32_t)h * 128u);
                const float4 va = vr[(uint32_t)(2 * j) ^ sw], vb = vr[(uint32_t)(2 * j + 1) ^ sw];
                o[0] = fmaf(S[m], va.x, o[0]); o[1] = fmaf(S[m], va.y, o[1]); o[2] = fmaf(S[m], va.z, o[2]); o[3] = fmaf(S[m], va.w, o[3]);
                o[4] = fmaf(S[m], vb.x, o[4]); o[5] = fmaf(S[m], vb.y, o[5]); o[6] = fmaf(S[m], vb.z, o[6]); o[7] = fmaf(S[m], vb.w, o[7]);
            }
            // channel = h*32 + 8j + e -> plane 4h + j of the K-major A operand of the to_out conv
            *reinterpret_cast<uint4*>(smem + p.xh_off + (uint32_t)(4 * h + j) * plane + (uint32_t)row * 16u) = pack8(o, p.fmt);
        } else if (wact) {
            const int h = part;
            float q[32];
            load_q(q);
            float S[NPX];
#pragma unroll
            for (int m = 0; m < NPX; ++m) {
                const float4* kr = reinterpret_cast<const float4*>(kst + (uint32_t)(row_s0 + m) * SM_KP + (uint32_t)h * 128u);
                float a0 = 0.f, a1 = 0.f, a2 = 0.f, a3 = 0.f;        // (the same association as the quarter-tile path: bit-equal results)
#pragma unroll
                for (int c4 = 0; c4 < 8; ++c4) {
                    const float4 kk = kr[(uint32_t)c4 ^ swz];
                    a0 = fmaf(q[c4 * 4], kk.x, a0); a1 = fmaf(q[c4 * 4 + 1], kk.y, a1);
                    a2 = fmaf(q[c4 * 4 + 2], kk.z, a2); a3 = fmaf(q[c4 * 4 + 3], kk.w, a3);
                }
                S[m] = (a0 + a1) + (a2 + a3);
            }
            if (!LINEAR) {                                      // softmax over the key pixels (unet.py:116-118)
                float m = S[0];
#pragma unroll
                for (int j = 1; j < NPX; ++j) m = fmaxf(m, S[j]);
                float sum = 0.f;
#pragma unroll
                for (int j = 0; j < NPX; ++j) { S[j] = fast_exp(S[j] - m); sum += S[j]; }
                const float inv = fast_rcp(sum);
#pragma unroll
                for (int j = 0; j < NPX; ++j) S[j] *= inv;
            }
            float o[32];
#pragma unroll
            for (int e = 0; e < 32; ++e) o[e] = 0.f;
#pragma unroll
            for (int m = 0; m < NPX; ++m) {
                const float4* vr = reinterpret_cast<const float4*>(vst + (uint32_t)(row_s0 + m) * SM_KP + (uint32_t)h * 128u);
#pragma unroll
                for (int c4 = 0; c4 < 8; ++c4) {
                    const float4 vv = vr[(uint32_t)c4 ^ swz];
                    o[c4 * 4] = fmaf(S[m], vv.x, o[c4 * 4]); o[c4 * 4 + 1] = fmaf(S[m], vv.y, o[c4 * 4 + 1]);
                    o[c4 * 4 + 2] = fmaf(S[m], vv.z, o[c4 * 4 + 2]); o[c4 * 4 + 3] = fmaf(S[m], vv.w, o[c4 * 4 + 3]);
                }
            }
            // channel = h*32 + e ('b h c (x y) -> b (h c) x y', unet.py:149 / 121), as the K-major A operand of the to_out conv
#pragma unroll
            for (int cb = 0; cb < 4; ++cb)
                *reinterpret_cast<uint4*>(smem + p.xh_off + (uint32_t)(4 * h + cb) * plane + (uint32_t)r * 16u) = pack8(o + cb * 8, p.fmt);
        }
        if (dbg && et == 0) dbg[11] = clock64();
        // ================= EPI-C: to_out bias [-> GroupNorm(1, C)] -> + x2 -> global =================
        // Up to four warp groups split the channels in whole 16-channel chunks (C = 128: 32 each, C = 64: 16 each, C = 32: two
        // groups); a thread holds at most two chunks, so the accumulators stay in registers between the statistics and the
        // normalisation, and the residual rows are requested BEFORE the to_out MMAs are waited for (an exposed L2 round trip per
        // chunk otherwise: 9.6k cycles for the x2-upsampled C = 128 output, profiles/r02_attn_small_timeline.txt).
        const int lgparts = (C & 63) == 0 ? 2 : ((C & 31) == 0 ? 1 : 0);
        const bool act = part < (1 << lgparts);
        const int cpp = C >> lgparts, c_lo = part * cpp, c_hi = (act && wact) ? c_lo + cpp : c_lo;
        uint4 xr[4];
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            xr[2 * k] = make_uint4(0, 0, 0, 0); xr[2 * k + 1] = xr[2 * k];
            const int c16 = c_lo + 16 * k;
            if (valid && c16 < c_hi) {
                xr[2 * k] = xsrc[(size_t)((c16 >> 3) * p.B + b) * NPX + px];
                xr[2 * k + 1] = xsrc[(size_t)(((c16 >> 3) + 1) * p.B + b) * NPX + px];
            }
        }
        fence_proxy_async();
        tc_fence_before();
        named_bar_arrive(2, n_epi + 32);
        if (act) {
        mbar_wait(bar_mma, 1);
        tc_fence_after();
        if (dbg && et == 0) dbg[26] = clock64();
        griddep_launch();            // PDL: the next stage kernel may become resident during the last epilogue
        const float* bias = par;
        const float* gamma = par + 128;
        const float* beta = par + 256;
        float v[2][16];
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            uint32_t u[16];
            if (c_lo + 16 * k < c_hi) tmem_ld16_issue(tlane + (uint32_t)(p.col_proj + c_lo + 16 * k), u);
            tmem_ld_wait();
#pragma unroll
            for (int j = 0; j < 16; ++j) v[k][j] = (c_lo + 16 * k < c_hi) ? __uint_as_float(u[j]) + bias[c_lo + 16 * k + j] : 0.f;
        }
        float mean = 0.f, rstd = 1.f;
        if (LINEAR) {
            float sx = 0.f, sq = 0.f;
#pragma unroll
            for (int k = 0; k < 2; ++k)
#pragma unroll
                for (int j = 0; j < 16; ++j) { sx += v[k][j]; sq = fmaf(v[k][j], v[k][j], sq); }
            if (!valid) { sx = 0.f; sq = 0.f; }
#pragma unroll
            for (int o = NPX >> 1; o > 0; o >>= 1) { sx += __shfl_xor_sync(0xffffffffu, sx, o); sq += __shfl_xor_sync(0xffffffffu, sq, o); }
            if (px == 0) hstat[part * 32 + s_loc] = make_float2(sx, sq);
            named_bar_sync(3, 128 << lgparts);
            if (dbg && et == 0) dbg[27] = clock64();
            sx = 0.f; sq = 0.f;
            for (int q = 0; q < (1 << lgparts); ++q) { const float2 a = hstat[q * 32 + s_loc]; sx += a.x; sq += a.y; }     // fixed order
            const float icnt = fast_rcp((float)(C * NPX));
            mean = sx * icnt;
            rstd = rsqrtf(fmaxf(sq * icnt - mean * mean, 0.f) + 1e-5f);
        }
#pragma unroll
        for (int k = 0; k < 2; ++k) {
            const int c16 = c_lo + 16 * k;
            if (c16 >= c_hi) continue;                 // warp-uniform
            float x2[16];
            unpack8(xr[2 * k], x2, p.fmt);
            unpack8(xr[2 * k + 1], x2 + 8, p.fmt);
#pragma unroll
            for (int j = 0; j < 16; ++j) {
                float y = v[k][j];
                if (LINEAR) y = (y - mean) * rstd * gamma[c16 + j] + beta[c16 + j];
                v[k][j] = y + x2[j];
            }
            attn_write_out_w(p, b, px, c16, v[k], valid, p.fmt);
        }
        }
        if (dbg && et == 0) dbg[28] = clock64();
    }
    tc_fence_before();
    __syncthreads();
    if (dbg && tid == 0) dbg[65] = clock64();
    if (p.dbg && tid == 0) { if (blockIdx.x == 0) p.dbg[102] = global_ns(); atomicMax(reinterpret_cast<unsigned long long*>(p.dbg + 103), (unsigned long long)global_ns()); }
    if (warp == w_mma) tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
}

cudaError_t attn_configure() {
    cudaError_t e = cudaFuncSetAttribute(k_attn<>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_attn<1, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_attn<1, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_attn<2, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_attn<2, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_attn_small<16, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_attn_small<4, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_attn_small<16, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_attn_small<4, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_attn_small<16, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_attn_small<4, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_attn_small<16, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_attn_small<4, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    return e;
}

cudaError_t launch_pdl(const void* fn, int grid, int block, size_t smem, cudaStream_t s, void** args, int cluster);
cudaError_t launch_attn_fused(const AttnFusedParams& p, const CUtensorMap& xh_map, int grid, cudaStream_t s) {
    void* args[2] = {(void*)&xh_map, (void*)&p};
    if (p.small) {
        const bool qt = p.nb * p.n == 32;
        const void* fn = p.n == 16 ? (p.full ? (qt ? (const void*)k_attn_small<16, false, true> : (const void*)k_attn_small<16, false>)
                                             : (qt ? (const void*)k_attn_small<16, true, true> : (const void*)k_attn_small<16, true>))
                                   : (p.full ? (qt ? (const void*)k_attn_small<4, false, true> : (const void*)k_attn_small<4, false>)
                                             : (qt ? (const void*)k_attn_small<4, true, true> : (const void*)k_attn_small<4, true>));
        return launch_pdl(fn, grid, SMALL_THREADS, (size_t)p.smem_bytes, s, args, 1);
    }
    // transposed K / V projections (linear attention): the planner sets them only for one M tile with 8 epilogue warps or two
    // with 16, the two LEAN instances
    const void* fn = (const void*)k_attn<>;
    if (p.ktrans && !p.full)
        fn = p.n_mtiles == 2 ? (p.fmt ? (const void*)k_attn<2, 1> : (const void*)k_attn<2, 0>)
                             : (p.fmt ? (const void*)k_attn<1, 1> : (const void*)k_attn<1, 0>);
    return launch_pdl(fn, grid, (p.epi_warps + 2) * 32, (size_t)p.smem_bytes, s, args, 1);
}

}  // namespace flo
