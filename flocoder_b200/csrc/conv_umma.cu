// Implicit-GEMM convolution on the 5th-generation tensor cores (tcgen05 / TMEM / TMA), sm_100a.
//
// GEMM view of a k x k (k = 1, 3 or 5, pad k/2) convolution over blocked bf16 activations:
//     D[pixel, cout] = sum_{tap, cin} A_tap[pixel, cin] * W[tap, cin, cout]
// * A operand: ONE TMA tensor-tile load per source brings the zero-padded image tile of `nb`
//   samples -- box {8ch, W+2p, H+2p, nb, C/8} at coordinates (0,-p,-p,b0,0), out-of-bounds = 0 --
//   into shared memory as [C/8][nb][H+2p][W+2p][8ch].  That is exactly the tcgen05 no-swizzle
//   K-major operand layout (16-byte rows, 8-row core matrices): the A tile of a tap is the
//   SAME bytes at a start address shifted by (dh*(W+2p)+dw)*16 B, so im2col costs no data
//   movement at all -- k*k descriptors instead of k*k copies.  torch.cat of two sources is two
//   TMA loads into consecutive planes (two K segments).
// * M tile = 128 output pixels = 16 groups of 8 consecutive padded pixels.  At 16x16 a tile is a
//   16-row x 8-column strip (group stride = padded row pitch, every row useful); at lower
//   resolutions a tile is 128 consecutive padded pixels of `nb` stacked samples (halo rows compute
//   junk that the epilogue discards).
// * B operand: weights pre-packed on the host into the canonical K-major core-matrix layout, streamed
//   through a ring of shared-memory stages by 1-D bulk TMA copies (cp.async.bulk, mbarrier tx).
// * D: fp32 accumulators in TMEM (one 128 x n_tile block per M tile); tcgen05.mma issued by one thread;
//   tcgen05.commit -> mbarrier hands stages back to the producer and the result to the epilogue.
// * Epilogue: 4 warps tcgen05.ld their 32 TMEM lanes, add bias (then SiLU, then the fp32 residual), and write fp32
//   and/or bf16 blocked outputs with 32-/16-byte vector stores, plus the pixel-unshuffled / nearest-x2 bf16 copies the
//   inpainting mask fusions hand to the next Downsample / Upsample conv.
// * Mask branches switched off at run time (*mask_mode < need_mode) do no MMA: the CTA copies the bypass tensor to every
//   output, or returns when there is none.  The flag is uniform over the grid, so one captured graph serves every mode.
//
// Warp roles (192 threads): warps 0-3 epilogue, warp 4 TMA producer, warp 5 TMEM owner + MMA issuer.
#include <cuda_fp16.h>
#include <string.h>

#include "flo_internal.h"
#include "umma_common.cuh"

namespace flo {

constexpr int UMMA_THREADS = 192;

// ------------------------------------------------------------------------------------------------
// geometry shared by the MMA issuer and the epilogue
// ------------------------------------------------------------------------------------------------
struct ConvGeom {
    int Wp, PP;        // padded row pitch and padded pixels per sample (H*W for 1x1)
};
__device__ __forceinline__ int tile_row0(const ConvUmmaParams& p, int t) {
    if (p.sbo_px != 8) {            // strip mode: tile = 16 image rows x 8 columns
        const int pad = p.ksize >> 1;
        const int tx_n = p.W >> 3;
        const int ty = t / tx_n, tx = t % tx_n;
        return (ty * 16 + pad) * (p.W + 2 * pad) + pad + 8 * tx;
    }
    return p.row0 + t * p.tile_stride;
}

// Pixels of shared memory past the A planes that a tile may address: the last M tile's rows run up to 127 pixels past the
// plane, and a tap shifts by up to pad*(Wp+1).  (1x1 keeps the 3x3 slack.)
__host__ __device__ __forceinline__ uint32_t a_slack_px(int pad, int Wp) {
    return 128u + (uint32_t)((pad > 1 ? pad : 1) * (Wp + 1) + 1);
}

// bf16 copies of one 8-channel pixel vector of a [cout/8][B][H][W][8] output: pixel-unshuffled ('b c (h p1) (w p2) ->
// b (c p1 p2) h w' in our (p1 p2 c) channel order, as k_gn writes it) and nearest x2
__device__ __forceinline__ void store_un_up(const ConvUmmaParams& p, int cb, int b, int h, int w, uint4 u) {
    const int HW = p.H * p.W;
    if (p.out_un) {
        const int plane = ((h & 1) * 2 + (w & 1)) * (p.cout >> 3) + cb;
        const int q = (h >> 1) * (p.W >> 1) + (w >> 1);
        *reinterpret_cast<uint4*>(p.out_un + ((size_t)(plane * p.B + b) * (HW >> 2) + q) * 8) = u;
    }
    if (p.out_up) {
        const int W2 = p.W * 2;
#pragma unroll
        for (int d = 0; d < 4; ++d) {
            const int q = (2 * h + (d >> 1)) * W2 + 2 * w + (d & 1);
            *reinterpret_cast<uint4*>(p.out_up + ((size_t)(cb * p.B + b) * (HW * 4) + q) * 8) = u;
        }
    }
}
__device__ __forceinline__ uint4 pack_bf16x8(const float* o) {
    uint4 u;
    __nv_bfloat162* h2 = reinterpret_cast<__nv_bfloat162*>(&u);
#pragma unroll
    for (int q = 0; q < 4; ++q) h2[q] = __floats2bfloat162_rn(o[2 * q], o[2 * q + 1]);
    return u;
}

// a mask branch switched off at run time: this CTA's samples and output channels are the bypass tensor
__device__ __forceinline__ void conv_umma_bypass(const ConvUmmaParams& p) {
    const int HW = p.H * p.W, ncb = p.n_tile >> 3;
    const int b0 = blockIdx.x * p.nb, nbh = min(p.nb, p.B - b0);
    const int cb0 = (blockIdx.y * p.n_tile) >> 3;
    const int n = nbh * HW * ncb;
    for (int i = threadIdx.x; i < n; i += blockDim.x) {
        const int px = i % HW, r = i / HW, s = r % nbh, cb = cb0 + r / nbh, b = b0 + s;
        const size_t off = ((size_t)(cb * p.B + b) * HW + px) * 8;
        const float4 v0 = *reinterpret_cast<const float4*>(p.bypass + off);
        const float4 v1 = *reinterpret_cast<const float4*>(p.bypass + off + 4);
        if (p.out_m) {
            *reinterpret_cast<float4*>(p.out_m + off) = v0;
            *reinterpret_cast<float4*>(p.out_m + off + 4) = v1;
        }
        const float o[8] = {v0.x, v0.y, v0.z, v0.w, v1.x, v1.y, v1.z, v1.w};
        const uint4 u = pack_bf16x8(o);
        if (p.out_o) *reinterpret_cast<uint4*>(p.out_o + off) = u;
        const int h = px / p.W;
        store_un_up(p, cb, b, h, px - h * p.W, u);
    }
}

__global__ void __launch_bounds__(UMMA_THREADS) k_conv_umma(const __grid_constant__ CUtensorMap tmA0,
                                                            const __grid_constant__ CUtensorMap tmA1,
                                                            const ConvUmmaParams p) {
    extern __shared__ __align__(128) uint8_t smem[];
    // run-time mask mode: read once, before any barrier or tensor memory exists (uniform over the grid)
    if (p.mask_mode && *p.mask_mode < p.need_mode) {
        if (p.bypass) conv_umma_bypass(p);
        return;
    }
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int ncbT = p.ncb0 + p.ncb1;
    const int pad = p.ksize >> 1;
    const int Wp = p.W + 2 * pad, Hp = p.H + 2 * pad, PP = Wp * Hp;
    const uint32_t plane_bytes = (uint32_t)p.plane_px * 16u;
    const uint32_t a_bytes = (uint32_t)ncbT * plane_bytes;
    const uint32_t a_region = (a_bytes + a_slack_px(pad, Wp) * 16u + 127u) & ~127u;
    const uint32_t stage_bytes = (uint32_t)p.slices_per_stage * (uint32_t)p.n_tile * 32u;
    const uint32_t ring_off = a_region;
    const uint32_t bar_off = ring_off + (uint32_t)p.n_wstages * stage_bytes;

    const uint32_t smem_base = smem_u32(smem);
    const uint32_t bar_full = smem_base + bar_off;                 // [MAX_WSTAGES]
    const uint32_t bar_empty = bar_full + 8 * MAX_WSTAGES;         // [MAX_WSTAGES]
    const uint32_t bar_a = bar_empty + 8 * MAX_WSTAGES;
    const uint32_t bar_done = bar_a + 8;
    const uint32_t tmem_slot = bar_done + 8;
    volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem + bar_off + 16 * MAX_WSTAGES + 16);

    const int b0 = blockIdx.x * p.nb;
    const int nt = blockIdx.y;
    const int taps = p.ksize * p.ksize;
    const int cpT = ncbT >> 1;                       // K16 slices per tap
    const int total_slices = taps * cpT;
    const int n_loads = total_slices / p.slices_per_stage;

    if (warp == 4 && lane == 0) {
        for (int i = 0; i < p.n_wstages; ++i) { mbar_init(bar_full + 8 * i, 1); mbar_init(bar_empty + 8 * i, 1); }
        mbar_init(bar_a, 1);
        mbar_init(bar_done, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA0) : "memory");
        if (p.ncb1) asm volatile("prefetch.tensormap [%0];" ::"l"(&tmA1) : "memory");
    }
    if (warp == 5) tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_ptr;

    if (warp == 4) {
        // ===================== TMA producer =====================
        if (lane == 0) {
            mbar_expect_tx(bar_a, a_bytes);
            tma_load_5d(smem_base, &tmA0, bar_a, 0, -pad, -pad, b0, 0);
            if (p.ncb1) tma_load_5d(smem_base + (uint32_t)p.ncb0 * plane_bytes, &tmA1, bar_a, 0, -pad, -pad, b0, 0);
            const uint8_t* wsrc = reinterpret_cast<const uint8_t*>(p.w) + (size_t)nt * total_slices * p.n_tile * 32;
            for (int i = 0; i < n_loads; ++i) {
                const int slot = i % p.n_wstages;
                if (i >= p.n_wstages) mbar_wait(bar_empty + 8 * slot, ((i / p.n_wstages) - 1) & 1);
                mbar_expect_tx(bar_full + 8 * slot, stage_bytes);
                bulk_load_1d(smem_base + ring_off + slot * stage_bytes, wsrc + (size_t)i * stage_bytes, stage_bytes,
                             bar_full + 8 * slot);
            }
        }
    } else if (warp == 5) {
        // ===================== MMA issuer =====================
        if (lane == 0) {
            const uint32_t idesc = make_idesc_bf16(128, p.n_tile);
            const uint32_t a_sbo = (uint32_t)p.sbo_px * 16u;
            const uint32_t b_lbo = (uint32_t)p.n_tile * 16u;
            mbar_wait(bar_a, 0);
            for (int i = 0; i < n_loads; ++i) {
                const int slot = i % p.n_wstages;
                mbar_wait(bar_full + 8 * slot, (i / p.n_wstages) & 1);
                tc_fence_after();
                const uint32_t bstage = smem_base + ring_off + slot * stage_bytes;
                for (int s = 0; s < p.slices_per_stage; ++s) {
                    const int ks = i * p.slices_per_stage + s;
                    const int tap = ks / cpT, cp = ks - tap * cpT;
                    const int shift = pad ? ((tap / p.ksize - pad) * Wp + (tap % p.ksize - pad)) : 0;
                    const uint64_t bdesc = make_smem_desc(bstage + (uint32_t)s * (uint32_t)p.n_tile * 32u, b_lbo, 128u);
                    for (int t = 0; t < p.n_mtiles; ++t) {
                        const uint32_t a_addr =
                            smem_base + (uint32_t)(2 * cp) * plane_bytes + (uint32_t)(tile_row0(p, t) + shift) * 16u;
                        const uint64_t adesc = make_smem_desc(a_addr, plane_bytes, a_sbo);
                        umma_bf16(tmem_base + (uint32_t)(t * p.n_tile), adesc, bdesc, idesc, ks > 0 ? 1u : 0u);
                    }
                }
                umma_commit(bar_empty + 8 * slot);      // frees the weight stage when these MMAs retire
            }
            umma_commit(bar_done);                      // accumulators complete
        }
    } else {
        // ===================== epilogue (warps 0-3 <-> TMEM lanes 32w..32w+31) =====================
        mbar_wait(bar_done, 0);
        tc_fence_after();
        const int HW = p.H * p.W;
        const int r = warp * 32 + lane;
        const int g = r >> 3, i8 = r & 7;
        for (int t = 0; t < p.n_mtiles; ++t) {
            const int pp = tile_row0(p, t) + g * p.sbo_px + i8;
            const int s = pp / PP, rem = pp - s * PP;
            bool valid;
            int px;
            if (pad) {
                const int hh = rem / Wp - pad, ww = rem % Wp - pad;
                valid = (s < p.nb) && (hh >= 0) && (hh < p.H) && (ww >= 0) && (ww < p.W);
                px = hh * p.W + ww;
            } else {
                valid = (s < p.nb);
                px = rem;
            }
            const int b = b0 + s;
            valid = valid && (b < p.B);
            const uint32_t trow = tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(t * p.n_tile);
            for (int c16 = 0; c16 < p.n_tile; c16 += 16) {
                float v[16];
                tmem_ld16(trow + (uint32_t)c16, v);
                if (!valid) continue;
                const int c = nt * p.n_tile + c16;
#pragma unroll
                for (int hb = 0; hb < 2; ++hb) {
                    float* o = v + hb * 8;
                    const int cc = c + hb * 8;
                    if (p.bias) {
                        const float4 b0v = *reinterpret_cast<const float4*>(p.bias + cc);
                        const float4 b1v = *reinterpret_cast<const float4*>(p.bias + cc + 4);
                        o[0] += b0v.x; o[1] += b0v.y; o[2] += b0v.z; o[3] += b0v.w;
                        o[4] += b1v.x; o[5] += b1v.y; o[6] += b1v.z; o[7] += b1v.w;
                    }
                    if (p.act_silu) {           // nn.SiLU of the mask-fusion convs, in k_conv_simt's IEEE form
#pragma unroll
                        for (int j = 0; j < 8; ++j) o[j] = o[j] / (1.0f + expf(-o[j]));
                    }
                    const size_t off = ((size_t)((cc >> 3) * p.B + b) * HW + px) * 8;
                    if (p.res) {
                        const float4 r0 = *reinterpret_cast<const float4*>(p.res + off);
                        const float4 r1 = *reinterpret_cast<const float4*>(p.res + off + 4);
                        o[0] += r0.x; o[1] += r0.y; o[2] += r0.z; o[3] += r0.w;
                        o[4] += r1.x; o[5] += r1.y; o[6] += r1.z; o[7] += r1.w;
                    }
                    if (p.out_m) {
                        *reinterpret_cast<float4*>(p.out_m + off) = make_float4(o[0], o[1], o[2], o[3]);
                        *reinterpret_cast<float4*>(p.out_m + off + 4) = make_float4(o[4], o[5], o[6], o[7]);
                    }
                    if (p.out_o || p.out_un || p.out_up) {
                        const uint4 u = pack_bf16x8(o);
                        if (p.out_o) *reinterpret_cast<uint4*>(p.out_o + off) = u;
                        if (p.out_un || p.out_up) {
                            const int h = px / p.W;
                            store_un_up(p, cc >> 3, b, h, px - h * p.W, u);
                        }
                    }
                }
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 5) tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
}

cudaError_t conv_umma_configure() {
    return cudaFuncSetAttribute(k_conv_umma, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
}

cudaError_t launch_conv_umma(const ConvUmmaParams& p, const CUtensorMap& a0, const CUtensorMap& a1, cudaStream_t s) {
    dim3 grid((p.B + p.nb - 1) / p.nb, p.cout / p.n_tile);
    k_conv_umma<<<grid, UMMA_THREADS, p.smem_bytes, s>>>(a0, a1, p);
    return cudaGetLastError();
}

// shared-memory bytes the kernel carves for a configuration (must mirror the kernel's arithmetic)
int conv_umma_smem_bytes(const ConvUmmaParams& p) {
    const int pad = p.ksize >> 1, Wp = p.W + 2 * pad;
    const uint32_t plane_bytes = (uint32_t)p.plane_px * 16u;
    const uint32_t a_bytes = (uint32_t)(p.ncb0 + p.ncb1) * plane_bytes;
    const uint32_t a_region = (a_bytes + a_slack_px(pad, Wp) * 16u + 127u) & ~127u;
    const uint32_t stage_bytes = (uint32_t)p.slices_per_stage * (uint32_t)p.n_tile * 32u;
    return (int)(a_region + p.n_wstages * stage_bytes + 16 * MAX_WSTAGES + 16 + 16);
}

// ------------------------------------------------------------------------------------------------
// host-side weight packing: OIHW fp32 -> per n-tile stream of K16 slices in core-matrix order
//   [n_tile index][slice = tap*(cin/16)+cp][k half][n/8][n%8][k%8]   (bf16)
// ------------------------------------------------------------------------------------------------
size_t pack_umma_weights(const float* w, int cout, int cin, int ksize, const int* perm, int n_tile, bool f16,
                         std::vector<__nv_bfloat16>& out) {
    const int taps = ksize * ksize, cpT = cin / 16;
    const size_t start = out.size();
    out.resize(start + (size_t)cout * cin * taps);
    __nv_bfloat16* dst = out.data() + start;
    size_t idx = 0;
    for (int nt = 0; nt < cout / n_tile; ++nt)
        for (int tap = 0; tap < taps; ++tap)
            for (int cp = 0; cp < cpT; ++cp)
                for (int h = 0; h < 2; ++h)
                    for (int n = 0; n < n_tile; ++n)
                        for (int j = 0; j < 8; ++j) {
                            const int ci_ours = (2 * cp + h) * 8 + j;
                            const int ci = perm ? perm[ci_ours] : ci_ours;
                            const int co = nt * n_tile + n;
                            const float x = w[((size_t)co * cin + ci) * taps + tap];
                            if (f16) { const __half hv = __float2half(x); memcpy(&dst[idx++], &hv, 2); }
                            else dst[idx++] = __float2bfloat16(x);
                        }
    return idx;
}

// ------------------------------------------------------------------------------------------------
// descriptor micro-test: D[128 x N] = A[128 x K] * B[N x K]^T with A placed at arbitrary
// (start shift, LBO, SBO) -- the exact descriptor forms the convolution relies on.
// ------------------------------------------------------------------------------------------------
struct MicroParams {
    const __nv_bfloat16* a;   // [128][K] row-major
    const __nv_bfloat16* b;   // [N][K] row-major
    float* d;                 // [128][N]
    int N, K;
    int a_lbo, a_sbo, a_shift;   // bytes
    int b_lbo, b_sbo;            // bytes
};
__global__ void __launch_bounds__(128) k_umma_micro(MicroParams p) {
    extern __shared__ __align__(128) uint8_t smem[];
    __shared__ __align__(8) uint64_t bar;
    __shared__ uint32_t tslot;
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t a_off = 0, b_off = 96 * 1024;
    // place A: element (m, k) at a_shift + (k/8)%2... general: k16 slice s, half h, row m
    for (int idx = tid; idx < 128 * p.K; idx += 128) {
        const int m = idx / p.K, k = idx % p.K;
        const int s = k / 16, h = (k / 8) & 1, j = k & 7;
        const uint32_t o = a_off + (uint32_t)p.a_shift + (uint32_t)s * 2u * (uint32_t)p.a_lbo + (uint32_t)h * p.a_lbo +
                           (uint32_t)(m / 8) * p.a_sbo + (uint32_t)(m % 8) * 16u + (uint32_t)j * 2u;
        *reinterpret_cast<__nv_bfloat16*>(smem + o) = p.a[idx];
    }
    for (int idx = tid; idx < p.N * p.K; idx += 128) {
        const int n = idx / p.K, k = idx % p.K;
        const int s = k / 16, h = (k / 8) & 1, j = k & 7;
        const uint32_t o = b_off + (uint32_t)s * 2u * (uint32_t)p.b_lbo + (uint32_t)h * p.b_lbo +
                           (uint32_t)(n / 8) * p.b_sbo + (uint32_t)(n % 8) * 16u + (uint32_t)j * 2u;
        *reinterpret_cast<__nv_bfloat16*>(smem + o) = p.b[idx];
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");   // generic-proxy writes -> async proxy (UMMA)
    if (tid == 0) {
        mbar_init(smem_u32(&bar), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    int cols = 32;
    while (cols < p.N) cols <<= 1;
    if (warp == 0) tmem_alloc(smem_u32(&tslot), cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tbase = *reinterpret_cast<volatile uint32_t*>(&tslot);
    if (tid == 0) {
        const uint32_t idesc = make_idesc_bf16(128, p.N);
        const uint32_t base = smem_u32(smem);
        for (int s = 0; s < p.K / 16; ++s) {
            const uint64_t ad = make_smem_desc(base + a_off + p.a_shift + s * 2 * p.a_lbo, p.a_lbo, p.a_sbo);
            const uint64_t bd = make_smem_desc(base + b_off + s * 2 * p.b_lbo, p.b_lbo, p.b_sbo);
            umma_bf16(tbase, ad, bd, idesc, s > 0);
        }
        umma_commit(smem_u32(&bar));
    }
    mbar_wait(smem_u32(&bar), 0);
    tc_fence_after();
    for (int c = 0; c < p.N; c += 16) {
        float v[16];
        tmem_ld16(tbase + ((uint32_t)(warp * 32) << 16) + c, v);
        for (int i = 0; i < 16; ++i) p.d[(size_t)(warp * 32 + lane) * p.N + c + i] = v[i];
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tbase, cols);
}

cudaError_t launch_umma_micro(const __nv_bfloat16* a, const __nv_bfloat16* b, float* d, int N, int K, int a_lbo,
                              int a_sbo, int a_shift, int b_lbo, int b_sbo, cudaStream_t s) {
    static bool configured = false;
    if (!configured) {
        cudaFuncSetAttribute(k_umma_micro, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        configured = true;
    }
    MicroParams p{a, b, d, N, K, a_lbo, a_sbo, a_shift, b_lbo, b_sbo};
    k_umma_micro<<<1, 128, 200 * 1024, s>>>(p);
    return cudaGetLastError();
}


// ------------------------------------------------------------------------------------------------
// swizzled-operand micro-test + issue-rate probe: K-major SWIZZLE_{32,64,128}B operands with shifted start
// addresses (base_offset) and non-atom-multiple group strides; also times `reps` back-to-back MMAs.
// ------------------------------------------------------------------------------------------------
struct Micro2Params {
    const __nv_bfloat16* a;   // [128][K]
    const __nv_bfloat16* b;   // [N][K]
    float* d;                 // [128][N]
    long long* cycles;        // [1]: SM cycles for `reps` MMA chains (issue -> commit -> barrier)
    int N, K;
    int layout;               // 0 none, 2 = 128B, 4 = 64B, 6 = 32B swizzle
    int row_bytes;            // bytes per operand row (K-major): 16 (none: core-matrix rows) / 32 / 64 / 128
    int a_sbo, a_shift, a_lbo;
    int use_base_offset;
    int reps;
};
__device__ __forceinline__ uint32_t swz(uint32_t lin, int layout) {
    const uint32_t mask = layout == 2 ? 7u : layout == 4 ? 3u : layout == 6 ? 1u : 0u;
    return lin ^ (((lin >> 7) & mask) << 4);
}
__global__ void __launch_bounds__(128) k_umma_micro2(Micro2Params p) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bar;
    __shared__ uint32_t tslot;
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const uint32_t a_off = 0, b_off = 96 * 1024;
    const int kpr = p.row_bytes / 2;          // K elements per row
    for (int idx = tid; idx < 128 * p.K; idx += 128) {
        const int m = idx / p.K, k = idx % p.K;
        uint32_t lin;
        if (p.layout == 0) lin = (uint32_t)p.a_shift + (uint32_t)(k / 8) * p.a_lbo + (uint32_t)(m / 8) * p.a_sbo + (uint32_t)(m % 8) * 16u + (uint32_t)(k % 8) * 2u;
        else lin = (uint32_t)p.a_shift + (uint32_t)(m / 8) * p.a_sbo + (uint32_t)(m % 8) * p.row_bytes + (uint32_t)(k % kpr) * 2u;
        *reinterpret_cast<__nv_bfloat16*>(smem + a_off + swz(lin, p.layout)) = p.a[idx];
    }
    const uint32_t b_sbo = p.layout == 0 ? 128u : 8u * p.row_bytes, b_lbo = (uint32_t)p.N * 16u;
    for (int idx = tid; idx < p.N * p.K; idx += 128) {
        const int n = idx / p.K, k = idx % p.K;
        uint32_t lin;
        if (p.layout == 0) lin = (uint32_t)(k / 8) * b_lbo + (uint32_t)(n / 8) * 128u + (uint32_t)(n % 8) * 16u + (uint32_t)(k % 8) * 2u;
        else lin = (uint32_t)(n / 8) * b_sbo + (uint32_t)(n % 8) * p.row_bytes + (uint32_t)(k % kpr) * 2u;
        *reinterpret_cast<__nv_bfloat16*>(smem + b_off + swz(lin, p.layout)) = p.b[idx];
    }
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    if (tid == 0) {
        mbar_init(smem_u32(&bar), 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    int cols = 32;
    while (cols < p.N) cols <<= 1;
    if (warp == 0) tmem_alloc(smem_u32(&tslot), cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tbase = *reinterpret_cast<volatile uint32_t*>(&tslot);
    long long t0 = 0;
    if (warp == 1) {
        const uint32_t idesc = make_idesc_bf16(128, p.N);
        const uint32_t base = smem_u32(smem);
        const uint64_t lt = (uint64_t)p.layout << 61;
        t0 = clock64();
        for (int rep = 0; rep < p.reps; ++rep) {
            for (int s = 0; s < p.K / 16; ++s) {
                uint32_t a_addr, b_addr, a_l, b_l, a_s, b_s;
                if (p.layout == 0) {
                    a_addr = base + a_off + p.a_shift + s * 2 * p.a_lbo; b_addr = base + b_off + s * 2 * b_lbo;
                    a_l = p.a_lbo; b_l = b_lbo; a_s = p.a_sbo; b_s = 128;
                } else {
                    a_addr = base + a_off + p.a_shift + s * 32; b_addr = base + b_off + s * 32;
                    a_l = 16; b_l = 16; a_s = p.a_sbo; b_s = b_sbo;
                }
                uint64_t ad = make_smem_desc(a_addr, a_l, a_s) | lt;
                uint64_t bd = make_smem_desc(b_addr, b_l, b_s) | lt;
                if (p.use_base_offset) ad |= (uint64_t)((a_addr >> 7) & 7u) << 49;
                if (elect_one()) umma_bf16(tbase, ad, bd, idesc, (rep | s) > 0);
            }
        }
        if (elect_one()) umma_commit(smem_u32(&bar));
        __syncwarp();
    }
    mbar_wait(smem_u32(&bar), 0);
    tc_fence_after();
    if (warp == 1 && lane == 0) p.cycles[0] = clock64() - t0;
    for (int c = 0; c < p.N; c += 16) {
        float v[16];
        tmem_ld16(tbase + ((uint32_t)(warp * 32) << 16) + c, v);
        for (int i = 0; i < 16; ++i) p.d[(size_t)(warp * 32 + lane) * p.N + c + i] = v[i];
    }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tbase, cols);
}
cudaError_t launch_umma_micro2(const __nv_bfloat16* a, const __nv_bfloat16* b, float* d, long long* cycles, int N, int K, int layout,
                               int row_bytes, int a_sbo, int a_shift, int a_lbo, int use_base_offset, int reps, cudaStream_t s) {
    static bool configured = false;
    if (!configured) {
        cudaFuncSetAttribute(k_umma_micro2, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        configured = true;
    }
    Micro2Params p{a, b, d, cycles, N, K, layout, row_bytes, a_sbo, a_shift, a_lbo, use_base_offset, reps};
    k_umma_micro2<<<1, 128, 200 * 1024, s>>>(p);
    return cudaGetLastError();
}


// Back-to-back tcgen05.mma throughput probe: one elected thread issues `n_mma` M=128 x N x K=16 MMAs on zeroed no-swizzle
// operands (A start address cycling through 4 tiles), one commit, then waits.  cycles[0] = issue loop, cycles[1] = until done.
// a_mode: 0 = A from shared memory; 1 = A from tensor memory (the .ts form: 8 TMEM columns per K16 slice);
// a_shift: byte offset added to the shared-memory A start (16 = one pixel of a 3x3 tap, i.e. off the 128-byte line).
__global__ void __launch_bounds__(128) k_umma_rate(long long* cycles, int N, int n_mma, int n_acc, int a_mode, int a_shift) {
    extern __shared__ uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bar;
    __shared__ uint32_t tslot;
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    for (int i = tid * 16; i < 96 * 1024; i += 128 * 16) *reinterpret_cast<uint4*>(smem + i) = make_uint4(0, 0, 0, 0);
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    if (tid == 0) {
        mbar_init(smem_u32(&bar), n_acc < 0 ? 2 : 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    int cols = 32;
    while (cols < N * (n_acc < 0 ? 2 : n_acc) + (a_mode == 1 ? 32 : 0)) cols <<= 1;
    if (warp == 0) tmem_alloc(smem_u32(&tslot), cols);
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tbase = *reinterpret_cast<volatile uint32_t*>(&tslot);
    long long t0 = 0, t1 = 0;
    const bool dual = n_acc < 0;                 // two issuing warps (1 and 2), one accumulator each, barrier count 2
    const int nacc = dual ? 1 : n_acc;
    if (warp == 1 || (dual && warp == 2)) {
        const uint32_t idesc = make_idesc_bf16(128, N);
        const uint32_t base = smem_u32(smem);
        // A: LBO = 2 KB plane, SBO = 128 B; a_mode >= 2: the strided row groups of the zero-copy im2col (SBO = a_mode * 16 bytes,
        // e.g. 18 = the padded row of a 16-pixel-wide image), LBO = 8 KB planes
        const uint64_t ad0 = a_mode >= 2 ? make_smem_desc(base + (uint32_t)a_shift, 8192u, (uint32_t)a_mode * 16u)
                                         : make_smem_desc(base + (uint32_t)a_shift, 2048u, 128u);
        const uint32_t a_t0 = tbase + (uint32_t)(N * nacc);                     // A tiles in TMEM (contents irrelevant for timing)
        const uint64_t bd0 = make_smem_desc(base + 64 * 1024, (uint32_t)N * 16u, 128u);
        const uint32_t tcol = tbase + (uint32_t)((warp - 1) * N);
        t0 = clock64();
        if (elect_one()) {
            const uint32_t acc_mask = (uint32_t)(nacc - 1);
#pragma unroll 4
            for (int i = 0; i < n_mma; ++i) {
                const uint32_t dcol = tcol + ((uint32_t)i & acc_mask) * (uint32_t)N;
                if (a_mode == 1) {
                    asm volatile(
                        "{\n\t.reg .pred p;\n\t"
                        "setp.ne.b32 p, %4, 0;\n\t"
                        "tcgen05.mma.cta_group::1.kind::f16 [%0], [%1], %2, %3, p;\n\t}"
                        ::"r"(dcol), "r"(a_t0 + (uint32_t)((i & 3) * 8)), "l"(bd0), "r"(idesc), "r"(1u)
                        : "memory");
                } else {
                    umma_bf16(dcol, ad0 + (uint64_t)((i & 3) * ((a_mode >= 2 ? 16384 : 4096) >> 4)), bd0, idesc, 1u);
                }
            }
            umma_commit(smem_u32(&bar));
        }
        __syncwarp();
        t1 = clock64();
    }
    mbar_wait(smem_u32(&bar), 0);
    tc_fence_after();
    if (warp == 1 && lane == 0) { cycles[0] = t1 - t0; cycles[1] = clock64() - t0; }
    tc_fence_before();
    __syncthreads();
    if (warp == 0) tmem_dealloc(tbase, cols);
}
cudaError_t launch_umma_rate(long long* cycles, int N, int n_mma, int n_acc, cudaStream_t s, int a_mode, int a_shift) {
    static bool configured = false;
    if (!configured) {
        cudaFuncSetAttribute(k_umma_rate, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        configured = true;
    }
    k_umma_rate<<<1, 128, 200 * 1024, s>>>(cycles, N, n_mma, n_acc, a_mode, a_shift);
    return cudaGetLastError();
}

// Micro-benchmark: how fast ONE CTA pulls a weight stream from L2 through a ring of bulk copies (what the chain stages do at the
// low resolutions): thread 0 issues cp.async.bulk copies (`pieces` per chunk) into an n_ring-deep ring, thread 32 consumes a chunk
// as soon as it is full.  Every CTA of the grid streams the same bytes (same_src) or its own region.
__global__ void __launch_bounds__(64) k_stream_rate(const uint8_t* src, long long* cycles, int total_bytes, int chunk_bytes, int n_ring,
                                                    int pieces, int same_src) {
    extern __shared__ __align__(128) uint8_t smem_raw[];
    __shared__ __align__(8) uint64_t bars[2 * 32];
    const uint32_t full = smem_u32(&bars[0]), empty = smem_u32(&bars[32]);
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 127) & ~(uintptr_t)127);
    const int tid = threadIdx.x;
    if (tid == 0) {
        for (int i = 0; i < n_ring; ++i) { mbar_init(full + 8 * i, 1); mbar_init(empty + 8 * i, 1); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    __syncthreads();
    const uint8_t* my = src + (same_src ? 0 : (size_t)blockIdx.x * (size_t)total_bytes);
    const int n_chunks = total_bytes / chunk_bytes;
    const long long t0 = clock64();
    // pieces > 0: thread 0 issues `pieces` copies per chunk; pieces < 0: lanes 0..-pieces-1 of warp 0 issue the chunks round-robin
    // (one whole-chunk copy each, all lanes in the same instruction)
    if (pieces < 0 && tid < -pieces) {
        const int P = -pieces;
        for (int c = tid; c < n_chunks; c += P) {
            const int slot = c % n_ring;
            if (c >= n_ring) mbar_wait(empty + 8 * slot, ((c / n_ring) - 1) & 1);
            mbar_expect_tx(full + 8 * slot, (uint32_t)chunk_bytes);
            bulk_load_1d(smem_u32(smem) + (uint32_t)slot * (uint32_t)chunk_bytes, my + (size_t)c * chunk_bytes, (uint32_t)chunk_bytes, full + 8 * slot);
        }
    } else if (pieces > 0 && tid == 0) {
        const uint32_t piece = (uint32_t)(chunk_bytes / pieces);
        for (int c = 0; c < n_chunks; ++c) {
            const int slot = c % n_ring;
            if (c >= n_ring) mbar_wait(empty + 8 * slot, ((c / n_ring) - 1) & 1);
            mbar_expect_tx(full + 8 * slot, (uint32_t)chunk_bytes);
            for (int q = 0; q < pieces; ++q)
                bulk_load_1d(smem_u32(smem) + (uint32_t)slot * (uint32_t)chunk_bytes + (uint32_t)q * piece,
                             my + (size_t)c * chunk_bytes + (size_t)q * piece, piece, full + 8 * slot);
        }
    } else if (tid == 32) {
        for (int c = 0; c < n_chunks; ++c) {
            const int slot = c % n_ring;
            mbar_wait(full + 8 * slot, (c / n_ring) & 1);
            mbar_arrive(empty + 8 * slot);
        }
        if (blockIdx.x == 0) cycles[0] = clock64() - t0;
    }
}
cudaError_t launch_stream_rate(const void* src, long long* cycles, int grid, int total_bytes, int chunk_bytes, int n_ring, int pieces,
                               int same_src, cudaStream_t s) {
    static bool configured = false;
    if (!configured) {
        cudaFuncSetAttribute(k_stream_rate, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
        configured = true;
    }
    k_stream_rate<<<grid, 64, (size_t)n_ring * chunk_bytes + 256, s>>>(reinterpret_cast<const uint8_t*>(src), cycles, total_bytes, chunk_bytes,
                                                                        n_ring, pieces, same_src);
    return cudaGetLastError();
}

}  // namespace flo
