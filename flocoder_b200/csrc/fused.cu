// Fused stage kernels (sm_100a): whole ResnetBlock chains of one resolution level in ONE kernel.
// A CTA owns `nb` complete samples; activations never leave the SM inside a stage -- 16-bit operands live in
// shared memory in the blocked/padded layout that doubles as the tcgen05 no-swizzle K-major operand (3x3 taps
// = shifted descriptors, torch.cat = two operand slots), fp32 accumulators live in TMEM, weights are streamed
// through a shared-memory ring by bulk TMA copies.
//
// k_chain   [conv -> GroupNorm+FiLM+SiLU(+residual)]* with
//           * the conv bias folded into the GEMM (one extra K slice: a constant "ones" A tile x a B tile holding the
//             bias split into a 16-bit high part and a 16-bit remainder, so it is exact to ~2^-17),
//           * the ResnetBlock 1x1 res_conv accumulated into a second TMEM region (never leaves TMEM),
//           * GroupNorm statistics reduced with warp shuffles on register-resident accumulator chunks wherever the row
//             geometry allows it (one sample per CTA: FAST; 2x2 N-split stages: a sample = one half-warp; 4x4 stages: a
//             sample's valid rows = one warp) -- otherwise per-row partial sums and ONE (scale, offset) pair per (sample,
//             channel) in shared memory, so that the normalise pass is one FMA + SiLU per element,
//           * the PreNorm of the following attention block fused into the last epilogue,
//           * init_conv (unet.py:295) as the first epilogue of the first stage and final_conv + the RK4 / Euler
//             / CFG stage update (unet.py:372, sampling.py:43-48,69-74) as the last epilogue of the last stage.
//
// Warp roles (320 threads): warps 0-7 = epilogue, warp 8 lane 0 = TMA producer (input tiles, weight ring), warp 9 =
// tcgen05.mma issuer (warp-uniform code, one elected lane issues a whole weight chunk of MMAs).
// The EIGHT epilogue warps are two warp groups that share the four TMEM lane quadrants: with several M tiles per
// CTA a warp group owns whole tiles (tile t -> group t & 1), with one M tile the groups split the output channels
// (group g -> channels [g C/2, (g+1) C/2)), so a thread normalises 8..16 accumulator values per step instead of 32:
// the epilogue is a latency chain (TMEM load -> FMA -> MUFU -> pack -> store), and its length, not the instruction
// count, is what a step costs.  The kernel is templated on everything that is uniform per launch -- M tiles per CTA,
// N-split, 16-bit operand format, FAST epilogue, the two-CTAs-per-SM register cap (WIDE lifts it for single-wave
// launches), init / final code (ENDS) -- and a stage launches the instance that matches it: tile loops, row bookkeeping
// and pack/unpack code are static, and no launch pays registers or spills for code it never runs (DESIGN.md 5.3).
// Steps alternate MMA(i) -> EPI(i) -> MMA(i+1) ...: bar_mma (tcgen05.commit) one way; back, inside one CTA a named
// barrier, across a cluster the output stores themselves (st.async completing transaction bytes on the consumers'
// mbarriers).  Overlap of one sample group's epilogue with another's MMAs comes from the co-resident CTA.
#include <cuda_fp16.h>

#include <cstring>
#include <type_traits>
#include "flo_internal.h"
#include "umma_common.cuh"
#include "fused_common.cuh"

namespace flo {

// geometry of the M tiles, in registers
struct Geo {
    int W, H, Wp, PP, nb, B, strips, sbo_px, tx_n;
};
__device__ __forceinline__ Geo make_geo(const ChainParams& p) {
    Geo g;
    g.W = p.W; g.H = p.H; g.Wp = p.W + 2; g.PP = g.Wp * (p.H + 2); g.nb = p.nb; g.B = p.B;
    g.strips = p.strips; g.sbo_px = p.strips ? g.Wp : 8; g.tx_n = p.W >> 3;
    return g;
}
__device__ __forceinline__ int tile_row0(const Geo& g, int t) {
    if (g.strips) return ((t / g.tx_n) * 16 + 1) * g.Wp + 1 + 8 * (t % g.tx_n);
    return g.Wp + 1 + t * 128;
}
struct RowInfo {
    int pp;        // flattened padded pixel index inside the CTA's planes
    int s, px;     // sample within the CTA, unpadded pixel index h*W+w
    bool valid;
};
__device__ __forceinline__ RowInfo make_row(const Geo& g, int t, int r, int b0) {
    RowInfo ri;
    ri.pp = tile_row0(g, t) + (r >> 3) * g.sbo_px + (r & 7);
    ri.s = ri.pp / g.PP;
    const int rem = ri.pp - ri.s * g.PP;
    const int hh = rem / g.Wp, ww = rem - hh * g.Wp;
    ri.px = (hh - 1) * g.W + (ww - 1);
    ri.valid = (ri.s < g.nb) && (b0 + ri.s < g.B) && hh >= 1 && hh <= g.H && ww >= 1 && ww <= g.W;
    return ri;
}

// ------------------------------------------------------------------------------------------------
// MMA issue: one convolution = taps x channel-pair slices (+ 1 bias slice), weights from the ring
// ------------------------------------------------------------------------------------------------
struct RingPos {               // ring slot and mbarrier phase, advanced without integer division
    int slot; uint32_t phase;
    __device__ __forceinline__ void next(int n_ring) { if (++slot == n_ring) { slot = 0; phase ^= 1u; } }
};
struct ConvIssue {
    const int32_t* tab;        // per-slice A start address (>>4, tap shift + Wp + 1; IssueCtx::row0 adds the tile's rest)
    int n, col, slices, S;
};
template <int MT>
struct IssueCtx {
    uint32_t tmem_base, bar_full, bar_empty, ring_lo, ring_slot16, ones_lo;
    uint32_t plane16;          // plane stride >> 4
    uint32_t desc_hi_a, desc_hi_ones;
    int n_ring;
    uint32_t row0[MT];
    int cc;                    // global ring chunk counter
    RingPos rp;
    long long* dbg;
};
__device__ __forceinline__ uint64_t desc64(uint32_t lo, uint32_t hi) {
    uint64_t d;
    asm("mov.b64 %0, {%1, %2};" : "=l"(d) : "r"(lo), "r"(hi));
    return d;
}
// The A operand of K16 slice ks = two channel-block planes of one input slot, shifted by the 3x3 tap: its start
// address comes from the table built at kernel start, so the issuing thread runs load / add / tcgen05.mma only.
template <int MT, int FMT>
__device__ __forceinline__ void issue_conv(IssueCtx<MT>& x, const ConvIssue& c) {
    const uint32_t idesc = make_idesc16(128, c.n, FMT, 0, 0);
    const uint32_t b_hi = (128u >> 4) | (1u << 14);
    const uint32_t b_lbo = ((uint32_t)c.n & 0x3FFFu) << 16;      // n*16 bytes >> 4 in the LBO field
    const uint32_t a_lbo = (x.plane16 & 0x3FFFu) << 16;
    const uint32_t slice16 = (uint32_t)c.n * 2u;                 // n*32 bytes >> 4
    const int conv_slices = c.slices - 1;                        // the last slice is the bias
    for (int ks0 = 0; ks0 < c.slices; ks0 += c.S) {
        const int cnt = min(c.S, c.slices - ks0);
        const int slot = x.rp.slot;
        mbar_wait(x.bar_full + 8 * slot, x.rp.phase);
        tc_fence_after();
        if (x.dbg && x.cc >= 8 && x.cc < 16 && (threadIdx.x & 31) == 0) x.dbg[104 + (x.cc - 8) * 3 + 2] = clock64();   // chunk seen full
        if (elect_one()) {
            uint32_t b_lo = (x.ring_lo + (uint32_t)slot * x.ring_slot16) | b_lbo;
            const int32_t* tp = c.tab + ks0;
            const int n_conv = min(cnt, conv_slices - ks0);      // slices of this chunk that are convolution slices
            uint32_t acc = ks0 > 0 ? 1u : 0u;                    // the very first slice overwrites the accumulator
            auto mma_slice = [&](int32_t e) {
                const uint64_t bdesc = desc64(b_lo, b_hi);
                const uint32_t a_base = (uint32_t)e | a_lbo;
#pragma unroll
                for (int t = 0; t < MT; ++t)
                    umma_bf16(x.tmem_base + (uint32_t)(c.col + t * c.n), desc64(a_base + x.row0[t], x.desc_hi_a), bdesc, idesc, acc);
                acc = 1u;
                b_lo += slice16;
            };
            int s = 0;
            if constexpr (MT == 1) {
                // groups of four slices: the table entries of the next group are loaded before this group's MMAs are issued
                int32_t e[4], f[4];
#pragma unroll
                for (int k = 0; k < 4; ++k) e[k] = (n_conv >= 4) ? tp[k] : 0;
                for (; s + 4 <= n_conv; s += 4) {
#pragma unroll
                    for (int k = 0; k < 4; ++k) f[k] = (s + 8 <= n_conv) ? tp[s + 4 + k] : 0;
#pragma unroll
                    for (int k = 0; k < 4; ++k) mma_slice(e[k]);
#pragma unroll
                    for (int k = 0; k < 4; ++k) e[k] = f[k];
                }
            } else {
                // several M tiles per slice: one entry ahead is enough (and keeps the register count of the kernel down)
                int32_t cur = n_conv > 0 ? tp[0] : 0;
                for (; s < n_conv; ++s) {
                    const int32_t nxt = tp[s + 1];               // the table has one spare entry per conv
                    mma_slice(cur);
                    cur = nxt;
                }
            }
            for (; s < n_conv; ++s) mma_slice(tp[s]);
            if (ks0 + cnt == c.slices) {
                // bias slice: rows [1,1,0..] x (bias hi, bias lo); K half 1 = zeros
                const uint64_t bdesc = desc64(b_lo, b_hi);
                const uint64_t adesc = desc64(x.ones_lo | (8u << 16), x.desc_hi_ones);
#pragma unroll
                for (int t = 0; t < MT; ++t) umma_bf16(x.tmem_base + (uint32_t)(c.col + t * c.n), adesc, bdesc, idesc, 1u);
            }
            umma_commit(x.bar_empty + 8 * slot);
        }
        __syncwarp();
        ++x.cc;
        x.rp.next(x.n_ring);
    }
}

// ------------------------------------------------------------------------------------------------
// epilogue helpers
// ------------------------------------------------------------------------------------------------
template <int N> struct IntTag { static constexpr int value = N; };

// Per-(sample, group) statistics from the per-row (sum, sumsq) partials in shared memory, then the collapsed
// (scale, offset) table:  y = x*scale + offset  ==  FiLM(GroupNorm(x)).
//   rowstat[row * GS + gs], rows = MT*128, GS = G * pm: `pm` partial columns per group (2 when the two warp groups of
//   a one-tile CTA each hold half of a group's channels).  A segment of `seg` lanes owns one (sample, group): every
//   lane sums a strided share of the rows in a fixed order, a shuffle tree combines them (deterministic), and the same
//   lanes then write the group's channels of coef[s*C + c].  Two named barriers per call.
// `gpar[c]` = (gamma, beta); with `has_film`, coef[s*C+c] holds (1+scale, shift) on entry.
struct XChg {                    // cross-CTA (cluster) reduction of per-sample statistics; nsplit == 1: unused
    int nsplit; uint32_t rank, smem_base, bar_x; int xpart_off; uint32_t* phase; uint8_t* smem;
};
__device__ __forceinline__ void stats_to_coef(const Geo& g, int R, const float2* rowstat, float2* coef, const float2* gpar, int G, int pm,
                                              int C, int HW, bool has_film, int et, const XChg* xc = nullptr) {
    // G, C, seg are powers of two: shifts instead of runtime integer divisions on this serial stretch
    const int lgG = 31 - __clz(G), combos = g.nb * G, cpg = C >> lgG, GS = G * pm;
    const int cpw = (combos + EPI_WARPS - 1) / EPI_WARPS;
    int seg = 32;
    while (seg * cpw > 32) seg >>= 1;
    const int warp = et >> 5, lane = et & 31;
    const int lgS = 31 - __clz(seg);
    const int combo = warp * (32 >> lgS) + (lane >> lgS), li = lane & (seg - 1);
    const bool active = combo < combos;
    const int s = active ? (combo >> lgG) : 0, gi = active ? (combo & (G - 1)) : 0;
    epi_sync();
    float sx = 0.f, sq = 0.f;
    if (active) {
        int lo = 0, hi = R;
        if (!g.strips) {
            lo = min(max(s * g.PP - (g.Wp + 1), 0), R);
            hi = min(max((s + 1) * g.PP - (g.Wp + 1), 0), R);
        }
        const float2* rs = rowstat + gi * pm;
        if (pm == 1) {
            for (int r = lo + li; r < hi; r += seg) { const float2 v = rs[r * GS]; sx += v.x; sq += v.y; }
        } else {
            for (int r = lo + li; r < hi; r += seg) {
                const float4 v = *reinterpret_cast<const float4*>(rs + r * GS);
                sx += v.x + v.z; sq += v.y + v.w;
            }
        }
    }
    for (int o = seg >> 1; o > 0; o >>= 1) {
        sx += __shfl_xor_sync(0xffffffffu, sx, o);
        sq += __shfl_xor_sync(0xffffffffu, sq, o);
    }
    int n_parts = 1;
    if (xc && xc->nsplit > 1) {
        // G == 1 here: every CTA of the cluster holds the sums over ITS channels; publish them to all CTAs, then
        // add the parts in rank order (deterministic, identical in every CTA)
        n_parts = xc->nsplit;
        // every CTA receives nsplit x nb (sum, sumsq) pairs of 8 bytes; one thread posts the expectation, the stores signal
        if (et == 0) mbar_expect_tx(xc->bar_x, (uint32_t)(n_parts * g.nb * 8));
        if (active && li == 0)
            for (int q = 0; q < n_parts; ++q)
                st_async_f2(mapa_shared(xc->smem_base + (uint32_t)xc->xpart_off + (uint32_t)((int)xc->rank * g.nb + s) * 8u, (uint32_t)q),
                            make_float2(sx, sq), mapa_shared(xc->bar_x, (uint32_t)q));
        mbar_wait_cluster(xc->bar_x, *xc->phase & 1u);
        ++*xc->phase;
        if (active) {
            const float2* xp = reinterpret_cast<const float2*>(xc->smem + xc->xpart_off);
            sx = 0.f; sq = 0.f;
            for (int q = 0; q < n_parts; ++q) { const float2 v = xp[q * g.nb + s]; sx += v.x; sq += v.y; }
        }
    }
    if (active) {
        // reciprocal and rsqrt through MUFU (2 ulp): the IEEE division / sqrt sequences are ~100 instructions on this
        // serial stretch between the two barriers
        const float icnt = fast_rcp((float)(cpg * HW * n_parts));
        const float mean = sx * icnt;
        const float var = fmaxf(sq * icnt - mean * mean, 0.f);
        const float rstd = rsqrtf(var + 1e-5f);
        for (int c = gi * cpg + li; c < (gi + 1) * cpg; c += seg) {
            const float2 gb = gpar[c];
            float a = rstd * gb.x, bb = gb.y - mean * a;
            if (has_film) {
                const float2 f = coef[s * C + c];
                a *= f.x; bb = bb * f.x + f.y;
            }
            coef[s * C + c] = make_float2(a, bb);
        }
    }
    epi_sync();
}

// Sum of NV values per lane over the 32 lanes of a warp.  A butterfly would move all NV values at every level (NV x 5
// shuffles); here every level also halves the values a lane is responsible for, so the exchange costs NV/2 + NV/4 + ...
// + 1 shuffles for the splitting levels and one per remaining level.  On return p[0] holds the warp total of value
// `idx` (the return value: bit k of idx = lane bit 4-k); the 32/NV lanes with the same upper lane bits hold the same
// total.  Fixed exchange pattern: deterministic.
template <int NV>
__device__ __forceinline__ int warp_sum_scatter(float (&p)[NV], int lane) {
    int idx = 0, o = 16;
#pragma unroll
    for (int h = NV / 2; h >= 1; h >>= 1, o >>= 1) {
        const bool upper = (lane & o) != 0;
#pragma unroll
        for (int j = 0; j < h; ++j) {
            const float send = upper ? p[j] : p[j + h];
            const float keep = upper ? p[j + h] : p[j];
            p[j] = keep + __shfl_xor_sync(0xffffffffu, send, o);
        }
        idx += upper ? h : 0;
    }
    for (; o >= 1; o >>= 1) p[0] += __shfl_xor_sync(0xffffffffu, p[0], o);
    return idx;
}

// ------------------------------------------------------------------------------------------------
// k_chain
// ------------------------------------------------------------------------------------------------
// SPLIT: the N-split (cluster) variant; false compiles every cluster / DSMEM path out (Q == 1, c0 == 0 fold away)
#ifndef FLO_CHAIN_MINB
#define FLO_CHAIN_MINB 2
#endif
constexpr int FINAL_MAX_CH = 4;     // latent channels the fused final epilogue handles (api.cu routes more to the layer-wise path)
// FAST: every GroupNorm step of the stage takes the warp-shuffle path (one sample per CTA, one accumulator chunk per
// thread: chosen by the planner); the generic row-statistics path is compiled out, and vice versa.
// WIDE: an instance without the two-CTAs-per-SM register cap, launched when the grid leaves at most one CTA per SM anyway; the
// barrier-free 4x4 GroupNorm epilogue lives there (it spills under the 96-register cap and then loses to the generic one).
// ENDS: bit 0 = the stage may hold the init conv (first stage), bit 1 = the final conv + integrator update (last stage).  The FAST
// instances are compiled per combination: the 96-register cap that keeps two CTAs on an SM made the all-in-one instance spill on
// its hot path (280 bytes of spill loads), and the stages that hold neither ran 2.5 % faster end to end without that code.
template <int MT, bool SPLIT, int FMT, bool FAST, bool WIDE = false, int ENDS = 3>
__global__ void __launch_bounds__(FUSED_THREADS, (MT <= 2 && !SPLIT && !WIDE) ? FLO_CHAIN_MINB : 1) k_chain(const __grid_constant__ CUtensorMap tm0,
                                                         const __grid_constant__ CUtensorMap tm1,
                                                         const __grid_constant__ CUtensorMap tm2,
                                                         const __grid_constant__ CUtensorMap tm3,
                                                         const __grid_constant__ ChainParams p) {
    extern __shared__ __align__(128) uint8_t smem[];
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, tid = threadIdx.x;
    constexpr int W_PROD = EPI_WARPS, W_MMA = EPI_WARPS + 1;
    const uint32_t smem_base = smem_u32(smem);
    const int bar_off = p.bar_off;
    const uint32_t bar_full = smem_base + bar_off;
    const uint32_t bar_empty = bar_full + 8 * MAX_WSTAGES;
    const uint32_t bar_load = bar_empty + 8 * MAX_WSTAGES;
    const uint32_t bar_mma = bar_load + 8;
    const uint32_t bar_epi = bar_mma + 8;
    const uint32_t tmem_slot = bar_epi + 8;
    const uint32_t bar_x = tmem_slot + 8;
    const uint32_t bar_epi2 = bar_x + 8;         // N-split step hand-off: steps alternate between bar_epi and bar_epi2
    volatile uint32_t* tmem_slot_ptr = reinterpret_cast<volatile uint32_t*>(smem + bar_off + 16 * MAX_WSTAGES + 24);
    const Geo geo = make_geo(p);
    // N-split: the Q CTAs of a cluster own the same samples and 1/Q of every step's output channels
    const int Q = SPLIT ? p.nsplit : 1;
    const uint32_t qrank = SPLIT ? cluster_ctarank() : 0u;
    const int lgQ = SPLIT ? 31 - __clz(Q) : 0;          // cluster sizes are powers of two
    const int b0 = ((int)blockIdx.x >> lgQ) * geo.nb;
    const uint32_t plane_bytes = (uint32_t)p.plane_px * 16u;
    const int n_steps = p.n_steps, n_ring = p.n_ring, n_loads = p.n_loads, tmem_cols = p.tmem_cols;
    const int ones_off = p.ones_off;
    long long* dbg = (blockIdx.x == 0) ? p.dbg : nullptr;
    if (p.dbg && tid == 0 && blockIdx.x == 0) p.dbg[100] = global_ns();

    if (warp == W_PROD && lane == 0) {
        for (int i = 0; i < n_ring; ++i) { mbar_init(bar_full + 8 * i, 1); mbar_init(bar_empty + 8 * i, 1); }
        mbar_init(bar_load, 1);
        mbar_init(bar_mma, 1);
        // N-split: the stores of every CTA of the cluster complete transaction bytes on these (one arrival: the expectation)
        mbar_init(bar_epi, SPLIT ? 1 : EPI_THREADS);
        mbar_init(bar_epi2, 1);
        mbar_init(bar_x, SPLIT ? 1 : EPI_THREADS);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == W_MMA) tmem_alloc(tmem_slot, (uint32_t)tmem_cols);
    {   // clear the slots the epilogues write (their halo must read as zero) and build the "ones" A tile
        const int zoff = p.zero_off, zbytes = p.zero_bytes;
        for (int i = tid * 16; i < zbytes; i += FUSED_THREADS * 16) *reinterpret_cast<uint4*>(smem + zoff + i) = make_uint4(0, 0, 0, 0);
        const uint32_t ones2 = pack2t<FMT>(1.0f, 1.0f);
        for (int i = tid; i < 256; i += FUSED_THREADS)      // plane 0: [1,1,0,0,0,0,0,0] per row (bias hi + lo); plane 1: zeros
            *reinterpret_cast<uint4*>(smem + ones_off + i * 16) = make_uint4(i < 128 ? ones2 : 0u, 0, 0, 0);
    }
    // the host-built tables (fused_plan.inc, end_chain) into shared memory; descriptor address field = 14 bits of
    // (CTA-local address >> 4): in a cluster the shared window address carries the CTA rank in its upper bits,
    // which must not leak into the LBO field
    int32_t* atab = reinterpret_cast<int32_t*>(smem + p.tab_off);
    {
        const int32_t* gtab = reinterpret_cast<const int32_t*>(p.fblob + p.tabs_off);
        const int base16 = (int)((smem_base >> 4) & 0x3FFFu);
        const int tab_n = p.tab_n, n_chunks = p.n_chunks;
        for (int i = tid; i < tab_n; i += FUSED_THREADS) atab[i] = gtab[i] + base16;
        const uint2* gw = reinterpret_cast<const uint2*>(gtab + tab_n) + (size_t)qrank * n_chunks;
        uint2* wtab_w = reinterpret_cast<uint2*>(smem + p.wtab_off);
        for (int i = tid; i < n_chunks; i += FUSED_THREADS) wtab_w[i] = gw[i];
    }
    fence_proxy_async();
    tc_fence_before();
    if (Q > 1) cluster_sync_all();       // barriers initialised and slots cleared in EVERY CTA before any remote store / arrive
    else __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot_ptr;
    if (dbg && tid == 0) dbg[CH_MAX_STEPS * 8] = clock64();
    if (dbg && tid == 0) dbg[101] = global_ns();

    if (warp == W_PROD) {
        // ============================ producer ============================
        // TWO issuing lanes (chunk cc -> lane cc & 1): the bulk copies of one thread do not overlap and two is what an SM keeps in
        // flight (profiles/r02_stream_rate.txt: 31.7 -> 55 B/clk for 16 KB chunks)
        if (dbg && lane == 8) {
            // timeline only: the cycle at which weight chunks 8..15 LAND in the ring (the MMA warp only sees them when it gets there);
            // walks every chunk in order so that the parity waits cannot alias an earlier phase of the same slot
            for (int cc = 0; cc < 16 && cc < p.n_chunks; ++cc) {
                mbar_wait(bar_full + 8 * (cc % n_ring), (uint32_t)(cc / n_ring) & 1u);
                if (cc >= 8) dbg[104 + (cc - 8) * 3] = clock64();
            }
        }
        constexpr int NL = 2;
        if (lane < NL) {
            const uint32_t ring_base = smem_base + p.ring_off, ring_slot_bytes = p.ring_slot_bytes;
            const uint2* wtab = reinterpret_cast<const uint2*>(smem + p.wtab_off);
            const uint8_t* wbase = reinterpret_cast<const uint8_t*>(p.wblob);
            const int n_chunks = p.n_chunks;
            auto issue = [&](int cc) {
                const uint2 e = wtab[cc];
                const int slot = cc % n_ring;
                const uint32_t full = bar_full + 8 * slot;
                if (cc >= n_ring) mbar_wait(bar_empty + 8 * slot, (uint32_t)((cc / n_ring) - 1) & 1u);
                if (dbg && cc >= 8 && cc < 16) dbg[104 + (cc - 8) * 3 + 1] = clock64();
                mbar_expect_tx(full, e.y);
                // ONE bulk copy per chunk: a cp.async.bulk costs ~520 cycles whatever its size (16 KB in one copy 31.7 B/clk, in four
                // 23.4, in sixteen 11.9), so chunks are as large as the ring allows
                bulk_load_1d(ring_base + (uint32_t)slot * ring_slot_bytes, wbase + e.x, e.y, full);
            };
            // the weights do not depend on the previous kernel: fill the ring before waiting for it
            const int pre = min(n_ring, n_chunks);
            int cc = lane;
            for (; cc < pre; cc += NL) issue(cc);
            griddep_wait();
            if (lane == 0 && n_loads > 0) {
                uint32_t lbytes = 0;
                for (int i = 0; i < n_loads; ++i) lbytes += (uint32_t)p.load_ncb[i] * plane_bytes;
                mbar_expect_tx(bar_load, lbytes);
                const CUtensorMap* maps[4] = {&tm0, &tm1, &tm2, &tm3};
                for (int i = 0; i < n_loads; ++i) tma_load_5d(smem_base + p.load_off[i], maps[i], bar_load, 0, -1, -1, b0, 0);
            }
            for (; cc < n_chunks; cc += NL) issue(cc);
        }
    } else if (warp == W_MMA) {
        // ============================ MMA issuer (whole warp, warp-uniform; one elected lane issues) ============================
        IssueCtx<MT> x;
        x.tmem_base = tmem_base; x.bar_full = bar_full; x.bar_empty = bar_empty;
        x.ring_lo = ((smem_base + p.ring_off) >> 4) & 0x3FFFu; x.ring_slot16 = (uint32_t)p.ring_slot_bytes >> 4;
        x.ones_lo = ((smem_base + ones_off) >> 4) & 0x3FFFu;
        x.plane16 = plane_bytes >> 4;
        x.desc_hi_a = (((uint32_t)geo.sbo_px * 16u) >> 4) | (1u << 14);
        x.desc_hi_ones = (128u >> 4) | (1u << 14);
        x.n_ring = n_ring; x.cc = 0; x.rp.slot = 0; x.rp.phase = 0; x.dbg = dbg;
#pragma unroll
        for (int t = 0; t < MT; ++t) x.row0[t] = (uint32_t)(tile_row0(geo, t) - (geo.Wp + 1));   // atab holds tile 0's Wp + 1
        if (n_loads > 0) mbar_wait(bar_load, 0);
        for (int i = 0; i < n_steps; ++i) {
            if (i > 0) {
                // epilogue -> MMA hand-off: inside one CTA a named barrier the 256 epilogue threads arrive on (no 256
                // serialised mbarrier arrivals); across a cluster the output stores themselves
                if (SPLIT) {
                    // every CTA of the cluster stores step i-1's 16-bit outputs into our slot with st.async: the barrier completes when
                    // all of them have landed -- (live rows) x (channel blocks of the step) x 16 bytes; steps alternate between two
                    // barriers, so a peer that is one step ahead signals the other one
                    const int live = min(geo.nb, geo.B - b0) * geo.H * geo.W;
                    const uint32_t bar = ((i - 1) & 1) ? bar_epi2 : bar_epi;
                    if (elect_one()) mbar_expect_tx(bar, (uint32_t)(live * (p.st[i - 1].C >> 3) * 16));
                    __syncwarp();
                    mbar_wait_cluster(bar, ((i - 1) >> 1) & 1);
                    fence_proxy_async_all();
                } else {
                    named_bar_sync(2, EPI_THREADS + 32);
                }
            }
            tc_fence_after();
            if (dbg && lane == 0) dbg[i * 8 + 0] = clock64();
            if (p.st[i].has_conv) {
                ConvIssue c;
                c.tab = atab + p.st[i].tab_idx;
                c.n = p.st[i].n; c.col = p.st[i].acc_col; c.slices = p.st[i].slices;
                c.S = p.st[i].slices_per_chunk;
                issue_conv<MT, FMT>(x, c);
                if (p.st[i].has_res) {
                    c.tab = atab + p.st[i].res_tab_idx;
                    c.col = p.st[i].res_col; c.slices = p.st[i].res_slices; c.S = p.st[i].res_slices_per_chunk;
                    issue_conv<MT, FMT>(x, c);
                }
                if (dbg && lane == 0) dbg[i * 8 + 1] = clock64();
                if (elect_one()) umma_commit(bar_mma);
            } else {
                if (elect_one()) mbar_arrive(bar_mma);
            }
            __syncwarp();
        }
    } else {
        // ============================ epilogue warps ============================
        const int wg = warp >> 2, quad = warp & 3;            // warp group; TMEM lane quadrant
        const int r = quad * 32 + lane;                       // row inside every M tile == TMEM lane
        const int et = tid;                                   // epilogue thread index (warps 0..7)
        const uint32_t tlane = tmem_base + ((uint32_t)(quad * 32) << 16);
        float2* rowstat = reinterpret_cast<float2*>(smem + p.stats_off);
        float2* coef = rowstat + MT * 128 * p.g_max;          // [nb][C] (scale, offset)
        float* cpar = reinterpret_cast<float*>(coef + p.coef_n);   // small per-step constants (init / final conv weights)
        const int cpar_n = p.cpar_n;
        float2* gpar = reinterpret_cast<float2*>(cpar + cpar_n);
        float* const fastbuf = reinterpret_cast<float*>(gpar + p.max_c);
        Ctrl* ctrl = p.ctrl;
        const float* fblob = p.fblob;
        const int HW = geo.H * geo.W;
        griddep_wait();              // ctrl, the FiLM table and every activation come from earlier kernels
        const int step_idx = ctrl->step;
        const Stage sg = ctrl->stages[step_idx];
        const float* film_tab = ctrl->film;
        const int film_per_sample = ctrl->film_per_sample, film_row = sg.film_row, film_dim = p.film_dim;
        // the M tiles of this thread's warp group: tile wg, wg + 2, ... (one tile: both groups work on tile 0)
        constexpr int TW = (MT + 1) / 2;
        RowInfo ri[TW];
#pragma unroll
        for (int k = 0; k < TW; ++k) {
            const int t = (MT == 1) ? 0 : wg + 2 * k;
            if (t < MT) ri[k] = make_row(geo, t, r, b0);
            else { ri[k].pp = 0; ri[k].s = 0; ri[k].px = 0; ri[k].valid = false; }
        }
        if (n_loads > 0) mbar_wait(bar_load, 0);
        uint32_t xphase = 0;
        XChg xc;
        xc.nsplit = Q; xc.rank = qrank; xc.smem_base = smem_base; xc.bar_x = bar_x; xc.xpart_off = p.xpart_off; xc.phase = &xphase;
        xc.smem = smem;

        for (int i = 0; i < n_steps; ++i) {
            // ---- step parameters into registers
            const int epi = p.st[i].epi, Ctot = p.st[i].C, acc_col = p.st[i].acc_col, res_col = p.st[i].res_col;
            const int C = Ctot >> lgQ, c0 = (int)qrank * C;      // this CTA's channels [c0, c0 + C) of the step's Ctot
            const int res_mode = p.st[i].res_mode, res_slot_off = p.st[i].res_slot_off;
            const int is_final = (ENDS & 2) ? p.st[i].final : 0, pn_g = p.st[i].pn_g;
            const int out_slot_off = p.st[i].out_slot_off;
            uint4* const og = p.st[i].out_g >= 0 ? reinterpret_cast<uint4*>(p.gt[p.st[i].out_g]) : nullptr;
            // this thread's channels of the step: one tile -> the warp groups split the channels (the final epilogue needs all
            // channels of a row in one thread: warp group 0 alone); several tiles -> all channels of the group's tiles
            int cbeg = 0, cend = C;
            if (MT == 1) {
                if (is_final) { cend = wg == 0 ? C : 0; }
                else { cbeg = wg * (C >> 1); cend = cbeg + (C >> 1); }
            }
            const bool cw8 = (cend - cbeg) == 8;
            // one 8-channel block of one row -> shared-memory slot(s) and/or the global tensor
            auto write8 = [&](const RowInfo& R, int cb, const float* v8) -> uint4 {
                const uint4 u = pack8t<FMT>(v8);
                if (out_slot_off >= 0) {
                    const uint32_t soff = (uint32_t)out_slot_off + (uint32_t)cb * plane_bytes + (uint32_t)R.pp * 16u;
                    if (!SPLIT) *reinterpret_cast<uint4*>(smem + soff) = u;
                    else if (i + 1 < n_steps) {
                        const uint32_t bar = (i & 1) ? bar_epi2 : bar_epi;
                        for (int q = 0; q < Q; ++q) st_async_v4(mapa_shared(smem_base + soff, (uint32_t)q), u, mapa_shared(bar, (uint32_t)q));
                    } else {
                        *reinterpret_cast<uint4*>(smem + soff) = u;      // last step: only this CTA reads the slot again (fused PreNorm)
                    }
                }
                if (og) og[(size_t)(cb * geo.B + b0 + R.s) * HW + R.px] = u;
                return u;
            };
            // calls fn(k, c, IntTag<CW>) for every (tile, channel chunk) of this thread
            auto for_chunks = [&](auto&& fn) {
                if (cw8) {
                    fn(0, cbeg, IntTag<8>());
                } else {
#pragma unroll
                    for (int k = 0; k < TW; ++k) {
                        if (MT > 1 && wg + 2 * k >= MT) continue;
                        for (int c = cbeg; c < cend; c += 16) fn(k, c, IntTag<16>());
                    }
                }
            };
            auto tile_of = [&](int k) { return (MT == 1) ? 0 : wg + 2 * k; };
            // ---- final_conv bias + RK4 / Euler / CFG stage update (sampling.py:43-48,69-74)
            // the integrator state this thread updates is requested in one batch (independent loads in flight instead of
            // a dependent chain per element); the control block's pointers are read once
            auto final_update = [&](const float (&kacc)[(MT + 1) / 2][FINAL_MAX_CH]) {
                float* const Y = ctrl->y; float* const ACC = ctrl->acc; float* const XS = ctrl->xs; float* const VOUT = ctrl->vout;
                float* const VC = ctrl->vcond; float* const VT = ctrl->vtrace;
                const float cfg_s = ctrl->cfg;
                const int nch = p.channels, dim = p.dim;
                const size_t plane = (size_t)geo.B * nch * HW;
#pragma unroll
                for (int k = 0; k < (MT + 1) / 2; ++k) {
                    if (MT > 1 && wg + 2 * k >= MT) continue;
                    if (!ri[k].valid) continue;
                    const int b = b0 + ri[k].s;
                    float fy[4], fa[4], fc[4];
#pragma unroll
                    for (int co = 0; co < 4; ++co) {
                        fy[co] = 0.f; fa[co] = 0.f; fc[co] = 0.f;
                        if (co < nch) {
                            const size_t o = ((size_t)b * nch + co) * HW + ri[k].px;
                            if (sg.kind != ST_PLAIN && sg.kind != ST_CFG_COND) fy[co] = Y[o];
                            if (sg.kind == ST_RK2 || sg.kind == ST_RK3 || sg.kind == ST_RK4) fa[co] = ACC[o];
                            if (sg.flags & SF_CFG_COMBINE) fc[co] = VC[o];
                        }
                    }
#pragma unroll
                    for (int co = 0; co < FINAL_MAX_CH; ++co) {
                        if (co >= nch) continue;
                        float kv = kacc[k][co] + cpar[nch * dim + co];
                        const size_t o = ((size_t)b * nch + co) * HW + ri[k].px;
                        if (sg.flags & SF_CFG_COMBINE) kv = __fadd_rn(kv, __fmul_rn(cfg_s, __fsub_rn(fc[co], kv)));
                        if (VT && sg.eval_idx >= 0) VT[(size_t)sg.eval_idx * plane + o] = kv;
                        switch (sg.kind) {
                            case ST_PLAIN: VOUT[o] = kv; break;
                            case ST_CFG_COND: VC[o] = kv; break;
                            case ST_RK1:
                                ACC[o] = kv;
                                XS[o] = __fadd_rn(fy[co], __fmul_rn(__fmul_rn(sg.dt, kv), 0.5f));
                                break;
                            case ST_RK2:
                                ACC[o] = __fadd_rn(fa[co], __fmul_rn(2.0f, kv));
                                XS[o] = __fadd_rn(fy[co], __fmul_rn(__fmul_rn(sg.dt, kv), 0.5f));
                                break;
                            case ST_RK3:
                                ACC[o] = __fadd_rn(fa[co], __fmul_rn(2.0f, kv));
                                XS[o] = __fadd_rn(fy[co], __fmul_rn(sg.dt, kv));
                                break;
                            case ST_RK4: {
                                const float yn = __fadd_rn(fy[co], __fmul_rn(sg.dt6, __fadd_rn(fa[co], kv)));
                                Y[o] = yn; XS[o] = yn;
                            } break;
                            case ST_EULER: {
                                const float yn = __fadd_rn(fy[co], __fmul_rn(kv, sg.dt));
                                Y[o] = yn; XS[o] = yn;
                            } break;
                            default: break;
                        }
                    }
                }
            };
            // ---- classifier-free guidance as ONE pass over 2B samples (SF_CFG_2B): rows [0,B) are the conditional evaluations, rows
            // [B,2B) the unconditional ones of the same latents.  Every CTA publishes its velocities; of the two CTAs that hold the
            // halves of a sample the LATER one (a per-sample arrival counter) forms v_nc + cfg (v_c - v_nc) (sampling.py:69-74) and
            // does the integrator update, writing the next evaluation's input for both halves.  Barriers: all epilogue threads.
            auto final_update_2b = [&](const float (&kacc)[(MT + 1) / 2][FINAL_MAX_CH], bool has_rows) {
                float* const Y = ctrl->y; float* const ACC = ctrl->acc; float* const XS = ctrl->xs; float* const VC = ctrl->vcond;
                float* const VT = ctrl->vtrace;
                const float cfg_s = ctrl->cfg;
                const int Bh = ctrl->cfg_half, nch = p.channels, dim = p.dim;
                int* const arrived = reinterpret_cast<int*>(smem + p.xpart_off);      // [nb] (the N-split exchange area: unused here)
                float kv[(MT + 1) / 2][FINAL_MAX_CH];
#pragma unroll
                for (int k = 0; k < (MT + 1) / 2; ++k) {
#pragma unroll
                    for (int co = 0; co < FINAL_MAX_CH; ++co) kv[k][co] = 0.f;
                    if (!has_rows || (MT > 1 && wg + 2 * k >= MT) || !ri[k].valid) continue;
                    const int b = b0 + ri[k].s;
#pragma unroll
                    for (int co = 0; co < FINAL_MAX_CH; ++co) {
                        if (co >= nch) continue;
                        kv[k][co] = kacc[k][co] + cpar[nch * dim + co];
                        __stcg(VC + ((size_t)b * nch + co) * HW + ri[k].px, kv[k][co]);
                    }
                }
                __threadfence();
                epi_sync();
                if (et < geo.nb) {
                    int old = 0;
                    const int b = b0 + et;
                    if (b < geo.B) {
                        const int bs = b >= Bh ? b - Bh : b;
                        old = atomicAdd(ctrl->pair_flags + bs, 1);
                        if (old == 1) { ctrl->pair_flags[bs] = 0; __threadfence(); }      // both halves are in: re-arm for the next pass
                    }
                    arrived[et] = old;
                }
                epi_sync();
                const size_t plane = (size_t)Bh * nch * HW;
#pragma unroll
                for (int k = 0; k < (MT + 1) / 2; ++k) {
                    if (!has_rows || (MT > 1 && wg + 2 * k >= MT) || !ri[k].valid) continue;
                    if (arrived[ri[k].s] != 1) continue;
                    const int b = b0 + ri[k].s;
                    const bool uncond = b >= Bh;
                    const int bs = uncond ? b - Bh : b, bp = uncond ? bs : bs + Bh;
#pragma unroll
                    for (int co = 0; co < FINAL_MAX_CH; ++co) {
                        if (co >= nch) continue;
                        const float other = __ldcg(VC + ((size_t)bp * nch + co) * HW + ri[k].px);
                        const float vc = uncond ? other : kv[k][co], vnc = uncond ? kv[k][co] : other;
                        const float v = __fadd_rn(vnc, __fmul_rn(cfg_s, __fsub_rn(vc, vnc)));
                        const size_t o = ((size_t)bs * nch + co) * HW + ri[k].px;
                        if (VT && sg.eval_idx >= 0) VT[(size_t)sg.eval_idx * plane + o] = v;
                        float xn = 0.f;
                        switch (sg.kind) {
                            case ST_RK1: ACC[o] = v; xn = __fadd_rn(Y[o], __fmul_rn(__fmul_rn(sg.dt, v), 0.5f)); break;
                            case ST_RK2: ACC[o] = __fadd_rn(ACC[o], __fmul_rn(2.0f, v)); xn = __fadd_rn(Y[o], __fmul_rn(__fmul_rn(sg.dt, v), 0.5f)); break;
                            case ST_RK3: ACC[o] = __fadd_rn(ACC[o], __fmul_rn(2.0f, v)); xn = __fadd_rn(Y[o], __fmul_rn(sg.dt, v)); break;
                            case ST_RK4: xn = __fadd_rn(Y[o], __fmul_rn(sg.dt6, __fadd_rn(ACC[o], v))); Y[o] = xn; break;
                            case ST_EULER: xn = __fadd_rn(Y[o], __fmul_rn(v, sg.dt)); Y[o] = xn; break;
                            default: break;
                        }
                        XS[o] = xn; XS[o + plane] = xn;
                    }
                }
            };
            // warp-shuffle GroupNorm path: one sample per CTA and one accumulator chunk per thread
            constexpr bool fast_gn_k = FAST;
            const bool fast_gn = FAST && epi == CE_GN;
            float* const wpart = fastbuf;                                           // [8 warps][8] block norm | [8][2] PreNorm at +64
            float2* const gcoef = reinterpret_cast<float2*>(fastbuf + 128) + (i & 1) * p.max_c;          // (gamma', beta') with FiLM folded
            float2* const pnpar = reinterpret_cast<float2*>(fastbuf + 128) + (2 + (i & 1)) * p.max_c;    // PreNorm (gamma, beta)

            // small constants staged while the MMAs of this step run
            if ((ENDS & 1) && epi == CE_INIT) {
                const float* w = fblob + p.init_w_off;
                const float* bias = fblob + p.init_b_off;
                const int cin0 = p.cin0;
                for (int k = et; k < C * cin0; k += EPI_THREADS) cpar[k] = w[k];
                for (int k = et; k < C; k += EPI_THREADS) cpar[C * cin0 + k] = bias[k];
                epi_sync();
            } else if (is_final) {
                const float* w = fblob + p.final_w_off;
                const float* bias = fblob + p.final_b_off;
                const int nch = p.channels, dim = p.dim;
                for (int k = et; k < nch * dim; k += EPI_THREADS) cpar[k] = w[k];
                for (int k = et; k < nch; k += EPI_THREADS) cpar[nch * dim + k] = bias[k];
            }
            if (fast_gn) {
                // per-channel GroupNorm affine with the sample's FiLM factors folded in, fetched while the MMAs run:
                //   FiLM(GN(x)) = xhat*gamma' + beta',  gamma' = gamma (1+scale), beta' = beta (1+scale) + shift   (unet.py:70)
                // The tables alternate between two buffers by step parity: a thread cannot be two steps ahead of another one.
                const float* gamma = fblob + p.st[i].gamma_off;
                const float* beta = fblob + p.st[i].beta_off;
                const int foff = p.st[i].film_off;
                const float* fl = film_tab + (size_t)(film_per_sample ? b0 : film_row) * film_dim + foff;
                for (int c = et; c < C; c += EPI_THREADS) {
                    float f1 = 1.0f, f2 = 0.0f;
                    if (foff >= 0) { f1 = fl[c] + 1.0f; f2 = fl[C + c]; }
                    gcoef[c] = make_float2(gamma[c] * f1, fmaf(beta[c], f1, f2));
                    if (pn_g >= 0) pnpar[c] = make_float2(fblob[p.st[i].pn_gamma_off + c], fblob[p.st[i].pn_beta_off + c]);
                }
            } else if (epi == CE_GN) {
                // per-channel GroupNorm affine and per-(sample, channel) FiLM factors, fetched while the MMAs run
                epi_sync();           // every thread is done reading the previous step's coef / gpar
                const float* gamma = fblob + p.st[i].gamma_off;
                const float* beta = fblob + p.st[i].beta_off;
                for (int c = et; c < C; c += EPI_THREADS) gpar[c] = make_float2(gamma[c0 + c], beta[c0 + c]);
                const int foff = p.st[i].film_off, lgC = 31 - __clz(C);
                for (int idx = et; idx < geo.nb * C; idx += EPI_THREADS) {
                    const int s = idx >> lgC, c = idx & (C - 1);
                    float2 f = make_float2(1.0f, 0.0f);
                    if (foff >= 0 && b0 + s < geo.B) {
                        const float* fl = film_tab + (size_t)(film_per_sample ? (b0 + s) : film_row) * film_dim + foff;
                        f = make_float2(fl[c0 + c] + 1.0f, fl[Ctot + c0 + c]);          // x*(scale+1)+shift, unet.py:70
                    }
                    coef[idx] = f;
                }
                // the PreNorm affine of the last step too: fetched from global memory behind the statistics it was an exposed L2
                // round trip on the tail of the kernel
                if (pn_g >= 0)
                    for (int c = et; c < C; c += EPI_THREADS) pnpar[c] = make_float2(fblob[p.st[i].pn_gamma_off + c0 + c], fblob[p.st[i].pn_beta_off + c0 + c]);
            }
            mbar_wait(bar_mma, i & 1);
            tc_fence_after();
            if (dbg && et == 0) dbg[i * 8 + 2] = clock64();
            // programmatic dependent launch: let the next stage kernel become resident only now, during the last epilogue
            // (its barrier init, TMEM allocation, table copy and weight prefetch overlap this kernel's tail); triggering at
            // kernel start was measured to slow the running kernel (profiles/r01_pdl_gaps.txt)
            if (i == n_steps - 1) griddep_launch();

            if ((ENDS & 1) && epi == CE_INIT) {
                // ---- init_conv 1x1 from the NCHW fp32 integrator state (unet.py:295)
                const float* xs = ctrl->xs;
                const int cin0 = p.cin0;
#pragma unroll
                for (int k = 0; k < TW; ++k) {
                    if (MT > 1 && wg + 2 * k >= MT) continue;
                    if (!ri[k].valid) continue;
                    const int b = b0 + ri[k].s;
                    float xin[16];
#pragma unroll
                    for (int ci = 0; ci < 16; ++ci) xin[ci] = ci < cin0 ? xs[((size_t)b * cin0 + ci) * HW + ri[k].px] : 0.f;
                    for (int c8 = cbeg; c8 < cend; c8 += 8) {
                        float v[8];
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            float a = cpar[C * cin0 + c8 + j];
                            if (cin0 == 4) {          // the usual latent: one 16-byte weight row per output channel
                                const float4 w4 = *reinterpret_cast<const float4*>(cpar + (c8 + j) * 4);
                                a = fmaf(xin[0], w4.x, a); a = fmaf(xin[1], w4.y, a); a = fmaf(xin[2], w4.z, a); a = fmaf(xin[3], w4.w, a);
                            } else {
#pragma unroll
                                for (int ci = 0; ci < 16; ++ci)
                                    if (ci < cin0) a = fmaf(xin[ci], cpar[(c8 + j) * cin0 + ci], a);
                            }
                            v[j] = a;
                        }
                        write8(ri[k], (c0 + c8) >> 3, v);
                    }
                }
            } else if (epi == CE_BIAS) {
                // ---- conv (+bias via the GEMM)
                for_chunks([&](int k, int c, auto tag) {
                    constexpr int CW = decltype(tag)::value;
                    uint32_t u[CW];
                    const uint32_t ta = tlane + (uint32_t)(acc_col + tile_of(k) * C + c);
                    if constexpr (CW == 16) tmem_ld16_issue(ta, u); else tmem_ld8_issue(ta, u);
                    tmem_ld_wait();
                    if (!ri[k].valid) return;
                    float v[CW];
#pragma unroll
                    for (int j = 0; j < CW; ++j) v[j] = __uint_as_float(u[j]);
#pragma unroll
                    for (int hb = 0; hb < CW / 8; ++hb) write8(ri[k], ((c0 + c) >> 3) + hb, v + hb * 8);
                });
            } else {
                // ---- conv (+bias) -> GroupNorm -> FiLM -> SiLU -> + residual     (unet.py:64-73,96)
                const int G = p.st[i].groups >> lgQ, lg_cpg = 31 - __clz(C) - (31 - __clz(G)), cpg = 1 << lg_cpg;
                float kacc[TW][FINAL_MAX_CH];       // final 1x1 conv accumulators (latent channels; fused path: <= 4)
                float psx[TW], psq[TW];
#pragma unroll
                for (int k = 0; k < TW; ++k) {
                    psx[k] = 0.f; psq[k] = 0.f;
#pragma unroll
                    for (int j = 0; j < FINAL_MAX_CH; ++j) kacc[k][j] = 0.f;
                }
                if constexpr (fast_gn_k) {
                    if (dbg && et == 0) dbg[i * 8 + 3] = clock64();
                    // ======== one sample per CTA, one accumulator chunk per thread: the values stay in registers between the
                    // statistics and the normalisation, the statistics are reduced with warp shuffles and ONE named barrier,
                    // and every thread derives mean / rstd of its own groups from the eight per-warp partial sums.
                    float y[16];
                    uint4 pk[2];
                    const bool has_work = cend > cbeg;             // warp-uniform (the idle warp group of a one-tile final step)
                    const int t = tile_of(0);
                    // warps whose partial sums make up this thread's groups
                    const int wlo = (MT == 1 && (G > 1 || is_final)) ? wg * 4 : 0;
                    const int whi = (MT == 1 && (G > 1 || is_final)) ? wg * 4 + 4 : EPI_WARPS;
                    const float icnt = fast_rcp((float)(cpg * HW));
                    auto head = [&](auto cw_tag, auto ng_tag) {
                        constexpr int CW = decltype(cw_tag)::value, NG = decltype(ng_tag)::value, NV = 2 * NG, CG = CW / NG;
                        if (has_work) {
                            uint32_t av[CW];
                            const uint32_t ta = tlane + (uint32_t)(acc_col + t * C + cbeg);
                            if constexpr (CW == 16) tmem_ld16_issue(ta, av); else tmem_ld8_issue(ta, av);
                            tmem_ld_wait();
                            if (dbg && et == 0) dbg[i * 8 + 6] = clock64();
                            float ps[NV];
#pragma unroll
                            for (int g = 0; g < NG; ++g) {
                                float s0 = 0.f, q0 = 0.f, s1 = 0.f, q1 = 0.f;
#pragma unroll
                                for (int j = 0; j < CG; j += 2) {
                                    const float xa = __uint_as_float(av[g * CG + j]), xb = __uint_as_float(av[g * CG + j + 1]);
                                    s0 += xa; q0 = fmaf(xa, xa, q0); s1 += xb; q1 = fmaf(xb, xb, q1);
                                }
                                const bool valid = ri[0].valid;
                                ps[2 * g] = valid ? s0 + s1 : 0.f; ps[2 * g + 1] = valid ? q0 + q1 : 0.f;
                            }
                            const int idx = warp_sum_scatter<NV>(ps, lane);
                            if ((lane & (32 / NV - 1)) == 0) wpart[warp * 8 + idx] = ps[0];
#pragma unroll
                            for (int j = 0; j < CW; ++j) y[j] = __uint_as_float(av[j]);
                        }
                        if (dbg && et == 0) dbg[i * 8 + 7] = clock64();
                        epi_sync();
                        if (dbg && et == 0) dbg[80 + i] = clock64();
                        // mean / rstd of every group ONCE (lane g of the first warp whose partial sums make up the group: warp 0, or
                        // warps 0 and 4 when the two warp groups hold different channels), then a second barrier and one small load per
                        // thread -- instead of sixteen loads, 64 adds and NG rsqrt sequences in each of the 256 threads.  Same order of
                        // additions and the same expressions: bit-identical statistics.
                        float2* const gstat = reinterpret_cast<float2*>(fastbuf + 96) + (wlo ? 4 : 0);
                        if (has_work && warp == wlo && lane < NG) {
                            float sx = 0.f, sq = 0.f;
#pragma unroll
                            for (int k = 0; k < EPI_WARPS; ++k) {
                                const int w = wlo + k;
                                if (w < whi) { const float2 a = *reinterpret_cast<const float2*>(wpart + w * 8 + 2 * lane); sx += a.x; sq += a.y; }
                            }
                            const float mean = sx * icnt;
                            const float var = fmaxf(sq * icnt - mean * mean, 0.f);
                            const float rstd = rsqrtf(var + 1e-5f);
                            gstat[lane] = make_float2(rstd, -mean * rstd);
                        }
                        epi_sync();
                        if (!has_work) return;
#pragma unroll
                        for (int g = 0; g < NG; ++g) {
                            const float2 st = gstat[g];
#pragma unroll
                            for (int j = 0; j < CG; ++j) y[g * CG + j] = fmaf(y[g * CG + j], st.x, st.y);
                        }
                    };
                    auto tail = [&](auto cw_tag) {
                        constexpr int CW = decltype(cw_tag)::value;
                        if (!has_work) return;
                        uint32_t rv[CW];
                        if (res_mode == 1) {
                            const uint32_t ta = tlane + (uint32_t)(res_col + t * C + cbeg);
                            if constexpr (CW == 16) tmem_ld16_issue(ta, rv); else tmem_ld8_issue(ta, rv);
                            tmem_ld_wait();
                        }
                        if (!ri[0].valid) return;
                        float rr[CW];
                        if (res_mode == 2) {
                            const uint8_t* src = smem + res_slot_off + (uint32_t)(cbeg >> 3) * plane_bytes + (uint32_t)ri[0].pp * 16u;
#pragma unroll
                            for (int hb = 0; hb < CW / 8; ++hb) unpack8t<FMT>(*reinterpret_cast<const uint4*>(src + hb * plane_bytes), rr + hb * 8);
                        } else if (res_mode == 1) {
#pragma unroll
                            for (int j = 0; j < CW; ++j) rr[j] = __uint_as_float(rv[j]);
                        } else {
#pragma unroll
                            for (int j = 0; j < CW; ++j) rr[j] = 0.f;
                        }
                        const float4* gc = reinterpret_cast<const float4*>(gcoef + cbeg);
                        float sxa = 0.f, sqa = 0.f, sxb = 0.f, sqb = 0.f;
#pragma unroll
                        for (int j = 0; j < CW; j += 2) {
                            const float4 ab = gc[j >> 1];
                            float ya = fmaf(y[j], ab.x, ab.y);
                            float yb = fmaf(y[j + 1], ab.z, ab.w);
                            ya = fast_silu(ya); yb = fast_silu(yb);          // every GroupNorm step of the U-Net is followed by SiLU (unet.py:67)
                            ya += rr[j]; yb += rr[j + 1];
                            y[j] = ya; y[j + 1] = yb;
                            sxa += ya; sqa = fmaf(ya, ya, sqa); sxb += yb; sqb = fmaf(yb, yb, sqb);
                        }
                        psx[0] = sxa + sxb; psq[0] = sqa + sqb;
                        if (is_final) {
                            const int nch = p.channels, dim = p.dim;
#pragma unroll
                            for (int co = 0; co < FINAL_MAX_CH; ++co) {
                                if (co < nch) {
                                    float a = 0.f;
#pragma unroll
                                    for (int j = 0; j < CW; ++j) a = fmaf(y[j], cpar[co * dim + cbeg + j], a);
                                    kacc[0][co] = a;
                                }
                            }
                        } else {
#pragma unroll
                            for (int hb = 0; hb < CW / 8; ++hb) pk[hb] = write8(ri[0], (cbeg >> 3) + hb, y + hb * 8);
                        }
                    };
                    const int ng = cpg >= 16 ? 1 : (cw8 ? 8 : 16) >> lg_cpg;          // groups inside this thread's chunk
                    if (cw8) {
                        if (ng == 2) head(IntTag<8>(), IntTag<2>()); else head(IntTag<8>(), IntTag<1>());
                        if (dbg && et == 0) dbg[i * 8 + 4] = clock64();
                        tail(IntTag<8>());
                    } else {
                        if (ng == 4) head(IntTag<16>(), IntTag<4>());
                        else if (ng == 2) head(IntTag<16>(), IntTag<2>());
                        else head(IntTag<16>(), IntTag<1>());
                        if (dbg && et == 0) dbg[i * 8 + 4] = clock64();
                        tail(IntTag<16>());
                    }
                    if (pn_g >= 0) {
                        // ---- fused PreNorm of the following attention block: GroupNorm(1, C) of the 16-bit result; every warp
                        // holds C/2 (one tile) or C (two tiles) channels of its rows
                        float ps[2];
                        ps[0] = ri[0].valid ? psx[0] : 0.f; ps[1] = ri[0].valid ? psq[0] : 0.f;
                        warp_sum_scatter<2>(ps, lane);
                        if ((lane & 15) == 0) wpart[64 + warp * 2 + (lane >> 4)] = ps[0];
                        epi_sync();
                        float sx = 0.f, sq = 0.f;
                        for (int w = 0; w < EPI_WARPS; ++w) { const float2 a = *reinterpret_cast<const float2*>(wpart + 64 + w * 2); sx += a.x; sq += a.y; }
                        const float icn = fast_rcp((float)(C * HW));
                        const float mean = sx * icn;
                        const float rstd = rsqrtf(fmaxf(sq * icn - mean * mean, 0.f) + 1e-5f);
                        if (ri[0].valid) {
                            uint4* dst = reinterpret_cast<uint4*>(p.gt[pn_g]);
                            const int nhb = cw8 ? 1 : 2;
#pragma unroll
                            for (int hb = 0; hb < 2; ++hb) {
                                if (hb >= nhb) break;
                                const int gcb = (cbeg >> 3) + hb;
                                float xv[8];
                                unpack8t<FMT>(pk[hb], xv);
                                const float4* pp4 = reinterpret_cast<const float4*>(pnpar + cbeg + hb * 8);
#pragma unroll
                                for (int j = 0; j < 8; j += 2) {
                                    const float4 gb = pp4[j >> 1];                       // (gamma, beta) x 2 channels
                                    const float a0 = rstd * gb.x, a1 = rstd * gb.z;
                                    xv[j] = fmaf(xv[j], a0, gb.y - mean * a0); xv[j + 1] = fmaf(xv[j + 1], a1, gb.w - mean * a1);
                                }
                                dst[(size_t)(gcb * geo.B + b0) * HW + ri[0].px] = pack8t<FMT>(xv);
                            }
                        }
                    }
                } else {
                const int pm = (MT == 1 && G == 1 && !is_final) ? 2 : 1;   // partial columns per group in rowstat
                const int GS = G * pm;
                // N-split stages at 2x2 pixels: a sample's 16 padded rows are exactly one half-warp and the CTA's channels one group, so
                // the statistics are four xor-shuffles away, the accumulator chunk stays in registers between the statistics and the
                // normalisation, and the two warp groups (the two channel halves) meet behind ONE barrier -- no per-row partials in
                // shared memory, no coefficient table, no second tensor-memory load.
                bool fast2 = false;
                if constexpr (SPLIT && MT == 1)
                    fast2 = G == 1 && geo.PP == 16 && !is_final && (cend - cbeg == 8 || cend - cbeg == 16);
                bool fast3 = false;
                if constexpr (!SPLIT && MT == 1 && WIDE)
                    fast3 = geo.H == 4 && geo.W == 4 && geo.nb <= 3 && !is_final && (cpg == 8 || cpg == 16) && ((cend - cbeg) & 15) == 0 &&
                            cend > cbeg;
                if (fast2) {
                    if (dbg && et == 0) dbg[i * 8 + 3] = clock64();
                    auto body = [&](auto cw_tag) {
                        constexpr int CW = decltype(cw_tag)::value;
                        uint32_t av[CW];
                        const uint32_t ta = tlane + (uint32_t)(acc_col + cbeg);
                        if constexpr (CW == 16) tmem_ld16_issue(ta, av); else tmem_ld8_issue(ta, av);
                        tmem_ld_wait();
                        const bool valid = ri[0].valid;
                        float s0 = 0.f, q0 = 0.f, s1 = 0.f, q1 = 0.f;
#pragma unroll
                        for (int j = 0; j < CW; j += 2) {
                            const float xa = __uint_as_float(av[j]), xb = __uint_as_float(av[j + 1]);
                            s0 += xa; q0 = fmaf(xa, xa, q0); s1 += xb; q1 = fmaf(xb, xb, q1);
                        }
                        float sx = valid ? s0 + s1 : 0.f, sq = valid ? q0 + q1 : 0.f;
#pragma unroll
                        for (int o = 8; o > 0; o >>= 1) { sx += __shfl_xor_sync(0xffffffffu, sx, o); sq += __shfl_xor_sync(0xffffffffu, sq, o); }
                        float2* const part = reinterpret_cast<float2*>(fastbuf);          // [2 warp groups][8 samples]
                        const int sl = r >> 4;                                             // sample of this row inside the CTA
                        if ((lane & 15) == 0) part[wg * 8 + sl] = make_float2(sx, sq);
                        epi_sync();
                        if (dbg && et == 0) dbg[i * 8 + 4] = clock64();
                        uint32_t rv[CW];
                        if (res_mode == 1) {
                            const uint32_t tr = tlane + (uint32_t)(res_col + cbeg);
                            if constexpr (CW == 16) tmem_ld16_issue(tr, rv); else tmem_ld8_issue(tr, rv);
                            tmem_ld_wait();
                        }
                        if (!valid) return;
                        const float2 pa = part[sl], pb = part[8 + sl];
                        const float icnt = fast_rcp((float)(C * HW));
                        const float mean = (pa.x + pb.x) * icnt;
                        const float rstd = rsqrtf(fmaxf((pa.y + pb.y) * icnt - mean * mean, 0.f) + 1e-5f);
                        float rr[CW];
                        if (res_mode == 2) {
                            const uint8_t* src = smem + res_slot_off + (uint32_t)((c0 + cbeg) >> 3) * plane_bytes + (uint32_t)ri[0].pp * 16u;
#pragma unroll
                            for (int hb = 0; hb < CW / 8; ++hb) unpack8t<FMT>(*reinterpret_cast<const uint4*>(src + hb * plane_bytes), rr + hb * 8);
                        } else if (res_mode == 1) {
#pragma unroll
                            for (int j = 0; j < CW; ++j) rr[j] = __uint_as_float(rv[j]);
                        } else {
#pragma unroll
                            for (int j = 0; j < CW; ++j) rr[j] = 0.f;
                        }
                        // FiLM(GroupNorm(x)) = x a + b with a = rstd gamma (1 + scale), b = (beta - mean rstd gamma)(1 + scale) + shift
                        const float4* gp = reinterpret_cast<const float4*>(gpar + cbeg);                    // (gamma, beta) x 2 channels
                        const float4* cf = reinterpret_cast<const float4*>(coef + ri[0].s * C + cbeg);      // (1 + scale, shift) x 2 channels
                        float v[CW];
                        float sxa = 0.f, sqa = 0.f, sxb = 0.f, sqb = 0.f;
#pragma unroll
                        for (int j = 0; j < CW; j += 2) {
                            const float4 gb = gp[j >> 1], f = cf[j >> 1];
                            float a0 = rstd * gb.x, b0 = gb.y - mean * a0, a1 = rstd * gb.z, b1 = gb.w - mean * a1;
                            a0 *= f.x; b0 = fmaf(b0, f.x, f.y); a1 *= f.z; b1 = fmaf(b1, f.z, f.w);
                            float ya = fmaf(__uint_as_float(av[j]), a0, b0);
                            float yb = fmaf(__uint_as_float(av[j + 1]), a1, b1);
                            ya = fast_silu(ya); yb = fast_silu(yb);
                            ya += rr[j]; yb += rr[j + 1];
                            v[j] = ya; v[j + 1] = yb;
                            sxa += ya; sqa = fmaf(ya, ya, sqa); sxb += yb; sqb = fmaf(yb, yb, sqb);
                        }
                        psx[0] += sxa + sxb; psq[0] += sqa + sqb;
#pragma unroll
                        for (int hb = 0; hb < CW / 8; ++hb) write8(ri[0], ((c0 + cbeg) >> 3) + hb, v + hb * 8);
                    };
                    if (cw8) body(IntTag<8>()); else body(IntTag<16>());
                } else if (fast3) {
                    // 4x4 pixels, up to three samples per CTA: the valid rows of sample s (padded positions 36 s + 7 ..) all lie in
                    // warp s of each warp group, and a 16-channel chunk holds whole groups -- so a (sample, group) sum is one warp
                    // butterfly away and every chunk is normalised out of registers with no barrier at all.
                    if (dbg && et == 0) dbg[i * 8 + 3] = clock64();
                    const bool valid = ri[0].valid;
                    const float icnt = fast_rcp((float)(cpg * HW));
                    for (int c = cbeg; c < cend; c += 16) {
                        uint32_t av[16], rv[16];
                        tmem_ld16_issue(tlane + (uint32_t)(acc_col + c), av);
                        if (res_mode == 1) tmem_ld16_issue(tlane + (uint32_t)(res_col + c), rv);
                        tmem_ld_wait();
                        // partial sums of the chunk's groups: one group of 16 channels, or two of 8
                        float s0 = 0.f, q0 = 0.f, s1 = 0.f, q1 = 0.f;
#pragma unroll
                        for (int j = 0; j < 8; ++j) {
                            const float xa = __uint_as_float(av[j]), xb = __uint_as_float(av[8 + j]);
                            s0 += xa; q0 = fmaf(xa, xa, q0); s1 += xb; q1 = fmaf(xb, xb, q1);
                        }
                        if (!valid) { s0 = 0.f; q0 = 0.f; s1 = 0.f; q1 = 0.f; }
                        if (cpg == 16) { s0 += s1; q0 += q1; }
#pragma unroll
                        for (int o = 16; o > 0; o >>= 1) {
                            s0 += __shfl_xor_sync(0xffffffffu, s0, o); q0 += __shfl_xor_sync(0xffffffffu, q0, o);
                            if (cpg == 8) { s1 += __shfl_xor_sync(0xffffffffu, s1, o); q1 += __shfl_xor_sync(0xffffffffu, q1, o); }
                        }
                        if (!valid) continue;
                        const float m0 = s0 * icnt, r0 = rsqrtf(fmaxf(q0 * icnt - m0 * m0, 0.f) + 1e-5f);
                        float m1 = m0, r1 = r0;
                        if (cpg == 8) { m1 = s1 * icnt; r1 = rsqrtf(fmaxf(q1 * icnt - m1 * m1, 0.f) + 1e-5f); }
                        float rr[16];
                        if (res_mode == 2) {
                            const uint8_t* src = smem + res_slot_off + (uint32_t)(c >> 3) * plane_bytes + (uint32_t)ri[0].pp * 16u;
#pragma unroll
                            for (int hb = 0; hb < 2; ++hb) unpack8t<FMT>(*reinterpret_cast<const uint4*>(src + hb * plane_bytes), rr + hb * 8);
                        } else if (res_mode == 1) {
#pragma unroll
                            for (int j = 0; j < 16; ++j) rr[j] = __uint_as_float(rv[j]);
                        } else {
#pragma unroll
                            for (int j = 0; j < 16; ++j) rr[j] = 0.f;
                        }
                        const float4* gp = reinterpret_cast<const float4*>(gpar + c);
                        const float4* cf = reinterpret_cast<const float4*>(coef + ri[0].s * C + c);
                        float v[16];
                        float sxa = 0.f, sqa = 0.f, sxb = 0.f, sqb = 0.f;
#pragma unroll
                        for (int j = 0; j < 16; j += 2) {
                            const float mean = j < 8 ? m0 : m1, rstd = j < 8 ? r0 : r1;
                            const float4 gb = gp[j >> 1], f = cf[j >> 1];
                            float a0 = rstd * gb.x, b0 = gb.y - mean * a0, a1 = rstd * gb.z, b1 = gb.w - mean * a1;
                            a0 *= f.x; b0 = fmaf(b0, f.x, f.y); a1 *= f.z; b1 = fmaf(b1, f.z, f.w);
                            float ya = fmaf(__uint_as_float(av[j]), a0, b0);
                            float yb = fmaf(__uint_as_float(av[j + 1]), a1, b1);
                            ya = fast_silu(ya); yb = fast_silu(yb);
                            ya += rr[j]; yb += rr[j + 1];
                            v[j] = ya; v[j + 1] = yb;
                            sxa += ya; sqa = fmaf(ya, ya, sqa); sxb += yb; sqb = fmaf(yb, yb, sqb);
                        }
                        psx[0] += sxa + sxb; psq[0] += sqa + sqb;
#pragma unroll
                        for (int hb = 0; hb < 2; ++hb) write8(ri[0], (c >> 3) + hb, v + hb * 8);
                    }
                    if (dbg && et == 0) dbg[i * 8 + 4] = clock64();
                } else {
                // pass 1: per-row (sum, sumsq) per group
                {
                    float run_sx = 0.f, run_sq = 0.f;
                    for_chunks([&](int k, int c, auto tag) {
                        constexpr int CW = decltype(tag)::value;
                        uint32_t u[CW];
                        const uint32_t ta = tlane + (uint32_t)(acc_col + tile_of(k) * C + c);
                        if constexpr (CW == 16) tmem_ld16_issue(ta, u); else tmem_ld8_issue(ta, u);
                        tmem_ld_wait();
                        float2* rs = rowstat + (size_t)(tile_of(k) * 128 + r) * GS;
                        const bool valid = ri[k].valid;
                        if (cpg == 4) {
#pragma unroll
                            for (int q = 0; q < CW / 4; ++q) {
                                float sx = 0.f, sq = 0.f;
#pragma unroll
                                for (int j = 0; j < 4; ++j) { const float xv = __uint_as_float(u[q * 4 + j]); sx += xv; sq = fmaf(xv, xv, sq); }
                                rs[(c >> 2) + q] = valid ? make_float2(sx, sq) : make_float2(0.f, 0.f);
                            }
                        } else if (cpg == 8) {
#pragma unroll
                            for (int q = 0; q < CW / 8; ++q) {
                                float sx = 0.f, sq = 0.f;
#pragma unroll
                                for (int j = 0; j < 8; ++j) { const float xv = __uint_as_float(u[q * 8 + j]); sx += xv; sq = fmaf(xv, xv, sq); }
                                rs[(c >> 3) + q] = valid ? make_float2(sx, sq) : make_float2(0.f, 0.f);
                            }
                        } else {
                            float sx0 = 0.f, sq0 = 0.f, sx1 = 0.f, sq1 = 0.f;
#pragma unroll
                            for (int j = 0; j < CW; j += 2) {
                                const float xa = __uint_as_float(u[j]), xb = __uint_as_float(u[j + 1]);
                                sx0 += xa; sq0 = fmaf(xa, xa, sq0); sx1 += xb; sq1 = fmaf(xb, xb, sq1);
                            }
                            run_sx += sx0 + sx1; run_sq += sq0 + sq1;
                            if (((c + CW) & (cpg - 1)) == 0 || c + CW == cend) {
                                rs[pm == 2 ? wg : (c >> lg_cpg)] = valid ? make_float2(run_sx, run_sq) : make_float2(0.f, 0.f);
                                run_sx = 0.f; run_sq = 0.f;
                            }
                        }
                    });
                }
                if (dbg && et == 0) dbg[i * 8 + 3] = clock64();
                stats_to_coef(geo, MT * 128, rowstat, coef, gpar, G, pm, C, HW, true, et);
                if (dbg && et == 0) dbg[i * 8 + 4] = clock64();
                // pass 2: y = x*scale + offset, SiLU, + residual, write
                for_chunks([&](int k, int c, auto tag) {
                    constexpr int CW = decltype(tag)::value;
                    uint32_t av[CW], rv[CW];
                    const int t = tile_of(k);
                    if constexpr (CW == 16) {
                        tmem_ld16_issue(tlane + (uint32_t)(acc_col + t * C + c), av);
                        if (res_mode == 1) tmem_ld16_issue(tlane + (uint32_t)(res_col + t * C + c), rv);
                    } else {
                        tmem_ld8_issue(tlane + (uint32_t)(acc_col + t * C + c), av);
                        if (res_mode == 1) tmem_ld8_issue(tlane + (uint32_t)(res_col + t * C + c), rv);
                    }
                    tmem_ld_wait();
                    if (!ri[k].valid) return;
                    float rr[CW];
                    if (res_mode == 2) {
                        const uint8_t* src = smem + res_slot_off + (uint32_t)((c0 + c) >> 3) * plane_bytes + (uint32_t)ri[k].pp * 16u;
#pragma unroll
                        for (int hb = 0; hb < CW / 8; ++hb) unpack8t<FMT>(*reinterpret_cast<const uint4*>(src + hb * plane_bytes), rr + hb * 8);
                    } else if (res_mode == 1) {
#pragma unroll
                        for (int j = 0; j < CW; ++j) rr[j] = __uint_as_float(rv[j]);
                    } else {
#pragma unroll
                        for (int j = 0; j < CW; ++j) rr[j] = 0.f;
                    }
                    const float4* cf = reinterpret_cast<const float4*>(coef + ri[k].s * C + c);
                    float v[CW];
                    float sxa = 0.f, sqa = 0.f, sxb = 0.f, sqb = 0.f;
#pragma unroll
                    for (int j = 0; j < CW; j += 2) {
                        const float4 ab = cf[j >> 1];
                        float ya = fmaf(__uint_as_float(av[j]), ab.x, ab.y);
                        float yb = fmaf(__uint_as_float(av[j + 1]), ab.z, ab.w);
                        ya = fast_silu(ya); yb = fast_silu(yb);          // every GroupNorm step of the U-Net is followed by SiLU (unet.py:67)
                        ya += rr[j]; yb += rr[j + 1];
                        v[j] = ya; v[j + 1] = yb;
                        sxa += ya; sqa = fmaf(ya, ya, sqa); sxb += yb; sqb = fmaf(yb, yb, sqb);
                    }
                    psx[k] += sxa + sxb; psq[k] += sqa + sqb;
                    if (is_final) {
                        const int nch = p.channels, dim = p.dim;
#pragma unroll
                        for (int co = 0; co < FINAL_MAX_CH; ++co) {
                            if (co < nch) {
                                float a = kacc[k][co];
#pragma unroll
                                for (int j = 0; j < CW; ++j) a = fmaf(v[j], cpar[co * dim + c + j], a);
                                kacc[k][co] = a;
                            }
                        }
                    } else {
#pragma unroll
                        for (int hb = 0; hb < CW / 8; ++hb) write8(ri[k], ((c0 + c) >> 3) + hb, v + hb * 8);
                    }
                });
                }
                if (pn_g >= 0) {
                    // ---- fused PreNorm of the following attention block: GroupNorm(1, C) of the 16-bit result
                    const int pm2 = (MT == 1) ? 2 : 1;
                    // (rowstat and gpar were last read before the final barrier of the block-norm stats_to_coef; coef is
                    // rewritten only behind the first barrier of the next one, which every thread reaches after its pass 2)
#pragma unroll
                    for (int k = 0; k < TW; ++k) {
                        if (MT > 1 && wg + 2 * k >= MT) continue;
                        const int t = tile_of(k);
                        rowstat[(size_t)(t * 128 + r) * pm2 + (pm2 == 2 ? wg : 0)] = ri[k].valid ? make_float2(psx[k], psq[k]) : make_float2(0.f, 0.f);
                    }
                    stats_to_coef(geo, MT * 128, rowstat, coef, pnpar, 1, pm2, C, HW, false, et, &xc);
                    uint4* dst = reinterpret_cast<uint4*>(p.gt[pn_g]);
                    for_chunks([&](int k, int c, auto tag) {
                        constexpr int CW = decltype(tag)::value;
                        if (!ri[k].valid) return;
                        const int b = b0 + ri[k].s;
                        const float4* cf = reinterpret_cast<const float4*>(coef + ri[k].s * C + c);
#pragma unroll
                        for (int hb = 0; hb < CW / 8; ++hb) {
                            const int gcb = ((c0 + c) >> 3) + hb;
                            float xv[8];
                            unpack8t<FMT>(*reinterpret_cast<const uint4*>(smem + out_slot_off + (uint32_t)gcb * plane_bytes + (uint32_t)ri[k].pp * 16u), xv);
#pragma unroll
                            for (int j = 0; j < 8; j += 2) {
                                const float4 ab = cf[hb * 4 + (j >> 1)];
                                xv[j] = fmaf(xv[j], ab.x, ab.y); xv[j + 1] = fmaf(xv[j + 1], ab.z, ab.w);
                            }
                            dst[(size_t)(gcb * geo.B + b) * HW + ri[k].px] = pack8t<FMT>(xv);
                        }
                    });
                }
                }
                if (is_final) {
                    if (sg.flags & SF_CFG_2B) final_update_2b(kacc, cend > cbeg);
                    else if (cend > cbeg) final_update(kacc);
                }
                if (is_final) {
                    // the last CTA to finish advances the stage counter (every CTA has read ctrl->step by now)
                    epi_sync();
                    if (et == 0) {
                        __threadfence();
                        const int done = atomicAdd(&ctrl->done_ctr, 1);
                        if (done == (int)gridDim.x - 1) {
                            ctrl->done_ctr = 0;
                            ctrl->step = step_idx + 1;
                            __threadfence();
                        }
                    }
                }
            }
            if (dbg && et == 0) dbg[i * 8 + 5] = clock64();
            tc_fence_before();
            if (!SPLIT) {                 // (N-split: the stores of write8 complete the consumers' barriers as they land)
                fence_proxy_async();      // shared-memory results -> visible to the next step's tcgen05.mma
                if (i + 1 < n_steps) named_bar_arrive(2, EPI_THREADS + 32);
            }
        }
    }
    tc_fence_before();
    __syncthreads();
    if (Q > 1) cluster_sync_all();       // no CTA may exit while a peer can still store into its shared memory
    if (dbg && tid == 0) dbg[CH_MAX_STEPS * 8 + 1] = clock64();
    if (p.dbg && tid == 0) { if (blockIdx.x == 0) p.dbg[102] = global_ns(); atomicMax(reinterpret_cast<unsigned long long*>(p.dbg + 103), (unsigned long long)global_ns()); }
    if (warp == W_MMA) tmem_dealloc(tmem_base, (uint32_t)tmem_cols);
}

cudaError_t attn_configure();
template <int MT, bool SPLIT, bool FAST>
static cudaError_t chain_attr() {
    cudaError_t e = cudaFuncSetAttribute(k_chain<MT, SPLIT, 0, FAST>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_chain<MT, SPLIT, 1, FAST>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    return e;
}
template <int MT, int ENDS>
static cudaError_t fast_ends_attr() {
    cudaError_t e = cudaFuncSetAttribute(k_chain<MT, false, 0, true, false, ENDS>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_chain<MT, false, 1, true, false, ENDS>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    return e;
}
cudaError_t fused_configure() {
    cudaError_t e = chain_attr<1, false, false>();
    if (e == cudaSuccess) e = chain_attr<1, true, false>();
    if (e == cudaSuccess) e = chain_attr<2, false, false>();
    if (e == cudaSuccess) e = chain_attr<3, false, false>();
    if (e == cudaSuccess) e = chain_attr<4, false, false>();
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_chain<1, true, 0, false, false, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_chain<1, true, 1, false, false, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_chain<1, false, 0, false, true, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_chain<1, false, 1, false, true, 0>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e == cudaSuccess) e = fast_ends_attr<1, 0>();
    if (e == cudaSuccess) e = fast_ends_attr<1, 1>();
    if (e == cudaSuccess) e = fast_ends_attr<1, 2>();
    if (e == cudaSuccess) e = fast_ends_attr<2, 0>();
    if (e == cudaSuccess) e = fast_ends_attr<2, 1>();
    if (e == cudaSuccess) e = fast_ends_attr<2, 2>();
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_chain<1, false, 0, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(k_chain<1, false, 1, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024);
    if (e != cudaSuccess) return e;
    return attn_configure();
}

cudaError_t launch_pdl(const void* fn, int grid, int block, size_t smem, cudaStream_t s, void** args, int cluster) {
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3((unsigned)grid); cfg.blockDim = dim3((unsigned)block); cfg.dynamicSmemBytes = smem; cfg.stream = s;
    cudaLaunchAttribute at[2];
    int n = 0;
    at[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;     // programmatic dependent launch between the stage kernels
    at[n].val.programmaticStreamSerializationAllowed = 1;
    ++n;
    if (cluster > 1) {
        at[n].id = cudaLaunchAttributeClusterDimension;
        at[n].val.clusterDim.x = (unsigned)cluster; at[n].val.clusterDim.y = 1; at[n].val.clusterDim.z = 1;
        ++n;
    }
    cfg.attrs = at; cfg.numAttrs = n;
    return cudaLaunchKernelExC(&cfg, fn, args);
}

// How many clusters of `nsplit` k_chain<1, true> CTAs with `smem_bytes` of dynamic shared memory the device keeps resident
// at once (clusters must sit inside one GPC, so this is less than SMs / nsplit: 148 SMs hold 32-36 clusters of four, not 37).
// Returns -1 when the query is not available; the caller then falls back to the SM-count estimate.
int fused_max_active_clusters(int nsplit, int smem_bytes) {
    if (nsplit <= 1) return -1;
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3((unsigned)(nsplit * 64)); cfg.blockDim = dim3((unsigned)FUSED_THREADS); cfg.dynamicSmemBytes = (size_t)smem_bytes;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = (unsigned)nsplit; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    int n = 0;
    if (cudaOccupancyMaxActiveClusters(&n, (const void*)k_chain<1, true, 1, false>, &cfg) != cudaSuccess) { cudaGetLastError(); return -1; }
    return n;
}

template <int FMT>
static const void* chain_fn(int mt, bool split, bool fast, bool wide, int ends) {
    if (ends == 0 && !fast && mt == 1) {
        if (split) return (const void*)k_chain<1, true, FMT, false, false, 0>;
        if (!split && wide) return (const void*)k_chain<1, false, FMT, false, true, 0>;
    }
    if (wide && !fast && !split && mt == 1) return (const void*)k_chain<1, false, FMT, false, true>;
    if (fast) {
        if (split || mt > 2) return nullptr;
        if (ends == 0) return mt == 1 ? (const void*)k_chain<1, false, FMT, true, false, 0> : (const void*)k_chain<2, false, FMT, true, false, 0>;
        if (ends == 1) return mt == 1 ? (const void*)k_chain<1, false, FMT, true, false, 1> : (const void*)k_chain<2, false, FMT, true, false, 1>;
        if (ends == 2) return mt == 1 ? (const void*)k_chain<1, false, FMT, true, false, 2> : (const void*)k_chain<2, false, FMT, true, false, 2>;
        return nullptr;          // no stage holds both the init conv and the final conv (fused_plan.inc)
    }
    switch (mt) {
        case 1: return split ? (const void*)k_chain<1, true, FMT, false> : (const void*)k_chain<1, false, FMT, false>;
        case 2: return (const void*)k_chain<2, false, FMT, false>;
        case 3: return (const void*)k_chain<3, false, FMT, false>;
        case 4: return (const void*)k_chain<4, false, FMT, false>;
        default: return nullptr;
    }
}
cudaError_t launch_chain(const ChainParams& p, const CUtensorMap* maps, int grid, cudaStream_t s) {
    if (p.nsplit > 1 && p.n_mtiles != 1) return cudaErrorInvalidValue;
    int ends = 0;
    for (int i = 0; i < p.n_steps; ++i) ends |= (p.st[i].epi == CE_INIT ? 1 : 0) | (p.st[i].final != 0 ? 2 : 0);
    const void* fn = p.fmt ? chain_fn<1>(p.n_mtiles, p.nsplit > 1, p.fast != 0, p.wide != 0, ends)
                           : chain_fn<0>(p.n_mtiles, p.nsplit > 1, p.fast != 0, p.wide != 0, ends);
    if (!fn) return cudaErrorInvalidValue;
    void* args[5] = {(void*)&maps[0], (void*)&maps[1], (void*)&maps[2], (void*)&maps[3], (void*)&p};
    return launch_pdl(fn, grid * p.nsplit, FUSED_THREADS, (size_t)p.smem_bytes, s, args, p.nsplit);
}

}  // namespace flo
