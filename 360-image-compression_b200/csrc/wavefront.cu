// Wavefront engine of the fused decoder.  Replaces the 12 CconvDc launches (+5 TileAdd) that the reference issues per
// wavefront step (test/lic360_demo.py:201-209,226-234; cconv_dc_cuda.cu:108-137; tile_add_cuda.cu:40-61).
//
// A decoder step p is strictly sequential across layers only through the SAME-wavefront terms (Q) of each layer, at
// most 25*cin_g MACs per output.  The canonical arithmetic (conv.cu header) therefore splits every output into
//     out = ((P + R) + Q) + bias
//   P : "old" terms, inputs of wavefronts <= p-2       -> wf_old_kernel : ALL 12 layers in one launch, fed by TMA box
//                                                         loads; launched for step p+1 on a side branch of step p's
//                                                         graph, i.e. off the critical path (it only needs data that is
//                                                         complete before step p starts)
//   R : inputs of wavefront p-1 (available at step start) -> wf_prev_kernel: all 12 layers in one launch
//   Q : inputs of wavefront p (the layer below, this step) -> wf_chain_kernel: one thread-block cluster per net walks
//                                                         the 12 layers with a cluster barrier between layers; bias,
//                                                         PReLU and the residual add (TileAdd) are fused here
// so the critical path of a step is  scatter -> R -> chain -> CDF rows  instead of 12 dependent full-size launches.
#include <algorithm>
#include <cooperative_groups.h>
#include <vector>
#include "conv_dev.cuh"
#include "tables_dev.cuh"
#include "wavefront.cuh"

namespace cg = cooperative_groups;

namespace lic360 {

WF_TRACE_DECL
void wf_trace_set(unsigned long long* buf, int sel) {
    cudaMemcpyToSymbol(g_wf_trace, &buf, sizeof(buf));
    cudaMemcpyToSymbol(g_wf_trace_sel, &sel, sizeof(sel));
}

// ------------------------------------------------------------------------------------------------ TMA / mbarrier
// The inner (h) coordinate of a TMA box must be 16-byte aligned (4 floats; an unaligned start faults with "illegal
// instruction" on sm_100, tools/tma_probe.cu), so the box starts at (hbase - 2) rounded down to 4 and is 40 wide.
constexpr int WF_BOX_W = 40;
constexpr int WF_BAND = 9 * WF_BOX_W;                 // cells per channel
#ifndef WF_STAGE_CH
#define WF_STAGE_CH 4
#endif
constexpr int WF_STAGE = WF_STAGE_CH;                 // input channels per TMA stage
constexpr int WF_BAND_BYTES = WF_STAGE * WF_BAND * 4;  // 5760 for 4 channels
constexpr int WF_STAGE_BYTES = ((WF_BAND_BYTES + WF_STAGE * TAPS * 16 + 127) / 128) * 128;  // band + weights, multiple of 128

__device__ __forceinline__ void mbar_init(unsigned bar, int count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;\n" ::"r"(bar), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(unsigned bar, int bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(unsigned bar, unsigned parity) {
    unsigned ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n"
        : "=r"(ok)
        : "r"(bar), "r"(parity)
        : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(unsigned bar, unsigned parity) {
    while (!mbar_try_wait(bar, parity)) {}
}
__device__ __forceinline__ void tma_load_3d(unsigned dst, const CUtensorMap* tm, int c0, int c1, int c2, unsigned bar) {
    asm volatile("cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];\n"
                 ::"r"(dst), "l"(tm), "r"(c0), "r"(c1), "r"(c2), "r"(bar) : "memory");
}
__device__ __forceinline__ void bulk_load(unsigned dst, const void* src, int bytes, unsigned bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];\n"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}

// CTA geometry shared by the old-term and previous-wavefront kernels:
//   blockIdx.x -> (diagonal of the slab, 32-position part), blockIdx.y -> 4-channel output chunk inside the group,
//   blockIdx.z -> (layer, net)
struct WfTile { int l, n, kc, psum, d, hbase, hmax, tc; bool ok; };

__device__ __forceinline__ WfTile wf_tile(const WfNetDev& net, int dp, int l0 = 0, bool swapped = false) {
    WfTile t;
    const int bx = swapped ? blockIdx.z : blockIdx.x, bz = swapped ? blockIdx.x : blockIdx.z;
    t.l = l0 + bz / net.nsets;
    t.n = bz % net.nsets;
    t.kc = blockIdx.y;
    t.psum = *net.ctr + dp;
    t.ok = t.kc < net.L[t.l].cpg4 && t.psum < net.nsteps;
    const int la = max(0, t.psum - net.G + 1), lb = min(t.psum, net.H + net.W - 2);
    t.d = la + bx / net.parts;
    t.ok = t.ok && t.d <= lb;
    const int hmin = max(0, t.d - net.W + 1);
    t.hmax = min(net.H - 1, t.d);
    t.hbase = hmin + (bx % net.parts) * 32;
    t.ok = t.ok && t.hbase <= t.hmax;
    t.tc = t.psum - t.d;
    return t;
}

// ------------------------------------------------------------------------------------------------ old terms (P)
// CTA = 32 consecutive positions of one anti-diagonal x one 4-channel output chunk x (layer, net); its 4 warps share
// out the canonical 16-channel input blocks that have old terms for this output group.  Per stage of 4 input channels ONE 3-D TMA box {36 h, 9 d, 4 c} of the planar skewed frame
// (out-of-image cells zero-filled by the TMA unit: no index math, no bounds checks) plus one bulk copy of the stage's
// 100 float4 weights land in the warp's private shared-memory slice and complete on the warp's own mbarrier.
constexpr int WF_OLD_WARPS = 4;  // warps per CTA; warp w walks the canonical blocks w, w+4, ... that have old terms

__global__ void __launch_bounds__(32 * WF_OLD_WARPS) wf_old_kernel(const __grid_constant__ WfNetDev net,
                                                                  const __grid_constant__ WfMaps maps, int dp) {
    extern __shared__ unsigned char wf_raw[];
    // grid = ((layer, net), chunk, (diagonal, part)): CTAs are dispatched x-fastest, so the tiles of the LARGEST output
    // groups (most old terms) of every layer start first and the light ones fill the tail
    const WfTile t = wf_tile(net, dp, 0, true);
    if (!t.ok) return;  // CTA-uniform
    if (threadIdx.x == 0 && threadIdx.y == 0) WF_TRACE_MIN(net.G, t.psum - dp, WF_TR_OLD0);
    const WfLayerDev& L = net.L[t.l];
    const unsigned raw_s = (unsigned)__cvta_generic_to_shared(wf_raw);
    unsigned char* base = wf_raw + ((128u - (raw_s & 127u)) & 127u);                            // 128-B aligned
    float4* part = reinterpret_cast<float4*>(base + (size_t)WF_OLD_WARPS * WF_STAGE_BYTES);    // [nblk][32]
    unsigned long long* bars = reinterpret_cast<unsigned long long*>(part + L.nblk * 32);      // [WF_OLD_WARPS]
    const int lane = threadIdx.x, seg = threadIdx.y;
    float* band = reinterpret_cast<float*>(base + (size_t)seg * WF_STAGE_BYTES);
    float4* wsm = reinterpret_cast<float4*>(band + WF_STAGE * WF_BAND);
    const unsigned band_s = (unsigned)__cvta_generic_to_shared(band);
    const unsigned wsm_s = band_s + WF_BAND_BYTES;
    const int h0 = (t.hbase - 2 + WF_HSHIFT) & ~3;   // aligned box start, in frame columns (row h = column h + WF_HSHIFT)
    const float* bandl = band + (t.hbase - 2 + WF_HSHIFT - h0);
    const unsigned bar = (unsigned)__cvta_generic_to_shared(bars + seg);
    if (lane == 0) {
        mbar_init(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    __syncthreads();
    const int Cin = L.Cin;
    const int lim = min(Cin, (t.tc + 3) * L.cin_g);  // old terms: g_in <= tc + 2
    const int nact = (lim + CB - 1) / CB;            // canonical blocks that have old terms
    const int chunk = t.tc * L.cpg4 + t.kc;
    unsigned phase = 0;
    for (int j = seg; j < nact; j += WF_OLD_WARPS) {
        float4 u = make_float4(0.f, 0.f, 0.f, 0.f);
        const int cb = min(CB, Cin - j * CB);
        const float4* wp4 = reinterpret_cast<const float4*>(L.wp) + (((size_t)t.n * L.nchunk + chunk) * Cin + j * CB) * TAPS;
        for (int c0 = 0; c0 < cb && j * CB + c0 < lim; c0 += WF_STAGE) {
            const int nc = min(WF_STAGE, cb - c0);
            __syncwarp();  // every lane is done with the previous stage
            if (lane == 0) {
                mbar_expect_tx(bar, WF_BAND_BYTES + nc * TAPS * 16);
                tma_load_3d(band_s, &maps.tm[t.l], h0, t.d - 4, t.n * Cin + j * CB + c0, bar);
                bulk_load(wsm_s, wp4 + c0 * TAPS, nc * TAPS * 16, bar);
            }
            mbar_wait(bar, phase);
            phase ^= 1;
            dc_stage_fma<1, WF_BOX_W, WF_BAND>(bandl, wsm, nc, lane, j * CB + c0, L.cin_g, t.tc, u);
        }
        part[j * 32 + lane] = u;
    }
    __syncthreads();
    const int h = t.hbase + lane;
    if (seg == 0 && h <= t.hmax) {
        float4 P = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int j = 0; j < nact; j++) {  // blocks without old terms add nothing (the encoder skips them too)
            const float4 v = part[j * 32 + lane];
            P.x = P.x + v.x; P.y = P.y + v.y; P.z = P.z + v.z; P.w = P.w + v.w;
        }
        L.pbuf[t.psum & 1][(((size_t)t.n * L.cpg4 + t.kc) * net.D + t.d) * net.HS + h] = P;
    }
    if (threadIdx.x == 0 && threadIdx.y == 0) WF_TRACE_MAX(net.G, t.psum - dp, WF_TR_OLD1);
}

// ------------------------------------------------------------------------------------------------ old terms, 4 positions / lane
// The old-term kernels are bound by shared-memory load wavefronts, and a two-positions-per-lane form spends 50 of its 88 per channel on
// the 25 weight vectors.  Here a warp takes TWO neighbouring diagonals of the slab -- output groups tc and tc - 1 -- 64 positions each:
// 16 lanes per diagonal, four adjacent positions per lane (dc_taps_fma4).  Both diagonals read the SAME input channels around the same
// rows, one diagonal apart: one TMA box {72 h, 10 d, 2 c} serves both (the second half-warp's band rows are one further down), and
// each half-warp reads its own group's weight vector with a single LDS.128 (two addresses per instruction cost what a broadcast
// costs).  114 wavefronts per channel for 400 packed FMAs instead of 88 for 200.  The lower group has fewer old terms: its missing
// tap rows and its missing last input group are zero in the packed weights (x * 0 added to an accumulator changes nothing), and its
// block sums beyond its own count are left out of the canonical sum like everywhere else.  Needs one output chunk per group.
constexpr int WF4_STAGE = 2;
constexpr int WF4_BOX_W = 72;
constexpr int WF4_ROWS = 10;
constexpr int WF4_BAND = WF4_ROWS * WF4_BOX_W;
constexpr int WF4_BAND_BYTES = WF4_STAGE * WF4_BAND * 4;
constexpr int WF4_W_BYTES = WF4_STAGE * TAPS * 16;  // weight vectors of one half-warp's group
constexpr int WF4_STAGE_BYTES = ((WF4_BAND_BYTES + 2 * WF4_W_BYTES + 127) / 128) * 128;

__global__ void __launch_bounds__(32 * WF_OLD_WARPS) wf_old4_kernel(const __grid_constant__ WfNetDev net,
                                                                   const __grid_constant__ WfMaps maps, int dp, int parts4, int psum_x,
                                                                   const int* __restrict__ scat_done) {
    extern __shared__ unsigned char wf_raw[];
    // grid = ((layer, net), 1, (diagonal pair, part)), x fastest: the heaviest output groups of every layer start first
    const int bx = blockIdx.z, bz = blockIdx.x;
    const int l = bz / net.nsets, n = bz % net.nsets;
    const int psum = psum_x >= 0 ? psum_x : *net.ctr + dp;  // explicit step: persistent decode (the host paces the steps)
    if (psum >= net.nsteps) return;
    const int la = max(0, psum - net.G + 1), lb = min(psum, net.H + net.W - 2);
    const int dA = la + 2 * (bx / parts4);  // half-warp 0: diagonal dA, group tcA; half-warp 1: diagonal dA + 1, group tcA - 1
    if (dA > lb) return;
    const bool hasB = dA + 1 <= lb;
    const int hminA = max(0, dA - net.W + 1), hmaxA = min(net.H - 1, dA);
    const int hminB = max(0, dA + 1 - net.W + 1), hmaxB = hasB ? min(net.H - 1, dA + 1) : -1;
    const int hb = (hminA & ~3) + (bx % parts4) * 64;  // a multiple of 4: the lane's four cells are one aligned float4 per band row
    if (hb > max(hmaxA, hmaxB)) return;                // CTA-uniform
    const int tcA = psum - dA;
    if (threadIdx.x == 0 && threadIdx.y == 0) WF_TRACE_MIN(net.G, psum - dp, WF_TR_OLD0);
    if (scat_done && l == 0) {
        // persistent decode: this launch was enqueued right behind the host's go for step psum - 1; layer 0 reads the symbols of steps
        // <= psum - 2, which the chain kernel scatters at the top of step psum - 1 -- normally long done, but not ordered by any stream
        if (threadIdx.x == 0 && threadIdx.y == 0) {
            unsigned long long t0 = 0, t1 = 0;
            for (unsigned spins = 1; reinterpret_cast<const volatile int*>(scat_done)[n] < psum - 1; spins++)
                if ((spins & 0xFFF) == 0) {
                    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
                    if (t0 == 0) t0 = t1;
                    else if (t1 - t0 > 5000000000ull) break;
                }
            __threadfence();
        }
        __syncthreads();
    }
    const WfLayerDev& L = net.L[l];
    const unsigned raw_s = (unsigned)__cvta_generic_to_shared(wf_raw);
    unsigned char* base = wf_raw + ((128u - (raw_s & 127u)) & 127u);                            // 128-B aligned
    float4* part = reinterpret_cast<float4*>(base + (size_t)WF_OLD_WARPS * WF4_STAGE_BYTES);   // [nblk][2 diagonals][64]
    unsigned long long* bars = reinterpret_cast<unsigned long long*>(part + L.nblk * 128);     // [WF_OLD_WARPS]
    const int lane = threadIdx.x, seg = threadIdx.y, half = lane >> 4, l16 = lane & 15;
    float* band = reinterpret_cast<float*>(base + (size_t)seg * WF4_STAGE_BYTES);
    float4* wsm = reinterpret_cast<float4*>(band + WF4_STAGE * WF4_BAND);                      // [half][channel][tap]
    const unsigned band_s = (unsigned)__cvta_generic_to_shared(band);
    const unsigned wsm_s = band_s + WF4_BAND_BYTES;
    // frame column of row hb - 2 is hb - 2 + WF_HSHIFT = hb: the box starts there; band row r + half <-> tap row r of this half's diagonal
    const float* bw0 = band + half * WF4_BOX_W + 4 * l16;
    const float4* wsm_h = wsm + half * (WF4_STAGE * TAPS);
    const unsigned bar = (unsigned)__cvta_generic_to_shared(bars + seg);
    if (lane == 0) {
        mbar_init(bar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    __syncthreads();
    const int Cin = L.Cin;
    const int limA = min(Cin, (tcA + 3) * L.cin_g);              // old terms: g_in <= tc + 2
    const int limB = hasB ? min(Cin, (tcA + 2) * L.cin_g) : 0;
    const int nactA = (limA + CB - 1) / CB, nactB = (limB + CB - 1) / CB;  // canonical blocks that have old terms
    unsigned phase = 0;
    for (int j = seg; j < nactA; j += WF_OLD_WARPS) {
        float4 u[4];
#pragma unroll
        for (int i = 0; i < 4; i++) u[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        const int cb = min(CB, Cin - j * CB);
        const float4* wpA = reinterpret_cast<const float4*>(L.wp) + (((size_t)n * L.nchunk + tcA) * Cin + j * CB) * TAPS;
        const float4* wpB = wpA - (size_t)Cin * TAPS;  // group tcA - 1
        for (int c0 = 0; c0 < cb && j * CB + c0 < limA; c0 += WF4_STAGE) {
            const int nc = min(WF4_STAGE, cb - c0);
            __syncwarp();  // every lane is done with the previous stage
            if (lane == 0) {
                mbar_expect_tx(bar, WF4_BAND_BYTES + (hasB ? 2 : 1) * nc * TAPS * 16);
                tma_load_3d(band_s, &maps.tm[l], hb, dA - 4, n * Cin + j * CB + c0, bar);
                bulk_load(wsm_s, wpA + c0 * TAPS, nc * TAPS * 16, bar);
                if (hasB) bulk_load(wsm_s + WF4_W_BYTES, wpB + c0 * TAPS, nc * TAPS * 16, bar);
            }
            mbar_wait(bar, phase);
            phase ^= 1;
            dc_stage_fma4<WF4_BOX_W, WF4_BAND>(bw0, wsm_h, nc, j * CB + c0, L.cin_g, tcA, u);
        }
#pragma unroll
        for (int i = 0; i < 4; i++) part[j * 128 + half * 64 + 4 * l16 + i] = u[i];
    }
    __syncthreads();
    {   // the block sums in canonical order: one thread per output position (warps 0, 1: diagonal dA; warps 2, 3: diagonal dA + 1)
        const int t = seg * 32 + lane, ho = t >> 6, pos = t & 63, h = hb + pos;
        const int nact = ho ? nactB : nactA, hmin = ho ? hminB : hminA, hmax = ho ? hmaxB : hmaxA;
        if (t < 128 && h >= hmin && h <= hmax) {
            float4 P = make_float4(0.f, 0.f, 0.f, 0.f);
            for (int j = 0; j < nact; j++) {  // blocks without old terms add nothing (the encoder skips them too)
                const float4 v = part[j * 128 + ho * 64 + pos];
                P.x = P.x + v.x; P.y = P.y + v.y; P.z = P.z + v.z; P.w = P.w + v.w;
            }
            L.pbuf[psum & 1][((size_t)n * net.D + dA + ho) * net.HS + h] = P;
        }
    }
    if (threadIdx.x == 0 && threadIdx.y == 0) WF_TRACE_MAX(net.G, psum - dp, WF_TR_OLD1);
}

// ------------------------------------------------------------------------------------------------ R / Q terms
// one canonical 16-channel block (jq) of the previous-wavefront (cls 0) or same-wavefront (cls 1) terms of output
// (d, h, group tc, chunk kc): every tap reads the cin_g channels of ONE input group from the channel-last frame.
// CG: read with ld.global.cg (the chain kernel consumes values produced by other CTAs of its cluster in the same launch).
template <bool CG>
__device__ __forceinline__ float4 wf_ldx4(const float* p) {
    return CG ? __ldcg(reinterpret_cast<const float4*>(p)) : __ldg(reinterpret_cast<const float4*>(p));
}

// The activation and weight loads of a whole kernel row (5 taps x 4 channels) are issued before the row's first FMA:
// these kernels run few warps per SM right after a cluster barrier (cold L1), so one L2 round trip per row instead of one
// per weight vector is the difference between ~1 us and ~15 us per layer.  The FMA order is the canonical one.
template <bool CG>
__device__ __forceinline__ float4 wf_rq_partial(const WfNetDev& net, const WfLayerDev& L, int n, int d, int h, int tc, int kc,
                                                int jq, int cls) {
    float4 u = make_float4(0.f, 0.f, 0.f, 0.f);
    const int cin_g = L.cin_g, C = L.Cin;
    const int gsel0 = tc + 3 + cls;
    const int cend = min((jq + 1) * CB, cin_g);
    const float4* w = reinterpret_cast<const float4*>(L.wq) +
                      ((size_t)(cls * net.nsets + n) * L.nchunk + tc * L.cpg4 + kc) * TAPS * cin_g;
    // cell (d-4+kh+kw, group gq, h-2+kh) of the padded frame = xb + (((kh+kw) * GP + gq) * Hp + kh) * cin_g
    const int Hp = net.Hp, GP = net.G + 2 * WF_GPAD;
    const float* xb = L.xc + ((((size_t)n * net.Dp + d) * GP + WF_GPAD) * Hp + h) * cin_g;
    (void)C;
    if ((cin_g & 3) == 0 && net.G == 1) {
        // one group: input group 0 is selected by exactly the taps with kh + kw == gsel0 (3 or 4)
        for (int c0 = jq * CB; c0 < cend; c0 += 4) {
            float4 xv[5], wv[5][4];
#pragma unroll
            for (int kh = 0; kh < 5; kh++) {
                const int kw = gsel0 - kh;
                const bool ok = kw >= 0 && kw < 5;
                xv[kh] = make_float4(0.f, 0.f, 0.f, 0.f);
                if (ok) xv[kh] = wf_ldx4<CG>(xb + ((size_t)gsel0 * GP * Hp + kh) * cin_g + c0);
#pragma unroll
                for (int c = 0; c < 4; c++) {
                    wv[kh][c] = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (ok) wv[kh][c] = __ldg(w + (kh * 5 + kw) * cin_g + c0 + c);
                }
            }
#pragma unroll
            for (int kh = 0; kh < 5; kh++) {
                const int kw = gsel0 - kh;
                if (kw < 0 || kw >= 5) continue;
                const float xs[4] = {xv[kh].x, xv[kh].y, xv[kh].z, xv[kh].w};
#pragma unroll
                for (int c = 0; c < 4; c++) {
                    fma4(u, xs[c], wv[kh][c]);
                }
            }
        }
    } else if ((cin_g & 3) == 0) {
        // row by row: the 5 activations and 20 weight vectors of a kernel row are in flight together
        for (int c0 = jq * CB; c0 < cend; c0 += 4) {
#pragma unroll
            for (int kh = 0; kh < 5; kh++) {
                float4 xv[5], wv[5][4];
#pragma unroll
                for (int kw = 0; kw < 5; kw++) {
                    const int gq = gsel0 - kh - kw;
                    const bool ok = gq >= 0 && gq < net.G;
                    xv[kw] = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (ok) xv[kw] = wf_ldx4<CG>(xb + (((size_t)(kh + kw) * GP + gq) * Hp + kh) * cin_g + c0);
#pragma unroll
                    for (int c = 0; c < 4; c++) {
                        wv[kw][c] = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (ok) wv[kw][c] = __ldg(w + (kh * 5 + kw) * cin_g + c0 + c);
                    }
                }
#pragma unroll
                for (int kw = 0; kw < 5; kw++) {
                    const int gq = gsel0 - kh - kw;
                    if (gq < 0 || gq >= net.G) continue;
                    const float xs[4] = {xv[kw].x, xv[kw].y, xv[kw].z, xv[kw].w};
#pragma unroll
                    for (int c = 0; c < 4; c++) {
                        fma4(u, xs[c], wv[kw][c]);
                    }
                }
            }
        }
    } else {
        for (int c0 = jq * CB; c0 < cend; c0 += 4) {
            const int nc = min(4, cend - c0);
#pragma unroll
            for (int kh = 0; kh < 5; kh++) {
#pragma unroll
                for (int kw = 0; kw < 5; kw++) {
                    const int gq = gsel0 - kh - kw;
                    if (gq < 0 || gq >= net.G) continue;
                    const float* xp = xb + (((size_t)(kh + kw) * GP + gq) * Hp + kh) * cin_g + c0;
                    const float4* wt = w + (kh * 5 + kw) * cin_g + c0;
                    for (int c = 0; c < nc; c++) {
                        const float xx = CG ? __ldcg(xp + c) : __ldg(xp + c);
                        const float4 w4 = __ldg(wt + c);
                        fma4(u, xx, w4);
                    }
                }
            }
        }
    }
    return u;
}

// previous-wavefront terms R of layers [l0, ..) of step *ctr + dp -> rbuf.  Same CTA geometry as wf_old_kernel, so a CTA
// has ONE output group: its row of class-0 weights ([tap][cin_g] float4, only the taps that select an existing group)
// is staged in shared memory with cp.async; warp jq = canonical 16-channel block jq of the group, and the activation
// loads of a whole 4-channel chunk (all taps) are in flight before its first FMA.
template <int MAXT>
__global__ void __launch_bounds__(MAXT, 1) wf_prev_kernel(const __grid_constant__ WfNetDev net, int wcap, int dp, int l0) {
    extern __shared__ float4 wf_psm[];  // [TAPS * cin_g (<= wcap)] weights, then [nqb][32] partials
    const WfTile t = wf_tile(net, dp, l0);
    if (!t.ok) return;
    if (threadIdx.x == 0 && threadIdx.y == 0) WF_TRACE_MIN(net.G, t.psum - dp, WF_TR_PREV);
    const WfLayerDev& L = net.L[t.l];
    const int lane = threadIdx.x, jq = threadIdx.y, tid = jq * 32 + lane, nthr = blockDim.x * blockDim.y;
    const int cin_g = L.cin_g, G = net.G, Hp = net.Hp;
    const int gsel0 = t.tc + 3;
    {
        const float4* src = reinterpret_cast<const float4*>(L.wq) + ((size_t)t.n * L.nchunk + t.tc * L.cpg4 + t.kc) * TAPS * cin_g;
        const unsigned dst = (unsigned)__cvta_generic_to_shared(wf_psm);
        for (int e = tid; e < TAPS * cin_g; e += nthr) {
            const int tap = e / cin_g, gq = gsel0 - tap / 5 - tap % 5;
            if (gq >= 0 && gq < G) cp_async16(dst + 16u * e, src + e);
        }
        cp_async_wait_all();
        __syncthreads();
    }
    float4* part = wf_psm + wcap;
    const int h = t.hbase + lane;
    const bool valid = h <= t.hmax;
    float4 u = make_float4(0.f, 0.f, 0.f, 0.f);
    if (jq < L.nqb && valid) {
        const int cend = min((jq + 1) * CB, cin_g);
        const int GP = G + 2 * WF_GPAD;
        const float* xb = L.xc + ((((size_t)t.n * net.Dp + t.d) * GP + WF_GPAD) * Hp + h) * cin_g;
        if ((cin_g & 3) == 0 && G == 1) {
            // one group: exactly the taps with kh + kw == gsel0 (== 3) contribute; all chunks of the block in flight
            float4 xv[4][5];
#pragma unroll
            for (int q = 0; q < 4; q++)
#pragma unroll
                for (int kh = 0; kh < 5; kh++) {
                    const int kw = gsel0 - kh, c0 = jq * CB + 4 * q;
                    xv[q][kh] = make_float4(0.f, 0.f, 0.f, 0.f);
                    if (kw >= 0 && kw < 5 && c0 < cend) xv[q][kh] = __ldg(reinterpret_cast<const float4*>(xb + ((size_t)gsel0 * GP * Hp + kh) * cin_g + c0));
                }
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const int c0 = jq * CB + 4 * q;
                if (c0 >= cend) break;
#pragma unroll
                for (int kh = 0; kh < 5; kh++) {
                    const int kw = gsel0 - kh;
                    if (kw < 0 || kw >= 5) continue;
                    const float xs[4] = {xv[q][kh].x, xv[q][kh].y, xv[q][kh].z, xv[q][kh].w};
                    const float4* wt = wf_psm + (kh * 5 + kw) * cin_g + c0;
#pragma unroll
                    for (int c = 0; c < 4; c++) {
                        const float4 w4 = wt[c];
                        fma4(u, xs[c], w4);
                    }
                }
            }
        } else if ((cin_g & 3) == 0) {
            for (int c0 = jq * CB; c0 < cend; c0 += 4) {
                float4 xv[TAPS];
#pragma unroll
                for (int kh = 0; kh < 5; kh++)
#pragma unroll
                    for (int kw = 0; kw < 5; kw++) {
                        const int gq = gsel0 - kh - kw;
                        xv[kh * 5 + kw] = make_float4(0.f, 0.f, 0.f, 0.f);
                        if (gq >= 0 && gq < G)
                            xv[kh * 5 + kw] = __ldg(reinterpret_cast<const float4*>(xb + (((size_t)(kh + kw) * GP + gq) * Hp + kh) * cin_g + c0));
                    }
#pragma unroll
                for (int kh = 0; kh < 5; kh++)
#pragma unroll
                    for (int kw = 0; kw < 5; kw++) {
                        const int gq = gsel0 - kh - kw;
                        if (gq < 0 || gq >= G) continue;
                        const float4 x4 = xv[kh * 5 + kw];
                        const float xs[4] = {x4.x, x4.y, x4.z, x4.w};
                        const float4* wt = wf_psm + (kh * 5 + kw) * cin_g + c0;
#pragma unroll
                        for (int c = 0; c < 4; c++) {
                            const float4 w4 = wt[c];
                            fma4(u, xs[c], w4);
                        }
                    }
            }
        } else {
            for (int c0 = jq * CB; c0 < cend; c0 += 4) {
                const int nc = min(4, cend - c0);
#pragma unroll
                for (int kh = 0; kh < 5; kh++)
#pragma unroll
                    for (int kw = 0; kw < 5; kw++) {
                        const int gq = gsel0 - kh - kw;
                        if (gq < 0 || gq >= G) continue;
                        const float* xp = xb + (((size_t)(kh + kw) * GP + gq) * Hp + kh) * cin_g + c0;
                        const float4* wt = wf_psm + (kh * 5 + kw) * cin_g + c0;
                        for (int c = 0; c < nc; c++) {
                            const float xx = __ldg(xp + c);
                            const float4 w4 = wt[c];
                            fma4(u, xx, w4);
                        }
                    }
            }
        }
    }
    float4 r = u;
    if (blockDim.y > 1) {
        part[jq * 32 + lane] = u;
        __syncthreads();
        if (jq != 0) return;
        r = make_float4(0.f, 0.f, 0.f, 0.f);
        for (int j = 0; j < L.nqb; j++) {
            const float4 v = part[j * 32 + lane];
            r.x = r.x + v.x; r.y = r.y + v.y; r.z = r.z + v.z; r.w = r.w + v.w;
        }
    } else {
        r.x = 0.f + r.x; r.y = 0.f + r.y; r.z = 0.f + r.z; r.w = 0.f + r.w;  // R = 0 + r_0, as everywhere else
    }
    if (!valid) return;
    L.rbuf[t.psum & 1][(((size_t)t.n * L.cpg4 + t.kc) * net.D + t.d) * net.HS + h] = r;
}

// ------------------------------------------------------------------------------------------------ the 12-layer chain
// One thread-block cluster per net.  Layer l: every (slab position, output chunk) item adds its same-wavefront terms
// (read from the layer below through L2) to P + R, applies bias / PReLU / residual and stores the 4 channels into both
// frame layouts; a cluster barrier (release / acquire) orders layer l's stores before layer l+1's loads.
template <int MAXT>
__global__ void __launch_bounds__(MAXT, 1) wf_chain_kernel(const __grid_constant__ WfNetDev net, int nc) {
    extern __shared__ float4 wf_part[];
    const int tid = threadIdx.x, nt = blockDim.x;
    const int n = blockIdx.x / nc, rank = blockIdx.x % nc;
    // programmatic dependent launch: the old-term kernel of the next step may start as soon as every CTA of this kernel is
    // resident (it does not read anything this kernel writes); without that launch attribute this is a no-op
    asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory");
    const StepDesc sd = net.steps[*net.ctr];
    const int HW = net.H * net.W;
    for (int l = 0; l < WF_LAYERS; l++) {
        const WfLayerDev& L = net.L[l];
        const int items = sd.len * L.cpg4;
        const int per = (items + nc - 1) / nc;
        const int i0 = min(items, rank * per), i1 = min(items, i0 + per), nloc = i1 - i0;
        const bool direct = L.nqb == 1;  // one canonical block per item: no exchange of partials through shared memory
        if (L.has_q && !direct) {
            for (int tsk = tid; tsk < nloc * L.nqb; tsk += nt) {
                const int jq = tsk / nloc, i = i0 + tsk % nloc;
                const int kc = i / sd.len, k = sd.start + i % sd.len;
                const int h = __ldg(net.idx + k), w = __ldg(net.idx + k + HW);
                wf_part[tsk] = wf_rq_partial<true>(net, L, n, h + w, h, sd.psum - h - w, kc, jq, 1);
            }
            __syncthreads();
        }
        for (int il = tid; il < nloc; il += nt) {
            const int i = i0 + il;
            const int kc = i / sd.len, k = sd.start + i % sd.len;
            const int h = __ldg(net.idx + k), w = __ldg(net.idx + k + HW);
            const int d = h + w, tc = sd.psum - d;
            // independent loads first: P + R, bias, slope, residual
            const size_t pi = (((size_t)n * L.cpg4 + kc) * net.D + d) * net.HS + h;
            float4 pr = __ldg(L.pbuf[sd.psum & 1] + pi);
            { const float4 rr = __ldg(L.rbuf[sd.psum & 1] + pi); pr.x = pr.x + rr.x; pr.y = pr.y + rr.y; pr.z = pr.z + rr.z; pr.w = pr.w + rr.w; }
            const size_t fc = wf_fc_index(net.Dp, net.Hp, net.G, L.cout_g, n, d, tc, h) + kc * 4;
            const int o0 = tc * L.cout_g + kc * 4;
            float bs[4], sl[4], rs[4];
#pragma unroll
            for (int q = 0; q < 4; q++) {
                const bool live = kc * 4 + q < L.cout_g;
                bs[q] = live ? __ldg(L.bias + n * L.Cout + o0 + q) : 0.f;
                sl[q] = live && L.slope ? __ldg(L.slope + n * L.Cout + o0 + q) : 0.f;
                rs[q] = live && L.rc ? __ldcg(L.rc + fc + q) : 0.f;
            }
            float Q[4] = {0.f, 0.f, 0.f, 0.f};
            if (L.has_q) {
                if (direct) {
                    const float4 v = wf_rq_partial<true>(net, L, n, d, h, tc, kc, 0, 1);
                    Q[0] = Q[0] + v.x; Q[1] = Q[1] + v.y; Q[2] = Q[2] + v.z; Q[3] = Q[3] + v.w;
                } else {
                    for (int j = 0; j < L.nqb; j++) {
                        const float4 v = wf_part[j * nloc + il];
                        Q[0] = Q[0] + v.x; Q[1] = Q[1] + v.y; Q[2] = Q[2] + v.z; Q[3] = Q[3] + v.w;
                    }
                }
            }
            const float PR[4] = {pr.x, pr.y, pr.z, pr.w};
            float v[4];
#pragma unroll
            for (int q = 0; q < 4; q++) {
                v[q] = 0.f;
                if (kc * 4 + q >= L.cout_g) continue;
                float y = (PR[q] + Q[q]) + bs[q];
                if (L.slope) y = y > 0.f ? y : y * sl[q];
                if (L.rc) y = y + rs[q];
                v[q] = y;
                if (L.op) L.op[wf_fp_index(net.D, net.HS, L.Cout, n, o0 + q, d, h)] = y;
            }
            if ((L.cout_g & 3) == 0) {
                *reinterpret_cast<float4*>(L.oc + fc) = make_float4(v[0], v[1], v[2], v[3]);
            } else {
#pragma unroll
                for (int q = 0; q < 4; q++)
                    if (kc * 4 + q < L.cout_g) L.oc[fc + q] = v[q];
            }
        }
        if (l + 1 < WF_LAYERS) {
            if (nc > 1) cg::this_cluster().sync();
            else __syncthreads();
        }
    }
}

// Fast chain for nets whose chained layers have 4 channels per input group and at most 4 per output group (the code
// stream: 48 groups x 4): one item = one slab position.  Everything that does not depend on the layer below is taken
// off the per-layer critical path:
//   - the same-wavefront weights of layer l+1 (one 100-float4 row per output group present in this CTA's item range)
//     are copied to shared memory with cp.async while layer l is being computed,
//   - P + R, bias, slope and the residual of layer l+1 are loaded into registers before the barrier that ends layer l,
//   - the 25 activation loads of an item (one float4 per tap) are all in flight before the first FMA.
// Per layer that leaves: cluster barrier -> one L2 round trip -> 400 FMAs against shared-memory weights -> stores.
// tap loads of the code-stream chain: plain loads (see wf_chain4_kernel); -DLIC360_WF_TAPS_CG restores ld.global.cg
#ifdef LIC360_WF_TAPS_CG
#define WF_TAP_LOAD(p) __ldcg(p)
#else
#define WF_TAP_LOAD(p) (*(p))
#endif
constexpr int WF_ROW_F4 = TAPS * 4;  // float4 per (output group) row of same-wavefront weights when cin_g == 4

struct WfPre { float4 pr, rr; float bs[4], sl[4], rs[4]; };  // P and R: added where they are consumed, a layer later

__device__ __forceinline__ void wf_chain4_prefetch(const WfNetDev& net, const WfLayerDev& L, int n, int par, int d, int h, int tc,
                                                   WfPre& p) {
    // L2 loads (not the read-only path): in the persistent decode these sums are produced while this kernel is running -- P by the
    // concurrently running old-term kernel, R by this cluster's own tail of the previous step
    p.pr = __ldcg(L.pbuf[par] + ((size_t)n * net.D + d) * net.HS + h);
    p.rr = __ldcg(L.rbuf[par] + ((size_t)n * net.D + d) * net.HS + h);
    const size_t fc = wf_fc_index(net.Dp, net.Hp, net.G, L.cout_g, n, d, tc, h);
    const int o0 = tc * L.cout_g;
#pragma unroll
    for (int q = 0; q < 4; q++) {
        const bool live = q < L.cout_g;
        p.bs[q] = live ? __ldg(L.bias + n * L.Cout + o0 + q) : 0.f;
        p.sl[q] = live && L.slope ? __ldg(L.slope + n * L.Cout + o0 + q) : 0.f;
        p.rs[q] = live && L.rc ? __ldcg(L.rc + fc + q) : 0.f;  // written by this very thread two layers ago
    }
}

// Previous-wavefront terms R of one item of LAYER 0 when it has one channel per group (the code stream's first layer):
// they read the symbols the host decoded a moment ago, so they cannot be computed a step ahead like the other layers'.
// 25 activations and 25 weight vectors, all in flight together; groups outside [0, G) read the zero padding of the group
// axis and carry zero weights.  Non-inlined: runs once per step, outside the layer loop.
// COHERENT: the symbols were scattered by THIS kernel (persistent decode) -> L2 loads instead of the read-only path
template <bool COHERENT = false>
__device__ __noinline__ float4 wf_r_layer0_c1(const WfNetDev& net, int n, int d, int h, int tc, int kc = 0) {
    const WfLayerDev& L = net.L[0];
    const int GP = net.G + 2 * WF_GPAD;
    const float* xr = L.xc + (((size_t)n * net.Dp + d) * GP + WF_GPAD + tc + 3) * net.Hp + h;
    const size_t srow = (size_t)(GP - 1) * net.Hp;
    const float4* w = reinterpret_cast<const float4*>(L.wq) + ((size_t)n * L.nchunk + tc * L.cpg4 + kc) * TAPS;
    float xv[TAPS];
    float4 wv[TAPS];
#pragma unroll
    for (int kh = 0; kh < 5; kh++)
#pragma unroll
        for (int kw = 0; kw < 5; kw++) {
            xv[kh * 5 + kw] = COHERENT ? __ldcg(xr + (kh + kw) * srow + kh) : __ldg(xr + (kh + kw) * srow + kh);
            wv[kh * 5 + kw] = __ldg(w + kh * 5 + kw);
        }
    float4 u = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int t = 0; t < TAPS; t++) {
        fma4(u, xv[t], wv[t]);
    }
    return make_float4(0.f + u.x, 0.f + u.y, 0.f + u.z, 0.f + u.w);  // R = 0 + r_0 (one canonical block)
}

// Previous-wavefront terms R of step p + 1 (layers 1..11) are evaluated by the chain kernel of step p behind its CDF rows (wf_chain4_rtail).
// This CTA takes the same chunk of the NEXT slab it will own in the next step's chain; the R weight rows of that chunk's output groups, for
// as many layers as fit (all 11 unless the chunk spans many groups), are copied to shared memory while the CTA waits for the other
// clusters in wf_chain4_rows -- the tail then runs from shared-memory weights like the chain itself.
struct WfTailPlan { int i0, nloc, tc_lo, nrows, lpg; };

// step s1 = step psum1 of the index plan idx (H * W positions); also evaluated on the host (wf_tail_rounds)
__host__ __device__ __forceinline__ WfTailPlan wf_tail_plan_of(const int32_t* idx, int HW, StepDesc s1, int rank, int nc, int psum1,
                                                               int smem_rows) {
#ifdef __CUDA_ARCH__
#define WF_IDX(k) __ldg(idx + (k))
#else
#define WF_IDX(k) idx[k]
#endif
    WfTailPlan t = {0, 0, 0, 0, 1};
    const int per = (s1.len + nc - 1) / nc;
    t.i0 = min(s1.len, rank * per);
    const int i1 = min(s1.len, t.i0 + per);
    t.nloc = i1 - t.i0;
    if (t.nloc > 0) {  // plan order is diagonal-major: the chunk's output groups are a contiguous range
        const int ka = s1.start + t.i0, kb = s1.start + i1 - 1;
        const int tc_hi = psum1 - WF_IDX(ka) - WF_IDX(ka + HW);
        t.tc_lo = psum1 - WF_IDX(kb) - WF_IDX(kb + HW);
        t.nrows = tc_hi - t.tc_lo + 1;
        t.lpg = max(1, min(WF_LAYERS - 1, smem_rows / t.nrows));
    }
#undef WF_IDX
    return t;
}

__device__ __forceinline__ WfTailPlan wf_tail_plan(const WfNetDev& net, int rank, int nc, int psum1, int smem_rows) {
    if (psum1 >= net.nsteps) return WfTailPlan{0, 0, 0, 0, 1};
    return wf_tail_plan_of(net.idx, net.H * net.W, net.steps[psum1], rank, nc, psum1, smem_rows);
}

// cp.async of the R rows [tc_lo, tc_lo + nrows) of layers l0 .. l0 + nl - 1 into the dynamic shared memory, issued by threads t0, t0 + 1, ..
__device__ __forceinline__ void wf_tail_stage(const WfNetDev& net, int n, const WfTailPlan& t, int l0, int nl, int tid, int t0, int nthr) {
    extern __shared__ float4 wf_wsm[];
    if (tid >= t0) {
        const int per_layer = t.nrows * WF_ROW_F4;
        for (int lr = 0; lr < nl; lr++) {
            const WfLayerDev& L = net.L[l0 + lr];
            const float4* src = reinterpret_cast<const float4*>(L.wq) + ((size_t)n * L.nchunk + t.tc_lo) * WF_ROW_F4;
            const unsigned dst = (unsigned)__cvta_generic_to_shared(wf_wsm + (size_t)lr * per_layer);
            for (int e = tid - t0; e < per_layer; e += nthr) cp_async16(dst + 16u * e, src + e);
        }
    }
    asm volatile("cp.async.commit_group;\n" ::);
}

// CDF rows of the step (TileExtract + EntropyGmmTable fused) at the end of the chain kernel: a row needs the outputs of all
// three nets, so the clusters meet at a monotone global counter first (every CTA of the grid is resident or becomes
// resident without needing anything from the waiting ones: no deadlock).  A separate, non-inlined function: its register
// needs (erff, the 9-bin row) stay out of the chain's layer loop.
__device__ __noinline__ void wf_chain4_rows(const WfNetDev& net, const WfRows& rows, int psum, int start, int len, int tid, int nt,
                                            int n, const WfTailPlan& tail) {
    __shared__ int s_abort;
    __threadfence();
    __syncthreads();
    // the layer loop is done with the weight buffers: warps 1.. fill them with the R rows of the tail while thread 0 meets the other clusters
    if (tail.nloc > 0) wf_tail_stage(net, n, tail, 1, min(tail.lpg, WF_LAYERS - 1), tid, 32, nt - 32);
    if (tid == 0) {
        atomicAdd(rows.sync, 1);
        const int target = (psum + 1) * (int)gridDim.x;
        // Bail-out: with more decodes in flight than the device can keep resident (codec.cu bounds that with a per-device
        // semaphore) a sibling cluster might never be placed; give up after ~2 s instead of spinning forever, the host sees the
        // negative flag and fails the decode.
        unsigned long long t0 = 0, t1 = 0;
        int ab = 0;
        for (unsigned spins = 1; *reinterpret_cast<volatile int*>(rows.sync) < target; spins++) {
            if ((spins & 0x3FFF) == 0) {
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
                if (t0 == 0) t0 = t1;
                else if (t1 - t0 > 2000000000ull) { ab = 1; break; }
            }
        }
        s_abort = ab;
        __threadfence();
        WF_TRACE_MIN(net.G, psum, WF_TR_ROWS0);
    }
    __syncthreads();
    if (s_abort) {
        if (tid == 0) {
            __threadfence_system();
            reinterpret_cast<volatile int*>(rows.flag)[blockIdx.x] = -(psum + 1);
        }
        return;
    }
    const int G = net.G, H = net.H, W = net.W, HW = H * W;
    const float* y = net.L[WF_LAYERS - 1].oc;
    // 4 lanes per symbol, lane j computes bins j + 1 and j + 5 (the 21 erff of a row are the latency of this phase; with 8 lanes
    // per symbol a full slab needed two passes over the grid's threads), lane 0 gathers, fixes up and stores the packed row
    const int total = ((len * 4 + 31) >> 5) << 5;  // whole warps
    for (int gt = blockIdx.x * nt + tid; gt < total; gt += (int)gridDim.x * nt) {
        const int li = gt >> 2, j = gt & 3;
        const bool live = li < len;
        float bin_a = 0.f, bin_b = 0.f;
        int th = 0, tw = 0, tc = 0;
        if (live) {
            th = __ldg(net.idx + start + li); tw = __ldg(net.idx + start + li + HW);
            tc = psum - th - tw;
            float wv[3], dv[3], mv[3];
#pragma unroll
            for (int i = 0; i < 3; i++) {
                wv[i] = __ldcg(y + wf_fc_index(net.Dp, net.Hp, G, 3, 0, th + tw, tc, th) + i);
                dv[i] = __ldcg(y + wf_fc_index(net.Dp, net.Hp, G, 3, 1, th + tw, tc, th) + i);
                mv[i] = __ldcg(y + wf_fc_index(net.Dp, net.Hp, G, 3, 2, th + tw, tc, th) + i);
            }
            gmm_prep(wv, dv, 3, 1e-6f);
            bin_a = gmm_bin_value(wv, dv, mv, j + 1, 3, 3.5f, 65536.f, rows.s2);
            if (j < 3) bin_b = gmm_bin_value(wv, dv, mv, j + 5, 3, 3.5f, 65536.f, rows.s2);
        }
        float o[9];
        o[0] = 0.f; o[8] = 65536.f;
        const int base = tid & 28;
#pragma unroll
        for (int k = 0; k < 4; k++) {
            o[1 + k] = __shfl_sync(0xffffffffu, bin_a, base + k);
            if (k < 3) o[5 + k] = __shfl_sync(0xffffffffu, bin_b, base + k);
        }
        if (live && j == 0) {
            fixup_row(o, 8, true);
            const int lvl = (int)(__ldcg(rows.levels + (th >> 1) * (W >> 1) + (tw >> 1)) + 1e-5f);  // written by the other stream's kernels
            pack_gmm_row(o, 0, code_mask_from_level(lvl, tc, th, tw), rows.rows + (size_t)li * 8, wf_row_tag(psum));
        }
    }
    // self-validating rows: no fence, no flag; the host decodes row i as soon as row i carries this step's tag
    if (tid == 0) WF_TRACE_MAX(net.G, psum, WF_TR_ROWS1);
}

// Previous-wavefront terms R of step psum1 = p + 1, layers 1..11, evaluated by the chain kernel of step p right behind its CDF
// rows: the activations of wavefront p are final, the cluster's SMs are idle while the host decodes, and a separate launch for
// them (wf_prev_kernel) was observed to start only when the concurrently running old-term kernel drained (+30 us on the step).
// One item = (layer, slab position of step p + 1); arithmetic = one canonical block of 4 channels, taps in (kh, kw, c) order,
// every tap read unconditionally from the group-padded frame (out-of-range groups are zeros times zero weights).
// One item = (layer, PAIR of adjacent positions of one diagonal of the next slab): the two positions share their output group, so
// every shared-memory weight vector feeds 8 FMAs, and 16 of their 2 x 25 taps (tap (kh, kw) of the upper position is tap
// (kh + 1, kw - 1) of the lower one).  Pairs are formed inside each diagonal's segment of the CTA's chunk, from the segment start; a
// segment of odd length ends in a single.  The item loop is bound by shared-memory wavefronts like the old-term kernels.
struct WfPairPos { int d, h, single; };

// pair q of the chunk [k0, k0 + nloc) of the plan (diagonal-major, rows ascending); q < 0: returns the number of pairs in .h
__device__ __forceinline__ WfPairPos wf_tail_pair(const WfNetDev& net, int k0, int nloc, int q) {
    const int HW = net.H * net.W;
    const int hf = __ldg(net.idx + k0);
    int d = hf + __ldg(net.idx + k0 + HW);
    int a = hf - max(0, d - net.W + 1);  // offset of the chunk's first position inside its diagonal
    int left = nloc, total = 0;
    WfPairPos r = {0, 0, 0};
    while (left > 0) {
        const int hmin = max(0, d - net.W + 1), dlen = min(net.H - 1, d) - hmin + 1;
        const int seg = min(dlen - a, left), np = (seg + 1) >> 1;
        if (q >= 0 && q < np) {
            r.d = d; r.h = hmin + a + 2 * q; r.single = 2 * q + 1 >= seg;
            return r;
        }
        q -= np; total += np; left -= seg; d++; a = 0;
    }
    r.h = total;
    return r;
}

__device__ __noinline__ void wf_chain4_rtail(const WfNetDev& net, int n, int psum1, int tid, int nt, const WfTailPlan& tail) {
    extern __shared__ float4 wf_wsm[];
    if (psum1 >= net.nsteps || tail.nloc == 0) return;  // uniform per CTA
    if (tid == 0) WF_TRACE_MIN(net.G, psum1 - 1, WF_TR_TAIL0);
    const StepDesc s1 = net.steps[psum1];
    const int GP = net.G + 2 * WF_GPAD;
    const size_t srow = (size_t)(GP - 1) * net.Hp;
    const int k0 = s1.start + tail.i0;
    const int npairs = wf_tail_pair(net, k0, tail.nloc, -1).h;
    for (int l0 = 1; l0 < WF_LAYERS; l0 += tail.lpg) {
        const int nl = min(tail.lpg, WF_LAYERS - l0);
        if (l0 > 1) {  // (the first group was staged in wf_chain4_rows)
            __syncthreads();
            wf_tail_stage(net, n, tail, l0, nl, tid, 0, nt);
        }
        asm volatile("cp.async.wait_group 0;\n" ::: "memory");
        __syncthreads();
        for (int it = tid; it < nl * npairs; it += nt) {
            const int lr = it / npairs;
            const WfPairPos pp = wf_tail_pair(net, k0, tail.nloc, it - lr * npairs);
            const WfLayerDev& L = net.L[l0 + lr];
            const int h = pp.h, d = pp.d, tc = psum1 - d;
            // tap (kh, kw), s = kh + kw, selects group tc + 3 - s: cell = xr + s * srow + kh (+ 1 for the upper position), float4 units
            const float4* xr = reinterpret_cast<const float4*>(L.xc) + (((size_t)n * net.Dp + d) * GP + WF_GPAD + tc + 3) * net.Hp + h;
            const float4* wr = wf_wsm + ((size_t)lr * tail.nrows + (tc - tail.tc_lo)) * WF_ROW_F4;
            float4 cell[9][6];
#pragma unroll
            for (int sd = 0; sd < 9; sd++) {
                const int khmin = sd > 4 ? sd - 4 : 0, khmax = sd < 4 ? sd : 4;
#pragma unroll
                for (int col = 0; col < 6; col++) {
                    if (col < khmin || col > khmax + 1) continue;
                    // this cluster's stores, behind its barriers; a single's upper cells would leave the diagonal: not read
                    if (col == khmax + 1 && pp.single) cell[sd][col] = make_float4(0.f, 0.f, 0.f, 0.f);
                    else cell[sd][col] = WF_TAP_LOAD(xr + sd * srow + col);
                }
            }
            float4 u0 = make_float4(0.f, 0.f, 0.f, 0.f), u1 = u0;
#pragma unroll
            for (int kh = 0; kh < 5; kh++)
#pragma unroll
                for (int kw = 0; kw < 5; kw++) {
                    const float4 a4 = cell[kh + kw][kh], b4 = cell[kh + kw][kh + 1];
                    const float as[4] = {a4.x, a4.y, a4.z, a4.w}, bs[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
                    for (int c = 0; c < 4; c++) {
                        const float4 w4 = wr[(kh * 5 + kw) * 4 + c];
                        fma4(u0, as[c], w4);
                        fma4(u1, bs[c], w4);
                    }
                }
            float4* dst = L.rbuf[psum1 & 1] + ((size_t)n * net.D + d) * net.HS + h;
            dst[0] = make_float4(0.f + u0.x, 0.f + u0.y, 0.f + u0.z, 0.f + u0.w);  // R = 0 + r_0
            if (!pp.single) dst[1] = make_float4(0.f + u1.x, 0.f + u1.y, 0.f + u1.z, 0.f + u1.w);
        }
    }
    __syncthreads();  // the next step's (or launch's) layer loop stages into these buffers again
    if (tid == 0) WF_TRACE_MAX(net.G, psum1 - 1, WF_TR_TAIL1);
}

// Persistent decode (WfPersist): what the chain kernel does between two steps instead of being re-launched.
// wf_chain4_wait_old: the old-term sums of step p are complete (the old-term kernel of step p was enqueued a whole step ago; normally
// this returns at once).  Runs BEFORE the go so that P, R, bias and slope of the step's first layer are in registers when it comes.
__device__ __noinline__ void wf_chain4_wait_old(const WfPersist& ps, int p, int tid) {
    if (tid == 0) {
        unsigned long long t0 = 0, t1 = 0;
        for (unsigned spins = 1; *reinterpret_cast<const volatile int*>(ps.old_done) < p + 1; spins++) {
            if ((spins & 0xFFF) == 0) {
                asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
                if (t0 == 0) t0 = t1;
                else if (t1 - t0 > 5000000000ull) break;  // the step then runs on incomplete sums and the decode fails on the host side
            }
        }
        __threadfence();
    }
    __syncthreads();
}

// wf_chain4_step_begin, top of step p:
//   warps 1..: TileInput (tile_input_cuda.cu:27-43) of the symbols of step p - 1 into this cluster's copy of the input frame, both
//     layouts.  The host publishes every symbol as it decodes it, as a self-validating word (tag of step p - 1 in the four low mantissa
//     bits), so each thread polls ITS word in mapped host memory and scatters it at once: when the host has decoded the last symbol the
//     frame is complete but for that symbol's PCIe read.
//   thread 0: waits for the host's go -- CTA 0 polls the mapped host flag and republishes the decision in device memory so that every
//     CTA of the grid takes the SAME decision at the same step boundary (run step p, or abort instead of running it).
//   then a cluster barrier publishes the scatter to the whole cluster, and CTA 0 of the cluster tells the old-term kernels.
// Every spin has a bail-out so that a lost host or a lost kernel ends in an error, not a hang.  Returns false when the decode is to be
// abandoned.
__device__ __noinline__ bool wf_chain4_step_begin(const WfNetDev& net, const WfPersist& ps, int p, int n, int rank, int nc, int tid, int nt) {
    __shared__ int s_go;  // 0 = undecided, 1 = run, -1 = abort
    if (tid == 0) s_go = 0;
    __syncthreads();
    if (tid == 0) {
        int decision = 0;
        unsigned long long t0 = 0, t1 = 0;
        if (blockIdx.x == 0) {
            for (unsigned spins = 1; decision == 0; spins++) {
                const int v = *reinterpret_cast<const volatile int*>(ps.go_host);
                if (v == WF_GO_ABORT) decision = -1;
                else if (v >= p) decision = 1;
                else if ((spins & 0xFF) == 0) {
                    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
                    if (t0 == 0) t0 = t1;
                    else if (t1 - t0 > 20000000000ull) decision = -1;  // 20 s without a host: give up
                }
            }
            WF_TRACE_MIN(net.G, p, WF_TR_SCATTER);  // debug timeline: the go of step p has reached the device
            *reinterpret_cast<volatile int*>(ps.go_dev) = decision > 0 ? p : -(p + 2);
            if (decision > 0) *reinterpret_cast<volatile int*>(ps.ctr) = p;
        } else {
            for (unsigned spins = 1; decision == 0; spins++) {
                const int v = *reinterpret_cast<const volatile int*>(ps.go_dev);
                if (v >= p) decision = 1;
                else if (v < -1 && -(v + 2) <= p) decision = -1;  // -1 is the initial value: nothing decided yet
                else if ((spins & 0xFFF) == 0) {
                    asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t1));
                    if (t0 == 0) t0 = t1;
                    else if (t1 - t0 > 30000000000ull) decision = -1;
                }
            }
        }
        *reinterpret_cast<volatile int*>(&s_go) = decision;
    } else if (tid >= 32 && p > 0) {
        const StepDesc d = net.steps[p - 1];
        const int HW = net.H * net.W, nw = nt - 32;
        const unsigned tag = (unsigned)wf_row_tag(p - 1);
        float* fp0 = const_cast<float*>(net.L[0].xp);
        float* fc0 = const_cast<float*>(net.L[0].xc);
        const unsigned* words = reinterpret_cast<const unsigned*>(ps.syms);
        bool dead = false;
        for (int l = rank * nw + tid - 32; l < d.len && !dead; l += nc * nw) {
            const int th = __ldg(net.idx + d.start + l), tw = __ldg(net.idx + d.start + l + HW);
            const int tc = d.psum - th - tw;
            unsigned bits;
            for (;;) {
                bits = __ldcv(words + l);  // mapped host memory: never from a cached line
                if ((bits & 15u) == tag) break;
                if (*reinterpret_cast<volatile int*>(&s_go) < 0) { dead = true; break; }  // the go can only come after the symbols
            }
            if (dead) break;
            const float v = fmaf(ps.scale, __uint_as_float(bits & ~15u), ps.bias);
            fp0[wf_fp_index(net.D, net.HS, net.G, n, tc, th + tw, th)] = v;
            fc0[wf_fc_index(net.Dp, net.Hp, net.G, 1, n, th + tw, tc, th)] = v;
        }
    }
    __syncthreads();
    if (s_go < 0) return false;
    if (nc > 1) cg::this_cluster().sync();
    else __syncthreads();
    if (rank == 0 && tid == 0) {  // this net's frame now holds the symbols of every step < p
        if (n == 0) WF_TRACE_MIN(net.G, p, WF_TR_PREV);  // debug timeline: scatter + cluster barrier done
        __threadfence();
        reinterpret_cast<volatile int*>(ps.scat_done)[n] = p;
    }
    return true;
}

__global__ void __launch_bounds__(384, 1) wf_chain4_kernel(const __grid_constant__ WfNetDev net, int nc, int rows_cap,
                                                         const __grid_constant__ WfRows rows,
                                                         const __grid_constant__ WfPersist persist, int smem_rows) {
    extern __shared__ float4 wf_wsm[];  // [2][rows_cap][WF_ROW_F4]
    const int tid = threadIdx.x, nt = blockDim.x;
    const int n = blockIdx.x / nc, rank = blockIdx.x % nc;
    // programmatic dependent launch: the old-term kernel of the next step may start as soon as every CTA of this kernel is
    // resident (it does not read anything this kernel writes); without that launch attribute this is a no-op
    asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory");
    const int HW = net.H * net.W;
    // one step per launch (graph replay: the step is read from the device counter) or all of them (persistent decode)
    const int step_first = persist.enabled ? 0 : *net.ctr, step_last = persist.enabled ? net.nsteps : step_first + 1;
  for (int step = step_first; step < step_last; step++) {
    const StepDesc sd = net.steps[step];
    const int par = sd.psum & 1;
    if (!persist.enabled && threadIdx.x == 0) WF_TRACE_MIN(net.G, sd.psum, WF_TR_CHAIN0);
    const int per = (sd.len + nc - 1) / nc;
    const int i0 = min(sd.len, rank * per), i1 = min(sd.len, i0 + per), nloc = i1 - i0;
    // plan order is diagonal-major, so the output groups of this CTA's items are the contiguous range [tc_lo, tc_hi]
    int tc_lo = 0, nrows = 0;
    if (nloc > 0) {
        const int ka = sd.start + i0, kb = sd.start + i1 - 1;
        const int tc_hi = sd.psum - __ldg(net.idx + ka) - __ldg(net.idx + ka + HW);
        tc_lo = sd.psum - __ldg(net.idx + kb) - __ldg(net.idx + kb + HW);
        nrows = tc_hi - tc_lo + 1;
    }
    // slot 0 item of this thread (the only one unless the slab is larger than the cluster's thread count)
    const bool has0 = tid < nloc;
    int h0 = 0, d0 = 0, tc0 = 0;
    if (has0) {
        const int k = sd.start + i0 + tid;
        h0 = __ldg(net.idx + k);
        d0 = h0 + __ldg(net.idx + k + HW);
        tc0 = sd.psum - d0;
    }
    WfPre pre;
    if (persist.enabled) wf_chain4_wait_old(persist, step, tid);
    if (has0) wf_chain4_prefetch(net, net.L[0], n, par, d0, h0, tc0, pre);
    if (persist.enabled) {  // everything above is in flight or done when the host's go arrives
        if (!wf_chain4_step_begin(net, persist, step, n, rank, nc, tid, nt)) return;
        if (threadIdx.x == 0) WF_TRACE_MIN(net.G, sd.psum, WF_TR_CHAIN0);
    }
    // layer 0's previous-wavefront terms read the symbols of step p - 1: evaluated here, not a step ahead like the other layers'
    if (has0) pre.rr = persist.enabled ? wf_r_layer0_c1<true>(net, n, d0, h0, tc0) : wf_r_layer0_c1<false>(net, n, d0, h0, tc0);
    // debug timeline (LIC360_WF_TRACE=1): ns spent by thread 0 of CTA 0 in the phases of every layer, accumulated behind the step slots
    const bool phase_trace = g_wf_trace && g_wf_trace_sel == 0 && blockIdx.x == 0 && tid == 0;
    unsigned long long tph = 0;
    auto phase = [&](int l, int ph) {
        if (!phase_trace) return;
        unsigned long long t_;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_));
        if (ph >= 0) atomicAdd(g_wf_trace + (size_t)(net.nsteps + 2) * WF_TR_SLOTS + l * 4 + ph, t_ - tph);
        tph = t_;
    };
    phase(0, -1);
    for (int l = 0; l < WF_LAYERS; l++) {
        const WfLayerDev& L = net.L[l];
        // stage the same-wavefront weights of the next layer: rows tc_lo .. tc_lo + nrows - 1 are contiguous in wq
        if (l + 1 < WF_LAYERS && nrows > 0) {
            const WfLayerDev& Ln = net.L[l + 1];
            const float4* src = reinterpret_cast<const float4*>(Ln.wq) + ((size_t)(net.nsets + n) * Ln.nchunk + tc_lo) * WF_ROW_F4;
            const unsigned dst = (unsigned)__cvta_generic_to_shared(wf_wsm + (size_t)((l + 1) & 1) * rows_cap * WF_ROW_F4);
            for (int e = tid; e < nrows * WF_ROW_F4; e += nt) cp_async16(dst + 16u * e, src + e);
            asm volatile("cp.async.commit_group;\n" ::);
        }
        const float4* wl = wf_wsm + (size_t)(l & 1) * rows_cap * WF_ROW_F4;
        phase(l, 0);
        for (int il = tid; il < nloc; il += nt) {
            int h = h0, d = d0, tc = tc0;
            WfPre p = pre;
            if (il != tid) {  // further slots: nothing was prefetched
                const int k = sd.start + i0 + il;
                h = __ldg(net.idx + k);
                d = h + __ldg(net.idx + k + HW);
                tc = sd.psum - d;
                wf_chain4_prefetch(net, L, n, par, d, h, tc, p);
                if (l == 0) p.rr = persist.enabled ? wf_r_layer0_c1<true>(net, n, d, h, tc) : wf_r_layer0_c1<false>(net, n, d, h, tc);
            }
            float4 u = make_float4(0.f, 0.f, 0.f, 0.f);
            if (L.has_q) {
                // tap (kh, kw), s = kh + kw, selects group tc + 4 - s: cell = xr + s * srow + kh, float4 units.  Groups outside
                // [0, G) fall into the zero padding of the group axis (and carry zero weights): no tests, no branches.
                const int GP = net.G + 2 * WF_GPAD;
                const float4* xr = reinterpret_cast<const float4*>(L.xc) + (((size_t)n * net.Dp + d) * GP + WF_GPAD + tc + 4) * net.Hp + h;
                const size_t srow = (size_t)(GP - 1) * net.Hp;
                const float4* wr = wl + (size_t)(tc - tc_lo) * WF_ROW_F4;
                float4 xv[TAPS];
                // Plain (L1-allocating) loads: the values were stored by CTAs of THIS cluster before the cluster barrier, whose
                // acquire makes them visible to weak loads as well, and neighbouring positions share most of their 25 taps -- with
                // ld.global.cg every tap of every lane went to L2 (90 KB per CTA and layer, 1.6 us); through L1 only the first touch does.
#pragma unroll
                for (int kh = 0; kh < 5; kh++)
#pragma unroll
                    for (int kw = 0; kw < 5; kw++) xv[kh * 5 + kw] = WF_TAP_LOAD(xr + (kh + kw) * srow + kh);
#ifdef LIC360_WF_FINE_TRACE
                if (phase_trace) {  // all 25 loads have landed when their sum is known
                    float acc = 0.f;
#pragma unroll
                    for (int t = 0; t < TAPS; t++) acc += xv[t].x;
                    if (acc == 123456.789f) u.x = 1.f;
                    phase(l, 0);
                }
#endif
#pragma unroll
                for (int kh = 0; kh < 5; kh++)
#pragma unroll
                    for (int kw = 0; kw < 5; kw++) {
                        const float4 x4 = xv[kh * 5 + kw];
                        const float xs[4] = {x4.x, x4.y, x4.z, x4.w};
#pragma unroll
                        for (int c = 0; c < 4; c++) {
                            const float4 w4 = wr[(kh * 5 + kw) * 4 + c];
                            fma4(u, xs[c], w4);
                        }
                    }
#ifdef LIC360_WF_FINE_TRACE
                if (phase_trace) { if (u.x == 123456.789f) u.y = 1.f; phase(l, 2); }
#endif
            }
            const float Q[4] = {0.f + u.x, 0.f + u.y, 0.f + u.z, 0.f + u.w};  // Q = 0 + q_0 (one canonical block)
            const float PR[4] = {p.pr.x + p.rr.x, p.pr.y + p.rr.y, p.pr.z + p.rr.z, p.pr.w + p.rr.w};
            const size_t fc = wf_fc_index(net.Dp, net.Hp, net.G, L.cout_g, n, d, tc, h);
            float v[4];
#pragma unroll
            for (int q = 0; q < 4; q++) {
                v[q] = 0.f;
                if (q >= L.cout_g) continue;
                float y = (PR[q] + Q[q]) + p.bs[q];
                if (L.slope) y = y > 0.f ? y : y * p.sl[q];
                if (L.rc) y = y + p.rs[q];
                v[q] = y;
                if (L.op) L.op[wf_fp_index(net.D, net.HS, L.Cout, n, tc * L.cout_g + q, d, h)] = y;
            }
            if (L.cout_g == 4) {
                *reinterpret_cast<float4*>(L.oc + fc) = make_float4(v[0], v[1], v[2], v[3]);
            } else {
#pragma unroll
                for (int q = 0; q < 4; q++)
                    if (q < L.cout_g) L.oc[fc + q] = v[q];
            }
        }
        phase(l, 1);
        if (l + 1 < WF_LAYERS) {
            if (has0) wf_chain4_prefetch(net, net.L[l + 1], n, par, d0, h0, tc0, pre);
            asm volatile("cp.async.wait_group 0;\n" ::: "memory");
            phase(l, 2);
            if (nc > 1) cg::this_cluster().sync();
            else __syncthreads();
        }
        phase(l, 3);
    }
    if (threadIdx.x == 0) WF_TRACE_MAX(net.G, sd.psum, WF_TR_CHAIN1);
    const WfTailPlan tail = wf_tail_plan(net, rank, nc, sd.psum + 1, smem_rows);
    wf_chain4_rows(net, rows, sd.psum, sd.start, sd.len, tid, nt, n, tail);
    wf_chain4_rtail(net, n, sd.psum + 1, tid, nt, tail);
    if (persist.enabled) {  // the next step prefetches the R sums the tail just stored (other CTAs of the cluster) before its go
        if (nc > 1) cg::this_cluster().sync();
        else __syncthreads();
    }
  }  // step
}

// Chain for single-group nets (the importance stream: G = 1, 144 channels).  A step is ONE anti-diagonal (<= min(H,W)
// positions) and the same-wavefront taps are the five with kh + kw == 4, all on that diagonal, so per layer
//   Q[pos][oc] = sum over (16-channel block jq | 4-channel chunk, kh, c) of X[pos + kh][c] * W[oc][kh][c]
// is a small dense product and the layer time is pure latency.  The cluster splits the OUTPUT CHUNKS: CTA r owns chunks
// [r*kpc, (r+1)*kpc) for all positions and keeps its slice of the next layer's weights in shared memory (cp.async, double
// buffered, issued a layer ahead).  The diagonal's activations never make a round trip through L2 inside the step: the
// epilogue of layer l stores its 4 channels straight into the activation tile of EVERY CTA of the cluster (distributed shared
// memory), the cluster barrier between layers publishes them, and layer l+1 starts computing right behind the barrier.  (The
// global frames are still written -- later steps' old / previous-wavefront kernels read them -- but nobody waits for that.)
// Warp task = (canonical block jq, 32 positions) for all kpc chunks of the CTA at once: one set of conflict-free float4
// activation reads (row stride cin_g + 4) feeds kpc independent accumulator chains, weights are broadcasts.
constexpr int C1_KB = 3;  // chunks a warp accumulates together
__global__ void __launch_bounds__(384, 1) wf_chain1_kernel(const __grid_constant__ WfNetDev net, int nc, int kpc, int lenp,
                                                         int cmax, WfRows rows, int dsm) {
    extern __shared__ float4 wf_sm1[];
    __shared__ unsigned long long wbar_mem;  // mbarrier of the weight staging
    cg::cluster_group cluster = cg::this_cluster();
    const int tid = threadIdx.x, nt = blockDim.x, lane = tid & 31, warp = tid >> 5, nwarps = nt >> 5;
    const int n = blockIdx.x / nc, rank = blockIdx.x % nc;
    // programmatic dependent launch: the old-term kernel of the next step may start as soon as every CTA of this kernel is
    // resident (it does not read anything this kernel writes); without that launch attribute this is a no-op
    asm volatile("griddepcontrol.launch_dependents;\n" ::: "memory");
    if (nc > 1) cluster.barrier_arrive();  // every CTA of the cluster is running before anyone stores into its shared memory
    const StepDesc sd = net.steps[*net.ctr];
    if (tid == 0) WF_TRACE_MIN(net.G, sd.psum, WF_TR_CHAIN0);
    const int par = sd.psum & 1, d = sd.psum, len = sd.len;
    const int hmin = max(0, d - net.W + 1);
    const int nqb_max = (cmax + CB - 1) / CB;
    const int xs = cmax + 4;                                            // padded row stride of the activation tile (floats)
    const int xt_floats = (lenp + 4) * xs;
    float4* wbuf = wf_sm1;                                              // [2][kpc][5][cmax] float4
    // dsm: input tile of layer l in half l & 1, filled by the previous layer's epilogues through distributed shared memory.
    // !dsm (diagonals too long for two tiles): one tile, reloaded from the L2-resident frame behind every cluster barrier.
    float* xt = reinterpret_cast<float*>(wbuf + (size_t)2 * kpc * 5 * cmax);   // [dsm ? 2 : 1][lenp + 4][xs]
    float4* part = reinterpret_cast<float4*>(xt + (size_t)(dsm ? 2 : 1) * xt_floats);  // [kpc][nqb_max][lenp]
    // [lenp][52]: the last layer's logits, gathered in CTA 0.  They live in weight buffer 0, which is idle by then: the last layer
    // (odd) computes out of buffer 1 and nothing is staged after it (host side checks that the buffer is large enough)
    static_assert(((WF_LAYERS - 1) & 1) == 1, "the logits reuse weight buffer 0 during the last layer");
    float* ylog = reinterpret_cast<float*>(wbuf);
    const unsigned wbar = (unsigned)__cvta_generic_to_shared(&wbar_mem);
    if (tid == 0) {
        mbar_init(wbar, 1);
        asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
    }
    __syncthreads();
    // rows hmin-2, hmin-1, hmin+len, hmin+len+1 of the diagonal are outside the image (or outside the frame's written part): zero;
    // rows 2 .. len+1 are completely rewritten by the producers of every layer
    for (int e = tid; e < (dsm ? 2 : 1) * 4 * xs; e += nt) {
        const int half = e / (4 * xs), r4 = (e / xs) % 4, c = e % xs;
        xt[(size_t)half * xt_floats + (size_t)(r4 < 2 ? r4 : len + r4) * xs + c] = 0.f;
    }
    // slot-0 epilogue item of this thread: (chunk kc0 + it / len, position it % len)
    WfPre pre;
    // weights of layer l (same-wavefront class, taps (kh, 4 - kh)) of this CTA's chunks: kn * 5 rows of cin_g float4, each one
    // contiguous in the packed array -> one bulk copy per row, issued by one thread, completing on the mbarrier
    unsigned wphase = 0;
    bool wpending = false;
    auto stage_weights = [&](int l) {
        const WfLayerDev& L = net.L[l];
        const int kc0 = rank * kpc, kn = max(0, min(kpc, L.cpg4 - kc0));
        if (!L.has_q || kn == 0) return;
        wpending = true;
        if (tid != nt - 32) return;  // lane 0 of the last warp: it has no product task when nqb * npg < nwarps
        const int cg = L.cin_g;
        const float4* src = reinterpret_cast<const float4*>(L.wq) + ((size_t)(net.nsets + n) * L.nchunk + kc0) * TAPS * cg;
        const unsigned dst = (unsigned)__cvta_generic_to_shared(wbuf + (size_t)(l & 1) * kpc * 5 * cmax);
        mbar_expect_tx(wbar, kn * 5 * cg * 16);
        for (int e = 0; e < kn * 5; e++) {
            const int kh = e % 5, k = e / 5;
            bulk_load(dst + 16u * (unsigned)(e * cmax), src + ((size_t)k * TAPS + kh * 5 + 4 - kh) * cg, cg * 16, wbar);
        }
    };
    auto wait_weights = [&]() {
        if (!wpending) return;
        mbar_wait(wbar, wphase);
        wphase ^= 1;
        wpending = false;
    };
    auto prefetch = [&](int l) {
        const WfLayerDev& L = net.L[l];
        const int kc0 = rank * kpc, kn = max(0, min(kpc, L.cpg4 - kc0));
        if (tid >= kn * len) return;
        const int kc = kc0 + tid / len, h = hmin + tid % len;
        pre.pr = __ldg(L.pbuf[par] + (((size_t)n * L.cpg4 + kc) * net.D + d) * net.HS + h);
        // layer 0 reads the symbols the scatter kernel wrote a moment ago: its previous-wavefront terms are evaluated here instead
        // of by one more launch in front of the chain
        if (l == 0) pre.rr = wf_r_layer0_c1(net, n, d, h, 0, kc);
        else pre.rr = __ldg(L.rbuf[par] + (((size_t)n * L.cpg4 + kc) * net.D + d) * net.HS + h);
        const size_t fc = wf_fc_index(net.Dp, net.Hp, 1, L.cout_g, n, d, 0, h) + kc * 4;
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const bool live = kc * 4 + q < L.cout_g;
            pre.bs[q] = live ? __ldg(L.bias + n * L.Cout + kc * 4 + q) : 0.f;
            pre.sl[q] = live && L.slope ? __ldg(L.slope + n * L.Cout + kc * 4 + q) : 0.f;
            pre.rs[q] = live && L.rc ? __ldcg(L.rc + fc + q) : 0.f;
        }
    };
    stage_weights(1);
    prefetch(0);
    // debug timeline (LIC360_WF_TRACE=2): ns spent by CTA 0 in the phases of every layer, accumulated behind the step slots
    const bool phase_trace = g_wf_trace && g_wf_trace_sel == 1 && blockIdx.x == 0 && tid == 0;
    unsigned long long tph = 0;
    auto phase = [&](int l, int ph) {
        if (!phase_trace) return;
        unsigned long long t_;
        asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_));
        if (ph >= 0) atomicAdd(g_wf_trace + (size_t)(net.nsteps + 2) * WF_TR_SLOTS + l * 4 + ph, t_ - tph);
        tph = t_;
    };
    if (nc > 1) cluster.barrier_wait();
    phase(0, -1);
    for (int l = 0; l < WF_LAYERS; l++) {
        const WfLayerDev& L = net.L[l];
        const int kc0 = rank * kpc, kn = max(0, min(kpc, L.cpg4 - kc0));
        if (l >= 1 && l + 1 < WF_LAYERS) {  // weights of layer l+1 (layer 1 was staged before the loop)
            stage_weights(l + 1);
        }
        phase(l, 0);
        if (L.has_q && kn > 0) {
            const int cg = L.cin_g;
            const float* xl = xt + (size_t)(dsm ? (l & 1) : 0) * xt_floats;  // rows hmin-2 .. hmin+len+1 of the diagonal
            if (!dsm) {  // one contiguous block of the channel-last frame, written by all CTAs of the cluster before the barrier
                const float4* xsrc = reinterpret_cast<const float4*>(L.xc + wf_fc_index(net.Dp, net.Hp, 1, cg, n, d, 0, hmin - 2));
                const int row_f4 = cg >> 2;
                for (int e = tid; e < (len + 4) * row_f4; e += nt) {
                    const int r = e / row_f4, c4 = e % row_f4;
                    *reinterpret_cast<float4*>(xt + (size_t)r * xs + 4 * c4) = __ldcg(xsrc + e);
                }
                __syncthreads();
            }
            const float4* wl = wbuf + (size_t)(l & 1) * kpc * 5 * cmax;
            const int npg = (len + 31) >> 5, nqb = L.nqb;
            for (int k0 = 0; k0 < kn; k0 += C1_KB) {
                const int kb = min(C1_KB, kn - k0);
                for (int wt = warp; wt < nqb * npg; wt += nwarps) {
                    const int pg = wt % npg, jq = wt / npg;
                    const int pos = pg * 32 + lane;
                    if (pos >= len) continue;
                    float4 u[C1_KB];
#pragma unroll
                    for (int k = 0; k < C1_KB; k++) u[k] = make_float4(0.f, 0.f, 0.f, 0.f);
                    const int cend = min((jq + 1) * CB, cg);
                    for (int c0 = jq * CB; c0 < cend; c0 += 4) {
                        float4 xv[5];
#pragma unroll
                        for (int kh = 0; kh < 5; kh++) xv[kh] = *reinterpret_cast<const float4*>(xl + (size_t)(pos + kh) * xs + c0);
#pragma unroll
                        for (int kh = 0; kh < 5; kh++) {
                            const float x4[4] = {xv[kh].x, xv[kh].y, xv[kh].z, xv[kh].w};
#pragma unroll
                            for (int c = 0; c < 4; c++) {
#pragma unroll
                                for (int k = 0; k < C1_KB; k++) {
                                    if (k >= kb) continue;  // warp-uniform
                                    const float4 w4 = wl[(size_t)((k0 + k) * 5 + kh) * cmax + c0 + c];
                                    fma4(u[k], x4[c], w4);
                                }
                            }
                        }
                    }
#pragma unroll
                    for (int k = 0; k < C1_KB; k++)
                        if (k < kb) part[((size_t)(k0 + k) * nqb_max + jq) * lenp + pos] = u[k];
                }
            }
            __syncthreads();
        }
        phase(l, 1);
        // ranks that consume this layer's output in the next layer (those that own output chunks there)
        const int nranks_next = (dsm && l + 1 < WF_LAYERS && net.L[l + 1].has_q) ? min(nc, (net.L[l + 1].cpg4 + kpc - 1) / kpc) : 0;
        float* xnext = xt + (size_t)((l + 1) & 1) * xt_floats;
        for (int it = tid; it < kn * len; it += nt) {
            const int k = it / len, pos = it % len, kc = kc0 + k, h = hmin + pos;
            WfPre p = pre;
            if (it != tid) {  // further slots (more items than threads): nothing was prefetched
                p.pr = __ldg(L.pbuf[par] + (((size_t)n * L.cpg4 + kc) * net.D + d) * net.HS + h);
                if (l == 0) p.rr = wf_r_layer0_c1(net, n, d, h, 0, kc);
                else p.rr = __ldg(L.rbuf[par] + (((size_t)n * L.cpg4 + kc) * net.D + d) * net.HS + h);
                const size_t fcr = wf_fc_index(net.Dp, net.Hp, 1, L.cout_g, n, d, 0, h) + kc * 4;
#pragma unroll
                for (int q = 0; q < 4; q++) {
                    const bool live = kc * 4 + q < L.cout_g;
                    p.bs[q] = live ? __ldg(L.bias + n * L.Cout + kc * 4 + q) : 0.f;
                    p.sl[q] = live && L.slope ? __ldg(L.slope + n * L.Cout + kc * 4 + q) : 0.f;
                    p.rs[q] = live && L.rc ? __ldcg(L.rc + fcr + q) : 0.f;
                }
            }
            float Q[4] = {0.f, 0.f, 0.f, 0.f};
            if (L.has_q)
                for (int j = 0; j < L.nqb; j++) {
                    const float4 v = part[((size_t)k * nqb_max + j) * lenp + pos];
                    Q[0] = Q[0] + v.x; Q[1] = Q[1] + v.y; Q[2] = Q[2] + v.z; Q[3] = Q[3] + v.w;
                }
            const float PR[4] = {p.pr.x + p.rr.x, p.pr.y + p.rr.y, p.pr.z + p.rr.z, p.pr.w + p.rr.w};
            const size_t fc = wf_fc_index(net.Dp, net.Hp, 1, L.cout_g, n, d, 0, h) + kc * 4;
            float v[4];
#pragma unroll
            for (int q = 0; q < 4; q++) {
                v[q] = 0.f;
                if (kc * 4 + q >= L.cout_g) continue;
                float y = (PR[q] + Q[q]) + p.bs[q];
                if (L.slope) y = y > 0.f ? y : y * p.sl[q];
                if (L.rc) y = y + p.rs[q];
                v[q] = y;
            }
            const float4 v4 = make_float4(v[0], v[1], v[2], v[3]);
            // next layer's input tile in every consuming CTA (cin_g of the next layer == cout_g of this one, a multiple of 4 there)
            if (nranks_next > 0 && kc * 4 + 3 < L.cout_g) {
                float* dst = xnext + (size_t)(pos + 2) * xs + kc * 4;
                if (nc > 1) {
                    for (int r = 0; r < nranks_next; r++) *reinterpret_cast<float4*>(cluster.map_shared_rank(dst, r)) = v4;
                } else {
                    *reinterpret_cast<float4*>(dst) = v4;
                }
            }
            if (l == WF_LAYERS - 1) {  // logits of the CDF rows, gathered in CTA 0
                float* yd = ylog + (size_t)pos * 52 + kc * 4;
                if (nc > 1) yd = cluster.map_shared_rank(yd, 0);
#pragma unroll
                for (int q = 0; q < 4; q++)
                    if (kc * 4 + q < L.cout_g) yd[q] = v[q];
            }
#pragma unroll
            for (int q = 0; q < 4; q++)
                if (kc * 4 + q < L.cout_g && L.op) L.op[wf_fp_index(net.D, net.HS, L.Cout, n, kc * 4 + q, d, h)] = v[q];
            if ((L.cout_g & 3) == 0) {
                *reinterpret_cast<float4*>(L.oc + fc) = v4;
            } else {
#pragma unroll
                for (int q = 0; q < 4; q++)
                    if (kc * 4 + q < L.cout_g) L.oc[fc + q] = v[q];
            }
        }
        phase(l, 2);
        if (l + 1 < WF_LAYERS) {
            prefetch(l + 1);
            wait_weights();
            if (nc > 1) cluster.sync();
            else __syncthreads();
        }
        phase(l, 3);
    }
    if (tid == 0) WF_TRACE_MAX(net.G, sd.psum, WF_TR_CHAIN1);
    // CDF rows of the step (EntropyTable over the 49 logits of every position): the last layer's epilogues stored the logits into
    // CTA 0's shared memory; one warp per symbol, then the host flag -- no further launch on the critical path of the stream
    if (nc > 1) cluster.sync();
    else __syncthreads();
    if (rank != 0) return;
    if (tid == 0) WF_TRACE_MIN(net.G, sd.psum, WF_TR_ROWS0);
    float* scratch = reinterpret_cast<float*>(part) + warp * 64;  // the partial sums are dead by now
    for (int l = warp; l < len; l += nwarps) {
        const int th = __ldg(net.idx + sd.start + l);
        const float* yp = ylog + (size_t)(th - hmin) * 52;
        entropy_row49_warp(yp[lane], lane + 32 < 49 ? yp[lane + 32] : -INFINITY, scratch, lane, 0, rows.rows + (size_t)l * 64);
    }
    __threadfence_system();
    __syncthreads();
    if (tid == 0) {
        __threadfence_system();  // thread 0's own fence between the barrier and the flag
        *reinterpret_cast<volatile int*>(rows.flag) = sd.psum + 1;
        WF_TRACE_MAX(net.G, sd.psum, WF_TR_ROWS1);
    }
}

// ------------------------------------------------------------------------------------------------ host side
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = nullptr;
    if (!fn) {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeTiledFn>(p);
    }
    return fn;
}

int wf_init(WfEngine& e, int G, int cpg, int nlast, int nsets, int H, int W, const int32_t* idx_dev, const StepDesc* steps_dev,
            const int* ctr_dev, int nsteps, int max_len) {
    WfNetDev& n = e.dev;
    memset(&n, 0, sizeof(n));
    n.nsets = nsets; n.G = G; n.H = H; n.W = W; n.Dp = H + W - 1 + 8; n.Hp = H + 4;
    n.D = H + W - 1; n.HS = (H + WF_HSHIFT + 3) & ~3;
    n.nsteps = nsteps; n.parts = (std::min(H, W) + 31) / 32; n.ndiag = std::min(G, n.D);
    n.steps = steps_dev; n.ctr = ctr_dev; n.idx = idx_dev;
    e.max_len = max_len;
    e.C[0] = G;  // network input: one channel per group
    for (int l = 0; l < WF_LAYERS; l++) e.C[l + 1] = G * (l == WF_LAYERS - 1 ? nlast : cpg);
    size_t pb = 0;
    for (int l = 0; l < WF_LAYERS; l++) {
        WfLayerDev& L = n.L[l];
        L.Cin = e.C[l]; L.Cout = e.C[l + 1];
        L.cin_g = L.Cin / G; L.cout_g = L.Cout / G; L.cpg4 = (L.cout_g + 3) / 4; L.nchunk = G * L.cpg4;
        L.nblk = (L.Cin + CB - 1) / CB; L.nqb = (L.cin_g + CB - 1) / CB; L.has_q = l != 0;
        e.cpg4_max = std::max(e.cpg4_max, L.cpg4); e.nblk_max = std::max(e.nblk_max, L.nblk); e.nqb_max = std::max(e.nqb_max, L.nqb);
        pb += 4 * (size_t)nsets * L.cpg4 * n.D * n.HS;  // P and R, two step parities each
    }
    if (e.nblk_max > 32) { set_error("wavefront engine: too many channels"); return LIC360_ERR_ARG; }
    // wf_prev_kernel runs one warp per canonical 16-channel block of a group's input channels, at most 10
    if (e.nqb_max > 10) { set_error("wavefront engine: more than 160 input channels per group"); return LIC360_ERR_ARG; }
    // a many-group net runs wf_chain4_kernel and wf_old4_kernel: at most 64 groups, one output chunk (<= 4 channels) per group
    // in every layer, 4 input channels per group in every layer after the first
    e.chain4 = G > 1 && G <= 64;
    for (int l = 0; l < WF_LAYERS; l++) e.chain4 = e.chain4 && n.L[l].cpg4 == 1 && (l == 0 || n.L[l].cin_g == 4);
    if (G > 1 && !e.chain4) {
        set_error("wavefront engine: a many-group net needs at most 64 groups, at most 4 output channels per group and 4 input "
                  "channels per group after the first layer");
        return LIC360_ERR_ARG;
    }
    e.old4 = G > 1;
    for (int i = 0; i <= WF_LAYERS; i++) {
        e.fc_floats[i] = (size_t)nsets * n.Dp * (G + 2 * WF_GPAD) * n.Hp * (e.C[i] / G);
        LIC360_CUDA(cudaMalloc(&e.fc[i], e.fc_floats[i] * sizeof(float)));
        if (i < WF_LAYERS) {
            e.fp_floats[i] = (size_t)nsets * e.C[i] * n.D * n.HS;
            LIC360_CUDA(cudaMalloc(&e.fp[i], e.fp_floats[i] * sizeof(float)));
        }
    }
    e.pbuf_f4 = pb;
    LIC360_CUDA(cudaMalloc(&e.pbuf, pb * sizeof(float4)));
    LIC360_CUDA(cudaMemset(e.pbuf, 0, pb * sizeof(float4)));
    float4* pp = e.pbuf;
    for (int l = 0; l < WF_LAYERS; l++) {
        WfLayerDev& L = n.L[l];
        L.xp = e.fp[l]; L.xc = e.fc[l];
        L.op = l + 1 < WF_LAYERS ? e.fp[l + 1] : nullptr;
        L.oc = e.fc[l + 1];
        L.rc = (l >= 2 && l <= 10 && (l % 2) == 0) ? e.fc[l - 1] : nullptr;  // conv2 of residual block b = layer 2b (y + x)
        for (int par = 0; par < 2; par++) { L.pbuf[par] = pp; pp += (size_t)nsets * L.cpg4 * n.D * n.HS; }
        for (int par = 0; par < 2; par++) { L.rbuf[par] = pp; pp += (size_t)nsets * L.cpg4 * n.D * n.HS; }
    }
    // TMA descriptors: FP frame of layer l as a 3-D tensor {HS, D, nsets*Cin}, box {40, 9, 4}, zero fill outside
    EncodeTiledFn enc = encode_tiled_fn();
    if (!enc) { set_error("wavefront engine: cuTensorMapEncodeTiled is not available from this driver"); return LIC360_ERR_CUDA; }
    for (int l = 0; l < WF_LAYERS; l++) {
        const cuuint64_t dims[3] = {(cuuint64_t)n.HS, (cuuint64_t)n.D, (cuuint64_t)nsets * e.C[l]};
        const cuuint64_t strides[2] = {(cuuint64_t)n.HS * 4, (cuuint64_t)n.D * n.HS * 4};
        const cuuint32_t box[3] = {WF_BOX_W, 9, WF_STAGE};
        const cuuint32_t estr[3] = {1, 1, 1};
        CUresult r = enc(&e.maps.tm[l], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, e.fp[l], dims, strides, box, estr,
                         CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                         CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { set_error("wavefront engine: cuTensorMapEncodeTiled failed (%d) for layer %d", (int)r, l); return LIC360_ERR_CUDA; }
        const cuuint32_t box4[3] = {WF4_BOX_W, WF4_ROWS, WF4_STAGE};
        r = enc(&e.maps4.tm[l], CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 3, e.fp[l], dims, strides, box4, estr,
                CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { set_error("wavefront engine: cuTensorMapEncodeTiled (10-row box) failed (%d) for layer %d", (int)r, l); return LIC360_ERR_CUDA; }
    }
    // launch shapes
    e.old_smem = 128 + (size_t)WF_OLD_WARPS * WF_STAGE_BYTES + (size_t)e.nblk_max * 32 * sizeof(float4) + (size_t)WF_OLD_WARPS * 8;
    // four positions per lane, two diagonals per warp for the many-group nets (e.old4).  The single-group net keeps the
    // one-position kernel: its diagonals are short (half-empty warps) and its old-term launch is latency-, not throughput-critical
    // (twice as many TMA round trips per warp made the importance stream gate the code stream at 2048x4096).
    e.parts4 = 1;
    for (int d = 0; d < n.D; d++) {  // a diagonal's tile starts at the multiple of 4 below its first row
        const int hmin = std::max(0, d - W + 1), hmax = std::min(H - 1, d);
        e.parts4 = std::max(e.parts4, (hmax - (hmin & ~3) + 64) / 64);
    }
    e.old4_smem = 128 + (size_t)WF_OLD_WARPS * WF4_STAGE_BYTES + (size_t)e.nblk_max * 128 * sizeof(float4) + (size_t)WF_OLD_WARPS * 8;
    e.prev_wcap = 0;
    for (int l = 0; l < WF_LAYERS; l++) e.prev_wcap = std::max(e.prev_wcap, TAPS * n.L[l].cin_g);
    e.prev_smem = ((size_t)e.prev_wcap + (size_t)e.nqb_max * 32) * sizeof(float4);
    // the attribute is per kernel AND per device, not per engine: only ever raise it (two engines with different channel counts
    // share it), and remember it for every device separately (SmemAttr, common.cuh)
    static SmemAttr prev_attr, old_attr, old4_attr, chain_attr_g, chain_attr_4, chain_attr_1;
    LIC360_CUDA(prev_attr.ensure(wf_prev_kernel<320>, e.prev_smem));
    LIC360_CUDA(old_attr.ensure(wf_old_kernel, e.old_smem));
    LIC360_CUDA(old4_attr.ensure(wf_old4_kernel, e.old4_smem));
    // chain kernels: one cluster per net.  16 CTAs (non-portable size, opt-in) when the device can co-schedule them,
    // else the portable maximum of 8.
    LIC360_CUDA(cudaFuncSetAttribute(wf_chain_kernel<384>, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    LIC360_CUDA(cudaFuncSetAttribute(wf_chain4_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    LIC360_CUDA(cudaFuncSetAttribute(wf_chain1_kernel, cudaFuncAttributeNonPortableClusterSizeAllowed, 1));
    // many-group nets (3 clusters, old-term kernel running beside them): 8 CTAs each measured best; the single-group net
    // has one cluster and splits output chunks: 16
    int want = G > 1 ? 8 : 16;
    if (const char* s = getenv(G > 1 ? "LIC360_WF_CLUSTER_CODE" : "LIC360_WF_CLUSTER_IMP")) want = std::max(1, std::min(16, atoi(s)));
    // the one limit of every chain kernel's dynamic shared memory: the per-block opt-in maximum (227 KB on B200) minus the largest
    // static shared memory of the three kernels
    int dev = 0, optin = 0;
    LIC360_CUDA(cudaGetDevice(&dev));
    LIC360_CUDA(cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, dev));
    size_t static_max = 0;
    cudaFuncAttributes fa;
    LIC360_CUDA(cudaFuncGetAttributes(&fa, wf_chain_kernel<384>)); static_max = std::max(static_max, fa.sharedSizeBytes);
    LIC360_CUDA(cudaFuncGetAttributes(&fa, wf_chain4_kernel)); static_max = std::max(static_max, fa.sharedSizeBytes);
    LIC360_CUDA(cudaFuncGetAttributes(&fa, wf_chain1_kernel)); static_max = std::max(static_max, fa.sharedSizeBytes);
    const size_t cap = (size_t)optin - static_max;
    for (e.cluster = want;; e.cluster = 8) {
        int tasks_max = 0;
        for (int l = 0; l < WF_LAYERS; l++) {
            const int per = (max_len * n.L[l].cpg4 + e.cluster - 1) / e.cluster;
            tasks_max = std::max(tasks_max, per * (n.L[l].has_q ? n.L[l].nqb : 1));
        }
        // a kernel row of an item (5 activations + 20 weight vectors) is kept in registers: at most 384 threads per CTA
        // (168 registers each); CTAs with more tasks loop
        e.chain_threads = std::min(384, std::max(128, ((tasks_max + 31) / 32) * 32));
        e.chain_tasks = tasks_max;
        e.chain_smem = (size_t)tasks_max * sizeof(float4);
        e.chain1 = G == 1;
        e.c1_cmax = 4;
        for (int l = 1; l < WF_LAYERS; l++) { e.chain1 = e.chain1 && (n.L[l].cin_g & 3) == 0; e.c1_cmax = std::max(e.c1_cmax, n.L[l].cin_g); }
        if (e.chain4) e.chain_smem = (size_t)2 * G * WF_ROW_F4 * sizeof(float4);
        if (e.chain1) {
            e.c1_kpc = (e.cpg4_max + e.cluster - 1) / e.cluster;
            e.c1_lenp = ((max_len + 31) / 32) * 32;
            const size_t wbuf1 = (size_t)e.c1_kpc * 5 * e.c1_cmax * sizeof(float4);                  // one weight buffer
            const size_t tile = (size_t)(e.c1_lenp + 4) * (e.c1_cmax + 4) * sizeof(float);            // one activation tile
            const size_t parts = (size_t)e.c1_kpc * ((e.c1_cmax + CB - 1) / CB) * e.c1_lenp * sizeof(float4);
            const bool logits_fit = (size_t)e.c1_lenp * 52 * sizeof(float) <= wbuf1;                 // they reuse weight buffer 0
            e.c1_dsm = logits_fit && 2 * wbuf1 + 2 * tile + parts <= cap;   // activations exchanged through distributed shared memory
            const size_t sm = 2 * wbuf1 + (e.c1_dsm ? 2 : 1) * tile + parts;
            if (logits_fit && sm <= cap) { e.chain_smem = sm; e.chain_threads = 384; }
            else e.chain1 = false;  // too large for shared memory: the generic chain kernel handles it
        }
        if (e.chain_smem > cap) { set_error("wavefront engine: slab too large for the chain kernel"); return LIC360_ERR_ARG; }
        // The old-term kernel of the next step runs concurrently (programmatic dependent launch): claim the whole shared
        // memory of the SM so that none of its CTAs lands next to a chain CTA and steals its issue slots.
        e.chain_smem = std::max(e.chain_smem, (size_t)196 * 1024);
        LIC360_CUDA(chain_attr_g.ensure(wf_chain_kernel<384>, e.chain_smem));
        LIC360_CUDA(chain_attr_4.ensure(wf_chain4_kernel, e.chain_smem));
        LIC360_CUDA(chain_attr_1.ensure(wf_chain1_kernel, e.chain_smem));
        if (e.cluster <= 8) break;
        // can nsets clusters of this size be resident at once?
        cudaLaunchConfig_t cfg;
        memset(&cfg, 0, sizeof(cfg));
        cfg.gridDim = dim3(nsets * e.cluster); cfg.blockDim = dim3(e.chain_threads); cfg.dynamicSmemBytes = e.chain_smem;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = e.cluster; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        int nclusters = 0;
        cudaError_t r = e.chain4 ? cudaOccupancyMaxActiveClusters(&nclusters, wf_chain4_kernel, &cfg)
                      : e.chain1 ? cudaOccupancyMaxActiveClusters(&nclusters, wf_chain1_kernel, &cfg)
                                 : cudaOccupancyMaxActiveClusters(&nclusters, wf_chain_kernel<384>, &cfg);
        if (r == cudaSuccess && nclusters >= nsets) break;
        cudaGetLastError();
    }
    return LIC360_OK;
}

// How many decodes may run their code-stream chain concurrently on this device without risking the deadlock of partially
// resident grids: the chain kernel's clusters wait for each other at a global counter (wf_chain4_rows), so ALL nsets clusters of
// every running chain must be resident at once.
int wf_chain_capacity(const WfEngine& e) {
    if (!e.chain4) return 1 << 20;  // the other chain kernels have no inter-cluster wait
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(e.dev.nsets * e.cluster); cfg.blockDim = dim3(e.chain_threads); cfg.dynamicSmemBytes = e.chain_smem;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = e.cluster; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr; cfg.numAttrs = e.cluster > 1 ? 1 : 0;
    int nclusters = 0;
    if (cudaOccupancyMaxActiveClusters(&nclusters, wf_chain4_kernel, &cfg) != cudaSuccess) { cudaGetLastError(); return 1; }
    return std::max(1, nclusters / e.dev.nsets);
}

int wf_tail_rounds(const WfEngine& e, const int32_t* idx, const StepDesc* steps) {
    if (!e.chain4) return 0;
    const int smem_rows = (int)(e.chain_smem / (WF_ROW_F4 * sizeof(float4)));  // as wf_launch_chain passes it
    int rounds = 0;
    for (int p = 1; p < e.dev.nsteps; p++)
        for (int rank = 0; rank < e.cluster; rank++) {
            const WfTailPlan t = wf_tail_plan_of(idx, e.dev.H * e.dev.W, steps[p], rank, e.cluster, p, smem_rows);
            if (t.nloc > 0) rounds = std::max(rounds, (WF_LAYERS - 1 + t.lpg - 1) / t.lpg);
        }
    return rounds;
}

const void* wf_old_kernel_ptr() { return reinterpret_cast<const void*>(&wf_old_kernel); }

void wf_set_layer(WfEngine& e, int l, const float* wp, const float* wq, const float* bias, const float* slope) {
    WfLayerDev& L = e.dev.L[l];
    L.wp = wp; L.wq = wq; L.bias = bias; L.slope = slope;
}

void wf_free(WfEngine& e) {
    for (int i = 0; i <= WF_LAYERS; i++) { cudaFree(e.fp[i]); cudaFree(e.fc[i]); e.fp[i] = e.fc[i] = nullptr; }
    cudaFree(e.pbuf);
    e.pbuf = nullptr;
}

cudaError_t wf_clear(const WfEngine& e, cudaStream_t s) {
    for (int i = 0; i <= WF_LAYERS; i++) {
        cudaError_t r = cudaMemsetAsync(e.fc[i], 0, e.fc_floats[i] * sizeof(float), s);
        if (r != cudaSuccess) return r;
        if (i < WF_LAYERS && (r = cudaMemsetAsync(e.fp[i], 0, e.fp_floats[i] * sizeof(float), s)) != cudaSuccess) return r;
    }
    return cudaMemsetAsync(e.pbuf, 0, e.pbuf_f4 * sizeof(float4), s);
}

// behind an old-term launch in the same stream: the sums of steps < value are complete and visible
__global__ void wf_old_done_kernel(int* done, int value) {
    __threadfence();
    *reinterpret_cast<volatile int*>(done) = value;
}

cudaError_t wf_launch_old(const WfEngine& e, int dp, cudaStream_t s, bool programmatic, int psum, int* done, const int* scat_done) {
    if (psum >= 0 && !e.old4) return cudaErrorInvalidValue;  // explicit steps: many-group engines only
    const WfNetDev& n = e.dev;
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = e.old4 ? dim3(WF_LAYERS * n.nsets, 1, ((n.ndiag + 1) / 2) * e.parts4)
                         : dim3(WF_LAYERS * n.nsets, e.cpg4_max, n.ndiag * n.parts);
    cfg.blockDim = dim3(32, WF_OLD_WARPS);
    cfg.dynamicSmemBytes = e.old4 ? e.old4_smem : e.old_smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;  // start once the previous kernel's CTAs have all
    attr[0].val.programmaticStreamSerializationAllowed = 1;          // executed griddepcontrol.launch_dependents
    cfg.attrs = attr;
    cfg.numAttrs = programmatic ? 1 : 0;
    g_launches++;
    const cudaError_t err = e.old4 ? cudaLaunchKernelEx(&cfg, wf_old4_kernel, n, e.maps4, dp, e.parts4, psum, scat_done)
                                   : cudaLaunchKernelEx(&cfg, wf_old_kernel, n, e.maps, dp);
    if (err != cudaSuccess) return err;
    if (done) {
        wf_old_done_kernel<<<1, 1, 0, s>>>(done, psum + 1);
        g_launches++;
        return cudaGetLastError();
    }
    return cudaSuccess;
}

cudaError_t wf_launch_prev(const WfEngine& e, int dp, int l0, int l1, cudaStream_t s) {
    const WfNetDev& n = e.dev;
    int cpg4 = 0, nqb = 0;
    for (int l = l0; l < l1; l++) { cpg4 = std::max(cpg4, n.L[l].cpg4); nqb = std::max(nqb, n.L[l].nqb); }
    dim3 grid(n.ndiag * n.parts, cpg4, (l1 - l0) * n.nsets), block(32, nqb);
    wf_prev_kernel<320><<<grid, block, e.prev_smem, s>>>(n, e.prev_wcap, dp, l0);  // nqb <= 10 (wf_init)
    g_launches++;
    return cudaGetLastError();
}

cudaError_t wf_launch_chain(const WfEngine& e, cudaStream_t s, const WfRows& rows, const WfPersist* persist) {
    WfPersist ps;
    memset(&ps, 0, sizeof(ps));
    if (persist) {
        if (!e.chain4) return cudaErrorInvalidValue;
        ps = *persist;
        ps.enabled = 1;
    }
    const WfNetDev& n = e.dev;
    cudaLaunchConfig_t cfg;
    memset(&cfg, 0, sizeof(cfg));
    cfg.gridDim = dim3(n.nsets * e.cluster);
    cfg.blockDim = dim3(e.chain_threads);
    cfg.dynamicSmemBytes = e.chain_smem;
    cfg.stream = s;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = e.cluster; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    cfg.attrs = attr;
    cfg.numAttrs = e.cluster > 1 ? 1 : 0;
    g_launches++;
    if (e.chain4) return cudaLaunchKernelEx(&cfg, wf_chain4_kernel, n, e.cluster, n.G, rows, ps, (int)(e.chain_smem / (WF_ROW_F4 * sizeof(float4))));
    if (e.chain1) return cudaLaunchKernelEx(&cfg, wf_chain1_kernel, n, e.cluster, e.c1_kpc, e.c1_lenp, e.c1_cmax, rows, (int)e.c1_dsm);
    return cudaLaunchKernelEx(&cfg, wf_chain_kernel<384>, n, e.cluster);
}

}  // namespace lic360
