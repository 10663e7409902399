// Device helpers shared by the per-op context-conv kernels (conv.cu) and the wavefront engine of the fused decoder
// (wavefront.cu): one definition of the canonical per-stage arithmetic (see the header of conv.cu), so that every
// kernel that produces a context-conv output produces the same bits.
#pragma once
#include "common.cuh"

namespace lic360 {

constexpr int CB = 16;    // canonical input-channel block
constexpr int TAPS = 25;  // 5x5
constexpr int DC_BAND = 36 * 9;          // cells per channel
constexpr int DC_STAGE = 4;              // channels staged per round
constexpr int DC_WARP_FLOATS = DC_STAGE * DC_BAND + DC_STAGE * TAPS * 4;  // band + weights of one stage

__device__ __forceinline__ void cp_async4(unsigned dst, const void* src, bool valid) {
    asm volatile("cp.async.ca.shared.global [%0], [%1], 4, %2;\n" ::"r"(dst), "l"(src), "r"(valid ? 4 : 0));
}
__device__ __forceinline__ void cp_async16(unsigned dst, const void* src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(dst), "l"(src));
}
// 16-byte copy, zero-filled when !valid (src must still be a valid address)
__device__ __forceinline__ void cp_async16z(unsigned dst, const void* src, bool valid) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;\n" ::"r"(dst), "l"(src), "r"(valid ? 16 : 0));
}
__device__ __forceinline__ void cp_async_wait_all() {
    asm volatile("cp.async.commit_group;\n" ::);
    asm volatile("cp.async.wait_group 0;\n" ::: "memory");
}

// 100 taps of one stage out of shared memory: x from the band (row stride 9: conflict free), weights broadcast
// old terms only: taps with kh + kw >= tc + 3 - group(channel) carry a zero weight and are skipped (warp-uniform)
// band cell of position `lane`, tap (kh,kw): band[ch*DC_BAND + (lane+kh)*RS + (kh+kw)*CS]
//   NCHW kernel  : rows = image rows, 9 columns         -> RS = 9, CS = 1,  CHS = 324
//   skewed kernel: rows = diagonals (kh+kw), 40 columns -> RS = 1, CS = 40, CHS = 360 (TMA box, wavefront.cu)
// u += x * w for the 4 output channels of a chunk.  With LIC360_FFMA2 the four fp32 FMAs are issued as two packed
// fma.rn.f32x2 (sm_100: two IEEE fp32 FMAs per instruction, bit-identical results, half the FMA issue slots).
__device__ __forceinline__ void fma4(float4& u, float xx, const float4& w4) {
#ifdef LIC360_FFMA2
    asm("{\n"
        ".reg .b64 xa, wa, wb, ua, ub;\n"
        "mov.b64 xa, {%4, %4};\n"
        "mov.b64 wa, {%5, %6};\n"
        "mov.b64 wb, {%7, %8};\n"
        "mov.b64 ua, {%0, %1};\n"
        "mov.b64 ub, {%2, %3};\n"
        "fma.rn.f32x2 ua, xa, wa, ua;\n"
        "fma.rn.f32x2 ub, xa, wb, ub;\n"
        "mov.b64 {%0, %1}, ua;\n"
        "mov.b64 {%2, %3}, ub;\n"
        "}\n"
        : "+f"(u.x), "+f"(u.y), "+f"(u.z), "+f"(u.w)
        : "f"(xx), "f"(w4.x), "f"(w4.y), "f"(w4.z), "f"(w4.w));
#else
    u.x = fmaf(xx, w4.x, u.x);
    u.y = fmaf(xx, w4.y, u.y);
    u.z = fmaf(xx, w4.z, u.z);
    u.w = fmaf(xx, w4.w, u.w);
#endif
}

// taps with kh + kw < NS, fully unrolled with compile-time tap predicates (no per-tap compare/branch at run time)
template <int RS, int CS, int NS>
__device__ __forceinline__ void dc_taps_fma(const float* bw, const float4* wrow, float4& u) {
#pragma unroll
    for (int kh = 0; kh < 5; kh++) {
#pragma unroll
        for (int kw = 0; kw < 5; kw++) {
            if (kh + kw >= NS) continue;
            const float xx = bw[kh * RS + (kh + kw) * CS];
            const float4 w4 = wrow[kh * 5 + kw];
            fma4(u, xx, w4);
        }
    }
}

template <int RS, int CS, int CHS>
__device__ __forceinline__ void dc_stage_fma(const float* band, const float4* wsm, int nc, int lane, int chan0, int cin_g,
                                             int tc, float4& u) {
    for (int ch = 0; ch < nc; ch++) {
        const float* bw = band + ch * CHS + lane * RS;
        const float4* wrow = wsm + ch * TAPS;
        const int bound = tc + 3 - (chan0 + ch) / cin_g;  // warp-uniform
        if (bound >= 9) { dc_taps_fma<RS, CS, 9>(bw, wrow, u); continue; }
        switch (bound) {
            case 8: dc_taps_fma<RS, CS, 8>(bw, wrow, u); break;
            case 7: dc_taps_fma<RS, CS, 7>(bw, wrow, u); break;
            case 6: dc_taps_fma<RS, CS, 6>(bw, wrow, u); break;
            case 5: dc_taps_fma<RS, CS, 5>(bw, wrow, u); break;
            case 4: dc_taps_fma<RS, CS, 4>(bw, wrow, u); break;
            case 3: dc_taps_fma<RS, CS, 3>(bw, wrow, u); break;
            case 2: dc_taps_fma<RS, CS, 2>(bw, wrow, u); break;
            case 1: dc_taps_fma<RS, CS, 1>(bw, wrow, u); break;
            default: break;
        }
    }
}

// Four adjacent positions of one diagonal per lane: 16 lanes cover 64 positions, and the other half-warp works on the NEXT diagonal
// of the same band (its band rows are one further down, its weight vectors belong to the next lower output group).  bw points at the
// 16-byte aligned cell of the lane's FIRST position for tap (0, 0); position i reads band cell [row][kh + i], so a row serves the four
// positions with the cells kh_min .. kh_max + 3: at most two aligned float4 (16 loads per channel for 400 FMAs).  A weight vector is
// one LDS.128 with ONE ADDRESS PER HALF-WARP -- the cost of a broadcast, 2 wavefronts (tools/lds_probe.cu) -- and feeds 16 FMAs.
// Per-accumulator FMA order = the canonical (kh, kw) order of dc_taps_fma.
template <int BW, int NS>
__device__ __forceinline__ void dc_taps_fma4(const float* bw, const float4* wrow, float4 (&u)[4]) {
    float cell[9][8];
#pragma unroll
    for (int r = 0; r < 9; r++) {
        if (r >= NS) continue;
        const int khmin = r > 4 ? r - 4 : 0, khmax = r < 4 ? r : 4;
#pragma unroll
        for (int m = 0; m < 8; m += 4) {
            if (m + 3 < khmin || m > khmax + 3) continue;
            const float4 v = *reinterpret_cast<const float4*>(bw + r * BW + m);
            cell[r][m] = v.x;
            cell[r][m + 1] = v.y;
            cell[r][m + 2] = v.z;
            cell[r][m + 3] = v.w;
        }
    }
#pragma unroll
    for (int kh = 0; kh < 5; kh++) {
#pragma unroll
        for (int kw = 0; kw < 5; kw++) {
            if (kh + kw >= NS) continue;
            const float4 w4 = wrow[kh * 5 + kw];
#pragma unroll
            for (int i = 0; i < 4; i++) fma4(u[i], cell[kh + kw][kh + i], w4);
        }
    }
}

// tc: the LARGER output group of the warp's pair (more old tap rows); the other half-warp's extra rows and channels carry zero weights
template <int BW, int CHS>
__device__ __forceinline__ void dc_stage_fma4(const float* bw0, const float4* wsm, int nc, int chan0, int cin_g, int tc, float4 (&u)[4]) {
    for (int ch = 0; ch < nc; ch++) {
        const float* bw = bw0 + ch * CHS;
        const float4* wrow = wsm + ch * TAPS;
        const int bound = tc + 3 - (chan0 + ch) / cin_g;  // warp-uniform
        if (bound >= 9) { dc_taps_fma4<BW, 9>(bw, wrow, u); continue; }
        switch (bound) {
            case 8: dc_taps_fma4<BW, 8>(bw, wrow, u); break;
            case 7: dc_taps_fma4<BW, 7>(bw, wrow, u); break;
            case 6: dc_taps_fma4<BW, 6>(bw, wrow, u); break;
            case 5: dc_taps_fma4<BW, 5>(bw, wrow, u); break;
            case 4: dc_taps_fma4<BW, 4>(bw, wrow, u); break;
            case 3: dc_taps_fma4<BW, 3>(bw, wrow, u); break;
            case 2: dc_taps_fma4<BW, 2>(bw, wrow, u); break;
            case 1: dc_taps_fma4<BW, 1>(bw, wrow, u); break;
            default: break;
        }
    }
}

// previous- (gsel0 = tc + 3) or same-wavefront (gsel0 = tc + 4) taps of one 4-channel chunk: canonical order (kh, kw, c)
template <int RS, int CS, int CHS>
__device__ __forceinline__ void dc_stage_q(const float* band, const float4* wsm, int nc, int lane, int gsel0, int G, float4& u) {
#pragma unroll
    for (int kh = 0; kh < 5; kh++) {
#pragma unroll
        for (int kw = 0; kw < 5; kw++) {
            const int gq = gsel0 - kh - kw;
            if (gq < 0 || gq >= G) continue;  // warp-uniform
            for (int ch = 0; ch < nc; ch++) {
                const float xx = band[ch * CHS + (lane + kh) * RS + (kh + kw) * CS];
                const float4 w4 = wsm[ch * TAPS + kh * 5 + kw];
                fma4(u, xx, w4);
            }
        }
    }
}


}  // namespace lic360
