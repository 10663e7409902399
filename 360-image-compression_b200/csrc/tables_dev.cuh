// Device functions that turn model outputs into integer CDF rows. Shared by the per-op kernels (tables.cu) and the
// fused codec kernels (codec.cu) so that both paths emit bit-identical tables.
// Bit-exact tier: every float/double promotion of the reference expressions is kept literally
// (entropy_gmm_table_cuda.cu:29-107, entropy_table_cuda.cu:24-76); do not compile with --use_fast_math.
#pragma once
#include <stdint.h>

namespace lic360 {

// strictly-increasing fix-up of one row (stride 1, ngroup+1 entries).
// gmm_rule: entropy_gmm_table_cuda.cu:85-107 tests T[i+1] <= T[i] (before adding the running bias),
// otherwise entropy_table_cuda.cu:53-76 tests T[i+1] + bias <= T[i].
__device__ __forceinline__ void fixup_row(float* o, int ngroup, bool gmm_rule) {
    float bias = 0.f, mval = 0.f;
    int midx = 0;
    for (int i = 0; i < ngroup; i++) {
        const bool bump = gmm_rule ? (o[i + 1] <= o[i]) : (o[i + 1] + bias <= o[i]);
        if (bump) bias += 1.f;
        o[i + 1] += bias;
        const float d = o[i + 1] - o[i];
        if (d > mval) { mval = d; midx = i; }
    }
    if (bias > 0.f)
        for (int i = midx; i < ngroup; i++) o[i + 1] -= bias;
}

// GMM row, part 1: wv = softmax of the mixture logits, dv = clamped delta, in place (what the reference writes back,
// entropy_gmm_table_cuda.cu:29-57)
__device__ __forceinline__ void gmm_prep(float* wv, float* dv, int ng, float beta) {
    float mval = wv[0], psum = 0.f;
    for (int i = 1; i < ng; i++) if (mval < wv[i]) mval = wv[i];
    for (int i = 0; i < ng; i++) { wv[i] = expf(wv[i] - mval); psum += wv[i]; }
    for (int i = 0; i < ng; i++) wv[i] = wv[i] / psum;
    for (int i = 0; i < ng; i++) { float t = dv[i]; dv[i] = t < 0 ? beta : t + beta; }
}

// GMM row, part 2: bin pt (1 <= pt <= nstep-1) from the prepared parameters (entropy_gmm_table_cuda.cu:60-83)
__device__ __forceinline__ float gmm_bin_value(const float* wv, const float* dv, const float* mv, int pt, int ng, float bias, float total,
                                               float s2) {
    float v = pt - 1 - bias + 0.5;  // (float)(pt-1) - bias in float, + 0.5 in double, rounded to float
    float ps = 0, f;
    for (int i = 0; i < ng; i++) {
        // reference: f = 0.5 + 0.5 * erff(..) evaluated in double and rounded to float.  0.5*e is exact and a double sum
        // of two floats rounded to float is the correctly rounded float sum (53 >= 2*24+2: innocuous double rounding), so
        // the single-rounding fmaf gives the same bits without the FP64 pipe.
        f = fmaf(0.5f, erff(s2 * (v - mv[i]) / dv[i]), 0.5f);
        ps = ps + wv[i] * f;                              // float, contracted to FFMA as in the reference
    }
    return static_cast<int>(total * ps + 0.5);  // float product, + 0.5 in double, truncation
}

// GMM row: wv/dv/mv hold the raw mixture logits / deltas / means on entry; on exit wv = softmax, dv = clamped delta
// (what the reference writes back in place); o receives nstep+1 bins.
__device__ __forceinline__ void gmm_row(float* wv, float* dv, const float* mv, float* o, int ng, int nstep, float bias,
                                        float total, float beta, float s2) {
    const int nt = nstep + 1;
    gmm_prep(wv, dv, ng, beta);
    o[0] = 0.f;
    o[nt - 1] = static_cast<int>(total);
    for (int pt = 1; pt < nt - 1; pt++) o[pt] = gmm_bin_value(wv, dv, mv, pt, ng, bias, total, s2);
    fixup_row(o, nstep, true);
}

// softmax row -> cumulative integer table. o has w+1 entries; on entry o[1+i] holds logit i.
__device__ __forceinline__ void entropy_row(float* o, int w, float total) {
    float mval = o[1], psum = 0.f;
    for (int i = 1; i < w; i++) if (mval < o[1 + i]) mval = o[1 + i];
    for (int i = 0; i < w; i++) { float t = expf(o[1 + i] - mval); o[1 + i] = t; psum += t; }
    o[0] = 0.f;
    const float dp = total / psum;
    float ts;
    for (int i = 0; i < w - 1; i++) {
        ts = o[i] + static_cast<int>(o[1 + i] * dp + 0.5);  // float product, + 0.5 in double, truncation
        o[i + 1] = ts < total ? ts : total;
    }
    o[w] = total;
    fixup_row(o, w, false);
}


// EntropyTable row of 49 logits by ONE WARP (the importance stream's rows sit on the critical path of the decoder: latency counts).
// Lanes hold logits i and i + 32 (v1 = -inf for i + 32 >= 49); the softmax denominator is accumulated in index order by every lane
// from shared memory (the serial order of entropy_row is part of the bit-exact contract), the cumulative table is a warp scan of
// integers (exact in fp32, so min(prefix, total) equals the serial clipped recurrence), lane 0 runs the serial fix-up and the warp
// stores the packed 128-byte row (coder_internal.h) with one coalesced write.  o: 64 floats of shared memory private to the warp.
__device__ __forceinline__ void entropy_row49_warp(float v0, float v1, float* o, int lane, int sym, uint16_t* dst) {
    const float total = 65536.f;
    const bool has1 = lane + 32 < 49;
    float m = fmaxf(v0, v1);
#pragma unroll
    for (int k = 16; k > 0; k >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, k));
    const float t0 = expf(v0 - m), t1 = has1 ? expf(v1 - m) : 0.f;
    __syncwarp();
    o[lane] = t0;
    if (has1) o[lane + 32] = t1;
    __syncwarp();
    float psum = 0.f;
    for (int i = 0; i < 49; i++) psum += o[i];   // index order, as the serial row
    const float dp = total / psum;
    const int a0 = static_cast<int>(t0 * dp + 0.5);                 // float product, + 0.5 in double, truncation
    const int a1 = has1 ? static_cast<int>(t1 * dp + 0.5) : 0;
    int s0 = a0, s1 = a1;
#pragma unroll
    for (int k = 1; k < 32; k <<= 1) {
        const int u0 = __shfl_up_sync(0xffffffffu, s0, k), u1 = __shfl_up_sync(0xffffffffu, s1, k);
        if (lane >= k) { s0 += u0; s1 += u1; }
    }
    s1 += __shfl_sync(0xffffffffu, s0, 31);
    __syncwarp();
    // T[i + 1] = min(prefix(i), total) for i < 48, T[0] = 0, T[49] = total
    if (lane == 0) { o[0] = 0.f; o[49] = total; }
    o[lane + 1] = fminf((float)s0, total);
    if (lane + 32 < 48) o[lane + 33] = fminf((float)s1, total);
    __syncwarp();
    if (lane == 0) fixup_row(o, 49, false);
    __syncwarp();
    // u16[0..47] = low words of T[1..48], [48] = symbol, [49..51] = bit 16 of T[1..48]
    const uint32_t e0 = lane < 24 ? (uint32_t)(int)o[2 * lane + 1] : 0u, e1 = lane < 24 ? (uint32_t)(int)o[2 * lane + 2] : 0u;
    const uint32_t be = __ballot_sync(0xffffffffu, lane < 24 && ((e0 >> 16) & 1u));
    const uint32_t bo = __ballot_sync(0xffffffffu, lane < 24 && ((e1 >> 16) & 1u));
    uint32_t ovf[3];
#pragma unroll
    for (int mth = 0; mth < 3; mth++) {
        uint32_t wv = 0;
#pragma unroll
        for (int q = 0; q < 8; q++) wv |= (((be >> (8 * mth + q)) & 1u) << (2 * q)) | (((bo >> (8 * mth + q)) & 1u) << (2 * q + 1));
        ovf[mth] = wv;
    }
    uint32_t word = 0;
    if (lane < 24) word = (e0 & 0xFFFFu) | ((e1 & 0xFFFFu) << 16);
    else if (lane == 24) word = ((uint32_t)sym & 0xFFFFu) | (ovf[0] << 16);
    else if (lane == 25) word = ovf[1] | (ovf[2] << 16);
    reinterpret_cast<uint32_t*>(dst)[lane] = word;
    __syncwarp();
}

// The symbol and mask rules of the encoder, shared by the kernels that pack rows for the host coder and the ones that cost the
// symbols without it (codec.cu), so the two cannot disagree on a fractional, negative or NaN input.
// code stream: 0..7, anything else (NaN included) is the out-of-range marker 8
__device__ __forceinline__ int code_symbol(float cv) { return (cv >= 0.f && cv < 8.f) ? (int)cv : 8; }
// code stream: a position is coded unless its mask is below 0.5 (NaN is coded)
__device__ __forceinline__ int code_mask_bit(float m) { return m < 0.5f ? 0 : 1; }
// importance stream: the level as the packed row stores it (u16); 49 or more is out of range
__device__ __forceinline__ uint32_t imp_symbol(float level) { return (uint16_t)(int)level; }

// bins T[s], T[s+1] (0 <= s < N) of a row of N symbols as the host coder reads them back from the packed row: T[0] = 0 and
// T[N] = 65536 are implied, the interior bins are the low 17 bits of (int)o[j] (16-bit word + overflow bit, pack_gmm_row /
// imp_rows_kernel).  Selected in an unrolled loop, so a row held in registers is not indexed dynamically.
template <int N>
__device__ __forceinline__ void coded_bins(const float* o, int s, uint32_t* lo, uint32_t* hi) {
    uint32_t a = 0u, b = 65536u;
#pragma unroll
    for (int j = 1; j < N; j++) {
        const uint32_t v = (uint32_t)(int)o[j] & 0x1FFFFu;
        if (j == s) a = v;
        if (j == s + 1) b = v;
    }
    *lo = a;
    *hi = b;
}

// packed code-stream row (coder_internal.h): 7 x u16 low words of T[1..7] + meta = sym | bad << 3 | mask << 8 | overflow bits << 9
// bad: the symbol is outside 0..7 (sym >= 8 or negative); the host encoder reports it like the per-op path does ("symbol out
// of range") instead of coding a wrapped, decodable but wrong symbol
// tag (4 bits, meta bits 4..7): publication tag of the decoder's per-step rows (wavefront.cu): a row is ONE aligned 16-byte store, so
// the host can validate every row by its tag instead of waiting for a fence + flag behind all of them
__device__ __forceinline__ void pack_gmm_row(const float* o, int sym, int maskbit, uint16_t* dst, int tag = 0) {
    uint32_t ovf = 0;
    uint16_t w[8];
#pragma unroll
    for (int j = 1; j <= 7; j++) {
        const uint32_t v = (uint32_t)(int)o[j];
        w[j - 1] = (uint16_t)(v & 0xFFFF);
        ovf |= ((v >> 16) & 1u) << (j - 1);
    }
    w[7] = (uint16_t)((sym & 7) | ((unsigned)sym > 7u ? 8 : 0) | ((tag & 15) << 4) | (maskbit << 8) | (ovf << 9));
    *reinterpret_cast<uint4*>(dst) = *reinterpret_cast<const uint4*>(w);
}


}  // namespace lic360
