// Tensor-core form of the encoder's old-term pass (P terms of CconvEc), OPT-IN (LIC360_EC_MMA=1).
//
// north_star asks for the masked context conv on tensor cores with fp32 accumulation in a fixed reduction order.  This kernel is
// that design for the whole-frame (encode) form, on the legacy tensor path: mma.sync.m16n8k8 TF32 (SASS HMMA.1688.F32.TF32) with
// the error-compensated 3-way split that the 1e-5 float tier needs,
//     x * w  ~=  x_lo*w_hi + x_hi*w_lo + x_hi*w_hi,     v_hi = v & 0xffffe000 (10-bit mantissa), v_lo = (v - v_hi) & 0xffffe000
// accumulated inside the tensor core for one canonical 16-channel block (2 stages x 25 taps x 3 MMAs), then folded into the fp32 sum
// P with an IEEE add -- the tensor core's accumulator rounds toward zero (tools/mma_probe.cu: 1 + 1.5*2^-24 -> 1), so short
// chains + RN folds keep the bias at the level of the sequential fp32 chain (measured: 2.4e-6 vs 1.5e-6 over K = 4800).
// Implicit GEMM: M = positions (a warp owns one image row of the 8x32 tile: two m16 tiles), N = 32 output channels of the CTA
// (four n8 tiles), K = 8 input channels of one tap per MMA; A fragments come straight out of the halo'd activation tile (channel
// stride padded to 440 floats: conflict-free), B fragments out of the masked weight tile (chunk stride padded to 816 floats).
// k-steps whose weights are all masked for an n-tile are skipped (warp-uniform); the probe shows that an all-zero B column leaves
// the accumulator untouched, so skipping and multiplying by zero are interchangeable.
//
// Why it is not the default (DESIGN.md s3, measured): mma.sync TF32 runs at 276 TFLOP/s on B200 = 3.7x the fp32 FMA peak; the 3-way
// split leaves 1.2x, mask padding inside the 32-channel tile (~0.85) and issue overhead take the rest -- and the DECODER would have
// to replay the same MMA sequence per output on its N = 4 wavefront tiles (half of every n8 tile wasted) to stay bit-identical,
// which is slower than its SIMT kernels.  With this kernel enabled the encoder no longer matches the (SIMT) decoder bit for bit:
// it is a measurement and parity (1e-5 vs the reference) vehicle of the per-op CconvEc, not a codec path (the codec's run_ec_net
// calls launch_cconv_ec with allow_mma = false).
#include <cstdlib>
#include "internal.cuh"
#include "conv_dev.cuh"

namespace lic360 {

constexpr int MM_TH = 8, MM_TW = 32, MM_XH = MM_TH + 4, MM_XW = MM_TW + 4;
constexpr int MM_CHUNKS = 8;      // 32 output channels per CTA
constexpr int MM_SB = 8;          // input channels per stage = K of one MMA
constexpr int MM_XS = 440;        // channel stride of the x tile in floats (12*36 = 432 padded; 440 % 32 == 24)
constexpr int MM_WS = 204;        // chunk stride of the weight tile in float4 (8*25 = 200 padded; 816 floats, 816 % 32 == 16)
constexpr int MM_STAGE_FLOATS = MM_SB * MM_XS + MM_CHUNKS * MM_WS * 4;
constexpr int MM_SMEM_BYTES = 2 * MM_STAGE_FLOATS * (int)sizeof(float);

__device__ __forceinline__ void split_tf32(float v, uint32_t& hi, uint32_t& lo) {
    hi = __float_as_uint(v) & 0xffffe000u;
    lo = __float_as_uint(v - __uint_as_float(hi)) & 0xffffe000u;
}

__device__ __forceinline__ void mma_tf32(float (&d)[4], const uint32_t (&a)[4], uint32_t b0, uint32_t b1) {
    asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};\n"
                 : "+f"(d[0]), "+f"(d[1]), "+f"(d[2]), "+f"(d[3])
                 : "r"(a[0]), "r"(a[1]), "r"(a[2]), "r"(a[3]), "r"(b0), "r"(b1));
}

__global__ void __launch_bounds__(256, 2) cconv_ec_mma_kernel(const ConvArgs a) {
    extern __shared__ float4 mm_smem4[];
    float* smem = reinterpret_cast<float*>(mm_smem4);
    const int tid = threadIdx.x, lane = tid & 31, ty = tid >> 5;
    const int g = lane >> 2, t = lane & 3;
    const int tiles_w = (a.W + MM_TW - 1) / MM_TW;
    const int w0 = (blockIdx.x % tiles_w) * MM_TW, h0 = (blockIdx.x / tiles_w) * MM_TH;
    const int ny = (a.nchunk + MM_CHUNKS - 1) / MM_CHUNKS;
    const int ytile = ny - 1 - (int)blockIdx.y;  // heaviest output groups first
    const int chunk0 = ytile * MM_CHUNKS;
    const int n = blockIdx.z, set = n / a.per;
    const int Cin = a.Cin, H = a.H, W = a.W;
    const int last_chunk = min(chunk0 + MM_CHUNKS - 1, a.nchunk - 1);
    const int lim_tile = min(Cin, (last_chunk / a.cpg4 + 3) * a.cin_g);  // old terms: g_in <= g_out + 2
    const int nstage = (lim_tile + MM_SB - 1) / MM_SB;
    // per n-tile (chunks 2nt, 2nt+1): the largest output group it holds -> taps with kh + kw < g_hi + 3 - (first input group of the stage)
    int g_hi[4];
#pragma unroll
    for (int nt = 0; nt < 4; nt++) g_hi[nt] = min(chunk0 + 2 * nt + 1, a.nchunk - 1) / a.cpg4;

    float P[2][4][4], u[2][4][4];
#pragma unroll
    for (int mt = 0; mt < 2; mt++)
#pragma unroll
        for (int nt = 0; nt < 4; nt++)
#pragma unroll
            for (int r = 0; r < 4; r++) { P[mt][nt][r] = 0.f; u[mt][nt][r] = 0.f; }

    const float4* wp4 = reinterpret_cast<const float4*>(a.wp);
    const unsigned smem_s = (unsigned)__cvta_generic_to_shared(smem);
    auto issue = [&](int st) {
        const int buf = st & 1, cb8 = min(MM_SB, Cin - st * MM_SB);
        const unsigned xd = smem_s + (unsigned)buf * (MM_STAGE_FLOATS * 4), wd = xd + MM_SB * MM_XS * 4;
        // all 8 channel slots are written: slots beyond the layer's channels are zero-filled (they meet zero weights, but 0 * garbage
        // could be NaN)
        for (int e = tid; e < MM_SB * MM_XH * MM_XW; e += 256) {
            const int ci = e / (MM_XH * MM_XW), rem = e % (MM_XH * MM_XW), r = rem / MM_XW, c = rem % MM_XW;
            const int h = h0 + r - 2, w = w0 + c - 2;
            const bool ok = ci < cb8 && h >= 0 && h < H && w >= 0 && w < W;
            cp_async4(xd + 4u * (ci * MM_XS + rem), ok ? a.x + (((size_t)n * Cin + st * MM_SB + ci) * H + h) * W + w : a.x, ok);
        }
        for (int e = tid; e < MM_CHUNKS * MM_SB * TAPS; e += 256) {
            const int ch = e / (MM_SB * TAPS), r = e % (MM_SB * TAPS), ci = r / TAPS;
            const int chunk = chunk0 + ch;
            const bool ok = chunk < a.nchunk && ci < cb8;
            cp_async16z(wd + 16u * (ch * MM_WS + r), ok ? wp4 + (((size_t)set * a.nchunk + chunk) * Cin + st * MM_SB) * TAPS + r : wp4, ok);
        }
        asm volatile("cp.async.commit_group;\n" ::);
    };
    if (nstage > 0) issue(0);
    for (int st = 0; st < nstage; st++) {
        if (st + 1 < nstage) {
            issue(st + 1);
            asm volatile("cp.async.wait_group 1;\n" ::: "memory");
        } else {
            asm volatile("cp.async.wait_group 0;\n" ::: "memory");
        }
        __syncthreads();
        const float* xb = smem + (st & 1) * MM_STAGE_FLOATS;
        const float* wb = xb + MM_SB * MM_XS;  // [chunk][ci][tap][4] with chunk stride MM_WS float4
        const int grp0 = (st * MM_SB) / a.cin_g;  // first input group of the stage (the least masked one)
        const int ns_max = g_hi[3] + 3 - grp0;
        // A: row ty of the tile, positions col = mt*16 + g (+8), channels t (+4); B: k = channel t (+4), n = 8 channels of the n-tile:
        // chunk 2nt + g/4, lane channel g%4
        const float* xa = xb + t * MM_XS + ty * MM_XW + g;
        const float* wl = wb + ((g >> 2) * MM_WS + t * TAPS) * 4 + (g & 3);
#pragma unroll 1
        for (int kh = 0; kh < 5; kh++) {
#pragma unroll
            for (int kw = 0; kw < 5; kw++) {
                const int s = kh + kw;
                if (s >= ns_max) continue;  // CTA-uniform
                uint32_t ah[2][4], al[2][4];
#pragma unroll
                for (int mt = 0; mt < 2; mt++) {
                    const float* p = xa + kh * MM_XW + kw + mt * 16;
                    split_tf32(p[0], ah[mt][0], al[mt][0]);
                    split_tf32(p[8], ah[mt][1], al[mt][1]);
                    split_tf32(p[4 * MM_XS], ah[mt][2], al[mt][2]);
                    split_tf32(p[4 * MM_XS + 8], ah[mt][3], al[mt][3]);
                }
                // B fragments of the four n-tiles, then the three split terms TERM-major: consecutive MMAs hit different accumulator
                // tiles (the per-accumulator order lo*hi, hi*lo, hi*hi -- the canonical one -- is unchanged), so the tensor pipe does not
                // wait on the previous MMA of the same tile
                uint32_t bh[4][2], bl[4][2];
                bool live[4];
#pragma unroll
                for (int nt = 0; nt < 4; nt++) {
                    live[nt] = s < g_hi[nt] + 3 - grp0;  // else every weight of this n-tile is masked at this tap (CTA-uniform)
                    const float* q = wl + (2 * nt * MM_WS + kh * 5 + kw) * 4;
                    split_tf32(q[0], bh[nt][0], bl[nt][0]);
                    split_tf32(q[4 * TAPS * 4], bh[nt][1], bl[nt][1]);
                }
#pragma unroll
                for (int term = 0; term < 3; term++)
#pragma unroll
                    for (int nt = 0; nt < 4; nt++) {
                        if (!live[nt]) continue;
#pragma unroll
                        for (int mt = 0; mt < 2; mt++) {
                            if (term == 0) mma_tf32(u[mt][nt], al[mt], bh[nt][0], bh[nt][1]);
                            else if (term == 1) mma_tf32(u[mt][nt], ah[mt], bl[nt][0], bl[nt][1]);
                            else mma_tf32(u[mt][nt], ah[mt], bh[nt][0], bh[nt][1]);
                        }
                    }
            }
        }
        if ((st & 1) == 1 || st + 1 == nstage) {  // the canonical 16-channel block is complete: fold with IEEE adds
#pragma unroll
            for (int mt = 0; mt < 2; mt++)
#pragma unroll
                for (int nt = 0; nt < 4; nt++)
#pragma unroll
                    for (int r = 0; r < 4; r++) { P[mt][nt][r] = P[mt][nt][r] + u[mt][nt][r]; u[mt][nt][r] = 0.f; }
        }
        __syncthreads();
    }
    // accumulator fragment: regs 0,1 = position g, channels 2t, 2t+1 of the n-tile; regs 2,3 = position g + 8
    const int h = h0 + ty;
    if (h >= H) return;
#pragma unroll
    for (int nt = 0; nt < 4; nt++)
#pragma unroll
        for (int r = 0; r < 4; r++) {
            const int cn = 2 * t + (r & 1);                  // channel inside the n-tile
            const int chunk = chunk0 + 2 * nt + (cn >> 2), oc = (chunk % a.cpg4) * 4 + (cn & 3);
            if (chunk >= a.nchunk || oc >= a.cout_g) continue;
            const int g_out = chunk / a.cpg4;
            const size_t row = (((size_t)n * a.Cout + g_out * a.cout_g + oc) * H + h) * W;
#pragma unroll
            for (int mt = 0; mt < 2; mt++) {
                const int w = w0 + mt * 16 + g + (r >> 1) * 8;
                if (w < W) a.out[row + w] = P[mt][nt][r];
            }
        }
}

bool cconv_ec_mma_enabled() {
    const char* e = getenv("LIC360_EC_MMA");
    return e && e[0] == '1';
}

// P terms of the whole frame into a.out (the R / Q pass follows as for the SIMT kernel)
cudaError_t launch_cconv_ec_mma(const ConvArgs& a, cudaStream_t s) {
    static SmemAttr attr;
    cudaError_t e = attr.ensure(cconv_ec_mma_kernel, MM_SMEM_BYTES);
    if (e != cudaSuccess) return e;
    const int ny = (a.nchunk + MM_CHUNKS - 1) / MM_CHUNKS, nxy = ((a.W + MM_TW - 1) / MM_TW) * ((a.H + MM_TH - 1) / MM_TH);
    dim3 grid(nxy, ny, a.N);
    cconv_ec_mma_kernel<<<grid, 256, MM_SMEM_BYTES, s>>>(a);
    g_launches++;
    return cudaGetLastError();
}

}  // namespace lic360
