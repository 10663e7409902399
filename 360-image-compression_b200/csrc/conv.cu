// Masked 3-D context convolution: encode form (CconvEc, whole frame) and wavefront decode form (CconvDc).
// Replaces /root/reference/extension/cconv_ec_cuda.cu:54-339 and cconv_dc_cuda.cu:58-398.
//
// CANONICAL PER-OUTPUT ARITHMETIC (shared by the EC kernel, the per-op DC kernel and the wavefront engine of the fused
// decoder, wavefront.cu, so that encoder and decoder produce bit-identical fp32 values -- the arithmetic decoder
// desynchronises otherwise, SURVEY.md s7 hard part 1).  The terms of one output (h, w, g_out), wavefront p = h+w+g_out,
// are split by the wavefront q = p - g_out - 4 + kh + kw + g_in of the input they read:
//
//   glim(kh,kw) = g_out + 4 - kh - kw                      (mask rule, cconv_ec_cuda.cu:71)
//   P = 0                                                  "old": q <= p-2, i.e. input groups g_in <= glim - 2
//   for j in 0 .. ceil(Cin/16)-1:                          16-channel blocks, ascending
//       u = 0
//       for ci in block j (ascending): for kh in 0..4: for kw in 0..4:
//           if tap inside the image and ci/cin_g <= glim-2: u = fmaf(x[ci,ph,pw], W[o,ci,kh,kw], u)
//       P = P + u
//   R = terms of the previous wavefront  (q == p-1: g_in == glim - 1), Q = terms of the same wavefront (q == p:
//   g_in == glim, constrain 6 only); both in the same order, with gsel = glim - 1 resp. glim:
//   for jq in 0 .. ceil(cin_g/16)-1:                       16-channel blocks of the group (one block when cin_g <= 16)
//     r = 0
//     for c0 in 16*jq, 16*jq+4, ..:                        4-channel chunks of the block
//       for kh: for kw: if tap inside the image and 0 <= gsel < G:
//         for c in c0 .. min(c0+4, cin_g)-1:               r = fmaf(x[gsel*cin_g+c,ph,pw], W[o,gsel*cin_g+c,kh,kw], r)
//     R = R + r
//   out = ((P + R) + Q) + bias[o];  PReLU: out > 0 ? out : out*slope[o];  optional residual: out = out + r
//
// Terms that are skipped in one kernel and multiplied by an exact zero in the other give identical values
// (fmaf(x, 0, u) == u for finite x).  The three-way split is what makes the decoder pipeline: P of step p+1 only
// needs data of steps <= p-1 and is computed while step p is still on its critical path (R, then the 12-layer chain
// of Q terms, <= 25*cin_g MACs each).
#include <algorithm>
#include "internal.cuh"
#include "conv_dev.cuh"

namespace lic360 {

constexpr int TH = 8, TW = 32, XH = TH + 4, XW = TW + 4;  // EC spatial tile and its halo'd smem tile
constexpr int EC_CHUNKS = 8;                              // 8 four-channel output chunks (32 channels) per EC block
constexpr int EC_THREADS = 256;
constexpr int EC_SB = 8;                                  // input channels per pipeline stage (two stages = one canonical block)
constexpr int EC_SMEM_BYTES = 2 * (EC_SB * XH * XW + EC_CHUNKS * EC_SB * TAPS * 4) * (int)sizeof(float);

// ---------------------------------------------------------------------------------------------------------
// weight packing: W (nsets,Cout,Cin,5,5) -> Wp [set][chunk][ci][tap][4] ("old" terms, everything else zeroed) and
//                                           Wq [cls][set][chunk][tap][c][4], cls 0 = previous-wavefront terms (R),
//                                                                          cls 1 = same-wavefront terms (Q)
// chunk = g_out * cpg4 + (4-channel chunk inside the group); channels beyond cout_g are zero padding.
// ---------------------------------------------------------------------------------------------------------
__global__ void cconv_pack_kernel(const float* __restrict__ w, float* __restrict__ wp, float* __restrict__ wq,
                                  int nsets, int Cin, int Cout, int G, int constrain) {
    const int cin_g = Cin / G, cout_g = Cout / G, cpg4 = (cout_g + 3) / 4, nchunk = G * cpg4;
    const size_t np = (size_t)nsets * nchunk * Cin * TAPS * 4;
    const size_t nq = (size_t)nsets * nchunk * TAPS * cin_g * 4;  // per class
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < np + 2 * nq; i += (size_t)gridDim.x * blockDim.x) {
        if (i < np) {
            int q = i % 4;
            int tap = (i / 4) % TAPS;
            int ci = (i / (4 * TAPS)) % Cin;
            int chunk = (i / ((size_t)4 * TAPS * Cin)) % nchunk;
            int set = i / ((size_t)4 * TAPS * Cin * nchunk);
            int g_out = chunk / cpg4, oc = (chunk % cpg4) * 4 + q;
            int glim = g_out + 4 - tap / 5 - tap % 5;
            float v = 0.f;
            if (oc < cout_g && ci / cin_g <= glim - 2)
                v = w[(((size_t)set * Cout + g_out * cout_g + oc) * Cin + ci) * TAPS + tap];
            wp[i] = v;
        } else {
            const int cls = (i - np) >= nq;
            size_t k = i - np - (cls ? nq : 0);
            int q = k % 4;
            int c = (k / 4) % cin_g;
            int tap = (k / ((size_t)4 * cin_g)) % TAPS;
            int chunk = (k / ((size_t)4 * cin_g * TAPS)) % nchunk;
            int set = k / ((size_t)4 * cin_g * TAPS * nchunk);
            int g_out = chunk / cpg4, oc = (chunk % cpg4) * 4 + q;
            int gsel = g_out + 3 + cls - tap / 5 - tap % 5;
            float v = 0.f;
            if (oc < cout_g && (cls == 0 || constrain == 6) && gsel >= 0 && gsel < G)
                v = w[(((size_t)set * Cout + g_out * cout_g + oc) * Cin + gsel * cin_g + c) * TAPS + tap];
            wq[i - np] = v;
        }
    }
}

// ---------------------------------------------------------------------------------------------------------
// EC, first pass (old terms P): implicit-GEMM style SIMT kernel. One CTA = 8x32 positions x 32 output channels (8 chunks) of one image.
// Thread tile = 4 positions (along w) x 2 chunks x 4 channels = 32 accumulators; K loop over 16-channel
// blocks staged in shared memory (x tile with halo + masked weight tile), 25 taps unrolled.
// ---------------------------------------------------------------------------------------------------------

// one input channel of the EC thread tile (4 positions along w x 2 chunks x 4 channels): taps with kh + kw < NS, fully unrolled
// with compile-time tap tests; x row = two float4 (8 consecutive columns), weights broadcast from shared memory
template <int NS>
__device__ __forceinline__ void ec_taps_fma(const float* xr, const float4* wA, const float4* wB, float4 (&u)[2][4]) {
#pragma unroll
    for (int kh = 0; kh < 5; kh++) {
        if (kh >= NS) continue;
        const float4 x0 = *reinterpret_cast<const float4*>(xr + kh * XW);
        const float4 x1 = *reinterpret_cast<const float4*>(xr + kh * XW + 4);
        const float xv[8] = {x0.x, x0.y, x0.z, x0.w, x1.x, x1.y, x1.z, x1.w};
#pragma unroll
        for (int kw = 0; kw < 5; kw++) {
            if (kh + kw >= NS) continue;
            const float4 a4 = wA[kh * 5 + kw], b4 = wB[kh * 5 + kw];
#pragma unroll
            for (int p = 0; p < 4; p++) {
                fma4(u[0][p], xv[p + kw], a4);
                fma4(u[1][p], xv[p + kw], b4);
            }
        }
    }
}

__global__ void __launch_bounds__(EC_THREADS, 2) cconv_ec_kernel(const ConvArgs a, int pair) {
    extern __shared__ float4 smem_f4[];
    float* xs = reinterpret_cast<float*>(smem_f4);       // [2][EC_SB][XH][XW]
    float4* ws4 = smem_f4 + (2 * EC_SB * XH * XW) / 4;   // [2][EC_CHUNKS][EC_SB][TAPS] float4

    const int tid = threadIdx.x;
    const int tx = tid & 7, ty = (tid >> 3) & 7, tz = tid >> 6;
    const int tiles_w = (a.W + TW - 1) / TW;
    const int w0 = (blockIdx.x % tiles_w) * TW, h0 = (blockIdx.x / tiles_w) * TH;
    // The K extent of a y tile grows with its output groups (old terms: g_in <= g_out + 2), so a CTA takes the PAIR (heaviest
    // remaining, lightest remaining) = y tiles (ny - 1 - b, b): every CTA of the launch then has nearly the same work and one wave
    // of CTAs finishes together instead of leaving a 20% tail of idle SMs behind the heavy tiles.
    const int ny = (a.nchunk + EC_CHUNKS - 1) / EC_CHUNKS;
    // (pair == 0: small grids that do not fill the machine anyway keep one y tile per CTA, heaviest first.)
  for (int pass = 0; pass < 1 + pair; pass++) {
    const int ytile = pass == 0 ? ny - 1 - (int)blockIdx.y : (int)blockIdx.y;
    if (pass == 1 && ytile >= ny - 1 - (int)blockIdx.y) break;  // middle tile of an odd count: done in pass 0
    if (pass == 1) __syncthreads();                             // everyone is done with the staging buffers of pass 0
    const int chunk0 = ytile * EC_CHUNKS;
    const int n = blockIdx.z, set = n / a.per;
    const int Cin = a.Cin, H = a.H, W = a.W;

    const int last_chunk = min(chunk0 + EC_CHUNKS - 1, a.nchunk - 1);
    const int lim_tile = min(Cin, (last_chunk / a.cpg4 + 3) * a.cin_g);  // old terms: g_in <= g_out + 2
    const int nj = (lim_tile + CB - 1) / CB;
    const int cA = chunk0 + 2 * tz;
    const int my_lim = min(Cin, (min(cA + 1, a.nchunk - 1) / a.cpg4 + 3) * a.cin_g);

    float P[2][4][4];
#pragma unroll
    for (int c = 0; c < 2; c++)
#pragma unroll
        for (int p = 0; p < 4; p++)
#pragma unroll
            for (int q = 0; q < 4; q++) P[c][p][q] = 0.f;

    // K loop: 8-channel stages, double buffered with cp.async (the x tile with its halo, zero-filled outside the image, and the
    // masked weight tile of the 8 chunks land while the previous stage is being consumed); two stages = one canonical 16-channel
    // block, whose partial sum u is added to P when it is complete.
    const float4* wp4 = reinterpret_cast<const float4*>(a.wp);
    const int nstage = (lim_tile + EC_SB - 1) / EC_SB;
    (void)nj;
    const unsigned xs_s = (unsigned)__cvta_generic_to_shared(xs), ws_s = (unsigned)__cvta_generic_to_shared(ws4);
    auto issue = [&](int st) {
        const int buf = st & 1, cb8 = min(EC_SB, Cin - st * EC_SB);
        const unsigned xd = xs_s + (unsigned)buf * (EC_SB * XH * XW * 4), wd = ws_s + (unsigned)buf * (EC_CHUNKS * EC_SB * TAPS * 16);
        for (int e = tid; e < cb8 * XH * XW; e += EC_THREADS) {
            const int ci = e / (XH * XW), r = (e % (XH * XW)) / XW, c = e % XW;
            const int h = h0 + r - 2, w = w0 + c - 2;
            const bool ok = h >= 0 && h < H && w >= 0 && w < W;
            cp_async4(xd + 4u * e, ok ? a.x + (((size_t)n * Cin + st * EC_SB + ci) * H + h) * W + w : a.x, ok);
        }
        for (int e = tid; e < EC_CHUNKS * cb8 * TAPS; e += EC_THREADS) {
            const int ch = e / (cb8 * TAPS), r = e % (cb8 * TAPS);
            const int chunk = chunk0 + ch;
            const bool ok = chunk < a.nchunk;
            cp_async16z(wd + 16u * (ch * EC_SB * TAPS + r), ok ? wp4 + (((size_t)set * a.nchunk + chunk) * Cin + st * EC_SB) * TAPS + r : wp4, ok);
        }
        asm volatile("cp.async.commit_group;\n" ::);
    };
    float4 u[2][4];
    if (nstage > 0) issue(0);
    for (int st = 0; st < nstage; st++) {
        if (st + 1 < nstage) {
            issue(st + 1);
            asm volatile("cp.async.wait_group 1;\n" ::: "memory");
        } else {
            asm volatile("cp.async.wait_group 0;\n" ::: "memory");
        }
        __syncthreads();
        const int j = st >> 1;             // canonical 16-channel block
        const bool mine = j * CB < my_lim;  // warp-uniform: tz is constant inside a warp
        if ((st & 1) == 0) {
#pragma unroll
            for (int c = 0; c < 2; c++)
#pragma unroll
                for (int p = 0; p < 4; p++) u[c][p] = make_float4(0.f, 0.f, 0.f, 0.f);
        }
        if (mine) {
            // old taps of input group g for output group g_out: kh + kw <= g_out + 2 - g; beyond that both chunks of this thread
            // carry zero weights (warp-uniform skip; a single-group net keeps 6 of its 25 taps)
            const int buf = st & 1, cb8 = min(EC_SB, Cin - st * EC_SB);
            const float* xb = xs + buf * (EC_SB * XH * XW);
            const float4* wb = ws4 + buf * (EC_CHUNKS * EC_SB * TAPS);
            const int gmax_out = min(cA + 1, a.nchunk - 1) / a.cpg4;
#pragma unroll 1
            for (int ci = 0; ci < cb8; ci++) {
                const float4* wA = wb + ((2 * tz) * EC_SB + ci) * TAPS;
                const float4* wB = wb + ((2 * tz + 1) * EC_SB + ci) * TAPS;
                const float* xr = xb + (ci * XH + ty) * XW + 4 * tx;
                const int ns = gmax_out + 3 - (st * EC_SB + ci) / a.cin_g;  // taps with kh + kw < ns (warp-uniform)
                if (ns >= 9) { ec_taps_fma<9>(xr, wA, wB, u); continue; }  // the common case: straight-line, no tap tests
                switch (ns) {
                    case 8: ec_taps_fma<8>(xr, wA, wB, u); break;
                    case 7: ec_taps_fma<7>(xr, wA, wB, u); break;
                    case 6: ec_taps_fma<6>(xr, wA, wB, u); break;
                    case 5: ec_taps_fma<5>(xr, wA, wB, u); break;
                    case 4: ec_taps_fma<4>(xr, wA, wB, u); break;
                    case 3: ec_taps_fma<3>(xr, wA, wB, u); break;
                    case 2: ec_taps_fma<2>(xr, wA, wB, u); break;
                    case 1: ec_taps_fma<1>(xr, wA, wB, u); break;
                    default: break;
                }
            }
            if ((st & 1) == 1 || st + 1 == nstage) {  // the canonical block is complete
#pragma unroll
                for (int c = 0; c < 2; c++)
#pragma unroll
                    for (int p = 0; p < 4; p++) {
                        P[c][p][0] = P[c][p][0] + u[c][p].x;
                        P[c][p][1] = P[c][p][1] + u[c][p].y;
                        P[c][p][2] = P[c][p][2] + u[c][p].z;
                        P[c][p][3] = P[c][p][3] + u[c][p].w;
                    }
            }
        }
        __syncthreads();  // everyone is done with this buffer before the stage after next lands in it
    }

    // P of every output goes to `out`; cconv_ec_rq_kernel adds the R / Q terms and the epilogue in place
    const int h = h0 + ty;
#pragma unroll
    for (int cc = 0; cc < 2; cc++) {
        const int chunk = cA + cc;
        if (chunk >= a.nchunk || h >= H) continue;
        const int g_out = chunk / a.cpg4;
#pragma unroll
        for (int q = 0; q < 4; q++) {
            const int oc = (chunk % a.cpg4) * 4 + q;
            if (oc >= a.cout_g) continue;
            const size_t row = (((size_t)n * a.Cout + g_out * a.cout_g + oc) * H + h) * W;
#pragma unroll
            for (int p = 0; p < 4; p++) {
                const int w = w0 + 4 * tx + p;
                if (w < W) a.out[row + w] = P[cc][p][q];
            }
        }
    }
  }  // pass
}

// EC, second pass: adds the previous-wavefront (R) and same-wavefront (Q) terms -- every tap reads the cin_g channels
// of ONE input group -- to the P sums that cconv_ec_kernel left in `out`, then bias / PReLU / residual, in place.
// The chunk's R and Q weights are staged once per CTA in shared memory and read as broadcasts; the activation loads are
// coalesced along w.  Two shapes:
//   cconv_ec_rq_kernel<CG>  (cin_g <= 16, one canonical block): one thread = one position x one 4-channel output chunk,
//                           CTA = 256 consecutive positions of one (image, chunk); CG = cin_g when it is 4 (unrolled), else 0
//   cconv_ec_rqb_kernel     (cin_g > 16): CTA = 32 positions of one (image, chunk); warp (cls, jq) computes the partial
//                           of canonical block jq, warp 0 combines them in the canonical order.
constexpr int RQ_THREADS = 256;

__device__ __forceinline__ void rq_epilogue(const ConvArgs& a, int n, int set, int chunk, int g_out, int pos, const float* R,
                                            const float* Q) {
    const int HW = a.H * a.W;
#pragma unroll
    for (int q = 0; q < 4; q++) {
        const int oc = (chunk % a.cpg4) * 4 + q;
        if (oc >= a.cout_g) continue;
        const int o = g_out * a.cout_g + oc;
        const size_t p = ((size_t)n * a.Cout + o) * HW + pos;
        float v = ((a.out[p] + R[q]) + Q[q]) + __ldg(a.bias + set * a.Cout + o);
        if (a.slope) { const float sl = __ldg(a.slope + set * a.Cout + o); v = v > 0.f ? v : v * sl; }
        if (a.resid) v = v + a.resid[p];
        a.out[p] = v;
    }
}

template <int CG>
__global__ void __launch_bounds__(RQ_THREADS, 2) cconv_ec_rq_kernel(const ConvArgs a) {
    extern __shared__ float4 rq_wsm[];  // [2 classes][TAPS][cin_g]
    const int chunk = blockIdx.y, n = blockIdx.z, set = n / a.per;
    const int g_out = chunk / a.cpg4;
    const int cin_g = CG ? CG : a.cin_g, H = a.H, W = a.W, HW = a.H * a.W;
    const int row_f4 = TAPS * cin_g;
    const size_t wq_cls = (size_t)(a.N / a.per) * a.nchunk * row_f4;  // float4 per class
    const float4* wq4 = reinterpret_cast<const float4*>(a.wq) + ((size_t)set * a.nchunk + chunk) * row_f4;
    const int ncls = a.has_q ? 2 : 1;
    for (int e = threadIdx.x; e < ncls * row_f4; e += RQ_THREADS) rq_wsm[e] = __ldg(wq4 + (e / row_f4) * wq_cls + e % row_f4);
    __syncthreads();
    const int pos = blockIdx.x * RQ_THREADS + threadIdx.x;
    if (pos >= HW) return;
    const int h = pos / W, w = pos % W;
    const float* xn = a.x + (size_t)n * a.Cin * HW;
    float RQ[2][4];
#pragma unroll
    for (int cls = 0; cls < 2; cls++) {
        float4 u = make_float4(0.f, 0.f, 0.f, 0.f);
        if (cls < ncls) {
            const float4* ws = rq_wsm + cls * row_f4;
            for (int c0 = 0; c0 < cin_g; c0 += 4) {  // canonical 4-channel chunks of the single block
                const int c1 = min(c0 + 4, cin_g);
#pragma unroll
                for (int kh = 0; kh < 5; kh++) {
                    const int ph = h + kh - 2;
                    if (ph < 0 || ph >= H) continue;
#pragma unroll
                    for (int kw = 0; kw < 5; kw++) {
                        const int gq = g_out + 3 + cls - kh - kw;
                        const int pw = w + kw - 2;
                        if (gq < 0 || gq >= a.G || pw < 0 || pw >= W) continue;
                        const float* xp = xn + ((size_t)(gq * cin_g) * H + ph) * W + pw;
                        const float4* wt = ws + (kh * 5 + kw) * cin_g;
                        if (CG == 4) {
                            float xx[4];
#pragma unroll
                            for (int c = 0; c < 4; c++) xx[c] = __ldg(xp + (size_t)c * HW);
#pragma unroll
                            for (int c = 0; c < 4; c++) {
                                const float4 w4 = wt[c];
                                fma4(u, xx[c], w4);
                            }
                        } else {
                            for (int c = c0; c < c1; c++) {
                                const float xx = __ldg(xp + (size_t)c * HW);
                                const float4 w4 = wt[c];
                                fma4(u, xx, w4);
                            }
                        }
                    }
                }
            }
        }
        RQ[cls][0] = 0.f + u.x; RQ[cls][1] = 0.f + u.y; RQ[cls][2] = 0.f + u.z; RQ[cls][3] = 0.f + u.w;
    }
    rq_epilogue(a, n, set, chunk, g_out, pos, RQ[0], RQ[1]);
}

// R / Q pass of the many-group nets (cin_g == 4, one 4-channel output chunk per group: every hidden and the last layer of the code
// stream).  The generic kernel above fetches its 200 activations per output straight from L2 (40 channel planes per output group,
// no reuse between the 25 taps, one broadcast weight load per FMA4: ~5 TB/s of L1/L2 traffic, 180 us per layer at 512x1024).
// Here a CTA owns an 8x32 spatial tile and FOUR adjacent output groups: the 13 input groups g0-5 .. g0+7 their taps select (52
// channels) are staged once in shared memory with their halo, as aligned 16-byte cp.async chunks (rows start at column w0-4;
// zero-filled outside the image / outside [0, G): the skipped terms of the canonical order become exact +0 products).  A warp owns a
// PAIR of output groups on a 4-row x 16-column piece of the tile, a lane 2 positions (columns 8 apart): the previous-wavefront tap
// of group g+1 and the same-wavefront tap of group g read the same activation, so 3 activation loads feed the 4 (group, class)
// accumulators of a position and each broadcast weight vector feeds 2 positions.  112 KB per CTA: two CTAs per SM, one loads while
// the other computes.  Per-output arithmetic and order are those of cconv_ec_rq_kernel<4> (canonical order, header of this file).
constexpr int RQ4_G = 4;                          // output groups per CTA
constexpr int RQ4_IN = RQ4_G + 9;                 // input groups staged: g0-5 .. g0+7
constexpr int RQ4_XW = 40;                        // staged row: columns w0-4 .. w0+35 (ten float4); lane (ty, tx) -> bank 8*ty + tx
constexpr int RQ4_PLANE = XH * RQ4_XW;
constexpr int RQ4_W_F4 = RQ4_G * 2 * TAPS * 4;    // [group][class][tap][c] float4
constexpr int RQ4_SMEM_BYTES = RQ4_W_F4 * 16 + RQ4_IN * 4 * RQ4_PLANE * 4;

__global__ void __launch_bounds__(256, 2) cconv_ec_rq_tile_kernel(const ConvArgs a) {
    extern __shared__ float4 rqt_smem[];
    float4* wsm = rqt_smem;
    float* xs = reinterpret_cast<float*>(rqt_smem + RQ4_W_F4);  // [RQ4_IN * 4][XH][RQ4_XW]
    const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int tiles_w = (a.W + TW - 1) / TW;
    const int w0 = (blockIdx.x % tiles_w) * TW, h0 = (blockIdx.x / tiles_w) * TH;
    const int g0 = RQ4_G * blockIdx.y, n = blockIdx.z, set = n / a.per;
    const int H = a.H, W = a.W, HW = a.H * a.W, G = a.G;
    const int ncls = a.has_q ? 2 : 1;
    // weights: wq [cls][set][chunk][tap][c] float4, chunk == group here
    const size_t wq_cls = (size_t)(a.N / a.per) * a.nchunk * (TAPS * 4);
    const float4* wq4 = reinterpret_cast<const float4*>(a.wq);
    for (int e = tid; e < RQ4_W_F4; e += 256) {
        const int grp = e / (2 * TAPS * 4), cls = (e / (TAPS * 4)) % 2, r = e % (TAPS * 4);
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (g0 + grp < G && cls < ncls) v = __ldg(wq4 + cls * wq_cls + ((size_t)set * a.nchunk + g0 + grp) * (TAPS * 4) + r);
        wsm[e] = v;
    }
    // activations: warp w stages channels w, w+8, ...; 12 rows x 10 aligned float4 per channel (W % 4 == 0 is checked by the launcher)
    const unsigned xs_s = (unsigned)__cvta_generic_to_shared(xs);
    const float* xn = a.x + (size_t)n * a.Cin * HW;
    for (int ch = warp; ch < RQ4_IN * 4; ch += 8) {
        const int grp = g0 - 5 + (ch >> 2);
        const bool gok = grp >= 0 && grp < G;
        const float* plane = xn + (size_t)(gok ? grp * 4 + (ch & 3) : 0) * HW;
        for (int id = lane; id < XH * (RQ4_XW / 4); id += 32) {
            const int r = id / (RQ4_XW / 4), c4 = id % (RQ4_XW / 4);
            const int h = h0 + r - 2, w = w0 - 4 + 4 * c4;
            const bool ok = gok && h >= 0 && h < H && w >= 0 && w + 3 < W;
            cp_async16z(xs_s + 4u * (ch * RQ4_PLANE + r * RQ4_XW + 4 * c4), ok ? plane + (size_t)h * W + w : xn, ok);
        }
    }
    cp_async_wait_all();
    __syncthreads();
    // warp -> (pair of output groups, 4-row half, 16-column half); lane -> row ty, columns tx and tx + 8 of that piece
    const int pi = warp >> 2, row = ((warp >> 1) & 1) * 4 + (lane >> 3), col = (warp & 1) * 16 + (lane & 7);
    if (g0 + 2 * pi >= G) return;  // warp-uniform
    float4 acc[2][4];  // [position j][pr * 2 + cls]
#pragma unroll
    for (int j = 0; j < 2; j++)
#pragma unroll
        for (int k = 0; k < 4; k++) acc[j][k] = make_float4(0.f, 0.f, 0.f, 0.f);
    const float4* wpair = wsm + (2 * pi) * 2 * TAPS * 4;
#pragma unroll 1
    for (int kh = 0; kh < 5; kh++) {
#pragma unroll
        for (int kw = 0; kw < 5; kw++) {
            // (pr, cls) reads input group g0 + 2pi + pr + cls + 3 - kh - kw = staged group 2pi + 8 + (pr + cls) - kh - kw;
            // image column w0 + col + kw - 2 = staged column col + kw + 2
            const float* xt = xs + ((2 * pi + 8 - kh - kw) * 4) * RQ4_PLANE + (row + kh) * RQ4_XW + col + kw + 2;
#pragma unroll
            for (int c = 0; c < 4; c++) {
                float xv[3][2];
#pragma unroll
                for (int k = 0; k < 3; k++)
#pragma unroll
                    for (int j = 0; j < 2; j++) xv[k][j] = xt[(k * 4 + c) * RQ4_PLANE + 8 * j];
#pragma unroll
                for (int pc = 0; pc < 4; pc++) {  // pc = pr * 2 + cls
                    const float4 w4 = wpair[pc * (TAPS * 4) + (kh * 5 + kw) * 4 + c];
#pragma unroll
                    for (int j = 0; j < 2; j++) fma4(acc[j][pc], xv[(pc >> 1) + (pc & 1)][j], w4);
                }
            }
        }
    }
    const int h = h0 + row;
    if (h >= H) return;
#pragma unroll
    for (int j = 0; j < 2; j++) {
        const int w = w0 + col + 8 * j;
        if (w >= W) continue;
#pragma unroll
        for (int pr = 0; pr < 2; pr++) {
            const int g_out = g0 + 2 * pi + pr;
            if (g_out >= G) continue;
            const float4 r4 = acc[j][pr * 2], q4 = acc[j][pr * 2 + 1];
            const float R[4] = {0.f + r4.x, 0.f + r4.y, 0.f + r4.z, 0.f + r4.w};
            const float Q[4] = {0.f + q4.x, 0.f + q4.y, 0.f + q4.z, 0.f + q4.w};
            rq_epilogue(a, n, set, g_out, g_out, h * W + w, R, Q);
        }
    }
}

__global__ void __launch_bounds__(640, 2) cconv_ec_rqb_kernel(const ConvArgs a, int nqb, int tap_cap) {
    extern __shared__ float4 rq_wsm[];  // [2 classes][tap_cap][cin_g] weights of the taps that select a valid group, then partials
    __shared__ int s_tap[2][TAPS], s_ntap[2];
    const int chunk = blockIdx.y, n = blockIdx.z, set = n / a.per;
    const int g_out = chunk / a.cpg4;
    const int cin_g = a.cin_g, H = a.H, W = a.W, HW = a.H * a.W;
    const int row_f4 = TAPS * cin_g;
    const size_t wq_cls = (size_t)(a.N / a.per) * a.nchunk * row_f4;
    const float4* wq4 = reinterpret_cast<const float4*>(a.wq) + ((size_t)set * a.nchunk + chunk) * row_f4;
    const int ncls = a.has_q ? 2 : 1;
    const int lane = threadIdx.x, wid = threadIdx.y, tid = wid * 32 + lane, nthr = blockDim.x * blockDim.y;
    float4* part = rq_wsm + 2 * tap_cap * cin_g;
    if (tid < 2) {  // taps of class tid whose selected input group exists, in canonical (kh, kw) order
        int m = 0;
        for (int t = 0; t < TAPS; t++) {
            const int gq = g_out + 3 + tid - t / 5 - t % 5;
            if (gq >= 0 && gq < a.G && tid < ncls) s_tap[tid][m++] = t;
        }
        s_ntap[tid] = m;
    }
    __syncthreads();
    for (int c = 0; c < ncls; c++)
        for (int e = tid; e < s_ntap[c] * cin_g; e += nthr)
            rq_wsm[c * tap_cap * cin_g + e] = __ldg(wq4 + c * wq_cls + (size_t)s_tap[c][e / cin_g] * cin_g + e % cin_g);
    __syncthreads();
    const int pos = blockIdx.x * 32 + lane;
    const bool valid = pos < HW;
    const int h = pos / W, w = pos % W;
    const int cls = wid / nqb, jq = wid % nqb;
    float4 u = make_float4(0.f, 0.f, 0.f, 0.f);
    if (valid && cls < ncls) {
        const float* xn = a.x + (size_t)n * a.Cin * HW;
        const float4* ws = rq_wsm + cls * tap_cap * cin_g;
        const int cend = min((jq + 1) * CB, cin_g), nt = s_ntap[cls];
        for (int c0 = jq * CB; c0 < cend; c0 += 4) {
            const int c1 = min(c0 + 4, cend);
            for (int ti = 0; ti < nt; ti++) {
                const int t = s_tap[cls][ti], kh = t / 5, kw = t % 5;
                const int ph = h + kh - 2, pw = w + kw - 2;
                if (ph < 0 || ph >= H || pw < 0 || pw >= W) continue;
                const int gq = g_out + 3 + cls - kh - kw;
                const float* xp = xn + ((size_t)(gq * cin_g) * H + ph) * W + pw;
                const float4* wt = ws + ti * cin_g;
                if (c1 - c0 == 4) {
                    float xx[4];
#pragma unroll
                    for (int c = 0; c < 4; c++) xx[c] = __ldg(xp + (size_t)(c0 + c) * HW);
#pragma unroll
                    for (int c = 0; c < 4; c++) {
                        const float4 w4 = wt[c0 + c];
                        fma4(u, xx[c], w4);
                    }
                } else {
                    for (int c = c0; c < c1; c++) {
                        const float xx = __ldg(xp + (size_t)c * HW);
                        const float4 w4 = wt[c];
                        fma4(u, xx, w4);
                    }
                }
            }
        }
    }
    part[wid * 32 + lane] = u;
    __syncthreads();
    if (wid != 0 || !valid) return;
    float RQ[2][4];
#pragma unroll
    for (int c = 0; c < 2; c++) {
        RQ[c][0] = RQ[c][1] = RQ[c][2] = RQ[c][3] = 0.f;
        for (int j = 0; j < nqb; j++) {
            const float4 v = part[(c * nqb + j) * 32 + lane];
            RQ[c][0] = RQ[c][0] + v.x; RQ[c][1] = RQ[c][1] + v.y; RQ[c][2] = RQ[c][2] + v.z; RQ[c][3] = RQ[c][3] + v.w;
        }
    }
    rq_epilogue(a, n, set, chunk, g_out, pos, RQ[0], RQ[1]);
}

// ---------------------------------------------------------------------------------------------------------
// DC: one wavefront step.  CTA = 32 consecutive positions of ONE anti-diagonal d (so the whole CTA shares the
// output group tc = psum - d and its weights) x (nblk past segments + 1 present segment) warps, one 4-channel
// output chunk, one image.  Positions are derived analytically (h = hmin(d) + i, w = d - h), no index plan needed.
//
// The 5x5 windows of 32 diagonal neighbours cover a band of 36 rows x 9 columns per input channel
// (row rr = i + kh, column cc = kh + kw in band coordinates).  Each past-segment warp stages the band of 4 input
// channels at a time in its private shared-memory slice with row-contiguous (coalesced) global reads, then every
// lane walks its window from shared memory (stride-9 rows: bank-conflict free) against warp-uniform float4 weight
// loads.  Segment partials meet in shared memory and are combined in the canonical order by warp 0.
// ---------------------------------------------------------------------------------------------------------
// canonical combine of the segment partials + bias / PReLU / residual; p = element offset of channel 0 of this
// position in the output frame, cstride = channel stride of that frame
__device__ __forceinline__ void dc_combine_store(const ConvArgs& a, const float4* part, int nblk, int nqb, int lane, int tc,
                                                 int set, int ochunk, size_t p0, size_t cstride) {
    float P[4] = {0.f, 0.f, 0.f, 0.f}, R[4] = {0.f, 0.f, 0.f, 0.f}, Q[4] = {0.f, 0.f, 0.f, 0.f};
    for (int j = 0; j < nblk; j++) {
        const float4 v = part[j * 32 + lane];
        P[0] = P[0] + v.x; P[1] = P[1] + v.y; P[2] = P[2] + v.z; P[3] = P[3] + v.w;
    }
    for (int j = nblk; j < nblk + nqb; j++) {
        const float4 v = part[j * 32 + lane];
        R[0] = R[0] + v.x; R[1] = R[1] + v.y; R[2] = R[2] + v.z; R[3] = R[3] + v.w;
    }
    for (int j = nblk + nqb; j < nblk + 2 * nqb; j++) {  // zero partials when !has_q
        const float4 v = part[j * 32 + lane];
        Q[0] = Q[0] + v.x; Q[1] = Q[1] + v.y; Q[2] = Q[2] + v.z; Q[3] = Q[3] + v.w;
    }
#pragma unroll
    for (int q = 0; q < 4; q++) {
        const int oc = ochunk * 4 + q;
        if (oc >= a.cout_g) continue;
        const int o = tc * a.cout_g + oc;
        float v = ((P[q] + R[q]) + Q[q]) + __ldg(a.bias + set * a.Cout + o);
        if (a.slope) { const float sl = __ldg(a.slope + set * a.Cout + o); v = v > 0.f ? v : v * sl; }
        const size_t p = p0 + (size_t)o * cstride;
        if (a.resid) v = v + a.resid[p];
        a.out[p] = v;
    }
}

__global__ void __launch_bounds__(1024) cconv_dc_kernel(const ConvArgs a, int psum, int nblk, int nqb, int parts,
                                                      const StepDesc* __restrict__ steps, const int* __restrict__ ctr) {
    extern __shared__ float4 dc_smem4[];
    const int nseg = nblk + 2 * nqb;                                       // old segments, then R, then Q segments
    float4* part = dc_smem4;                                               // [nseg][32]
    int* boff = reinterpret_cast<int*>(dc_smem4 + nseg * 32);              // [DC_BAND] band cell -> row*W+col or -1
    float* stage_all = reinterpret_cast<float*>(boff + DC_BAND);           // [nseg][DC_WARP_FLOATS]
    const int lane = threadIdx.x, seg = threadIdx.y;
    if (steps) psum = steps[*ctr].psum;  // graph replay: the step is read on the device
    const int H = a.H, W = a.W, HW = a.H * a.W, Cin = a.Cin;
    const int la = max(0, psum - a.G + 1), lb = min(psum, H + W - 2);
    const int d = la + blockIdx.x / parts;
    if (d > lb) return;
    const int hmin = max(0, d - W + 1), hmax = min(H - 1, d);
    const int hbase = hmin + (blockIdx.x % parts) * 32;
    if (hbase > hmax) return;
    for (int r = seg * 32 + lane; r < DC_BAND; r += 32 * nseg) {
        const int rr = r / 9, cc = r % 9;
        const int row = hbase + rr - 2, col = d - hbase - rr - 2 + cc;
        boff[r] = (row >= 0 && row < H && col >= 0 && col < W) ? row * W + col : -1;
    }
    __syncthreads();
    const int th = hbase + lane, tw = d - th;
    const bool valid = th <= hmax;
    const int tc = psum - d;  // output group of this diagonal in this step
    const int n = blockIdx.z, set = n / a.per;
    const int chunk = tc * a.cpg4 + blockIdx.y;
    float* band = stage_all + seg * DC_WARP_FLOATS;
    float4* wsm = reinterpret_cast<float4*>(band + DC_STAGE * DC_BAND);
    const unsigned band_s = (unsigned)__cvta_generic_to_shared(band);
    const unsigned wsm_s = (unsigned)__cvta_generic_to_shared(wsm);
    float4 u = make_float4(0.f, 0.f, 0.f, 0.f);
    if (seg < nblk) {
        const int lim = min(Cin, (tc + 3) * a.cin_g);  // old terms: g_in <= tc + 2
        if (seg * CB < lim) {
            const int cb = min(CB, Cin - seg * CB);
            const float4* wp4 = reinterpret_cast<const float4*>(a.wp) + (((size_t)set * a.nchunk + chunk) * Cin + seg * CB) * TAPS;
            const float* xb = a.x + ((size_t)n * Cin + seg * CB) * HW;
            for (int c0 = 0; c0 < cb; c0 += DC_STAGE) {
                if (c0 + seg * CB >= lim) break;  // only masked-out channels remain (warp-uniform)
                const int nc = min(DC_STAGE, cb - c0);
                __syncwarp();
                for (int ch = 0; ch < nc; ch++) {
                    const float* xc = xb + (size_t)(c0 + ch) * HW;
#pragma unroll 4
                    for (int r = lane; r < DC_BAND; r += 32) {
                        const int off = boff[r];
                        cp_async4(band_s + 4u * (ch * DC_BAND + r), off >= 0 ? xc + off : xc, off >= 0);
                    }
                }
                for (int e = lane; e < nc * TAPS; e += 32) cp_async16(wsm_s + 16u * e, wp4 + c0 * TAPS + e);
                cp_async_wait_all();
                __syncwarp();
                dc_stage_fma<9, 1, DC_BAND>(band, wsm, nc, lane, seg * CB + c0, a.cin_g, tc, u);
            }
        }
    } else if (seg < nblk + nqb || a.has_q) {
        // R (cls 0) / Q (cls 1) terms, 16-channel block jq of the group: tap (kh,kw) reads group gq = tc + 3 + cls - (kh+kw)
        // at band column cc = kh+kw, so the stage holds, for every column cc, the 4-channel chunk [c0, c0+4) of that group
        const int cls = seg >= nblk + nqb;
        const int jq = seg - nblk - cls * nqb;
        const int gsel0 = tc + 3 + cls;
        const int cend = min((jq + 1) * CB, a.cin_g);
        const float4* wq4 = reinterpret_cast<const float4*>(a.wq) +
                            ((size_t)(cls * (a.N / a.per) + set) * a.nchunk + chunk) * TAPS * a.cin_g;
        const float* xn = a.x + (size_t)n * Cin * HW;
        for (int c0 = jq * CB; c0 < cend; c0 += DC_STAGE) {
            const int nc = min(DC_STAGE, cend - c0);
            __syncwarp();
            for (int ch = 0; ch < nc; ch++) {
#pragma unroll 4
                for (int r = lane; r < DC_BAND; r += 32) {
                    const int off = boff[r];
                    const int gq = gsel0 - r % 9;
                    const bool ok = off >= 0 && gq >= 0 && gq < a.G;
                    cp_async4(band_s + 4u * (ch * DC_BAND + r), ok ? xn + (size_t)(gq * a.cin_g + c0 + ch) * HW + off : xn, ok);
                }
            }
            // weights of this chunk: wq layout [tap][cin_g] float4 -> stage layout [ch][tap]
            for (int e = lane; e < nc * TAPS; e += 32) cp_async16(wsm_s + 16u * e, wq4 + (e % TAPS) * a.cin_g + c0 + e / TAPS);
            cp_async_wait_all();
            __syncwarp();
            dc_stage_q<9, 1, DC_BAND>(band, wsm, nc, lane, gsel0, a.G, u);
        }
    }
    part[seg * 32 + lane] = u;
    __syncthreads();
    if (seg == 0 && valid)
        dc_combine_store(a, part, nblk, nqb, lane, tc, set, blockIdx.y, ((size_t)n * a.Cout * H + th) * W + tw, (size_t)HW);
}

int fill_conv_args(ConvArgs& a, const float* x, const float* wp, const float* wq, const float* bias,
                   const float* slope, const float* resid, float* out, int N, int Cin, int H, int W, int Cout, int G,
                   int constrain, int nsets) {
    if (N <= 0 || Cin <= 0 || Cout <= 0 || G <= 0 || H <= 0 || W <= 0 || nsets <= 0) return 1;
    if (Cin % G || Cout % G || N % nsets) return 1;
    if (constrain != 5 && constrain != 6) return 1;
    a.x = x; a.wp = wp; a.wq = wq; a.bias = bias; a.slope = slope; a.resid = resid; a.out = out;
    a.N = N; a.Cin = Cin; a.H = H; a.W = W; a.Cout = Cout; a.G = G;
    a.cin_g = Cin / G; a.cout_g = Cout / G; a.cpg4 = (a.cout_g + 3) / 4; a.nchunk = G * a.cpg4;
    a.per = N / nsets; a.has_q = constrain == 6;
    return 0;
}

cudaError_t launch_cconv_ec(const ConvArgs& a, cudaStream_t s, bool allow_mma) {
    static SmemAttr ec_attr;  // per device (ADVICE r1: a process-wide flag left cuda:1 at the 48 KB default)
    {
        cudaError_t e = ec_attr.ensure(cconv_ec_kernel, EC_SMEM_BYTES);
        if (e != cudaSuccess) return e;
    }
    const int ny = (a.nchunk + EC_CHUNKS - 1) / EC_CHUNKS, nxy = ((a.W + TW - 1) / TW) * ((a.H + TH - 1) / TH);
    cudaError_t e;
    // opt-in tensor-core form of the old-term pass (conv_mma.cu), per-op CconvEc only: it is NOT bit-identical to the decoder,
    // so the codec (run_ec_net, allow_mma = false) never uses it and its streams do not depend on LIC360_EC_MMA
    if (allow_mma && cconv_ec_mma_enabled()) {
        e = launch_cconv_ec_mma(a, s);
    } else {
        const int pair = (long long)nxy * ny * a.N > 2 * 148 ? 1 : 0;  // more than one wave of CTAs (2 per SM): balance them in pairs
        dim3 grid(nxy, pair ? (ny + 1) / 2 : ny, a.N);
        cconv_ec_kernel<<<grid, EC_THREADS, EC_SMEM_BYTES, s>>>(a, pair);
        g_launches++;
        e = cudaGetLastError();
    }
    if (e != cudaSuccess) return e;
    const int nqb = (a.cin_g + CB - 1) / CB;
    if (a.cin_g == 4 && a.cpg4 == 1 && a.G >= 8 && a.W % 4 == 0 && (reinterpret_cast<uintptr_t>(a.x) & 15) == 0) {
        static SmemAttr rqt_attr;
        e = rqt_attr.ensure(cconv_ec_rq_tile_kernel, RQ4_SMEM_BYTES);
        if (e != cudaSuccess) return e;
        dim3 grid2(nxy, (a.G + RQ4_G - 1) / RQ4_G, a.N);
        cconv_ec_rq_tile_kernel<<<grid2, 256, RQ4_SMEM_BYTES, s>>>(a);
    } else if (nqb == 1) {
        const size_t rq_smem = (size_t)2 * TAPS * a.cin_g * sizeof(float4);  // <= 12.8 KB
        dim3 grid2((a.H * a.W + RQ_THREADS - 1) / RQ_THREADS, a.nchunk, a.N);
        if (a.cin_g == 4) cconv_ec_rq_kernel<4><<<grid2, RQ_THREADS, rq_smem, s>>>(a);
        else cconv_ec_rq_kernel<0><<<grid2, RQ_THREADS, rq_smem, s>>>(a);
    } else {
        if (2 * nqb > 20) return cudaErrorInvalidConfiguration;  // cin_g <= 160
        int tap_cap = 0;  // most taps of one class that select an existing input group, over all output groups
        for (int g = 0; g < a.G; g++)
            for (int cls = 0; cls < 2; cls++) {
                int m = 0;
                for (int t = 0; t < TAPS; t++) { const int gq = g + 3 + cls - t / 5 - t % 5; m += gq >= 0 && gq < a.G; }
                tap_cap = std::max(tap_cap, m);
            }
        const size_t rq_smem = ((size_t)2 * tap_cap * a.cin_g + (size_t)2 * nqb * 32) * sizeof(float4);
        static SmemAttr rq_attr;
        e = rq_attr.ensure(cconv_ec_rqb_kernel, rq_smem);
        if (e != cudaSuccess) return e;
        dim3 grid2((a.H * a.W + 31) / 32, a.nchunk, a.N), block2(32, 2 * nqb);
        cconv_ec_rqb_kernel<<<grid2, block2, rq_smem, s>>>(a, nqb, tap_cap);
    }
    g_launches++;
    return cudaGetLastError();
}

cudaError_t launch_cconv_dc(const ConvArgs& a, const int32_t* idx_dev, int start, int len, int psum, const StepDesc* steps,
                            const int* ctr, int max_len, cudaStream_t s) {
    (void)idx_dev; (void)start; (void)max_len;
    const int nblk = (a.Cin + CB - 1) / CB;
    if (!steps && len <= 0) return cudaSuccess;
    const int parts = (std::min(a.H, a.W) + 31) / 32;          // 32-position chunks per anti-diagonal
    const int ndiag = std::min(a.G, a.H + a.W - 1);            // a slab holds at most G diagonals
    const int nqb = (a.cin_g + CB - 1) / CB;
    const int nseg = nblk + 2 * nqb;
    if (nseg > 32) return cudaErrorInvalidConfiguration;
    const size_t smem = (size_t)nseg * 32 * sizeof(float4) + DC_BAND * sizeof(int) + (size_t)nseg * DC_WARP_FLOATS * sizeof(float);
    static SmemAttr dc_attr;
    {
        cudaError_t e = dc_attr.ensure(cconv_dc_kernel, smem);
        if (e != cudaSuccess) return e;
    }
    dim3 grid(ndiag * parts, a.cpg4, a.N), block(32, nseg);
    cconv_dc_kernel<<<grid, block, smem, s>>>(a, psum, nblk, nqb, parts, steps, ctr);
    g_launches++;
    return cudaGetLastError();
}

}  // namespace lic360

using namespace lic360;

extern "C" size_t lic360_cconv_wp_floats(int nsets, int Cin, int Cout, int G) {
    int cpg4 = (Cout / G + 3) / 4;
    return (size_t)nsets * G * cpg4 * Cin * TAPS * 4;
}
extern "C" size_t lic360_cconv_wq_floats(int nsets, int Cin, int Cout, int G) {
    int cpg4 = (Cout / G + 3) / 4;
    return (size_t)2 * nsets * G * cpg4 * TAPS * (Cin / G) * 4;  // two classes: previous-wavefront and same-wavefront terms
}

extern "C" int lic360_cconv_pack(const float* w_dev, float* wp_dev, float* wq_dev, int nsets, int Cin, int Cout, int G,
                                 int ksize, int constrain, void* stream) {
    LIC360_CHECK_ARG(ksize == 5, "only 5x5 context kernels are supported (every reference call site uses 5)");
    LIC360_CHECK_ARG(constrain == 5 || constrain == 6, "constrain must be 5 (first layer) or 6 (hidden)");
    LIC360_CHECK_ARG(G > 0 && Cin % G == 0 && Cout % G == 0 && nsets > 0, "channels must be multiples of ngroup");
    size_t total = lic360_cconv_wp_floats(nsets, Cin, Cout, G) + lic360_cconv_wq_floats(nsets, Cin, Cout, G);
    cconv_pack_kernel<<<stream_grid(total, 256 * 4), 256, 0, as_stream(stream)>>>(w_dev, wp_dev, wq_dev, nsets, Cin, Cout, G, constrain);
    LAUNCH_CHECK();
    return LIC360_OK;
}

extern "C" int lic360_cconv_ec_forward(const float* x_dev, const float* wp_dev, const float* wq_dev,
                                       const float* bias_dev, const float* slope_dev, const float* resid_dev,
                                       float* out_dev, int N, int Cin, int H, int W, int Cout, int G, int constrain,
                                       int nsets, void* stream) {
    ConvArgs a;
    LIC360_CHECK_ARG(fill_conv_args(a, x_dev, wp_dev, wq_dev, bias_dev, slope_dev, resid_dev, out_dev, N, Cin, H, W, Cout, G,
                               constrain, nsets) == 0, "bad shape / constrain");
    LIC360_CUDA(launch_cconv_ec(a, as_stream(stream), true));
    return LIC360_OK;
}

extern "C" int lic360_cconv_dc_forward(const float* x_dev, const float* wp_dev, const float* wq_dev,
                                       const float* bias_dev, const float* slope_dev, const float* resid_dev,
                                       float* out_dev, int N, int Cin, int H, int W, int Cout, int G, int constrain,
                                       int nsets, const int32_t* idx_dev, const int32_t* plan_host, int psum,
                                       void* stream) {
    ConvArgs a;
    LIC360_CHECK_ARG(fill_conv_args(a, x_dev, wp_dev, wq_dev, bias_dev, slope_dev, resid_dev, out_dev, N, Cin, H, W, Cout, G,
                               constrain, nsets) == 0, "bad shape / constrain");
    const int nblk = (Cin + CB - 1) / CB;
    LIC360_CHECK_ARG(nblk + 2 * ((Cin / G + CB - 1) / CB) <= 32, "Cin too large for the wavefront kernel");
    const int mod = H + W + G - 2;
    int start, len;
    slab_of(plan_host, H, W, G, psum, &start, &len);
    if (!(psum < mod && len > 0)) return LIC360_OK;  // cconv_dc_cuda.cu:121
    if (psum == 0)                                   // cconv_dc_cuda.cu:124-126 (stream-ordered here)
        LIC360_CUDA(cudaMemsetAsync(out_dev, 0, sizeof(float) * (size_t)N * Cout * H * W, as_stream(stream)));
    LIC360_CUDA(launch_cconv_dc(a, idx_dev, start, len, psum, nullptr, nullptr, 0, as_stream(stream)));
    return LIC360_OK;
}
