/* Bit-exact CPU model of the canonical fp32 order of one masked context-conv layer (header of csrc/conv.cu).
 *
 * Every kernel that computes a context-conv output (encoder P and R/Q passes, per-op decoder, fused wavefront decoder)
 * must produce exactly these bits: the arithmetic decoder reads tables built from them.  Per output (n, o, h, w), with
 * g_out = o / cout_g and glim(kh, kw) = g_out + 4 - kh - kw:
 *   P: blocks of 16 input channels, ascending; inside a block a fresh u = 0 and one fmaf chain over (ci, kh, kw) of the
 *      taps with ci / cin_g <= glim - 2; then P = P + u
 *   R (g_in == glim - 1) and Q (g_in == glim, constrain 6 only): 16-channel blocks of the selected group; inside a block
 *      a fresh r = 0 and, per 4-channel chunk, (kh, kw) then c; then R = R + r
 *   v = ((P + R) + Q) + bias;  v = v > 0 ? v : v * slope;  v = v + resid
 * The input is zero padded: fmaf(0, w, u) == u for finite w, and u is never -0, so an out-of-image tap that is multiplied
 * by zero gives the bits of one that is skipped.  A tap the mask forbids is never read (NaN there is harmless).
 *
 * variant selects a deliberately different order, used by the tests to show that the model can tell orders apart:
 *   0 canonical, 1 one flat fmaf chain over every kept tap in (ci, kh, kw) order, 2 ((P + Q) + R) + bias.
 *
 * Loop order across outputs is free; this one vectorises across w (one output row per inner loop).
 * Build: gcc -O3 -mavx2 -mfma -ffp-contract=off -fopenmp (fmaf is then the correctly rounded FMA instruction).
 */
#include <math.h>
#include <stdlib.h>
#include <string.h>

#define CB 16

static void fma_row(float* restrict u, const float* restrict x, float wt, int W) {
    for (int w = 0; w < W; w++) u[w] = fmaf(x[w], wt, u[w]);
}

void canon_cconv(const float* x, const float* wt, const float* bias, const float* slope, const float* resid, float* out,
                 int N, int Cin, int Cout, int G, int H, int W, int constrain, int nsets, int variant) {
    const int cin_g = Cin / G, cout_g = Cout / G, per = N / nsets;
    const int Hp = H + 4, Wp = W + 4;
    float* xp = (float*)calloc((size_t)N * Cin * Hp * Wp, sizeof(float));
    for (size_t p = 0; p < (size_t)N * Cin; p++)
        for (int h = 0; h < H; h++)
            memcpy(xp + (p * Hp + h + 2) * Wp + 2, x + (p * H + h) * W, (size_t)W * sizeof(float));
#pragma omp parallel
    {
        float* buf = (float*)malloc(5 * (size_t)W * sizeof(float));
        float *P = buf, *R = buf + W, *Q = buf + 2 * W, *u = buf + 3 * W, *r = buf + 4 * W;
#pragma omp for collapse(3) schedule(dynamic)
        for (int n = 0; n < N; n++)
            for (int o = 0; o < Cout; o++)
                for (int h = 0; h < H; h++) {
                    const int set = n / per, g_out = o / cout_g;
                    const float* wo = wt + ((size_t)set * Cout + o) * Cin * 25;
                    const float* xn = xp + (size_t)n * Cin * Hp * Wp;
                    memset(P, 0, sizeof(float) * (size_t)W);
                    memset(R, 0, sizeof(float) * (size_t)W);
                    memset(Q, 0, sizeof(float) * (size_t)W);
                    if (variant == 1) {  /* one flat chain over every kept tap */
                        for (int ci = 0; ci < Cin; ci++)
                            for (int kh = 0; kh < 5; kh++)
                                for (int kw = 0; kw < 5; kw++) {
                                    const int glim = g_out + 4 - kh - kw, g_in = ci / cin_g;
                                    if (g_in <= glim - 2 || g_in == glim - 1 || (g_in == glim && constrain == 6))
                                        fma_row(P, xn + ((size_t)ci * Hp + h + kh) * Wp + kw, wo[ci * 25 + kh * 5 + kw], W);
                                }
                    } else {
                        for (int j = 0; j * CB < Cin; j++) {
                            memset(u, 0, sizeof(float) * (size_t)W);
                            const int c1 = j * CB + CB < Cin ? j * CB + CB : Cin;
                            for (int ci = j * CB; ci < c1; ci++)
                                for (int kh = 0; kh < 5; kh++)
                                    for (int kw = 0; kw < 5; kw++)
                                        if (ci / cin_g <= g_out + 2 - kh - kw)
                                            fma_row(u, xn + ((size_t)ci * Hp + h + kh) * Wp + kw, wo[ci * 25 + kh * 5 + kw], W);
                            for (int w = 0; w < W; w++) P[w] = P[w] + u[w];
                        }
                        for (int cls = 0; cls < (constrain == 6 ? 2 : 1); cls++) {
                            float* S = cls ? Q : R;
                            for (int jq = 0; jq * CB < cin_g; jq++) {
                                memset(r, 0, sizeof(float) * (size_t)W);
                                const int cend = jq * CB + CB < cin_g ? jq * CB + CB : cin_g;
                                for (int c0 = jq * CB; c0 < cend; c0 += 4)
                                    for (int kh = 0; kh < 5; kh++)
                                        for (int kw = 0; kw < 5; kw++) {
                                            const int gsel = g_out + 3 + cls - kh - kw;
                                            if (gsel < 0 || gsel >= G) continue;
                                            for (int c = c0; c < c0 + 4 && c < cend; c++) {
                                                const int ci = gsel * cin_g + c;
                                                fma_row(r, xn + ((size_t)ci * Hp + h + kh) * Wp + kw, wo[ci * 25 + kh * 5 + kw], W);
                                            }
                                        }
                                for (int w = 0; w < W; w++) S[w] = S[w] + r[w];
                            }
                        }
                    }
                    const float b = bias[set * Cout + o];
                    const float sl = slope ? slope[set * Cout + o] : 0.f;
                    const size_t row = (((size_t)n * Cout + o) * H + h) * W;
                    for (int w = 0; w < W; w++) {
                        float v = variant == 2 ? ((P[w] + Q[w]) + R[w]) + b : ((P[w] + R[w]) + Q[w]) + b;
                        if (slope) v = v > 0.f ? v : v * sl;
                        if (resid) v = v + resid[row + w];
                        out[row + w] = v;
                    }
                }
        free(buf);
    }
    free(xp);
}
