// Wavefront engine of the fused decoder (wavefront.cu): data structures shared with codec.cu.
//
// One engine = the 12-layer context network of one bitstream (code stream: 48 groups x 3 nets, importance stream:
// 1 group) in its decoder form.  Activations live in two persistent layouts per layer:
//   FP  "planar skewed"   [set*C + c][D][HS]          d = h + w, HS = H rounded up to 4.  Source of the TMA box loads
//                                                      of the old-term kernel (a 5x5 window of 32 diagonal neighbours
//                                                      is the rectangle 36 x 9 in (h, d) coordinates).
//   FC  "group-major channel-last"  [set][D + 8][G + 10][H + 4][C/G]   zero border of 4 diagonals / 5 groups / 2 rows: the previous- and
//                                                      same-wavefront terms read one float4 (4 channels of a group)
//                                                      per tap with no bounds checks, and the 32 lanes of a warp
//                                                      (consecutive h on one diagonal, one group) read 512 contiguous bytes.
// Cells outside the image (w = d - h not in [0, W)) exist in both layouts, are never written and stay zero.
#pragma once
#include <cuda.h>
#include "internal.cuh"

namespace lic360 {

constexpr int WF_LAYERS = 12;

struct WfLayerDev {
    const float* xp;     // FP input frame (nullptr never: every layer has one)
    const float* xc;     // FC input frame
    float* op;           // FP output frame (nullptr for the last layer: nobody convolves it)
    float* oc;           // FC output frame
    const float* rc;     // FC residual frame (same shape as oc) or nullptr
    const float* wp;     // old-term weights      [set][chunk][ci][tap] float4
    const float* wq;     // R / Q weights    [cls][set][chunk][tap][c]  float4
    const float* bias;   // [set][Cout]
    const float* slope;  // [set][Cout] or nullptr (no PReLU)
    float4* pbuf[2];     // old-term sums P by step parity: [set][kc][D][HS]
    float4* rbuf[2];     // previous-wavefront sums R by step parity, same shape
    int Cin, Cout, cin_g, cout_g, cpg4, nchunk, nblk, nqb, has_q, pad;
};

struct WfNetDev {
    WfLayerDev L[WF_LAYERS];
    const StepDesc* steps;  // [nsteps]
    const int* ctr;         // current step (device counter, advanced at the end of every step graph)
    const int32_t* idx;     // index plan (row plane, column plane), code_contex_cuda.cu:11-32
    int nsets, G, H, W, D, HS, Dp, Hp, nsteps, parts, ndiag, pad;
};

// The CDF rows of the step are produced at the end of wf_chain4_kernel and wf_chain1_kernel (no extra launch on the critical path).
// wf_chain4_kernel (code stream) publishes every row by its tag wf_row_tag(step), with no system fence + flag behind the rows: the host
// validates row by row; it also evaluates the previous-wavefront terms of the NEXT step (layers 1..11) behind the rows.
// wf_chain1_kernel (importance stream) raises the flag once its rows are written.
// The tag of a step is never 0 (the value of a row nobody has written) and differs from the previous step's.  The persistent decode
// tags the decoded symbol words of a step with it too.
__host__ __device__ __forceinline__ int wf_row_tag(int step) { return step % 15 + 1; }
struct WfRows {
    uint16_t* rows;       // mapped pinned: packed rows of the step
    const float* levels;  // decoded importance levels (mask bit = Imp2mask + Dtow of the symbol's 2x2 cell)
    int* flag;            // mapped pinned: step + 1 once the rows are written (wf_chain1_kernel); -(step + 1): a wf_chain4_kernel CTA gave up
    int* sync;            // monotone counter: all nets have finished layer 11 of step p when it reaches (p + 1) * gridDim.x
    float s2;
};

// Low-latency ("persistent") decode of the many-group stream: ONE launch of the chain kernel walks all wavefront steps; between steps it
// waits for the host instead of being re-launched (no graph launch, no scatter kernel, no kernel prologue on the critical path).
struct WfPersist {
    const float* syms;   // mapped pinned: the symbols the host decoded for the previous step
    const int* go_host;  // mapped pinned, host -> device: step p may run once *go_host >= p; WF_GO_ABORT: stop at the next step boundary
    int* go_dev;         // device: CTA 0 republishes the host's decision here (p = run step p, -(p + 2) = abort instead of running p)
    const int* old_done; // device: old-term sums of steps < *old_done are complete (set by wf_old_done_kernel behind every old-term launch)
    int* ctr;            // device step counter kept up to date for the kernels that follow the decode (final scatter)
    int* scat_done;      // device, one per net: the symbols of steps < scat_done[n] are in net n's input frame (the old-term kernel of
                         // step q, enqueued by the host right behind go(q - 1), reads wavefronts <= q - 2 of that frame: it waits for q - 1)
    float bias, scale;   // TileInput: value = scale * symbol + bias
    int enabled;
};
constexpr int WF_GO_ABORT = -2;

struct WfMaps { CUtensorMap tm[WF_LAYERS]; };  // FP input frame of every layer, box {40 h, 9 d, 4 c}

struct WfEngine {
    WfNetDev dev;
    WfMaps maps;
    WfMaps maps4;         // box {72 h, 10 d, 2 c} of the four-positions-per-lane, two-diagonals-per-warp old-term kernel
    bool old4 = false;    // many-group net: wf_old4_kernel (else wf_old_kernel)
    int parts4 = 1;
    size_t old4_smem = 0;
    float* fp[WF_LAYERS + 1] = {nullptr};
    float* fc[WF_LAYERS + 1] = {nullptr};
    size_t fp_floats[WF_LAYERS + 1] = {0}, fc_floats[WF_LAYERS + 1] = {0};
    float4* pbuf = nullptr;
    size_t pbuf_f4 = 0;
    int C[WF_LAYERS + 1];
    int max_len = 0, cpg4_max = 0, nblk_max = 0, nqb_max = 0;
    int cluster = 1, chain_threads = 0;
    int chain_tasks = 0;  // wf_chain_kernel: (item, block) tasks of one CTA in the longest step's most expensive layer
    // chain4 and chain1 also produce the step's CDF rows and compute layer 0's previous-wavefront terms themselves (no launch for them)
    bool chain4 = false;  // many-group net (every chained layer has 4 channels per group): the staged-weight chain kernel
    bool chain1 = false;  // single-group net: the output-chunk-split chain kernel applies
    bool c1_dsm = false;  // chain1: both activation tiles fit, layers exchange activations through distributed shared memory
    int c1_kpc = 0, c1_lenp = 0, c1_cmax = 0, prev_wcap = 0;
    size_t old_smem = 0, prev_smem = 0, chain_smem = 0;
};

// G groups, cpg hidden channels per group, nlast output channels per group of the last layer, latent H x W
int wf_init(WfEngine& e, int G, int cpg, int nlast, int nsets, int H, int W, const int32_t* idx_dev, const StepDesc* steps_dev,
            const int* ctr_dev, int nsteps, int max_len);
void wf_set_layer(WfEngine& e, int l, const float* wp, const float* wq, const float* bias, const float* slope);
void wf_free(WfEngine& e);
int wf_chain_capacity(const WfEngine& e);  // decodes whose code-stream chains may be in flight together on the device
// wf_chain4_kernel's R tail: the most rounds in which a CTA stages its weight rows, over all steps (0: not a chain4 engine).
// idx, steps: the host copies of the index plan and the step list the engine was created with
int wf_tail_rounds(const WfEngine& e, const int32_t* idx, const StepDesc* steps);
const void* wf_old_kernel_ptr();  // to give the importance stream's old-term kernel node its own (lowest) priority in the step graph
cudaError_t wf_clear(const WfEngine& e, cudaStream_t s);                    // zero every frame (start of a decode)
// P of step *ctr + dp, all layers.  programmatic: launch as a programmatic dependent of the previous kernel in the stream
// psum >= 0: explicit step (persistent decode: the host knows it), else *ctr + dp.  done != nullptr: a one-thread kernel behind the launch
// publishes *done = psum + 1 (stream order: the old-term sums of that step are complete)
cudaError_t wf_launch_old(const WfEngine& e, int dp, cudaStream_t s, bool programmatic = false, int psum = -1, int* done = nullptr,
                          const int* scat_done = nullptr);
// R of step *ctr + dp for layers [l0, l1): layer 0 at dp = 0 right after the scatter (it reads the symbols just decoded),
// layers 1..11 at dp = 1 right after the chain (underneath the host decoder)
cudaError_t wf_launch_prev(const WfEngine& e, int dp, int l0, int l1, cudaStream_t s);
// the 12-layer chain of step *ctr; rows: where chain4 and chain1 put the step's CDF rows (the generic chain kernel ignores them);
// persist != nullptr (chain4 engines only): all steps in one launch, paced by the host through persist->go_host
cudaError_t wf_launch_chain(const WfEngine& e, cudaStream_t s, const WfRows& rows, const WfPersist* persist = nullptr);

// first channel of group g at (d, h); cpg = channels per group of that frame.  The group axis carries WF_GPAD zero
// groups on each side: a tap of the R / Q terms may select group -5 .. G+3, which then reads zeros instead of needing a test.
constexpr int WF_GPAD = 5;
__host__ __device__ inline size_t wf_fc_index(int Dp, int Hp, int G, int cpg, int n, int d, int g, int h) {
    return ((((size_t)n * Dp + d + 4) * (G + 2 * WF_GPAD) + g + WF_GPAD) * Hp + h + 2) * cpg;
}
// Debug timeline (LIC360_WF_TRACE=1): per step 8 slots of %globaltimer stamps.  Each translation unit has its own copy of
// the device pointer (no relocatable device code); wf_trace_set() / codec_trace_set() point both at the same buffer.
enum { WF_TR_SCATTER = 0, WF_TR_PREV, WF_TR_CHAIN0, WF_TR_CHAIN1, WF_TR_ROWS0, WF_TR_ROWS1, WF_TR_OLD0, WF_TR_OLD1, WF_TR_TAIL0, WF_TR_TAIL1, WF_TR_SLOTS };
void wf_trace_set(unsigned long long* buf, int sel);  // sel: 0 = trace the multi-group (code) stream, 1 = the single-group (importance) stream
#define WF_TRACE_DECL static __device__ unsigned long long* g_wf_trace = nullptr; static __device__ int g_wf_trace_sel = 0;
#define WF_TRACE_MIN(G, step, slot)                                                                       \
    do {                                                                                                  \
        if (g_wf_trace && ((G) > 1 ? 0 : 1) == g_wf_trace_sel) {                                                                                 \
            unsigned long long t_;                                                                        \
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_));                                        \
            atomicMin(g_wf_trace + (size_t)(step) * WF_TR_SLOTS + (slot), t_);                            \
        }                                                                                                 \
    } while (0)
#define WF_TRACE_MAX(G, step, slot)                                                                       \
    do {                                                                                                  \
        if (g_wf_trace && ((G) > 1 ? 0 : 1) == g_wf_trace_sel) {                                                                                 \
            unsigned long long t_;                                                                        \
            asm volatile("mov.u64 %0, %%globaltimer;" : "=l"(t_));                                        \
            atomicMax(g_wf_trace + (size_t)(step) * WF_TR_SLOTS + (slot), t_);                            \
        }                                                                                                 \
    } while (0)

// Planar skewed frame: row h of diagonal d lives in column h + WF_HSHIFT.  A 5x5 window starts two rows above its position, and the
// TMA unit wants box starts that are multiples of 4 floats: with the shift the box of a tile starting at row hb (a multiple of 4) starts
// at column hb, and a lane's first cell is 16-byte aligned in shared memory (wf_old4_kernel reads the band as float4).  Columns 0, 1
// and everything right of the image are never written: zeros (or the TMA unit's out-of-bounds fill).
constexpr int WF_HSHIFT = 2;
__host__ __device__ inline size_t wf_fp_index(int D, int HS, int C, int n, int c, int d, int h) {
    return (((size_t)n * C + c) * D + d) * HS + h + WF_HSHIFT;
}

}  // namespace lic360
