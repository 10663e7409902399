// Fused entropy codec of one ERP latent: the 238-step (code stream) and 95-step (importance stream) loops that the
// reference drives from Python with ~25 launches, 3 blocking copies and a per-op Coder call per step
// (test/lic360_demo.py:124-141,173-189,220-238,272-290) run here as one host C++ loop per stream:
//
//   encode : prep -> 12 whole-frame context convs (residual add fused) -> ONE kernel that emits the CDF rows of ALL
//            symbols in coding order (packed 16 B / 128 B rows) -> one D2H copy -> host arithmetic coder.
//   decode : per wavefront step ONE CUDA graph replay with two branches (wavefront.cu):
//              critical branch : scatter previous symbols -> previous-wavefront terms of all 12 layers (one launch) ->
//                                12-layer chain of same-wavefront terms (one cluster launch per step, TileAdd fused) ->
//                                CDF rows of the slab written straight into mapped pinned memory + completion flag
//              side branch     : old terms of ALL 12 layers of the NEXT step (one TMA-fed launch)
//            The host spins on the flag (no stream sync: the side branch may still be running), runs the arithmetic
//            decoder and writes the symbols into mapped pinned memory that the next replay's scatter kernel reads.
//            The step is read on the device from a counter, so the same graph is replayed for every step and image.
//
// The bitstream is the reference's (coder.cpp: same coder, same symbol order, same tables); the conv kernels are the
// ones behind CconvEcOp/CconvDcOp (conv.cu) and the row arithmetic is shared with EntropyGmmTableOp/EntropyTableOp
// (tables_dev.cuh), so per-op and fused paths are interchangeable bit for bit.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <functional>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <sched.h>
#include <thread>
#include <cmath>
#include <vector>
#include "coder_internal.h"
#include "internal.cuh"
#include "tables_dev.cuh"
#include "wavefront.cuh"

namespace lic360 {

struct NetDesc {
    int G = 0, cpg = 0, nlast = 0, nsets = 1, H = 0, W = 0;
    int Cin[12], Cout[12], constrain[12];
    bool act[12];
    float* wp[12] = {nullptr}; float* wq[12] = {nullptr}; float* bias[12] = {nullptr}; float* slope[12] = {nullptr};
    bool set[12] = {false};
    float* frame[13] = {nullptr};  // frame[0] = network input, frame[i+1] = output of layer i (persistent in decode)
    size_t frame_floats[13];
    int32_t* idx_dev = nullptr;
    std::vector<int32_t> plan;
    std::vector<StepDesc> steps;
    std::vector<int> row_off;  // first row of each step in coding order
    StepDesc* steps_dev = nullptr;
    int* row_off_dev = nullptr;
    int nsteps = 0, max_len = 0, total_rows = 0;
    cudaGraphExec_t graph = nullptr;
    int graph_nodes = 0;
    WfEngine wf;       // decoder form of the network (wavefront.cu)
    double t_kernel[5] = {0, 0, 0, 0, 0};  // profile mode: ms in old / prev / chain / scatter+rows kernels, steps
    // per-bitstream execution context: the two streams of an image are coded concurrently
    cudaStream_t stream = nullptr, side = nullptr;
    cudaEvent_t ev_fork = nullptr, ev_join = nullptr, ev_prof[6] = {nullptr};
    int* ctr_dev = nullptr;             // current wavefront step (device counter)
    int* done_dev = nullptr;            // CTA counter of the rows kernel
    int* arrived_dev = nullptr;         // CTA counter of the scatter kernel (the last CTA advances ctr_dev)
    int* sync_dev = nullptr;            // code stream: monotone cross-cluster counter of the chain kernel's rows phase
    int* flag_host = nullptr;           // mapped pinned: step + 1 once the rows of a step are in rows_step_host
    int nflags = 1;                     // host flags the rows producer raises (one per CTA of the fused code-stream chain)
    int* go_host = nullptr;             // mapped pinned: the stream may run step p once this is >= p (launch-ahead / persistent decode)
    int* go_dev = nullptr;              // persistent decode: CTA 0's republished go / abort decision
    int* old_done_dev = nullptr;        // persistent decode: old-term sums of steps < this are complete
    int* scat_done_dev = nullptr;       // persistent decode, one per net: symbols of steps < this are in the net's input frame
    uint16_t* rows_dev = nullptr;       // encode: all rows of the stream
    uint16_t* rows_host = nullptr;      // pinned
    uint16_t* rows_step_host = nullptr; // mapped pinned: rows of one decode step
    float* syms_host = nullptr;         // mapped pinned: decoded symbols of one step
    std::vector<float> step_wait_us, step_decode_us, step_levels_us;  // debug timeline (LIC360_WF_TRACE_FILE): host time per step waiting for rows / decoding
    int row_bytes = 16;                 // packed row size (16 B code stream, 128 B importance stream)
    bool tagged = false;                // decode: the step's rows carry a publication tag and are validated row by row (no fence + flag)
    double t_host_coder = 0, t_gpu_wait = 0, t_done = 0;
    lic360_coder* coder = nullptr;
    char err[256] = {0};                // error text of a worker thread (set_error is thread-local)
    double* bits_partial_dev = nullptr; // estimate: one partial sum per block of the bits kernel
    int bits_blocks = 0;
};

constexpr int BITS_THREADS = 256;  // block size of the estimate's bits and sum kernels

// device-side results of an estimate, copied back with one cudaMemcpyAsync; index = stream_id (0 code, 1 importance)
struct EstimateTotals {
    double bits[2];
    unsigned long long err[2];
};

}  // namespace lic360

using namespace lic360;

namespace lic360 {
// Per-device admission of concurrent decodes (ADVICE r1): the code-stream chain kernel's three clusters meet at a global
// counter, which only works while every cluster of every running chain is resident.  A decode takes a slot for its duration;
// the capacity comes from cudaOccupancyMaxActiveClusters (wf_chain_capacity), further decodes queue here on the host.
struct ChainSlots {
    std::mutex m;
    std::condition_variable cv;
    int in_use[kMaxDevices] = {0};
    void acquire(int dev, int cap, int units) {
        std::unique_lock<std::mutex> lk(m);
        cv.wait(lk, [&] { return in_use[dev] + units <= cap; });
        in_use[dev] += units;
    }
    void release(int dev, int units) {
        { std::lock_guard<std::mutex> lk(m); in_use[dev] -= units; }
        cv.notify_all();
    }
};
static ChainSlots g_chain_slots;
// units = 1: a graph-replay decode; units = cap: a low-latency decode, which owns the device while it runs -- its chain clusters stay
// resident from the first to the last step, and with several of them pinned (24 SMs each, wherever the hardware found room) the
// 16-CTA cluster of an importance stream may not find a GPC with enough free SMs for as long as they run (observed: decodes timing
// out waiting for importance levels with two or more resident chains and decodes starting and finishing around them)
struct ChainSlot {
    int dev, units;
    ChainSlot(int d, int cap, int u) : dev(d), units(std::max(1, std::min(u, cap))) { g_chain_slots.acquire(d, cap, units); }
    ~ChainSlot() { g_chain_slots.release(dev, units); }
};

// the importance stream of a decode runs on a second host thread: one persistent worker per codec (not a std::thread per call)
struct StreamWorker {
    std::thread th;
    std::mutex m;
    std::condition_variable cv;
    std::function<void()> job;
    bool has_job = false, quit = false, busy = false;
    void loop() {
        std::unique_lock<std::mutex> lk(m);
        for (;;) {
            cv.wait(lk, [&] { return has_job || quit; });
            if (quit) return;
            std::function<void()> j = std::move(job);
            has_job = false;
            lk.unlock();
            j();
            lk.lock();
            busy = false;
            cv.notify_all();
        }
    }
    void submit(std::function<void()> j) {
        std::unique_lock<std::mutex> lk(m);
        if (!th.joinable()) th = std::thread([this] { loop(); });
        job = std::move(j);
        has_job = true; busy = true;
        cv.notify_all();
    }
    void wait() {
        std::unique_lock<std::mutex> lk(m);
        cv.wait(lk, [&] { return !busy; });
    }
    ~StreamWorker() {
        { std::lock_guard<std::mutex> lk(m); quit = true; }
        cv.notify_all();
        if (th.joinable()) th.join();
    }
};
}  // namespace lic360

struct lic360_codec {
    int device = 0, H = 0, W = 0;
    int chain_cap = 1;                  // concurrent decodes the device can hold (wf_chain_capacity)
    lic360::StreamWorker imp_worker;
    int mode = 0;                       // 0: pipelined graph replay, 1: serialized launches with per-kernel event timing
    NetDesc code, imp;
    float* levels_dev = nullptr;        // decoded importance levels (1,1,H/2,W/2), filled diagonal by diagonal
    float* mask192_dev = nullptr;       // scratch: Imp2mask output
    std::atomic<int> imp_ready{0};      // decode: importance levels of diagonals < imp_ready are in levels_dev
    std::atomic<int> abort_flag{0};     // decode: one of the two stream loops failed
    lic360::EstimateTotals* est_dev = nullptr;   // estimate: totals and error keys of both streams
    lic360::EstimateTotals* est_host = nullptr;  // pinned copy of est_dev
    cudaEvent_t ev_est = nullptr;                // estimate: the importance stream's results are in est_dev
    double t_host_coder = 0, t_total = 0, t_gpu_wait = 0, t_imp = 0, t_gpu_steps = 0, t_gpu_steps_imp = 0;
};

namespace lic360 {

WF_TRACE_DECL
static void codec_trace_set(unsigned long long* buf, int sel) {
    cudaMemcpyToSymbol(g_wf_trace, &buf, sizeof(buf));
    cudaMemcpyToSymbol(g_wf_trace_sel, &sel, sizeof(sel));
}

// ------------------------------------------------------------------------------------------------ kernels
// code stream encoder input: x = (code - 3.5) * mask replicated for the 3 nets (lic360_demo.py:130-131)
__global__ void prep_code_kernel(const float* __restrict__ code, const float* __restrict__ mask, float* __restrict__ x,
                                 int n, float bias) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float v = (code[i] - bias) * mask[i];
        x[i] = v; x[i + n] = v; x[i + 2 * n] = v;
    }
}

// y: (3, G*3, H, W) outputs of [weight_net, delta_net, mean_net]; one thread = one symbol (tc, k) in plan order.
// all_steps != 0: encoder, every symbol, row index = coding order; else: decoder, the slab of steps[*ctr].
__global__ void gmm_rows_kernel(const float* __restrict__ y, const float* __restrict__ code, const float* __restrict__ mask,
                                const int32_t* __restrict__ idx, const StepDesc* __restrict__ steps,
                                const int* __restrict__ row_off, const int* __restrict__ ctr, uint16_t* __restrict__ rows,
                                int G, int H, int W, int all_steps, float s2) {
    const int HW = H * W;
    int th, tw, tc, row;
    if (all_steps) {
        const int i = blockIdx.x * blockDim.x + threadIdx.x;
        if (i >= G * HW) return;
        const int k = i % HW;
        tc = i / HW;
        th = __ldg(idx + k); tw = __ldg(idx + k + HW);
        const int p = th + tw + tc;
        row = __ldg(row_off + p) + k - steps[p].start;
    } else {
        const StepDesc d = steps[*ctr];
        const int l = blockIdx.x * blockDim.x + threadIdx.x;
        if (l >= d.len) return;
        th = __ldg(idx + d.start + l); tw = __ldg(idx + d.start + l + HW);
        tc = d.psum - th - tw;
        row = l;
    }
    float wv[3], dv[3], mv[3], o[9];
    const size_t net = (size_t)G * 3 * HW;
    const size_t base = ((size_t)tc * 3 * H + th) * W + tw;
#pragma unroll
    for (int i = 0; i < 3; i++) {
        wv[i] = y[base + (size_t)i * HW];
        dv[i] = y[net + base + (size_t)i * HW];
        mv[i] = y[2 * net + base + (size_t)i * HW];
    }
    gmm_row(wv, dv, mv, o, 3, 8, 3.5f, 65536.f, 1e-6f, s2);
    const size_t pos = ((size_t)tc * H + th) * W + tw;
    const int sym = code ? code_symbol(code[pos]) : 0;  // NaN and anything outside [0, 8) become the out-of-range marker of the row
    pack_gmm_row(o, sym, code_mask_bit(mask[pos]), rows + (size_t)row * 8);
}

// importance stream: y (1, 49, h, w) logits; one thread = one position in plan order (G = 1: step p = diagonal p)
__global__ void imp_rows_kernel(const float* __restrict__ y, const float* __restrict__ levels, const int32_t* __restrict__ idx,
                                const StepDesc* __restrict__ steps, const int* __restrict__ ctr, uint16_t* __restrict__ rows,
                                int H, int W, int all_steps) {
    const int HW = H * W;
    int k, row;
    if (all_steps) {
        k = blockIdx.x * blockDim.x + threadIdx.x;
        if (k >= HW) return;
        row = k;
    } else {
        const StepDesc d = steps[*ctr];
        const int l = blockIdx.x * blockDim.x + threadIdx.x;
        if (l >= d.len) return;
        k = d.start + l;
        row = l;
    }
    const int th = __ldg(idx + k), tw = __ldg(idx + k + HW);
    float o[50];
    for (int i = 0; i < 49; i++) o[1 + i] = y[((size_t)i * H + th) * W + tw];
    entropy_row(o, 49, 65536.f);
    uint16_t* dst = rows + (size_t)row * 64;
    uint32_t ovf[3] = {0, 0, 0};
    for (int j = 1; j <= 48; j++) {
        const uint32_t v = (uint32_t)(int)o[j];
        dst[j - 1] = (uint16_t)(v & 0xFFFF);
        ovf[(j - 1) / 16] |= ((v >> 16) & 1u) << ((j - 1) % 16);
    }
    dst[48] = levels ? (uint16_t)imp_symbol(levels[th * W + tw]) : 0;
    dst[49] = (uint16_t)ovf[0]; dst[50] = (uint16_t)ovf[1]; dst[51] = (uint16_t)ovf[2];
}

// ---- rate estimate (lic360_codec_estimate): the ideal code length 16 - log2(T[s+1] - T[s]) bits of every symbol the encoder would
// code, from the rows the two kernels above build (same row functions, same symbol and mask rules), without packing the rows or
// running the host coder.  One thread per symbol, in any order.  A symbol's cost goes into its block's partial in a fixed tree order
// and bits_sum_kernel adds the partials in a fixed order too, so a total depends on the inputs only (no floating-point atomics).
// The first error in CODING order -- the row the host coder would stop at -- is kept as the smallest key (row << 32) | symbol;
// symbol >= number of symbols: out of range, else: a zero-width bin.
constexpr unsigned long long kNoError = ~0ull;

// sum of v over the block in a fixed order (a shuffle tree per warp, then one over the warp sums); valid in thread 0
__device__ __forceinline__ double block_sum_fixed(double v) {
    __shared__ double warp_sum[BITS_THREADS / 32];
#pragma unroll
    for (int k = 16; k > 0; k >>= 1) v += __shfl_down_sync(0xffffffffu, v, k);
    if ((threadIdx.x & 31) == 0) warp_sum[threadIdx.x >> 5] = v;
    __syncthreads();
    if (threadIdx.x < 32) {
        v = threadIdx.x < BITS_THREADS / 32 ? warp_sum[threadIdx.x] : 0.0;
#pragma unroll
        for (int k = 16; k > 0; k >>= 1) v += __shfl_down_sync(0xffffffffu, v, k);
    }
    return v;
}

// cost of symbol s (0 <= s < N) of a row; false: zero-width bin, which the host coder refuses ("symbol has zero frequency")
template <int N>
__device__ __forceinline__ bool symbol_bits(const float* o, int s, double* bits) {
    uint32_t lo, hi;
    coded_bins<N>(o, s, &lo, &hi);
    if (lo == hi) return false;
    *bits = 16.0 - log2((double)hi - (double)lo);
    return true;
}

// code stream: y as in gmm_rows_kernel; thread i = symbol (tc = i / HW, k = i % HW in plan order), bits in (G, H, W) layout
__global__ void __launch_bounds__(BITS_THREADS) gmm_bits_kernel(const float* __restrict__ y, const float* __restrict__ code,
                                const float* __restrict__ mask, const int32_t* __restrict__ idx, const StepDesc* __restrict__ steps,
                                const int* __restrict__ row_off, float* __restrict__ bits, double* __restrict__ partial,
                                unsigned long long* err, int G, int H, int W, float s2) {
    const int HW = H * W;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    double cost = 0.0;
    if (i < G * HW) {
        const int k = i % HW, tc = i / HW;
        const int th = __ldg(idx + k), tw = __ldg(idx + k + HW);
        const size_t pos = ((size_t)tc * H + th) * W + tw;
        if (code_mask_bit(mask[pos])) {  // a position the encoder skips costs nothing, whatever its symbol
            float wv[3], dv[3], mv[3], o[9];
            const size_t net = (size_t)G * 3 * HW;
            const size_t base = ((size_t)tc * 3 * H + th) * W + tw;
#pragma unroll
            for (int j = 0; j < 3; j++) {
                wv[j] = y[base + (size_t)j * HW];
                dv[j] = y[net + base + (size_t)j * HW];
                mv[j] = y[2 * net + base + (size_t)j * HW];
            }
            gmm_row(wv, dv, mv, o, 3, 8, 3.5f, 65536.f, 1e-6f, s2);
            const int s = code_symbol(code[pos]);
            if (s > 7 || !symbol_bits<8>(o, s, &cost)) {
                const int p = th + tw + tc;
                const unsigned long long row = (unsigned)(__ldg(row_off + p) + k - steps[p].start);
                atomicMin(err, (row << 32) | (unsigned)s);
                cost = 0.0;
            }
        }
        bits[pos] = (float)cost;
    }
    cost = block_sum_fixed(cost);
    if (threadIdx.x == 0) partial[blockIdx.x] = cost;
}

// importance stream: y (1, 49, h, w) logits; thread k = position k of the plan = row k of the stream, bits in (h, w) layout
__global__ void __launch_bounds__(BITS_THREADS) imp_bits_kernel(const float* __restrict__ y, const float* __restrict__ levels,
                                const int32_t* __restrict__ idx, float* __restrict__ bits, double* __restrict__ partial,
                                unsigned long long* err, int H, int W) {
    const int HW = H * W;
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    double cost = 0.0;
    if (k < HW) {
        const int th = __ldg(idx + k), tw = __ldg(idx + k + HW);
        float o[50];
        for (int j = 0; j < 49; j++) o[1 + j] = y[((size_t)j * H + th) * W + tw];
        entropy_row(o, 49, 65536.f);
        const uint32_t s = imp_symbol(levels[th * W + tw]);
        if (s >= 49 || !symbol_bits<49>(o, (int)s, &cost)) {
            atomicMin(err, ((unsigned long long)k << 32) | s);
            cost = 0.0;
        }
        bits[th * W + tw] = (float)cost;
    }
    cost = block_sum_fixed(cost);
    if (threadIdx.x == 0) partial[blockIdx.x] = cost;
}

// one block: thread t adds partials t, t + BITS_THREADS, ... in index order, then the block's fixed tree
__global__ void __launch_bounds__(BITS_THREADS) bits_sum_kernel(const double* __restrict__ partial, int n, double* __restrict__ total) {
    double v = 0.0;
    for (int i = threadIdx.x; i < n; i += BITS_THREADS) v += partial[i];
    v = block_sum_fixed(v);
    if (threadIdx.x == 0) *total = v;
}

// TileInput of the previous step read from mapped pinned memory (tile_input_cuda.cu:27-43) into both layouts of the
// engine's input frame, replicated for the nsets nets; no-op at step 0.  This is the FIRST kernel of a step and it also advances
// the device step counter: every CTA reads the old value on entry (step = old + 1), the last CTA to finish publishes the new
// one, and every later kernel of the step reads it at its own start -- no one-thread "advance" launch at the end of the step.
__global__ void scatter_prev_kernel(const float* __restrict__ syms, float* __restrict__ fp0, float* __restrict__ fc0,
                                    const int32_t* __restrict__ idx, const StepDesc* __restrict__ steps, int* __restrict__ ctr,
                                    int* __restrict__ arrived, int G, int H, int W, int D, int HS, int Dp, int Hp, float bias,
                                    float scale, int rep, float* __restrict__ keep) {
    const int c = *reinterpret_cast<volatile int*>(ctr) + 1;
    if (threadIdx.x == 0 && blockIdx.x == 0) WF_TRACE_MIN(G, c, WF_TR_SCATTER);
    if (c > 0) {
        const StepDesc d = steps[c - 1];
        const int HW = H * W;
        for (int l = blockIdx.x * blockDim.x + threadIdx.x; l < d.len; l += gridDim.x * blockDim.x) {
            const int th = __ldg(idx + d.start + l), tw = __ldg(idx + d.start + l + HW);
            const int tc = d.psum - th - tw;
            const float s = syms[l];
            const float v = fmaf(scale, s, bias);
            for (int r = 0; r < rep; r++) {
                fp0[wf_fp_index(D, HS, G, r, tc, th + tw, th)] = v;
                fc0[wf_fc_index(Dp, Hp, G, 1, r, th + tw, tc, th)] = v;
            }
            if (keep) keep[th * W + tw] = s;  // importance stream: the decoded level itself
        }
    }
    __syncthreads();
    if (threadIdx.x == 0) {
        __threadfence();
        if (atomicAdd(arrived, 1) == (int)gridDim.x - 1) {
            *arrived = 0;
            *ctr = c;
        }
    }
}

// code = frame[0:1] + 3.5 * mask (lic360_demo.py:236-237), gathered from the channel-last engine frame
__global__ void finish_code_kernel(const float* __restrict__ fc0, const float* __restrict__ mask, float* __restrict__ out,
                                   int G, int H, int W, int Dp, int Hp, float bias) {
    const int n = G * H * W;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int w = i % W, h = (i / W) % H, g = i / (W * H);
        out[i] = fc0[wf_fc_index(Dp, Hp, G, 1, 0, h + w, g, h)] + bias * mask[i];
    }
}

// all rows of a step are in mapped pinned memory: the last CTA raises the host flag
__device__ __forceinline__ void rows_done(int* done, volatile int* flag, int step, int G) {
    __threadfence_system();
    __syncthreads();
    if (threadIdx.x == 0) {
        if (atomicAdd(done, 1) == (int)gridDim.x - 1) {
            *done = 0;
            __threadfence_system();
            *flag = step + 1;
            WF_TRACE_MAX(G, step, WF_TR_ROWS1);
        }
    }
}

// decoder: CDF rows of the slab of step *ctr from the engine's last frame (group-major channel-last, 3 nets x G x 3).
// 8 lanes per symbol: lane j computes bin j (the 21 erff of a row are the critical path of this latency-bound kernel),
// lane 0 gathers the bins, runs the monotonic fix-up and stores the packed 16-byte row.
// The mask bit of a symbol comes straight from the decoded importance level of its 2x2 cell (Imp2mask + Dtow fused:
// mask_up[g][h][w] = (4g + 2(h%2) + (w%2)) < 4*level[h/2][w/2], imp2mask_cuda.cu:25-38, dtow_cuda.cu:38-56), so the code
// stream only needs the importance diagonals that are already decoded and the two streams decode concurrently.
__global__ void gmm_rows_wf_kernel(const float* __restrict__ y, const float* __restrict__ levels, const int32_t* __restrict__ idx,
                                   const StepDesc* __restrict__ steps, const int* __restrict__ ctr, uint16_t* __restrict__ rows,
                                   int G, int H, int W, int Dp, int Hp, float s2, int* done, int* flag) {
    const int step = *ctr;
    if (threadIdx.x == 0) WF_TRACE_MIN(G, step, WF_TR_ROWS0);
    const StepDesc d = steps[step];
    const int gt = blockIdx.x * blockDim.x + threadIdx.x;
    const int l = gt >> 3, j = gt & 7;
    const bool live = l < d.len;
    float bin = 0.f;
    int th = 0, tw = 0, tc = 0;
    if (live) {
        const int HW = H * W;
        th = __ldg(idx + d.start + l); tw = __ldg(idx + d.start + l + HW);
        tc = d.psum - th - tw;
        float wv[3], dv[3], mv[3];
#pragma unroll
        for (int i = 0; i < 3; i++) {
            wv[i] = y[wf_fc_index(Dp, Hp, G, 3, 0, th + tw, tc, th) + i];
            dv[i] = y[wf_fc_index(Dp, Hp, G, 3, 1, th + tw, tc, th) + i];
            mv[i] = y[wf_fc_index(Dp, Hp, G, 3, 2, th + tw, tc, th) + i];
        }
        gmm_prep(wv, dv, 3, 1e-6f);
        if (j >= 1) bin = gmm_bin_value(wv, dv, mv, j, 3, 3.5f, 65536.f, s2);
    }
    float o[9];
    o[0] = 0.f; o[8] = 65536.f;
#pragma unroll
    for (int k = 1; k < 8; k++) o[k] = __shfl_sync(0xffffffffu, bin, (threadIdx.x & 24) + k);
    if (live && j == 0) {
        fixup_row(o, 8, true);
        const int lvl = (int)(levels[(th >> 1) * (W >> 1) + (tw >> 1)] + 1e-5f);
        pack_gmm_row(o, 0, (4 * tc + 2 * (th & 1) + (tw & 1)) < 4 * lvl ? 1 : 0, rows + (size_t)l * 8);
    }
    rows_done(done, flag, step, G);
}

// decoder, importance stream: CDF row of every position of the step's diagonal from the 49 logits of the engine's last frame.
// One WARP per symbol (the step has <= min(H, W) symbols and sits on the critical path of BOTH streams, so it is latency that
// counts): lanes hold logits i and i + 32, the softmax denominator is accumulated in index order by every lane from shared memory
// (the serial order of entropy_row, tables_dev.cuh, is part of the bit-exact contract), the cumulative table is a warp scan of
// integers (exact in fp32, so min(prefix, total) equals the serial clipped recurrence), lane 0 runs the serial fix-up and the
// warp stores the packed 128-byte row with one coalesced write.
constexpr int IMP_ROWS_WARPS = 8;
__global__ void __launch_bounds__(32 * IMP_ROWS_WARPS) imp_rows_wf_kernel(const float* __restrict__ y, const int32_t* __restrict__ idx,
                                   const StepDesc* __restrict__ steps, const int* __restrict__ ctr, uint16_t* __restrict__ rows,
                                   int H, int W, int Dp, int Hp, int* done, int* flag) {
    __shared__ float sh[IMP_ROWS_WARPS][64];
    const int step = *ctr;
    if (threadIdx.x == 0) WF_TRACE_MIN(1, step, WF_TR_ROWS0);
    const StepDesc d = steps[step];
    const int lane = threadIdx.x & 31, wp = threadIdx.x >> 5;
    for (int l = blockIdx.x * IMP_ROWS_WARPS + wp; l < d.len; l += gridDim.x * IMP_ROWS_WARPS) {  // warp-uniform
        const int th = __ldg(idx + d.start + l), tw = __ldg(idx + d.start + l + H * W);
        const float* yp = y + wf_fc_index(Dp, Hp, 1, 49, 0, th + tw, 0, th);
        entropy_row49_warp(yp[lane], lane + 32 < 49 ? yp[lane + 32] : -INFINITY, sh[wp], lane, 0, rows + (size_t)l * 64);
    }
    rows_done(done, flag, step, 1);
}

// ------------------------------------------------------------------------------------------------ host helpers
static void net_init(NetDesc& n, int G, int cpg, int nlast, int nsets, int H, int W) {
    n.G = G; n.cpg = cpg; n.nlast = nlast; n.nsets = nsets; n.H = H; n.W = W;
    for (int l = 0; l < 12; l++) {
        n.Cin[l] = G * (l == 0 ? 1 : cpg);
        n.Cout[l] = G * (l == 11 ? nlast : cpg);
        n.constrain[l] = l == 0 ? 5 : 6;
        n.act[l] = l != 11;
    }
    n.frame_floats[0] = (size_t)nsets * G * H * W;
    for (int l = 0; l < 12; l++) n.frame_floats[l + 1] = (size_t)nsets * n.Cout[l] * H * W;
}

static int net_alloc(NetDesc& n) {
    for (int i = 0; i < 13; i++) LIC360_CUDA(cudaMalloc(&n.frame[i], n.frame_floats[i] * sizeof(float)));
    const int H = n.H, W = n.W, G = n.G;
    std::vector<int32_t> idx(2 * (size_t)H * W);
    n.plan.resize(H + W);
    lic360_code_contex(H, W, idx.data(), n.plan.data());
    LIC360_CUDA(cudaMalloc(&n.idx_dev, idx.size() * sizeof(int32_t)));
    LIC360_CUDA(cudaMemcpy(n.idx_dev, idx.data(), idx.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
    n.nsteps = H + W + G - 2;
    n.steps.resize(n.nsteps);
    n.row_off.resize(n.nsteps + 1);
    int off = 0;
    for (int p = 0; p < n.nsteps; p++) {
        int s, l;
        slab_of(n.plan.data(), H, W, G, p, &s, &l);
        n.steps[p] = {p, s, l, 0};
        n.row_off[p] = off;
        off += l;
        if (l > n.max_len) n.max_len = l;
    }
    n.row_off[n.nsteps] = off;
    n.total_rows = off;
    LIC360_CUDA(cudaMalloc(&n.steps_dev, n.nsteps * sizeof(StepDesc)));
    LIC360_CUDA(cudaMemcpy(n.steps_dev, n.steps.data(), n.nsteps * sizeof(StepDesc), cudaMemcpyHostToDevice));
    LIC360_CUDA(cudaMalloc(&n.row_off_dev, (n.nsteps + 1) * sizeof(int)));
    LIC360_CUDA(cudaMemcpy(n.row_off_dev, n.row_off.data(), (n.nsteps + 1) * sizeof(int), cudaMemcpyHostToDevice));
    return LIC360_OK;
}

static void net_free(NetDesc& n) {
    for (int i = 0; i < 13; i++) cudaFree(n.frame[i]);
    for (int l = 0; l < 12; l++) { cudaFree(n.wp[l]); cudaFree(n.wq[l]); cudaFree(n.bias[l]); cudaFree(n.slope[l]); }
    cudaFree(n.idx_dev); cudaFree(n.steps_dev); cudaFree(n.row_off_dev);
    if (n.graph) cudaGraphExecDestroy(n.graph);
}

// layer l: input frame, output frame, fused residual (the `y + x` / TileAdd of the residual blocks)
static void layer_io(const NetDesc& n, int l, const float** x, const float** resid, float** out) {
    *x = n.frame[l];
    *out = n.frame[l + 1];
    *resid = (l >= 2 && l <= 10 && (l % 2) == 0) ? n.frame[l - 1] : nullptr;  // conv2 of block b = layer 2b+2
}

static int conv_args(const NetDesc& n, int l, ConvArgs& a) {
    const float *x, *r;
    float* out;
    layer_io(n, l, &x, &r, &out);
    if (fill_conv_args(a, x, n.wp[l], n.wq[l], n.bias[l], n.act[l] ? n.slope[l] : nullptr, r, out, n.nsets, n.Cin[l], n.H, n.W,
                       n.Cout[l], n.G, n.constrain[l], n.nsets)) {
        set_error("codec: bad layer geometry");
        return LIC360_ERR_ARG;
    }
    return LIC360_OK;
}

static int run_ec_net(const NetDesc& n, cudaStream_t s) {
    for (int l = 0; l < 12; l++) {
        ConvArgs a;
        int rc = conv_args(n, l, a);
        if (rc) return rc;
        LIC360_CUDA(launch_cconv_ec(a, s, false));  // the canonical P pass: the decoder reproduces these outputs bit for bit
    }
    return LIC360_OK;
}

static int check_params(const NetDesc& n) {
    for (int l = 0; l < 12; l++)
        if (!n.set[l]) { set_error("codec: layer %d has no parameters (call lic360_codec_set_layer)", l); return LIC360_ERR_ARG; }
    return LIC360_OK;
}

// the kernels of one decode step.  side == s (serialized / profile mode): everything in stream order, the old terms of
// the NEXT step last.  side != s (graph capture): the old terms run on a parallel low-priority branch; either way the
// host is released by the flag that the rows kernel raises, so the bulk of the arithmetic also overlaps the host coder.
// ev != nullptr: profile mode, events bracket the kernel classes (everything on `s`).
#define WF_DEBUG_SYNC(what)                                                                               \
    do {                                                                                                \
        if (dbg) {                                                                                      \
            cudaError_t e_ = cudaStreamSynchronize(s);                                                  \
            if (e_ != cudaSuccess) { set_error("codec: %s failed -> %s", what, cudaGetErrorString(e_)); return LIC360_ERR_CUDA; } \
        }                                                                                               \
    } while (0)

static int launch_step(lic360_codec* c, NetDesc& n, bool is_code, cudaStream_t s, cudaStream_t side, cudaEvent_t* ev) {
    const WfNetDev& w = n.wf.dev;
    static const bool dbg_env = getenv("LIC360_DEBUG_SYNC") != nullptr;
    const bool dbg = dbg_env && ev != nullptr;  // only in the serialized mode
    const int tgrid = (n.max_len + 127) / 128;
    if (ev) LIC360_CUDA(cudaEventRecord(ev[0], s));
    if (is_code)
        scatter_prev_kernel<<<tgrid, 128, 0, s>>>(n.syms_host, n.wf.fp[0], n.wf.fc[0], n.idx_dev, n.steps_dev, n.ctr_dev, n.arrived_dev, n.G, n.H, n.W,
                                                  w.D, w.HS, w.Dp, w.Hp, -3.5f, 1.0f, 3, nullptr);
    else
        scatter_prev_kernel<<<tgrid, 128, 0, s>>>(n.syms_host, n.wf.fp[0], n.wf.fc[0], n.idx_dev, n.steps_dev, n.ctr_dev, n.arrived_dev, 1, n.H, n.W,
                                                  w.D, w.HS, w.Dp, w.Hp, -1.0f, (float)(2. / (48 - 1.)), 1, c->levels_dev);
    LAUNCH_CHECK();
    WF_DEBUG_SYNC("scatter kernel");
    const bool fork = side != s;  // graph capture: overlap the old terms of the next step with the chain (see below)
    if (ev) LIC360_CUDA(cudaEventRecord(ev[1], s));
    const bool fused_rows = (is_code ? n.wf.chain4 : n.wf.chain1) && !getenv("LIC360_WF_ROWS_KERNEL");
    if (!(fused_rows && n.wf.r0_inline)) {  // else the chain kernel evaluates them in its prologue
        LIC360_CUDA(wf_launch_prev(n.wf, 0, 0, 1, s));  // layer 0 only: its taps read the symbols scattered a moment ago
        WF_DEBUG_SYNC("previous-wavefront kernel (layer 0)");
    }
    if (ev) LIC360_CUDA(cudaEventRecord(ev[2], s));
    // the chain; for the code stream it also emits the CDF rows of the step and raises the host flag
    WfRows rows;
    memset(&rows, 0, sizeof(rows));
    if (fused_rows) {
        rows.rows = n.rows_step_host; rows.levels = c->levels_dev; rows.done = n.done_dev; rows.flag = n.flag_host;
        rows.sync = n.sync_dev; rows.s2 = (float)(1. / sqrt(2.0)); rows.enabled = 1;
    }
    // code stream: the chain kernel also leaves the previous-wavefront terms of the next step behind (no launch, no side branch)
    n.nflags = fused_rows && is_code ? n.wf.dev.nsets * n.wf.cluster : 1;
    if (n.nflags > 64) { set_error("codec: %d chain CTAs exceed the 64 host flags", n.nflags); return LIC360_ERR_ARG; }
    const bool rtail = fused_rows && is_code && n.wf.chain4 && !getenv("LIC360_WF_PREV_KERNEL");
    rows.rtail = rtail ? 1 : 0;
    // code stream: every 16-byte row is published by its own tag (step % 15 + 1 in the meta word; 0 = never written); the host decodes row i as soon as
    // it has arrived -- no system fence and no flag write behind the rows, and the PCIe flight of the later rows overlaps the decoding
    n.tagged = fused_rows && is_code && n.wf.chain4 && !getenv("LIC360_WF_ROWS_FLAGS");
    rows.tagged = n.tagged ? 1 : 0;
    LIC360_CUDA(wf_launch_chain(n.wf, s, fused_rows ? &rows : nullptr));
    WF_DEBUG_SYNC("chain kernel");
    if (ev) LIC360_CUDA(cudaEventRecord(ev[3], s));
    // The old terms of step p+1 only read wavefronts <= p-1: they are launched right behind the chain kernel as its
    // PROGRAMMATIC dependent -- they start once every chain CTA is resident (so the chain's clusters got their SMs first)
    // and fill the SMs the chain leaves idle.  Whatever still needs the chain's RESULTS (a separate rows kernel, the
    // previous-wavefront kernel of the next step) waits for the chain's completion on the side stream; when the chain kernel
    // does all of that itself (rtail) there is no side branch at all.
    cudaStream_t rs = s;  // stream of the kernels behind the chain
    if (fork) {
        LIC360_CUDA(cudaEventRecord(n.ev_fork, s));
        LIC360_CUDA(wf_launch_old(n.wf, 1, s, true));
        if (!rtail) {
            LIC360_CUDA(cudaStreamWaitEvent(side, n.ev_fork, 0));
            rs = side;
        }
    }
    if (fused_rows) {
    } else if (is_code)
        gmm_rows_wf_kernel<<<(n.max_len * 8 + 127) / 128, 128, 0, rs>>>(n.wf.fc[12], c->levels_dev, n.idx_dev,
                                                 n.steps_dev, n.ctr_dev, n.rows_step_host, n.G, n.H, n.W, w.Dp, w.Hp,
                                                 (float)(1. / sqrt(2.0)), n.done_dev, n.flag_host);
    else
        imp_rows_wf_kernel<<<std::max(1, std::min(4, (n.max_len + IMP_ROWS_WARPS - 1) / IMP_ROWS_WARPS)), 32 * IMP_ROWS_WARPS, 0, rs>>>(n.wf.fc[12], n.idx_dev, n.steps_dev, n.ctr_dev, n.rows_step_host, n.H, n.W, w.Dp, w.Hp,
                                                 n.done_dev, n.flag_host);
    if (!fused_rows) LAUNCH_CHECK();
    WF_DEBUG_SYNC("rows kernel");
    // previous-wavefront terms of layers 1..11 for step p+1 (the activations of wavefront p are final): behind the rows
    // kernel, i.e. underneath the host decoder instead of on the critical path
    if (!rtail) LIC360_CUDA(wf_launch_prev(n.wf, 1, 1, WF_LAYERS, rs));
    WF_DEBUG_SYNC("previous-wavefront kernel (layers 1..11 of the next step)");
    if (ev) LIC360_CUDA(cudaEventRecord(ev[4], s));
    if (fork && rtail) {
        // the old-term kernel is only a PROGRAMMATIC dependent of the chain: give the end of the step a full edge from the chain too
        LIC360_CUDA(cudaStreamWaitEvent(s, n.ev_fork, 0));
    } else if (fork) {
        LIC360_CUDA(cudaEventRecord(n.ev_join, side));
        LIC360_CUDA(cudaStreamWaitEvent(s, n.ev_join, 0));
    } else {
        LIC360_CUDA(wf_launch_old(n.wf, 1, s));
    }
    WF_DEBUG_SYNC("old-term kernel");
    if (ev) LIC360_CUDA(cudaEventRecord(ev[5], s));
    return LIC360_OK;
}

// capture one decode step of a stream into a graph (replayed for every step)
static int build_step_graph(lic360_codec* c, NetDesc& n, bool is_code) {
    if (n.graph) return LIC360_OK;
    cudaStream_t s = n.stream;
    cudaGraph_t g;
    const long long l0 = g_launches;
    LIC360_CUDA(cudaStreamBeginCapture(s, cudaStreamCaptureModeThreadLocal));
    const bool overlap = getenv("LIC360_WF_NO_OVERLAP") == nullptr;  // (graph build time: not on a hot path)
    const int rc = launch_step(c, n, is_code, s, overlap ? n.side : s, nullptr);
    cudaError_t e = cudaStreamEndCapture(s, &g);
    n.graph_nodes = (int)(g_launches - l0);
    g_launches = l0;  // captured, not launched: replays are counted in decode_stream
    if (rc != LIC360_OK) { if (e == cudaSuccess) cudaGraphDestroy(g); return rc; }
    LIC360_CUDA(e);
    {   // kernel-node priorities: old-term kernel lowest, everything on the critical path highest
        int prio_lo = 0, prio_hi = 0;
        cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
        size_t nn = 0;
        LIC360_CUDA(cudaGraphGetNodes(g, nullptr, &nn));
        std::vector<cudaGraphNode_t> nodes(nn);
        LIC360_CUDA(cudaGraphGetNodes(g, nodes.data(), &nn));
        for (size_t i = 0; i < nn; i++) {
            cudaGraphNodeType ty;
            if (cudaGraphNodeGetType(nodes[i], &ty) != cudaSuccess || ty != cudaGraphNodeTypeKernel) continue;
            cudaKernelNodeParams kp;
            if (cudaGraphKernelNodeGetParams(nodes[i], &kp) != cudaSuccess) continue;
            cudaKernelNodeAttrValue v;
            memset(&v, 0, sizeof(v));
            // code stream: critical kernels highest, its old-term kernel lowest; the importance stream has slack (it only has
            // to stay ahead of the code stream): one level below the code stream's critical kernels, old terms lowest
            const int hi = is_code ? prio_hi : std::min(prio_lo, prio_hi + 2);
            v.priority = (kp.func == wf_old_kernel_ptr() || kp.func == wf_old2_kernel_ptr()) ? prio_lo : hi;
            cudaGraphKernelNodeSetAttribute(nodes[i], cudaKernelNodeAttributePriority, &v);
        }
        cudaGetLastError();
    }
    LIC360_CUDA(cudaGraphInstantiate(&n.graph, g, 0));
    cudaGraphDestroy(g);
    return LIC360_OK;
}

using clk = std::chrono::steady_clock;
static double ms_since(clk::time_point t0) { return std::chrono::duration<double, std::milli>(clk::now() - t0).count(); }

}  // namespace lic360

extern "C" {

static int ctx_alloc(NetDesc& n, int row_bytes, float fill, int prio_hi, int prio_lo) {
    n.row_bytes = row_bytes;
    LIC360_CUDA(cudaStreamCreateWithPriority(&n.stream, cudaStreamNonBlocking, prio_hi));
    LIC360_CUDA(cudaStreamCreateWithPriority(&n.side, cudaStreamNonBlocking, prio_lo));
    LIC360_CUDA(cudaEventCreateWithFlags(&n.ev_fork, cudaEventDisableTiming));
    LIC360_CUDA(cudaEventCreateWithFlags(&n.ev_join, cudaEventDisableTiming));
    for (int i = 0; i < 6; i++) LIC360_CUDA(cudaEventCreate(&n.ev_prof[i]));
    LIC360_CUDA(cudaMalloc(&n.ctr_dev, sizeof(int)));
    LIC360_CUDA(cudaMalloc(&n.done_dev, sizeof(int)));
    LIC360_CUDA(cudaMalloc(&n.arrived_dev, sizeof(int)));
    LIC360_CUDA(cudaMalloc(&n.sync_dev, sizeof(int)));
    LIC360_CUDA(cudaMalloc(&n.go_dev, sizeof(int)));
    LIC360_CUDA(cudaMalloc(&n.old_done_dev, sizeof(int)));
    LIC360_CUDA(cudaMalloc(&n.scat_done_dev, 4 * sizeof(int)));
    LIC360_CUDA(cudaHostAlloc(&n.flag_host, 64 * sizeof(int), cudaHostAllocMapped));
    LIC360_CUDA(cudaHostAlloc(&n.go_host, 64, cudaHostAllocMapped));
    *n.go_host = 0;
    n.coder = lic360_coder_create("", fill);
    return n.coder ? LIC360_OK : LIC360_ERR_ARG;
}

static int ctx_buffers(NetDesc& n) {
    LIC360_CUDA(cudaMalloc(&n.rows_dev, (size_t)n.total_rows * n.row_bytes));
    LIC360_CUDA(cudaHostAlloc(&n.rows_host, (size_t)n.total_rows * n.row_bytes, cudaHostAllocDefault));
    LIC360_CUDA(cudaHostAlloc(&n.rows_step_host, (size_t)n.max_len * n.row_bytes, cudaHostAllocMapped));
    LIC360_CUDA(cudaHostAlloc(&n.syms_host, (size_t)n.max_len * sizeof(float), cudaHostAllocMapped));
    n.bits_blocks = (n.G * n.H * n.W + BITS_THREADS - 1) / BITS_THREADS;
    LIC360_CUDA(cudaMalloc(&n.bits_partial_dev, (size_t)n.bits_blocks * sizeof(double)));
    return LIC360_OK;
}

static void ctx_free(NetDesc& n) {
    cudaFree(n.ctr_dev); cudaFree(n.done_dev); cudaFree(n.arrived_dev); cudaFree(n.sync_dev); cudaFree(n.go_dev); cudaFree(n.old_done_dev); cudaFree(n.scat_done_dev);
    cudaFreeHost(n.flag_host); cudaFreeHost(n.go_host);
    cudaFree(n.rows_dev); cudaFreeHost(n.rows_host); cudaFreeHost(n.rows_step_host); cudaFreeHost(n.syms_host);
    cudaFree(n.bits_partial_dev);
    if (n.ev_fork) cudaEventDestroy(n.ev_fork);
    if (n.ev_join) cudaEventDestroy(n.ev_join);
    for (int i = 0; i < 6; i++) if (n.ev_prof[i]) cudaEventDestroy(n.ev_prof[i]);
    if (n.side) cudaStreamDestroy(n.side);
    if (n.stream) cudaStreamDestroy(n.stream);
    lic360_coder_destroy(n.coder);
}

lic360_codec* lic360_codec_create(int device, int H, int W) {
    if (H <= 0 || W <= 0 || (H % 2) || (W % 2)) { set_error("codec: latent size must be positive and even"); return nullptr; }
    DeviceGuard guard(device);  // the caller's current device is restored on return
    if (guard.err != cudaSuccess) { set_error("codec: cudaSetDevice(%d) failed", device); return nullptr; }
    lic360_codec* c = new lic360_codec();
    c->device = device; c->H = H; c->W = W;
    net_init(c->code, 48, 4, 3, 3, H, W);
    net_init(c->imp, 1, 144, 49, 1, H / 2, W / 2);
    int prio_lo = 0, prio_hi = 0;
    cudaDeviceGetStreamPriorityRange(&prio_lo, &prio_hi);
    bool ok = ctx_alloc(c->code, 16, 3.5f, prio_hi, prio_lo) == LIC360_OK && ctx_alloc(c->imp, 128, 3.5f, prio_hi, prio_lo) == LIC360_OK;
    ok = ok && net_alloc(c->code) == LIC360_OK && net_alloc(c->imp) == LIC360_OK;
    ok = ok && ctx_buffers(c->code) == LIC360_OK && ctx_buffers(c->imp) == LIC360_OK;
    const bool pre_ok = ok;
    ok = ok && wf_init(c->code.wf, 48, 4, 3, 3, H, W, c->code.idx_dev, c->code.steps_dev, c->code.ctr_dev, c->code.nsteps, c->code.max_len) == LIC360_OK;
    ok = ok && wf_init(c->imp.wf, 1, 144, 49, 1, H / 2, W / 2, c->imp.idx_dev, c->imp.steps_dev, c->imp.ctr_dev, c->imp.nsteps, c->imp.max_len) == LIC360_OK;
    const bool wf_ok = ok || !pre_ok;
    if (ok) c->chain_cap = wf_chain_capacity(c->code.wf);
    ok = ok && cudaMalloc(&c->levels_dev, (size_t)(H / 2) * (W / 2) * sizeof(float)) == cudaSuccess;
    ok = ok && cudaMalloc(&c->mask192_dev, (size_t)192 * (H / 2) * (W / 2) * sizeof(float)) == cudaSuccess;
    ok = ok && cudaMalloc(&c->est_dev, sizeof(EstimateTotals)) == cudaSuccess;
    ok = ok && cudaHostAlloc(&c->est_host, sizeof(EstimateTotals), cudaHostAllocDefault) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&c->ev_est, cudaEventDisableTiming) == cudaSuccess;
    if (!ok) {
        if (wf_ok) set_error("codec: allocation failed (%s)", cudaGetErrorString(cudaGetLastError()));  // else: wf_init's message
        lic360_codec_destroy(c);
        return nullptr;
    }
    return c;
}

void lic360_codec_destroy(lic360_codec* c) {
    if (!c) return;
    DeviceGuard guard(c->device);
    net_free(c->code); net_free(c->imp);
    wf_free(c->code.wf); wf_free(c->imp.wf);
    ctx_free(c->code); ctx_free(c->imp);
    cudaFree(c->levels_dev); cudaFree(c->mask192_dev);
    cudaFree(c->est_dev); cudaFreeHost(c->est_host);
    if (c->ev_est) cudaEventDestroy(c->ev_est);
    delete c;
}

int lic360_codec_set_layer(lic360_codec* c, int stream_id, int layer, const float* w_dev, const float* bias_dev,
                           const float* slope_dev) {
    LIC360_CHECK_ARG(c && (stream_id == 0 || stream_id == 1) && layer >= 0 && layer < 12 && w_dev && bias_dev, "bad arguments");
    DeviceGuard guard(c->device);
    LIC360_CUDA(guard.err);
    NetDesc& n = stream_id == 0 ? c->code : c->imp;
    LIC360_CHECK_ARG(!n.act[layer] || slope_dev, "this layer has a PReLU: slope_dev must not be NULL");
    const size_t npf = lic360_cconv_wp_floats(n.nsets, n.Cin[layer], n.Cout[layer], n.G);
    const size_t nqf = lic360_cconv_wq_floats(n.nsets, n.Cin[layer], n.Cout[layer], n.G);
    const size_t nb = (size_t)n.nsets * n.Cout[layer];
    if (!n.wp[layer]) {
        LIC360_CUDA(cudaMalloc(&n.wp[layer], npf * sizeof(float)));
        LIC360_CUDA(cudaMalloc(&n.wq[layer], std::max(nqf, (size_t)4) * sizeof(float)));
        LIC360_CUDA(cudaMalloc(&n.bias[layer], nb * sizeof(float)));
        LIC360_CUDA(cudaMalloc(&n.slope[layer], nb * sizeof(float)));
    }
    int rc = lic360_cconv_pack(w_dev, n.wp[layer], n.wq[layer], n.nsets, n.Cin[layer], n.Cout[layer], n.G, 5, n.constrain[layer], n.stream);
    if (rc) return rc;
    LIC360_CUDA(cudaMemcpyAsync(n.bias[layer], bias_dev, nb * sizeof(float), cudaMemcpyDeviceToDevice, n.stream));
    if (slope_dev) LIC360_CUDA(cudaMemcpyAsync(n.slope[layer], slope_dev, nb * sizeof(float), cudaMemcpyDeviceToDevice, n.stream));
    LIC360_CUDA(cudaStreamSynchronize(n.stream));
    wf_set_layer(n.wf, layer, n.wp[layer], n.wq[layer], n.bias[layer], n.act[layer] ? n.slope[layer] : nullptr);
    if (n.graph) { cudaGraphExecDestroy(n.graph); n.graph = nullptr; }  // the graph holds the kernel parameters by value
    n.set[layer] = true;
    return LIC360_OK;
}

// The network part of an encode, shared with the rate estimate: the input frame of one stream from the caller's tensors and the
// stream's 12 layers, enqueued on its own CUDA stream; the outputs land in n.frame[12].
//   importance stream (lic360_demo.py:173-189): Scale(-1, 2/47) of the levels
//   code stream (lic360_demo.py:124-131): (code - 3.5) * mask, once for each of the three nets
static int run_encoder_net(lic360_codec* c, bool is_code, const float* code_dev, const float* mask_dev, const float* imp_dev) {
    NetDesc& n = is_code ? c->code : c->imp;
    if (is_code) {
        const int nel = n.G * n.H * n.W;
        prep_code_kernel<<<stream_grid(nel, 256), 256, 0, n.stream>>>(code_dev, mask_dev, n.frame[0], nel, 3.5f);
        LAUNCH_CHECK();
    } else {
        const int rc = lic360_scale(imp_dev, n.frame[0], n.H * n.W, -1.0f, (float)(2. / (48 - 1.)), n.stream);
        if (rc) return rc;
    }
    return run_ec_net(n, n.stream);
}

int lic360_codec_encode(lic360_codec* c, const float* code_dev, const float* mask_dev, const float* imp_dev) {
    LIC360_CHECK_ARG(c && code_dev && mask_dev && imp_dev, "bad arguments");
    DeviceGuard guard(c->device);
    LIC360_CUDA(guard.err);
    int rc = check_params(c->code);
    if (rc == LIC360_OK) rc = check_params(c->imp);
    if (rc) return rc;
    const auto t0 = clk::now();
    c->t_host_coder = 0; c->t_gpu_wait = 0; c->t_imp = 0; c->t_gpu_steps = 0; c->t_gpu_steps_imp = 0;
    // The two bitstreams are independent: both networks are enqueued on their own CUDA streams first, then the host
    // codes the (small) importance stream while the code-stream network is still running.
    // ---- importance stream: net -> rows of all symbols
    {
        NetDesc& n = c->imp;
        cudaStream_t s = n.stream;
        const int HW = n.H * n.W;
        rc = run_encoder_net(c, false, code_dev, mask_dev, imp_dev);
        if (rc) return rc;
        imp_rows_kernel<<<(HW + 127) / 128, 128, 0, s>>>(n.frame[12], imp_dev, n.idx_dev, n.steps_dev, n.ctr_dev, n.rows_dev, n.H, n.W, 1);
        LAUNCH_CHECK();
        LIC360_CUDA(cudaMemcpyAsync(n.rows_host, n.rows_dev, (size_t)n.total_rows * 128, cudaMemcpyDeviceToHost, s));
        c->t_gpu_steps_imp = ms_since(t0);  // host time spent enqueueing the importance-stream work
    }
    // ---- code stream (lic360_demo.py:124-141)
    {
        NetDesc& n = c->code;
        cudaStream_t s = n.stream;
        const auto tq0 = clk::now();
        const int nel = n.G * n.H * n.W;
        rc = run_encoder_net(c, true, code_dev, mask_dev, imp_dev);
        if (rc) return rc;
        gmm_rows_kernel<<<(nel + 127) / 128, 128, 0, s>>>(n.frame[12], code_dev, mask_dev, n.idx_dev, n.steps_dev, n.row_off_dev,
                                                          n.ctr_dev, n.rows_dev, n.G, n.H, n.W, 1, (float)(1. / sqrt(2.0)));
        LAUNCH_CHECK();
        LIC360_CUDA(cudaMemcpyAsync(n.rows_host, n.rows_dev, (size_t)n.total_rows * 16, cudaMemcpyDeviceToHost, s));
        c->t_gpu_steps = ms_since(tq0);  // host time spent enqueueing the code-stream work
    }
    {
        NetDesc& n = c->imp;
        auto tw = clk::now();
        LIC360_CUDA(cudaStreamSynchronize(n.stream));
        c->t_gpu_wait += ms_since(tw);
        auto th = clk::now();
        lic360_coder_start_encoder_mem(n.coder);
        rc = coder_encode_packed_imp(n.coder, n.rows_host, n.total_rows);
        if (rc) return rc;
        if (lic360_coder_finish_mem(n.coder) < 0) return LIC360_ERR_CODER;
        c->t_host_coder += ms_since(th);
        c->t_imp = ms_since(t0);
    }
    {
        NetDesc& n = c->code;
        auto tw = clk::now();
        LIC360_CUDA(cudaStreamSynchronize(n.stream));
        c->t_gpu_wait += ms_since(tw);
        auto th = clk::now();
        lic360_coder_start_encoder_mem(n.coder);
        rc = coder_encode_packed_gmm(n.coder, n.rows_host, n.total_rows);
        if (rc) return rc;
        if (lic360_coder_finish_mem(n.coder) < 0) return LIC360_ERR_CODER;
        c->t_host_coder += ms_since(th);
    }
    c->t_total = ms_since(t0);
    return LIC360_OK;
}

// the GPU work of an estimate on the codec's two streams; the code stream ends with the copy of both streams' results
static int enqueue_estimate(lic360_codec* c, const float* code_dev, const float* mask_dev, const float* imp_dev, float* code_bits_dev,
                            float* imp_bits_dev) {
    EstimateTotals* r = c->est_dev;
    {
        NetDesc& n = c->imp;
        cudaStream_t s = n.stream;
        LIC360_CUDA(cudaMemsetAsync(&r->err[1], 0xFF, sizeof(r->err[1]), s));
        int rc = run_encoder_net(c, false, code_dev, mask_dev, imp_dev);
        if (rc) return rc;
        imp_bits_kernel<<<n.bits_blocks, BITS_THREADS, 0, s>>>(n.frame[12], imp_dev, n.idx_dev, imp_bits_dev, n.bits_partial_dev,
                                                               &r->err[1], n.H, n.W);
        LAUNCH_CHECK();
        bits_sum_kernel<<<1, BITS_THREADS, 0, s>>>(n.bits_partial_dev, n.bits_blocks, &r->bits[1]);
        LAUNCH_CHECK();
        LIC360_CUDA(cudaEventRecord(c->ev_est, s));
    }
    {
        NetDesc& n = c->code;
        cudaStream_t s = n.stream;
        LIC360_CUDA(cudaMemsetAsync(&r->err[0], 0xFF, sizeof(r->err[0]), s));
        int rc = run_encoder_net(c, true, code_dev, mask_dev, imp_dev);
        if (rc) return rc;
        gmm_bits_kernel<<<n.bits_blocks, BITS_THREADS, 0, s>>>(n.frame[12], code_dev, mask_dev, n.idx_dev, n.steps_dev, n.row_off_dev,
                                                               code_bits_dev, n.bits_partial_dev, &r->err[0], n.G, n.H, n.W,
                                                               (float)(1. / sqrt(2.0)));
        LAUNCH_CHECK();
        bits_sum_kernel<<<1, BITS_THREADS, 0, s>>>(n.bits_partial_dev, n.bits_blocks, &r->bits[0]);
        LAUNCH_CHECK();
        LIC360_CUDA(cudaStreamWaitEvent(s, c->ev_est, 0));
        LIC360_CUDA(cudaMemcpyAsync(c->est_host, r, sizeof(EstimateTotals), cudaMemcpyDeviceToHost, s));
    }
    return LIC360_OK;
}

int lic360_codec_estimate(lic360_codec* c, const float* code_dev, const float* mask_dev, const float* imp_dev, float* code_bits_dev,
                          float* imp_bits_dev, double* bits_host) {
    LIC360_CHECK_ARG(c && code_dev && mask_dev && imp_dev && code_bits_dev && imp_bits_dev && bits_host, "bad arguments");
    DeviceGuard guard(c->device);
    LIC360_CUDA(guard.err);
    int rc = check_params(c->code);
    if (rc == LIC360_OK) rc = check_params(c->imp);
    if (rc) return rc;
    const auto t0 = clk::now();
    c->t_host_coder = 0; c->t_gpu_wait = 0; c->t_imp = 0; c->t_gpu_steps = 0; c->t_gpu_steps_imp = 0;
    rc = enqueue_estimate(c, code_dev, mask_dev, imp_dev, code_bits_dev, imp_bits_dev);
    // both streams are drained on every path: the caller may reuse the inputs and the maps as soon as the call returns
    const auto tw = clk::now();
    const cudaError_t e_imp = cudaStreamSynchronize(c->imp.stream);
    const cudaError_t e_code = cudaStreamSynchronize(c->code.stream);
    c->t_gpu_wait = ms_since(tw);
    c->t_total = ms_since(t0);
    if (rc) return rc;
    LIC360_CUDA(e_imp);
    LIC360_CUDA(e_code);
    // the errors encode reports, with its messages: the importance stream is coded (and checked) first
    const EstimateTotals& r = *c->est_host;
    if (r.err[1] != kNoError) {
        const unsigned s = (unsigned)r.err[1];
        if (s >= 49) set_error("coder: importance level %u out of range", s);
        else set_error("coder: symbol has zero frequency");
        return LIC360_ERR_CODER;
    }
    if (r.err[0] != kNoError) {
        const int row = (int)(r.err[0] >> 32);
        if ((unsigned)r.err[0] > 7) set_error("coder: symbol out of range in packed row %d", row);
        else set_error("coder: symbol has zero frequency (row %d)", row);
        return LIC360_ERR_CODER;
    }
    bits_host[0] = r.bits[0];
    bits_host[1] = r.bits[1];
    return LIC360_OK;
}

long lic360_codec_stream_size(lic360_codec* c, int stream_id) {
    long n = 0;
    coder_bytes(stream_id ? c->imp.coder : c->code.coder, &n);
    return n;
}

long lic360_codec_stream_copy(lic360_codec* c, int stream_id, uint8_t* out, long cap) {
    return lic360_coder_get_bytes(stream_id ? c->imp.coder : c->code.coder, out, cap);
}

// cuStreamWaitValue32 through the runtime's driver entry point lookup (no link-time dependency on libcuda)
typedef CUresult (*StreamWaitValue32Fn)(CUstream, CUdeviceptr, cuuint32_t, unsigned int);
static StreamWaitValue32Fn stream_wait_value_fn() {
    static StreamWaitValue32Fn fn = nullptr;
    static bool tried = false;
    if (!tried) {
        tried = true;
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (getenv("LIC360_WF_LAUNCH_AHEAD") &&
            cudaGetDriverEntryPoint("cuStreamWaitValue32", &p, cudaEnableDefault, &q) == cudaSuccess && q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<StreamWaitValue32Fn>(p);
        else
            cudaGetLastError();
    }
    return fn;
}

// releases a stream that may be parked on its go flag, whatever way decode_stream is left (a parked stream never drains)
struct GoRelease {
    int* go;
    ~GoRelease() { __atomic_store_n(go, 0x7fffffff, __ATOMIC_RELEASE); }
};

// wait for the rows of step p without synchronising the stream (a later kernel of the step graph may still be running)
static int wait_rows(lic360_codec* c, NetDesc& n, int p) {
    const int* f = n.flag_host;
    const auto t0 = clk::now();
    const int nf = n.nflags;
    bool dev_abort = false;
    // acquire loads: the rows the device wrote before raising a flag are read (non-atomically) by the coder right after
    auto ready = [&]() {
        for (int i = 0; i < nf; i++) {
            const int v = __atomic_load_n(f + i, __ATOMIC_ACQUIRE);
            if (v < 0) { dev_abort = true; return true; }
            if (v != p + 1) return false;
        }
        return true;
    };
    for (unsigned spins = 1; !ready(); spins++) {
        if ((spins & 0x3FFF) == 0) {
            if (c->abort_flag.load()) { set_error("codec: aborted (the other stream failed)"); return LIC360_ERR_CUDA; }
            const cudaError_t e = cudaStreamQuery(n.stream);
            if (e == cudaSuccess) {
                if (ready()) break;
                set_error("codec: step %d finished without producing its rows", p);
                return LIC360_ERR_CUDA;
            }
            if (e != cudaErrorNotReady) { set_error("codec: step %d failed -> %s", p, cudaGetErrorString(e)); return LIC360_ERR_CUDA; }
            if (ms_since(t0) > 20000.) { set_error("codec: step %d timed out", p); return LIC360_ERR_CUDA; }
        }
#if defined(__x86_64__)
        __builtin_ia32_pause();
#endif
        if ((spins & 0x7F) == 0) sched_yield();  // several ranks / images per box: do not starve the other polling threads
    }
    if (dev_abort) {
        set_error("codec: step %d: a chain cluster gave up waiting for the other nets' clusters (too many decodes in flight on this device?)", p);
        return LIC360_ERR_CUDA;
    }
    return LIC360_OK;
}

// called by the tagged row decoder every few thousand polls of a row that has not arrived: the same give-up conditions as wait_rows
struct StallCtx { lic360_codec* c; NetDesc* n; int p; clk::time_point t0; };
static int rows_stalled(void* vp) {
    StallCtx* x = static_cast<StallCtx*>(vp);
    NetDesc& n = *x->n;
    if (x->c->abort_flag.load()) { set_error("codec: aborted (the other stream failed)"); return LIC360_ERR_CUDA; }
    for (int i = 0; i < n.nflags; i++)
        if (__atomic_load_n(n.flag_host + i, __ATOMIC_ACQUIRE) < 0) {
            set_error("codec: step %d: a chain cluster gave up waiting for the other nets' clusters (too many decodes in flight on this device?)", x->p);
            return LIC360_ERR_CUDA;
        }
    const cudaError_t e = cudaStreamQuery(n.stream);
    if (e != cudaSuccess && e != cudaErrorNotReady) { set_error("codec: step %d failed -> %s", x->p, cudaGetErrorString(e)); return LIC360_ERR_CUDA; }
    if (ms_since(x->t0) > 20000.) { set_error("codec: step %d timed out waiting for its rows", x->p); return LIC360_ERR_CUDA; }
    sched_yield();
    return 0;
}

static int final_scatter(lic360_codec* c, NetDesc& n, bool is_code) {
    // scatter the symbols of the last step (the final TileInput of lic360_demo.py:236,285)
    const WfNetDev& w = n.wf.dev;
    const int tgrid = (n.max_len + 127) / 128;
    cudaStream_t s = n.stream;
    if (is_code)
        scatter_prev_kernel<<<tgrid, 128, 0, s>>>(n.syms_host, n.wf.fp[0], n.wf.fc[0], n.idx_dev, n.steps_dev, n.ctr_dev, n.arrived_dev, n.G, n.H, n.W,
                                                  w.D, w.HS, w.Dp, w.Hp, -3.5f, 1.0f, 3, nullptr);
    else
        scatter_prev_kernel<<<tgrid, 128, 0, s>>>(n.syms_host, n.wf.fp[0], n.wf.fc[0], n.idx_dev, n.steps_dev, n.ctr_dev, n.arrived_dev, 1, n.H, n.W,
                                                  w.D, w.HS, w.Dp, w.Hp, -1.0f, (float)(2. / (48 - 1.)), 1, c->levels_dev);
    LAUNCH_CHECK();
    return LIC360_OK;
}

// code stream: the importance levels step p needs are decoded (cells on importance diagonals <= min(p, H+W-2)/2), published by the
// importance loop running concurrently on another host thread and CUDA stream
static int wait_levels(lic360_codec* c, const NetDesc& n, int p) {
    const int need = std::min(p, n.H + n.W - 2) / 2 + 1;
    const auto t0 = clk::now();
    for (unsigned spins = 1; c->imp_ready.load(std::memory_order_acquire) < need; spins++) {
        if ((spins & 0xFFF) == 0 && (c->abort_flag.load() || ms_since(t0) > 20000.)) {
            set_error("codec: the importance stream did not deliver the levels the code stream needs");
            return LIC360_ERR_CODER;
        }
#if defined(__x86_64__)
        __builtin_ia32_pause();
#endif
        if ((spins & 0x1F) == 0) sched_yield();
    }
    return LIC360_OK;
}

// stops a persistent chain kernel at its next step boundary, whatever way the host loop is left (after a normal decode the kernel has
// already exited and the store is harmless)
struct PersistStop {  // every exit path: the chain kernel stops at its next step boundary
    int* go;
    ~PersistStop() { __atomic_store_n(go, WF_GO_ABORT, __ATOMIC_RELEASE); }
};

// Low-latency decode of the code stream (mode 2): ONE launch of the chain kernel walks all wavefront steps (wavefront.cu, WfPersist).
// Per step the host only (1) stores the go flag -- the symbols of the previous step are in mapped memory by then --, (2) enqueues an
// old-term kernel on the low-priority side stream, (3) decodes the rows as they arrive.  Against the graph replay per step this
// takes the graph launch, the scatter kernel and the chain kernel's prologue off the critical path; the price is that the chain's 24
// SMs stay occupied for the whole decode (fine for one image at a time, the wrong trade with several in flight).
static int decode_stream_persistent(lic360_codec* c, NetDesc& n) {
    cudaStream_t s = n.stream, side = n.side;
    for (int i = 0; i < 64; i++) n.flag_host[i] = 0;
    memset(n.rows_step_host, 0, (size_t)n.max_len * n.row_bytes);
    memset(n.syms_host, 0, (size_t)n.max_len * sizeof(float));  // tag 0 = not published
    __atomic_store_n(n.go_host, -1, __ATOMIC_RELEASE);
    PersistStop stop{n.go_host};
    n.t_host_coder = 0; n.t_gpu_wait = 0;
    const bool trace_file = getenv("LIC360_WF_TRACE_FILE") != nullptr;
    n.step_wait_us.clear(); n.step_decode_us.clear(); n.step_levels_us.clear();
    for (int i = 0; i < 5; i++) n.t_kernel[i] = 0;
    LIC360_CUDA(wf_clear(n.wf, s));
    LIC360_CUDA(cudaMemsetAsync(n.ctr_dev, 0xFF, sizeof(int), s));
    LIC360_CUDA(cudaMemsetAsync(n.done_dev, 0, sizeof(int), s));
    LIC360_CUDA(cudaMemsetAsync(n.arrived_dev, 0, sizeof(int), s));
    LIC360_CUDA(cudaMemsetAsync(n.sync_dev, 0, sizeof(int), s));
    LIC360_CUDA(cudaMemsetAsync(n.go_dev, 0xFF, sizeof(int), s));
    LIC360_CUDA(cudaMemsetAsync(n.old_done_dev, 0, sizeof(int), s));
    LIC360_CUDA(cudaMemsetAsync(n.scat_done_dev, 0, 4 * sizeof(int), s));
    LIC360_CUDA(cudaEventRecord(n.ev_fork, s));
    LIC360_CUDA(cudaStreamWaitEvent(side, n.ev_fork, 0));
    LIC360_CUDA(wf_launch_old(n.wf, 0, side, false, 0, n.old_done_dev, n.scat_done_dev));  // old terms of step 0 (all zero; keeps the protocol uniform)
    WfRows rows;
    memset(&rows, 0, sizeof(rows));
    rows.rows = n.rows_step_host; rows.levels = c->levels_dev; rows.done = n.done_dev; rows.flag = n.flag_host;
    rows.sync = n.sync_dev; rows.s2 = (float)(1. / sqrt(2.0)); rows.enabled = 1; rows.rtail = 1; rows.tagged = 1;
    n.tagged = true;
    n.nflags = n.wf.dev.nsets * n.wf.cluster;
    if (n.nflags > 64) { set_error("codec: %d chain CTAs exceed the 64 host flags", n.nflags); return LIC360_ERR_ARG; }
    WfPersist ps;
    memset(&ps, 0, sizeof(ps));
    ps.syms = n.syms_host; ps.go_host = n.go_host; ps.go_dev = n.go_dev; ps.old_done = n.old_done_dev; ps.ctr = n.ctr_dev; ps.scat_done = n.scat_done_dev;
    ps.bias = -3.5f; ps.scale = 1.0f;
    LIC360_CUDA(wf_launch_chain(n.wf, s, &rows, &ps));
    int rc = LIC360_OK;
    for (int p = 0; p < n.nsteps; p++) {
        auto tw = clk::now();
        rc = wait_levels(c, n, p);
        if (rc) return rc;
        if (trace_file) n.step_levels_us.push_back((float)(ms_since(tw) * 1e3));
        __atomic_store_n(n.go_host, p, __ATOMIC_RELEASE);  // step p may run: the symbols of step p - 1 are in syms_host
        // old terms of step p + 1: they read wavefronts <= p - 1, complete now; enqueued behind the go so that the launch costs no time on
        // the critical path (the GPU is busy with step p for the next ~60 us)
        if (p + 1 < n.nsteps) LIC360_CUDA(wf_launch_old(n.wf, 0, side, false, p + 1, n.old_done_dev, n.scat_done_dev));
        StallCtx sc{c, &n, p, clk::now()};
        for (unsigned spins = 1; ((__atomic_load_n(n.rows_step_host + 7, __ATOMIC_ACQUIRE) >> 4) & 15) != (unsigned)(p % 15 + 1); spins++) {
#if defined(__x86_64__)
            __builtin_ia32_pause();
#endif
            if ((spins & 0x3FFF) == 0) { rc = rows_stalled(&sc); if (rc) return rc; }
        }
        n.t_gpu_wait += ms_since(tw);
        if (trace_file) n.step_wait_us.push_back((float)(ms_since(tw) * 1e3));
        auto th = clk::now();
        rc = coder_decode_packed_gmm_tagged(n.coder, n.rows_step_host, n.steps[p].len, n.syms_host, p % 15 + 1, rows_stalled, &sc,
                                            p + 1 < n.nsteps ? (unsigned)(p % 15 + 1) : 0u);  // symbol words tagged too: the chain kernel polls
                                            // them one by one (not the last step's: the final scatter reads plain floats)
        n.t_host_coder += ms_since(th);
        if (trace_file) n.step_decode_us.push_back((float)(ms_since(th) * 1e3));
        if (rc) return rc;
    }
    LIC360_CUDA(cudaEventRecord(n.ev_join, side));
    LIC360_CUDA(cudaStreamWaitEvent(s, n.ev_join, 0));
    return final_scatter(c, n, true);  // behind the chain kernel in stream order; the device step counter is nsteps - 1
}

// The wavefront loop of one bitstream.  is_code: before step p the importance levels of every 2x2 cell the slab touches
// must be decoded (cells on importance diagonals <= min(p, H+W-2)/2): the loop waits on c->imp_ready, which the
// importance loop (running concurrently on another host thread and CUDA stream) publishes.
static bool persistent_ok(const lic360_codec* c, const NetDesc& n) {
    return c->mode == 2 && n.wf.chain4 && n.wf.r0_inline && n.wf.old2 && !getenv("LIC360_WF_ROWS_KERNEL") && !getenv("LIC360_WF_PREV_KERNEL");
}

static int decode_stream(lic360_codec* c, NetDesc& n, bool is_code) {
    if (is_code && persistent_ok(c, n)) return decode_stream_persistent(c, n);
    cudaStream_t s = n.stream;
    int rc = LIC360_OK;
    for (int i = 0; i < 64; i++) n.flag_host[i] = 0;
    memset(n.rows_step_host, 0, (size_t)n.max_len * n.row_bytes);  // publication tags of a previous decode must not match step 0
    // Launch-ahead (experiment, LIC360_WF_LAUNCH_AHEAD=1; measured ~1 ms SLOWER per 512x1024 decode than launching each step's
    // graph when its symbols are ready, so it is off by default): while the GPU works on step p the host already enqueues
    // [wait until *go >= p+1][graph of step p+1]; once the symbols of step p are decoded (and, for the code stream, the importance
    // levels step p+1 needs are there) one store to the mapped flag lets the stream's front end start the step.  The wait is a
    // stream memory operation (no kernel spins); GoRelease un-parks the stream on every exit path.
    StreamWaitValue32Fn wait_value = c->mode != 1 ? stream_wait_value_fn() : nullptr;
    CUdeviceptr go_dev = 0;
    if (wait_value) {
        void* dp = nullptr;
        if (cudaHostGetDevicePointer(&dp, n.go_host, 0) != cudaSuccess) { cudaGetLastError(); wait_value = nullptr; }
        go_dev = (CUdeviceptr)(uintptr_t)dp;
    }
    __atomic_store_n(n.go_host, 0, __ATOMIC_RELEASE);
    GoRelease go_release{n.go_host};
    n.t_host_coder = 0; n.t_gpu_wait = 0;
    const bool trace_file = getenv("LIC360_WF_TRACE_FILE") != nullptr;
    n.step_wait_us.clear(); n.step_decode_us.clear(); n.step_levels_us.clear();
    LIC360_CUDA(wf_clear(n.wf, s));
    LIC360_CUDA(cudaMemsetAsync(n.ctr_dev, 0xFF, sizeof(int), s));  // -1: the scatter kernel of step p makes it p
    LIC360_CUDA(cudaMemsetAsync(n.done_dev, 0, sizeof(int), s));
    LIC360_CUDA(cudaMemsetAsync(n.arrived_dev, 0, sizeof(int), s));
    LIC360_CUDA(cudaMemsetAsync(n.sync_dev, 0, sizeof(int), s));
    LIC360_CUDA(wf_launch_old(n.wf, 1, s));  // old terms of step 0 = counter (-1) + 1 (all zero, but it keeps the schedule uniform)
    if (getenv("LIC360_DEBUG_SYNC")) LIC360_CUDA(cudaStreamSynchronize(s));
    for (int i = 0; i < 5; i++) n.t_kernel[i] = 0;
    bool ahead = false;  // the graph of the current step is already enqueued (behind its go flag)
    for (int p = 0; p < n.nsteps; p++) {
        auto tw = clk::now();
        if (c->mode != 1) {
            if (!ahead) {
                if (is_code) { rc = wait_levels(c, n, p); if (rc) return rc; }
                if (trace_file && is_code) n.step_levels_us.push_back((float)(ms_since(tw) * 1e3));
                LIC360_CUDA(cudaGraphLaunch(n.graph, s));
                g_launches += n.graph_nodes;
            }
            ahead = false;
            if (wait_value && p + 1 < n.nsteps) {
                if (wait_value(s, go_dev, (cuuint32_t)(p + 1), 0 /* CU_STREAM_WAIT_VALUE_GEQ */) == CUDA_SUCCESS) {
                    LIC360_CUDA(cudaGraphLaunch(n.graph, s));
                    g_launches += n.graph_nodes;
                    ahead = true;
                } else {
                    wait_value = nullptr;  // not supported here: plain launch per step
                }
            }
            if (!n.tagged) {
                rc = wait_rows(c, n, p);
                if (rc) return rc;
            }
        } else {
            if (is_code) { rc = wait_levels(c, n, p); if (rc) return rc; }
            rc = launch_step(c, n, is_code, s, s, n.ev_prof);
            if (rc) return rc;
            LIC360_CUDA(cudaStreamSynchronize(s));
            float ms[5];
            for (int i = 0; i < 5; i++) cudaEventElapsedTime(&ms[i], n.ev_prof[i], n.ev_prof[i + 1]);
            n.t_kernel[0] += ms[4]; n.t_kernel[1] += ms[1]; n.t_kernel[2] += ms[2]; n.t_kernel[3] += ms[0] + ms[3]; n.t_kernel[4] += 1;
        }
        n.t_gpu_wait += ms_since(tw);
        if (!is_code) c->imp_ready.store(p, std::memory_order_release);  // the scatter of this step wrote diagonal p-1
        auto th = clk::now();
        const int len = n.steps[p].len;
        if (is_code && n.tagged) {
            StallCtx sc{c, &n, p, clk::now()};
            // time until the first row is there = waiting for the GPU; the rest of the call decodes while the later rows arrive
            for (unsigned spins = 1; ((__atomic_load_n(n.rows_step_host + 7, __ATOMIC_ACQUIRE) >> 4) & 15) != (unsigned)(p % 15 + 1); spins++) {
#if defined(__x86_64__)
                __builtin_ia32_pause();
#endif
                if ((spins & 0x3FFF) == 0) { rc = rows_stalled(&sc); if (rc) return rc; }
            }
            n.t_gpu_wait += ms_since(th);
            if (trace_file) n.step_wait_us.push_back((float)(ms_since(tw) * 1e3));
            th = clk::now();
            rc = coder_decode_packed_gmm_tagged(n.coder, n.rows_step_host, len, n.syms_host, p % 15 + 1, rows_stalled, &sc);
        } else {
            rc = is_code ? coder_decode_packed_gmm(n.coder, n.rows_step_host, len, n.syms_host)
                         : coder_decode_packed_imp(n.coder, n.rows_step_host, len, n.syms_host);
        }
        n.t_host_coder += ms_since(th);
        if (trace_file && is_code && n.tagged) n.step_decode_us.push_back((float)(ms_since(th) * 1e3));
        if (rc) return rc;
        if (ahead) {
            if (is_code) { rc = wait_levels(c, n, p + 1); if (rc) return rc; }
            __atomic_store_n(n.go_host, p + 1, __ATOMIC_RELEASE);  // symbols of step p are in syms_host: step p+1 may run
        }
    }
    rc = final_scatter(c, n, is_code);
    if (rc) return rc;
    if (!is_code) {
        LIC360_CUDA(cudaStreamSynchronize(s));
        c->imp_ready.store(n.nsteps + 1, std::memory_order_release);  // every diagonal is in levels_dev
    }
    return LIC360_OK;
}

int lic360_codec_decode(lic360_codec* c, const uint8_t* imp_bytes, long n_imp, const uint8_t* code_bytes, long n_code,
                        float* code_out_dev, float* mask_out_dev) {
    LIC360_CHECK_ARG(c && imp_bytes && code_bytes && code_out_dev && mask_out_dev && n_imp >= 0 && n_code >= 0, "bad arguments");
    DeviceGuard guard(c->device);
    LIC360_CUDA(guard.err);
    int rc = check_params(c->code);
    if (rc == LIC360_OK) rc = check_params(c->imp);
    if (rc) return rc;
    const auto t0 = clk::now();
    c->t_host_coder = 0; c->t_gpu_wait = 0; c->t_gpu_steps = 0; c->t_gpu_steps_imp = 0; c->t_imp = 0;
    c->imp_ready.store(0);
    c->abort_flag.store(0);
    // debug timeline of the code stream (LIC360_WF_TRACE=1): %globaltimer stamps per step, summarised on stderr
    unsigned long long* trace_dev = nullptr;
    const int tr_sel = getenv("LIC360_WF_TRACE") && atoi(getenv("LIC360_WF_TRACE")) == 2 ? 1 : 0;  // 2: trace the importance stream
    const NetDesc& tr_net = tr_sel ? c->imp : c->code;
    const int tr_steps = tr_net.nsteps + 2;
    if (getenv("LIC360_WF_TRACE")) {
        std::vector<unsigned long long> init((size_t)tr_steps * WF_TR_SLOTS + 64, 0ull);  // + per-layer phase sums of the G = 1 chain
        for (int p = 0; p < tr_steps; p++)
            for (int k = 0; k < WF_TR_SLOTS; k++)
                init[(size_t)p * WF_TR_SLOTS + k] = (k == WF_TR_CHAIN1 || k == WF_TR_ROWS1 || k == WF_TR_OLD1 || k == WF_TR_TAIL1) ? 0ull : ~0ull;
        LIC360_CUDA(cudaMalloc(&trace_dev, init.size() * 8));
        LIC360_CUDA(cudaMemcpy(trace_dev, init.data(), init.size() * 8, cudaMemcpyHostToDevice));
        wf_trace_set(trace_dev, tr_sel);
        codec_trace_set(trace_dev, tr_sel);
    }
    // Admission first: a decode queues here when the device already runs as many decodes as it can hold, and a low-latency decode takes
    // the device for itself.  Everything below -- graph capture and instantiation included, which may allocate and therefore wait for the
    // device -- runs inside the slot: a thread that blocks in the driver while ANOTHER decode's persistent kernel waits for its host
    // would stall that decode's importance-stream launches (observed as a 20 s "levels" time-out under a 7-thread stress).
    std::unique_ptr<ChainSlot> slot;
    if (c->mode != 1) slot.reset(new ChainSlot(c->device, c->chain_cap, persistent_ok(c, c->code) ? c->chain_cap : 1));
    if (c->mode != 1) {  // both step graphs exist before the second host thread starts (the persistent code stream needs none)
        rc = build_step_graph(c, c->imp, false);
        if (rc == LIC360_OK && !persistent_ok(c, c->code)) rc = build_step_graph(c, c->code, true);
        if (rc) return rc;
    }
    lic360_coder_start_decoder_mem(c->imp.coder, imp_bytes, n_imp);
    lic360_coder_start_decoder_mem(c->code.coder, code_bytes, n_code);
    // ---- importance stream (lic360_demo.py:272-290) and code stream (:220-238), concurrently in the pipelined mode: the
    // code stream only reads importance levels that are already decoded (decode_stream).  Serialized in profile mode.
    int rc_imp = LIC360_OK;
    c->imp.err[0] = 0;
    auto imp_loop = [&]() {
        cudaSetDevice(c->device);
        rc_imp = decode_stream(c, c->imp, false);
        if (rc_imp) {
            snprintf(c->imp.err, sizeof(c->imp.err), "%s", lic360_last_error());
            c->abort_flag.store(1);
        }
        c->t_imp = ms_since(t0);
    };
    if (c->mode != 1) {
        c->imp_worker.submit(imp_loop);
        rc = decode_stream(c, c->code, true);
        std::string code_err;
        if (rc) { code_err = lic360_last_error(); c->abort_flag.store(1); }
        c->imp_worker.wait();
        // both failed: the stream that failed FIRST carries the cause, the other one only reports the abort it was told about
        if (rc && rc_imp && strstr(c->imp.err, "aborted (the other stream failed)")) {
            set_error("%s", code_err.c_str());
            cudaStreamSynchronize(c->code.stream); cudaStreamSynchronize(c->imp.stream);
            return rc;
        }
    } else {
        imp_loop();
        if (rc_imp == LIC360_OK) rc = decode_stream(c, c->code, true);
    }
    if (rc_imp) { set_error("%s", c->imp.err); cudaStreamSynchronize(c->code.stream); cudaStreamSynchronize(c->imp.stream); return rc_imp; }
    if (rc) { cudaStreamSynchronize(c->code.stream); cudaStreamSynchronize(c->imp.stream); return rc; }
    // ---- outputs: mask_up = Dtow(Imp2mask(levels)) (lic360_demo.py:285-290), code = frame + 3.5 * mask (:236-237)
    cudaStream_t s = c->code.stream;
    rc = lic360_imp2mask(c->levels_dev, c->mask192_dev, 1, 192, c->imp.H, c->imp.W, 48, s);
    if (rc) return rc;
    rc = lic360_dtow(c->mask192_dev, mask_out_dev, 1, 192, c->imp.H, c->imp.W, 2, 1, s);
    if (rc) return rc;
    const int nel = 48 * c->H * c->W;
    finish_code_kernel<<<stream_grid(nel, 256), 256, 0, s>>>(c->code.wf.fc[0], mask_out_dev, code_out_dev, 48, c->H, c->W,
                                                             c->code.wf.dev.Dp, c->code.wf.dev.Hp, 3.5f);
    LAUNCH_CHECK();
    LIC360_CUDA(cudaStreamSynchronize(s));
    if (trace_dev) {
        std::vector<unsigned long long> tr((size_t)tr_steps * WF_TR_SLOTS + 64);
        cudaMemcpy(tr.data(), trace_dev, tr.size() * 8, cudaMemcpyDeviceToHost);
        wf_trace_set(nullptr, 0);
        codec_trace_set(nullptr, 0);
        cudaFree(trace_dev);
        const char* names[WF_TR_SLOTS] = {"scatter start", "prev start", "chain start", "chain end", "rows start", "rows flag", "old start", "old end", "R tail start", "R tail end"};
        for (int w0 = 0; w0 < 2; w0++) {  // two windows: while the importance stream still runs / after it finished
            const int pa = tr_sel ? (w0 == 0 ? 10 : 50) : (w0 == 0 ? 20 : 140), pb = tr_sel ? (w0 == 0 ? 45 : 90) : (w0 == 0 ? 80 : 220);
            double acc[WF_TR_SLOTS] = {0}, period = 0;
            int cnt = 0;
            for (int p = pa; p < pb && p + 1 < tr_net.nsteps; p++) {
                const unsigned long long* r = &tr[(size_t)p * WF_TR_SLOTS];
                for (int k = 0; k < WF_TR_SLOTS; k++) acc[k] += (double)(long long)(r[k] - r[0]) * 1e-3;
                period += (double)(long long)(tr[(size_t)(p + 1) * WF_TR_SLOTS] - r[0]) * 1e-3;
                cnt++;
            }
            fprintf(stderr, "lic360 trace, %s-stream steps %d..%d: period %.1f us;", tr_sel ? "importance" : "code", pa, pb, period / cnt);
            for (int k = 1; k < WF_TR_SLOTS; k++) fprintf(stderr, " %s +%.1f;", names[k], acc[k] / cnt);
            fprintf(stderr, "\n");
        }
        if (const char* fn = getenv("LIC360_WF_TRACE_FILE")) {  // per-step dump: step, slab length, us relative to the step's slot 0, period
            if (FILE* f = fopen(fn, "w")) {
                fprintf(f, "step,len,prev_start,chain_start,chain_end,rows_start,rows_last,old_start,old_end,tail_start,tail_end,period,host_wait_us,host_decode_us,levels_wait_us\n");
                for (int p = 0; p + 1 < tr_net.nsteps; p++) {
                    const unsigned long long* r = &tr[(size_t)p * WF_TR_SLOTS];
                    fprintf(f, "%d,%d", p, tr_net.steps[p].len);
                    for (int k = 1; k < WF_TR_SLOTS; k++) fprintf(f, ",%.1f", (double)(long long)(r[k] - r[0]) * 1e-3);
                    fprintf(f, ",%.1f", (double)(long long)(tr[(size_t)(p + 1) * WF_TR_SLOTS] - r[0]) * 1e-3);
                    fprintf(f, ",%.1f,%.1f,%.1f\n", (size_t)p < tr_net.step_wait_us.size() ? tr_net.step_wait_us[p] : 0.f,
                            (size_t)p < tr_net.step_decode_us.size() ? tr_net.step_decode_us[p] : 0.f,
                            (size_t)p < tr_net.step_levels_us.size() ? tr_net.step_levels_us[p] : 0.f);
                }
                fclose(f);
            }
        }
        if (!tr_sel) {
            fprintf(stderr, "lic360 trace, code-stream chain, CTA 0 thread 0, us per layer [weight staging issue | item: 25 loads, 100 FMA4, stores | prefetch issue + weights landed | cluster barrier]:");
            for (int l = 0; l < 12; l++) {
                fprintf(stderr, " L%d", l);
                for (int ph = 0; ph < 4; ph++) fprintf(stderr, "%c%.2f", ph ? '|' : ' ', (double)tr[(size_t)tr_steps * WF_TR_SLOTS + l * 4 + ph] * 1e-3 / tr_net.nsteps);
            }
            fprintf(stderr, "\n");
        }
        if (tr_sel) {
            fprintf(stderr, "lic360 trace, G=1 chain, CTA 0, us per layer [weight staging | Q product | epilogue + DSMEM stores | prefetch + cluster barrier]:");
            for (int l = 0; l < 12; l++) {
                fprintf(stderr, " L%d", l);
                for (int ph = 0; ph < 4; ph++) fprintf(stderr, "%c%.2f", ph ? '|' : ' ', (double)tr[(size_t)tr_steps * WF_TR_SLOTS + l * 4 + ph] * 1e-3 / tr_net.nsteps);
            }
            fprintf(stderr, "\n");
        }
    }
    c->t_host_coder = c->code.t_host_coder + c->imp.t_host_coder;
    c->t_gpu_wait = c->code.t_gpu_wait;
    c->t_total = ms_since(t0);
    return LIC360_OK;
}

int lic360_codec_last_timing(lic360_codec* c, double* out, int n) {
    const double v[6] = {c->t_total, c->t_host_coder, c->t_gpu_wait, c->t_imp, c->t_gpu_steps, c->t_gpu_steps_imp};
    for (int i = 0; i < n && i < 6; i++) out[i] = v[i];
    return LIC360_OK;
}

int lic360_codec_set_mode(lic360_codec* c, int mode) {
    LIC360_CHECK_ARG(c && (mode == 0 || mode == 1 || mode == 2),
                     "mode must be 0 (pipelined graph replay per step), 1 (serialized, per-kernel timing) or 2 (low latency: persistent code-stream chain)");
    c->mode = mode;
    return LIC360_OK;
}

int lic360_codec_kernel_times(lic360_codec* c, int stream_id, double* out, int n) {
    LIC360_CHECK_ARG(c && out, "bad arguments");
    const NetDesc& d = stream_id == 0 ? c->code : c->imp;
    for (int i = 0; i < n && i < 5; i++) out[i] = d.t_kernel[i];
    return LIC360_OK;
}

}  // extern "C"
