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
#include <deque>
#include <functional>
#include <cstring>
#include <memory>
#include <mutex>
#include <string>
#include <sched.h>
#include <system_error>
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
    float* frame[13] = {nullptr};  // encoder: frame[0] = network input, frame[i+1] = output of layer i, for lic360_codec::batch_cap latents
    size_t frame_floats[13];       // floats of one latent
    int32_t* idx_dev = nullptr;
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
    int* flag_host = nullptr;           // mapped pinned, importance stream: step + 1 once the rows of a step are in rows_step_host;
                                        // code stream: one per chain CTA, negative when that CTA gave up waiting for the other clusters
    int nflags = 1;                     // code stream: chain CTAs, each with its own host flag
    int* go_host = nullptr;             // mapped pinned: the stream may run step p once this is >= p (persistent decode)
    int* go_dev = nullptr;              // persistent decode: CTA 0's republished go / abort decision
    int* old_done_dev = nullptr;        // persistent decode: old-term sums of steps < this are complete
    int* scat_done_dev = nullptr;       // persistent decode, one per net: symbols of steps < this are in the net's input frame
    uint16_t* rows_dev = nullptr;       // encode: all rows of the stream
    uint16_t* rows_host = nullptr;      // pinned
    uint16_t* rows_step_host = nullptr; // mapped pinned: rows of one decode step
    float* syms_host = nullptr;         // mapped pinned: decoded symbols of one step
    std::vector<float> step_wait_us, step_decode_us, step_levels_us;  // debug timeline (LIC360_WF_TRACE_FILE): host time per step waiting for rows / decoding
    int row_bytes = 16;                 // packed row size (16 B code stream, 128 B importance stream)
    double t_host_coder = 0, t_gpu_wait = 0;
    lic360_coder* coder = nullptr;
    double* bits_partial_dev = nullptr; // estimate: one partial sum per block of the bits kernel and latent
    int* count_partial_dev = nullptr;   // estimate: coded symbols per block of the bits kernel and latent
    int bits_blocks = 0;                // blocks of the bits kernel per latent
};

constexpr int BITS_THREADS = 256;  // block size of the estimate's bits and sum kernels

// device-side results of an estimate of K latents, copied back with one cudaMemcpyAsync: the totals, the first-error keys and the
// coded-symbol counts, each indexed [stream_id * K + k] (stream_id 0 code, 1 importance)
struct EstimateTotals {
    double* bits;
    unsigned long long* err;
    long long* count;
};
inline size_t estimate_bytes(int K) { return (size_t)2 * K * (sizeof(double) + sizeof(unsigned long long) + sizeof(long long)); }
inline EstimateTotals estimate_totals(void* base, int K) {
    EstimateTotals r;
    r.bits = static_cast<double*>(base);
    r.err = reinterpret_cast<unsigned long long*>(r.bits + 2 * K);
    r.count = reinterpret_cast<long long*>(r.err + 2 * K);
    return r;
}
// a batch of K latents runs the code network with 3K images (grid.z of the conv kernels, at most 65535) and indexes its input frame
// with int
constexpr int kMaxBatch = 65535 / 3;

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

// the host coding of a batch encode: persistent workers per codec (not a std::thread per call), each with its own coder, started
// on demand and joined when the codec is destroyed.  Jobs start in the order they were posted.
constexpr int kMaxCoderWorkers = 16;
struct CoderPool {
    std::vector<std::thread> th;
    std::vector<lic360_coder*> coders;  // coders[i] belongs to th[i]
    std::mutex m;
    std::condition_variable cv, idle;
    std::deque<std::function<void(lic360_coder*)>> jobs;
    int running = 0;
    bool quit = false;
    void loop(lic360_coder* coder) {
        std::unique_lock<std::mutex> lk(m);
        for (;;) {
            cv.wait(lk, [&] { return quit || !jobs.empty(); });
            if (quit) return;
            std::function<void(lic360_coder*)> j = std::move(jobs.front());
            jobs.pop_front();
            running++;
            lk.unlock();
            j(coder);
            lk.lock();
            if (--running == 0 && jobs.empty()) idle.notify_all();
        }
    }
    // at least n workers, or as many as the system lets us start; returns the number of workers
    int grow(int n) {
        while ((int)th.size() < n) {
            lic360_coder* coder = lic360_coder_create("", 3.5f);
            try {
                th.emplace_back([this, coder] { loop(coder); });
            } catch (const std::system_error&) {
                lic360_coder_destroy(coder);
                break;
            }
            coders.push_back(coder);
        }
        return (int)th.size();
    }
    void post(std::function<void(lic360_coder*)> j) {
        { std::lock_guard<std::mutex> lk(m); jobs.push_back(std::move(j)); }
        cv.notify_one();
    }
    void wait() {  // until every posted job has finished
        std::unique_lock<std::mutex> lk(m);
        idle.wait(lk, [&] { return jobs.empty() && running == 0; });
    }
    ~CoderPool() {
        { std::lock_guard<std::mutex> lk(m); quit = true; }
        cv.notify_all();
        for (std::thread& t : th) t.join();
        for (lic360_coder* coder : coders) lic360_coder_destroy(coder);
    }
};

// one stream of a batch encode: its bytes, or the status and message of the coder that refused it
struct EncodedStream {
    std::vector<uint8_t> bytes;
    int rc = 0;
    std::string err;
};
}  // namespace lic360

struct lic360_codec {
    int device = 0, H = 0, W = 0;
    int chain_cap = 1;                  // concurrent decodes the device can hold (wf_chain_capacity)
    lic360::StreamWorker imp_worker;
    lic360::CoderPool coder_pool;       // encode_batch: codes the 2K streams
    int mode = 0;                       // 0: pipelined graph replay, 1: serialized launches with per-kernel event timing
    NetDesc code, imp;
    float* levels_dev = nullptr;        // decoded importance levels (1,1,H/2,W/2), filled diagonal by diagonal
    float* mask192_dev = nullptr;       // scratch: Imp2mask output
    std::atomic<int> imp_ready{0};      // decode: importance levels of diagonals < imp_ready are in levels_dev
    std::atomic<int> abort_flag{0};     // decode: one of the two stream loops failed
    int batch_cap = 0;                  // latents the encoder frames, the bits partials and est_dev / est_host hold (grown on demand)
    void* est_dev = nullptr;            // estimate: totals, error keys and counts of both streams (EstimateTotals layout)
    void* est_host = nullptr;           // pinned copy of est_dev
    cudaEvent_t ev_est = nullptr;                // estimate: the importance stream's results are in est_dev
    int2* cand_dev = nullptr;           // estimate_ / encode_candidates: the (source latent, offset) table, batch_cap entries
    float* cand_levels_dev = nullptr;   // estimate_ / encode_candidates: the candidates' levels (batch_cap,1,H/2,W/2), the importance net's input
    int rows_cap = 1;                   // latents the encoder's row buffers (rows_dev / rows_host of both streams) hold (grown on demand)
    int enc_k = 0;                      // latents of the last successful encode / encode_batch (0 after a failure or a decode)
    std::vector<lic360::EncodedStream> enc_out = std::vector<lic360::EncodedStream>(2);  // [2k + stream_id]: the streams of the last encode (empty after a failed one)
    double t_host_coder = 0, t_total = 0, t_gpu_wait = 0, t_imp = 0, t_gpu_steps = 0, t_gpu_steps_imp = 0;
};

namespace lic360 {

WF_TRACE_DECL
static void codec_trace_set(unsigned long long* buf, int sel) {
    cudaMemcpyToSymbol(g_wf_trace, &buf, sizeof(buf));
    cudaMemcpyToSymbol(g_wf_trace_sel, &sel, sizeof(sel));
}

// Debug timeline of a decode (LIC360_WF_TRACE=1: the code stream, 2: the importance stream): %globaltimer stamps in the WF_TR_SLOTS
// slots of every step, then the per-layer phase sums of the traced stream's chain kernel
struct DecodeTrace {
    unsigned long long* dev = nullptr;  // nullptr: no trace
    int sel = 0;                        // 0: code stream, 1: importance stream
    int steps = 0;                      // steps with slots
};

static int decode_trace_begin(lic360_codec* c, DecodeTrace& t) {
    const char* env = getenv("LIC360_WF_TRACE");
    if (!env) return LIC360_OK;
    t.sel = atoi(env) == 2 ? 1 : 0;
    t.steps = (t.sel ? c->imp : c->code).nsteps + 2;
    std::vector<unsigned long long> init((size_t)t.steps * WF_TR_SLOTS + 64, 0ull);  // + per-layer phase sums of the chain
    for (int p = 0; p < t.steps; p++)
        for (int k = 0; k < WF_TR_SLOTS; k++)
            init[(size_t)p * WF_TR_SLOTS + k] = (k == WF_TR_CHAIN1 || k == WF_TR_ROWS1 || k == WF_TR_OLD1 || k == WF_TR_TAIL1) ? 0ull : ~0ull;
    LIC360_CUDA(cudaMalloc(&t.dev, init.size() * 8));
    LIC360_CUDA(cudaMemcpy(t.dev, init.data(), init.size() * 8, cudaMemcpyHostToDevice));
    wf_trace_set(t.dev, t.sel);
    codec_trace_set(t.dev, t.sel);
    return LIC360_OK;
}

// after a decode: the trace's summary on stderr, and one line per step in the CSV file LIC360_WF_TRACE_FILE names
static void decode_trace_report(lic360_codec* c, DecodeTrace& t) {
    if (!t.dev) return;
    const NetDesc& net = t.sel ? c->imp : c->code;
    std::vector<unsigned long long> tr((size_t)t.steps * WF_TR_SLOTS + 64);
    cudaMemcpy(tr.data(), t.dev, tr.size() * 8, cudaMemcpyDeviceToHost);
    wf_trace_set(nullptr, 0);
    codec_trace_set(nullptr, 0);
    cudaFree(t.dev);
    t.dev = nullptr;
    const char* names[WF_TR_SLOTS] = {"scatter start", "prev start", "chain start", "chain end", "rows start", "rows flag", "old start", "old end", "R tail start", "R tail end"};
    for (int w0 = 0; w0 < 2; w0++) {  // two windows: while the importance stream still runs / after it finished
        const int pa = t.sel ? (w0 == 0 ? 10 : 50) : (w0 == 0 ? 20 : 140), pb = t.sel ? (w0 == 0 ? 45 : 90) : (w0 == 0 ? 80 : 220);
        double acc[WF_TR_SLOTS] = {0}, period = 0;
        int cnt = 0;
        for (int p = pa; p < pb && p + 1 < net.nsteps; p++) {
            const unsigned long long* r = &tr[(size_t)p * WF_TR_SLOTS];
            for (int k = 0; k < WF_TR_SLOTS; k++) acc[k] += (double)(long long)(r[k] - r[0]) * 1e-3;
            period += (double)(long long)(tr[(size_t)(p + 1) * WF_TR_SLOTS] - r[0]) * 1e-3;
            cnt++;
        }
        fprintf(stderr, "lic360 trace, %s-stream steps %d..%d: period %.1f us;", t.sel ? "importance" : "code", pa, pb, period / cnt);
        for (int k = 1; k < WF_TR_SLOTS; k++) fprintf(stderr, " %s +%.1f;", names[k], acc[k] / cnt);
        fprintf(stderr, "\n");
    }
    if (const char* fn = getenv("LIC360_WF_TRACE_FILE")) {  // per-step dump: step, slab length, us relative to the step's slot 0, period
        if (FILE* f = fopen(fn, "w")) {
            fprintf(f, "step,len,prev_start,chain_start,chain_end,rows_start,rows_last,old_start,old_end,tail_start,tail_end,period,host_wait_us,host_decode_us,levels_wait_us\n");
            for (int p = 0; p + 1 < net.nsteps; p++) {
                const unsigned long long* r = &tr[(size_t)p * WF_TR_SLOTS];
                fprintf(f, "%d,%d", p, net.steps[p].len);
                for (int k = 1; k < WF_TR_SLOTS; k++) fprintf(f, ",%.1f", (double)(long long)(r[k] - r[0]) * 1e-3);
                fprintf(f, ",%.1f", (double)(long long)(tr[(size_t)(p + 1) * WF_TR_SLOTS] - r[0]) * 1e-3);
                fprintf(f, ",%.1f,%.1f,%.1f\n", (size_t)p < net.step_wait_us.size() ? net.step_wait_us[p] : 0.f,
                        (size_t)p < net.step_decode_us.size() ? net.step_decode_us[p] : 0.f,
                        (size_t)p < net.step_levels_us.size() ? net.step_levels_us[p] : 0.f);
            }
            fclose(f);
        }
    }
    fprintf(stderr, "%s", t.sel ? "lic360 trace, G=1 chain, CTA 0, us per layer [weight staging | Q product | epilogue + DSMEM stores | prefetch + cluster barrier]:"
                                : "lic360 trace, code-stream chain, CTA 0 thread 0, us per layer [weight staging issue | item: 25 loads, 100 FMA4, stores | prefetch issue + weights landed | cluster barrier]:");
    for (int l = 0; l < 12; l++) {
        fprintf(stderr, " L%d", l);
        for (int ph = 0; ph < 4; ph++) fprintf(stderr, "%c%.2f", ph ? '|' : ' ', (double)tr[(size_t)t.steps * WF_TR_SLOTS + l * 4 + ph] * 1e-3 / net.nsteps);
    }
    fprintf(stderr, "\n");
}

// ------------------------------------------------------------------------------------------------ kernels
// code stream encoder input: x = (code - 3.5) * mask replicated for the 3 nets (lic360_demo.py:130-131).  n = K latents x (48, H, W):
// x is set-major, [net][k][48][H][W], the layout the conv kernels read with N = 3K images and 3 weight sets (image / K = set)
__global__ void prep_code_kernel(const float* __restrict__ code, const float* __restrict__ mask, float* __restrict__ x,
                                 int n, float bias) {
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const float v = (code[i] - bias) * mask[i];
        x[i] = v; x[i + n] = v; x[i + 2 * n] = v;
    }
}

// level of one cell in candidate t: max(s - max(t - P, 0), 0), s = imp_symbol(level) the symbol encode codes, P = protect[cell] clamped
// to [0, 48] (0 without a protection map, where this is max(s - t, 0))
__device__ __forceinline__ int candidate_level(const float* __restrict__ levels, const int32_t* __restrict__ protect, int cell, int t) {
    const int drop = protect ? max(t - min(max(protect[cell], 0), 48), 0) : t;
    return max((int)imp_symbol(levels[cell]) - drop, 0);
}

// Candidates of lic360_codec_estimate_candidates and lic360_codec_encode_candidates: candidate j (the batch's latent j) is source latent
// tab[j].x lowered by offset tab[j].y (candidate_level), with the levels, code and protection map of that source; the mask bit of a code
// symbol is code_mask_from_level of its cell's candidate level, the bit lic360_imp_levels_to_mask_protected stores.
struct Candidates {
    const int2* tab;
    const float* levels;     // (S,1,h,w) source levels
    const int32_t* protect;  // (S,1,h,w) or NULL
};

// the mask bit of code symbol (tc, th, tw) of an H x W latent in the candidate of source src and offset t
__device__ __forceinline__ int candidate_mask_bit(const Candidates& cd, int src, int t, int tc, int th, int tw, int H, int W) {
    const size_t cells = (size_t)src * (H >> 1) * (W >> 1);
    const int lvl = candidate_level(cd.levels + cells, cd.protect ? cd.protect + cells : nullptr, (th >> 1) * (W >> 1) + (tw >> 1), t);
    return code_mask_from_level(lvl, tc, th, tw);
}

// prep_code_kernel of J candidates: x = (code - 3.5) * mask with the source's code and the candidate's mask bit as a float, the
// arithmetic prep_code_kernel does on a materialised candidate.  n = J x (48, H, W), same set-major layout.
__global__ void prep_candidate_code_kernel(const float* __restrict__ code, Candidates cd, float* __restrict__ x, int n, int G, int H,
                                           int W, float bias) {
    const int plane = G * H * W;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int j = i / plane, p = i - j * plane;
        const int2 e = cd.tab[j];
        const int tw = p % W, th = (p / W) % H, tc = p / (W * H);
        const float v = (code[(size_t)e.x * plane + p] - bias) * (float)candidate_mask_bit(cd, e.x, e.y, tc, th, tw, H, W);
        x[i] = v; x[i + n] = v; x[i + 2 * n] = v;
    }
}

// the candidate levels (J,1,h,w) as float, candidate j in blockIdx.y: the importance network's input and the levels its bits kernel reads
__global__ void candidate_levels_kernel(Candidates cd, int hw, float* __restrict__ out) {
    const int2 e = cd.tab[blockIdx.y];
    const size_t cells = (size_t)e.x * hw;
    out += (size_t)blockIdx.y * hw;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < hw; i += gridDim.x * blockDim.x)
        out[i] = (float)candidate_level(cd.levels + cells, cd.protect ? cd.protect + cells : nullptr, i, e.y);
}

// The encoder's kernels run a batch of latents: latent blockIdx.y of gridDim.y.  The helpers below give each stream's batch layout, network
// outputs and CDF row once, for the row kernels (which pack the rows for the host coder) and the bits kernels (the rate estimate).
// code stream: y [net][latent][G*3][H][W], the outputs of [weight_net, delta_net, mean_net]; code, mask and the rest (G, H, W) per latent.
// Moves y to the block's latent and returns the offset of its symbols.
__device__ __forceinline__ size_t gmm_latent(const float* __restrict__& y, int G, int HW) {
    const size_t lat = blockIdx.y, plane = (size_t)G * HW;
    y += lat * 3 * plane;
    return lat * plane;
}

// code stream: the CDF row o[9] of symbol (tc, th, tw) from its 3x3 network outputs (y as gmm_latent left it)
__device__ __forceinline__ void gmm_symbol_row(const float* y, int G, int H, int W, int tc, int th, int tw, float s2, float* o) {
    const int HW = H * W;
    float wv[3], dv[3], mv[3];
    const size_t net = (size_t)gridDim.y * G * 3 * HW;
    const size_t base = ((size_t)tc * 3 * H + th) * W + tw;
#pragma unroll
    for (int i = 0; i < 3; i++) {
        wv[i] = y[base + (size_t)i * HW];
        dv[i] = y[net + base + (size_t)i * HW];
        mv[i] = y[2 * net + base + (size_t)i * HW];
    }
    gmm_row(wv, dv, mv, o, 3, 8, 3.5f, 65536.f, 1e-6f, s2);
}

// code stream: the row of plan position k of group tc in coding order (its step is th + tw + tc)
__device__ __forceinline__ int gmm_coding_row(const int* row_off, const StepDesc* steps, int k, int tc, int th, int tw) {
    const int p = th + tw + tc;
    return __ldg(row_off + p) + k - steps[p].start;
}

// importance stream: y [latent][49][h][w] logits, the levels and the rest (h, w) per latent.  Moves y to the block's latent and
// returns the offset of its cells.
__device__ __forceinline__ size_t imp_latent(const float* __restrict__& y, int HW) {
    const size_t lat = blockIdx.y;
    y += lat * 49 * HW;
    return lat * HW;
}

// importance stream: the CDF row o[1..49] of cell (th, tw) from its 49 logits (y as imp_latent left it)
__device__ __forceinline__ void imp_symbol_row(const float* y, int H, int W, int th, int tw, float* o) {
    for (int i = 0; i < 49; i++) o[1 + i] = y[((size_t)i * H + th) * W + tw];
    entropy_row(o, 49, 65536.f);
}

// code stream: one thread = one symbol (tc = i / HW, k = i % HW in plan order); its packed row (8 u16) at its coding-order row.
// CAND: latent blockIdx.y is candidate blockIdx.y of `cd`, as in gmm_bits_kernel<true>; `mask` is not read.
template <bool CAND>
__global__ void gmm_rows_kernel(const float* __restrict__ y, const float* __restrict__ code, const float* __restrict__ mask,
                                Candidates cd, const int32_t* __restrict__ idx, const StepDesc* __restrict__ steps,
                                const int* __restrict__ row_off, uint16_t* __restrict__ rows, int G, int H, int W, float s2) {
    const int HW = H * W;
    const size_t lat = gmm_latent(y, G, HW);
    int2 cand = make_int2(0, 0);
    if constexpr (CAND) {
        cand = cd.tab[blockIdx.y];
        code += (size_t)cand.x * G * HW;
    } else {
        code += lat; mask += lat;
    }
    rows += lat * 8;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= G * HW) return;
    const int k = i % HW, tc = i / HW;
    const int th = __ldg(idx + k), tw = __ldg(idx + k + HW);
    rows += (size_t)gmm_coding_row(row_off, steps, k, tc, th, tw) * 8;
    const size_t pos = ((size_t)tc * H + th) * W + tw;
    // NaN and anything outside [0, 8) become the out-of-range marker of the row.  Symbol and mask bit are read before the row is built:
    // it keeps the kernel at 32 registers.
    const int sym = code_symbol(code[pos]);
    int maskbit;
    if constexpr (CAND) maskbit = candidate_mask_bit(cd, cand.x, cand.y, tc, th, tw, H, W);
    else maskbit = code_mask_bit(mask[pos]);
    float o[9];
    gmm_symbol_row(y, G, H, W, tc, th, tw, s2, o);
    pack_gmm_row(o, sym, maskbit, rows);
}

// importance stream: one thread = one position k of the plan = row k of the stream (64 u16)
__global__ void imp_rows_kernel(const float* __restrict__ y, const float* __restrict__ levels, const int32_t* __restrict__ idx,
                                uint16_t* __restrict__ rows, int H, int W) {
    const int HW = H * W;
    const size_t lat = imp_latent(y, HW);
    levels += lat; rows += lat * 64;
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    if (k >= HW) return;
    const int th = __ldg(idx + k), tw = __ldg(idx + k + HW);
    float o[50];
    imp_symbol_row(y, H, W, th, tw, o);
    uint16_t* dst = rows + (size_t)k * 64;
    uint32_t ovf[3] = {0, 0, 0};
    for (int j = 1; j <= 48; j++) {
        const uint32_t v = (uint32_t)(int)o[j];
        dst[j - 1] = (uint16_t)(v & 0xFFFF);
        ovf[(j - 1) / 16] |= ((v >> 16) & 1u) << ((j - 1) % 16);
    }
    dst[48] = (uint16_t)imp_symbol(levels[th * W + tw]);
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

// A batch: latent blockIdx.y of gridDim.y, each with the block partition, the partials and the error key of a single latent, so its
// totals and map do not depend on the other latents.
// code stream: thread i = symbol (tc = i / HW, k = i % HW in plan order), bits (optional) in (G, H, W) layout per latent; count: coded
// symbols (mask >= 0.5) per block.  CAND: latent blockIdx.y is candidate blockIdx.y of `cd`, its code read from its source latent and
// its mask bit derived from the candidate level (candidate_mask_bit); `mask` is not read.
template <bool CAND>
__global__ void __launch_bounds__(BITS_THREADS) gmm_bits_kernel(const float* __restrict__ y, const float* __restrict__ code,
                                const float* __restrict__ mask, Candidates cd, const int32_t* __restrict__ idx,
                                const StepDesc* __restrict__ steps, const int* __restrict__ row_off, float* __restrict__ bits,
                                double* __restrict__ partial, int* __restrict__ count, unsigned long long* err, int G, int H, int W,
                                float s2) {
    const int HW = H * W;
    const size_t lat = gmm_latent(y, G, HW);
    int2 cand = make_int2(0, 0);
    if constexpr (CAND) {
        cand = cd.tab[blockIdx.y];
        code += (size_t)cand.x * G * HW;
    } else {
        code += lat; mask += lat;
    }
    err += blockIdx.y;
    if (bits) bits += lat;
    partial += (size_t)blockIdx.y * gridDim.x; count += (size_t)blockIdx.y * gridDim.x;
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    double cost = 0.0;
    int coded = 0;
    if (i < G * HW) {
        const int k = i % HW, tc = i / HW;
        const int th = __ldg(idx + k), tw = __ldg(idx + k + HW);
        const size_t pos = ((size_t)tc * H + th) * W + tw;
        if constexpr (CAND) coded = candidate_mask_bit(cd, cand.x, cand.y, tc, th, tw, H, W);
        else coded = code_mask_bit(mask[pos]);
        if (coded) {  // a position the encoder skips costs nothing, whatever its symbol
            float o[9];
            gmm_symbol_row(y, G, H, W, tc, th, tw, s2, o);
            const int s = code_symbol(code[pos]);
            if (s > 7 || !symbol_bits<8>(o, s, &cost)) {
                const unsigned long long row = (unsigned)gmm_coding_row(row_off, steps, k, tc, th, tw);
                atomicMin(err, (row << 32) | (unsigned)s);
                cost = 0.0;
            }
        }
        if (bits) bits[pos] = (float)cost;
    }
    coded = __syncthreads_count(coded);
    cost = block_sum_fixed(cost);
    if (threadIdx.x == 0) { partial[blockIdx.x] = cost; count[blockIdx.x] = coded; }
}

// importance stream: thread k = position k of the plan = row k of the stream, bits (optional) in (h, w) layout per latent; every
// position is coded
__global__ void __launch_bounds__(BITS_THREADS) imp_bits_kernel(const float* __restrict__ y, const float* __restrict__ levels,
                                const int32_t* __restrict__ idx, float* __restrict__ bits, double* __restrict__ partial,
                                int* __restrict__ count, unsigned long long* err, int H, int W) {
    const int HW = H * W;
    const size_t lat = imp_latent(y, HW);
    levels += lat; err += blockIdx.y;
    if (bits) bits += lat;
    partial += (size_t)blockIdx.y * gridDim.x; count += (size_t)blockIdx.y * gridDim.x;
    const int k = blockIdx.x * blockDim.x + threadIdx.x;
    double cost = 0.0;
    if (k < HW) {
        const int th = __ldg(idx + k), tw = __ldg(idx + k + HW);
        float o[50];
        imp_symbol_row(y, H, W, th, tw, o);
        const uint32_t s = imp_symbol(levels[th * W + tw]);
        if (s >= 49 || !symbol_bits<49>(o, (int)s, &cost)) {
            atomicMin(err, ((unsigned long long)k << 32) | s);
            cost = 0.0;
        }
        if (bits) bits[th * W + tw] = (float)cost;
    }
    const int coded = __syncthreads_count(k < HW);
    cost = block_sum_fixed(cost);
    if (threadIdx.x == 0) { partial[blockIdx.x] = cost; count[blockIdx.x] = coded; }
}

// block b = latent b: thread t adds the latent's n partials t, t + BITS_THREADS, ... in index order, then the block's fixed tree; the
// counts are integers, added in any order
__global__ void __launch_bounds__(BITS_THREADS) bits_sum_kernel(const double* __restrict__ partial, const int* __restrict__ count, int n,
                                                                double* __restrict__ total, long long* __restrict__ total_count) {
    __shared__ unsigned long long coded;
    partial += (size_t)blockIdx.x * n; count += (size_t)blockIdx.x * n;
    if (threadIdx.x == 0) coded = 0;
    double v = 0.0;
    long long m = 0;
    for (int i = threadIdx.x; i < n; i += BITS_THREADS) { v += partial[i]; m += count[i]; }
    v = block_sum_fixed(v);  // its barrier orders the reset of `coded` before the adds
    atomicAdd(&coded, (unsigned long long)m);
    __syncthreads();
    if (threadIdx.x == 0) { total[blockIdx.x] = v; total_count[blockIdx.x] = (long long)coded; }
}

// candidate j (blockIdx.y) of lic360_imp_levels_to_mask_batch: the candidate level of every cell of source latent off.src[j] at offset
// off.k[j] (candidate_level) and the (48, 2h, 2w) code mask the decoder derives from it (Imp2mask + Dtow)
struct LevelOffsets { int k[32]; int src[32]; };
__global__ void imp_levels_to_mask_kernel(const float* __restrict__ levels, const int32_t* __restrict__ protect, int h, int w,
                                          LevelOffsets off, float* __restrict__ levels_out, float* __restrict__ mask_out) {
    const int j = blockIdx.y, k = off.k[j], hw = h * w, W = 2 * w, n = 48 * 4 * hw;
    levels += (size_t)off.src[j] * hw;
    if (protect) protect += (size_t)off.src[j] * hw;
    levels_out += (size_t)j * hw;
    mask_out += (size_t)j * n;
    for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < n; i += gridDim.x * blockDim.x) {
        const int tw = i % W, th = (i / W) % (2 * h), tc = i / (W * 2 * h);
        const int cell = (th >> 1) * w + (tw >> 1);
        mask_out[i] = (float)code_mask_from_level(candidate_level(levels, protect, cell, k), tc, th, tw);
        if (i < hw) levels_out[i] = (float)candidate_level(levels, protect, i, k);
    }
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
    const int H = n.H, W = n.W, G = n.G;
    std::vector<int32_t> idx(2 * (size_t)H * W), plan(H + W);
    lic360_code_contex(H, W, idx.data(), plan.data());
    LIC360_CUDA(cudaMalloc(&n.idx_dev, idx.size() * sizeof(int32_t)));
    LIC360_CUDA(cudaMemcpy(n.idx_dev, idx.data(), idx.size() * sizeof(int32_t), cudaMemcpyHostToDevice));
    n.nsteps = H + W + G - 2;
    n.steps.resize(n.nsteps);
    n.row_off.resize(n.nsteps + 1);
    int off = 0;
    for (int p = 0; p < n.nsteps; p++) {
        int s, l;
        slab_of(plan.data(), H, W, G, p, &s, &l);
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

// K latents: N = nsets * K images, set-major (image / K = weight set)
static int conv_args(const NetDesc& n, int l, int K, ConvArgs& a) {
    const float *x, *r;
    float* out;
    layer_io(n, l, &x, &r, &out);
    if (fill_conv_args(a, x, n.wp[l], n.wq[l], n.bias[l], n.act[l] ? n.slope[l] : nullptr, r, out, n.nsets * K, n.Cin[l], n.H, n.W,
                       n.Cout[l], n.G, n.constrain[l], n.nsets)) {
        set_error("codec: bad layer geometry");
        return LIC360_ERR_ARG;
    }
    return LIC360_OK;
}

static int run_ec_net(const NetDesc& n, int K, cudaStream_t s) {
    for (int l = 0; l < 12; l++) {
        ConvArgs a;
        int rc = conv_args(n, l, K, a);
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

// s2 of gmm_row: 1 / sqrt(2)
static const float kGmmS2 = (float)(1. / sqrt(2.0));
// importance stream network input: Scale(-1, 2/47) of the levels (lic360_demo.py:173-189)
static const float kImpScale = (float)(2. / (48 - 1.));

// TileInput of a decoded symbol into the stream's network input: scale * symbol + bias, once for each of its rep nets
struct TileIn { float bias, scale; int rep; };
static TileIn tile_input(bool is_code) { return is_code ? TileIn{-3.5f, 1.0f, 3} : TileIn{-1.0f, kImpScale, 1}; }

// LIC360_DEBUG_SYNC: synchronise after every kernel of a serialized (mode 1) decode step, and after the set-up of every decode
static bool debug_sync() {
    static const bool on = getenv("LIC360_DEBUG_SYNC") != nullptr;
    return on;
}

// the error paths that leave work on both CUDA streams: wait for it, so that the caller may reuse its buffers once the call returns
static void drain(lic360_codec* c) {
    cudaStreamSynchronize(c->code.stream);
    cudaStreamSynchronize(c->imp.stream);
}

// where the chain kernels of a decode step put its CDF rows
static WfRows wf_rows(lic360_codec* c, NetDesc& n) {
    WfRows rows;
    rows.rows = n.rows_step_host; rows.levels = c->levels_dev; rows.flag = n.flag_host; rows.sync = n.sync_dev;
    rows.s2 = kGmmS2;
    return rows;
}

// the symbols of the previous step into the network input (TileInput); the importance stream also keeps them as the decoded levels
static int launch_scatter(lic360_codec* c, NetDesc& n, bool is_code, cudaStream_t s) {
    const WfNetDev& w = n.wf.dev;
    const TileIn t = tile_input(is_code);
    scatter_prev_kernel<<<(n.max_len + 127) / 128, 128, 0, s>>>(n.syms_host, n.wf.fp[0], n.wf.fc[0], n.idx_dev, n.steps_dev, n.ctr_dev,
                                                              n.arrived_dev, n.G, n.H, n.W, w.D, w.HS, w.Dp, w.Hp, t.bias, t.scale, t.rep,
                                                              is_code ? nullptr : c->levels_dev);
    LAUNCH_CHECK();
    return LIC360_OK;
}

// the kernels of one decode step.  side == s (serialized / profile mode): everything in stream order, the old terms of
// the NEXT step last.  side != s (graph capture): the old terms run beside the chain as its programmatic dependent; either way the
// host is released by the step's rows (published row by row in the code stream, by a flag in the importance stream), so the bulk
// of the arithmetic also overlaps the host coder.
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
    const bool dbg = debug_sync() && ev != nullptr;  // only in the serialized mode
    if (ev) LIC360_CUDA(cudaEventRecord(ev[0], s));
    const int rc = launch_scatter(c, n, is_code, s);
    if (rc) return rc;
    WF_DEBUG_SYNC("scatter kernel");
    const bool fork = side != s;  // graph capture: overlap the old terms of the next step with the chain (see below)
    if (ev) LIC360_CUDA(cudaEventRecord(ev[1], s));
    // wf_chain4_kernel (code stream) and wf_chain1_kernel evaluate layer 0's previous-wavefront terms in their prologue and emit the
    // step's CDF rows themselves; the generic chain kernel (importance stream, long diagonals) needs a launch for each
    const bool fused = n.wf.chain4 || n.wf.chain1;
    if (!fused) {
        LIC360_CUDA(wf_launch_prev(n.wf, 0, 0, 1, s));  // layer 0 only: its taps read the symbols scattered a moment ago
        WF_DEBUG_SYNC("previous-wavefront kernel (layer 0)");
    }
    if (ev) LIC360_CUDA(cudaEventRecord(ev[2], s));
    LIC360_CUDA(wf_launch_chain(n.wf, s, wf_rows(c, n)));
    WF_DEBUG_SYNC("chain kernel");
    if (ev) LIC360_CUDA(cudaEventRecord(ev[3], s));
    // The old terms of step p+1 only read wavefronts <= p-1: they are launched right behind the chain kernel as its
    // PROGRAMMATIC dependent -- they start once every chain CTA is resident (so the chain's clusters got their SMs first)
    // and fill the SMs the chain leaves idle.  In the importance stream, whatever still needs the chain's RESULTS (the rows
    // kernel of the generic chain, the previous-wavefront kernel of the next step) waits for the chain's completion on the side
    // stream.  The code stream's chain kernel also leaves the previous-wavefront terms of the next step behind: no side branch.
    cudaStream_t rs = s;  // stream of the kernels behind the chain
    if (fork) {
        LIC360_CUDA(cudaEventRecord(n.ev_fork, s));
        LIC360_CUDA(wf_launch_old(n.wf, 1, s, true));
        if (!is_code) {
            LIC360_CUDA(cudaStreamWaitEvent(side, n.ev_fork, 0));
            rs = side;
        }
    }
    if (!fused) {
        imp_rows_wf_kernel<<<std::max(1, std::min(4, (n.max_len + IMP_ROWS_WARPS - 1) / IMP_ROWS_WARPS)), 32 * IMP_ROWS_WARPS, 0, rs>>>(n.wf.fc[12], n.idx_dev, n.steps_dev, n.ctr_dev, n.rows_step_host, n.H, n.W, w.Dp, w.Hp,
                                                 n.done_dev, n.flag_host);
        LAUNCH_CHECK();
        WF_DEBUG_SYNC("rows kernel");
    }
    if (!is_code) {
        // previous-wavefront terms of layers 1..11 for step p+1 (the activations of wavefront p are final): behind the rows,
        // i.e. underneath the host decoder instead of on the critical path
        LIC360_CUDA(wf_launch_prev(n.wf, 1, 1, WF_LAYERS, rs));
        WF_DEBUG_SYNC("previous-wavefront kernel (layers 1..11 of the next step)");
    }
    if (ev) LIC360_CUDA(cudaEventRecord(ev[4], s));
    if (fork && is_code) {
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
    const int rc = launch_step(c, n, is_code, s, n.side, nullptr);
    cudaError_t e = cudaStreamEndCapture(s, &g);
    n.graph_nodes = (int)(g_launches - l0);
    g_launches = l0;  // captured, not launched: replays are counted in decode_stream
    if (rc != LIC360_OK) { if (e == cudaSuccess) cudaGraphDestroy(g); return rc; }
    LIC360_CUDA(e);
    {   // kernel-node priorities: the importance stream's old-term kernel lowest, everything else at its stream's level
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
            // code stream: every kernel highest -- its old-term kernel, wf_old4_kernel, is not singled out here; the importance
            // stream has slack (it only has to stay ahead of the code stream): one level below, its old-term kernel
            // (wf_old_kernel) lowest
            const int hi = is_code ? prio_hi : std::min(prio_lo, prio_hi + 2);
            v.priority = kp.func == wf_old_kernel_ptr() ? prio_lo : hi;
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
    return LIC360_OK;
}

// Replaces every buffer of `bufs` with one of its new size, or none of them: the old ones are kept unless every new one was allocated.
struct GrowBuf { void** slot; size_t bytes; bool pinned; };
static int grow_buffers(lic360_codec* c, const std::vector<GrowBuf>& bufs, int K) {
    // the old buffers may still be in use by work enqueued on the codec's streams
    LIC360_CUDA(cudaStreamSynchronize(c->code.stream));
    LIC360_CUDA(cudaStreamSynchronize(c->imp.stream));
    std::vector<void*> fresh(bufs.size(), nullptr);
    cudaError_t e = cudaSuccess;
    for (size_t i = 0; i < bufs.size() && e == cudaSuccess; i++)
        e = bufs[i].pinned ? cudaHostAlloc(&fresh[i], bufs[i].bytes, cudaHostAllocDefault) : cudaMalloc(&fresh[i], bufs[i].bytes);
    for (size_t i = 0; i < bufs.size(); i++) {
        void* old = e == cudaSuccess ? *bufs[i].slot : fresh[i];
        if (bufs[i].pinned) cudaFreeHost(old); else cudaFree(old);
        if (e == cudaSuccess) *bufs[i].slot = fresh[i];
    }
    if (e != cudaSuccess) {
        cudaGetLastError();
        set_error("codec: cannot allocate the buffers of %d latents (%s)", K, cudaGetErrorString(e));
        return LIC360_ERR_CUDA;
    }
    return LIC360_OK;
}

// The buffers that scale with the number of latents an encode or an estimate runs at once: both networks' encoder frames, the bits
// kernels' partials, the estimate's results and the candidate table and levels of estimate_ / encode_candidates.  They only grow.
static int batch_reserve(lic360_codec* c, int K) {
    if (K <= c->batch_cap) return LIC360_OK;
    std::vector<GrowBuf> bufs;
    for (NetDesc* n : {&c->code, &c->imp}) {
        for (int i = 0; i < 13; i++) bufs.push_back({reinterpret_cast<void**>(&n->frame[i]), n->frame_floats[i] * K * sizeof(float), false});
        bufs.push_back({reinterpret_cast<void**>(&n->bits_partial_dev), (size_t)n->bits_blocks * K * sizeof(double), false});
        bufs.push_back({reinterpret_cast<void**>(&n->count_partial_dev), (size_t)n->bits_blocks * K * sizeof(int), false});
    }
    bufs.push_back({reinterpret_cast<void**>(&c->cand_dev), (size_t)K * sizeof(int2), false});
    bufs.push_back({reinterpret_cast<void**>(&c->cand_levels_dev), (size_t)K * c->imp.H * c->imp.W * sizeof(float), false});
    bufs.push_back({&c->est_dev, estimate_bytes(K), false});
    bufs.push_back({&c->est_host, estimate_bytes(K), true});
    const int rc = grow_buffers(c, bufs, K);
    if (rc == LIC360_OK) c->batch_cap = K;
    return rc;
}

// The encoder's CDF rows of K latents, on the device and in pinned host memory, for both streams.  Only an encode grows them (an
// estimate packs no rows), and they only grow.
static int rows_reserve(lic360_codec* c, int K) {
    if (K <= c->rows_cap) return LIC360_OK;
    std::vector<GrowBuf> bufs;
    for (NetDesc* n : {&c->code, &c->imp}) {
        const size_t bytes = (size_t)n->total_rows * n->row_bytes * K;
        bufs.push_back({reinterpret_cast<void**>(&n->rows_dev), bytes, false});
        bufs.push_back({reinterpret_cast<void**>(&n->rows_host), bytes, true});
    }
    const int rc = grow_buffers(c, bufs, K);
    if (rc == LIC360_OK) c->rows_cap = K;
    return rc;
}

static void ctx_free(NetDesc& n) {
    cudaFree(n.ctr_dev); cudaFree(n.done_dev); cudaFree(n.arrived_dev); cudaFree(n.sync_dev); cudaFree(n.go_dev); cudaFree(n.old_done_dev); cudaFree(n.scat_done_dev);
    cudaFreeHost(n.flag_host); cudaFreeHost(n.go_host);
    cudaFree(n.rows_dev); cudaFreeHost(n.rows_host); cudaFreeHost(n.rows_step_host); cudaFreeHost(n.syms_host);
    cudaFree(n.bits_partial_dev); cudaFree(n.count_partial_dev);
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
    if (ok) {
        c->chain_cap = wf_chain_capacity(c->code.wf);
        c->code.nflags = c->code.wf.dev.nsets * c->code.wf.cluster;  // at most 3 x 16 of the 64 flags
    }
    ok = ok && cudaMalloc(&c->levels_dev, (size_t)(H / 2) * (W / 2) * sizeof(float)) == cudaSuccess;
    ok = ok && cudaMalloc(&c->mask192_dev, (size_t)192 * (H / 2) * (W / 2) * sizeof(float)) == cudaSuccess;
    ok = ok && cudaEventCreateWithFlags(&c->ev_est, cudaEventDisableTiming) == cudaSuccess;
    if (!ok && wf_ok) set_error("codec: allocation failed (%s)", cudaGetErrorString(cudaGetLastError()));  // else: wf_init's message
    ok = ok && batch_reserve(c, 1) == LIC360_OK;  // (its own message)
    if (!ok) {
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
    cudaFree(c->cand_dev); cudaFree(c->cand_levels_dev);
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
// stream's 12 layers, enqueued on its own CUDA stream; the outputs land in n.frame[12].  K latents (K <= c->batch_cap) run as one
// batch of the same kernels: each latent's outputs are those of a run of that latent alone (the conv kernels compute every image
// alike, whatever else is in the batch).
//   importance stream (lic360_demo.py:173-189): Scale(-1, 2/47) of the levels
//   code stream (lic360_demo.py:124-131): (code - 3.5) * mask, once for each of the three nets
// cand: the K latents are candidates (lic360_codec_estimate_candidates, lic360_codec_encode_candidates): code_dev holds their sources
// and the masks are derived, imp_dev holds the candidate levels
static int run_encoder_net(lic360_codec* c, bool is_code, int K, const float* code_dev, const float* mask_dev, const float* imp_dev,
                           const Candidates* cand = nullptr) {
    NetDesc& n = is_code ? c->code : c->imp;
    if (is_code) {
        const int nel = K * n.G * n.H * n.W;
        if (cand)
            prep_candidate_code_kernel<<<stream_grid(nel, 256), 256, 0, n.stream>>>(code_dev, *cand, n.frame[0], nel, n.G, n.H, n.W, 3.5f);
        else
            prep_code_kernel<<<stream_grid(nel, 256), 256, 0, n.stream>>>(code_dev, mask_dev, n.frame[0], nel, 3.5f);
        LAUNCH_CHECK();
    } else {
        const int rc = lic360_scale(imp_dev, n.frame[0], (size_t)K * n.H * n.W, -1.0f, kImpScale, n.stream);
        if (rc) return rc;
    }
    return run_ec_net(n, K, n.stream);
}

// The candidates of an estimate or an encode of K candidates: the table cand_host goes to c->cand_dev (cd.tab) and their levels to
// c->cand_levels_dev, on the importance stream; both streams read the table, so the code stream waits for it (ev_est).
static int enqueue_candidates(lic360_codec* c, int K, const int2* cand_host, const Candidates& cd) {
    cudaStream_t s = c->imp.stream;
    const int hw = c->imp.H * c->imp.W;
    LIC360_CUDA(cudaMemcpyAsync(c->cand_dev, cand_host, (size_t)K * sizeof(int2), cudaMemcpyHostToDevice, s));
    candidate_levels_kernel<<<dim3((hw + 255) / 256, K), 256, 0, s>>>(cd, hw, c->cand_levels_dev);
    LAUNCH_CHECK();
    LIC360_CUDA(cudaEventRecord(c->ev_est, s));
    LIC360_CUDA(cudaStreamWaitEvent(c->code.stream, c->ev_est, 0));
    return LIC360_OK;
}

// the (source latent, offset) table of J candidates of K sources; a source outside [0, K) or a negative offset is an argument error of
// the entry point fn
static int candidate_table(const char* fn, int K, int J, const int* cand_latent_host, const int* cand_offset_host, std::vector<int2>& tab) {
    tab.resize(J);
    for (int j = 0; j < J; j++) {
        const char* bad = cand_latent_host[j] < 0 || cand_latent_host[j] >= K ? "cand_latent must lie in [0, K)"
                        : cand_offset_host[j] < 0                            ? "offsets must not be negative" : nullptr;
        if (bad) {
            set_error("%s: %s", fn, bad);
            return LIC360_ERR_ARG;
        }
        tab[j] = make_int2(cand_latent_host[j], cand_offset_host[j]);
    }
    return LIC360_OK;
}

// the GPU work of an encode of K latents on the codec's two streams: both networks at batch K, the CDF rows of every latent in coding
// order (latent k's rows at k * total_rows) and their copy to the host, one per stream.  cand (K candidates, enqueue_candidates done):
// code_dev holds the sources, imp_dev the candidate levels, and the code stream's mask bits are derived (mask_dev is not read).
static int enqueue_encode(lic360_codec* c, int K, const float* code_dev, const float* mask_dev, const float* imp_dev, clk::time_point t0,
                          const Candidates* cand = nullptr) {
    // The two bitstreams are independent: both networks are enqueued on their own CUDA streams first, then the host
    // codes the (small) importance stream while the code-stream network is still running.
    // ---- importance stream: net -> rows of all symbols
    {
        NetDesc& n = c->imp;
        cudaStream_t s = n.stream;
        const int HW = n.H * n.W;
        int rc = run_encoder_net(c, false, K, code_dev, mask_dev, imp_dev);
        if (rc) return rc;
        imp_rows_kernel<<<dim3((HW + 127) / 128, K), 128, 0, s>>>(n.frame[12], imp_dev, n.idx_dev, n.rows_dev, n.H, n.W);
        LAUNCH_CHECK();
        LIC360_CUDA(cudaMemcpyAsync(n.rows_host, n.rows_dev, (size_t)K * n.total_rows * 128, cudaMemcpyDeviceToHost, s));
        c->t_gpu_steps_imp = ms_since(t0);  // host time spent enqueueing the importance-stream work
    }
    // ---- code stream (lic360_demo.py:124-141)
    {
        NetDesc& n = c->code;
        cudaStream_t s = n.stream;
        const auto tq0 = clk::now();
        const int nel = n.G * n.H * n.W;
        int rc = run_encoder_net(c, true, K, code_dev, mask_dev, imp_dev, cand);
        if (rc) return rc;
        const dim3 grid((nel + 127) / 128, K);
        if (cand)
            gmm_rows_kernel<true><<<grid, 128, 0, s>>>(n.frame[12], code_dev, nullptr, *cand, n.idx_dev, n.steps_dev, n.row_off_dev,
                                                       n.rows_dev, n.G, n.H, n.W, kGmmS2);
        else
            gmm_rows_kernel<false><<<grid, 128, 0, s>>>(n.frame[12], code_dev, mask_dev, Candidates{}, n.idx_dev, n.steps_dev,
                                                        n.row_off_dev, n.rows_dev, n.G, n.H, n.W, kGmmS2);
        LAUNCH_CHECK();
        LIC360_CUDA(cudaMemcpyAsync(n.rows_host, n.rows_dev, (size_t)K * n.total_rows * 16, cudaMemcpyDeviceToHost, s));
        c->t_gpu_steps = ms_since(tq0);  // host time spent enqueueing the code-stream work
    }
    return LIC360_OK;
}

// one stream of one latent from its rows into `out`, with `coder`
static void code_stream_job(lic360_coder* coder, const uint16_t* rows, int nrows, int sid, EncodedStream* out) {
    lic360_coder_start_encoder_mem(coder);
    int rc = sid ? coder_encode_packed_imp(coder, rows, nrows) : coder_encode_packed_gmm(coder, rows, nrows);
    if (rc == LIC360_OK && lic360_coder_finish_mem(coder) < 0) rc = LIC360_ERR_CODER;
    out->rc = rc;
    if (rc) {
        out->err = lic360_last_error();  // the message is thread-local
        out->bytes.clear();
        return;
    }
    long nb = 0;
    const uint8_t* b = coder_bytes(coder, &nb);
    out->bytes.assign(b, b + nb);
}

// appends " (<what> k)" to the message of the calling thread's last error
static void add_index_suffix(const char* what, int k) {
    const std::string msg = lic360_last_error();
    set_error("%s (%s %d)", msg.c_str(), what, k);
}

// The host coding of an encode of K latents, every stream into enc_out: the K importance streams as soon as their rows are on the host
// (the code network may still be running), then the K code streams.  K = 1 codes on the calling thread with the codec's two coders,
// K > 1 on the coder pool.  Both CUDA streams are drained on every path.  suffix: NULL, or the word of the " (<suffix> k)" an error gets
static int code_streams(lic360_codec* c, int K, const char* suffix, clk::time_point t0) {
    const bool pooled = K > 1;
    if (pooled) {
        const unsigned hw = std::thread::hardware_concurrency();
        if (c->coder_pool.grow(std::min(std::min(K, kMaxCoderWorkers), std::max(1, (int)hw))) == 0) {
            drain(c);
            set_error("codec: cannot start a coder thread");
            return LIC360_ERR_CODER;
        }
    }
    c->enc_out.resize(2 * (size_t)K);
    auto code_stream = [&](NetDesc& n, int sid) {
        const size_t row_u16 = (size_t)n.total_rows * n.row_bytes / 2;
        for (int k = 0; k < K; k++) {
            const uint16_t* rows = n.rows_host + k * row_u16;
            EncodedStream* out = &c->enc_out[2 * (size_t)k + sid];
            const int nrows = n.total_rows;
            if (pooled) c->coder_pool.post([=](lic360_coder* coder) { code_stream_job(coder, rows, nrows, sid, out); });
            else code_stream_job(n.coder, rows, nrows, sid, out);
        }
    };
    auto tw = clk::now();
    const cudaError_t e_imp = cudaStreamSynchronize(c->imp.stream);
    c->t_gpu_wait += ms_since(tw);
    const auto th = clk::now();
    if (e_imp == cudaSuccess) code_stream(c->imp, 1);
    const double t_imp_coder = ms_since(th);
    if (!pooled) c->t_imp = ms_since(t0);
    tw = clk::now();
    const cudaError_t e_code = cudaStreamSynchronize(c->code.stream);
    c->t_gpu_wait += ms_since(tw);
    const auto tc = clk::now();
    if (e_imp == cudaSuccess && e_code == cudaSuccess) code_stream(c->code, 0);
    if (pooled) c->coder_pool.wait();
    // K = 1: the coder's time; K > 1: the wall time of the coding phase
    c->t_host_coder = pooled ? ms_since(th) : t_imp_coder + ms_since(tc);
    int rc = LIC360_OK;
    if (e_imp != cudaSuccess || e_code != cudaSuccess) {
        set_error("codec: the batch encode's GPU work failed -> %s", cudaGetErrorString(e_imp != cudaSuccess ? e_imp : e_code));
        rc = LIC360_ERR_CUDA;
    }
    // the error encode reports for the lowest bad latent alone, whichever worker finished first; within a latent the importance
    // stream's (encode codes it first)
    for (int k = 0; k < K && rc == LIC360_OK; k++)
        for (int sid : {1, 0}) {
            const EncodedStream& r = c->enc_out[2 * (size_t)k + sid];
            if (r.rc == LIC360_OK) continue;
            set_error("%s", r.err.c_str());
            if (suffix) add_index_suffix(suffix, k);
            rc = r.rc;
            break;
        }
    if (rc)
        for (EncodedStream& e : c->enc_out) e.bytes.clear();
    return rc;
}

// the start of an encode or an estimate of K latents on the codec's device (guard): both networks have their parameters, the buffers
// that scale with K hold K latents, and the timing of the last call is reset
static int begin_latents(lic360_codec* c, const DeviceGuard& guard, int K) {
    LIC360_CUDA(guard.err);
    int rc = check_params(c->code);
    if (rc == LIC360_OK) rc = check_params(c->imp);
    if (rc == LIC360_OK) rc = batch_reserve(c, K);
    if (rc) return rc;
    c->t_host_coder = 0; c->t_gpu_wait = 0; c->t_imp = 0; c->t_gpu_steps = 0; c->t_gpu_steps_imp = 0;
    return LIC360_OK;
}

// lic360_codec_encode (K = 1, no suffix), lic360_codec_encode_batch (suffix "latent") and lic360_codec_encode_candidates (suffix
// "candidate", the table in cand_host, imp_dev the sources' levels); protect may be NULL
static int encode_latents(lic360_codec* c, int K, const float* code_dev, const float* mask_dev, const float* imp_dev, const char* suffix,
                          const int2* cand_host = nullptr, const int32_t* protect = nullptr) {
    DeviceGuard guard(c->device);
    c->enc_k = 0;
    int rc = begin_latents(c, guard, K);
    if (rc == LIC360_OK) rc = rows_reserve(c, K);
    if (rc) return rc;
    const auto t0 = clk::now();
    const Candidates cd{c->cand_dev, imp_dev, protect};
    if (cand_host) rc = enqueue_candidates(c, K, cand_host, cd);
    if (rc == LIC360_OK && cand_host) rc = enqueue_encode(c, K, code_dev, nullptr, c->cand_levels_dev, t0, &cd);
    else if (rc == LIC360_OK) rc = enqueue_encode(c, K, code_dev, mask_dev, imp_dev, t0);
    if (rc) { drain(c); return rc; }
    rc = code_streams(c, K, suffix, t0);
    c->t_total = ms_since(t0);
    if (rc == LIC360_OK) c->enc_k = K;
    return rc;
}

// K within the launch limits of a batch
#define LIC360_CHECK_BATCH(c, K)                                                                                \
    LIC360_CHECK_ARG(K <= kMaxBatch && (long long)3 * K * (c)->code.G * (c)->H * (c)->W <= 0x7fffffffLL,       \
                     "K exceeds the launch limits of a batch (3K conv images, 3 * K * 48 * H * W input floats)")

int lic360_codec_encode(lic360_codec* c, const float* code_dev, const float* mask_dev, const float* imp_dev) {
    LIC360_CHECK_ARG(c && code_dev && mask_dev && imp_dev, "bad arguments");
    return encode_latents(c, 1, code_dev, mask_dev, imp_dev, nullptr);
}

int lic360_codec_encode_batch(lic360_codec* c, int K, const float* code_dev, const float* mask_dev, const float* imp_dev) {
    LIC360_CHECK_ARG(K >= 1, "K must be at least 1");
    LIC360_CHECK_ARG(c && code_dev && mask_dev && imp_dev, "bad arguments");
    LIC360_CHECK_BATCH(c, K);
    return encode_latents(c, K, code_dev, mask_dev, imp_dev, "latent");
}

int lic360_codec_encode_candidates(lic360_codec* c, int K, const float* code_dev, const float* imp_dev, const int32_t* protect_dev, int J,
                                   const int* cand_latent_host, const int* cand_offset_host) {
    LIC360_CHECK_ARG(K >= 1, "K must be at least 1");
    LIC360_CHECK_ARG(J >= 1, "J must be at least 1");
    LIC360_CHECK_ARG(c && code_dev && imp_dev && cand_latent_host && cand_offset_host, "bad arguments");
    LIC360_CHECK_BATCH(c, J);
    std::vector<int2> tab;
    const int rc = candidate_table(__func__, K, J, cand_latent_host, cand_offset_host, tab);
    if (rc) return rc;
    return encode_latents(c, J, code_dev, nullptr, imp_dev, "candidate", tab.data(), protect_dev);
}

// the GPU work of an estimate of K latents on the codec's two streams; the code stream ends with the copy of both streams' results.
// cand (K candidates, lic360_codec_estimate_candidates): its table is uploaded to c->cand_dev first, code_dev holds the sources, and
// the importance stream's input is the candidate levels, written to c->cand_levels_dev (imp_dev and mask_dev are not read).
static int enqueue_estimate(lic360_codec* c, int K, const float* code_dev, const float* mask_dev, const float* imp_dev,
                            float* code_bits_dev, float* imp_bits_dev, const int2* cand_host = nullptr, const float* src_levels = nullptr,
                            const int32_t* protect = nullptr) {
    const EstimateTotals r = estimate_totals(c->est_dev, K);
    const Candidates cd{c->cand_dev, src_levels, protect};
    if (cand_host) {
        const int rc = enqueue_candidates(c, K, cand_host, cd);  // ev_est is recorded again below for the results
        if (rc) return rc;
        imp_dev = c->cand_levels_dev;
    }
    {
        NetDesc& n = c->imp;
        cudaStream_t s = n.stream;
        LIC360_CUDA(cudaMemsetAsync(r.err + K, 0xFF, K * sizeof(*r.err), s));
        int rc = run_encoder_net(c, false, K, code_dev, mask_dev, imp_dev);
        if (rc) return rc;
        imp_bits_kernel<<<dim3(n.bits_blocks, K), BITS_THREADS, 0, s>>>(n.frame[12], imp_dev, n.idx_dev, imp_bits_dev, n.bits_partial_dev,
                                                                        n.count_partial_dev, r.err + K, n.H, n.W);
        LAUNCH_CHECK();
        bits_sum_kernel<<<K, BITS_THREADS, 0, s>>>(n.bits_partial_dev, n.count_partial_dev, n.bits_blocks, r.bits + K, r.count + K);
        LAUNCH_CHECK();
        LIC360_CUDA(cudaEventRecord(c->ev_est, s));
    }
    {
        NetDesc& n = c->code;
        cudaStream_t s = n.stream;
        LIC360_CUDA(cudaMemsetAsync(r.err, 0xFF, K * sizeof(*r.err), s));
        int rc = run_encoder_net(c, true, K, code_dev, mask_dev, imp_dev, cand_host ? &cd : nullptr);
        if (rc) return rc;
        if (cand_host)
            gmm_bits_kernel<true><<<dim3(n.bits_blocks, K), BITS_THREADS, 0, s>>>(n.frame[12], code_dev, nullptr, cd, n.idx_dev, n.steps_dev,
                                                                                  n.row_off_dev, code_bits_dev, n.bits_partial_dev,
                                                                                  n.count_partial_dev, r.err, n.G, n.H, n.W, kGmmS2);
        else
            gmm_bits_kernel<false><<<dim3(n.bits_blocks, K), BITS_THREADS, 0, s>>>(n.frame[12], code_dev, mask_dev, cd, n.idx_dev, n.steps_dev,
                                                                                   n.row_off_dev, code_bits_dev, n.bits_partial_dev,
                                                                                   n.count_partial_dev, r.err, n.G, n.H, n.W, kGmmS2);
        LAUNCH_CHECK();
        bits_sum_kernel<<<K, BITS_THREADS, 0, s>>>(n.bits_partial_dev, n.count_partial_dev, n.bits_blocks, r.bits, r.count);
        LAUNCH_CHECK();
        LIC360_CUDA(cudaStreamWaitEvent(s, c->ev_est, 0));
        LIC360_CUDA(cudaMemcpyAsync(c->est_host, c->est_dev, estimate_bytes(K), cudaMemcpyDeviceToHost, s));
    }
    return LIC360_OK;
}

// lic360_codec_estimate (K = 1, no suffix), lic360_codec_estimate_batch (suffix "latent") and lic360_codec_estimate_candidates (suffix
// "candidate", the table in cand_host); the maps may be NULL
static int estimate_latents(lic360_codec* c, int K, const float* code_dev, const float* mask_dev, const float* imp_dev,
                            float* code_bits_dev, float* imp_bits_dev, double* bits_host, long long* counts_host, const char* suffix,
                            const int2* cand_host = nullptr, const int32_t* protect = nullptr) {
    DeviceGuard guard(c->device);
    int rc = begin_latents(c, guard, K);
    if (rc) return rc;
    const auto t0 = clk::now();
    rc = enqueue_estimate(c, K, code_dev, mask_dev, imp_dev, code_bits_dev, imp_bits_dev, cand_host, imp_dev, protect);
    // both streams are drained on every path: the caller may reuse the inputs and the maps as soon as the call returns
    const auto tw = clk::now();
    const cudaError_t e_imp = cudaStreamSynchronize(c->imp.stream);
    const cudaError_t e_code = cudaStreamSynchronize(c->code.stream);
    c->t_gpu_wait = ms_since(tw);
    c->t_total = ms_since(t0);
    if (rc) return rc;
    LIC360_CUDA(e_imp);
    LIC360_CUDA(e_code);
    // the error encode reports for the first bad latent, with its message: the importance stream is coded (and checked) first
    const EstimateTotals r = estimate_totals(c->est_host, K);
    for (int k = 0; k < K; k++)
        for (int sid : {1, 0}) {
            const unsigned long long e = r.err[sid * K + k];
            if (e == kNoError) continue;
            coder_row_error(sid, (int)(e >> 32), (unsigned)e);
            if (suffix) add_index_suffix(suffix, k);
            return LIC360_ERR_CODER;
        }
    for (int k = 0; k < K; k++)
        for (int sid = 0; sid < 2; sid++) {
            bits_host[2 * k + sid] = r.bits[sid * K + k];
            if (counts_host) counts_host[2 * k + sid] = r.count[sid * K + k];
        }
    return LIC360_OK;
}

int lic360_codec_estimate(lic360_codec* c, const float* code_dev, const float* mask_dev, const float* imp_dev, float* code_bits_dev,
                          float* imp_bits_dev, double* bits_host) {
    LIC360_CHECK_ARG(c && code_dev && mask_dev && imp_dev && code_bits_dev && imp_bits_dev && bits_host, "bad arguments");
    return estimate_latents(c, 1, code_dev, mask_dev, imp_dev, code_bits_dev, imp_bits_dev, bits_host, nullptr, nullptr);
}

int lic360_codec_estimate_batch(lic360_codec* c, int K, const float* code_dev, const float* mask_dev, const float* imp_dev,
                                float* code_bits_dev, float* imp_bits_dev, double* bits_host, long long* counts_host) {
    LIC360_CHECK_ARG(K >= 1, "K must be at least 1");
    LIC360_CHECK_ARG(c && code_dev && mask_dev && imp_dev && bits_host && counts_host, "bad arguments");
    LIC360_CHECK_BATCH(c, K);
    return estimate_latents(c, K, code_dev, mask_dev, imp_dev, code_bits_dev, imp_bits_dev, bits_host, counts_host, "latent");
}

int lic360_codec_estimate_candidates(lic360_codec* c, int K, const float* code_dev, const float* imp_dev, const int32_t* protect_dev, int J,
                                     const int* cand_latent_host, const int* cand_offset_host, double* bits_host, long long* counts_host) {
    LIC360_CHECK_ARG(K >= 1, "K must be at least 1");
    LIC360_CHECK_ARG(J >= 1, "J must be at least 1");
    LIC360_CHECK_ARG(c && code_dev && imp_dev && cand_latent_host && cand_offset_host && bits_host && counts_host, "bad arguments");
    LIC360_CHECK_BATCH(c, J);
    std::vector<int2> tab;
    const int rc = candidate_table(__func__, K, J, cand_latent_host, cand_offset_host, tab);
    if (rc) return rc;
    return estimate_latents(c, J, code_dev, nullptr, imp_dev, nullptr, nullptr, bits_host, counts_host, "candidate", tab.data(), protect_dev);
}

int lic360_imp_levels_to_mask(const float* levels_dev, int h, int w, const int* offsets_host, int K, float* levels_out_dev,
                              float* mask_out_dev, void* stream) {
    return lic360_imp_levels_to_mask_protected(levels_dev, h, w, offsets_host, K, nullptr, levels_out_dev, mask_out_dev, stream);
}

// the launches of the candidate maps: candidate j is source latent src_host[j] (0 when src_host is NULL) at offset offsets_host[j]
static int enqueue_levels_to_mask(const float* levels_dev, int h, int w, const int32_t* protect_dev, int J, const int* src_host,
                                  const int* offsets_host, float* levels_out_dev, float* mask_out_dev, void* stream) {
    const int n = 48 * 4 * h * w;
    for (int j0 = 0; j0 < J; j0 += 32) {  // 32 candidates per launch (the table travels as a kernel parameter)
        LevelOffsets off;
        const int nj = std::min(32, J - j0);
        for (int j = 0; j < nj; j++) {
            off.k[j] = offsets_host[j0 + j];
            off.src[j] = src_host ? src_host[j0 + j] : 0;
        }
        imp_levels_to_mask_kernel<<<dim3(std::max(1, stream_grid(n, 256) / nj), nj), 256, 0, as_stream(stream)>>>(
            levels_dev, protect_dev, h, w, off, levels_out_dev + (size_t)j0 * h * w, mask_out_dev + (size_t)j0 * n);
        LAUNCH_CHECK();
    }
    return LIC360_OK;
}

int lic360_imp_levels_to_mask_protected(const float* levels_dev, int h, int w, const int* offsets_host, int K, const int32_t* protect_dev,
                                        float* levels_out_dev, float* mask_out_dev, void* stream) {
    LIC360_CHECK_ARG(K >= 1, "K must be at least 1");
    LIC360_CHECK_ARG(levels_dev && offsets_host && levels_out_dev && mask_out_dev, "bad arguments");
    LIC360_CHECK_ARG(h > 0 && w > 0 && (long long)48 * 4 * h * w <= 0x7fffffffLL, "bad importance map size");
    for (int j = 0; j < K; j++) LIC360_CHECK_ARG(offsets_host[j] >= 0, "offsets must not be negative");
    return enqueue_levels_to_mask(levels_dev, h, w, protect_dev, K, nullptr, offsets_host, levels_out_dev, mask_out_dev, stream);
}

int lic360_imp_levels_to_mask_batch(const float* levels_dev, int K, int h, int w, const int32_t* protect_dev, int J,
                                    const int* cand_latent_host, const int* cand_offset_host, float* levels_out_dev, float* mask_out_dev,
                                    void* stream) {
    LIC360_CHECK_ARG(K >= 1, "K must be at least 1");
    LIC360_CHECK_ARG(J >= 1, "J must be at least 1");
    LIC360_CHECK_ARG(levels_dev && cand_latent_host && cand_offset_host && levels_out_dev && mask_out_dev, "bad arguments");
    LIC360_CHECK_ARG(h > 0 && w > 0 && (long long)48 * 4 * h * w <= 0x7fffffffLL, "bad importance map size");
    for (int j = 0; j < J; j++) {
        LIC360_CHECK_ARG(cand_latent_host[j] >= 0 && cand_latent_host[j] < K, "cand_latent must lie in [0, K)");
        LIC360_CHECK_ARG(cand_offset_host[j] >= 0, "offsets must not be negative");
    }
    return enqueue_levels_to_mask(levels_dev, h, w, protect_dev, J, cand_latent_host, cand_offset_host, levels_out_dev, mask_out_dev,
                                  stream);
}

// stream stream_id of latent k of the last encode (none before the first encode and after a failed one)
static long copy_stream(lic360_codec* c, int k, int stream_id, uint8_t* out, long cap) {
    const std::vector<uint8_t>& b = c->enc_out[2 * (size_t)k + (stream_id ? 1 : 0)].bytes;
    const long n = (long)b.size();
    if (out && cap > 0) memcpy(out, b.data(), (size_t)std::min(n, cap));
    return n;
}

long lic360_codec_stream_size(lic360_codec* c, int stream_id) {
    return copy_stream(c, 0, stream_id, nullptr, 0);
}

long lic360_codec_stream_copy(lic360_codec* c, int stream_id, uint8_t* out, long cap) {
    return copy_stream(c, 0, stream_id, out, cap);
}

long lic360_codec_batch_stream_size(lic360_codec* c, int k, int stream_id) {
    return lic360_codec_batch_stream_copy(c, k, stream_id, nullptr, 0);
}

long lic360_codec_batch_stream_copy(lic360_codec* c, int k, int stream_id, uint8_t* out, long cap) {
    if (!c || (stream_id != 0 && stream_id != 1)) { set_error("codec: bad arguments to a batch stream accessor"); return -1; }
    if (k < 0 || k >= c->enc_k) {
        set_error("codec: latent %d is not in the last encode (%d latents)", k, c->enc_k);
        return -1;
    }
    return copy_stream(c, k, stream_id, out, cap);
}

// importance stream: wait for the rows of step p without synchronising the stream (a later kernel of the step graph may still be
// running).  An acquire load: the rows the device wrote before raising the flag are read (non-atomically) by the coder right after.
static int wait_rows(lic360_codec* c, NetDesc& n, int p) {
    const auto t0 = clk::now();
    auto ready = [&]() { return __atomic_load_n(n.flag_host, __ATOMIC_ACQUIRE) == p + 1; };
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
    return LIC360_OK;
}

// code stream: called by the tagged row decoder every few thousand polls of a row that has not arrived.  The give-up conditions of
// wait_rows, and a negative flag: a chain CTA gave up waiting for the other nets' clusters
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

// code stream: spin until the first row of step sc.p carries its tag (the time until then is waiting for the GPU; the coder decodes the
// later rows as they arrive)
static int wait_first_row(StallCtx& sc) {
    const uint16_t* meta = sc.n->rows_step_host + 7;
    for (unsigned spins = 1; ((__atomic_load_n(meta, __ATOMIC_ACQUIRE) >> 4) & 15) != (unsigned)wf_row_tag(sc.p); spins++) {
#if defined(__x86_64__)
        __builtin_ia32_pause();
#endif
        if ((spins & 0x3FFF) == 0) {
            const int rc = rows_stalled(&sc);
            if (rc) return rc;
        }
    }
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
// The state every decode of a stream starts from: host flags and publication tags, timers, the trace vectors, the engine's frames and
// the device counters (enqueued on the stream's CUDA stream)
static int decode_reset(NetDesc& n) {
    cudaStream_t s = n.stream;
    for (int i = 0; i < 64; i++) n.flag_host[i] = 0;
    memset(n.rows_step_host, 0, (size_t)n.max_len * n.row_bytes);  // publication tags of a previous decode must not match step 0
    n.t_host_coder = 0; n.t_gpu_wait = 0;
    for (int i = 0; i < 5; i++) n.t_kernel[i] = 0;
    n.step_wait_us.clear(); n.step_decode_us.clear(); n.step_levels_us.clear();
    LIC360_CUDA(wf_clear(n.wf, s));
    LIC360_CUDA(cudaMemsetAsync(n.ctr_dev, 0xFF, sizeof(int), s));  // -1: the scatter kernel of step p makes it p
    LIC360_CUDA(cudaMemsetAsync(n.done_dev, 0, sizeof(int), s));
    LIC360_CUDA(cudaMemsetAsync(n.arrived_dev, 0, sizeof(int), s));
    LIC360_CUDA(cudaMemsetAsync(n.sync_dev, 0, sizeof(int), s));
    return LIC360_OK;
}

static int decode_stream_persistent(lic360_codec* c, NetDesc& n) {
    cudaStream_t s = n.stream, side = n.side;
    int rc = decode_reset(n);
    if (rc) return rc;
    memset(n.syms_host, 0, (size_t)n.max_len * sizeof(float));  // tag 0 = not published
    __atomic_store_n(n.go_host, -1, __ATOMIC_RELEASE);
    PersistStop stop{n.go_host};
    const bool trace_file = getenv("LIC360_WF_TRACE_FILE") != nullptr;
    LIC360_CUDA(cudaMemsetAsync(n.go_dev, 0xFF, sizeof(int), s));
    LIC360_CUDA(cudaMemsetAsync(n.old_done_dev, 0, sizeof(int), s));
    LIC360_CUDA(cudaMemsetAsync(n.scat_done_dev, 0, 4 * sizeof(int), s));
    LIC360_CUDA(cudaEventRecord(n.ev_fork, s));
    LIC360_CUDA(cudaStreamWaitEvent(side, n.ev_fork, 0));
    LIC360_CUDA(wf_launch_old(n.wf, 0, side, false, 0, n.old_done_dev, n.scat_done_dev));  // old terms of step 0 (all zero; keeps the protocol uniform)
    WfPersist ps;
    memset(&ps, 0, sizeof(ps));
    ps.syms = n.syms_host; ps.go_host = n.go_host; ps.go_dev = n.go_dev; ps.old_done = n.old_done_dev; ps.ctr = n.ctr_dev; ps.scat_done = n.scat_done_dev;
    const TileIn t = tile_input(true);
    ps.bias = t.bias; ps.scale = t.scale;
    LIC360_CUDA(wf_launch_chain(n.wf, s, wf_rows(c, n), &ps));
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
        rc = wait_first_row(sc);
        if (rc) return rc;
        n.t_gpu_wait += ms_since(tw);
        if (trace_file) n.step_wait_us.push_back((float)(ms_since(tw) * 1e3));
        auto th = clk::now();
        rc = coder_decode_packed_gmm_tagged(n.coder, n.rows_step_host, n.steps[p].len, n.syms_host, wf_row_tag(p), rows_stalled, &sc,
                                            p + 1 < n.nsteps ? (unsigned)wf_row_tag(p) : 0u);  // symbol words tagged too: the chain kernel polls
                                            // them one by one (not the last step's: the final scatter reads plain floats)
        n.t_host_coder += ms_since(th);
        if (trace_file) n.step_decode_us.push_back((float)(ms_since(th) * 1e3));
        if (rc) return rc;
    }
    LIC360_CUDA(cudaEventRecord(n.ev_join, side));
    LIC360_CUDA(cudaStreamWaitEvent(s, n.ev_join, 0));
    // the final TileInput of lic360_demo.py:236: behind the chain kernel in stream order; the device step counter is nsteps - 1
    return launch_scatter(c, n, true, s);
}

// The wavefront loop of one bitstream.  is_code: before step p the importance levels of every 2x2 cell the slab touches
// must be decoded (cells on importance diagonals <= min(p, H+W-2)/2): the loop waits on c->imp_ready, which the
// importance loop (running concurrently on another host thread and CUDA stream) publishes.
static int decode_stream(lic360_codec* c, NetDesc& n, bool is_code) {
    if (is_code && c->mode == 2) return decode_stream_persistent(c, n);
    cudaStream_t s = n.stream;
    int rc = decode_reset(n);
    if (rc) return rc;
    const bool trace_file = getenv("LIC360_WF_TRACE_FILE") != nullptr;
    LIC360_CUDA(wf_launch_old(n.wf, 1, s));  // old terms of step 0 = counter (-1) + 1 (all zero, but it keeps the schedule uniform)
    if (debug_sync()) LIC360_CUDA(cudaStreamSynchronize(s));
    for (int p = 0; p < n.nsteps; p++) {
        auto tw = clk::now();
        if (is_code) { rc = wait_levels(c, n, p); if (rc) return rc; }
        if (c->mode != 1) {
            if (trace_file && is_code) n.step_levels_us.push_back((float)(ms_since(tw) * 1e3));
            LIC360_CUDA(cudaGraphLaunch(n.graph, s));
            g_launches += n.graph_nodes;
            if (!is_code) {
                rc = wait_rows(c, n, p);
                if (rc) return rc;
            }
        } else {
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
        if (is_code) {
            StallCtx sc{c, &n, p, clk::now()};
            rc = wait_first_row(sc);
            if (rc) return rc;
            n.t_gpu_wait += ms_since(th);
            if (trace_file) n.step_wait_us.push_back((float)(ms_since(tw) * 1e3));
            th = clk::now();
            rc = coder_decode_packed_gmm_tagged(n.coder, n.rows_step_host, len, n.syms_host, wf_row_tag(p), rows_stalled, &sc);
        } else {
            rc = coder_decode_packed_imp(n.coder, n.rows_step_host, len, n.syms_host);
        }
        n.t_host_coder += ms_since(th);
        if (trace_file && is_code) n.step_decode_us.push_back((float)(ms_since(th) * 1e3));
        if (rc) return rc;
    }
    rc = launch_scatter(c, n, is_code, s);  // the symbols of the last step (the final TileInput of lic360_demo.py:236,285)
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
    c->enc_k = 0;  // the streams of the last encode are no longer returned by the batch accessors
    c->imp_ready.store(0);
    c->abort_flag.store(0);
    DecodeTrace trace;
    rc = decode_trace_begin(c, trace);
    if (rc) return rc;
    // Admission first: a decode queues here when the device already runs as many decodes as it can hold, and a low-latency decode takes
    // the device for itself.  Everything below -- graph capture and instantiation included, which may allocate and therefore wait for the
    // device -- runs inside the slot: a thread that blocks in the driver while ANOTHER decode's persistent kernel waits for its host
    // would stall that decode's importance-stream launches (observed as a 20 s "levels" time-out under a 7-thread stress).
    std::unique_ptr<ChainSlot> slot;
    if (c->mode != 1) slot.reset(new ChainSlot(c->device, c->chain_cap, c->mode == 2 ? c->chain_cap : 1));
    if (c->mode != 1) {  // both step graphs exist before the second host thread starts (the persistent code stream needs none)
        rc = build_step_graph(c, c->imp, false);
        if (rc == LIC360_OK && c->mode != 2) rc = build_step_graph(c, c->code, true);
        if (rc) return rc;
    }
    lic360_coder_start_decoder_mem(c->imp.coder, imp_bytes, n_imp);
    lic360_coder_start_decoder_mem(c->code.coder, code_bytes, n_code);
    // ---- importance stream (lic360_demo.py:272-290) and code stream (:220-238), concurrently in the pipelined mode: the
    // code stream only reads importance levels that are already decoded (decode_stream).  Serialized in profile mode.
    int rc_imp = LIC360_OK;
    char imp_err[256] = {0};  // error text of the importance loop's thread (set_error is thread-local)
    auto imp_loop = [&]() {
        cudaSetDevice(c->device);
        rc_imp = decode_stream(c, c->imp, false);
        if (rc_imp) {
            snprintf(imp_err, sizeof(imp_err), "%s", lic360_last_error());
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
        if (rc && rc_imp && strstr(imp_err, "aborted (the other stream failed)")) {
            set_error("%s", code_err.c_str());
            drain(c);
            return rc;
        }
    } else {
        imp_loop();
        if (rc_imp == LIC360_OK) rc = decode_stream(c, c->code, true);
    }
    if (rc_imp) { set_error("%s", imp_err); drain(c); return rc_imp; }
    if (rc) { drain(c); return rc; }
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
    decode_trace_report(c, trace);
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

int lic360_codec_engine_info(lic360_codec* c, int stream_id, int* out, int n) {
    LIC360_CHECK_ARG(c && out && (stream_id == 0 || stream_id == 1), "bad arguments");
    const NetDesc& d = stream_id == 0 ? c->code : c->imp;
    const WfEngine& e = d.wf;
    int tail_rounds = 0;
    if (e.chain4 && n > 12) {
        std::vector<int32_t> idx(2 * (size_t)d.H * d.W), plan(d.H + d.W);
        lic360_code_contex(d.H, d.W, idx.data(), plan.data());
        tail_rounds = wf_tail_rounds(e, idx.data(), d.steps.data());
    }
    const int v[13] = {e.chain1 ? 2 : e.chain4 ? 1 : 0, e.chain1 && e.c1_dsm, e.cluster, e.chain_threads, (int)e.chain_smem, e.max_len,
                       e.chain1 ? e.c1_lenp : 0, e.chain1 ? e.c1_kpc : 0, e.chain_tasks, e.old4 ? 4 : 1, e.parts4,
                       e.dev.parts, tail_rounds};
    for (int i = 0; i < n && i < 13; i++) out[i] = v[i];
    return LIC360_OK;
}

}  // extern "C"
