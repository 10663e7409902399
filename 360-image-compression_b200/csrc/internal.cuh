// Internal (non-ABI) declarations shared between the op entry points and the fused codec pipeline.
#pragma once
#include <cuda.h>
#include "common.cuh"

namespace lic360 {

struct ConvArgs {
    const float* x; const float* wp; const float* wq; const float* bias; const float* slope; const float* resid;
    float* out;
    int N, Cin, H, W, Cout, G, cin_g, cout_g, cpg4, nchunk, per, has_q;
};

// one wavefront step as seen by device code: slab [start, start+len) of the index plan, step number psum
struct StepDesc { int psum, start, len, pad; };

int fill_conv_args(ConvArgs& a, const float* x, const float* wp, const float* wq, const float* bias, const float* slope,
                   const float* resid, float* out, int N, int Cin, int H, int W, int Cout, int G, int constrain, int nsets);
// allow_mma: the per-op CconvEc honours LIC360_EC_MMA; the codec passes false, its streams need the canonical P pass
cudaError_t launch_cconv_ec(const ConvArgs& a, cudaStream_t s, bool allow_mma);
// conv_mma.cu: opt-in (LIC360_EC_MMA=1) tensor-core form of the encoder's old-term pass, mma.sync TF32 with a 3-way split
bool cconv_ec_mma_enabled();
cudaError_t launch_cconv_ec_mma(const ConvArgs& a, cudaStream_t s);
// explicit step (steps == nullptr) or step read on the device from steps[*ctr + ctr_off] (graph replay; grid sized for max_len)
cudaError_t launch_cconv_dc(const ConvArgs& a, const int32_t* idx_dev, int start, int len, int psum, const StepDesc* steps,
                            const int* ctr, int max_len, cudaStream_t s);

}  // namespace lic360
