/*
 * lic360_b200 -- C-ABI of the B200-native LIC360 context-model entropy path.
 *
 * This header is the drop-in boundary.  Every entry point replaces one method of the reference's pybind11
 * module `lic360` (/root/reference/extension/main.cpp:4-178); the file:line each one replaces is cited.
 * Conventions
 *   - plain pointers and sizes only; all tensors are dense fp32 NCHW unless stated; `*_dev` = device memory,
 *     `*_host` = host memory; the caller owns every buffer (the reference's op-owned `top_data_` caching,
 *     base_opt.hpp:43-72, lives in the host-side mirror, 360-image-compression_b200/lic360/).
 *   - `stream` is a cudaStream_t passed as void* (the reference captures one stream per op at construction,
 *     base_opt.hpp:20-23; here it is per call so several images can be in flight per GPU).
 *   - return value: 0 on success, non-zero on error; lic360_last_error() returns a thread-local message.
 *     (The reference only printf()s CUDA errors, caffe_cuda_macro.h:21-26, and throws C strings from the
 *     coder, ArithmeticCoder.cpp:17-49; the Python mirror turns a non-zero status into RuntimeError.)
 *   - stateful wavefront ops take the step number `psum` explicitly (the reference keeps a private counter
 *     `plan_sum_` per op, cconv_dc.hpp:21, tile_*.hpp); the index plan is the pair (idx_dev, plan_host) of
 *     CodeContexOp (code_contex_cuda.cu:11-32).
 */
#ifndef LIC360_B200_H
#define LIC360_B200_H
#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define LIC360_OK 0
#define LIC360_ERR_ARG 1
#define LIC360_ERR_CUDA 2
#define LIC360_ERR_CODER 3

const char* lic360_last_error(void);
int lic360_version(void);
/* number of kernels this library has launched in the calling process (bench.py's "gpu_launches") */
long long lic360_launch_count(void);

/* ---- CodeContexOp.forward (main.cpp:80-84, code_contex_cuda.cu:11-38) ------------------------------------
 * idx_host: 2*H*W int32 (row plane, column plane), plan_host: H+W int32. Host-only; copy idx to the device. */
int lic360_code_contex(int H, int W, int32_t* idx_host, int32_t* plan_host);
/* slab [start, start+len) of step psum (cconv_dc_cuda.cu:113-117) */
int lic360_slab(const int32_t* plan_host, int H, int W, int G, int psum, int* start, int* len);

/* ---- context convolution: weight packing ------------------------------------------------------------------
 * The kernels consume weights re-laid out per 4-channel output chunk with the context mask applied
 * (mask rule cconv_ec_cuda.cu:71 == mask_constrain_cuda.cu:24,38). Call once per weight update.
 *   w_dev    : (nsets, Cout, Cin, 5, 5) reference layout (CconvEc.py:67,87)
 *   wp_dev   : lic360_cconv_wp_floats() floats  (strictly-earlier-wavefront terms)
 *   wq_dev   : lic360_cconv_wq_floats() floats  (same-wavefront terms; all zero for constrain 5)            */
size_t lic360_cconv_wp_floats(int nsets, int Cin, int Cout, int G);
size_t lic360_cconv_wq_floats(int nsets, int Cin, int Cout, int G);
int lic360_cconv_pack(const float* w_dev, float* wp_dev, float* wq_dev, int nsets, int Cin, int Cout, int G,
                      int ksize, int constrain, void* stream);

/* ---- CconvEcOp.forward / forward_act / forward_batch / forward_act_batch (main.cpp:96-102,
 *      cconv_ec_cuda.cu:99-121,170-192,242-265,317-339) ------------------------------------------------------
 * x (N,Cin,H,W) -> out (N,Cout,H,W); weight set = n / (N/nsets); slope_dev == NULL: no PReLU;
 * resid_dev != NULL: out += resid after the activation (the `y + x` of EntropyResidualBlockD*Fast,
 * lic360_demo.py:39-41,61-63, fused).                                                                       */
int lic360_cconv_ec_forward(const float* x_dev, const float* wp_dev, const float* wq_dev, const float* bias_dev,
                            const float* slope_dev, const float* resid_dev, float* out_dev, int N, int Cin, int H,
                            int W, int Cout, int G, int constrain, int nsets, void* stream);

/* ---- CconvDcOp.forward* (main.cpp:86-94, cconv_dc_cuda.cu:108-137,193-224,280-312,368-398) ---------------
 * One wavefront step: recomputes only the slab entries of the persistent frame out (N,Cout,H,W); zeroes it at
 * psum == 0 (cconv_dc_cuda.cu:125). resid_dev != NULL fuses TileAdd (tile_add_cuda.cu:22-38).               */
int lic360_cconv_dc_forward(const float* x_dev, const float* wp_dev, const float* wq_dev, const float* bias_dev,
                            const float* slope_dev, const float* resid_dev, float* out_dev, int N, int Cin, int H,
                            int W, int Cout, int G, int constrain, int nsets, const int32_t* idx_dev,
                            const int32_t* plan_host, int psum, void* stream);

/* ---- TileExtractOp.forward / forward_batch (main.cpp:104-110, tile_extract_cuda.cu:48-98,120-151) --------
 * *count_host receives the value of the reference's CPU int tensor top_num_.                                */
int lic360_tile_extract(const float* x_dev, float* out_dev, int N, int C, int H, int W, int G, int label,
                        const int32_t* idx_dev, const int32_t* plan_host, int psum, int* count_host, void* stream);
int lic360_tile_extract_batch(const float* x_dev, float* out_dev, int N, int C, int H, int W, int G,
                              const int32_t* idx_dev, const int32_t* plan_host, int psum, int* count_host,
                              void* stream);
/* ---- TileInputOp.forward (main.cpp:112-117, tile_input_cuda.cu:46-76) ------------------------------------ */
int lic360_tile_input(const float* in_dev, float* frame_dev, int N, int G, int H, int W, float bias, float scale,
                      int rep, const int32_t* idx_dev, const int32_t* plan_host, int psum, void* stream);
/* ---- TileAddOp.forward (main.cpp:119-124, tile_add_cuda.cu:40-61): y[slab] += x[slab] in place ----------- */
int lic360_tile_add(float* y_dev, const float* x_dev, int N, int C, int H, int W, int G, const int32_t* idx_dev,
                    const int32_t* plan_host, int psum, void* stream);

/* ---- EntropyGmmTableOp.forward / forward_batch (main.cpp:126-130, entropy_gmm_table_cuda.cu:109-191) -----
 * weight/delta/mean: rows x ng; weight is soft-maxed and delta clamped IN PLACE like the reference
 * (:29-57); out: rows x (nstep+1) floats holding integers.  For forward_batch pass the three planes of the
 * TileExtractBatch buffer (plane stride = N*C*H*W/3 floats, :167).                                          */
int lic360_gmm_table(float* weight_dev, float* delta_dev, const float* mean_dev, float* out_dev, int rows, int ng,
                     int nstep, float bias, int total_region, float beta, void* stream);
/* ---- EntropyTableOp.forward (main.cpp:150-153, entropy_table_cuda.cu:78-96) ------------------------------ */
int lic360_entropy_table(const float* in_dev, float* out_dev, int rows, int nstep, int total_region, void* stream);

/* ---- EntropyGmmOp.forward / backward (main.cpp:67-71, entropy_gmm_cuda.cu:70-124) ------------------------ */
int lic360_entropy_gmm_forward(const float* weight_dev, const float* delta_dev, const float* mean_dev,
                               const float* label_dev, float* wdiff_dev, float* ddiff_dev, float* mdiff_dev,
                               float* ldiff_dev, float* loss_dev, int S, int ng, void* stream);
int lic360_entropy_gmm_backward(float* wdiff_dev, float* ddiff_dev, float* mdiff_dev, float* ldiff_dev,
                                const float* top_diff_dev, int S, int ng, void* stream);

/* ---- ContextReshapeOp (main.cpp:61-65, context_reshape_cuda.cu:43-110) ----------------------------------- */
int lic360_context_reshape(const float* in_dev, float* out_dev, int N, int C, int H, int W, int G, int backward,
                           void* stream);
/* ---- ContexShiftOp (main.cpp:55-59, contex_shift_cuda.cu:66-144). H is the un-skewed height.
 * mode 0: scatter (N,C,H,W)->(N,C,H+W+G-2,W) (forward, and backward of inv, which zero-fills first, :128)
 * mode 1: gather back (forward of inv, backward of non-inv).                                                */
int lic360_contex_shift(const float* in_dev, float* out_dev, int N, int C, int H, int W, int cpn, int mode,
                        int zero_fill, void* stream);
/* ---- MaskConstrainOp.forward/backward (main.cpp:73-78, mask_constrain_cuda.cu:43-94): in place ----------- */
int lic360_mask_constrain(float* w_dev, int Cout, int Cin, int ksize, int G, int constrain, void* stream);

/* ---- QuantOp (main.cpp:42-46, quant_cuda.cu:136-169 forward, :237-266 backward, :119-134 level repair) ---
 * levels_dev (C x L) receives exp()-ed levels, qint_dev int32 indices, count_dev (C x L) is zeroed then
 * decremented per hit (:149,56,74). q_dev may be NULL (ntop == 1).                                          */
int lic360_quant_forward(const float* x_dev, const float* wb_dev, float* levels_dev, float* y_dev, float* q_dev,
                         int32_t* qint_dev, float* count_dev, int N, int C, int H, int W, int L, void* stream);
int lic360_quant_update_weight(float* wb_dev, float* ncount_dev, int C, int L, float decay, void* stream);
int lic360_quant_backward(const float* top_diff0_dev, const float* top_diff1_dev, const float* x_dev,
                          const float* y_dev, const int32_t* qint_dev, const float* levels_dev,
                          float* bottom_diff_dev, float* weight_diff_dev, int N, int C, int H, int W, int L,
                          float top_alpha, void* stream);
/* ---- DquantOp.forward (main.cpp:145-148, dquant_cuda.cu:49-69) -------------------------------------------- */
int lic360_dquant_forward(const float* q_dev, const float* mask_dev, const float* wb_dev, float* cum_dev,
                          float* y_dev, int N, int C, int H, int W, int L, void* stream);

/* ---- ImpMapOp (main.cpp:30-34, imp_map_cuda.cu:112-136 forward, :239-298 backward) -----------------------
 * mask_dev may be NULL (ntop == 1). constrain/alpha_t initialisation: imp_map_cuda.cu:27-69.                */
int lic360_imp_map_forward(const float* x_dev, const float* imp_dev, float* out_dev, float* mask_dev, int N, int C,
                           int H, int W, int levels, void* stream);
int lic360_imp_map_init(float* constrain_dev, float* alpha_t_dev, int N, int H, float alpha, float rt, float sc,
                        float sw, void* stream);
int lic360_imp_map_backward(const float* top_diff_dev, const float* imp_dev, const float* sphere_constrain_dev,
                            const float* alpha_t_dev, float* data_diff_dev, float* imp_diff_dev, int N, int C,
                            int H, int W, int levels, float gamma, int imp_kernel, void* stream);
/* ---- Imp2maskOp.forward (main.cpp:160-163, imp2mask_cuda.cu:40-57) ---------------------------------------- */
int lic360_imp2mask(const float* in_dev, float* out_dev, int N, int C, int H, int W, int levels, void* stream);
/* ---- ScaleOp.forward (main.cpp:155-158, scale_cuda.cu:32-48) ---------------------------------------------- */
int lic360_scale(const float* in_dev, float* out_dev, size_t n, float bias, float scale, void* stream);

/* ---- SpherePadOp (main.cpp:12-16, sphere_pad_cuda.cu:67-105 forward, :172-204 backward) ------------------
 * NC = N*C planes. forward: in (NC,H,W) -> out (NC,H+2p,W+2p). inplace: data (NC,Hp,Wp) already padded.     */
int lic360_sphere_pad(const float* in_dev, float* out_dev, int NC, int H, int W, int pad, void* stream);
int lic360_sphere_pad_inplace(float* data_dev, int NC, int Hp, int Wp, int pad, void* stream);
int lic360_sphere_pad_backward(float* bottom_dev, float* top_dev, int NC, int H, int W, int pad, int inplace,
                               void* stream);
/* ---- SphereTrimOp fwd == bwd (main.cpp:18-22, sphere_trim_cuda.cu:28-63): zero the border in place ------- */
int lic360_sphere_trim(float* data_dev, int NC, int H, int W, int pad, void* stream);
/* ---- SphereCutEdgeOp (main.cpp:24-28, sphere_cut_edge_cuda.cu:43-97) -------------------------------------- */
int lic360_sphere_cut_edge(const float* in_dev, float* out_dev, int NC, int H, int W, int pad, int backward,
                           void* stream);
/* ---- SphereLatScaleOp fwd == bwd kernel (main.cpp:48-53, sphere_lat_scale_cuda.cu:40-85) ------------------ */
int lic360_sphere_lat_scale(const float* in_dev, const float* weight_dev, float* out_dev, int NC, int H, int W,
                            int npart, void* stream);
/* ---- DtowOp (main.cpp:36-40, dtow_cuda.cu:77-175) -- SURVEY s8(f)-1 "next" row --------------------------- */
int lic360_dtow(const float* in_dev, float* out_dev, int N, int C, int H, int W, int stride, int d2w, void* stream);

/* ---- ProjectsOp (main.cpp:6-10, projects.hpp:6-34, projects_cuda.cu) -- SURVEY s8(f)-2 "next" row: MultiProject --------------
 * The 14 rectilinear viewports (h_out x w_out each) of an ERP image, bilinear or nearest; used by `--test` for viewport PSNR / SSIM
 * (lic360_demo.py:424-441) and by the training loss (trainDDP_IMP_ENT.py:33-36).
 *   init    : rays of all viewport pixels, xyz_dev (14, h_out*w_out, 3); theta14 / phi14 / fov in units of pi as the reference
 *             constructor takes them (projects.hpp:8-19, projects_cuda.cu:84-126)
 *   update  : ERP sampling coordinates for an H x W input, tf_dev (14, h_out*w_out, 2) = (x, y) (projects_cuda.cu:51-68,127-136);
 *             call when the input size changes (projects_opt::reshape)
 *   forward : in (NC = N*C planes, H, W) -> out (14*N, C, h_out, w_out), viewport-major: out[(v*NC + plane)*h_out*w_out + ps] (:181-252)
 *   backward: top_diff (same layout as out) -> bottom_diff (NC, H, W) and the accumulated weights count (NC, H, W), both zeroed
 *             first (:257-329; fp32 atomics, so the sums are order-dependent in their last bits like the reference's)        */
int lic360_projects_init(float* xyz_dev, int h_out, int w_out, const float* theta14, const float* phi14, float fov, void* stream);
int lic360_projects_update(const float* xyz_dev, float* tf_dev, int h_out, int w_out, int H, int W, void* stream);
int lic360_projects_forward(const float* in_dev, const float* tf_dev, float* out_dev, int NC, int H, int W, int h_out, int w_out,
                            int nearest, void* stream);
int lic360_projects_backward(const float* top_diff_dev, const float* tf_dev, float* bottom_diff_dev, float* count_dev, int NC, int H,
                             int W, int h_out, int w_out, int nearest, void* stream);

/* ---- View footprint: the cells of an h x w ERP grid that a rectilinear view of any direction touches --------------------------
 * Cell (i, j) is the closed spherical rectangle x in [j - 1/2, j + 1/2], y in [i - 1/2, i + 1/2] of ProjectsOp's ERP coordinates
 * (x = theta / pi * hx + hx, y = -2 lat / pi * hy + hy, hx = (w - 1) / 2, hy = (h - 1) / 2), clamped to the sphere: columns 0 and
 * w - 1 are the half cells beside the +-pi seam, rows 0 and h - 1 end in a pole.  View v is (theta, phi, fov) in units of pi, as
 * MultiProject's: its axes (f, r, u) are the columns of the rotation lic360_projects_init builds (view (0, 0) looks along +x), and its
 * field is the closed frustum {d : |d.r| <= tan(a) d.f, |d.u| <= tan(a) d.f}, a = fov * pi / 2.  out_dev (nviews, h, w) int32:
 * 1 exactly where the cell and the field intersect (float64 predicate: a corner of one inside the other, or a field edge across a
 * cell edge), else 0.  h, w even and positive; 0 < fov < 1; finite angles.                                                          */
int lic360_view_footprint(int h, int w, int nviews, const float* theta_host, const float* phi_host, const float* fov_host,
                          int32_t* out_dev, void* stream);

/* ---- Coder (main.cpp:132-143, coder.h:10-63, coder.cpp:30-114; ArithmeticCoder.cpp, BitIoStream.cpp) -----
 * Same bitstream format (32-bit state range coder, MSB-first bits, `1` terminator + zero padding).
 * Tables are int32 rows of ncode+1 cumulative counts, total = row[ncode].                                   */
typedef struct lic360_coder lic360_coder;
lic360_coder* lic360_coder_create(const char* fname, float fill_value);
void lic360_coder_destroy(lic360_coder* c);
int lic360_coder_reset_fname(lic360_coder* c, const char* fname);
int lic360_coder_start_encoder(lic360_coder* c);           /* coder.h:15-21 */
int lic360_coder_end_encoder(lic360_coder* c);             /* coder.h:22-26, writes the file */
int lic360_coder_start_decoder(lic360_coder* c);           /* coder.h:30-35, reads the file */
int lic360_coder_encodes(lic360_coder* c, const int32_t* table_host, int ncode, const int32_t* label_host,
                         const float* mask_host /* NULL: encodes, else encodes_mask */, int num);
int lic360_coder_decodes(lic360_coder* c, const int32_t* table_host, int ncode, const float* mask_host, int num,
                         float* out_host);
/* Coder.encode / Coder.decode (main.cpp:134-135, coder.cpp:13-29): one symbol, explicit total */
int lic360_coder_encode_one(lic360_coder* c, const int32_t* table_host, int ncode, int total, int symbol);
int lic360_coder_decode_one(lic360_coder* c, const int32_t* table_host, int ncode, int total, int* symbol);
/* in-memory variants used by the fused pipeline and the tests */
int lic360_coder_start_encoder_mem(lic360_coder* c);
long lic360_coder_finish_mem(lic360_coder* c);             /* returns byte count */
long lic360_coder_get_bytes(lic360_coder* c, uint8_t* out, long cap);
int lic360_coder_start_decoder_mem(lic360_coder* c, const uint8_t* bytes, long n);
/* the slab loops of coder.cpp:62-114 (encodes_mask / decodes_mask / encodes / decodes) over PACKED CDF rows, the format the fused
 * codec's kernels write into pinned memory (same integers as the int32 tables, end points 0 and 65536 dropped):
 *   kind 0, code stream      :  8 x u16 per symbol = T[1..7] low words, meta = symbol(3 bits) | out-of-range << 3 | publication tag << 4
 *                               | mask << 8 | bit 16 of T[1..7] << 9  (the tag is only used between the decoder's kernels and its host loop)
 *   kind 1, importance stream: 64 x u16 per symbol = T[1..48] low words, [48] = symbol, [49..51] = bit 16 of T[1..48]
 * decode writes the symbols (fill_value where the mask bit is 0) to out[nrows] */
int lic360_coder_encode_rows(lic360_coder* c, const uint16_t* rows, int nrows, int kind);
int lic360_coder_decode_rows(lic360_coder* c, const uint16_t* rows, int nrows, int kind, float* out);

/* ---- fused entropy codec of one ERP latent --------------------------------------------------------------------
 * Replaces the four Python drivers of the reference demo -- EntEncoderFast / ImpEntEncoderFast / EntDecoder /
 * ImpEntDecoder (test/lic360_demo.py:95-290) together with `encoding`/`decoding` (:339-404) for the entropy part:
 * same networks, same symbol order, same coder, same two bitstreams (<name>_imp, <name>).
 * H, W: size of the code latent (image/8; 64x128 for a 512x1024 ERP image); the importance map is (H/2, W/2).
 * One codec = one image in flight on its own CUDA stream; instances are independent and thread-safe against each
 * other (one host thread + one codec per image overlaps host coding of one image with GPU steps of another).
 * stream_id: 0 = code stream (48 groups, 3 nets [weight, delta, mean], 8 symbols), 1 = importance stream (49 symbols).
 * layer: 0..11 = net.0, net.1.conv1, net.1.conv2, ..., net.5.conv2, net.6 (lic360_demo.py:104-112,153-161,296-322),
 * weights in the reference layout ((3,)Cout,Cin,5,5).                                                           */
typedef struct lic360_codec lic360_codec;
lic360_codec* lic360_codec_create(int device, int H, int W);
void lic360_codec_destroy(lic360_codec* c);
int lic360_codec_set_layer(lic360_codec* c, int stream_id, int layer, const float* w_dev, const float* bias_dev,
                           const float* slope_dev);
/* code_dev (1,48,H,W) symbols 0..7, mask_dev (1,48,H,W) 0/1, imp_dev (1,1,H/2,W/2) importance levels 0..48 */
int lic360_codec_encode(lic360_codec* c, const float* code_dev, const float* mask_dev, const float* imp_dev);
/* Exact-table rate of one latent without arithmetic coding: runs the same two networks as lic360_codec_encode and, for
 * every symbol the encoder would code, its ideal code length 16 - log2(T[s+1] - T[s]) bits from the same integer CDF row.
 *   code_bits_dev (1,48,H,W) float32: bits of each code symbol; exactly 0 where mask < 0.5 (not coded)
 *   imp_bits_dev  (1,1,H/2,W/2) float32: bits of each importance level
 *   bits_host[0] = code stream total, bits_host[1] = importance stream total (stream_id order), summed in double in a fixed
 *   order (the same inputs give the same totals on every call and every codec)
 * Rejects exactly the inputs lic360_codec_encode rejects, with the same status and message.  A stream of N coded symbols and
 * I = its total is len bytes long with -(1 + u + N/8192) <= 8*len - I <= 8 + N/8192, u = the coder's pending underflow bits at
 * the end, which the terminator makes unnecessary (a few at most in practice; derivation in tests/test_rate_estimate.py). */
int lic360_codec_estimate(lic360_codec* c, const float* code_dev, const float* mask_dev, const float* imp_dev,
                          float* code_bits_dev, float* imp_bits_dev, double* bits_host);
/* lic360_codec_estimate of K latents of the codec's size in one pass: both networks run once at batch K (the code network as 3K
 * images over its 3 weight sets), the bits kernels once with the latent in blockIdx.y.  Latent k's totals and map are bit-identical
 * to lic360_codec_estimate of that latent alone (same block partition, same fixed-order sums, no floating-point atomics).
 *   code_dev, mask_dev (K,48,H,W), imp_dev (K,1,H/2,W/2): the inputs of K encodes, stacked
 *   code_bits_dev (K,48,H,W), imp_bits_dev (K,1,H/2,W/2): the maps; either may be NULL (not written; the totals still are)
 *   bits_host[2k + stream_id]: totals of latent k; counts_host[2k + stream_id]: its coded symbols, counted on the device (code
 *   stream: positions with mask >= 0.5; importance stream: every position)
 * The encoder buffers grow to the largest K seen and are freed by lic360_codec_destroy.  A bad latent fails the call with the status
 * and message lic360_codec_encode gives for it, followed by " (latent k)", for the lowest such k.  K < 1, or K beyond the launch
 * limits (3K <= 65535 and 3 * K * 48 * H * W < 2^31), is an argument error. */
int lic360_codec_estimate_batch(lic360_codec* c, int K, const float* code_dev, const float* mask_dev, const float* imp_dev,
                                float* code_bits_dev, float* imp_bits_dev, double* bits_host, long long* counts_host);
/* lic360_codec_estimate_batch of J rate-control candidates given as (source latent, offset) pairs, without materialising them.
 *   code_dev (K,48,H,W), imp_dev (K,1,H/2,W/2): K source latents; protect_dev: NULL or (K,1,H/2,W/2) int32 protection maps
 *   candidate j: source cand_latent_host[j] in [0, K) lowered by offset cand_offset_host[j] >= 0, cell by cell as
 *   lic360_imp_levels_to_mask_protected lowers it (P clamped to [0, 48]; NULL: no map)
 *   bits_host[2j + stream_id], counts_host[2j + stream_id]: totals and coded symbols of candidate j
 * The outputs are bit-identical to lic360_codec_estimate_batch run on the candidates' levels and masks from
 * lic360_imp_levels_to_mask_protected with the source's code.  No candidate's code or (48,H,W) mask is stored: the code network's input
 * (code - 3.5) * mask is built from the source code and each symbol's mask bit, which the code stream's bits kernel derives again; the
 * candidates' levels (H/2 x W/2 floats each) live in a codec buffer that grows with J.  J has the limits of K in
 * lic360_codec_estimate_batch.  A candidate lic360_codec_encode would refuse fails the call with encode's status and message followed
 * by " (candidate j)", for the lowest such j; validity is judged on the candidate (lowering can bring a level into range, and a
 * masked-out code symbol is never checked).  K < 1, J < 1, a source outside [0, K) or a negative offset is an argument error. */
int lic360_codec_estimate_candidates(lic360_codec* c, int K, const float* code_dev, const float* imp_dev, const int32_t* protect_dev,
                                     int J, const int* cand_latent_host, const int* cand_offset_host, double* bits_host,
                                     long long* counts_host);
/* lic360_codec_encode of K latents of the codec's size in one pass: both networks run once at batch K, as in
 * lic360_codec_estimate_batch, the row kernels once with the latent in blockIdx.y, and each stream's rows come back with one copy.
 * The host codes the K importance streams as soon as their rows are on the host, while the code network still runs, then the K
 * code streams.  Latent k's two streams are byte-identical to lic360_codec_encode of that latent alone.
 *   code_dev, mask_dev (K,48,H,W), imp_dev (K,1,H/2,W/2): the inputs of K encodes, stacked
 * Workers: K = 1 codes on the calling thread, exactly as lic360_codec_encode.  K > 1 codes the 2K streams on a pool of persistent
 * host threads owned by the codec, each with its own coder: min(K, hardware threads, 16) workers, started on demand the first time a
 * batch needs them and joined by lic360_codec_destroy.
 * Results: latent k's streams stay in codec-owned buffers until the next encode, encode_batch or decode on this codec; read them
 * with lic360_codec_batch_stream_size / _copy.  lic360_codec_stream_size / _copy return latent 0's.
 * Buffers: the encoder frames grow as in lic360_codec_estimate_batch; the CDF-row buffers of both streams (device and pinned host)
 * grow to the largest K an encode has seen (an estimate does not grow them).  A failed allocation keeps the old buffers.
 * Errors: a bad latent fails the whole call with the status and message lic360_codec_encode gives for it, followed by " (latent k)",
 * for the lowest such k; within a latent the importance stream's error comes first.  A failed call returns no streams.  K < 1, or
 * K beyond the launch limits of lic360_codec_estimate_batch, is an argument error.
 * lic360_codec_last_timing after a batch: [0] wall time of the call, [1] wall time of the host-coding phase (from the importance
 * rows' arrival to the last stream coded), [2] time the calling thread waited for the GPU. */
int lic360_codec_encode_batch(lic360_codec* c, int K, const float* code_dev, const float* mask_dev, const float* imp_dev);
/* bytes of stream stream_id (0 code, 1 importance) of latent k of the last encode or encode_batch; the copy writes at most cap of
 * them to out and returns the stream's size.  -1 (and a message) when k is not a latent of the last successful encode. */
long lic360_codec_batch_stream_size(lic360_codec* c, int k, int stream_id);
long lic360_codec_batch_stream_copy(lic360_codec* c, int k, int stream_id, uint8_t* out, long cap);
/* lic360_codec_encode_batch of J rate-control candidates given as (source latent, offset) pairs, without materialising them: the
 * arguments and their limits are those of lic360_codec_estimate_candidates.  Candidate j's two streams are byte-identical to
 * lic360_codec_encode_batch run on the source's code with the candidate's levels and mask from lic360_imp_levels_to_mask_batch.  No
 * candidate's code or (48,H,W) mask is stored: the code network's input is built as in lic360_codec_estimate_candidates, and the code
 * stream's row kernel reads the source code and derives each mask bit again; the importance stream codes the candidate levels.
 * Results: candidate j's streams are read with lic360_codec_batch_stream_size / _copy (k = j) and stay valid until the next encode,
 * encode_batch, encode_candidates or decode.  Buffers and lic360_codec_last_timing are those of lic360_codec_encode_batch at K = J.
 * Errors: a candidate lic360_codec_encode would refuse fails the whole call with encode's status and message followed by
 * " (candidate j)", for the lowest such j; within a candidate the importance stream's error comes first; validity is judged on the
 * candidate, as the estimate judges it (a masked-out code symbol is never checked).  A failed call returns no streams.  K < 1, J < 1,
 * J beyond the launch limits, a source outside [0, K) or a negative offset is an argument error. */
int lic360_codec_encode_candidates(lic360_codec* c, int K, const float* code_dev, const float* imp_dev, const int32_t* protect_dev,
                                   int J, const int* cand_latent_host, const int* cand_offset_host);
/* Candidate importance maps and the code masks the decoder derives from them, for rate control.  levels_dev (h,w) are importance
 * levels as lic360_codec_encode reads them: s = the symbol it codes for a level ((int) of it).  For each offsets_host[j] >= 0:
 *   levels_out_dev[j] (K,1,h,w) = max(s - offsets_host[j], 0)
 *   mask_out_dev[j]  (K,48,2h,2w) = the decoder's mask of that level, Imp2mask + Dtow in one pass: channel c at (y, x) is 1 iff
 *                                   4c + 2 (y % 2) + x % 2 < 4 * level(y/2, x/2)
 * Encoding a pair (levels_out[j], mask_out[j]) gives streams that decode to exactly that mask.  Enqueued on `stream`.
 * The case protect_dev = NULL of lic360_imp_levels_to_mask_protected. */
int lic360_imp_levels_to_mask(const float* levels_dev, int h, int w, const int* offsets_host, int K, float* levels_out_dev,
                              float* mask_out_dev, void* stream);
/* lic360_imp_levels_to_mask with a protection map: protect_dev (h,w) int32 per importance cell, or NULL.  Candidate t = offsets_host[j]
 * lowers a cell with protection P = min(max(protect_dev[cell], 0), 48) by max(t - P, 0):
 *   levels_out_dev[j] = max(s - max(t - P, 0), 0),  mask_out_dev[j] = the decoder's mask of that level, as above
 * all in integer arithmetic; the outputs are integers stored as float.  A cell keeps its level until t > P, so the masks are nested
 * in t and every level is 0 at t = 48 + max P.  NULL (or a map of zeros) gives the levels max(s - t, 0) of lic360_imp_levels_to_mask,
 * bit for bit.  Same argument checks and messages as lic360_imp_levels_to_mask. */
int lic360_imp_levels_to_mask_protected(const float* levels_dev, int h, int w, const int* offsets_host, int K, const int32_t* protect_dev,
                                        float* levels_out_dev, float* mask_out_dev, void* stream);
/* lic360_imp_levels_to_mask_protected of J candidates of K source maps: levels_dev (K,1,h,w), protect_dev NULL or (K,1,h,w) int32;
 * candidate j is source cand_latent_host[j] in [0, K) at offset cand_offset_host[j] >= 0.  levels_out_dev (J,1,h,w) and mask_out_dev
 * (J,48,2h,2w): entry j is bit-identical to lic360_imp_levels_to_mask_protected of its source's map and protection at its offset.
 * Enqueued on `stream`; a source outside [0, K) or a negative offset is an argument error. */
int lic360_imp_levels_to_mask_batch(const float* levels_dev, int K, int h, int w, const int32_t* protect_dev, int J,
                                    const int* cand_latent_host, const int* cand_offset_host, float* levels_out_dev, float* mask_out_dev,
                                    void* stream);
long lic360_codec_stream_size(lic360_codec* c, int stream_id);
long lic360_codec_stream_copy(lic360_codec* c, int stream_id, uint8_t* out, long cap);
/* -> code_out_dev (1,48,H,W) = symbols where mask == 1, else 0 (lic360_demo.py:236-237); mask_out_dev (1,48,H,W) */
int lic360_codec_decode(lic360_codec* c, const uint8_t* imp_bytes, long n_imp, const uint8_t* code_bytes, long n_code,
                        float* code_out_dev, float* mask_out_dev);
/* milliseconds of the last encode/decode/estimate call: [0] total, [1] host arithmetic coder, [2] waiting for the GPU,
 * [3] importance stream part of a decode, [4] CUDA-event time of all decode graph replays, [5] of the importance stream ones
 * (an estimate fills [0] and [2] only; an encode_batch of K > 1 fills [1] with the wall time of its host-coding phase) */
int lic360_codec_last_timing(lic360_codec* c, double* out, int n);
/* mode 0 (default): pipelined graph replay per wavefront step.  mode 1: the same kernels launched one by one on the codec
 * stream with CUDA events between them (the decode is serialized and slower; used by bench.py for the roofline block).
 * mode 2 (low latency, opt-in): the code stream's chain kernel is launched ONCE per decode and walks all wavefront steps; between
 * steps it polls the symbols the host publishes in mapped memory (every symbol word carries a publication tag) instead of being
 * re-launched, so no graph launch, scatter kernel or kernel prologue sits between the host's last decoded symbol and the next
 * step.  Same bitstreams, same results.  Its three 8-CTA clusters stay resident for the whole decode, so a mode-2 decode takes the device
 * for itself: other decodes on the same GPU queue until it is done (encodes do not).  Caveat: while it runs, a call from ANOTHER host
 * thread that makes the driver wait for the device (cudaFree, a graph instantiation, ...) can hold the driver lock the decode's own
 * launches need; the kernel's bail-outs (20 s) then fail the decode instead of hanging.  A latency mode for one image at a time. */
int lic360_codec_set_mode(lic360_codec* c, int mode);
/* after a mode-1 decode: total milliseconds of the last decode spent in [0] the old-term kernel, [1] the previous-wavefront
 * kernel, [2] the 12-layer chain kernel, [3] scatter + CDF-row kernels, and [4] the number of steps, for one stream */
int lic360_codec_kernel_times(lic360_codec* c, int stream_id, double* out, int n);
/* the decoder's kernel choices for one stream (0 = code, 1 = importance), fixed when the codec is created (they depend on the
 * latent size; DESIGN.md s8 lists the overrides of the cluster size [2]); read-only.  out[0 .. n-1], at most 13 values:
 *   [0] chain kernel: 0 wf_chain_kernel (generic), 1 wf_chain4_kernel, 2 wf_chain1_kernel
 *   [1] wf_chain1_kernel exchanges activations through distributed shared memory (1) or reloads its tile every layer (0)
 *   [2] CTAs per cluster  [3] chain threads per CTA  [4] chain dynamic shared memory, bytes, as launched
 *   [5] longest wavefront step (positions)  [6] wf_chain1_kernel's padded step length lenp  [7] its output chunks per CTA
 *       ([6], [7]: 0 for the other chain kernels)
 *   [8] wf_chain_kernel's tasks per CTA in the longest step (its thread loop takes a second round when [8] > [3])
 *   [9] old-term kernel positions per lane (4 or 1)  [10] parts4  [11] parts: 64- and 32-position tiles per diagonal
 *   [12] wf_chain4_kernel: most rounds in which a CTA's R tail stages its weight rows (0 for the other chain kernels) */
int lic360_codec_engine_info(lic360_codec* c, int stream_id, int* out, int n);

#ifdef __cplusplus
}
#endif
#endif /* LIC360_B200_H */
