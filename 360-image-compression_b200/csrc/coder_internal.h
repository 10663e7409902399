// Packed CDF rows exchanged between the fused codec kernels (codec.cu) and the host coder (coder.cpp).
// The tables are the same integers the per-op path produces as float rows; packing only drops the constant end
// points T[0] = 0 and T[last] = 65536 and stores the rest as 16-bit words plus one overflow bit each (a bin can
// reach 65536 + a few counts before the monotonic fix-up pulls it back, entropy_gmm_table_cuda.cu:85-107).
//   code stream row  :  8 x u16 = T[1..7] low words, meta = sym(3 bits) | out-of-range << 3 | tag(4 bits) << 4 | mask << 8 | overflow(T[1..7]) << 9
//                       (tag: wf_row_tag(step) (wavefront.cuh) on the decoder's per-step rows, 0 elsewhere; a row is one aligned 16-byte store, so the tag
//                       publishes the whole row and the host decodes row by row without a fence + flag behind the step's rows)
//   importance row   : 64 x u16 = T[1..48] low words, [48] = sym, [49..51] = overflow bits of T[1..48]
#pragma once
#include <stdint.h>
#include "../../include/lic360_b200.h"

namespace lic360 {
int coder_encode_packed_gmm(lic360_coder* c, const uint16_t* rows, int nrows);
int coder_decode_packed_gmm(lic360_coder* c, const uint16_t* rows, int nrows, float* out);
// the decoder's per-step rows when they carry a publication tag (meta bits 4..7): row i is decoded as soon as its tag equals `tag`;
// `stalled` is called every few thousand polls of a missing row and returns non-zero to give up (its value is returned)
// sym_tag != 0: the decoded symbol words carry that tag in their four low mantissa bits (polled by the persistent chain kernel)
int coder_decode_packed_gmm_tagged(lic360_coder* c, const uint16_t* rows, int nrows, float* out, int tag, int (*stalled)(void*), void* ctx,
                                   unsigned sym_tag = 0);
int coder_encode_packed_imp(lic360_coder* c, const uint16_t* rows, int nrows);
int coder_decode_packed_imp(lic360_coder* c, const uint16_t* rows, int nrows, float* out);
// the message the packed encoders set when they refuse row `row` of stream stream_id (0 code, 1 importance), whose symbol is `sym`:
// out of range (code stream: sym > 7, importance stream: sym >= 49), else a zero-width bin.  Returns LIC360_ERR_CODER.
int coder_row_error(int stream_id, int row, unsigned sym);
const uint8_t* coder_bytes(lic360_coder* c, long* n);
}  // namespace lic360
