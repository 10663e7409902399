// Host arithmetic coder: same bitstream as the reference's Coder / ArithmeticEncoder / ArithmeticDecoder /
// BitOutputStream / BitInputStream (/root/reference/extension/coder.{h,cpp}, ArithmeticCoder.cpp:15-171,
// BitIoStream.cpp:13-71): 32-bit state range coder, MSB-first bit order, terminator = a single `1` bit followed by
// zero padding to a byte boundary, EOF reads as zero bits.
//
// Written from the arithmetic, not from the reference classes: the per-bit renormalisation loops
// (ArithmeticCoder.cpp:56-68) are collapsed with count-leading-zeros into one multi-bit shift for the
// "matching top bits" phase and one for the underflow phase, bits go through a 64-bit accumulator instead of an
// iostream, and the power-of-two total (65536 for every table of this codec) turns the two divisions of the range
// update into shifts.  tests/test_oracle_coder.py checks byte-identical streams against oracle/_ref/libref_coder.so
// (the reference's own classes).
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <string>
#include <vector>
#include "../../include/lic360_b200.h"

namespace lic360 {
void set_error(const char* fmt, ...);
}

namespace {

constexpr uint64_t kMask = 0xFFFFFFFFull, kTop = 0x80000000ull, kSecond = 0x40000000ull;
constexpr uint64_t kMinRange = (1ull << 30) + 2;  // ArithmeticCoder.cpp:20, also MAX_TOTAL (:21)

struct BitWriter {
    std::vector<uint8_t> bytes;
    uint64_t acc = 0;  // pending bits, right-aligned
    int nacc = 0;
    void reset() { bytes.clear(); acc = 0; nacc = 0; }
    inline void flush_bytes() {
        while (nacc >= 8) {
            nacc -= 8;
            bytes.push_back((uint8_t)(acc >> nacc));
        }
        acc &= (1ull << nacc) - 1;
    }
    inline void put(uint32_t value, int n) {  // n <= 32
        if (n == 0) return;
        acc = (acc << n) | (value & ((n == 32) ? 0xFFFFFFFFu : ((1u << n) - 1)));
        nacc += n;
        flush_bytes();
    }
    inline void put_run(int bit, uint64_t count) {
        while (count > 0) {
            int n = count > 32 ? 32 : (int)count;
            put(bit ? 0xFFFFFFFFu : 0u, n);
            count -= n;
        }
    }
    void finish() {  // BitIoStream.cpp:68-71
        if (nacc > 0) put(0, 8 - nacc);
    }
};

struct BitReader {
    const uint8_t* p = nullptr;
    size_t len = 0, pos = 0;
    uint64_t acc = 0;
    int nacc = 0;
    void reset(const uint8_t* data, size_t n) { p = data; len = n; pos = 0; acc = 0; nacc = 0; }
    inline uint32_t get(int n) {  // 0 <= n <= 32 (n == 0 yields 0); past EOF reads zeros (ArithmeticCoder.cpp:131-136)
        if (nacc < n && pos + 4 <= len) {  // refill 32 bits at once (nacc < 32 here, so the 64-bit accumulator cannot overflow)
            uint32_t w;
            memcpy(&w, p + pos, 4);
            acc = (acc << 32) | __builtin_bswap32(w);
            nacc += 32;
            pos += 4;
        }
        while (nacc < n) {
            uint64_t b = pos < len ? p[pos] : 0;
            pos++;
            acc = (acc << 8) | b;
            nacc += 8;
        }
        nacc -= n;
        uint32_t v = (uint32_t)((acc >> nacc) & ((n == 32) ? 0xFFFFFFFFull : ((1ull << n) - 1)));
        acc &= (1ull << nacc) - 1;
        return v;
    }
};

}  // namespace

struct lic360_coder {
    std::string fname;
    float fill = 3.5f;
    uint64_t low = 0, high = kMask, code = 0, underflow = 0;
    BitWriter bw;
    BitReader br;
    std::vector<uint8_t> input;
    bool encoding = false, decoding = false, to_file = false;
};

namespace {

// ArithmeticCoder.cpp:34-69 with both renormalisation loops collapsed.
template <bool kDecode>
inline int ac_update(lic360_coder* c, uint32_t sym_low, uint32_t sym_high, uint32_t total) {
    const uint64_t range = c->high - c->low + 1;
    if (sym_low == sym_high) { lic360::set_error("coder: symbol has zero frequency"); return LIC360_ERR_CODER; }
    if (total > kMinRange) { lic360::set_error("coder: total too large"); return LIC360_ERR_CODER; }
    uint64_t nl, nh;
    if ((total & (total - 1)) == 0) {
        const int sh = __builtin_ctz(total);
        nl = c->low + (((uint64_t)sym_low * range) >> sh);
        nh = c->low + (((uint64_t)sym_high * range) >> sh) - 1;
    } else {
        nl = c->low + (uint64_t)sym_low * range / total;
        nh = c->low + (uint64_t)sym_high * range / total - 1;
    }
    uint32_t lo = (uint32_t)nl, hi = (uint32_t)nh;
    const uint32_t diff = lo ^ hi;
    if (diff == 0) { lic360::set_error("coder: low == high"); return LIC360_ERR_CODER; }
    const int n = __builtin_clz(diff);  // leading bits shared by low and high: shifted out (":56-60")
    if (n > 0) {
        if (kDecode) {
            c->code = ((c->code << n) & kMask) | c->br.get(n);
        } else {
            const int first = lo >> 31;
            c->bw.put(first, 1);
            if (c->underflow) { c->bw.put_run(first ^ 1, c->underflow); c->underflow = 0; }
            if (n > 1) c->bw.put(lo >> (32 - n), n - 1);  // low n-1 bits of the top n bits of lo
        }
        lo <<= n;
        hi = (hi << n) | ((1u << n) - 1);
    }
    // underflow phase (":62-68"): low = 01..., high = 10...  -> drop the second-highest bit k times
    const uint32_t m = (lo & ~hi) << 1;
    const int k = __builtin_clz(~m | 1u);  // consecutive ones from the top of m (k <= 31)
    if (k > 0) {
        if (kDecode) c->code = (c->code & kTop) | ((c->code << k) & (kMask >> 1)) | c->br.get(k);
        else c->underflow += k;
        lo = (lo << k) & 0x7FFFFFFFu;
        hi = ((hi << k) & 0x7FFFFFFFu) | 0x80000000u | ((1u << k) - 1);
    }
    c->low = lo;
    c->high = hi;
    return LIC360_OK;
}

}  // namespace

// ---- packed-row fast paths of the fused pipeline (codec.cu); see coder_internal.h for the row formats ----------
namespace lic360 {

int coder_row_error(int stream_id, int row, unsigned sym) {
    if (stream_id == 0 && sym > 7) set_error("coder: symbol out of range in packed row %d", row);
    else if (stream_id == 0) set_error("coder: symbol has zero frequency (row %d)", row);
    else if (sym >= 49) set_error("coder: importance level %u out of range", sym);
    else set_error("coder: symbol has zero frequency");
    return LIC360_ERR_CODER;
}

static inline uint32_t gmm_bin(const uint16_t* r, int j) {  // j in 0..8
    if (j == 0) return 0;
    if (j == 8) return 65536;
    return (uint32_t)r[j - 1] | (((uint32_t)(r[7] >> (9 + j - 1)) & 1u) << 16);
}

// Encoder state kept in locals for a whole run of rows (like DecState below): low / high / pending-underflow count in registers,
// bits through a 64-bit accumulator that is drained 32 bits at a time into a pre-sized buffer (no per-byte vector growth), and
// the common case "no pending underflow" emits the n matching top bits with one put.  Same bits as ac_update<false>
// (tests/test_oracle_coder.py pins both against the reference's classes).
struct EncState {
    uint32_t low, high;
    uint64_t underflow;
    uint64_t acc;
    int nacc;
    uint8_t* p;
    inline void put(uint32_t v, int n) {  // n in 1..32, v < 2^n
        acc = (acc << n) | v;
        nacc += n;
        if (nacc >= 32) {
            nacc -= 32;
            const uint32_t w = __builtin_bswap32((uint32_t)(acc >> nacc));
            memcpy(p, &w, 4);
            p += 4;
        }
    }
    inline bool update(uint32_t t_lo, uint32_t t_hi) {  // total = 65536
        const uint64_t range = (uint64_t)high - low + 1;
        uint32_t lo = low + (uint32_t)(((uint64_t)t_lo * range) >> 16), hi = low + (uint32_t)(((uint64_t)t_hi * range) >> 16) - 1;
        const uint32_t diff = lo ^ hi;
        if (t_lo == t_hi || diff == 0) return false;
        const int n = __builtin_clz(diff);
        if (n > 0) {
            if (underflow == 0) {
                put(lo >> (32 - n), n);
            } else {
                const uint32_t first = lo >> 31;
                put(first, 1);
                for (uint64_t left = underflow; left > 0;) {
                    const int k = left > 32 ? 32 : (int)left;
                    put(first ? 0u : (k == 32 ? 0xFFFFFFFFu : ((1u << k) - 1)), k);
                    left -= k;
                }
                underflow = 0;
                if (n > 1) put((lo >> (32 - n)) & ((1u << (n - 1)) - 1), n - 1);
            }
            lo <<= n;
            hi = (hi << n) | ((1u << n) - 1);
        }
        const uint32_t m = (lo & ~hi) << 1;
        const int k = __builtin_clz(~m | 1u);
        if (k > 0) {
            underflow += k;
            lo = (lo << k) & 0x7FFFFFFFu;
            hi = ((hi << k) & 0x7FFFFFFFu) | 0x80000000u | ((1u << k) - 1);
        }
        low = lo; high = hi;
        return true;
    }
};

// runs `body(EncState&)` over the coder's state with room for `max_bits` more bits in the output buffer
template <typename F>
static int with_enc_state(lic360_coder* c, size_t max_bits, F body) {
    BitWriter& bw = c->bw;
    const size_t used = bw.bytes.size();
    bw.bytes.resize(used + max_bits / 8 + 16);
    EncState e{(uint32_t)c->low, (uint32_t)c->high, c->underflow, bw.acc, bw.nacc, bw.bytes.data() + used};
    const int rc = body(e);
    while (e.nacc >= 8) { e.nacc -= 8; *e.p++ = (uint8_t)(e.acc >> e.nacc); }
    bw.acc = e.acc & ((1ull << e.nacc) - 1);
    bw.nacc = e.nacc;
    bw.bytes.resize((size_t)(e.p - bw.bytes.data()));
    c->low = e.low; c->high = e.high; c->underflow = e.underflow;
    return rc;
}

int coder_encode_packed_gmm(lic360_coder* c, const uint16_t* rows, int nrows) {
    // a symbol costs at most 16 bits of information (total 65536) + 1; pending underflow bits were counted when they arose
    return with_enc_state(c, (size_t)nrows * 34 + (size_t)c->underflow + 64, [&](EncState& e) -> int {
        for (int i = 0; i < nrows; i++) {
            const uint16_t* r = rows + (size_t)i * 8;
            if (!((r[7] >> 8) & 1)) continue;  // mask < 0.5: not coded (coder.cpp:79)
            if (r[7] & 8) return coder_row_error(0, i, 8);
            const int s = r[7] & 7;
            if (!e.update(gmm_bin(r, s), gmm_bin(r, s + 1))) return coder_row_error(0, i, s);
        }
        return LIC360_OK;
    });
}

// Decoder state kept in locals for a whole slab; `code` is refilled through the 64-bit accumulator of the bit reader.
// The symbol search is division-free: with value = floor(num / range), num = ((code - low + 1) << 16) - 1,
//     T[j] <= value  <=>  T[j] * range <= num          (T[j] integer, range > 0)
// so the symbol is the number of interior bins whose 48-bit product does not exceed num (the rows are strictly increasing after the
// fix-up, the same symbol the reference's binary search ArithmeticCoder.cpp:92-116 returns), the seven products are independent
// (no 64-bit divide, no data-dependent branch) and the two the range update needs (ArithmeticCoder.cpp:50-53) are among them.
struct DecState {
    uint32_t low, high, code;
    BitReader* br;
    inline bool update(uint64_t pl, uint64_t ph) {  // pl, ph = T[s] * range, T[s+1] * range; total = 65536
        uint32_t lo = low + (uint32_t)(pl >> 16), hi = low + (uint32_t)(ph >> 16) - 1;
        const uint32_t diff = lo ^ hi;
        if (pl == ph || diff == 0) return false;
        const int n = __builtin_clz(diff);  // 0..31 matching top bits; n == 0 flows through the same shifts (no data-dependent branch)
        code = (code << n) | br->get(n);
        lo <<= n;
        hi = (hi << n) | ((1u << n) - 1);
        const uint32_t m = (lo & ~hi) << 1;
        const int k = __builtin_clz(~m | 1u);
        if (k > 0) {
            code = (code & 0x80000000u) | ((code << k) & 0x7FFFFFFFu) | br->get(k);
            lo = (lo << k) & 0x7FFFFFFFu;
            hi = ((hi << k) & 0x7FFFFFFFu) | 0x80000000u | ((1u << k) - 1);
        }
        low = lo; high = hi;
        return code >= lo && code <= hi;
    }
};

template <bool kTagged>
static int decode_packed_gmm_impl(lic360_coder* c, const uint16_t* rows, int nrows, float* out, int tag, int (*stalled)(void*), void* ctx,
                                  uint32_t sym_tag = 0) {
    DecState st{(uint32_t)c->low, (uint32_t)c->high, (uint32_t)c->code, &c->br};
    // sym_tag != 0 (persistent decode): every symbol word is self-validating for the GPU threads that poll it -- the low 4 mantissa
    // bits of the float (zero for 0..7 and for the fill value) carry the step's publication tag
    auto put = [sym_tag](float* dst, float v) {
        if (kTagged && sym_tag) {
            uint32_t b;
            memcpy(&b, &v, 4);
            b |= sym_tag;
            __atomic_store_n(reinterpret_cast<uint32_t*>(dst), b, __ATOMIC_RELAXED);
        } else {
            *dst = v;
        }
    };
    const float fill = c->fill;
    int rc = LIC360_OK;
    for (int i = 0; i < nrows; i++) {
        const uint16_t* r = rows + (size_t)i * 8;
        if (kTagged) {
            // the row is one 16-byte device store: once the meta word shows this step's tag the whole row is there (acquire: the
            // loads of the bins below must not be satisfied before it)
            unsigned spins = 0;
            while (((__atomic_load_n(r + 7, __ATOMIC_ACQUIRE) >> 4) & 15) != (unsigned)(tag & 15)) {
#if defined(__x86_64__)
                __builtin_ia32_pause();
#endif
                if ((++spins & 0x3FFF) == 0 && stalled) {
                    const int give_up = stalled(ctx);
                    if (give_up) { c->low = st.low; c->high = st.high; c->code = st.code; return give_up; }
                }
            }
        }
        // the rows were just written by the GPU into pinned memory: every cache line is a miss, and the serial state chain leaves
        // the hardware prefetcher little to go on -- ask for the lines ahead
        __builtin_prefetch(r + 8 * 24);
        const uint32_t meta = r[7];
        if (!((meta >> 8) & 1)) { put(out + i, fill); continue; }  // coder.cpp:101-102
        const uint64_t range = (uint64_t)st.high - st.low + 1;
        const uint64_t num = (((uint64_t)(st.code - st.low) + 1) << 16) - 1;
        uint64_t prod[9];
        prod[0] = 0;
        prod[8] = range << 16;
        uint32_t s = 0;
#pragma GCC unroll 7
        for (int j = 1; j <= 7; j++) {
            const uint64_t t = (uint64_t)r[j - 1] | ((uint64_t)((meta >> (9 + j - 1)) & 1u) << 16);
            prod[j] = t * range;
            s += prod[j] <= num;
        }
        if (!st.update(prod[s], prod[s + 1])) {
            set_error("coder: corrupt stream or table mismatch (zero-frequency symbol or code out of range)");
            rc = LIC360_ERR_CODER;
            break;
        }
        put(out + i, (float)s);
    }
    c->low = st.low; c->high = st.high; c->code = st.code;
    return rc;
}

int coder_decode_packed_gmm(lic360_coder* c, const uint16_t* rows, int nrows, float* out) {
    return decode_packed_gmm_impl<false>(c, rows, nrows, out, 0, nullptr, nullptr);
}

int coder_decode_packed_gmm_tagged(lic360_coder* c, const uint16_t* rows, int nrows, float* out, int tag, int (*stalled)(void*), void* ctx,
                                   unsigned sym_tag) {
    if (sym_tag) {
        uint32_t fb;
        memcpy(&fb, &c->fill, 4);
        if ((fb & 15u) || sym_tag > 15u) { set_error("coder: symbol tags need a fill value with four zero low mantissa bits"); return LIC360_ERR_ARG; }
    }
    return decode_packed_gmm_impl<true>(c, rows, nrows, out, tag, stalled, ctx, sym_tag);
}

static inline uint32_t imp_bin(const uint16_t* r, int j) {  // j in 0..49
    if (j == 0) return 0;
    if (j == 49) return 65536;
    return (uint32_t)r[j - 1] | (((uint32_t)(r[49 + (j - 1) / 16] >> ((j - 1) % 16)) & 1u) << 16);
}

int coder_encode_packed_imp(lic360_coder* c, const uint16_t* rows, int nrows) {
    for (int i = 0; i < nrows; i++) {
        const uint16_t* r = rows + (size_t)i * 64;
        const int s = r[48];
        if (s >= 49) return coder_row_error(1, i, s);
        const uint32_t lo = imp_bin(r, s), hi = imp_bin(r, s + 1);
        if (lo == hi) return coder_row_error(1, i, s);
        int rc = ac_update<false>(c, lo, hi, 65536);
        if (rc) return rc;
    }
    return LIC360_OK;
}

int coder_decode_packed_imp(lic360_coder* c, const uint16_t* rows, int nrows, float* out) {
    for (int i = 0; i < nrows; i++) {
        const uint16_t* r = rows + (size_t)i * 64;
        const uint64_t range = c->high - c->low + 1;
        const uint64_t offset = c->code - c->low;
        const uint64_t value = (((offset + 1) << 16) - 1) / range;
        uint32_t s = 0, e = 49;
        while (e - s > 1) {
            const uint32_t mid = (s + e) >> 1;
            if (imp_bin(r, mid) > value) e = mid; else s = mid;
        }
        int rc = ac_update<true>(c, imp_bin(r, s), imp_bin(r, s + 1), 65536);
        if (rc) return rc;
        if (c->code < c->low || c->code > c->high) { set_error("coder: code out of range (corrupt stream or table mismatch)"); return LIC360_ERR_CODER; }
        out[i] = (float)s;
    }
    return LIC360_OK;
}

const uint8_t* coder_bytes(lic360_coder* c, long* n) { *n = (long)c->bw.bytes.size(); return c->bw.bytes.data(); }

}  // namespace lic360

extern "C" {

int lic360_coder_encode_rows(lic360_coder* c, const uint16_t* rows, int nrows, int kind) {
    if (!c || !rows || nrows < 0 || (kind != 0 && kind != 1)) { lic360::set_error("coder: bad arguments"); return LIC360_ERR_ARG; }
    if (!c->encoding) { lic360::set_error("coder: encode without start_encoder"); return LIC360_ERR_CODER; }
    return kind == 0 ? lic360::coder_encode_packed_gmm(c, rows, nrows) : lic360::coder_encode_packed_imp(c, rows, nrows);
}

int lic360_coder_decode_rows(lic360_coder* c, const uint16_t* rows, int nrows, int kind, float* out) {
    if (!c || !rows || !out || nrows < 0 || (kind != 0 && kind != 1)) { lic360::set_error("coder: bad arguments"); return LIC360_ERR_ARG; }
    if (!c->decoding) { lic360::set_error("coder: decode without start_decoder"); return LIC360_ERR_CODER; }
    return kind == 0 ? lic360::coder_decode_packed_gmm(c, rows, nrows, out) : lic360::coder_decode_packed_imp(c, rows, nrows, out);
}

lic360_coder* lic360_coder_create(const char* fname, float fill_value) {
    lic360_coder* c = new lic360_coder();
    c->fname = fname ? fname : "";
    c->fill = fill_value;
    return c;
}

void lic360_coder_destroy(lic360_coder* c) { delete c; }

int lic360_coder_reset_fname(lic360_coder* c, const char* fname) {
    c->fname = fname ? fname : "";
    return LIC360_OK;
}

int lic360_coder_start_encoder_mem(lic360_coder* c) {
    c->low = 0; c->high = kMask; c->underflow = 0;
    c->bw.reset();
    c->encoding = true; c->decoding = false; c->to_file = false;
    return LIC360_OK;
}

int lic360_coder_start_encoder(lic360_coder* c) {
    // the reference opens (truncates) the output file here, coder.h:15-21
    FILE* f = fopen(c->fname.c_str(), "wb");
    if (!f) { lic360::set_error("coder: cannot open '%s' for writing", c->fname.c_str()); return LIC360_ERR_CODER; }
    fclose(f);
    lic360_coder_start_encoder_mem(c);
    c->to_file = true;
    return LIC360_OK;
}

long lic360_coder_finish_mem(lic360_coder* c) {
    if (!c->encoding) { lic360::set_error("coder: end_encoder without start_encoder"); return -1; }
    c->bw.put(1, 1);  // ArithmeticCoder.cpp:152-154
    c->bw.finish();
    c->encoding = false;
    return (long)c->bw.bytes.size();
}

int lic360_coder_end_encoder(lic360_coder* c) {
    if (lic360_coder_finish_mem(c) < 0) return LIC360_ERR_CODER;
    if (c->to_file) {
        FILE* f = fopen(c->fname.c_str(), "wb");
        if (!f) { lic360::set_error("coder: cannot open '%s' for writing", c->fname.c_str()); return LIC360_ERR_CODER; }
        size_t n = fwrite(c->bw.bytes.data(), 1, c->bw.bytes.size(), f);
        fclose(f);
        if (n != c->bw.bytes.size()) { lic360::set_error("coder: short write to '%s'", c->fname.c_str()); return LIC360_ERR_CODER; }
    }
    return LIC360_OK;
}

long lic360_coder_get_bytes(lic360_coder* c, uint8_t* out, long cap) {
    long n = (long)c->bw.bytes.size();
    if (out && cap > 0) memcpy(out, c->bw.bytes.data(), (size_t)(n < cap ? n : cap));
    return n;
}

int lic360_coder_start_decoder_mem(lic360_coder* c, const uint8_t* bytes, long n) {
    c->input.assign(bytes, bytes + (n > 0 ? n : 0));
    c->br.reset(c->input.data(), c->input.size());
    c->low = 0; c->high = kMask;
    c->code = c->br.get(32);  // ArithmeticCoder.cpp:77-78
    c->decoding = true; c->encoding = false;
    return LIC360_OK;
}

int lic360_coder_start_decoder(lic360_coder* c) {
    FILE* f = fopen(c->fname.c_str(), "rb");
    if (!f) { lic360::set_error("coder: cannot open '%s' for reading", c->fname.c_str()); return LIC360_ERR_CODER; }
    std::vector<uint8_t> buf;
    uint8_t tmp[65536];
    size_t n;
    while ((n = fread(tmp, 1, sizeof(tmp), f)) > 0) buf.insert(buf.end(), tmp, tmp + n);
    fclose(f);
    return lic360_coder_start_decoder_mem(c, buf.data(), (long)buf.size());
}

// coder.cpp:30-47 (mask_host == NULL) and :70-89
int lic360_coder_encodes(lic360_coder* c, const int32_t* table_host, int ncode, const int32_t* label_host,
                         const float* mask_host, int num) {
    if (!c->encoding) { lic360::set_error("coder: encodes without start_encoder"); return LIC360_ERR_CODER; }
    const size_t stride = (size_t)ncode + 1;
    for (int i = 0; i < num; i++) {
        if (mask_host && mask_host[i] < 0.5f) continue;
        const uint32_t* t = reinterpret_cast<const uint32_t*>(table_host) + i * stride;
        const uint32_t s = (uint32_t)label_host[i];
        if (s >= (uint32_t)ncode) { lic360::set_error("coder: symbol %u out of range [0,%d)", s, ncode); return LIC360_ERR_CODER; }
        int rc = ac_update<false>(c, t[s], t[s + 1], t[ncode]);
        if (rc) return rc;
    }
    return LIC360_OK;
}

// coder.cpp:49-69 (mask_host == NULL) and :90-114; ArithmeticCoder.cpp:82-116
int lic360_coder_decodes(lic360_coder* c, const int32_t* table_host, int ncode, const float* mask_host, int num,
                         float* out_host) {
    if (!c->decoding) { lic360::set_error("coder: decodes without start_decoder"); return LIC360_ERR_CODER; }
    const size_t stride = (size_t)ncode + 1;
    for (int i = 0; i < num; i++) {
        if (mask_host && mask_host[i] < 0.5f) { out_host[i] = c->fill; continue; }
        const uint32_t* t = reinterpret_cast<const uint32_t*>(table_host) + i * stride;
        const uint32_t total = t[ncode];
        if (total == 0 || total > kMinRange) { lic360::set_error("coder: bad total %u", total); return LIC360_ERR_CODER; }
        const uint64_t range = c->high - c->low + 1;
        const uint64_t offset = c->code - c->low;
        const uint64_t value = ((offset + 1) * total - 1) / range;
        uint32_t s = 0, e = (uint32_t)ncode;
        while (e - s > 1) {
            const uint32_t mid = (s + e) >> 1;
            if (t[mid] > value) e = mid; else s = mid;
        }
        int rc = ac_update<true>(c, t[s], t[s + 1], total);
        if (rc) return rc;
        if (c->code < c->low || c->code > c->high) { lic360::set_error("coder: code out of range (corrupt stream or table mismatch)"); return LIC360_ERR_CODER; }
        out_host[i] = (float)s;
    }
    return LIC360_OK;
}

// Coder::encode / Coder::decode (main.cpp:134-135, coder.cpp:13-29): one symbol with an explicit total
int lic360_coder_encode_one(lic360_coder* c, const int32_t* table_host, int ncode, int total, int symbol) {
    if (!c->encoding) { lic360::set_error("coder: encode without start_encoder"); return LIC360_ERR_CODER; }
    if (symbol < 0 || symbol >= ncode) { lic360::set_error("coder: symbol %d out of range [0,%d)", symbol, ncode); return LIC360_ERR_CODER; }
    const uint32_t* t = reinterpret_cast<const uint32_t*>(table_host);
    return ac_update<false>(c, t[symbol], t[symbol + 1], (uint32_t)total);
}

int lic360_coder_decode_one(lic360_coder* c, const int32_t* table_host, int ncode, int total, int* symbol) {
    if (!c->decoding) { lic360::set_error("coder: decode without start_decoder"); return LIC360_ERR_CODER; }
    const uint32_t* t = reinterpret_cast<const uint32_t*>(table_host);
    const uint64_t range = c->high - c->low + 1;
    const uint64_t offset = c->code - c->low;
    const uint64_t value = ((offset + 1) * (uint32_t)total - 1) / range;
    uint32_t s = 0, e = (uint32_t)ncode;
    while (e - s > 1) {
        const uint32_t mid = (s + e) >> 1;
        if (t[mid] > value) e = mid; else s = mid;
    }
    int rc = ac_update<true>(c, t[s], t[s + 1], (uint32_t)total);
    *symbol = (int)s;
    return rc;
}

}  // extern "C"
