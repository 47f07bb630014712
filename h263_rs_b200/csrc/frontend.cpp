// frontend.cpp -- host front end: serial bitstream parse, one parser per stream, threaded
// across streams.  It stands in for H263Reader plus the serial loop of
// H263State::decode_next_picture (h263/src/decoder/state.rs:142-427, parser/*.rs,
// decoder/cpu/mvd_pred.rs) and emits the compact side info of include/h263cu.h.
//
// Written from the bitstream syntax (SURVEY.md Appendix A/B), not from the reference's
// control flow: table-driven VLC decode over a 64-bit window, no per-picture allocation,
// motion-vector prediction on the host.  Error values and the
// transactional "nothing changes on failure" contract follow the reference.
#include <algorithm>
#include <atomic>
#include <condition_variable>
#include <cstring>
#include <functional>
#include <mutex>
#include <new>
#include <pthread.h>
#include <thread>
#include <vector>

#include "../../include/h263cu.h"
#include "bitio.hpp"
#include "parse_mb.h"

namespace h263fe {

#include "vlc_codes.inc"

void VlcTable::build(const VlcCode* codes, int n) {
    max_len = 0;
    for (int i = 0; i < n; i++) max_len = std::max(max_len, codes[i].len);
    lut.assign((size_t)1 << max_len, VlcEntry{(uint8_t)(2u << 5), 0, 0, 0});
    for (int i = 0; i < n; i++) {
        uint32_t v = 0;
        for (int k = 0; k < codes[i].len; k++) v = (v << 1) | (uint32_t)(codes[i].bits[k] - '0');
        int rest = max_len - codes[i].len;
        VlcEntry e{(uint8_t)((unsigned)codes[i].len | ((unsigned)codes[i].kind << 5)), (int8_t)codes[i].a,
                   (uint8_t)codes[i].b, (uint8_t)codes[i].c};
        for (uint32_t s = 0; s < (1u << rest); s++) lut[((size_t)v << rest) | s] = e;
    }
}

namespace {
struct Tables {
    VlcTable t[5];
    // TCOEF again, laid out for the event loop: one word per (max code length + 1)-bit prefix, i.e. code AND sign bit =
    //   bits consumed[4:0] (code + sign) | kind[6:5] | last[7] | (run << 10 | level as a signed 10-bit field)[31:16]
    // so that one load yields the length to skip and the finished narrow event unit.  Escapes / invalid prefixes
    // carry the code length alone.
    std::vector<uint32_t> tcoef_fast;
    int tcoef_bits = 0;
    Tables() {
        t[T_MCBPC_I].build(MCBPC_I_CODES, MCBPC_I_CODES_COUNT);
        t[T_MCBPC_P].build(MCBPC_P_CODES, MCBPC_P_CODES_COUNT);
        t[T_CBPY].build(CBPY_CODES, CBPY_CODES_COUNT);
        t[T_MVD].build(MVD_CODES, MVD_CODES_COUNT);
        t[T_TCOEF].build(TCOEF_CODES, TCOEF_CODES_COUNT);
        tcoef_bits = t[T_TCOEF].max_len + 1;
        tcoef_fast.resize(t[T_TCOEF].lut.size() * 2);
        for (size_t i = 0; i < tcoef_fast.size(); i++) {
            const VlcEntry& e = t[T_TCOEF].lut[i >> 1];
            uint32_t w = e.len() | (e.kind() << 5);
            if (e.kind() == 0) {
                // the sign bit is the bit right after the code: bit (max_len - len) of the index, counted from the LSB
                const uint32_t sign = (uint32_t)(i >> (t[T_TCOEF].max_len - e.len())) & 1u;
                const uint32_t level = sign ? (0u - (uint32_t)e.c) & 0x3FFu : (uint32_t)e.c;
                w = (e.len() + 1u) | ((uint32_t)(e.a != 0) << 7) | ((((uint32_t)e.b << 10) | level) << 16);
            }
            tcoef_fast[i] = w;
        }
    }
};
const Tables& tables() {
    static const Tables T;
    return T;
}
}  // namespace

const VlcTable& vlc_table(int id) { return tables().t[id]; }
static const uint32_t* tcoef_fast_table(int* bits) {
    *bits = tables().tcoef_bits;
    return tables().tcoef_fast.data();
}
const VlcCode* vlc_codes(int id, int* count) {
    switch (id) {
        case T_MCBPC_I: *count = MCBPC_I_CODES_COUNT; return MCBPC_I_CODES;
        case T_MCBPC_P: *count = MCBPC_P_CODES_COUNT; return MCBPC_P_CODES;
        case T_CBPY: *count = CBPY_CODES_COUNT; return CBPY_CODES;
        case T_MVD: *count = MVD_CODES_COUNT; return MVD_CODES;
        default: *count = TCOEF_CODES_COUNT; return TCOEF_CODES;
    }
}

// ---------------------------------------------------------------------------------------
// Picture header
// ---------------------------------------------------------------------------------------
struct Header {
    int version = -1;  // Sorenson version field, -1 for baseline
    uint16_t tr = 0;
    int fmt_kind = -1;  // 0..4 standard sizes, 5 reserved, 6 custom
    uint16_t w = 0, h = 0;
    bool dims_valid = false;
    uint8_t pic_type = H263CU_PIC_I;
    bool type_supported = true;  // false: PB / reserved types (every coded MB is unimplemented)
    bool deblock = false;
    uint8_t quant = 0;
};

static bool std_dims(int kind, uint16_t* w, uint16_t* h) {
    static const uint16_t W[5] = {128, 176, 352, 704, 1408}, H[5] = {96, 144, 288, 576, 1152};
    if (kind < 0 || kind > 4) return false;
    *w = W[kind], *h = H[kind];
    return true;
}

// Start code search (reader.rs:240-258): 17 bits 0...01, preceded by stuffing that may not
// exceed the distance to the next byte boundary (plus the reference's off-by-one).
static int find_start_code(BitReader& r, uint32_t* skipped) {
    const size_t save = r.pos();
    uint32_t max_skip = (uint32_t)((8 - (r.pos() & 7)) & 7);
    uint32_t skip = 0;
    for (;;) {
        if (r.avail() < 17) {
            r.seek(save);
            return H263CU_ERR_UNHANDLED_IO_ERROR;
        }
        if (r.peek_padded(17) == 1) break;
        if (skip > max_skip) {
            r.seek(save);
            return H263CU_ERR_MIDDLE_OF_BITSTREAM;
        }
        r.consume(1);
        skip += 1;
    }
    r.seek(save);
    *skipped = skip;
    return 0;
}

#define RD(n, var)                                         \
    do {                                                   \
        if (!r.read((n), &(var))) return H263CU_ERR_UNHANDLED_IO_ERROR; \
    } while (0)

// picture.rs:611-817 (Sorenson branch :628-659, baseline PTYPE :21-81).
// prev_fmt_*: format of the previous picture header (baseline only; a change reaches the
// reference's RPRP stub, picture.rs:541-546,758-768).
static int parse_header(BitReader& r, uint32_t options, bool have_prev, int prev_kind, uint16_t prev_w,
                        uint16_t prev_h, Header* out) {
    uint32_t skipped = 0, v = 0;
    int e = find_start_code(r, &skipped);
    if (e) return e;
    if (!r.skip(17 + skipped)) return H263CU_ERR_UNHANDLED_IO_ERROR;
    uint32_t gob_id;
    RD(5, gob_id);
    Header h;
    if (options & H263CU_OPT_SORENSON_SPARK_BITSTREAM) {
        RD(8, v);
        h.tr = (uint16_t)v;
        uint32_t code;
        RD(3, code);
        switch (code) {
            case 0: {
                uint32_t cw, ch;
                RD(8, cw);
                RD(8, ch);
                h.fmt_kind = 6, h.w = (uint16_t)cw, h.h = (uint16_t)ch, h.dims_valid = true;
                break;
            }
            case 1: {
                uint32_t cw, ch;
                RD(16, cw);
                RD(16, ch);
                h.fmt_kind = 6, h.w = (uint16_t)cw, h.h = (uint16_t)ch, h.dims_valid = true;
                break;
            }
            case 2: h.fmt_kind = 2; break;
            case 3: h.fmt_kind = 1; break;
            case 4: h.fmt_kind = 0; break;
            case 5: h.fmt_kind = 6, h.w = 320, h.h = 240, h.dims_valid = true; break;
            case 6: h.fmt_kind = 6, h.w = 160, h.h = 120, h.dims_valid = true; break;
            default: h.fmt_kind = 5; break;
        }
        if (h.fmt_kind <= 4) h.dims_valid = std_dims(h.fmt_kind, &h.w, &h.h);
        RD(2, v);
        h.pic_type = (uint8_t)v;  // 0 I, 1 P, 2 disposable P
        if (v == 3) h.type_supported = false;
        RD(1, v);
        h.deblock = v == 1;
        RD(5, v);
        h.quant = (uint8_t)v;
        for (;;) {  // PEI / PSUPP
            RD(1, v);
            if (v != 1) break;
            RD(8, v);
        }
        h.version = (int)gob_id;
        *out = h;
        return 0;
    }
    if (gob_id != 0) return H263CU_ERR_MIDDLE_OF_BITSTREAM;  // decode_picture -> Ok(None)
    RD(8, v);
    h.tr = (uint16_t)v;
    uint32_t hi;
    RD(8, hi);
    if ((hi & 0xC0) != 0x80) return H263CU_ERR_INVALID_PTYPE;
    switch (hi & 7) {
        case 0: return H263CU_ERR_INVALID_PTYPE;
        case 7: return H263CU_ERR_UNIMPLEMENTED_DECODING;  // PLUSPTYPE: out of scope
        case 6: h.fmt_kind = 5; break;
        default: h.fmt_kind = (int)(hi & 7) - 1; break;
    }
    h.dims_valid = std_dims(h.fmt_kind, &h.w, &h.h);
    uint32_t lo;
    RD(5, lo);
    h.pic_type = (lo & 0x10) ? H263CU_PIC_I : H263CU_PIC_P;  // sic (picture.rs:57-61)
    if (lo & 1) h.pic_type = H263CU_PIC_OTHER, h.type_supported = false;  // PB frames (picture.rs:75-77)
    // UMV / SAC / AP bits are OPPTYPE options: masked out of the running options for
    // pictures without PLUSPTYPE (state.rs:152-155), hence without effect.
    if (have_prev && !(prev_kind == h.fmt_kind && (h.fmt_kind != 6 || (prev_w == h.w && prev_h == h.h))))
        return H263CU_ERR_UNIMPLEMENTED_DECODING;
    RD(5, v);
    h.quant = (uint8_t)v;
    RD(1, v);  // CPM
    if (v) RD(2, v);
    if (lo & 1) {
        RD(3, v);  // TRB
        RD(2, v);  // DBQUANT
    }
    for (;;) {
        RD(1, v);
        if (v != 1) break;
        RD(8, v);
    }
    h.version = -1;
    *out = h;
    return 0;
}

// ---------------------------------------------------------------------------------------
// Motion vector helpers (types.rs:736-798, mvd_pred.rs)
// ---------------------------------------------------------------------------------------
static inline int median3(int a, int b, int c) {
    int lo = std::min(a, b), hi = std::max(a, b);
    return std::max(lo, std::min(hi, c));
}
static inline int wrap_mv(int pred, int mvd) {
    int out = mvd + pred;
    if (out < -32 || out >= 32) out = (mvd > 0 ? mvd - 64 : (mvd < 0 ? mvd + 64 : 0)) + pred;
    return out;
}

struct Mv {
    int8_t x, y;
};

}  // namespace h263fe

using namespace h263fe;

// ---------------------------------------------------------------------------------------
// Parser object
// ---------------------------------------------------------------------------------------
struct h263cu_parser {
    uint32_t options = 0;
    // Stream state mirrored from H263State (state.rs:16-38)
    bool has_last = false;
    bool has_reference = false;
    int last_fmt_kind = -1;
    uint16_t last_w = 0, last_h = 0;
    uint16_t ref_w = 0, ref_h = 0;  // size of the last non-disposable picture (H263CU_OPT_DECODE_DISPOSABLE)
    // scratch
    std::vector<Mv> mvs;  // 4 per MB, current picture
    // per-picture staging used by h263cu_parse_step
    std::vector<h263cu_mb> st_mbs;
    std::vector<h263cu_event> st_events;
    h263cu_pic st_pic;
    int st_err = 0;
    // stream state after the picture parsed last by a deferred-commit parse step (h263fe::parse_step_deferred);
    // it becomes the parser's state only when the device stage has accepted the step
    struct Pending {
        bool valid = false;
        bool has_last = false, has_reference = false;
        int fmt_kind = -1;
        uint16_t w = 0, h = 0, ref_w = 0, ref_h = 0;
    } pending;
};

namespace {

struct PendingState {
    bool has_last, has_reference;
    int fmt_kind;
    uint16_t w, h, ref_w, ref_h;
};

// One block (block.rs:670-755).  Events go to ev_run/ev_level; returns 0 or an error.
// *overflow is set when the run lengths push the zig-zag index past 63 (rle.rs:125-127).
static inline int parse_block(BitReader& r_io, const Header& hd, uint32_t options, bool intra, bool coded, int* dc_code,
                              uint8_t* __restrict ev_run, int16_t* __restrict ev_level, int* nev, bool* overflow) {
    const VlcTable& T = vlc_table(T_TCOEF);
    // The reader works on a private copy whose address never escapes: the byte stores into ev_run / the records
    // may alias anything the compiler cannot prove local, and would otherwise force the bit window through memory
    // on every event.
    BitReader r = r_io;
    uint32_t v;
    *dc_code = -1;
    *nev = 0;
    *overflow = false;
    if (intra) {
        if (!r.read(8, &v)) return H263CU_ERR_UNHANDLED_IO_ERROR;
        if (v == 0 || v == 128) return H263CU_ERR_INVALID_INTRA_DC;
        *dc_code = (int)v;
    }
    if (!coded) {
        r_io = r;
        return 0;
    }
    const bool sorenson_v1 = (options & H263CU_OPT_SORENSON_SPARK_BITSTREAM) && hd.version == 1;
    int idx = intra ? 1 : 0;
    int n = 0;
    bool ovf = false;
    for (;;) {
        const VlcEntry* e;
        bool eof_sign;
        if (!r.read_vlc_bits(T, 1, &e, &v, &eof_sign)) return H263CU_ERR_UNHANDLED_IO_ERROR;  // code + sign bit from one window
        int last, run, level;
        if (e->kind() == 0) {
            last = e->a, run = e->b, level = v ? -(int)e->c : (int)e->c;
        } else if (e->kind() == 3) {
            unsigned width = 8;
            if (sorenson_v1) {
                if (!r.read(1, &v)) return H263CU_ERR_UNHANDLED_IO_ERROR;
                width = v ? 11 : 7;
            }
            uint32_t l, rn;
            int32_t lv;
            if (!r.read(1, &l) || !r.read(6, &rn) || !r.read_signed(width, &lv)) return H263CU_ERR_UNHANDLED_IO_ERROR;
            if (lv == 0) return H263CU_ERR_INVALID_LONG_COEFFICIENT;
            last = (int)l, run = (int)rn, level = lv;
        } else {
            return H263CU_ERR_INVALID_SHORT_COEFFICIENT;
        }
        idx += run;
        ovf |= idx >= 64;
        if (!ovf) {
            ev_run[n] = (uint8_t)run;
            ev_level[n] = (int16_t)level;
            n++;
        }
        idx += 1;
        if (last) break;
    }
    *overflow = ovf;
    *nev = ovf ? 0 : n;
    r_io = r;
    return 0;
}

// One block, the fast form (block.rs:670-755): events are written straight into the output as narrow units
// (RUN << 10 | LEVEL as a signed 10-bit field); *wide is set when some level does not fit, and the caller then
// re-reads the macroblock with parse_block (rare: Sorenson 11-bit escapes beyond +-511).  The reader is a local of the
// caller whose address never escapes, so the bit window stays in registers across the stores.
// A block whose runs overflow the zig-zag is dropped (*nev = 0, rle.rs:125-127) but still parsed to its end.
static H263_AI int parse_block_fast(BitReader& r, const uint32_t* __restrict tf, int tf_bits, bool sorenson_v1, bool intra, bool coded,
                                    int* dc_code, h263cu_event* __restrict out, int* nev, bool* overflow, bool* wide) {
    uint32_t v;
    *dc_code = -1;
    *nev = 0;
    *overflow = false;
    if (intra) {
        if (!r.read(8, &v)) return H263CU_ERR_UNHANDLED_IO_ERROR;
        if (v == 0 || v == 128) return H263CU_ERR_INVALID_INTRA_DC;
        *dc_code = (int)v;
    }
    if (!coded) return 0;
    int idx = intra ? 1 : 0;
    int n = 0;
    bool ovf = false;
    for (;;) {
        const uint64_t w = r.window();
        const uint32_t e = tf[(uint32_t)(w >> (64 - tf_bits))];
        const unsigned len = e & 31u, kind = (e >> 5) & 3u;
        int last, run, level;
        uint32_t unit;
        if (__builtin_expect(kind == 0, 1)) {
            if (__builtin_expect(len > r.avail(), 0)) return H263CU_ERR_UNHANDLED_IO_ERROR;  // the code or its sign bit is cut off
            r.consume(len);
            last = (int)((e >> 7) & 1u);
            unit = e >> 16;
            run = (int)(e >> 26);
        } else if (kind == 3) {
            if (len > r.avail()) return H263CU_ERR_UNHANDLED_IO_ERROR;
            r.consume(len);
            unsigned width = 8;
            if (sorenson_v1) {
                if (!r.read(1, &v)) return H263CU_ERR_UNHANDLED_IO_ERROR;
                width = v ? 11 : 7;
            }
            uint32_t l, rn;
            int32_t lv;
            if (!r.read(1, &l) || !r.read(6, &rn) || !r.read_signed(width, &lv)) return H263CU_ERR_UNHANDLED_IO_ERROR;
            if (lv == 0) return H263CU_ERR_INVALID_LONG_COEFFICIENT;
            last = (int)l, run = (int)rn, level = lv;
            *wide |= level < -512 || level > 511;
            unit = ((uint32_t)run << 10) | ((uint32_t)level & 0x3FFu);
        } else {
            if (len > r.avail()) return H263CU_ERR_UNHANDLED_IO_ERROR;
            return H263CU_ERR_INVALID_SHORT_COEFFICIENT;
        }
        idx += run;
        if (__builtin_expect(idx >= 64, 0))
            ovf = true;
        else if (!ovf)
            out[n++] = (h263cu_event)unit;
        idx += 1;
        if (last) break;
    }
    *overflow = ovf;
    *nev = ovf ? 0 : n;
    return 0;
}

// The serial loop of decode_next_picture (state.rs:142-427) for one packet.
static int parse_picture_impl(h263cu_parser* p, const uint8_t* data, size_t len, uint32_t stream, uint16_t pic_index,
                              uint32_t mb_base, uint32_t ev_base, h263cu_pic* pic, h263cu_mb* mbs, uint32_t mb_cap,
                              h263cu_event* events, uint32_t ev_cap, PendingState* pending) {
    BitReader r0(data, len);
    Header hd;
    int e = parse_header(r0, p->options, p->has_last, p->last_fmt_kind, p->last_w, p->last_h, &hd);
    if (e) return e;
    // The macroblock loop works on its own copy of the reader, every use of which is inlined: its address never
    // escapes, so the 64-bit window stays in registers across the byte stores into the records (which may alias
    // anything the compiler cannot prove local).  Out-of-line helpers get a copy.
    BitReader r = r0;
    int tf_bits;
    const uint32_t* const tf = tcoef_fast_table(&tf_bits);
    const bool sorenson_v1 = (p->options & H263CU_OPT_SORENSON_SPARK_BITSTREAM) && hd.version == 1;
    if (!hd.dims_valid) return H263CU_ERR_PICTURE_FORMAT_INVALID;
    const uint32_t W = hd.w, H = hd.h;
    const uint32_t mb_w = (W + 15) / 16, mb_h = (H + 15) / 16;
    if (mb_w == 0) return H263CU_ERR_REFERENCE_WOULD_ABORT;  // `len % mb_per_line` (state.rs:200)
    if (mb_w > 255 || mb_h > 255) return H263CU_ERR_CAPACITY;
    const uint32_t capacity = mb_w * mb_h;
    if (capacity > mb_cap) return H263CU_ERR_CAPACITY;

    const bool is_sorenson = (p->options & H263CU_OPT_SORENSON_SPARK_BITSTREAM) != 0;
    // EXTENSION: disposable P pictures parse like P pictures and never become the reference
    const bool decode_disposable = (p->options & H263CU_OPT_DECODE_DISPOSABLE) != 0;
    const bool is_i = hd.pic_type == H263CU_PIC_I;
    const VlcTable& TMt = vlc_table(is_i ? T_MCBPC_I : T_MCBPC_P);
    const VlcTable& TCt = vlc_table(T_CBPY);
    const VlcTable& TVt = vlc_table(T_MVD);
    const VlcEntry* const TM = TMt.lut.data();
    const VlcEntry* const TC = TCt.lut.data();
    const VlcEntry* const TV = TVt.lut.data();
    const unsigned TM_len = (unsigned)TMt.max_len, TC_len = (unsigned)TCt.max_len, TV_len = (unsigned)TVt.max_len;

    p->mvs.assign((size_t)capacity * 4, Mv{0, 0});
    Mv* mvs = p->mvs.data();

    int quant = hd.quant;
    uint32_t n = 0;        // macroblocks decoded so far (may exceed capacity with trailing COD=1 bits)
    uint32_t col = 0, row = 0;  // = n % mb_w, n / mb_w, kept by increments
    uint32_t ev_used = 0;  // event units written
    bool any_inter = false;
    bool mv_in_range = true;  // halfpel_decode wraps every component into [-32, 31] (mvd_pred.rs:70-117); checked anyway
    uint8_t ev_run[6][64];
    int16_t ev_level[6][64];

    for (;;) {
        const size_t mb_start = r.pos();
        uint32_t v;
        int err = 0;
        bool uncoded = false, stuffing = false;
        int mb_type = 0;
        bool cbp[6] = {false, false, false, false, false, false};
        int dquant = 0;
        Mv mvd[4] = {{0, 0}, {0, 0}, {0, 0}, {0, 0}};

        // ---- macroblock header (macroblock.rs:445-549) ----
        do {
            if (!is_i) {
                if (!r.read(1, &v)) {
                    err = H263CU_ERR_UNHANDLED_IO_ERROR;
                    break;
                }
                if (v) {
                    uncoded = true;
                    break;
                }
            }
            if (!is_i && hd.pic_type != H263CU_PIC_P && !(decode_disposable && hd.pic_type == H263CU_PIC_DISPOSABLE_P)) {
                err = H263CU_ERR_UNIMPLEMENTED_DECODING;  // disposable (without the extension) / unsupported types
                break;
            }
            if (!hd.type_supported) {
                err = H263CU_ERR_UNIMPLEMENTED_DECODING;
                break;
            }
            const VlcEntry* en;
            if (!r.read_vlc(TM, TM_len, &en)) {
                err = H263CU_ERR_UNHANDLED_IO_ERROR;
                break;
            }
            if (en->kind() == 1) {
                stuffing = true;
                break;
            }
            if (en->kind() != 0) {
                err = H263CU_ERR_INVALID_MACROBLOCK_HEADER;
                break;
            }
            mb_type = en->a;
            cbp[4] = en->b != 0, cbp[5] = en->c != 0;
            if (!r.read_vlc(TC, TC_len, &en)) {
                err = H263CU_ERR_UNHANDLED_IO_ERROR;
                break;
            }
            if (en->kind() != 0) {
                err = H263CU_ERR_INVALID_MACROBLOCK_CODED_BITS;
                break;
            }
            const bool intra = mb_type == 3 || mb_type == 4;
            int y = intra ? en->a : (~en->a & 15);
            cbp[0] = (y & 8) != 0, cbp[1] = (y & 4) != 0, cbp[2] = (y & 2) != 0, cbp[3] = (y & 1) != 0;
            if (mb_type == 1 || mb_type == 4 || mb_type == 5) {
                if (!r.read(2, &v)) {
                    err = H263CU_ERR_UNHANDLED_IO_ERROR;
                    break;
                }
                static const int DQ[4] = {-1, -2, 1, 2};
                dquant = DQ[v];
            }
            if (!intra) {
                int nmv = (mb_type == 2 || mb_type == 5) ? 4 : 1;
                for (int k = 0; k < nmv && !err; k++) {
                    for (int c = 0; c < 2; c++) {
                        if (!r.read_vlc(TV, TV_len, &en)) {
                            err = H263CU_ERR_UNHANDLED_IO_ERROR;
                            break;
                        }
                        if (en->kind() != 0) {
                            err = H263CU_ERR_INVALID_MVD;
                            break;
                        }
                        (c ? mvd[k].y : mvd[k].x) = en->a;
                    }
                }
            }
        } while (0);

        if (err) {
            r.seek(mb_start);  // decode_macroblock is a transaction
            if (err == H263CU_ERR_UNHANDLED_IO_ERROR) break;  // EOF ends the picture (state.rs:411)
            if ((err == H263CU_ERR_INVALID_MACROBLOCK_HEADER || err == H263CU_ERR_INVALID_MACROBLOCK_CODED_BITS) &&
                !is_sorenson) {
                // GOB resynchronisation stub (state.rs:387-408, gob.rs:50-71)
                uint32_t skipped = 0;
                BitReader probe = r;
                int ge = find_start_code(probe, &skipped);
                if (ge == H263CU_ERR_MIDDLE_OF_BITSTREAM) break;  // InvalidGobHeader ends the picture
                if (ge) break;                                    // EOF ends the picture
                if (r.avail() < 17 + skipped + 5) break;          // EOF while reading the GOB number
                const size_t save = r.pos();
                r.seek(save + 17 + skipped);
                uint32_t gn = r.peek_padded(5);
                r.seek(save);
                if (gn == 0 || gn == 15) break;  // picture start / EOS: end of this picture
                return H263CU_ERR_UNIMPLEMENTED_DECODING;
            }
            return err;
        }
        if (stuffing) continue;  // consumes no macroblock slot (state.rs:206)

        if (uncoded) {
            if (is_i) return H263CU_ERR_UNCODED_IFRAME_BLOCKS;  // unreachable: I pictures have no COD
            if (n < capacity) {
                h263cu_mb& m = mbs[n];
                std::memset(&m, 0, sizeof(m));
                m.ev_off = ev_used;
                m.pic = pic_index;
                m.mbx = (uint8_t)col, m.mby = (uint8_t)row;
                m.flags = H263CU_MB_INTER;
                m.quant = (uint8_t)quant;
                any_inter = true;
            }
            n++;
            if (++col == mb_w) col = 0, row++;
            continue;
        }

        // ---- coded macroblock ----
        quant = std::min(std::max(quant + dquant, 1), 31);
        const bool intra = mb_type == 3 || mb_type == 4;
        if (n >= capacity) {
            // One macroblock too many: the reference still parses the first block (whose
            // errors win) and then indexes past its coefficient array and aborts (rle.rs:89-90).
            int dc, nev0;
            bool ovf;
            BitReader tmp = r;
            int be = parse_block(tmp, hd, p->options, intra, cbp[0], &dc, ev_run[0], ev_level[0], &nev0, &ovf);
            return be ? be : H263CU_ERR_REFERENCE_WOULD_ABORT;
        }
        Mv* cur = mvs + (size_t)n * 4;
        if (!intra) {
            const bool four = mb_type == 2 || mb_type == 5;
            const Mv zero{0, 0};
            for (int k = 0; k < (four ? 4 : 1); k++) {
                // candidates (mvd_pred.rs:27-67)
                Mv c1, c2, c3;
                if (k == 0 || k == 2)
                    c1 = col == 0 ? zero : mvs[(size_t)(n - 1) * 4 + k + 1];
                else
                    c1 = cur[k - 1];
                if (k < 2) {
                    c2 = row == 0 ? c1 : mvs[(size_t)(n - mb_w) * 4 + k + 2];
                    if (col == mb_w - 1)
                        c3 = zero;
                    else if (row == 0)
                        c3 = c1;
                    else
                        c3 = mvs[(size_t)(n - mb_w + 1) * 4 + 2];
                } else {
                    c2 = cur[0];
                    c3 = cur[1];
                }
                int px = median3(c1.x, c2.x, c3.x), py = median3(c1.y, c2.y, c3.y);
                cur[k].x = (int8_t)wrap_mv(px, mvd[k].x);
                cur[k].y = (int8_t)wrap_mv(py, mvd[k].y);
                mv_in_range &= cur[k].x >= -32 && cur[k].x <= 31 && cur[k].y >= -32 && cur[k].y <= 31;
            }
            if (!four) cur[1] = cur[2] = cur[3] = cur[0];
            any_inter = true;
        }

        h263cu_mb& m = mbs[n];
        std::memset(&m, 0, sizeof(m));
        m.ev_off = ev_used;
        m.pic = pic_index;
        m.mbx = (uint8_t)col, m.mby = (uint8_t)row;
        m.quant = (uint8_t)quant;
        m.flags = (uint8_t)(H263CU_MB_CODED | (intra ? 0 : H263CU_MB_INTER) |
                            ((mb_type == 2 || mb_type == 5) ? H263CU_MB_FOURMV : 0));
        int nev[6];
        bool wide = false;
        uint32_t units = 0;
        if (ev_cap - ev_used >= 6 * 65) {
            // fast path: narrow units straight into the output (a block writes at most 65 units before it stops counting)
            const size_t blocks_start = r.pos();
            h263cu_event* ev = events + ev_used;
            int be = 0;
            for (int b = 0; b < 6 && !be; b++) {
                int dc;
                bool ovf;
                be = parse_block_fast(r, tf, tf_bits, sorenson_v1, intra, cbp[b], &dc, ev, &nev[b], &ovf, &wide);
                if (intra) m.u.intradc[b] = ovf ? 0 : (uint8_t)dc;
                m.nev[b] = (uint8_t)nev[b];
                ev += nev[b];
            }
            if (be) return be;  // `?`: block errors, EOF included, fail the whole picture
            if (!wide) {
                units = (uint32_t)(ev - (events + ev_used));
            } else {
                r.seek(blocks_start);  // some level needs 16 bits: read the macroblock again in the wide form
            }
        } else {
            wide = true;  // almost out of room: take the careful path, which checks the capacity exactly
        }
        if (wide) {
            wide = false;
            BitReader tmp = r;
            for (int b = 0; b < 6; b++) {
                int dc;
                bool ovf;
                int be = parse_block(tmp, hd, p->options, intra, cbp[b], &dc, ev_run[b], ev_level[b], &nev[b], &ovf);
                if (be) return be;
                if (intra) m.u.intradc[b] = ovf ? 0 : (uint8_t)dc;
                m.nev[b] = (uint8_t)nev[b];
                for (int k = 0; k < nev[b]; k++) wide |= ev_level[b][k] < -512 || ev_level[b][k] > 511;
            }
            r = tmp;
            uint32_t total = 0;
            for (int b = 0; b < 6; b++) total += (uint32_t)nev[b];
            units = wide ? total * 2 : total;
            if (ev_used + units > ev_cap) return H263CU_ERR_CAPACITY;
            h263cu_event* ev = events + ev_used;
            if (wide) {
                m.flags |= H263CU_MB_WIDE;
                for (int b = 0; b < 6; b++)
                    for (int k = 0; k < nev[b]; k++) {
                        *ev++ = ev_run[b][k];
                        *ev++ = (uint16_t)ev_level[b][k];
                    }
            } else {
                for (int b = 0; b < 6; b++)
                    for (int k = 0; k < nev[b]; k++)
                        *ev++ = (uint16_t)(((uint32_t)ev_run[b][k] << 10) | ((uint32_t)ev_level[b][k] & 0x3FF));
            }
        }
        if (!intra)
            for (int k = 0; k < 4; k++) m.u.mv[k][0] = cur[k].x, m.u.mv[k][1] = cur[k].y;
        ev_used += units;
        n++;
        if (++col == mb_w) col = 0, row++;
    }

    // A picture that ended early is padded with uncoded inter MBs (state.rs:419-427)
    for (uint32_t i = n; i < capacity; i++) {
        h263cu_mb& m = mbs[i];
        std::memset(&m, 0, sizeof(m));
        m.ev_off = ev_used;
        m.pic = pic_index;
        m.mbx = (uint8_t)(i % mb_w), m.mby = (uint8_t)(i / mb_w);
        m.flags = H263CU_MB_INTER;
        m.quant = (uint8_t)quant;
        any_inter = true;
    }

    // gather()'s checks (gather.rs:148-149; SURVEY.md 7.0 on mismatching dimensions)
    if (any_inter) {
        if (!(p->has_reference && p->has_last)) return H263CU_ERR_UNCODED_IFRAME_BLOCKS;
        // the prediction source: the last picture (the reference's get_reference_picture, state.rs:72-78), or the last
        // non-disposable one under the extension
        const uint16_t rw = decode_disposable ? p->ref_w : p->last_w, rh = decode_disposable ? p->ref_h : p->last_h;
        if (rw != W || rh != H) return H263CU_ERR_REFERENCE_WOULD_ABORT;
    }

    std::memset(pic, 0, sizeof(*pic));
    pic->stream = stream;
    pic->width = (uint16_t)W, pic->height = (uint16_t)H;
    pic->mb_w = (uint8_t)mb_w, pic->mb_h = (uint8_t)mb_h;
    pic->pic_type = hd.pic_type;
    pic->pquant = hd.quant;
    const bool disposable = decode_disposable && hd.pic_type == H263CU_PIC_DISPOSABLE_P;
    pic->flags = (uint8_t)((hd.deblock ? H263CU_PICFLAG_DEBLOCK : 0) | (any_inter ? H263CU_PICFLAG_HAS_INTER : 0) |
                           (mv_in_range ? H263CU_PICFLAG_MV_IN_RANGE : 0) | (disposable ? H263CU_PICFLAG_DISPOSABLE : 0));
    pic->version = hd.version < 0 ? 0xFF : (uint8_t)hd.version;
    pic->first_mb = mb_base;
    pic->n_mbs = capacity;
    pic->first_event = ev_base;
    pic->n_event_units = ev_used;
    pic->temporal_reference = hd.tr;

    // reference bookkeeping (state.rs:464-483)
    pending->has_last = true;
    pending->has_reference = p->has_reference;
    if (is_i) pending->has_reference = false;
    if (hd.pic_type != H263CU_PIC_DISPOSABLE_P) pending->has_reference = true;
    pending->fmt_kind = hd.fmt_kind;
    pending->w = (uint16_t)W, pending->h = (uint16_t)H;
    pending->ref_w = disposable ? p->ref_w : (uint16_t)W, pending->ref_h = disposable ? p->ref_h : (uint16_t)H;
    return 0;
}

static inline void commit(h263cu_parser* p, const PendingState& s) {
    p->has_last = s.has_last;
    p->has_reference = s.has_reference;
    p->last_fmt_kind = s.fmt_kind;
    p->last_w = s.w, p->last_h = s.h;
    p->ref_w = s.ref_w, p->ref_h = s.ref_h;
}

}  // namespace

namespace {
// Persistent worker threads for h263cu_parse_step: a step is parsed every few milliseconds, and creating and joining
// 2 x (threads - 1) std::threads per step cost a sixth of the parse itself.  One job at a time (callers serialise on
// the job mutex); the workers are detached and live until the process ends.
class WorkerPool {
  public:
    // runs fn on `threads` threads (the caller is one of them) and returns when all have finished
    void run(int threads, const std::function<void()>& fn) {
        if (threads <= 1) {
            fn();
            return;
        }
        std::lock_guard<std::mutex> job(job_mutex_);
        {
            std::unique_lock<std::mutex> lk(m_);
            while ((int)n_workers_ < threads - 1) {
                std::thread(&WorkerPool::worker, this, n_workers_).detach();
                n_workers_++;
            }
            fn_ = &fn;
            wanted_ = threads - 1;
            running_ = threads - 1;
            generation_++;
        }
        cv_.notify_all();
        fn();
        std::unique_lock<std::mutex> lk(m_);
        done_.wait(lk, [&] { return running_ == 0; });
        fn_ = nullptr;
    }

  private:
    void worker(size_t index) {
        uint64_t seen = 0;
        for (;;) {
            const std::function<void()>* fn;
            {
                std::unique_lock<std::mutex> lk(m_);
                cv_.wait(lk, [&] { return generation_ != seen; });
                seen = generation_;
                if ((int)index >= wanted_) continue;  // this job uses fewer workers
                fn = fn_;
            }
            (*fn)();
            std::lock_guard<std::mutex> lk(m_);
            if (--running_ == 0) done_.notify_all();
        }
    }
    std::mutex job_mutex_, m_;
    std::condition_variable cv_, done_;
    const std::function<void()>* fn_ = nullptr;
    size_t n_workers_ = 0;
    int wanted_ = 0, running_ = 0;
    uint64_t generation_ = 0;
};
// never destroyed: the detached workers may outlive static destructors.  Threads do not survive fork(): the child
// starts with a fresh pool (the old object, with its possibly locked mutexes, is abandoned).
WorkerPool* g_pool = nullptr;
std::once_flag g_pool_once;
WorkerPool& worker_pool() {
    std::call_once(g_pool_once, [] {
        g_pool = new WorkerPool();
        pthread_atfork(nullptr, nullptr, [] { g_pool = new WorkerPool(); });
    });
    return *g_pool;
}
}  // namespace

extern "C" {

h263cu_parser* h263cu_parser_create(uint32_t decoder_options) {
    h263cu_parser* p = new (std::nothrow) h263cu_parser();
    if (p) p->options = decoder_options;
    (void)tables();
    return p;
}
void h263cu_parser_destroy(h263cu_parser* p) { delete p; }
uint32_t h263cu_parser_options(const h263cu_parser* p) { return p ? p->options : 0u; }
void h263cu_parser_reset(h263cu_parser* p) {
    if (!p) return;
    p->has_last = p->has_reference = false;
    p->last_fmt_kind = -1;
    p->last_w = p->last_h = 0;
    p->ref_w = p->ref_h = 0;
}

int h263cu_peek_picture(uint32_t decoder_options, const uint8_t* data, size_t len, h263cu_pic* pic) {
    if (!data || !pic) return H263CU_ERR_BAD_ARGUMENT;
    BitReader r(data, len);
    Header hd;
    int e = parse_header(r, decoder_options, false, -1, 0, 0, &hd);
    if (e) return e;
    std::memset(pic, 0, sizeof(*pic));
    if (hd.dims_valid) {
        pic->width = hd.w, pic->height = hd.h;
        uint32_t mw = (hd.w + 15u) / 16u, mh = (hd.h + 15u) / 16u;
        pic->mb_w = (uint8_t)std::min(mw, 255u), pic->mb_h = (uint8_t)std::min(mh, 255u);
        pic->n_mbs = mw * mh;
    }
    pic->pic_type = hd.pic_type;
    pic->pquant = hd.quant;
    pic->flags = hd.deblock ? H263CU_PICFLAG_DEBLOCK : 0;
    pic->version = hd.version < 0 ? 0xFF : (uint8_t)hd.version;
    pic->temporal_reference = hd.tr;
    return 0;
}

int h263cu_parse_picture(h263cu_parser* p, const uint8_t* data, size_t len, uint32_t stream, uint16_t pic_index,
                         uint32_t mb_base, uint32_t ev_base, h263cu_pic* pic, h263cu_mb* mbs, uint32_t mb_cap,
                         h263cu_event* events, uint32_t ev_cap) {
    if (!p || !data || !pic || !mbs || (!events && ev_cap)) return H263CU_ERR_BAD_ARGUMENT;
    PendingState s;
    int e = parse_picture_impl(p, data, len, stream, pic_index, mb_base, ev_base, pic, mbs, mb_cap, events, ev_cap, &s);
    if (e) return e;
    commit(p, s);
    return 0;
}

static int parse_step_impl(h263cu_parser* const* parsers, const uint8_t* const* packets, const size_t* lens,
                           const uint32_t* stream_ids, uint32_t n, int threads, h263cu_pic* pics, h263cu_mb* mbs,
                           uint32_t mb_cap, h263cu_event* events, uint32_t ev_cap, uint32_t* n_pics_out,
                           uint32_t* n_mbs_out, uint32_t* n_units_out, int* per_pic_err, int32_t* pic_of_input,
                           bool commit_now, uint32_t max_w, uint32_t max_h, const uint32_t* min_size) {
    if (!parsers || !packets || !lens || !pics || !mbs || !n_pics_out || !n_mbs_out || !n_units_out)
        return H263CU_ERR_BAD_ARGUMENT;
    for (uint32_t i = 0; i < n; i++)
        if (parsers[i]) parsers[i]->pending.valid = false;
    if (n > 65535) return H263CU_ERR_CAPACITY;
    if (threads <= 0) threads = (int)std::max(1u, std::thread::hardware_concurrency());
    threads = (int)std::min<uint32_t>((uint32_t)threads, std::max(1u, n));
    std::vector<PendingState> pend(n);

    // phase 1: parse every packet into its parser's staging buffers (parallel over streams)
    std::atomic<uint32_t> next{0};
    auto work1 = [&]() {
        for (;;) {
            uint32_t i = next.fetch_add(1);
            if (i >= n) break;
            h263cu_parser* p = parsers[i];
            if (!p) continue;  // reported as H263CU_ERR_BAD_ARGUMENT below
            int e = 0;
            h263cu_pic hdr;
            if (!packets[i]) e = H263CU_ERR_BAD_ARGUMENT;
            if (!e) e = h263cu_peek_picture(p->options, packets[i], lens[i], &hdr);
            if (!e && hdr.n_mbs == 0) e = H263CU_ERR_PICTURE_FORMAT_INVALID;
            // a hostile header (Sorenson's 16-bit custom size) must not size the staging: more than 255 macroblocks
            // per row / column cannot be described by a record, and a picture beyond the context is this picture's
            // error, not the step's
            if (!e && ((hdr.width + 15u) / 16u > 255u || (hdr.height + 15u) / 16u > 255u)) e = H263CU_ERR_CAPACITY;
            if (!e && max_w && (hdr.width > max_w || hdr.height > max_h)) e = H263CU_ERR_CAPACITY;
            // a crop box of the caller's that does not fit the picture (h263cu_decode_step_device_tensor_fit)
            if (!e && min_size && (hdr.width < min_size[2 * i] || hdr.height < min_size[2 * i + 1])) e = H263CU_ERR_BAD_ARGUMENT;
            if (!e) {
                try {
                    p->st_mbs.resize(hdr.n_mbs);
                    // every event costs at least 3 bits and takes at most 2 units (wide MBs)
                    p->st_events.resize(lens[i] * 16 / 3 + 16);
                } catch (const std::bad_alloc&) {
                    e = H263CU_ERR_OUT_OF_MEMORY;
                }
            }
            if (!e) {
                e = parse_picture_impl(p, packets[i], lens[i], stream_ids ? stream_ids[i] : i, 0, 0, 0, &p->st_pic,
                                       p->st_mbs.data(), (uint32_t)p->st_mbs.size(), p->st_events.data(),
                                       (uint32_t)p->st_events.size(), &pend[i]);
            }
            p->st_err = e;
        }
    };
    worker_pool().run(threads, work1);

    // phase 2: pack the successful pictures densely
    uint32_t np = 0, nm = 0, nu = 0;
    std::vector<uint32_t> mb_base(n), ev_base(n);
    std::vector<int32_t> packed(n, -1);
    for (uint32_t i = 0; i < n; i++) {
        h263cu_parser* p = parsers[i];
        if (!p) {
            if (per_pic_err) per_pic_err[i] = H263CU_ERR_BAD_ARGUMENT;
            continue;
        }
        if (per_pic_err) per_pic_err[i] = p->st_err;
        if (p->st_err) continue;
        if ((uint64_t)nm + p->st_pic.n_mbs > mb_cap || (uint64_t)nu + p->st_pic.n_event_units > ev_cap)
            return H263CU_ERR_CAPACITY;
        packed[i] = (int32_t)np;
        mb_base[i] = nm, ev_base[i] = nu;
        np++;
        nm += p->st_pic.n_mbs;
        nu += p->st_pic.n_event_units;
    }
    next.store(0);
    auto work2 = [&]() {
        for (;;) {
            uint32_t i = next.fetch_add(1);
            if (i >= n) break;
            if (packed[i] < 0) continue;
            h263cu_parser* p = parsers[i];
            h263cu_pic pc = p->st_pic;
            pc.first_mb = mb_base[i];
            pc.first_event = ev_base[i];
            pics[packed[i]] = pc;
            h263cu_mb* dst = mbs + mb_base[i];
            std::memcpy(dst, p->st_mbs.data(), (size_t)pc.n_mbs * sizeof(h263cu_mb));
            for (uint32_t k = 0; k < pc.n_mbs; k++) dst[k].pic = (uint16_t)packed[i];
            if (pc.n_event_units)
                std::memcpy(events + ev_base[i], p->st_events.data(), (size_t)pc.n_event_units * sizeof(h263cu_event));
            if (commit_now) {
                commit(p, pend[i]);
            } else {
                p->pending.valid = true;
                p->pending.has_last = pend[i].has_last, p->pending.has_reference = pend[i].has_reference;
                p->pending.fmt_kind = pend[i].fmt_kind, p->pending.w = pend[i].w, p->pending.h = pend[i].h;
                p->pending.ref_w = pend[i].ref_w, p->pending.ref_h = pend[i].ref_h;
            }
        }
    };
    worker_pool().run(threads, work2);
    if (pic_of_input) std::memcpy(pic_of_input, packed.data(), n * sizeof(int32_t));
    *n_pics_out = np;
    *n_mbs_out = nm;
    *n_units_out = nu;
    return 0;
}

int h263cu_parse_step(h263cu_parser* const* parsers, const uint8_t* const* packets, const size_t* lens,
                      const uint32_t* stream_ids, uint32_t n, int threads, h263cu_pic* pics, h263cu_mb* mbs,
                      uint32_t mb_cap, h263cu_event* events, uint32_t ev_cap, uint32_t* n_pics_out,
                      uint32_t* n_mbs_out, uint32_t* n_units_out, int* per_pic_err, int32_t* pic_of_input) {
    try {
        return parse_step_impl(parsers, packets, lens, stream_ids, n, threads, pics, mbs, mb_cap, events, ev_cap, n_pics_out,
                               n_mbs_out, n_units_out, per_pic_err, pic_of_input, true, 0, 0, nullptr);
    } catch (const std::bad_alloc&) {
        return H263CU_ERR_OUT_OF_MEMORY;
    }
}

// ---- test hooks: the front end's own bit reader, tables and block decoder behind plain C calls, so that the
// reference's parser known-answer tests (reader.rs:448-559, macroblock.rs:551-1010, block.rs:757-2124) are replayed
// on the PRODUCT code and not only on the oracle (tests/test_frontend_kats.py).  Not on any decode path.
int h263cu_test_read_bits(const uint8_t* data, size_t len, size_t* bitpos, int nbits, int is_signed, int peek, int64_t* value) {
    if (!data || !bitpos || !value || nbits < 0 || nbits > 32) return H263CU_ERR_BAD_ARGUMENT;
    BitReader r(data, len);
    if (*bitpos > len * 8) return H263CU_ERR_BAD_ARGUMENT;
    r.seek(*bitpos);
    if (nbits == 0) {
        *value = 0;
        return 0;
    }
    if (is_signed) {
        int32_t v;
        if (!r.read_signed((unsigned)nbits, &v)) return H263CU_ERR_UNHANDLED_IO_ERROR;
        *value = v;
    } else {
        uint32_t v;
        if (!r.read((unsigned)nbits, &v)) return H263CU_ERR_UNHANDLED_IO_ERROR;
        *value = v;
    }
    if (!peek) *bitpos = r.pos();
    return 0;
}

int h263cu_test_start_code(const uint8_t* data, size_t len, size_t bitpos, int* skipped) {
    if (!data || !skipped || bitpos > len * 8) return H263CU_ERR_BAD_ARGUMENT;
    BitReader r(data, len);
    r.seek(bitpos);
    uint32_t sk = 0;
    const int e = find_start_code(r, &sk);
    *skipped = e ? -1 : (int)sk;
    return e;
}

int h263cu_test_read_vlc(int table, const uint8_t* data, size_t len, size_t* bitpos, int* out4) {
    if (table < 0 || table > 4 || !data || !bitpos || !out4 || *bitpos > len * 8) return H263CU_ERR_BAD_ARGUMENT;
    BitReader r(data, len);
    r.seek(*bitpos);
    const VlcEntry* e;
    if (!r.read_vlc(vlc_table(table), &e)) return H263CU_ERR_UNHANDLED_IO_ERROR;
    *bitpos = r.pos();
    out4[0] = (int)e->kind(), out4[1] = e->a, out4[2] = e->b, out4[3] = e->c;
    return 0;
}

int h263cu_test_decode_block(const uint8_t* data, size_t len, size_t* bitpos, uint32_t decoder_options, int version, int is_intra,
                             int tcoef_present, int* intradc_code, int* n_events, uint8_t* run, int16_t* level, int* overflow) {
    if (!data || !bitpos || !intradc_code || !n_events || !run || !level || *bitpos > len * 8) return H263CU_ERR_BAD_ARGUMENT;
    BitReader r(data, len);
    r.seek(*bitpos);
    Header hd;
    hd.version = version;
    uint8_t ev_run[64];
    int16_t ev_level[64];
    bool ovf = false;
    const int e = parse_block(r, hd, decoder_options, is_intra != 0, tcoef_present != 0, intradc_code, ev_run, ev_level, n_events, &ovf);
    if (e) return e;
    for (int k = 0; k < *n_events; k++) run[k] = ev_run[k], level[k] = ev_level[k];
    if (overflow) *overflow = ovf;
    *bitpos = r.pos();
    return 0;
}

int h263cu_is_eof_error(int err) { return err == H263CU_ERR_UNHANDLED_IO_ERROR; }
int h263cu_is_macroblock_error(int err) {
    return err == H263CU_ERR_INVALID_MACROBLOCK_HEADER || err == H263CU_ERR_INVALID_MACROBLOCK_CODED_BITS;
}
int h263cu_is_gob_error(int err) { return err == H263CU_ERR_INVALID_GOB_HEADER; }

const char* h263cu_strerror(int err) {
    switch (err) {
        case H263CU_OK: return "ok";
        case H263CU_ERR_INTERNAL_DECODER_ERROR: return "the H.263 decoder failed internally, this is a bug";
        case H263CU_ERR_MIDDLE_OF_BITSTREAM: return "the H.263 bitstream doesn't start with a picture";
        case H263CU_ERR_INVALID_MACROBLOCK_HEADER: return "the H.263 bitstream contains an invalid macroblock header";
        case H263CU_ERR_INVALID_MACROBLOCK_CODED_BITS: return "the H.263 bitstream contains invalid macroblock coded bits";
        case H263CU_ERR_INVALID_INTRA_DC: return "the H.263 bitstream contains an invalid intra-dc coefficient";
        case H263CU_ERR_INVALID_SHORT_COEFFICIENT: return "the H.263 bitstream contains an invalid short ac coefficient";
        case H263CU_ERR_INVALID_LONG_COEFFICIENT: return "the H.263 bitstream contains an invalid long ac coefficient";
        case H263CU_ERR_INVALID_MVD: return "the H.263 bitstream contains an invalid motion vector";
        case H263CU_ERR_INVALID_PTYPE: return "the H.263 bitstream has an invalid picture type";
        case H263CU_ERR_INVALID_PLUSPTYPE: return "the H.263 bitstream has an invalid extension picture type";
        case H263CU_ERR_INVALID_GOB_HEADER: return "the H.263 bitstream has an invalid group-of-blocks header";
        case H263CU_ERR_INVALID_BITSTREAM: return "the H.263 bitstream could not be decoded";
        case H263CU_ERR_PICTURE_FORMAT_MISSING: return "the decoded H.263 bitstream is missing its picture format";
        case H263CU_ERR_PICTURE_FORMAT_INVALID: return "the decoded H.263 bitstream has an invalid picture format";
        case H263CU_ERR_UNCODED_IFRAME_BLOCKS: return "the decoded H.263 bitstream has uncoded iframe blocks";
        case H263CU_ERR_UNHANDLED_IO_ERROR: return "an I/O error occurred: unexpected end of packet";
        case H263CU_ERR_UNIMPLEMENTED_DECODING: return "a feature in the H.263 bitstream being decoded is not yet supported";
        case H263CU_ERR_BAD_ARGUMENT: return "bad argument";
        case H263CU_ERR_CUDA: return "CUDA runtime error";
        case H263CU_ERR_NO_DEVICE: return "no usable CUDA device (this library has no CPU fallback)";
        case H263CU_ERR_CAPACITY: return "stream, macroblock or event capacity exceeded";
        case H263CU_ERR_REFERENCE_WOULD_ABORT: return "input on which the reference decoder aborts";
        case H263CU_ERR_NO_PICTURE: return "no picture has been decoded on this stream yet";
        case H263CU_ERR_OUT_OF_MEMORY: return "out of memory";
        default: return "unknown error";
    }
}

int h263cu_version(void) { return 100; }

}  // extern "C"

// ---- deferred-commit form used by h263cu_decode_step (context.cu): the parsers advance only when the device stage
// has accepted the step, so that decode_next_picture stays a transaction end to end (state.rs:120-137) ----
namespace h263fe {
int parse_step_deferred(h263cu_parser* const* parsers, const uint8_t* const* packets, const size_t* lens,
                        const uint32_t* stream_ids, uint32_t n, int threads, h263cu_pic* pics, h263cu_mb* mbs, uint32_t mb_cap,
                        h263cu_event* events, uint32_t ev_cap, uint32_t* n_pics_out, uint32_t* n_mbs_out, uint32_t* n_units_out,
                        int* per_pic_err, int32_t* pic_of_input, uint32_t max_w, uint32_t max_h, const uint32_t* min_size) {
    try {
        return parse_step_impl(parsers, packets, lens, stream_ids, n, threads, pics, mbs, mb_cap, events, ev_cap, n_pics_out,
                               n_mbs_out, n_units_out, per_pic_err, pic_of_input, false, max_w, max_h, min_size);
    } catch (const std::bad_alloc&) {
        return H263CU_ERR_OUT_OF_MEMORY;
    }
}
void parse_step_finish(h263cu_parser* const* parsers, uint32_t n, bool accept) {
    for (uint32_t i = 0; i < n; i++) {
        h263cu_parser* p = parsers[i];
        if (!p || !p->pending.valid) continue;
        if (accept) {
            p->has_last = p->pending.has_last, p->has_reference = p->pending.has_reference;
            p->last_fmt_kind = p->pending.fmt_kind, p->last_w = p->pending.w, p->last_h = p->pending.h;
            p->ref_w = p->pending.ref_w, p->ref_h = p->pending.ref_h;
        }
        p->pending.valid = false;
    }
}
}  // namespace h263fe

// ---- the host half of a step whose macroblock layer is parsed on the device (H263CU_PARSE_ON_DEVICE, parse_mb.cu):
// the host keeps the stream state and the picture layer, the device gets the bits after each header ----
namespace h263fe {
using h263dev::ParseJob;
using h263dev::ParseResult;

// The device parse's table image (parse_mb.h), copied from the tables the host parser decodes with
int device_parse_tables(uint32_t* out) {
    const Tables& T = tables();
    static const int spec[4][3] = {{T_MCBPC_I, h263dev::PT_MCBPC_I, h263dev::PT_MCBPC_I_BITS},
                                   {T_MCBPC_P, h263dev::PT_MCBPC_P, h263dev::PT_MCBPC_P_BITS},
                                   {T_CBPY, h263dev::PT_CBPY, h263dev::PT_CBPY_BITS},
                                   {T_MVD, h263dev::PT_MVD, h263dev::PT_MVD_BITS}};
    static_assert(sizeof(VlcEntry) == 4, "one word per table entry");
    for (const auto& t : spec) {
        if (T.t[t[0]].max_len != t[2]) return H263CU_ERR_INTERNAL_DECODER_ERROR;
        std::memcpy(out + t[1], T.t[t[0]].lut.data(), ((size_t)1 << t[2]) * sizeof(uint32_t));
    }
    if (T.tcoef_bits != h263dev::PT_TCOEF_BITS) return H263CU_ERR_INTERNAL_DECODER_ERROR;
    std::memcpy(out + h263dev::PT_TCOEF, T.tcoef_fast.data(), ((size_t)1 << h263dev::PT_TCOEF_BITS) * sizeof(uint32_t));
    return 0;
}

// Before the kernel: per input, the checks of parse_step_impl's first phase and parse_picture_impl up to its
// macroblock loop (the header with the parser's previous format, the size checks), in that order and with the same
// errors.  An input that passes becomes job job_of_input[i] (jobs in input order): its packet is copied to
// stage + pkt_off[i] and followed by 12 zero bytes, pics[i] gets its header fields and its parser's pending state the
// stream state after the picture (not valid yet: device_parse_finish decides).  Its records go to the next mb_w * mb_h
// of *n_mbs_out, its events to a region of the host parser's staging bound (lens * 16 / 3 + 16) of *n_units_out.
// errs[i]: the input's error, 0 for a job.
int device_parse_prepare(h263cu_parser* const* parsers, const uint8_t* const* packets, const size_t* lens, const uint32_t* stream_ids,
                         uint32_t n, int threads, uint32_t max_w, uint32_t max_h, const uint32_t* min_size, const uint64_t* pkt_off,
                         uint8_t* stage, h263cu_pic* pics, int* errs, ParseJob* jobs, int32_t* job_of_input, uint32_t* n_jobs_out,
                         uint32_t* n_mbs_out, uint32_t* n_units_out) {
    if (!parsers || !packets || !lens) return H263CU_ERR_BAD_ARGUMENT;
    for (uint32_t i = 0; i < n; i++)
        if (parsers[i]) parsers[i]->pending.valid = false;
    if (n > 65535) return H263CU_ERR_CAPACITY;
    if (threads <= 0) threads = (int)std::max(1u, std::thread::hardware_concurrency());
    threads = (int)std::min<uint32_t>((uint32_t)threads, std::max(1u, n));
    std::atomic<uint32_t> next{0};
    auto work = [&]() {
        for (;;) {
            const uint32_t i = next.fetch_add(1);
            if (i >= n) break;
            h263cu_parser* p = parsers[i];
            int e = 0;
            h263cu_pic hdr;
            if (!p || !packets[i]) e = H263CU_ERR_BAD_ARGUMENT;
            if (!e) e = h263cu_peek_picture(p->options, packets[i], lens[i], &hdr);
            if (!e && hdr.n_mbs == 0) e = H263CU_ERR_PICTURE_FORMAT_INVALID;
            if (!e && ((hdr.width + 15u) / 16u > 255u || (hdr.height + 15u) / 16u > 255u)) e = H263CU_ERR_CAPACITY;
            if (!e && max_w && (hdr.width > max_w || hdr.height > max_h)) e = H263CU_ERR_CAPACITY;
            if (!e && min_size && (hdr.width < min_size[2 * i] || hdr.height < min_size[2 * i + 1])) e = H263CU_ERR_BAD_ARGUMENT;
            Header hd;
            BitReader r(packets[i] ? packets[i] : (const uint8_t*)"", packets[i] ? lens[i] : 0);
            if (!e) e = parse_header(r, p->options, p->has_last, p->last_fmt_kind, p->last_w, p->last_h, &hd);
            if (!e && !hd.dims_valid) e = H263CU_ERR_PICTURE_FORMAT_INVALID;
            const uint32_t W = hd.w, H = hd.h, mb_w = (W + 15) / 16, mb_h = (H + 15) / 16;
            if (!e && mb_w == 0) e = H263CU_ERR_REFERENCE_WOULD_ABORT;
            if (!e && (mb_w > 255 || mb_h > 255)) e = H263CU_ERR_CAPACITY;
            errs[i] = e;
            if (e) continue;
            const bool is_i = hd.pic_type == H263CU_PIC_I;
            const bool decode_disposable = (p->options & H263CU_OPT_DECODE_DISPOSABLE) != 0;
            const bool is_sorenson = (p->options & H263CU_OPT_SORENSON_SPARK_BITSTREAM) != 0;
            const bool disposable = decode_disposable && hd.pic_type == H263CU_PIC_DISPOSABLE_P;
            ParseJob& J = jobs[i];  // compacted below
            std::memset(&J, 0, sizeof(J));
            J.bit_pos = (uint32_t)r.pos();
            J.bits = (uint32_t)(lens[i] * 8);
            J.mb_w = (uint8_t)mb_w, J.mb_h = (uint8_t)mb_h;
            J.quant = hd.quant;
            J.mode = (uint8_t)((is_i ? h263dev::PJ_INTRA : 0) | (is_sorenson ? h263dev::PJ_SORENSON : 0) |
                               ((is_sorenson && hd.version == 1) ? h263dev::PJ_ESC_V1 : 0));
            if ((!is_i && hd.pic_type != H263CU_PIC_P && !disposable) || !hd.type_supported) J.mode |= h263dev::PJ_UNSUPPORTED;
            h263cu_pic& pc = pics[i];
            std::memset(&pc, 0, sizeof(pc));
            pc.stream = stream_ids ? stream_ids[i] : i;
            pc.width = (uint16_t)W, pc.height = (uint16_t)H;
            pc.mb_w = (uint8_t)mb_w, pc.mb_h = (uint8_t)mb_h;
            pc.pic_type = hd.pic_type;
            pc.pquant = hd.quant;
            pc.flags = (uint8_t)((hd.deblock ? H263CU_PICFLAG_DEBLOCK : 0) | (disposable ? H263CU_PICFLAG_DISPOSABLE : 0));
            pc.version = hd.version < 0 ? 0xFF : (uint8_t)hd.version;
            pc.n_mbs = mb_w * mb_h;
            pc.temporal_reference = hd.tr;
            // reference bookkeeping (parse_picture_impl's end)
            auto& pd = p->pending;
            pd.has_last = true;
            pd.has_reference = p->has_reference;
            if (is_i) pd.has_reference = false;
            if (hd.pic_type != H263CU_PIC_DISPOSABLE_P) pd.has_reference = true;
            pd.fmt_kind = hd.fmt_kind;
            pd.w = (uint16_t)W, pd.h = (uint16_t)H;
            pd.ref_w = disposable ? p->ref_w : (uint16_t)W, pd.ref_h = disposable ? p->ref_h : (uint16_t)H;
            uint8_t* dst = stage + pkt_off[i];
            std::memcpy(dst, packets[i], lens[i]);
            std::memset(dst + lens[i], 0, (size_t)(pkt_off[i + 1] - pkt_off[i]) - lens[i]);
        }
    };
    worker_pool().run(threads, work);
    uint32_t nj = 0;
    uint64_t nm = 0, nu = 0;
    for (uint32_t i = 0; i < n; i++) {
        job_of_input[i] = -1;
        if (errs[i]) continue;
        ParseJob J = jobs[i];
        J.pkt_word = (uint32_t)(pkt_off[i] / 4);
        J.first_mb = (uint32_t)nm;
        J.first_event = (uint32_t)nu;
        J.ev_cap = (uint32_t)(lens[i] * 16 / 3 + 16);
        J.pic = (uint16_t)nj;
        nm += pics[i].n_mbs;
        nu += J.ev_cap;
        job_of_input[i] = (int32_t)nj;
        jobs[nj++] = J;
    }
    if (nm > 0xFFFFFFFFull || nu > 0xFFFFFFFFull) return H263CU_ERR_CAPACITY;
    *n_jobs_out = nj;
    *n_mbs_out = (uint32_t)nm;
    *n_units_out = (uint32_t)nu;
    return 0;
}

// After the kernel: each job's outcome -- the device's error, or else parse_picture_impl's closing checks (HAS_INTER
// needs a reference of the picture's size) against the parser's state before the picture.  A picture that passes gets
// its flags and unit count in pics[i], and its parser's pending state becomes valid (parse_step_finish commits it).
void device_parse_finish(h263cu_parser* const* parsers, uint32_t n, const int32_t* job_of_input, const ParseResult* res,
                         h263cu_pic* pics, int* errs) {
    for (uint32_t i = 0; i < n; i++) {
        const int32_t j = job_of_input[i];
        if (j < 0) continue;
        h263cu_parser* p = parsers[i];
        const ParseResult& r = res[j];
        int e = r.err;
        if (!e && (r.flags & H263CU_PICFLAG_HAS_INTER)) {
            if (!(p->has_reference && p->has_last)) {
                e = H263CU_ERR_UNCODED_IFRAME_BLOCKS;
            } else {
                const bool dd = (p->options & H263CU_OPT_DECODE_DISPOSABLE) != 0;
                const uint16_t rw = dd ? p->ref_w : p->last_w, rh = dd ? p->ref_h : p->last_h;
                if (rw != pics[i].width || rh != pics[i].height) e = H263CU_ERR_REFERENCE_WOULD_ABORT;
            }
        }
        errs[i] = e;
        if (e) continue;
        pics[i].flags |= (uint8_t)r.flags;
        pics[i].n_event_units = r.units;
        p->pending.valid = true;
    }
}
}  // namespace h263fe

static_assert(sizeof(h263cu_pic) == 32, "h263cu_pic layout");
static_assert(sizeof(h263cu_mb) == 24, "h263cu_mb layout");
