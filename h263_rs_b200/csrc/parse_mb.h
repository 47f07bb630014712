// parse_mb.h -- what the host front end (frontend.cpp) and the device macroblock parse (parse_mb.cu) exchange for a
// step decoded with H263CU_PARSE_ON_DEVICE.  Plain C++: frontend.cpp includes it without the CUDA headers.
#pragma once
#include <stdint.h>

namespace h263dev {

// The VLC tables of the device parse, one image of 32-bit words (VlcEntry as a word for the four header tables, the
// TCOEF code + sign table of the host's event loop), in this order.  Each table is indexed by the next max-length
// bits of the stream; the lengths are the longest code of each table in vlc_codes.inc (plus the sign bit for TCOEF).
enum {
    PT_MCBPC_I_BITS = 9, PT_MCBPC_P_BITS = 13, PT_CBPY_BITS = 6, PT_MVD_BITS = 13, PT_TCOEF_BITS = 13,
    PT_MCBPC_I = 0,
    PT_MCBPC_P = PT_MCBPC_I + (1 << PT_MCBPC_I_BITS),
    PT_CBPY = PT_MCBPC_P + (1 << PT_MCBPC_P_BITS),
    PT_MVD = PT_CBPY + (1 << PT_CBPY_BITS),
    PT_TCOEF = PT_MVD + (1 << PT_MVD_BITS),
    PT_WORDS = PT_TCOEF + (1 << PT_TCOEF_BITS),  // 25152 words, 98.25 KiB
};

// One picture of a device-parse step: the macroblock layer of its packet, from the first bit after the picture
// header (which the host has parsed), into `first_mb` of the step's records and `first_event` of its events.
struct ParseJob {  // 32 bytes
    uint32_t pkt_word;     // the packet's first byte, in 4-byte words from the start of the step's packet buffer
    uint32_t bit_pos;      // first bit after the picture header
    uint32_t bits;         // packet length in bits
    uint32_t first_mb;     // where the picture's mb_w * mb_h records go
    uint32_t first_event;  // where its events go (h263cu_mb.ev_off counts from here) ...
    uint32_t ev_cap;       // ... and how many units it may write (the host parser's staging bound)
    uint16_t pic;          // h263cu_mb.pic of its records
    uint8_t mb_w, mb_h;
    uint8_t quant;         // PQUANT
    uint8_t mode;          // PJ_* below
    uint8_t pad[2];
};
enum {
    PJ_INTRA = 1,        // I picture: no COD bits, MCBPC from the I table
    PJ_UNSUPPORTED = 2,  // a coded macroblock is H263CU_ERR_UNIMPLEMENTED_DECODING (PB, reserved, disposable types)
    PJ_SORENSON = 4,     // no GOB resynchronisation stub after a macroblock header error
    PJ_ESC_V1 = 8,       // Sorenson version 1: 7- or 11-bit escaped levels
};

// What the device returns per picture; the host finishes the picture from it (the reference checks, the pending
// stream state).
struct ParseResult {  // 16 bytes
    int32_t err;     // 0 or the picture's error
    uint32_t units;  // event units written
    uint32_t flags;  // H263CU_PICFLAG_HAS_INTER | H263CU_PICFLAG_MV_IN_RANGE
    uint32_t pad;
};

// Compaction of the records after a picture failed: the n records at src_first move to dst_first as picture `pic`.
struct PackMove {  // 16 bytes
    uint32_t src_first, dst_first, n, pic;
};

}  // namespace h263dev
