// parse_mb.cu -- the macroblock layer of the host parser (frontend.cpp, parse_picture_impl's macroblock loop) on the
// device, for steps decoded with H263CU_PARSE_ON_DEVICE.  The parse is serial inside a picture, but a step holds
// hundreds of independent pictures: one warp parses one picture, eight warps per CTA share one copy of the VLC tables
// in shared memory.  Lane 0 walks the bitstream; the warp pads the picture's uncoded tail.  The output is the host
// parser's, byte for byte: the same records (zeroed union bytes included), the same event units, the same errors.
#include <cuda_runtime.h>

#include "kernels.cuh"

namespace h263dev {
namespace {

constexpr int PARSE_WARPS = 8;
constexpr int MV_RING = 256;  // > the widest row (255 macroblocks): the left, upper and upper-right neighbours

__device__ __forceinline__ uint32_t bswap32(uint32_t x) { return __byte_perm(x, 0, 0x0123); }

// MSB-first reader over a packet in global memory, 4-byte aligned and followed by at least 12 zero bytes, so that
// the zero-padded look-ahead of the host's BitReader::peek_padded needs no test (pos <= end: the window's three words
// never reach past the padding).  A peek of up to 32 bits reads the first two words; the load of the third runs ahead
// of the consumption.
struct Bits {
    const uint32_t* p;
    uint32_t pos, end;  // bits
    uint32_t k;         // word index of w0
    uint32_t w0, w1, w2;
    __device__ __forceinline__ void seek(uint32_t b) {
        pos = b;
        k = b >> 5;
        w0 = bswap32(__ldg(p + k)), w1 = bswap32(__ldg(p + k + 1));
        w2 = bswap32(__ldg(p + k + 2));
    }
    __device__ __forceinline__ uint32_t avail() const { return end - pos; }
    __device__ __forceinline__ uint32_t peek32() const { return __funnelshift_l(w1, w0, pos & 31); }
    __device__ __forceinline__ void consume(uint32_t n) {  // n <= 32
        pos += n;
        if ((pos >> 5) != k) {
            k++;
            w0 = w1, w1 = w2;
            w2 = bswap32(__ldg(p + k + 2));
        }
    }
    // BitReader::read: n (1..32) bits, false when fewer remain
    __device__ __forceinline__ bool read(uint32_t n, uint32_t* v) {
        if (n > avail()) return false;
        *v = peek32() >> (32 - n);
        consume(n);
        return true;
    }
    // BitReader::read_vlc over a word table indexed by the next `bits` bits (VlcEntry as a little-endian word)
    __device__ __forceinline__ bool read_vlc(const uint32_t* t, uint32_t bits, uint32_t* e) {
        const uint32_t w = t[peek32() >> (32 - bits)];
        if ((w & 31u) > avail()) return false;
        consume(w & 31u);
        *e = w;
        return true;
    }
};
// Any bits of the packet (peek_padded at an arbitrary position): the GOB stub's probe
__device__ __forceinline__ uint32_t peek_at(const uint32_t* p, uint32_t pos) {
    const uint32_t k = pos >> 5;
    return __funnelshift_l(bswap32(__ldg(p + k + 1)), bswap32(__ldg(p + k)), pos & 31);
}

union MbWords {  // a record built in registers and stored as three 8-byte words
    h263cu_mb m;
    uint2 w[3];
};
__device__ __forceinline__ void store_mb(h263cu_mb* dst, const MbWords& r) {
    uint2* d = reinterpret_cast<uint2*>(dst);
    d[0] = r.w[0], d[1] = r.w[1], d[2] = r.w[2];
}

__device__ __forceinline__ uint32_t vlc_kind(uint32_t e) { return (e >> 5) & 7u; }
__device__ __forceinline__ int vlc_a(uint32_t e) { return (int)(int8_t)(e >> 8); }
__device__ __forceinline__ uint32_t vlc_b(uint32_t e) { return (e >> 16) & 0xFFu; }
__device__ __forceinline__ uint32_t vlc_c(uint32_t e) { return e >> 24; }

__device__ __forceinline__ int median3(int a, int b, int c) { return max(min(a, b), min(max(a, b), c)); }
__device__ __forceinline__ int wrap_mv(int pred, int mvd) {
    int out = mvd + pred;
    if (out < -32 || out >= 32) out = (mvd > 0 ? mvd - 64 : (mvd < 0 ? mvd + 64 : 0)) + pred;
    return out;
}

// One block (frontend.cpp parse_block): events staged as (run << 16 | level & 0xFFFF) in `ev`.  Returns 0 or the error.
__device__ __forceinline__ int parse_block(Bits& r, const uint32_t* __restrict__ tf, bool v1, bool intra, bool coded, int* dc,
                                           uint32_t* ev, int* nev, bool* ovf_out, bool* wide) {
    uint32_t v;
    *dc = -1;
    *nev = 0;
    *ovf_out = false;
    if (intra) {
        if (!r.read(8, &v)) return H263CU_ERR_UNHANDLED_IO_ERROR;
        if (v == 0 || v == 128) return H263CU_ERR_INVALID_INTRA_DC;
        *dc = (int)v;
    }
    if (!coded) return 0;
    int idx = intra ? 1 : 0, n = 0;
    bool ovf = false, wd = false;
    for (;;) {
        const uint32_t e = tf[r.peek32() >> (32 - PT_TCOEF_BITS)];
        const uint32_t len = e & 31u, kind = (e >> 5) & 3u;
        if (len > r.avail()) return H263CU_ERR_UNHANDLED_IO_ERROR;  // the code (kind 0: or its sign bit) is cut off
        r.consume(len);
        int last, run, level;
        if (kind == 0) {
            last = (int)((e >> 7) & 1u);
            run = (int)(e >> 26);
            level = ((int)(e << 6)) >> 22;  // the signed 10-bit field at bits 16..25
        } else if (kind == 3) {
            uint32_t width = 8, l, rn;
            if (v1) {
                if (!r.read(1, &v)) return H263CU_ERR_UNHANDLED_IO_ERROR;
                width = v ? 11 : 7;
            }
            if (!r.read(1, &l) || !r.read(6, &rn) || !r.read(width, &v)) return H263CU_ERR_UNHANDLED_IO_ERROR;
            const int lv = ((int)(v << (32 - width))) >> (32 - width);
            if (lv == 0) return H263CU_ERR_INVALID_LONG_COEFFICIENT;
            last = (int)l, run = (int)rn, level = lv;
        } else {
            return H263CU_ERR_INVALID_SHORT_COEFFICIENT;
        }
        idx += run;
        ovf |= idx >= 64;
        if (!ovf) {
            ev[n++] = ((uint32_t)run << 16) | ((uint32_t)level & 0xFFFFu);
            wd |= level < -512 || level > 511;
        }
        idx += 1;
        if (last) break;
    }
    *ovf_out = ovf;
    *nev = ovf ? 0 : n;
    if (!ovf) *wide |= wd;
    return 0;
}

// The macroblock loop of parse_picture_impl for one picture (lane 0).  *n_out: macroblocks decoded (records written
// for the first min(n, capacity)); *quant_out: QUANT after the last one.
__device__ int parse_picture(const ParseJob& J, const uint32_t* __restrict__ words, const uint32_t* __restrict__ T,
                             uint32_t* __restrict__ stage, int8_t (*__restrict__ ring)[4][2], h263cu_mb* __restrict__ mbs,
                             h263cu_event* __restrict__ events, uint32_t* n_out, int* quant_out, uint32_t* units_out, bool* any_inter_out,
                             bool* in_range_out) {
    Bits r;
    r.p = words + J.pkt_word;
    r.end = J.bits;
    r.seek(J.bit_pos);
    const bool is_i = (J.mode & PJ_INTRA) != 0, v1 = (J.mode & PJ_ESC_V1) != 0;
    const uint32_t* TM = T + (is_i ? PT_MCBPC_I : PT_MCBPC_P);
    const uint32_t TM_bits = is_i ? PT_MCBPC_I_BITS : PT_MCBPC_P_BITS;
    const uint32_t* TC = T + PT_CBPY;
    const uint32_t* TV = T + PT_MVD;
    const uint32_t* TF = T + PT_TCOEF;
    const uint32_t mb_w = J.mb_w, capacity = (uint32_t)J.mb_w * J.mb_h;
    const uint32_t R = mb_w + 1;  // ring slot of macroblock n: n % R; n - mb_w sits one slot ahead, n - mb_w + 1 two
    int quant = J.quant;
    uint32_t n = 0, col = 0, row = 0, slot = 0, ev_used = 0;
    bool any_inter = false, mv_in_range = true;
    int err = 0;
    for (;;) {
        const uint32_t mb_start = r.pos;
        uint32_t v, e;
        err = 0;
        bool uncoded = false, stuffing = false;
        int mb_type = 0;
        uint32_t cbp = 0;  // bit b: block b coded
        int dquant = 0;
        int mvd[4][2] = {{0, 0}, {0, 0}, {0, 0}, {0, 0}};
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
            if (J.mode & PJ_UNSUPPORTED) {
                err = H263CU_ERR_UNIMPLEMENTED_DECODING;
                break;
            }
            if (!r.read_vlc(TM, TM_bits, &e)) {
                err = H263CU_ERR_UNHANDLED_IO_ERROR;
                break;
            }
            if (vlc_kind(e) == 1) {
                stuffing = true;
                break;
            }
            if (vlc_kind(e) != 0) {
                err = H263CU_ERR_INVALID_MACROBLOCK_HEADER;
                break;
            }
            mb_type = vlc_a(e);
            cbp = (vlc_b(e) != 0 ? 16u : 0u) | (vlc_c(e) != 0 ? 32u : 0u);
            if (!r.read_vlc(TC, PT_CBPY_BITS, &e)) {
                err = H263CU_ERR_UNHANDLED_IO_ERROR;
                break;
            }
            if (vlc_kind(e) != 0) {
                err = H263CU_ERR_INVALID_MACROBLOCK_CODED_BITS;
                break;
            }
            const bool intra = mb_type == 3 || mb_type == 4;
            const int y = intra ? vlc_a(e) : (~vlc_a(e) & 15);
            cbp |= ((y & 8) ? 1u : 0u) | ((y & 4) ? 2u : 0u) | ((y & 2) ? 4u : 0u) | ((y & 1) ? 8u : 0u);
            if (mb_type == 1 || mb_type == 4 || mb_type == 5) {
                if (!r.read(2, &v)) {
                    err = H263CU_ERR_UNHANDLED_IO_ERROR;
                    break;
                }
                dquant = v == 0 ? -1 : v == 1 ? -2 : v == 2 ? 1 : 2;
            }
            if (!intra) {
                const int nmv = (mb_type == 2 || mb_type == 5) ? 4 : 1;
                for (int k = 0; k < nmv && !err; k++)
                    for (int c = 0; c < 2; c++) {
                        if (!r.read_vlc(TV, PT_MVD_BITS, &e)) {
                            err = H263CU_ERR_UNHANDLED_IO_ERROR;
                            break;
                        }
                        if (vlc_kind(e) != 0) {
                            err = H263CU_ERR_INVALID_MVD;
                            break;
                        }
                        mvd[k][c] = vlc_a(e);
                    }
            }
        } while (0);

        if (err) {
            if (err == H263CU_ERR_UNHANDLED_IO_ERROR) {  // EOF ends the picture
                err = 0;
                break;
            }
            if ((err == H263CU_ERR_INVALID_MACROBLOCK_HEADER || err == H263CU_ERR_INVALID_MACROBLOCK_CODED_BITS) &&
                !(J.mode & PJ_SORENSON)) {
                // GOB resynchronisation stub (frontend.cpp: find_start_code from the macroblock's first bit)
                const uint32_t max_skip = (8u - (mb_start & 7u)) & 7u;
                uint32_t skip = 0, p = mb_start;
                bool found = false, give_up = false;
                for (;;) {
                    if (J.bits - p < 17) {
                        give_up = true;  // EOF ends the picture
                        break;
                    }
                    if ((peek_at(r.p, p) >> 15) == 1u) {
                        found = true;
                        break;
                    }
                    if (skip > max_skip) {
                        give_up = true;  // InvalidGobHeader ends the picture
                        break;
                    }
                    p++, skip++;
                }
                err = 0;
                if (give_up || !found) break;
                if (J.bits - mb_start < 17 + skip + 5) break;  // EOF while reading the GOB number
                const uint32_t gn = peek_at(r.p, mb_start + 17 + skip) >> 27;
                if (gn == 0 || gn == 15) break;  // picture start / EOS: end of this picture
                return H263CU_ERR_UNIMPLEMENTED_DECODING;
            }
            return err;
        }
        if (stuffing) continue;  // consumes no macroblock slot

        if (uncoded) {
            if (is_i) return H263CU_ERR_UNCODED_IFRAME_BLOCKS;  // unreachable: I pictures have no COD
            if (n < capacity) {
                MbWords r;
                r.w[0] = r.w[1] = r.w[2] = make_uint2(0u, 0u);
                r.m.ev_off = ev_used;
                r.m.pic = J.pic;
                r.m.mbx = (uint8_t)col, r.m.mby = (uint8_t)row;
                r.m.flags = H263CU_MB_INTER;
                r.m.quant = (uint8_t)quant;
                store_mb(mbs + n, r);
                *reinterpret_cast<uint2*>(ring[slot]) = make_uint2(0u, 0u);
                any_inter = true;
            }
            n++;
            if (++col == mb_w) col = 0, row++;
            if (++slot == R) slot = 0;
            continue;
        }

        // ---- coded macroblock ----
        quant = min(max(quant + dquant, 1), 31);
        const bool intra = mb_type == 3 || mb_type == 4;
        const bool four = mb_type == 2 || mb_type == 5;
        bool wide = false;
        if (n >= capacity) {
            // one macroblock too many: the first block's errors win, else the reference aborts
            int dc, nev0;
            bool ovf;
            const int be = parse_block(r, TF, v1, intra, (cbp & 1u) != 0, &dc, stage, &nev0, &ovf, &wide);
            return be ? be : H263CU_ERR_REFERENCE_WOULD_ABORT;
        }
        int8_t cur[4][2] = {{0, 0}, {0, 0}, {0, 0}, {0, 0}};
        if (!intra) {
            const uint32_t left = slot == 0 ? R - 1 : slot - 1;
            const uint32_t up = slot + 1 >= R ? slot + 1 - R : slot + 1;
            const uint32_t upr = slot + 2 >= R ? slot + 2 - R : slot + 2;
            for (int k = 0; k < (four ? 4 : 1); k++) {
                int c1x, c1y, c2x, c2y, c3x, c3y;
                if (k == 0 || k == 2) {
                    c1x = col == 0 ? 0 : ring[left][k + 1][0];
                    c1y = col == 0 ? 0 : ring[left][k + 1][1];
                } else {
                    c1x = cur[k - 1][0], c1y = cur[k - 1][1];
                }
                if (k < 2) {
                    if (row == 0) {
                        c2x = c1x, c2y = c1y;
                    } else {
                        c2x = ring[up][k + 2][0], c2y = ring[up][k + 2][1];
                    }
                    if (col == mb_w - 1) {
                        c3x = c3y = 0;
                    } else if (row == 0) {
                        c3x = c1x, c3y = c1y;
                    } else {
                        c3x = ring[upr][2][0], c3y = ring[upr][2][1];
                    }
                } else {
                    c2x = cur[0][0], c2y = cur[0][1];
                    c3x = cur[1][0], c3y = cur[1][1];
                }
                const int px = median3(c1x, c2x, c3x), py = median3(c1y, c2y, c3y);
                cur[k][0] = (int8_t)wrap_mv(px, mvd[k][0]);
                cur[k][1] = (int8_t)wrap_mv(py, mvd[k][1]);
                mv_in_range &= cur[k][0] >= -32 && cur[k][0] <= 31 && cur[k][1] >= -32 && cur[k][1] <= 31;
            }
            if (!four)
                for (int k = 1; k < 4; k++) cur[k][0] = cur[0][0], cur[k][1] = cur[0][1];
            any_inter = true;
        }
        for (int k = 0; k < 4; k++) ring[slot][k][0] = cur[k][0], ring[slot][k][1] = cur[k][1];

        MbWords rec;
        rec.w[0] = rec.w[1] = rec.w[2] = make_uint2(0u, 0u);
        h263cu_mb& m = rec.m;
        m.ev_off = ev_used;
        m.pic = J.pic;
        m.mbx = (uint8_t)col, m.mby = (uint8_t)row;
        m.quant = (uint8_t)quant;
        m.flags = (uint8_t)(H263CU_MB_CODED | (intra ? 0 : H263CU_MB_INTER) | (four ? H263CU_MB_FOURMV : 0));
        uint32_t total = 0;
        for (int b = 0; b < 6; b++) {
            int dc, nev;
            bool ovf;
            const int be = parse_block(r, TF, v1, intra, (cbp >> b) & 1u, &dc, stage + total, &nev, &ovf, &wide);
            if (be) return be;  // block errors, EOF included, fail the whole picture
            if (intra) m.u.intradc[b] = ovf ? 0 : (uint8_t)dc;
            m.nev[b] = (uint8_t)nev;
            total += (uint32_t)nev;
        }
        const uint32_t units = wide ? total * 2 : total;
        if (ev_used + units > J.ev_cap) return H263CU_ERR_CAPACITY;
        h263cu_event* ev = events + ev_used;
        if (wide) {
            m.flags |= H263CU_MB_WIDE;
            for (uint32_t k = 0; k < total; k++) {
                const uint32_t s = stage[k];
                ev[2 * k] = (h263cu_event)(s >> 16);
                ev[2 * k + 1] = (h263cu_event)(s & 0xFFFFu);
            }
        } else {
            for (uint32_t k = 0; k < total; k++) {
                const uint32_t s = stage[k];
                ev[k] = (h263cu_event)(((s >> 16) << 10) | (s & 0x3FFu));
            }
        }
        if (!intra)
            for (int k = 0; k < 4; k++) m.u.mv[k][0] = cur[k][0], m.u.mv[k][1] = cur[k][1];
        store_mb(mbs + n, rec);
        ev_used += units;
        n++;
        if (++col == mb_w) col = 0, row++;
        if (++slot == R) slot = 0;
    }
    *n_out = n;
    *quant_out = quant;
    *units_out = ev_used;
    *any_inter_out = any_inter;
    *in_range_out = mv_in_range;
    return 0;
}

__global__ void __launch_bounds__(PARSE_WARPS * 32, 1) parse_mb_kernel(const ParseJob* __restrict__ jobs, uint32_t n_jobs,
                                                                     const uint32_t* __restrict__ tables, const uint32_t* __restrict__ words,
                                                                     h263cu_mb* __restrict__ mbs, h263cu_event* __restrict__ events,
                                                                     ParseResult* __restrict__ results) {
    extern __shared__ __align__(16) uint32_t smem[];
    uint32_t* T = smem;                                              // PT_WORDS
    uint32_t* stage_all = smem + PT_WORDS;                           // 6 * 64 per warp
    int8_t(*ring_all)[4][2] = reinterpret_cast<int8_t(*)[4][2]>(stage_all + PARSE_WARPS * 384);  // MV_RING per warp
    for (uint32_t i = threadIdx.x; i < PT_WORDS / 4; i += blockDim.x)
        reinterpret_cast<uint4*>(T)[i] = __ldg(reinterpret_cast<const uint4*>(tables) + i);
    __syncthreads();
    const uint32_t warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t j = blockIdx.x * PARSE_WARPS + warp;
    if (j >= n_jobs) return;
    const ParseJob J = jobs[j];
    uint32_t n = 0, units = 0;
    int quant = 0, err = 0;
    bool any_inter = false, in_range = true;
    if (lane == 0)
        err = parse_picture(J, words, T, stage_all + warp * 384, ring_all + warp * MV_RING, mbs + J.first_mb, events + J.first_event, &n,
                            &quant, &units, &any_inter, &in_range);
    err = __shfl_sync(0xFFFFFFFFu, err, 0);
    n = __shfl_sync(0xFFFFFFFFu, n, 0);
    quant = __shfl_sync(0xFFFFFFFFu, quant, 0);
    units = __shfl_sync(0xFFFFFFFFu, units, 0);
    // a picture that ended early is padded with uncoded inter macroblocks
    const uint32_t capacity = (uint32_t)J.mb_w * J.mb_h;
    if (!err && n < capacity) {
        for (uint32_t i = n + lane; i < capacity; i += 32) {
            MbWords r;
            r.w[0] = r.w[1] = r.w[2] = make_uint2(0u, 0u);
            r.m.ev_off = units;
            r.m.pic = J.pic;
            r.m.mbx = (uint8_t)(i % J.mb_w), r.m.mby = (uint8_t)(i / J.mb_w);
            r.m.flags = H263CU_MB_INTER;
            r.m.quant = (uint8_t)quant;
            store_mb(mbs + J.first_mb + i, r);
        }
        any_inter = true;
    }
    if (lane == 0) {
        ParseResult res;
        res.err = err;
        res.units = err ? 0u : units;
        res.flags = err ? 0u : ((any_inter ? H263CU_PICFLAG_HAS_INTER : 0u) | (in_range ? H263CU_PICFLAG_MV_IN_RANGE : 0u));
        res.pad = 0;
        results[j] = res;
    }
}

// The records of the pictures that survived, moved to their packed positions with their packed index
__global__ void pack_mbs_kernel(const h263cu_mb* __restrict__ src, h263cu_mb* __restrict__ dst, const PackMove* __restrict__ moves) {
    const PackMove mv = moves[blockIdx.x];
    for (uint32_t i = threadIdx.x; i < mv.n; i += blockDim.x) {
        h263cu_mb m = src[mv.src_first + i];
        m.pic = (uint16_t)mv.pic;
        dst[mv.dst_first + i] = m;
    }
}

constexpr size_t PARSE_SMEM = (size_t)PT_WORDS * 4 + (size_t)PARSE_WARPS * 384 * 4 + (size_t)PARSE_WARPS * MV_RING * 8;

}  // namespace

cudaError_t launch_parse_mb(const ParseJob* jobs, uint32_t n_jobs, const uint32_t* tables, const uint32_t* words, h263cu_mb* mbs,
                            h263cu_event* events, ParseResult* results, cudaStream_t stream) {
    // per device: the attribute belongs to the current device's module
    const cudaError_t attr = cudaFuncSetAttribute(parse_mb_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)PARSE_SMEM);
    if (attr != cudaSuccess || n_jobs == 0) return attr;
    const uint32_t blocks = (n_jobs + PARSE_WARPS - 1) / PARSE_WARPS;
    parse_mb_kernel<<<blocks, PARSE_WARPS * 32, PARSE_SMEM, stream>>>(jobs, n_jobs, tables, words, mbs, events, results);
    return cudaGetLastError();
}

void launch_pack_mbs(const h263cu_mb* src, h263cu_mb* dst, const PackMove* moves, uint32_t n_moves, cudaStream_t stream) {
    if (n_moves) pack_mbs_kernel<<<n_moves, 256, 0, stream>>>(src, dst, moves);
}

}  // namespace h263dev
