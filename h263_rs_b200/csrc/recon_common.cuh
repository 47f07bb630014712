// recon_common.cuh -- device helpers shared by the generic (kernels.cu) and the tiled
// (recon_tile.cu) reconstruction kernels.
#pragma once
#include "device_math.cuh"
#include "kernels.cuh"

namespace h263dev {

static __constant__ float c_basis[8][8] = H263_BASIS_TABLE;
static __constant__ uint8_t c_dezigzag[64] = H263_DEZIGZAG_LINEAR;

constexpr int WARPS_PER_CTA = 8;
constexpr int COEF_STRIDE = 68;  // floats per coefficient block: 64 + 4 pad (keeps 16 B alignment,
                                 // staggers the blocks over the banks)
constexpr unsigned FULL = 0xFFFFFFFFu;

enum { CLS_ZERO = 0, CLS_DC = 1, CLS_VERT = 3, CLS_FULL = 4 };  // Horiz is computed as Full (bit-identical)

// per-block info bits gathered while scattering events
constexpr uint32_t INFO_ROWS = 0xFFu;   // bit y: a coefficient event landed in row y
constexpr uint32_t INFO_COL = 0x100u;   // some event landed in a column x > 0
constexpr uint32_t INFO_DC = 0x200u;    // intra DC present
constexpr uint32_t INFO_OVF = 0x400u;   // zig-zag overflow: the block stays Zero (rle.rs:125-127)

struct __align__(16) WarpScratch {
    float coef[6 * COEF_STRIDE];  // dequantised coefficients, [block][y*8+x]
    float tbuf[64];               // row-pass output of the block in flight, [y*8+i]
    int16_t res[6][64];           // rounded residuals, [block][row*8+col]
    uint8_t rec[384];             // reconstructed MB: Y 16x16 | Cb 8x8 | Cr 8x8
};

__device__ __forceinline__ uint32_t byte_of(uint32_t w, int k) { return (w >> (8 * k)) & 0xFFu; }

// clamp(pred + r, 0, 255) on four packed pixels
__device__ __forceinline__ uint32_t add_clamp4(uint32_t pred, int r0, int r1, int r2, int r3) {
    uint32_t o0 = (uint32_t)clamp_u8((int)byte_of(pred, 0) + r0);
    uint32_t o1 = (uint32_t)clamp_u8((int)byte_of(pred, 1) + r1);
    uint32_t o2 = (uint32_t)clamp_u8((int)byte_of(pred, 2) + r2);
    uint32_t o3 = (uint32_t)clamp_u8((int)byte_of(pred, 3) + r3);
    return o0 | (o1 << 8) | (o2 << 16) | (o3 << 24);
}

// Prediction for 8 horizontally adjacent pixels at (x0, y0) of a W x H plane, displaced by
// the half-pel vector (mvx, mvy).  Sample coordinates clamp to the plane (read_sample,
// gather.rs:16-31 = unrestricted-MV border extension); one direction interpolates with
// (a+b+1)>>1, both with (a+b+c+d+2)>>2 (gather.rs:34-40, 103-113).
__device__ __forceinline__ void mc_fetch8(const uint8_t* __restrict__ ref, int pitch, int W, int H, int x0, int y0,
                                          int mvx, int mvy, uint32_t& o0, uint32_t& o1) {
    const int dx = mvx >> 1, ix = mvx & 1, dy = mvy >> 1, iy = mvy & 1;  // floor / odd (types.rs:721-729)
    const int sx = x0 + dx, sy = y0 + dy;
    uint32_t a0, a1, b0 = 0, b1 = 0, c0 = 0, c1 = 0, d0 = 0, d1 = 0;
    const bool inside = sx >= 0 && sy >= 0 && sx + 8 + ix <= W && sy + 1 + iy <= H;
    if (inside) {
        const int a = sx & 3;
        const uint32_t* wp = reinterpret_cast<const uint32_t*>(ref + (size_t)sy * pitch + (sx - a));
        const int sh = a * 8;
        uint32_t w0 = __ldg(wp), w1 = __ldg(wp + 1), w2 = __ldg(wp + 2);
        a0 = __funnelshift_r(w0, w1, sh);
        a1 = __funnelshift_r(w1, w2, sh);
        if (ix) {
            b0 = __funnelshift_rc(w0, w1, sh + 8);
            b1 = __funnelshift_rc(w1, w2, sh + 8);
        }
        if (iy) {
            const uint32_t* wq = wp + (pitch >> 2);
            uint32_t v0 = __ldg(wq), v1 = __ldg(wq + 1), v2 = __ldg(wq + 2);
            c0 = __funnelshift_r(v0, v1, sh);
            c1 = __funnelshift_r(v1, v2, sh);
            if (ix) {
                d0 = __funnelshift_rc(v0, v1, sh + 8);
                d1 = __funnelshift_rc(v1, v2, sh + 8);
            }
        }
    } else {
        uint32_t px[2][9];
#pragma unroll
        for (int r = 0; r < 2; r++) {
            const int cy = min(max(sy + r, 0), H - 1);
            const uint8_t* row = ref + (size_t)cy * pitch;
#pragma unroll
            for (int k = 0; k < 9; k++) px[r][k] = row[min(max(sx + k, 0), W - 1)];
        }
        a0 = px[0][0] | (px[0][1] << 8) | (px[0][2] << 16) | (px[0][3] << 24);
        a1 = px[0][4] | (px[0][5] << 8) | (px[0][6] << 16) | (px[0][7] << 24);
        b0 = px[0][1] | (px[0][2] << 8) | (px[0][3] << 16) | (px[0][4] << 24);
        b1 = px[0][5] | (px[0][6] << 8) | (px[0][7] << 16) | (px[0][8] << 24);
        c0 = px[1][0] | (px[1][1] << 8) | (px[1][2] << 16) | (px[1][3] << 24);
        c1 = px[1][4] | (px[1][5] << 8) | (px[1][6] << 16) | (px[1][7] << 24);
        d0 = px[1][1] | (px[1][2] << 8) | (px[1][3] << 16) | (px[1][4] << 24);
        d1 = px[1][5] | (px[1][6] << 8) | (px[1][7] << 16) | (px[1][8] << 24);
    }
    if (ix && iy) {
        o0 = avg4_u8x4(a0, b0, c0, d0);
        o1 = avg4_u8x4(a1, b1, c1, d1);
    } else if (ix) {
        o0 = avg2_u8x4(a0, b0);
        o1 = avg2_u8x4(a1, b1);
    } else if (iy) {
        o0 = avg2_u8x4(a0, c0);
        o1 = avg2_u8x4(a1, c1);
    } else {
        o0 = a0;
        o1 = a1;
    }
}

// One prediction sample of a plane whose samples are `step` bytes apart, through read_sample's clamp
// (gather.rs:16-31) and lerp (gather.rs:34-40, 103-113).
__device__ __forceinline__ uint32_t mc_fetch1(const uint8_t* __restrict__ ref, int pitch, int step, int W, int H, int x, int y,
                                              int mvx, int mvy) {
    const int sx = x + (mvx >> 1), sy = y + (mvy >> 1), ix = mvx & 1, iy = mvy & 1;
    const int x0 = min(max(sx, 0), W - 1), x1 = min(max(sx + 1, 0), W - 1);
    const int y0 = min(max(sy, 0), H - 1), y1 = min(max(sy + 1, 0), H - 1);
    const uint32_t a = ref[(size_t)y0 * pitch + x0 * step];
    if (ix && iy) {
        const uint32_t b = ref[(size_t)y0 * pitch + x1 * step], c = ref[(size_t)y1 * pitch + x0 * step],
                       d = ref[(size_t)y1 * pitch + x1 * step];
        return (a + b + c + d + 2u) >> 2;
    }
    if (ix) return (a + ref[(size_t)y0 * pitch + x1 * step] + 1u) >> 1;
    if (iy) return (a + ref[(size_t)y1 * pitch + x0 * step] + 1u) >> 1;
    return a;
}

__device__ __forceinline__ void load_event(const h263cu_event* __restrict__ ev, uint32_t idx, bool wide, int& run,
                                           int& level) {
    if (wide) {
        run = __ldg(ev + 2 * idx) & 63;
        level = (int16_t)__ldg(ev + 2 * idx + 1);
    } else {
        uint32_t u = __ldg(ev + idx);
        run = (int)(u >> 10);
        level = ((int)(u << 22)) >> 22;  // sign-extend the 10-bit level
    }
}


// Four RGBA pixels at a 16-byte aligned address, of which the first `valid` (> 0) lie inside the picture: one 128-bit
// store, or one 32-bit store per pixel for the last quad of a row whose width is not a multiple of 4.
__device__ __forceinline__ void store_rgba_quad(uint8_t* dst, const uint4& o, int valid) {
    if (valid >= 4) {
        *reinterpret_cast<uint4*>(dst) = o;
    } else {
        uint32_t* d = reinterpret_cast<uint32_t*>(dst);
        d[0] = o.x;
        if (valid > 1) d[1] = o.y;
        if (valid > 2) d[2] = o.z;
    }
}

// Plane output (OUT_YUV): the first `valid` bytes of a little-endian word at a 4-byte aligned address (nothing when
// valid <= 0).  The caller's planes may end inside a word: a row's last bytes leave through 16- and 8-bit stores.
__device__ __forceinline__ void store_word_cut(uint8_t* dst, uint32_t v, int valid) {
    if (valid >= 4) {
        *reinterpret_cast<uint32_t*>(dst) = v;
    } else if (valid >= 2) {
        *reinterpret_cast<uint16_t*>(dst) = (uint16_t)v;
        if (valid > 2) dst[2] = (uint8_t)(v >> 16);
    } else if (valid == 1) {
        dst[0] = (uint8_t)v;
    }
}
// The same for the two low bytes of `v` at a 2-byte aligned address.
__device__ __forceinline__ void store_pair_cut(uint8_t* dst, uint32_t v, int valid) {
    if (valid >= 2)
        *reinterpret_cast<uint16_t*>(dst) = (uint16_t)v;
    else if (valid == 1)
        dst[0] = (uint8_t)v;
}
// Chroma samples cx..cx+3 (cx a multiple of 4) of row cy of both planes, cb / cr one word each, of which the first
// `valid` lie inside the picture: I420 one word per plane, NV12 two words of CbCr pairs.
__device__ __forceinline__ void store_chroma4_cut(const YuvDst& d, uint32_t slot, int cy, int cx, uint32_t cb, uint32_t cr, int valid) {
    if (d.nv12) {
        uint8_t* o = yuv_row(d, 1, slot, (uint32_t)cy) + 2 * cx;
        store_word_cut(o, __byte_perm(cb, cr, 0x5140), 2 * valid);      // cb0 cr0 cb1 cr1
        store_word_cut(o + 4, __byte_perm(cb, cr, 0x7362), 2 * valid - 4);  // cb2 cr2 cb3 cr3
    } else {
        store_word_cut(yuv_row(d, 1, slot, (uint32_t)cy) + cx, cb, valid);
        store_word_cut(yuv_row(d, 2, slot, (uint32_t)cy) + cx, cr, valid);
    }
}

}  // namespace h263dev
