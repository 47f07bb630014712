// deblock_tile.cu -- deblocking post-filter (deblock/src/deblock.rs:29-42,99-127,136-299) fused
// with the BT.601 conversion (yuv/src/bt601.rs:12-59), register-resident: no shared memory, no
// barrier.  For planes whose sizes are multiples of 8 (luma sizes multiples of 16), where every
// edge sample uses the reference's SIMD arithmetic (arithmetic shifts = floor division); other
// sizes take deblock_rgba_kernel in kernels.cu, which also implements the scalar-tail rounding.
//
// Every output pixel depends only on input pixels of its own 8x8 cell shifted by (4,4)
// ([8k-4, 8k+4) x [8j-4, 8j+4)): the cell holds one horizontal edge (its rows 2..5) and one
// vertical edge (its columns 2..5), horizontal first (deblock.rs:305-315).  A thread owns one
// shifted luma cell and the 4x4 chroma samples under it of both planes, which are a quadrant of
// the chroma region [8M-2, 8M+6) x [8N-2, 8N+6): that region holds exactly one chroma edge per
// direction, whose four filter taps are the first four columns (rows) of the region, so the
// quadrants filter independently: the top two filter the horizontal edge, then the left two the
// vertical edge.  The deblocked planes never go back to the context: the reference frames stay
// un-deblocked (deblock/src/lib.rs:1-2); RGBA leaves the kernel, or in the plane-output form (YUV)
// the deblocked samples themselves go to the caller's planes.
//
// The filter runs on two samples per instruction in 16-bit lanes (VIADD.16x2, VIMNMX.S16x2,
// VIADDMNMX.S16x2.RELU); biased non-negative intermediates make floor division a plain shift.
#include "recon_common.cuh"

namespace h263dev {

namespace {

__device__ __forceinline__ uint32_t add2(uint32_t a, uint32_t b) { return __vadd2(a, b); }  // VIADD.16x2
__device__ __forceinline__ uint32_t neg2(uint32_t a) { return __vadd2(~a, 0x00010001u); }
__device__ __forceinline__ uint32_t max2(uint32_t a, uint32_t b) { return __vmaxs2(a, b); }  // VIMNMX.S16x2
__device__ __forceinline__ uint32_t min2(uint32_t a, uint32_t b) { return __vmins2(a, b); }

// process_simd (deblock.rs:99-127) on two sample quadruples, lanes hold 0..255:
//   d  = (A - 4B + 4C - D) >> 3
//   d1 = sign(d) * max(0, |d| - max(0, 2 (|d| - S)))          = clamp(d, -r, r), r = max(0, min(|d|, 2S - |d|))
//   d2 = clamp((A - D) >> 2, -|d1 >> 1|, |d1 >> 1|)
//   A -= d2 (wrapping u8), B = clamp(B + d1), C = clamp(C - d1), D += d2 (wrapping u8)
// s2 = (2S, 2S).
__device__ __forceinline__ void deblock2(uint32_t& A, uint32_t& B, uint32_t& C, uint32_t& D, uint32_t s2) {
    const uint32_t nB = B ^ 0x00FF00FFu, nD = D ^ 0x00FF00FFu;  // 255 - x
    const uint32_t e5 = A + nD + 0x00050005u;                    // A - D + 260
    const uint32_t s = e5 + 4u * (C + nB);                       // A - 4B + 4C - D + 1280, in [5, 2555]
    const uint32_t d = add2((s >> 3) & 0x1FFF1FFFu, 0xFF60FF60u);  // floor(./8) - 160
    const uint32_t nd = neg2(d);
    const uint32_t ad = max2(d, nd), r = __vimin_s16x2_relu(ad, add2(min2(d, nd), s2));
    const uint32_t nr = neg2(r);
    const uint32_t d1 = min2(max2(d, nr), r), nd1 = min2(max2(nd, nr), r);
    // |d1 >> 1| with floor: (|d1| + (d1 < 0)) >> 1
    const uint32_t lim = ((r + ((d >> 15) & 0x00010001u)) >> 1) & 0x7FFF7FFFu;
    const uint32_t q = add2((e5 >> 2) & 0x3FFF3FFFu, 0xFFBFFFBFu);  // floor((A - D + 260) / 4) - 65 = (A - D) >> 2
    const uint32_t d2 = min2(max2(q, neg2(lim)), lim);
    A = ~add2(~A, d2) & 0x00FF00FFu;
    D = add2(D, d2) & 0x00FF00FFu;
    B = __viaddmin_s16x2_relu(B, d1, 0x00FF00FFu);
    C = __viaddmin_s16x2_relu(C, nd1, 0x00FF00FFu);
}

__device__ __forceinline__ uint32_t pack_sat(int a, int b, uint32_t c) {
    uint32_t d;  // d = c[15:0] << 16 | sat_u8(a) << 8 | sat_u8(b)
    asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
struct CT {
    int r, g, b;
};
__device__ __forceinline__ CT chroma_terms_folded(int cb, int cr) {
    CT t;
    t.r = cr * 104597 + (32768 - 128 * 104597 - 16 * 76309);
    t.g = cr * -53279 + (cb * -25675 + (32768 + 128 * 53279 + 128 * 25675 - 16 * 76309));
    t.b = cb * 132201 + (32768 - 128 * 132201 - 16 * 76309);
    return t;
}
__device__ __forceinline__ uint32_t rgba_px(int y, const CT& t) {
    const int r = (y * 76309 + t.r) >> 16, g = (y * 76309 + t.g) >> 16, b = (y * 76309 + t.b) >> 16;
    return pack_sat(g, r, pack_sat(255, b, 0));
}

constexpr int DB_THREADS = 128;  // 4 warps = the four cells (a, b) of 32 consecutive 16x16 groups

}  // namespace

// grid = (ceil(groups / 32), n_pics); group (M, N) = luma region [16M-4, 16M+12) x [16N-4, 16N+12)
template <bool YUV>
__global__ void __launch_bounds__(DB_THREADS) deblock_rgba_tile_kernel(const PicDev* __restrict__ pics, const YuvDst yuv) {
    const PicDev& P = pics[blockIdx.y];
    const int W = P.w, H = P.h;
    const int GX = (W >> 4) + 1, GY = (H >> 4) + 1;
    const int gid = blockIdx.x * 32 + (threadIdx.x & 31);
    if (gid >= GX * GY) return;
    const int a = (threadIdx.x >> 5) & 1, b = threadIdx.x >> 6;  // warp-uniform
    const int N = gid / GX, M = gid - N * GX;
    const int x0 = 16 * M - 4 + 8 * a, y0 = 16 * N - 4 + 8 * b;
    if (x0 >= W || y0 >= H) return;  // the cell lies beyond the right / bottom border
    const int pitch_y = P.pitch_y, pitch_c = P.pitch_c;
    const uint32_t s2 = 2u * P.strength * 0x00010001u;

    // ---- luma cell: 8 rows x 8 pixels in 16-bit lanes (p0,p2) (p1,p3) (p4,p6) (p5,p7) ----
    uint32_t e0[8], o0[8], e1[8], o1[8];
    {
        const uint8_t* src = P.cur[0] + (ptrdiff_t)y0 * pitch_y + x0;  // 4-byte aligned; the planes carry a border
#pragma unroll
        for (int j = 0; j < 8; j++) {
            const uint32_t w0 = __ldg(reinterpret_cast<const uint32_t*>(src + j * pitch_y));
            const uint32_t w1 = __ldg(reinterpret_cast<const uint32_t*>(src + j * pitch_y + 4));
            e0[j] = __byte_perm(w0, 0, 0x4240), o0[j] = __byte_perm(w0, 0, 0x4341);
            e1[j] = __byte_perm(w1, 0, 0x4240), o1[j] = __byte_perm(w1, 0, 0x4341);
        }
        // horizontal edge at y0 + 4: rows 2..5; edges on the picture border are not filtered (deblock.rs:139-140)
        const int ey = y0 + 4;
        if (ey >= 8 && ey <= H - 2) {
            deblock2(e0[2], e0[3], e0[4], e0[5], s2);
            deblock2(o0[2], o0[3], o0[4], o0[5], s2);
            deblock2(e1[2], e1[3], e1[4], e1[5], s2);
            deblock2(o1[2], o1[3], o1[4], o1[5], s2);
        }
        // vertical edge at x0 + 4: columns 2..5 = (e0.hi, o0.hi, e1.lo, o1.lo), two rows per instruction
        const int ex = x0 + 4;
        if (W >= 10 && ex >= 8 && ex + 2 <= W) {
#pragma unroll
            for (int j = 0; j < 8; j += 2) {
                uint32_t A = __byte_perm(e0[j], e0[j + 1], 0x7632), B = __byte_perm(o0[j], o0[j + 1], 0x7632);
                uint32_t C = __byte_perm(e1[j], e1[j + 1], 0x5410), D = __byte_perm(o1[j], o1[j + 1], 0x5410);
                deblock2(A, B, C, D, s2);
                e0[j] = __byte_perm(e0[j], A, 0x5410), e0[j + 1] = __byte_perm(e0[j + 1], A, 0x7610);
                o0[j] = __byte_perm(o0[j], B, 0x5410), o0[j + 1] = __byte_perm(o0[j + 1], B, 0x7610);
                e1[j] = __byte_perm(e1[j], C, 0x3254), e1[j + 1] = __byte_perm(e1[j + 1], C, 0x3276);
                o1[j] = __byte_perm(o1[j], D, 0x3254), o1[j + 1] = __byte_perm(o1[j + 1], D, 0x3276);
            }
        }
    }

    // ---- chroma quadrant: 4 rows x 4 samples of both planes, lanes (c0,c2) (c1,c3) ----
    uint32_t ce[2][4], co[2][4];
    {
        const int CW = P.cw, CH = P.ch;
        const int cx0 = 8 * M - 2 + 4 * a, cy0 = 8 * N - 2 + 4 * b;  // = x0 / 2, y0 / 2
        const bool do_h = b == 0 && 8 * N >= 8 && 8 * N <= CH - 2;              // chroma edge row 8N: quadrant rows 0..3
        const bool do_v = a == 0 && CW >= 10 && 8 * M >= 8 && 8 * M + 2 <= CW;  // chroma edge column 8M: columns 0..3
        // the planes are interleaved (CbCr pairs): samples cx0..cx0+3 of both planes are the 8 bytes at 2 * cx0,
        // which is a multiple of 4: two aligned words per row serve both planes
        const uint8_t* src = P.cur[1] + (ptrdiff_t)cy0 * pitch_c + (ptrdiff_t)cx0 * CHROMA_STEP;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            const uint32_t w0 = __ldg(reinterpret_cast<const uint32_t*>(src + j * pitch_c));      // cb0 cr0 cb1 cr1
            const uint32_t w1 = __ldg(reinterpret_cast<const uint32_t*>(src + j * pitch_c + 4));  // cb2 cr2 cb3 cr3
            ce[0][j] = __byte_perm(w0, w1, 0x0400) & 0x00FF00FFu, co[0][j] = __byte_perm(w0, w1, 0x0602) & 0x00FF00FFu;
            ce[1][j] = __byte_perm(w0, w1, 0x0501) & 0x00FF00FFu, co[1][j] = __byte_perm(w0, w1, 0x0703) & 0x00FF00FFu;
        }
#pragma unroll
        for (int pl = 0; pl < 2; pl++) {
            if (do_h) {
                deblock2(ce[pl][0], ce[pl][1], ce[pl][2], ce[pl][3], s2);
                deblock2(co[pl][0], co[pl][1], co[pl][2], co[pl][3], s2);
            }
            if (do_v) {
#pragma unroll
                for (int j = 0; j < 4; j += 2) {
                    // columns 0..3 = (ce.lo, co.lo, ce.hi, co.hi)
                    uint32_t A = __byte_perm(ce[pl][j], ce[pl][j + 1], 0x5410), B = __byte_perm(co[pl][j], co[pl][j + 1], 0x5410);
                    uint32_t C = __byte_perm(ce[pl][j], ce[pl][j + 1], 0x7632), D = __byte_perm(co[pl][j], co[pl][j + 1], 0x7632);
                    deblock2(A, B, C, D, s2);
                    ce[pl][j] = __byte_perm(A, C, 0x5410), ce[pl][j + 1] = __byte_perm(A, C, 0x7632);
                    co[pl][j] = __byte_perm(B, D, 0x5410), co[pl][j + 1] = __byte_perm(B, D, 0x7632);
                }
            }
        }
    }

    // ---- BT.601 RGBA of the part of the cell that lies inside the picture ----
    if (!P.rgba) return;
    const bool left_cut = x0 < 0, right_cut = x0 + 8 > W;  // border cells: only 4 of the 8 columns exist
    if constexpr (YUV) {
        // plane output: the cell's luma rows as two words at x0 (4-byte aligned), the quadrant's chroma rows at
        // cx0 = x0 / 2, which the same cuts apply to (a border cell's quadrant holds 2 of its 4 columns)
        const uint32_t slot = P.rgba_row0 >> 12;
#pragma unroll
        for (int j = 0; j < 8; j++) {
            if (y0 + j < 0 || y0 + j >= H) continue;
            uint8_t* o = yuv_row(yuv, 0, slot, (uint32_t)(y0 + j)) + x0;
            if (!left_cut) *reinterpret_cast<uint32_t*>(o) = __byte_perm(e0[j], o0[j], 0x6240);
            if (!right_cut) *reinterpret_cast<uint32_t*>(o + 4) = __byte_perm(e1[j], o1[j], 0x6240);
        }
        const int cx0 = x0 / 2, cy0 = y0 / 2;
#pragma unroll
        for (int j = 0; j < 4; j++) {
            if (cy0 + j < 0 || cy0 + j >= (int)P.ch) continue;
            if (yuv.nv12) {
                // (cb0 cr0 cb2 cr2), (cb1 cr1 cb3 cr3) -> (cb0 cr0 cb1 cr1), (cb2 cr2 cb3 cr3) at 2 * cx0 (4-byte aligned)
                const uint32_t x = __byte_perm(ce[0][j], ce[1][j], 0x6240), y = __byte_perm(co[0][j], co[1][j], 0x6240);
                uint8_t* o = yuv_row(yuv, 1, slot, (uint32_t)(cy0 + j)) + 2 * cx0;
                if (!left_cut) *reinterpret_cast<uint32_t*>(o) = __byte_perm(x, y, 0x5410);
                if (!right_cut) *reinterpret_cast<uint32_t*>(o + 4) = __byte_perm(x, y, 0x7632);
            } else {
                // I420: samples c0..c3 of each plane at cx0 (2-byte aligned): two 16-bit stores per plane
#pragma unroll
                for (int pl = 0; pl < 2; pl++) {
                    const uint32_t v = __byte_perm(ce[pl][j], co[pl][j], 0x6240);
                    uint8_t* o = yuv_row(yuv, 1 + pl, slot, (uint32_t)(cy0 + j)) + cx0;
                    if (!left_cut) *reinterpret_cast<uint16_t*>(o) = (uint16_t)v;
                    if (!right_cut) *reinterpret_cast<uint16_t*>(o + 2) = (uint16_t)(v >> 16);
                }
            }
        }
        return;
    }
    uint8_t* out = P.rgba + (ptrdiff_t)y0 * P.rgba_pitch + (ptrdiff_t)x0 * 4;
#pragma unroll
    for (int cj = 0; cj < 4; cj++) {
        // chroma row cj serves luma rows 2cj, 2cj+1; sample i serves pixels 2i, 2i+1
        const CT t0 = chroma_terms_folded((int)(ce[0][cj] & 0xFFFFu), (int)(ce[1][cj] & 0xFFFFu));
        const CT t1 = chroma_terms_folded((int)(co[0][cj] & 0xFFFFu), (int)(co[1][cj] & 0xFFFFu));
        const CT t2 = chroma_terms_folded((int)(ce[0][cj] >> 16), (int)(ce[1][cj] >> 16));
        const CT t3 = chroma_terms_folded((int)(co[0][cj] >> 16), (int)(co[1][cj] >> 16));
#pragma unroll
        for (int rr = 0; rr < 2; rr++) {
            const int j = 2 * cj + rr;
            if (y0 + j < 0 || y0 + j >= H) continue;
            uint4 lo, hi;
            lo.x = rgba_px((int)(e0[j] & 0xFFFFu), t0), lo.y = rgba_px((int)(o0[j] & 0xFFFFu), t0);
            lo.z = rgba_px((int)(e0[j] >> 16), t1), lo.w = rgba_px((int)(o0[j] >> 16), t1);
            hi.x = rgba_px((int)(e1[j] & 0xFFFFu), t2), hi.y = rgba_px((int)(o1[j] & 0xFFFFu), t2);
            hi.z = rgba_px((int)(e1[j] >> 16), t3), hi.w = rgba_px((int)(o1[j] >> 16), t3);
            uint8_t* o = out + (ptrdiff_t)j * P.rgba_pitch;
            if (!left_cut) *reinterpret_cast<uint4*>(o) = lo;
            if (!right_cut) *reinterpret_cast<uint4*>(o + 16) = hi;
        }
    }
}

void launch_deblock_rgba_tile(const PicDev* pics, uint32_t n_pics, uint32_t max_w, uint32_t max_h, const YuvDst* yuv,
                              cudaStream_t stream) {
    if (n_pics == 0) return;
    const uint32_t groups = ((max_w >> 4) + 1) * ((max_h >> 4) + 1);
    dim3 grid((groups + 31) / 32, n_pics);
    if (yuv)
        deblock_rgba_tile_kernel<true><<<grid, DB_THREADS, 0, stream>>>(pics, *yuv);
    else
        deblock_rgba_tile_kernel<false><<<grid, DB_THREADS, 0, stream>>>(pics, YuvDst{});
}

}  // namespace h263dev
