// kernels.cu -- hand-written sm_100a kernels of the reconstruction path.
//
//   recon_kernel          one warp per macroblock: inverse RLE + dequantisation + block
//                         classification (rle.rs:82-172), f32 IDCT in the reference's
//                         operation order (idct.rs:52-65, 82-201), full/half-pel motion
//                         compensation with edge clamping (gather.rs:16-126, 140-204),
//                         residual add + clamp, plane stores, fused BT.601 RGBA
//                         (bt601.rs:12-59) with 128-bit stores.
//   deblock_rgba_kernel   deblocking post-filter (deblock.rs:29-42, 99-127, 136-299) on
//                         32x32 tiles with a 2-pixel halo, fused with the RGBA conversion.
//   yuv420_to_rgba_kernel / deblock_plane_kernel   stateless sibling-crate drop-ins.
//   checksum_kernel       position-weighted checksums for full-size parity checks.
//
// Bound: HBM bandwidth / FP32+INT issue rate; no tensor cores (the 8x8 transform must keep
// the reference's summation order, and is not a dense contraction worth them).
// Compile with -fmad=false; the transform additionally uses __fmul_rn/__fadd_rn, which are
// never contracted.
#include "recon_common.cuh"

namespace h263dev {

// ---------------------------------------------------------------------------------------
// recon_mb_kernel (v0): one warp per macroblock, generic (any picture size, any vector,
// clamped sample fetches).  Kept as the fallback for pictures whose size is not a multiple
// of 16 and as an independent second implementation for on-GPU A/B checks of the tiled
// kernel below.
// YUV (OUT_YUV): no RGBA; with emit_rgba the macroblock's planes also go to the caller's planes `yuv`.
// ---------------------------------------------------------------------------------------
template <bool YUV>
__global__ void __launch_bounds__(WARPS_PER_CTA * 32)
    recon_mb_kernel(const PicDev* __restrict__ pics, const h263cu_mb* __restrict__ mbs,
                    const h263cu_event* __restrict__ events, uint32_t n_mbs, int emit_rgba, const YuvDst yuv) {
    __shared__ WarpScratch scratch[WARPS_PER_CTA];
    __shared__ uint8_t s_dezigzag[64];
    if (threadIdx.x < 64) s_dezigzag[threadIdx.x] = c_dezigzag[threadIdx.x];
    __syncthreads();

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t mb_idx = blockIdx.x * WARPS_PER_CTA + warp;
    if (mb_idx >= n_mbs) return;  // warp-uniform
    WarpScratch& S = scratch[warp];

    // ---- macroblock record (24 bytes = 6 words) -------------------------------------------
    const uint32_t* mw = reinterpret_cast<const uint32_t*>(mbs + mb_idx);
    const uint32_t mword = lane < 6 ? __ldg(mw + lane) : 0u;
    const uint32_t w0 = __shfl_sync(FULL, mword, 0), w1 = __shfl_sync(FULL, mword, 1);
    const uint32_t w2 = __shfl_sync(FULL, mword, 2), w3 = __shfl_sync(FULL, mword, 3);
    const uint32_t w4 = __shfl_sync(FULL, mword, 4), w5 = __shfl_sync(FULL, mword, 5);
    const PicDev& P = pics[w1 & 0xFFFFu];
    const int mbx = (w1 >> 16) & 0xFF, mby = w1 >> 24;
    const bool inter = (w2 & H263CU_MB_INTER) != 0;
    const bool wide = (w2 & H263CU_MB_WIDE) != 0;
    const int quant = (w2 >> 8) & 0xFF;
    const uint32_t c1 = (w2 >> 16) & 0xFF, c2 = c1 + (w2 >> 24), c3 = c2 + (w3 & 0xFF), c4 = c3 + ((w3 >> 8) & 0xFF),
                   c5 = c4 + ((w3 >> 16) & 0xFF), total = c5 + (w3 >> 24);
    const h263cu_event* ev = events + P.first_event + w0;

    uint32_t info[6] = {0, 0, 0, 0, 0, 0};
    const bool has_coefs = total > 0 || !inter;
    if (has_coefs) {
        // ---- zero the coefficient blocks, then scatter the dequantised events ----------------
        float4* cz = reinterpret_cast<float4*>(S.coef);
        for (int i = lane; i < 6 * COEF_STRIDE / 4; i += 32) cz[i] = make_float4(0.f, 0.f, 0.f, 0.f);
        __syncwarp();
        const int first_idx = inter ? 0 : 1;  // intra: DC occupies zig-zag index 0 (rle.rs:117-121)
        if (total <= 32) {
            // one event per lane; the zig-zag position is a segmented prefix sum of (run + 1)
            const bool active = (uint32_t)lane < total;
            const uint32_t e = (uint32_t)lane;
            const int b = (e >= c1) + (e >= c2) + (e >= c3) + (e >= c4) + (e >= c5);
            const int seg_start = b == 0 ? 0 : (b == 1 ? c1 : (b == 2 ? c2 : (b == 3 ? c3 : (b == 4 ? c4 : c5))));
            int run = 0, level = 1;
            if (active) load_event(ev, e, wide, run, level);
            int v = active ? run + 1 : 0;
#pragma unroll
            for (int d = 1; d < 32; d <<= 1) {
                int t = __shfl_up_sync(FULL, v, d);
                if (lane - d >= seg_start) v += t;
            }
            const int pos = first_idx + v - 1;
            const bool ok = active && pos < 64;
            const uint32_t ovf_ballot = __ballot_sync(FULL, active && pos >= 64);
            uint32_t bits = 0;
            if (ok) {
                const int lin = s_dezigzag[pos];
                S.coef[b * COEF_STRIDE + lin] = (float)dequant(level, quant);
                bits = (1u << (lin >> 3)) | ((lin & 7) ? INFO_COL : 0u);
            }
            const uint32_t cs[7] = {0, c1, c2, c3, c4, c5, total};
#pragma unroll
            for (int bb = 0; bb < 6; bb++) {
                uint32_t m = __reduce_or_sync(FULL, (ok && b == bb) ? bits : 0u);
                const uint64_t seg = ((1ull << cs[bb + 1]) - 1ull) ^ ((1ull << cs[bb]) - 1ull);
                if (ovf_ballot & (uint32_t)seg) m |= INFO_OVF;
                info[bb] = m;
            }
        } else {
            // rare: more than 32 events in the macroblock -> lanes 0..5 walk one block each
            uint32_t mine = 0;
            if (lane < 6) {
                const uint32_t cs[7] = {0, c1, c2, c3, c4, c5, total};
                int idx = first_idx;
                for (uint32_t k = cs[lane]; k < cs[lane + 1]; k++) {
                    int run, level;
                    load_event(ev, k, wide, run, level);
                    idx += run;
                    if (idx >= 64) {
                        mine |= INFO_OVF;
                        break;
                    }
                    const int lin = s_dezigzag[idx];
                    S.coef[lane * COEF_STRIDE + lin] = (float)dequant(level, quant);
                    mine |= (1u << (lin >> 3)) | ((lin & 7) ? INFO_COL : 0u);
                    idx += 1;
                }
            }
#pragma unroll
            for (int bb = 0; bb < 6; bb++) info[bb] = __shfl_sync(FULL, mine, bb);
        }
        if (!inter) {
            // INTRADC codes: bytes 0..3 of w4, 0..1 of w5; 0 = dropped block
            uint32_t code = 0;
            if (lane < 6) code = lane < 4 ? byte_of(w4, lane) : byte_of(w5, lane - 4);
            uint32_t my_info = __shfl_sync(FULL, 0u, 0);
#pragma unroll
            for (int bb = 0; bb < 6; bb++)
                if (lane == bb) my_info = info[bb];
            const bool dc_ok = lane < 6 && code != 0 && !(my_info & INFO_OVF);
            if (dc_ok) S.coef[lane * COEF_STRIDE] = (float)intradc_level((int)code);
            const uint32_t dc_ballot = __ballot_sync(FULL, dc_ok);
#pragma unroll
            for (int bb = 0; bb < 6; bb++)
                if ((dc_ballot >> bb) & 1u) info[bb] |= INFO_DC;
        }
        __syncwarp();
    }

    // ---- classification (rle.rs:94-171) and block-serial IDCT ---------------------------------
    int cls[6];
    int dcres[6];
#pragma unroll
    for (int bb = 0; bb < 6; bb++) {
        const uint32_t m = info[bb];
        const uint32_t rows_ev = m & INFO_ROWS;
        int c;
        if ((m & INFO_OVF) || !(m & (INFO_ROWS | INFO_DC)))
            c = CLS_ZERO;
        else if (!(rows_ev & 0xFEu) && !(m & INFO_COL))
            c = CLS_DC;
        else if (!(m & INFO_COL))
            c = CLS_VERT;
        else
            c = CLS_FULL;
        cls[bb] = c;
        dcres[bb] = 0;
        if (c == CLS_DC) dcres[bb] = round_residual_dc(S.coef[bb * COEF_STRIDE]);
    }

    {
        const int i = lane & 7, jg = lane >> 3;
        float bi[8], bj0[8], bj1[8];
#pragma unroll
        for (int k = 0; k < 8; k++) {
            bi[k] = c_basis[k][i];
            bj0[k] = c_basis[k][jg];
            bj1[k] = c_basis[k][jg + 4];
        }
#pragma unroll
        for (int bb = 0; bb < 6; bb++) {
            if (cls[bb] != CLS_FULL && cls[bb] != CLS_VERT) continue;  // warp-uniform
            const bool vert = cls[bb] == CLS_VERT;
            const uint32_t rows = (info[bb] & INFO_ROWS) | ((info[bb] & INFO_DC) ? 1u : 0u);
            const int n = __popc(rows);
            const float* cb = S.coef + bb * COEF_STRIDE;
            // row pass: t[y][i] = sum_x c[y][x] * B[x][i], ascending x (idct_1d, idct.rs:52-65);
            // only rows that hold a coefficient (all-zero rows give +0 and add nothing later)
            for (int base = 0; base < n; base += 4) {
                const int ridx = base + jg;
                if (ridx < n) {
                    const int y = __fns(rows, 0, ridx + 1);
                    float t;
                    if (vert) {
                        t = cb[y * 8];  // Vert: idct_1d runs over the first column directly (idct.rs:152-153)
                    } else {
                        const float4 ca = *reinterpret_cast<const float4*>(cb + y * 8);
                        const float4 cc = *reinterpret_cast<const float4*>(cb + y * 8 + 4);
                        t = 0.0f;
                        t = fadd(t, fmul(ca.x, bi[0]));
                        t = fadd(t, fmul(ca.y, bi[1]));
                        t = fadd(t, fmul(ca.z, bi[2]));
                        t = fadd(t, fmul(ca.w, bi[3]));
                        t = fadd(t, fmul(cc.x, bi[4]));
                        t = fadd(t, fmul(cc.y, bi[5]));
                        t = fadd(t, fmul(cc.z, bi[6]));
                        t = fadd(t, fmul(cc.w, bi[7]));
                    }
                    S.tbuf[y * 8 + i] = t;
                }
            }
            __syncwarp();
            // column pass: out[i][j] = sum_y t[y][i] * B[y][j], ascending y; pixel (x=i, y=j)
            float a0 = 0.0f, a1 = 0.0f;
#pragma unroll
            for (int y = 0; y < 8; y++) {
                if ((rows >> y) & 1u) {
                    const float tv = S.tbuf[y * 8 + i];
                    a0 = fadd(a0, fmul(tv, bj0[y]));
                    a1 = fadd(a1, fmul(tv, bj1[y]));
                }
            }
            const int r0 = vert ? round_residual_scaled(a0) : round_residual(a0);
            const int r1 = vert ? round_residual_scaled(a1) : round_residual(a1);
            S.res[bb][jg * 8 + i] = (int16_t)r0;
            S.res[bb][(jg + 4) * 8 + i] = (int16_t)r1;
            __syncwarp();
        }
    }

    // ---- motion compensation + residual add + clamp -> planes ---------------------------------
    const int mv0x = (int8_t)byte_of(w4, 0), mv0y = (int8_t)byte_of(w4, 1);
    const int mv1x = (int8_t)byte_of(w4, 2), mv1y = (int8_t)byte_of(w4, 3);
    const int mv2x = (int8_t)byte_of(w5, 0), mv2y = (int8_t)byte_of(w5, 1);
    const int mv3x = (int8_t)byte_of(w5, 2), mv3y = (int8_t)byte_of(w5, 3);
    {
        // luma: lane -> pixel row (lane >> 1), 8-pixel half (lane & 1)
        const int rowpix = lane >> 1, half = lane & 1;
        const int b = ((rowpix >> 3) << 1) | half, j = rowpix & 7;
        const int c = half ? (rowpix >= 8 ? cls[3] : cls[1]) : (rowpix >= 8 ? cls[2] : cls[0]);
        const int dcv = half ? (rowpix >= 8 ? dcres[3] : dcres[1]) : (rowpix >= 8 ? dcres[2] : dcres[0]);
        uint32_t p0 = 0, p1 = 0;
        if (inter && P.ref[0]) {
            const int mvx = half ? (rowpix >= 8 ? mv3x : mv1x) : (rowpix >= 8 ? mv2x : mv0x);
            const int mvy = half ? (rowpix >= 8 ? mv3y : mv1y) : (rowpix >= 8 ? mv2y : mv0y);
            mc_fetch8(P.ref[0], P.pitch_y, P.w, P.h, mbx * 16 + half * 8, mby * 16 + rowpix, mvx, mvy, p0, p1);
        }
        if (c == CLS_DC) {
            p0 = add_clamp4(p0, dcv, dcv, dcv, dcv);
            p1 = add_clamp4(p1, dcv, dcv, dcv, dcv);
        } else if (c != CLS_ZERO) {
            const int4 rv = *reinterpret_cast<const int4*>(&S.res[b][j * 8]);
            p0 = add_clamp4(p0, (int16_t)(rv.x & 0xFFFF), rv.x >> 16, (int16_t)(rv.y & 0xFFFF), rv.y >> 16);
            p1 = add_clamp4(p1, (int16_t)(rv.z & 0xFFFF), rv.z >> 16, (int16_t)(rv.w & 0xFFFF), rv.w >> 16);
        }
        *reinterpret_cast<uint2*>(P.cur[0] + (size_t)(mby * 16 + rowpix) * P.pitch_y + mbx * 16 + half * 8) =
            make_uint2(p0, p1);
        *reinterpret_cast<uint2*>(&S.rec[rowpix * 16 + half * 8]) = make_uint2(p0, p1);
    }
    if (lane < 16) {
        // chroma: lane -> plane (lane >> 3), row (lane & 7); both planes share one vector.  The planes are
        // interleaved (CbCr pairs): samples of one plane are CHROMA_STEP bytes apart.
        const int plane = lane >> 3, j = lane & 7, b = 4 + plane;
        const int c = plane ? cls[5] : cls[4];
        const int dcv = plane ? dcres[5] : dcres[4];
        uint32_t px[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        if (inter && P.ref[1 + plane]) {
            const int cx = average_sum_of_mvs(mv0x + mv1x + mv2x + mv3x);
            const int cy = average_sum_of_mvs(mv0y + mv1y + mv2y + mv3y);
#pragma unroll
            for (int k = 0; k < 8; k++) px[k] = mc_fetch1(P.ref[1 + plane], P.pitch_c, CHROMA_STEP, P.cw, P.ch, mbx * 8 + k, mby * 8 + j, cx, cy);
        }
        uint32_t p0 = px[0] | (px[1] << 8) | (px[2] << 16) | (px[3] << 24), p1 = px[4] | (px[5] << 8) | (px[6] << 16) | (px[7] << 24);
        if (c == CLS_DC) {
            p0 = add_clamp4(p0, dcv, dcv, dcv, dcv);
            p1 = add_clamp4(p1, dcv, dcv, dcv, dcv);
        } else if (c != CLS_ZERO) {
            const int4 rv = *reinterpret_cast<const int4*>(&S.res[b][j * 8]);
            p0 = add_clamp4(p0, (int16_t)(rv.x & 0xFFFF), rv.x >> 16, (int16_t)(rv.y & 0xFFFF), rv.y >> 16);
            p1 = add_clamp4(p1, (int16_t)(rv.z & 0xFFFF), rv.z >> 16, (int16_t)(rv.w & 0xFFFF), rv.w >> 16);
        }
        uint8_t* dst = P.cur[1 + plane] + (size_t)(mby * 8 + j) * P.pitch_c + (size_t)(mbx * 8) * CHROMA_STEP;
#pragma unroll
        for (int k = 0; k < 4; k++) dst[k * CHROMA_STEP] = (uint8_t)byte_of(p0, k), dst[(k + 4) * CHROMA_STEP] = (uint8_t)byte_of(p1, k);
        *reinterpret_cast<uint2*>(&S.rec[256 + plane * 64 + j * 8]) = make_uint2(p0, p1);
    }

    // ---- plane output (OUT_YUV) from the staged macroblock, cut to the picture ------------------
    if (YUV && emit_rgba && P.rgba) {
        __syncwarp();
        const uint32_t slot = P.rgba_row0 >> 12;
        // luma: 16 rows x 4 words
#pragma unroll
        for (int g = lane; g < 64; g += 32) {
            const int row = g >> 2, xq = g & 3;
            const int px = mbx * 16 + xq * 4, py = mby * 16 + row;
            if (py >= P.h) continue;
            store_word_cut(yuv_row(yuv, 0, slot, (uint32_t)py) + px, *reinterpret_cast<const uint32_t*>(&S.rec[row * 16 + xq * 4]),
                           P.w - px);
        }
        // chroma: 8 rows x 2 words of 4 samples per plane
        if (lane < 16) {
            const int row = lane >> 1, half = lane & 1;
            const int cx = mbx * 8 + half * 4, cy = mby * 8 + row, valid = P.cw - cx;
            if (cy < P.ch)
                store_chroma4_cut(yuv, slot, cy, cx, *reinterpret_cast<const uint32_t*>(&S.rec[256 + row * 8 + half * 4]),
                                  *reinterpret_cast<const uint32_t*>(&S.rec[320 + row * 8 + half * 4]), valid);
        }
    }

    // ---- fused BT.601 YUV420 -> RGBA (bt601.rs:12-59), one 128-bit store per 4 pixels ---------
    // Only the picture's own pixels are stored (rows < h, the last quad cut at w): RGBA may go to a caller-owned
    // buffer whose slot is exactly the picture's size.
    if (!YUV && emit_rgba && P.rgba) {
        __syncwarp();
#pragma unroll
        for (int g = lane; g < 64; g += 32) {
            const int row = g >> 2, xq = g & 3;
            const int px = mbx * 16 + xq * 4, py = mby * 16 + row;
            if (px >= P.w || py >= P.h) continue;
            const uint32_t yw = *reinterpret_cast<const uint32_t*>(&S.rec[row * 16 + xq * 4]);
            const uint32_t cbp = *reinterpret_cast<const uint16_t*>(&S.rec[256 + (row >> 1) * 8 + xq * 2]);
            const uint32_t crp = *reinterpret_cast<const uint16_t*>(&S.rec[320 + (row >> 1) * 8 + xq * 2]);
            const ChromaTerms t0 = chroma_terms((int)(cbp & 0xFF), (int)(crp & 0xFF));
            const ChromaTerms t1 = chroma_terms((int)(cbp >> 8), (int)(crp >> 8));
            uint4 o;
            o.x = yuv_pixel((int)byte_of(yw, 0), t0);
            o.y = yuv_pixel((int)byte_of(yw, 1), t0);
            o.z = yuv_pixel((int)byte_of(yw, 2), t1);
            o.w = yuv_pixel((int)byte_of(yw, 3), t1);
            store_rgba_quad(P.rgba + (size_t)py * P.rgba_pitch + (size_t)px * 4, o, P.w - px);
        }
    }
}

void launch_recon(const PicDev* pics, const h263cu_mb* mbs, const h263cu_event* events, uint32_t n_mbs, int emit_rgba,
                  int tiled, int wide_mv, const Pools& pools, const CUtensorMap* rgba_map, int out, const YuvDst* yuv,
                  cudaStream_t stream) {
    if (n_mbs == 0) return;
    if (tiled) {
        launch_recon_tile(pics, mbs, events, n_mbs, emit_rgba, tiled == 2, wide_mv, pools, rgba_map, out, yuv, stream);
    } else {
        const uint32_t grid = (n_mbs + WARPS_PER_CTA - 1) / WARPS_PER_CTA;
        YuvDst yd{};
        if (yuv) yd = *yuv;
        if (out == OUT_YUV)
            recon_mb_kernel<true><<<grid, WARPS_PER_CTA * 32, 0, stream>>>(pics, mbs, events, n_mbs, emit_rgba, yd);
        else
            recon_mb_kernel<false><<<grid, WARPS_PER_CTA * 32, 0, stream>>>(pics, mbs, events, n_mbs, emit_rgba, yd);
    }
}

// =======================================================================================
// Deblocking post-filter on a tile held in shared memory.
//   region = (TW + 4) x (TH + 4) pixels starting at plane position (ox - 2, oy - 2), stored
//   with row stride RS at column offset CO (so that the tile interior is 4-byte aligned).
//   Every output pixel depends only on input pixels at most 2 rows / columns away across an
//   8-aligned edge, so tiles whose origin is a multiple of 8 are independent given the halo.
//   Horizontal edges first over the whole plane, then vertical edges (deblock.rs:305-315).
// =======================================================================================
template <int TW, int TH, int RS, int CO>
__device__ __forceinline__ void deblock_tile(uint8_t* sm, const uint8_t* __restrict__ src, int pitch, int step, int W, int H,
                                             int ox, int oy, int strength, int tid, int nthreads) {
    constexpr int RW = TW + 4, RH = TH + 4;
    for (int idx = tid; idx < RW * RH; idx += nthreads) {
        const int rx = idx % RW, ry = idx / RW;
        const int gx = min(max(ox - 2 + rx, 0), W - 1), gy = min(max(oy - 2 + ry, 0), H - 1);
        sm[ry * RS + CO + rx] = src[(size_t)gy * pitch + (size_t)gx * step];
    }
    __syncthreads();
    // horizontal edges: rows ey-2 .. ey+1 for ey = 8, 16, ... <= H - 2 (deblock.rs:136-181);
    // columns below 8*floor(W/8) use the SIMD (floor) arithmetic, the rest the scalar one.
    constexpr int NEH = TH / 8 + 1;
    const int simd_cols = (W >> 3) << 3;
    for (int item = tid; item < NEH * RW; item += nthreads) {
        const int e = item / RW, rx = item % RW;
        const int ey = oy + 8 * e, gx = ox - 2 + rx;
        if (ey < 8 || ey > H - 2 || gx < 0 || gx >= W) continue;
        uint8_t* p = sm + (8 * e) * RS + CO + rx;  // region row of sample A = 8e + 2 - 2
        int A = p[0], B = p[RS], C = p[2 * RS], D = p[3 * RS];
        deblock_process(A, B, C, D, strength, gx >= simd_cols);
        p[0] = (uint8_t)A, p[RS] = (uint8_t)B, p[2 * RS] = (uint8_t)C, p[3 * RS] = (uint8_t)D;
    }
    __syncthreads();
    // vertical edges: columns ex-2 .. ex+1 for ex = 8, 16, ... with ex + 2 <= W, only when
    // W >= 10 (deblock.rs:185-299); rows below 8*floor(H/8) use the SIMD arithmetic.
    constexpr int NEV = TW / 8 + 1;
    const int simd_rows = (H >> 3) << 3;
    for (int item = tid; item < NEV * TH; item += nthreads) {
        const int e = item / TH, ty = item % TH;
        const int ex = ox + 8 * e, gy = oy + ty;
        if (W < 10 || ex < 8 || ex + 2 > W || gy >= H) continue;
        uint8_t* p = sm + (ty + 2) * RS + CO + 8 * e;  // region column of sample A = 8e + 2 - 2
        int A = p[0], B = p[1], C = p[2], D = p[3];
        deblock_process(A, B, C, D, strength, gy >= simd_rows);
        p[0] = (uint8_t)A, p[1] = (uint8_t)B, p[2] = (uint8_t)C, p[3] = (uint8_t)D;
    }
    __syncthreads();
}

// Fused deblock (Y, Cb, Cr) + RGBA for one 32x32 luma tile of one picture; YUV: the deblocked planes go to the
// caller's planes `yuv` instead of RGBA (OUT_YUV).
template <bool YUV>
__global__ void __launch_bounds__(256) deblock_rgba_kernel(const PicDev* __restrict__ pics, const YuvDst yuv) {
    __shared__ __align__(16) uint8_t sy[36 * 40];
    __shared__ __align__(16) uint8_t scb[20 * 24];
    __shared__ __align__(16) uint8_t scr[20 * 24];
    const PicDev& P = pics[blockIdx.y];
    const int W = P.w, H = P.h;
    const int tiles_x = (W + 31) >> 5, tiles_y = (H + 31) >> 5;
    if ((int)blockIdx.x >= tiles_x * tiles_y) return;
    const int tx = blockIdx.x % tiles_x, ty = blockIdx.x / tiles_x;
    const int tid = threadIdx.x;
    const int strength = P.strength;
    deblock_tile<32, 32, 40, 2>(sy, P.cur[0], P.pitch_y, 1, W, H, tx * 32, ty * 32, strength, tid, 256);
    deblock_tile<16, 16, 24, 2>(scb, P.cur[1], P.pitch_c, CHROMA_STEP, P.cw, P.ch, tx * 16, ty * 16, strength, tid, 256);
    deblock_tile<16, 16, 24, 2>(scr, P.cur[2], P.pitch_c, CHROMA_STEP, P.cw, P.ch, tx * 16, ty * 16, strength, tid, 256);
    if (!P.rgba) return;
    const int row = tid >> 3, xq = tid & 7;
    const int gx = tx * 32 + xq * 4, gy = ty * 32 + row;
    if constexpr (YUV) {
        // luma: one word of 4 samples per thread; chroma: threads 0..63 take 4 samples of both planes
        const uint32_t slot = P.rgba_row0 >> 12;
        if (gx < W && gy < H)
            store_word_cut(yuv_row(yuv, 0, slot, (uint32_t)gy) + gx, *reinterpret_cast<const uint32_t*>(&sy[(row + 2) * 40 + 4 + xq * 4]),
                           W - gx);
        if (tid < 64) {
            const int crow = tid >> 2, k = tid & 3;
            const int cx = tx * 16 + k * 4, cy = ty * 16 + crow, valid = P.cw - cx;
            if (cy < P.ch)
                store_chroma4_cut(yuv, slot, cy, cx, *reinterpret_cast<const uint32_t*>(&scb[(crow + 2) * 24 + 4 + k * 4]),
                                  *reinterpret_cast<const uint32_t*>(&scr[(crow + 2) * 24 + 4 + k * 4]), valid);
        }
        return;
    }
    if (gx >= W || gy >= H) return;
    const uint32_t yw = *reinterpret_cast<const uint32_t*>(&sy[(row + 2) * 40 + 4 + xq * 4]);
    const uint32_t cbp = *reinterpret_cast<const uint16_t*>(&scb[((row >> 1) + 2) * 24 + 4 + xq * 2]);
    const uint32_t crp = *reinterpret_cast<const uint16_t*>(&scr[((row >> 1) + 2) * 24 + 4 + xq * 2]);
    const ChromaTerms t0 = chroma_terms((int)(cbp & 0xFF), (int)(crp & 0xFF));
    const ChromaTerms t1 = chroma_terms((int)(cbp >> 8), (int)(crp >> 8));
    uint4 o;
    o.x = yuv_pixel((int)byte_of(yw, 0), t0);
    o.y = yuv_pixel((int)byte_of(yw, 1), t0);
    o.z = yuv_pixel((int)byte_of(yw, 2), t1);
    o.w = yuv_pixel((int)byte_of(yw, 3), t1);
    store_rgba_quad(P.rgba + (size_t)gy * P.rgba_pitch + (size_t)gx * 4, o, W - gx);
}

void launch_deblock_rgba(const PicDev* pics, uint32_t n_pics, uint32_t max_w, uint32_t max_h, const YuvDst* yuv,
                         cudaStream_t stream) {
    if (n_pics == 0) return;
    dim3 grid(((max_w + 31) / 32) * ((max_h + 31) / 32), n_pics);
    if (yuv)
        deblock_rgba_kernel<true><<<grid, 256, 0, stream>>>(pics, *yuv);
    else
        deblock_rgba_kernel<false><<<grid, 256, 0, stream>>>(pics, YuvDst{});
}

// ---- stateless drop-ins ---------------------------------------------------------------
// yuv420_to_rgba (bt601.rs:105-196) on tight planes of any size: pixel (x, y) uses the
// chroma sample (x >> 1, y >> 1) of a ceil(w/2)-wide chroma plane (bt601.rs:115,133,182).
__global__ void __launch_bounds__(256)
    yuv420_to_rgba_kernel(const uint8_t* __restrict__ y, const uint8_t* __restrict__ cb, const uint8_t* __restrict__ cr,
                          uint32_t w, uint32_t h, uint32_t* __restrict__ rgba) {
    const uint32_t cw = (w + 1) >> 1;
    const size_t n = (size_t)w * h;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const uint32_t px = (uint32_t)(i % w), py = (uint32_t)(i / w);
        const size_t ci = (size_t)(py >> 1) * cw + (px >> 1);
        rgba[i] = yuv_pixel(y[i], chroma_terms(cb[ci], cr[ci]));
    }
}

void launch_yuv420_to_rgba(const uint8_t* y, const uint8_t* cb, const uint8_t* cr, uint32_t w, uint32_t h, uint8_t* rgba,
                           cudaStream_t stream) {
    const size_t n = (size_t)w * h;
    if (n == 0) return;
    const uint32_t grid = (uint32_t)((n + 255) / 256 > 148 * 16 ? 148 * 16 : (n + 255) / 256);
    yuv420_to_rgba_kernel<<<grid, 256, 0, stream>>>(y, cb, cr, w, h, reinterpret_cast<uint32_t*>(rgba));
}

__global__ void __launch_bounds__(256)
    deblock_plane_kernel(const uint8_t* __restrict__ in, uint8_t* __restrict__ out, int W, int H, int strength) {
    __shared__ __align__(16) uint8_t sm[36 * 40];
    const int tiles_x = (W + 31) >> 5;
    const int tx = blockIdx.x % tiles_x, ty = blockIdx.x / tiles_x;
    deblock_tile<32, 32, 40, 2>(sm, in, W, 1, W, H, tx * 32, ty * 32, strength, threadIdx.x, 256);
    for (int idx = threadIdx.x; idx < 32 * 32; idx += 256) {
        const int rx = idx & 31, ry = idx >> 5;
        const int gx = tx * 32 + rx, gy = ty * 32 + ry;
        if (gx < W && gy < H) out[(size_t)gy * W + gx] = sm[(ry + 2) * 40 + 4 + rx];
    }
}

void launch_deblock_plane(const uint8_t* in, uint8_t* out, uint32_t w, uint32_t h, int strength, cudaStream_t stream) {
    if (w == 0 || h == 0) return;
    const uint32_t grid = ((w + 31) / 32) * ((h + 31) / 32);
    deblock_plane_kernel<<<grid, 256, 0, stream>>>(in, out, (int)w, (int)h, strength);
}

// ---- checksums --------------------------------------------------------------------------
__global__ void __launch_bounds__(256) checksum_kernel(const ChecksumJob* __restrict__ jobs, unsigned long long* out) {
    const ChecksumJob J = jobs[blockIdx.y];
    const uint64_t n = (uint64_t)J.row_bytes * J.rows;
    unsigned long long s = 0;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint32_t x = (uint32_t)(i % J.row_bytes), yy = (uint32_t)(i / J.row_bytes);
        const uint32_t v = J.base[(size_t)yy * J.pitch + (size_t)x * J.step];
        s += (unsigned long long)(v + 1u) * (unsigned long long)(((uint32_t)i * 2654435761u) | 1u);
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) s += __shfl_down_sync(FULL, s, d);
    __shared__ unsigned long long ws[8];
    if ((threadIdx.x & 31) == 0) ws[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long t = 0;
        for (int k = 0; k < 8; k++) t += ws[k];
        atomicAdd(out + J.out_index, t);
    }
}

void launch_checksums(const ChecksumJob* jobs, uint32_t n_jobs, unsigned long long* out, cudaStream_t stream) {
    if (n_jobs == 0) return;
    dim3 grid(8, n_jobs);
    checksum_kernel<<<grid, 256, 0, stream>>>(jobs, out);
}

}  // namespace h263dev
