// resample_filter.cu -- resample_filter_kernel: the decoded planes of a step, resized with torch's antialiased
// bilinear or bicubic filter under a fit and converted into the caller's [slot][channel][row][column] tensor
// (h263cu_decode_step_device_tensor_filter; include/h263cu.h defines the output).
//
// A CTA per 32 x 8 output tile of one picture (grid = (tiles, pictures)), one thread per output pixel.  The filter is
// separable, so the CTA works in the "footprint form":
//  1. the taps of the tile's 32 columns and 8 rows (first sample, count, normalised weights) are computed once into
//     shared memory (aa_span / aa_raw / aa_total / aa_weight of device_math.cuh);
//  2. the tile's source footprint -- the rectangle of samples any of its outputs reads -- is converted once from Y /
//     CbCr to packed RGB in shared memory (chroma_terms / yuv_pixel, as resample_rgb_kernel);
//  3. the horizontal pass runs over the footprint rows of each column into an fp32 shared buffer;
//  4. the vertical pass runs per output pixel and stores the three channels.
// Each source sample is converted once per CTA instead of once per tap of every output that reads it (9-36 per output
// for the CIF -> 224 centre crop), and each tap's weight is computed once per column or row.
//
// The fast path needs the footprint to fit the shared buffers: at most RF_ROWS rows and RF_FOOT samples, and a
// support of at most RF_SUPPORT_MAX on both axes (so at most RF_TAPS taps per output).  A CTA whose footprint is larger
// (downscales beyond about 2.5x; any crop into a 1 x 1 output) takes the general path instead: each thread computes
// the same sums in the same order straight from the planes, recomputing the weights on the fly, so the two paths are
// bit-identical by construction.  The choice is per CTA, from the geometry alone.  Tiles wholly outside the placed
// picture store only the fill.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "device_math.cuh"
#include "kernels.cuh"

namespace h263dev {

namespace {

constexpr int RF_TX = 32, RF_TY = 8;
constexpr int RF_TAPS = 16;               // taps per output on the fast path (supports <= 7 give at most 15)
constexpr float RF_SUPPORT_MAX = 7.0f;
constexpr int RF_ROWS = 32;               // footprint rows on the fast path
constexpr int RF_FOOT = 4096;             // footprint samples on the fast path

// Step 4 with the filters' U8 rule: max(0, min(255, (int)(v + 0.5f))) (bicubic overshoots below 0); floats unclamped
template <uint32_t DT>
__device__ __forceinline__ void store_filtered(void* base, int64_t off, float v, float mul, float add) {
    if constexpr (DT == H263CU_TENSOR_U8) {
        const int q = trunc_to_int(fadd(v, 0.5f));
        static_cast<uint8_t*>(base)[off] = (uint8_t)(q < 0 ? 0 : q < 255 ? q : 255);
    } else {
        const float t = fadd(fmul(v, mul), add);
        if constexpr (DT == H263CU_TENSOR_F32)
            static_cast<float*>(base)[off] = t;
        else if constexpr (DT == H263CU_TENSOR_F16)
            static_cast<__half*>(base)[off] = __float2half_rn(t);
        else
            static_cast<__nv_bfloat16*>(base)[off] = __float2bfloat16_rn(t);
    }
}

__device__ __forceinline__ uint32_t rgb_at(const uint8_t* py, const uint8_t* pc, uint32_t pitch_y, uint32_t pitch_c, int x, int y) {
    const uint32_t luma = __ldg(py + (size_t)y * pitch_y + x);
    const uint32_t cbcr = __ldg(reinterpret_cast<const uint16_t*>(pc + (size_t)(y >> 1) * pitch_c + (size_t)(x >> 1) * CHROMA_STEP));
    return yuv_pixel((int)luma, chroma_terms((int)(cbcr & 0xFFu), (int)(cbcr >> 8)));
}

__device__ __forceinline__ float chan(uint32_t px, int c) { return (float)((px >> (8 * c)) & 0xFFu); }

}  // namespace

template <uint32_t DT, int BICUBIC>
__global__ void __launch_bounds__(RF_TX * RF_TY)
    resample_filter_kernel(const PicDev* __restrict__ pics, const YuvDst src, const TensorDst dst, const FitArgs fit) {
    __shared__ uint32_t s_pix[RF_FOOT];          // packed RGB of the footprint, row-major, fw samples per row
    __shared__ float s_h[3][RF_ROWS][RF_TX];     // horizontal pass: [channel][footprint row][tile column]
    __shared__ float s_wx[RF_TAPS][RF_TX], s_wy[RF_TY][RF_TAPS];
    __shared__ int s_x0[RF_TX], s_nx[RF_TX], s_y0[RF_TY], s_ny[RF_TY];  // first tap (footprint-relative), tap count

    const PicDev& P = pics[blockIdx.y];
    const FitGeom g = fit.geo[blockIdx.y];
    const int W = (int)dst.width, H = (int)dst.height;
    const int tiles_x = (W + RF_TX - 1) / RF_TX;
    const int X0 = (int)(blockIdx.x % tiles_x) * RF_TX, Y0 = (int)(blockIdx.x / tiles_x) * RF_TY;
    const int tx = (int)threadIdx.x, ty = (int)threadIdx.y;
    const int X = X0 + tx, Y = Y0 + ty;
    const int xo = X - g.px, yo = Y - g.py;  // the index into the resized picture
    const bool in_out = X < W && Y < H;
    const bool inside = in_out && (unsigned)xo < (unsigned)g.rw && (unsigned)yo < (unsigned)g.rh;
    const int64_t o = (int64_t)P.out_slot * dst.stride[0] + (int64_t)Y * dst.stride[2] + (int64_t)X * dst.stride[3];
    if (in_out && !inside) {
#pragma unroll
        for (int c = 0; c < 3; c++) store_filtered<DT>(dst.base, o + c * dst.stride[1], fit.fill[c], dst.mul[c], dst.add[c]);
    }
    // the tile's columns xa..xb and rows ya..yb of the resized picture (uniform over the CTA)
    const int xa = max(X0 - g.px, 0), xb = min(min(X0 + RF_TX, W) - g.px, g.rw) - 1;
    const int ya = max(Y0 - g.py, 0), yb = min(min(Y0 + RF_TY, H) - g.py, g.rh) - 1;
    if (xa > xb || ya > yb) return;  // the whole tile is fill

    const uint8_t *py, *pc;
    uint32_t pitch_y, pitch_c;
    if (src.base[0]) {  // deblocked copies: NV12 slot blockIdx.y of the context's scratch planes
        py = yuv_row(src, 0, blockIdx.y, 0), pc = yuv_row(src, 1, blockIdx.y, 0);
        pitch_y = src.pitch[0], pitch_c = src.pitch[1];
    } else {
        py = P.cur[0], pc = P.cur[1];
        pitch_y = P.pitch_y, pitch_c = P.pitch_c;
    }
    const float sx = axis_scale(g.cw, g.rw), sy = axis_scale(g.ch, g.rh);
    const float sup_x = aa_support(sx, BICUBIC ? 2 : 1), sup_y = aa_support(sy, BICUBIC ? 2 : 1);
    const float inv_x = aa_invscale(sx), inv_y = aa_invscale(sy);
    // the footprint: spans are monotone in the output index, so the first and last ones bound it
    const AaSpan fa = aa_span(xa, sx, sup_x, g.cw), fb = aa_span(xb, sx, sup_x, g.cw);
    const AaSpan ga = aa_span(ya, sy, sup_y, g.ch), gb = aa_span(yb, sy, sup_y, g.ch);
    const int fx0 = fa.min, fw = fb.min + fb.size - fx0, fy0 = ga.min, fh = gb.min + gb.size - fy0;

    if (!(sup_x <= RF_SUPPORT_MAX && sup_y <= RF_SUPPORT_MAX && fh <= RF_ROWS && fw * fh <= RF_FOOT)) {
        // general path: the same sums in the same order, straight from the planes
        if (!inside) return;
        const AaSpan spx = aa_span(xo, sx, sup_x, g.cw), spy = aa_span(yo, sy, sup_y, g.ch);
        const float tot_x = aa_total(spx, inv_x, BICUBIC), tot_y = aa_total(spy, inv_y, BICUBIC);
        float v[3] = {0.0f, 0.0f, 0.0f};
        for (int k = 0; k < spy.size; k++) {
            const float wy = aa_weight(aa_raw(spy, k, inv_y, BICUBIC), tot_y);
            const int y = g.cy + spy.min + k;
            float h[3] = {0.0f, 0.0f, 0.0f};
            for (int j = 0; j < spx.size; j++) {
                const float wx = aa_weight(aa_raw(spx, j, inv_x, BICUBIC), tot_x);
                const uint32_t px = rgb_at(py, pc, pitch_y, pitch_c, g.cx + spx.min + j, y);
#pragma unroll
                for (int c = 0; c < 3; c++) h[c] = j == 0 ? fmul(wx, chan(px, c)) : fadd(h[c], fmul(wx, chan(px, c)));
            }
#pragma unroll
            for (int c = 0; c < 3; c++) v[c] = k == 0 ? fmul(wy, h[c]) : fadd(v[c], fmul(wy, h[c]));
        }
#pragma unroll
        for (int c = 0; c < 3; c++) store_filtered<DT>(dst.base, o + c * dst.stride[1], v[c], dst.mul[c], dst.add[c]);
        return;
    }

    // 1. taps: warp 0 the columns, lanes 0..7 of warp 1 the rows
    if (ty == 0 && xo >= xa && xo <= xb) {
        const AaSpan s = aa_span(xo, sx, sup_x, g.cw);
        const float tot = aa_total(s, inv_x, BICUBIC);
        for (int j = 0; j < s.size; j++) s_wx[j][tx] = aa_weight(aa_raw(s, j, inv_x, BICUBIC), tot);
        s_x0[tx] = s.min - fx0, s_nx[tx] = s.size;
    } else if (ty == 1 && tx < RF_TY && Y0 + tx - g.py >= ya && Y0 + tx - g.py <= yb) {
        const AaSpan s = aa_span(Y0 + tx - g.py, sy, sup_y, g.ch);
        const float tot = aa_total(s, inv_y, BICUBIC);
        for (int k = 0; k < s.size; k++) s_wy[tx][k] = aa_weight(aa_raw(s, k, inv_y, BICUBIC), tot);
        s_y0[tx] = s.min - fy0, s_ny[tx] = s.size;
    }
    // 2. the footprint to packed RGB
    const int tid = ty * RF_TX + tx;
    for (int k = tid; k < fw * fh; k += RF_TX * RF_TY) {
        const int r = k / fw, c = k - r * fw;
        s_pix[k] = rgb_at(py, pc, pitch_y, pitch_c, g.cx + fx0 + c, g.cy + fy0 + r);
    }
    __syncthreads();
    // 3. horizontal pass: column tx of footprint rows ty, ty + 8, ...
    const bool col = xo >= xa && xo <= xb;
    if (col) {
        const int x0 = s_x0[tx], nx = s_nx[tx];
        float w[RF_TAPS];
#pragma unroll
        for (int j = 0; j < RF_TAPS; j++) w[j] = j < nx ? s_wx[j][tx] : 0.0f;
        for (int r = ty; r < fh; r += RF_TY) {
            const uint32_t* row = s_pix + r * fw + x0;
            uint32_t px = row[0];
            float h0 = fmul(w[0], chan(px, 0)), h1 = fmul(w[0], chan(px, 1)), h2 = fmul(w[0], chan(px, 2));
#pragma unroll
            for (int j = 1; j < RF_TAPS; j++) {
                if (j >= nx) break;
                px = row[j];
                h0 = fadd(h0, fmul(w[j], chan(px, 0))), h1 = fadd(h1, fmul(w[j], chan(px, 1))), h2 = fadd(h2, fmul(w[j], chan(px, 2)));
            }
            s_h[0][r][tx] = h0, s_h[1][r][tx] = h1, s_h[2][r][tx] = h2;
        }
    }
    __syncthreads();
    // 4. vertical pass per output pixel
    if (!inside) return;
    const int y0 = s_y0[ty], ny = s_ny[ty];
#pragma unroll
    for (int c = 0; c < 3; c++) {
        float v = fmul(s_wy[ty][0], s_h[c][y0][tx]);
        for (int k = 1; k < ny; k++) v = fadd(v, fmul(s_wy[ty][k], s_h[c][y0 + k][tx]));
        store_filtered<DT>(dst.base, o + c * dst.stride[1], v, dst.mul[c], dst.add[c]);
    }
}

template <uint32_t DT>
static void launch_filter_dtype(dim3 grid, dim3 block, const PicDev* pics, const YuvDst& s, const TensorDst& dst, uint32_t filter,
                                const FitArgs& fit, cudaStream_t stream) {
    if (filter == H263CU_FILTER_BICUBIC_AA)
        resample_filter_kernel<DT, 1><<<grid, block, 0, stream>>>(pics, s, dst, fit);
    else
        resample_filter_kernel<DT, 0><<<grid, block, 0, stream>>>(pics, s, dst, fit);
}

void launch_resample_filter(const PicDev* pics, uint32_t n_pics, const YuvDst* src, const TensorDst& dst, uint32_t dtype,
                            uint32_t filter, const FitArgs& fit, cudaStream_t stream) {
    if (n_pics == 0) return;
    const dim3 grid(((dst.width + RF_TX - 1) / RF_TX) * ((dst.height + RF_TY - 1) / RF_TY), n_pics), block(RF_TX, RF_TY);
    const YuvDst s = src ? *src : YuvDst{};
    switch (dtype) {
        case H263CU_TENSOR_U8: launch_filter_dtype<H263CU_TENSOR_U8>(grid, block, pics, s, dst, filter, fit, stream); break;
        case H263CU_TENSOR_F32: launch_filter_dtype<H263CU_TENSOR_F32>(grid, block, pics, s, dst, filter, fit, stream); break;
        case H263CU_TENSOR_F16: launch_filter_dtype<H263CU_TENSOR_F16>(grid, block, pics, s, dst, filter, fit, stream); break;
        default: launch_filter_dtype<H263CU_TENSOR_BF16>(grid, block, pics, s, dst, filter, fit, stream); break;
    }
}

}  // namespace h263dev
