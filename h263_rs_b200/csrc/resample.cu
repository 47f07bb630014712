// resample.cu -- resample_rgb_kernel: the decoded planes of a step, bilinearly resized and converted into the caller's
// [slot][channel][row][column] tensor (h263cu_decode_step_device_tensor; include/h263cu.h defines the output).
//
// One thread per output pixel, a CTA per 32 x 8 output tile of one picture (grid = (tiles, pictures): every picture of
// a call has the same output size, so no CTA idles).  Each thread gathers its four source pixels straight from the
// planes (Y byte + CbCr pair, L1 / L2 resident for neighbouring threads), converts them with the reference's integer
// BT.601 (chroma_terms / yuv_pixel), interpolates each channel in fp32 in the stated order and stores the three
// channels: a warp writes 32 consecutive columns of one channel row, whole sectors for a column stride of 1.
//
// The fit form (FIT = true, h263cu_decode_step_device_tensor_fit) does the same per output pixel for the picture's
// crop box resized to (rw, rh) and placed at (px, py) (FitGeom, one record per picture), and stores the fill value
// outside the placed picture.  FIT = false is the stretch of the whole picture, without the extra parameters.
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include <type_traits>

#include "device_math.cuh"
#include "kernels.cuh"

namespace h263dev {

namespace {

constexpr int RS_TX = 32, RS_TY = 8;

template <uint32_t DT>
__device__ __forceinline__ void store_channel(void* base, int64_t off, float v, float mul, float add) {
    if constexpr (DT == H263CU_TENSOR_U8) {
        const int q = trunc_to_int(fadd(v, 0.5f));
        static_cast<uint8_t*>(base)[off] = (uint8_t)(q < 255 ? q : 255);
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

}  // namespace

struct NoFit {};

template <uint32_t DT, bool FIT>
__global__ void __launch_bounds__(RS_TX * RS_TY)
    resample_rgb_kernel(const PicDev* __restrict__ pics, const YuvDst src, const TensorDst dst,
                        const typename std::conditional<FIT, FitArgs, NoFit>::type fit) {
    const PicDev& P = pics[blockIdx.y];
    int cw = P.w, ch = P.h;  // the source rectangle: cw x ch samples from (cx, cy) below
    const int W = (int)dst.width, H = (int)dst.height;
    const int tiles_x = (W + RS_TX - 1) / RS_TX;
    const int X = (int)(blockIdx.x % tiles_x) * RS_TX + (int)threadIdx.x, Y = (int)(blockIdx.x / tiles_x) * RS_TY + (int)threadIdx.y;
    if (X >= W || Y >= H) return;
    int x_out = X, y_out = Y, cx = 0, cy = 0, rw = W, rh = H;  // the index resampled and the size the source is resized to
    if constexpr (FIT) {
        const FitGeom g = fit.geo[blockIdx.y];
        x_out = X - g.px, y_out = Y - g.py;
        if ((unsigned)x_out >= (unsigned)g.rw || (unsigned)y_out >= (unsigned)g.rh) {  // outside the placed picture
            const int64_t o = (int64_t)P.out_slot * dst.stride[0] + (int64_t)Y * dst.stride[2] + (int64_t)X * dst.stride[3];
#pragma unroll
            for (int c = 0; c < 3; c++) store_channel<DT>(dst.base, o + c * dst.stride[1], fit.fill[c], dst.mul[c], dst.add[c]);
            return;
        }
        cx = g.cx, cy = g.cy, cw = g.cw, ch = g.ch, rw = g.rw, rh = g.rh;
    }
    const uint8_t *py, *pc;
    uint32_t pitch_y, pitch_c;
    if (src.base[0]) {  // deblocked copies: NV12 slot blockIdx.y of the context's scratch planes
        py = yuv_row(src, 0, blockIdx.y, 0), pc = yuv_row(src, 1, blockIdx.y, 0);
        pitch_y = src.pitch[0], pitch_c = src.pitch[1];
    } else {
        py = P.cur[0], pc = P.cur[1];
        pitch_y = P.pitch_y, pitch_c = P.pitch_c;
    }
    const AxisTap tx = axis_tap(x_out, axis_scale(cw, rw), cw), ty = axis_tap(y_out, axis_scale(ch, rh), ch);
    uint32_t px[4];  // packed RGBA of P(x0, y0), P(x1, y0), P(x0, y1), P(x1, y1)
#pragma unroll
    for (int k = 0; k < 4; k++) {
        const int x = cx + ((k & 1) ? tx.i1 : tx.i0), y = cy + ((k & 2) ? ty.i1 : ty.i0);
        const uint32_t luma = __ldg(py + (size_t)y * pitch_y + x);
        const uint32_t cbcr = __ldg(reinterpret_cast<const uint16_t*>(pc + (size_t)(y >> 1) * pitch_c + (size_t)(x >> 1) * CHROMA_STEP));
        px[k] = yuv_pixel((int)luma, chroma_terms((int)(cbcr & 0xFFu), (int)(cbcr >> 8)));
    }
    const int64_t o = (int64_t)P.out_slot * dst.stride[0] + (int64_t)Y * dst.stride[2] + (int64_t)X * dst.stride[3];
#pragma unroll
    for (int c = 0; c < 3; c++) {
        const int sh = 8 * c;
        const float v = bilinear(tx, ty, (float)((px[0] >> sh) & 0xFFu), (float)((px[1] >> sh) & 0xFFu),
                                 (float)((px[2] >> sh) & 0xFFu), (float)((px[3] >> sh) & 0xFFu));
        store_channel<DT>(dst.base, o + c * dst.stride[1], v, dst.mul[c], dst.add[c]);
    }
}

template <uint32_t DT>
static void launch_dtype(dim3 grid, dim3 block, const PicDev* pics, const YuvDst& s, const TensorDst& dst, const FitArgs* fit,
                  cudaStream_t stream) {
    if (fit)
        resample_rgb_kernel<DT, true><<<grid, block, 0, stream>>>(pics, s, dst, *fit);
    else
        resample_rgb_kernel<DT, false><<<grid, block, 0, stream>>>(pics, s, dst, NoFit{});
}

void launch_resample_rgb(const PicDev* pics, uint32_t n_pics, const YuvDst* src, const TensorDst& dst, uint32_t dtype,
                         const FitArgs* fit, cudaStream_t stream) {
    if (n_pics == 0) return;
    const dim3 grid(((dst.width + RS_TX - 1) / RS_TX) * ((dst.height + RS_TY - 1) / RS_TY), n_pics), block(RS_TX, RS_TY);
    const YuvDst s = src ? *src : YuvDst{};
    switch (dtype) {
        case H263CU_TENSOR_U8: launch_dtype<H263CU_TENSOR_U8>(grid, block, pics, s, dst, fit, stream); break;
        case H263CU_TENSOR_F32: launch_dtype<H263CU_TENSOR_F32>(grid, block, pics, s, dst, fit, stream); break;
        case H263CU_TENSOR_F16: launch_dtype<H263CU_TENSOR_F16>(grid, block, pics, s, dst, fit, stream); break;
        default: launch_dtype<H263CU_TENSOR_BF16>(grid, block, pics, s, dst, fit, stream); break;
    }
}

}  // namespace h263dev
