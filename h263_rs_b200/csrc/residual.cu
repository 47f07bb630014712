// residual.cu -- the prediction residuals of h263cu_decode_step_device_residual (include/h263cu.h): each picture's
// decoded planes minus the motion-compensated prediction the reference's gather builds (gather.rs:140-204), 0 where
// gather writes nothing (intra macroblocks, I pictures).  The kernel reads the step's planes, the stream's reference
// planes and the step's h263cu_mb records, all still in device memory after the step's other kernels, and writes
// through the caller's strides.
#include "kernels.cuh"

namespace h263dev {

// Two macroblock cells of a slot per CTA, three warps per cell: luma rows 0-7, luma rows 8-15, both chroma planes.
constexpr int RES_CELLS = 2, RES_THREADS = 96 * RES_CELLS;

__device__ __forceinline__ int clamp_to(int v, int hi) { return min(max(v, 0), hi); }

// types.rs:759-768, on the int16 sum of the four luma vectors' components
__device__ __forceinline__ int average_sum_of_mvs(int s) {
    const int whole = (s >> 4) * 2, frac = s & 15;
    return frac <= 2 ? whole : frac >= 14 ? whole + 2 : whole + 1;
}

// gather_block (gather.rs:47-126) for N consecutive samples of one row, from (x, y) on: the reference plane `ref`
// (samples STEP bytes apart, rows `pitch` bytes apart; with STEP 2 a CbCr pair is read as one 16-bit word and both
// planes come out, Cb in bits 0-7 and Cr in bits 8-15 of every element of `out`).  Every read is clamped to the
// picture's true w x h, as read_sample does (gather.rs:16-31): the planes' borders are never relied on.
template <int N, int STEP>
__device__ __forceinline__ void predict(const uint8_t* __restrict__ ref, uint32_t pitch, int w, int h, int x, int y, int mvx,
                                        int mvy, uint32_t (&out)[N]) {
    const int dx = mvx >> 1, dy = mvy >> 1;  // floor: HalfPel::into_lerp_parameters
    const bool ix = mvx & 1, iy = mvy & 1;
    const uint8_t* r0 = ref + (size_t)clamp_to(y + dy, h - 1) * pitch;
    const uint8_t* r1 = ref + (size_t)clamp_to(y + dy + 1, h - 1) * pitch;
    uint32_t a[N + 1], b[N + 1];
#pragma unroll
    for (int j = 0; j <= N; j++) {
        const int sx = clamp_to(x + dx + j, w - 1) * STEP;
        if (j < N || ix) a[j] = STEP == 2 ? __ldg(reinterpret_cast<const uint16_t*>(r0 + sx)) : __ldg(r0 + sx);
        if (iy && (j < N || ix)) b[j] = STEP == 2 ? __ldg(reinterpret_cast<const uint16_t*>(r1 + sx)) : __ldg(r1 + sx);
    }
#pragma unroll
    for (int j = 0; j < N; j++) {
#pragma unroll
        for (int p = 0; p < STEP; p++) {
            const int sh = 8 * p;
            const uint32_t s00 = (a[j] >> sh) & 0xFF;
            uint32_t v = s00;
            if (ix && iy)
                v = (s00 + ((a[j + 1] >> sh) & 0xFF) + ((b[j] >> sh) & 0xFF) + ((b[j + 1] >> sh) & 0xFF) + 2) >> 2;
            else if (ix)
                v = (s00 + ((a[j + 1] >> sh) & 0xFF) + 1) >> 1;
            else if (iy)
                v = (s00 + ((b[j] >> sh) & 0xFF) + 1) >> 1;
            if (p == 0) out[j] = v;
            else out[j] |= v << 8;
        }
    }
}

// N residual values of one row of one plane from column x on: one N * 2-byte store when the columns are contiguous and
// aligned and all N lie in the slot, else one store per column inside the slot (width W)
template <int N>
__device__ __forceinline__ void store_row(int16_t* p, int64_t col_stride, int x, uint32_t W, const int (&v)[N]) {
    if (col_stride == 1 && x + N <= (int)W && !((uintptr_t)p & (2 * N - 1))) {
        uint32_t pair[N / 2];
#pragma unroll
        for (int i = 0; i < N / 2; i++) pair[i] = (uint32_t)(uint16_t)v[2 * i] | (uint32_t)(uint16_t)v[2 * i + 1] << 16;
        if constexpr (N == 4)
            *reinterpret_cast<uint2*>(p) = make_uint2(pair[0], pair[1]);
        else
            *reinterpret_cast<uint32_t*>(p) = pair[0];
        return;
    }
#pragma unroll
    for (int j = 0; j < N; j++)
        if (x + j < (int)W) p[j * col_stride] = (int16_t)v[j];
}

__global__ void __launch_bounds__(RES_THREADS) residual_kernel(const PicDev* __restrict__ pics, const MotionJob* __restrict__ jobs,
                                                               const h263cu_mb* __restrict__ mbs, const ResidualDst d) {
    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, role = warp % 3;
    const uint32_t cells_w = (d.width + 15) / 16, cells_h = (d.height + 15) / 16;
    const uint32_t cell = blockIdx.x * RES_CELLS + warp / 3;
    if (cell >= cells_w * cells_h) return;
    if (role < 2 ? !d.base[0] : !d.base[1] && !d.base[2]) return;
    const int X = (int)(cell % cells_w), Y = (int)(cell / cells_w);
    const PicDev& P = pics[blockIdx.y];
    const MotionJob J = jobs[blockIdx.y];
    const int w = P.w, h = P.h;
    // the record's flags (byte 8) and, when INTER, its four (x, y) int8 vectors (bytes 16..23)
    bool inter = false;
    uint2 mv = make_uint2(0, 0);
    if (X < J.mb_w && Y < J.mb_h) {
        const uint8_t* r = reinterpret_cast<const uint8_t*>(mbs + J.first_mb + Y * J.mb_w + X);
        inter = __ldg(r + 8) & H263CU_MB_INTER;
        if (inter) mv = __ldg(reinterpret_cast<const uint2*>(r + 16));
    }
    const int64_t slot = J.slot;
    if (role < 2) {
        const int t = role * 32 + lane, row = t >> 2, col = (t & 3) * 4;
        const int x = 16 * X + col, y = 16 * Y + row;
        if (y >= (int)d.height) return;
        int v[4] = {0, 0, 0, 0};
        if (y < h && x < w) {
            const uint32_t c4 = *reinterpret_cast<const uint32_t*>(P.cur[0] + (size_t)y * P.pitch_y + x);
            uint32_t pred[4] = {0, 0, 0, 0};
            if (inter) {
                const uint32_t k = 2 * (row >= 8) + (col >= 8);
                const uint32_t m = (k < 2 ? mv.x : mv.y) >> (16 * (k & 1));
                predict<4, 1>(P.ref[0], P.pitch_y, w, h, x, y, (int8_t)(m & 0xFF), (int8_t)(m >> 8), pred);
            }
#pragma unroll
            for (int j = 0; j < 4; j++) v[j] = x + j < w ? (int)((c4 >> (8 * j)) & 0xFF) - (int)pred[j] : 0;
        }
        store_row<4>(d.base[0] + slot * d.stride[0][0] + y * d.stride[0][1] + x * d.stride[0][2], d.stride[0][2], x, d.width, v);
    } else {
        const uint32_t cwS = (d.width + 1) / 2, chS = (d.height + 1) / 2;
        const int row = lane >> 2, col = (lane & 3) * 2;
        const int x = 8 * X + col, y = 8 * Y + row;
        if (y >= (int)chS) return;
        const int cw = P.cw, ch = P.ch;
        int vb[2] = {0, 0}, vr[2] = {0, 0};
        if (y < ch && x < cw) {
            // Cb Cr Cb Cr of columns x, x + 1
            const uint32_t c4 = *reinterpret_cast<const uint32_t*>(P.cur[1] + (size_t)y * P.pitch_c + 2 * x);
            uint32_t pred[2] = {0, 0};
            if (inter) {
                const int sx = (int8_t)(mv.x & 0xFF) + (int8_t)((mv.x >> 16) & 0xFF) + (int8_t)(mv.y & 0xFF) + (int8_t)((mv.y >> 16) & 0xFF);
                const int sy = (int8_t)((mv.x >> 8) & 0xFF) + (int8_t)(mv.x >> 24) + (int8_t)((mv.y >> 8) & 0xFF) + (int8_t)(mv.y >> 24);
                predict<2, CHROMA_STEP>(P.ref[1], P.pitch_c, cw, ch, x, y, average_sum_of_mvs(sx), average_sum_of_mvs(sy), pred);
            }
#pragma unroll
            for (int j = 0; j < 2; j++)
                if (x + j < cw) {
                    vb[j] = (int)((c4 >> (16 * j)) & 0xFF) - (int)(pred[j] & 0xFF);
                    vr[j] = (int)((c4 >> (16 * j + 8)) & 0xFF) - (int)(pred[j] >> 8);
                }
        }
        if (d.base[1])
            store_row<2>(d.base[1] + slot * d.stride[1][0] + y * d.stride[1][1] + x * d.stride[1][2], d.stride[1][2], x, cwS, vb);
        if (d.base[2])
            store_row<2>(d.base[2] + slot * d.stride[2][0] + y * d.stride[2][1] + x * d.stride[2][2], d.stride[2][2], x, cwS, vr);
    }
}

void launch_residual(const PicDev* pics, const MotionJob* jobs, uint32_t n_pics, const h263cu_mb* mbs, const ResidualDst& dst,
                     cudaStream_t stream) {
    const uint32_t cells = ((dst.width + 15) / 16) * ((dst.height + 15) / 16);
    const dim3 grid((cells + RES_CELLS - 1) / RES_CELLS, n_pics);
    residual_kernel<<<grid, RES_THREADS, 0, stream>>>(pics, jobs, mbs, dst);
}

}  // namespace h263dev
