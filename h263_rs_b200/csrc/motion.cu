// motion.cu -- the motion fields of h263cu_decode_step_device_motion (include/h263cu.h): per macroblock cell of each
// picture's slot grid, the record's flags (INTER | FOURMV | CODED), its quantiser and its four luma vectors, read from
// the step's h263cu_mb records where they already are and written through the caller's strides.
#include "kernels.cuh"

namespace h263dev {

constexpr int MOTION_THREADS = 128;

__global__ void __launch_bounds__(MOTION_THREADS) motion_field_kernel(const MotionJob* __restrict__ jobs, const h263cu_mb* __restrict__ mbs,
                                                                      const MotionDst d) {
    const uint32_t cell = blockIdx.x * MOTION_THREADS + threadIdx.x;
    if (cell >= d.mb_width * d.mb_height) return;
    const MotionJob J = jobs[blockIdx.y];
    const uint32_t X = cell % d.mb_width, Y = cell / d.mb_width;
    uint32_t flags = H263CU_MOTION_OUTSIDE, quant = 0, mv[4] = {0, 0, 0, 0};  // mv[k]: x in bits 0..7, y in 8..15
    if (X < J.mb_w && Y < J.mb_h) {
        // the record's bytes 8..11 (mbx, mby, flags, quant) and 16..23 (the union: four (x, y) int8 pairs when INTER)
        const uint8_t* r = reinterpret_cast<const uint8_t*>(mbs + J.first_mb + Y * J.mb_w + X);
        const uint32_t w2 = __ldg(reinterpret_cast<const uint32_t*>(r + 8));
        const uint2 u = __ldg(reinterpret_cast<const uint2*>(r + 16));
        flags = w2 & (H263CU_MB_INTER | H263CU_MB_FOURMV | H263CU_MB_CODED);
        quant = (w2 >> 8) & 0xFFu;
        if (flags & H263CU_MB_INTER) mv[0] = u.x & 0xFFFFu, mv[1] = u.x >> 16, mv[2] = u.y & 0xFFFFu, mv[3] = u.y >> 16;
    }
    const int64_t slot = J.slot;
    if (d.flags) d.flags[slot * d.flags_stride[0] + Y * d.flags_stride[1] + X * d.flags_stride[2]] = (uint8_t)flags;
    if (d.quant) d.quant[slot * d.quant_stride[0] + Y * d.quant_stride[1] + X * d.quant_stride[2]] = (uint8_t)quant;
    if (d.mv) {
        int16_t* base = d.mv + slot * d.mv_stride[0];
#pragma unroll
        for (int k = 0; k < 4; k++) {
            int16_t* p = base + (int64_t)(2 * Y + (k >> 1)) * d.mv_stride[2] + (int64_t)(2 * X + (k & 1)) * d.mv_stride[3];
            p[0] = (int16_t)(int8_t)(mv[k] & 0xFFu);
            p[d.mv_stride[1]] = (int16_t)(int8_t)(mv[k] >> 8);
        }
    }
}

void launch_motion_field(const MotionJob* jobs, uint32_t n_pics, const h263cu_mb* mbs, const MotionDst& dst, cudaStream_t stream) {
    const uint32_t cells = dst.mb_width * dst.mb_height;
    const dim3 grid((cells + MOTION_THREADS - 1) / MOTION_THREADS, n_pics);
    motion_field_kernel<<<grid, MOTION_THREADS, 0, stream>>>(jobs, mbs, dst);
}

}  // namespace h263dev
