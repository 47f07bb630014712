// device_math.cuh -- arithmetic primitives of the reconstruction path.
//
// Every function is `HD` (host + device) and branch-light so that the same code is
// (a) inlined into the sm_100a kernels and (b) compiled with g++ into the CPU self-test
// (tests/test_device_math.py) which checks it against the oracle without a GPU.
// Floating point uses explicit round-to-nearest intrinsics on the device (never
// contracted into FMA; the build also passes -fmad=false) and plain operators under
// -ffp-contract=off on the host, so both follow the reference's operation order
// (h263/src/decoder/cpu/idct.rs:52-65).
#pragma once
#include <stdint.h>

#if defined(__CUDACC__)
#define HD __host__ __device__ __forceinline__
#else
#define HD static inline
#endif

namespace h263dev {

#if defined(__CUDA_ARCH__)
HD float fmul(float a, float b) { return __fmul_rn(a, b); }
HD float fadd(float a, float b) { return __fadd_rn(a, b); }
#else
HD float fmul(float a, float b) {
    volatile float r = a * b;  // volatile: keep the product a separately rounded f32
    return r;
}
HD float fadd(float a, float b) {
    volatile float r = a + b;
    return r;
}
#endif

// BASIS_TABLE[freq][i] (idct.rs:39-48): the reference's f32 literals.
#define H263_BASIS_TABLE                                                                                         \
    {                                                                                                            \
        {0.70710677f, 0.70710677f, 0.70710677f, 0.70710677f, 0.70710677f, 0.70710677f, 0.70710677f, 0.70710677f}, \
        {0.98078525f, 0.8314696f, 0.5555702f, 0.19509023f, -0.19509032f, -0.55557036f, -0.83146966f, -0.9807853f}, \
        {0.9238795f, 0.38268343f, -0.38268352f, -0.9238796f, -0.9238795f, -0.38268313f, 0.3826836f, 0.92387956f},  \
        {0.8314696f, -0.19509032f, -0.9807853f, -0.55557f, 0.55557007f, 0.98078525f, 0.19509007f, -0.8314698f},    \
        {0.70710677f, -0.70710677f, -0.70710665f, 0.707107f, 0.70710677f, -0.70710725f, -0.70710653f, 0.7071068f}, \
        {0.5555702f, -0.9807853f, 0.19509041f, 0.83146936f, -0.8314698f, -0.19508928f, 0.9807853f, -0.55557007f},  \
        {0.38268343f, -0.9238795f, 0.92387974f, -0.3826839f, -0.38268384f, 0.9238793f, -0.92387974f, 0.3826839f},  \
        {0.19509023f, -0.55557f, 0.83146936f, -0.9807852f, 0.98078525f, -0.83147013f, 0.55557114f, -0.19508967f},  \
    }
#define H263_B00 0.70710677f

// Zig-zag scan position -> y*8+x (rle.rs:6-71 stores (x, y); we store the linear index).
#define H263_DEZIGZAG_LINEAR                                                                                      \
    {                                                                                                             \
        0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, 7, \
            14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, 31,   \
            39, 46, 53, 60, 61, 54, 47, 55, 62, 63                                                                \
    }

// H.263 dequantisation in wrapping i16 (rle.rs:130-133):
//   clamp(sign(level) * (QP*(2|level|+1) - (QP even ? 1 : 0)), -2048, 2047)
HD int dequant(int level, int quant) {
    int absl = (int16_t)(level < 0 ? -level : level);
    int deq = (int16_t)(quant * (int16_t)(2 * absl + 1));
    int parity = (quant & 1) ? 0 : -1;
    int mag = (int16_t)(deq + parity);
    int sgn = level > 0 ? 1 : (level < 0 ? -1 : 0);
    int value = (int16_t)(sgn * mag);
    return value < -2048 ? -2048 : (value > 2047 ? 2047 : value);
}

// IntraDc::into_level (types.rs:955-961)
HD int intradc_level(int code) { return code == 0xFF ? 1024 : (code << 3); }

HD float copysign_half(float v) {
#if defined(__CUDA_ARCH__)
    return __int_as_float((__float_as_int(v) & 0x80000000) | 0x3F000000);
#else
    union {
        float f;
        uint32_t u;
    } a;
    a.f = v;
    a.u = (a.u & 0x80000000u) | 0x3F000000u;
    return a.f;
#endif
}

HD int trunc_to_int(float v) {
#if defined(__CUDA_ARCH__)
    return __float2int_rz(v);
#else
    if (v >= 2147483520.0f) return 2147483647;
    if (v <= -2147483648.0f) return (int)0x80000000;
    return (int)v;
#endif
}

// `((idct / 4.0 + idct.signum() * 0.5) as i16).clamp(-256, 255)` (idct.rs:189-190).
// v/4 is an exact power-of-two scaling, so v*0.25 rounds identically.
HD int round_residual(float v) {
    int r = trunc_to_int(fadd(fmul(v, 0.25f), copysign_half(v)));
    return r < -256 ? -256 : (r > 255 ? 255 : r);
}
// Horiz / Vert form: `idct * BASIS_TABLE[0][0] / 4.0 + idct.signum() * 0.5` (idct.rs:143-145,
// 161-163); the sign is that of the unscaled value.
HD int round_residual_scaled(float v) {
    int r = trunc_to_int(fadd(fmul(fmul(v, H263_B00), 0.25f), copysign_half(v)));
    return r < -256 ? -256 : (r > 255 ? 255 : r);
}
// Dc form: `dc * 0.5 / 4.0 + dc.signum() * 0.5` (idct.rs:119-121)
HD int round_residual_dc(float dc) {
    int r = trunc_to_int(fadd(fmul(fmul(dc, 0.5f), 0.25f), copysign_half(dc)));
    return r < -256 ? -256 : (r > 255 ? 255 : r);
}

HD int clamp_u8(int v) { return v < 0 ? 0 : (v > 255 ? 255 : v); }

// ---- packed-byte motion compensation (gather.rs:34-40, 103-113) -----------------------
// per byte (a + b + 1) >> 1
HD uint32_t avg2_u8x4(uint32_t a, uint32_t b) { return (a | b) - (((a ^ b) >> 1) & 0x7F7F7F7Fu); }
// per byte (a + b + c + d + 2) >> 2, exact
HD uint32_t avg4_u8x4(uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
    uint32_t lo = (a & 0x03030303u) + (b & 0x03030303u) + (c & 0x03030303u) + (d & 0x03030303u) + 0x02020202u;
    uint32_t hi = ((a >> 2) & 0x3F3F3F3Fu) + ((b >> 2) & 0x3F3F3F3Fu) + ((c >> 2) & 0x3F3F3F3Fu) +
                  ((d >> 2) & 0x3F3F3F3Fu);
    return hi + ((lo >> 2) & 0x0F0F0F0Fu);
}

// HalfPel::average_sum_of_mvs (types.rs:759-768) on one component
HD int average_sum_of_mvs(int s) {
    int whole = (s >> 4) << 1;
    int frac = s & 15;
    return frac <= 2 ? whole : (frac >= 14 ? whole + 2 : whole + 1);
}

// ---- BT.601 (yuv/src/bt601.rs:12-59) ------------------------------------------------
// Per-chroma-sample terms, shared by the pixels under one chroma sample.
struct ChromaTerms {
    int r, g, b;
};
HD ChromaTerms chroma_terms(int cb, int cr) {
    ChromaTerms t;
    int cbp = cb - 128, crp = cr - 128;
    t.r = crp * 104597 + 32768;
    t.g = crp * -53279 + cbp * -25675 + 32768;
    t.b = cbp * 132201 + 32768;
    return t;
}
// One pixel -> packed R | G<<8 | B<<16 | 255<<24
HD uint32_t yuv_pixel(int y, const ChromaTerms& t) {
    int gray = (y - 16) * 76309;
    int r = clamp_u8((gray + t.r) >> 16);
    int g = clamp_u8((gray + t.g) >> 16);
    int b = clamp_u8((gray + t.b) >> 16);
    return (uint32_t)r | ((uint32_t)g << 8) | ((uint32_t)b << 16) | 0xFF000000u;
}

// ---- bilinear resampling (h263cu_decode_step_device_tensor) ----------------------------
// One axis of torch's align_corners=False rule: output index X of an axis of `out` samples taken from an axis of `in`
// samples reads source samples i0 and i1 with weights l0 and l1 (include/h263cu.h states the definition).
struct AxisTap {
    int i0, i1;
    float l0, l1;
};
HD float axis_scale(int in, int out) {
#if defined(__CUDA_ARCH__)
    return __fdiv_rn((float)in, (float)out);
#else
    volatile float r = (float)in / (float)out;
    return r;
#endif
}
HD AxisTap axis_tap(int X, float scale, int in) {
    float s = fadd(fmul(scale, fadd((float)X, 0.5f)), -0.5f);
    if (!(s > 0.0f)) s = 0.0f;
    AxisTap t;
    t.i0 = (int)s;
    t.i1 = t.i0 + (t.i0 < in - 1 ? 1 : 0);
    t.l1 = fadd(s, -(float)t.i0);
    t.l0 = fadd(1.0f, -t.l1);
    return t;
}
// v = ly0 * (lx0 * p00 + lx1 * p10) + ly1 * (lx0 * p01 + lx1 * p11), p<x><y>, in this order
HD float bilinear(const AxisTap& tx, const AxisTap& ty, float p00, float p10, float p01, float p11) {
    return fadd(fmul(ty.l0, fadd(fmul(tx.l0, p00), fmul(tx.l1, p10))), fmul(ty.l1, fadd(fmul(tx.l0, p01), fmul(tx.l1, p11))));
}

// ---- antialiased resampling (h263cu_decode_step_device_tensor_filter) -------------------------------------------------
// One axis of torch's antialias=True rule (ATen/native/cuda/UpSample.cuh: _compute_weights_span, _compute_weights):
// output index i reads the `size` source samples from `min` with weights aa_weight(aa_raw(span, j, ...), total).
// include/h263cu.h states the definition and the operation order.
HD float fdiv(float a, float b) {
#if defined(__CUDA_ARCH__)
    return __fdiv_rn(a, b);
#else
    volatile float r = a / b;
    return r;
#endif
}
struct AaSpan {
    float center;
    int min, size;
};
// r = 1 (bilinear) or 2 (bicubic): half the filter's width
HD float aa_support(float scale, int r) { return scale >= 1.0f ? fmul((float)r, scale) : (float)r; }
HD float aa_invscale(float scale) { return scale >= 1.0f ? fdiv(1.0f, scale) : 1.0f; }
HD AaSpan aa_span(int i, float scale, float support, int in) {
    AaSpan s;
    s.center = fmul(scale, fadd((float)i, 0.5f));
    s.min = trunc_to_int(fadd(fadd(s.center, -support), 0.5f));
    if (s.min < 0) s.min = 0;
    int hi = trunc_to_int(fadd(fadd(s.center, support), 0.5f));
    if (hi > in) hi = in;
    s.size = hi - s.min;
    return s;
}
// The triangle max(0, 1 - |t|), or Keys' cubic with a = -0.5 in torch's cubic_convolution1 / 2 order
// (ATen/native/UpSample.h): ((a + 2) * x - (a + 3)) * x * x + 1 below 1, ((a * x - 5a) * x + 8a) * x - 4a below 2.
HD float aa_filter(float t, int bicubic) {
    const float x = t < 0.0f ? -t : t;
    if (!bicubic) return x < 1.0f ? fadd(1.0f, -x) : 0.0f;
    if (x < 1.0f) return fadd(fmul(fmul(fadd(fmul(1.5f, x), -2.5f), x), x), 1.0f);
    if (x < 2.0f) return fadd(fmul(fadd(fmul(fadd(fmul(-0.5f, x), 2.5f), x), -4.0f), x), 2.0f);
    return 0.0f;
}
// filter(((float)(min + j) - center + 0.5f) * invscale), before normalisation
HD float aa_raw(const AaSpan& s, int j, float invscale, int bicubic) {
    return aa_filter(fmul(fadd(fadd((float)(s.min + j), -s.center), 0.5f), invscale), bicubic);
}
// the sum of the raw weights in ascending j
HD float aa_total(const AaSpan& s, float invscale, int bicubic) {
    float t = 0.0f;
    for (int j = 0; j < s.size; j++) t = fadd(t, aa_raw(s, j, invscale, bicubic));
    return t;
}
HD float aa_weight(float raw, float total) { return total != 0.0f ? fdiv(raw, total) : raw; }

// ---- deblocking filter (deblock/src/deblock.rs:29-42, 99-127) -------------------------
// trunc == 0: `process_simd` lane semantics (arithmetic shifts = floor division);
// trunc != 0: scalar `process` semantics (truncating division).  The two differ for
// negative operands and the reference uses both (SIMD body vs scalar tail), SURVEY.md T10.
HD void deblock_process(int& A, int& B, int& C, int& D, int strength, int trunc) {
    int s = A - 4 * B + 4 * C - D;
    int d = trunc ? s / 8 : s >> 3;
    int ad = d < 0 ? -d : d;
    int inner = 2 * (ad - strength);
    if (inner < 0) inner = 0;
    int ramp = ad - inner;
    if (ramp < 0) ramp = 0;
    int d1 = d < 0 ? -ramp : ramp;
    int half = trunc ? d1 / 2 : d1 >> 1;
    int lim = half < 0 ? -half : half;
    int q = trunc ? (A - D) / 4 : (A - D) >> 2;
    int d2 = q < -lim ? -lim : (q > lim ? lim : q);
    A = (A - d2) & 0xFF;
    B = clamp_u8(B + d1);
    C = clamp_u8(C - d1);
    D = (D + d2) & 0xFF;
}

#define H263_QUANT_TO_STRENGTH \
    { 0, 1, 1, 2, 2, 3, 3, 4, 4, 4, 5, 5, 6, 6, 7, 7, 7, 8, 8, 8, 9, 9, 9, 10, 10, 10, 11, 11, 11, 12, 12, 12 }

}  // namespace h263dev
