// Host build of the resampling arithmetic of device_math.cuh (axis_scale, axis_tap, bilinear) for
// tests/test_device_tensor_abi.py: g++ -ffp-contract=off, checked bit for bit against tests/resample_ref.py.
#include <stddef.h>

#include "../../h263_rs_b200/csrc/device_math.cuh"

using namespace h263dev;

extern "C" {

// the taps of every output index of one axis of n_out samples taken from n_in
void rs_axis(int n_in, int n_out, int* i0, int* i1, float* l0, float* l1) {
    const float scale = axis_scale(n_in, n_out);
    for (int x = 0; x < n_out; x++) {
        const AxisTap t = axis_tap(x, scale, n_in);
        i0[x] = t.i0, i1[x] = t.i1, l0[x] = t.l0, l1[x] = t.l1;
    }
}

// v[c][Y][X] of a tight RGB picture rgb[h][w][3]
void rs_resample(const uint8_t* rgb, int w, int h, int W, int H, float* v) {
    const float sx = axis_scale(w, W), sy = axis_scale(h, H);
    for (int Y = 0; Y < H; Y++) {
        const AxisTap ty = axis_tap(Y, sy, h);
        for (int X = 0; X < W; X++) {
            const AxisTap tx = axis_tap(X, sx, w);
            for (int c = 0; c < 3; c++) {
                const auto p = [&](int x, int y) { return (float)rgb[((size_t)y * w + x) * 3 + c]; };
                v[((size_t)c * H + Y) * W + X] = bilinear(tx, ty, p(tx.i0, ty.i0), p(tx.i1, ty.i0), p(tx.i0, ty.i1), p(tx.i1, ty.i1));
            }
        }
    }
}
}
