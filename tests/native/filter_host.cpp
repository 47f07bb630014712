// Host build of the antialiased weights of device_math.cuh (aa_support, aa_invscale, aa_span, aa_raw, aa_total,
// aa_weight) for tests/test_device_tensor_filter_abi.py: g++ -ffp-contract=off, checked bit for bit against
// tests/filter_ref.py.
#include <stddef.h>

#include "../../h263_rs_b200/csrc/device_math.cuh"

using namespace h263dev;

extern "C" {

// the taps of every output index of one axis of n_out samples taken from n_in: xmin[i], xsize[i] and the normalised
// weights w[i * max_taps + j] for j < min(xsize[i], max_taps)
void aa_axis(int n_in, int n_out, int bicubic, int max_taps, int* xmin, int* xsize, float* w) {
    const float scale = axis_scale(n_in, n_out);
    const float support = aa_support(scale, bicubic ? 2 : 1), invscale = aa_invscale(scale);
    for (int i = 0; i < n_out; i++) {
        const AaSpan s = aa_span(i, scale, support, n_in);
        const float total = aa_total(s, invscale, bicubic);
        xmin[i] = s.min, xsize[i] = s.size;
        for (int j = 0; j < s.size && j < max_taps; j++) w[(size_t)i * max_taps + j] = aa_weight(aa_raw(s, j, invscale, bicubic), total);
    }
}
}
