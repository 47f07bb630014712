"""numpy float32 restatement of the output of h263cu_decode_step_device_tensor (include/h263cu.h, steps 2-4): the
reference the GPU tests compare the resample kernel against, bit for bit.  Every operation is one IEEE fp32 operation
rounded to nearest, in the order the header states."""
import numpy as np

F = np.float32


def axis_taps(n_in, n_out):
    """Per output index of one axis: source indices i0, i1 and weights l0, l1 (torch's align_corners=False rule)."""
    scale = F(n_in) / F(n_out)
    s = scale * (np.arange(n_out, dtype=F) + F(0.5)) - F(0.5)
    s = np.maximum(s, F(0))
    i0 = s.astype(np.int32)
    i1 = i0 + (i0 < n_in - 1).astype(np.int32)
    l1 = s - i0.astype(F)
    l0 = F(1) - l1
    return i0, i1, l0, l1


def resample(rgb, height, width, taps=axis_taps):
    """v: [3, height, width] float32 from an RGB picture [h, w, 3] (uint8 or the RGBA [h, w, 4] the oracle gives).
    `taps` computes the per-axis taps (a test swaps in torch's contracted coordinate)."""
    p = np.asarray(rgb)[..., :3].astype(F)
    h, w = p.shape[:2]
    xi0, xi1, lx0, lx1 = taps(w, width)
    yi0, yi1, ly0, ly1 = taps(h, height)
    lx0, lx1 = lx0[None, :, None], lx1[None, :, None]
    ly0, ly1 = ly0[:, None, None], ly1[:, None, None]
    top = lx0 * p[yi0][:, xi0] + lx1 * p[yi0][:, xi1]
    bottom = lx0 * p[yi1][:, xi0] + lx1 * p[yi1][:, xi1]
    v = ly0 * top + ly1 * bottom
    return np.ascontiguousarray(v.transpose(2, 0, 1))


def store(v, mul=(1.0, 1.0, 1.0), add=(0.0, 0.0, 0.0), u8=False):
    """Step 4: uint8 min(255, (int)(v + 0.5)), or float32 t = v * mul[c] + add[c] (to be cast to f16 / bf16 by the
    caller, round to nearest even)."""
    if u8:
        return np.minimum((v + F(0.5)).astype(np.int32), 255).astype(np.uint8)
    mul = np.asarray(mul, F)[:, None, None]
    add = np.asarray(add, F)[:, None, None]
    return (v * mul + add).astype(F)


def normalisation(mean, std):
    """mul = 1 / (255 * std), add = -mean / std: computed in float64, rounded once to float32."""
    std = np.asarray(std, np.float64)
    return (1.0 / (255.0 * std)).astype(F), (-np.asarray(mean, np.float64) / std).astype(F)
