"""Restatement of h263cu_decode_step_device_tensor_filter (include/h263cu.h): torch's antialiased bilinear / bicubic
weights and the separable passes as numpy float32 operations in the header's order, under the fit geometry of
fit_ref.py.  The GPU tests compare the kernel against it bit for bit; the CPU tests pin it to torch / torchvision."""
import numpy as np

F = np.float32
BILINEAR, BILINEAR_AA, BICUBIC_AA = 0, 1, 2


def aa_filter(t, bicubic):
    """The triangle max(0, 1 - |t|), or Keys' cubic (a = -0.5) in torch's cubic_convolution1 / 2 order."""
    x = np.abs(np.asarray(t, F))
    if not bicubic:
        return np.where(x < F(1), F(1) - x, F(0)).astype(F)
    c1 = ((F(1.5) * x + F(-2.5)) * x) * x + F(1)
    c2 = ((F(-0.5) * x + F(2.5)) * x + F(-4)) * x + F(2)
    return np.where(x < F(1), c1, np.where(x < F(2), c2, F(0))).astype(F)


def aa_taps(n_in, n_out, bicubic):
    """Per output index of one axis: the first source sample xmin, the tap count xsize and the normalised weights
    w[n_out, max xsize] (0 past xsize)."""
    scale = F(n_in) / F(n_out)
    r = F(2 if bicubic else 1)
    support = r * scale if scale >= F(1) else r
    invscale = F(1) / scale if scale >= F(1) else F(1)
    center = scale * (np.arange(n_out, dtype=F) + F(0.5))
    xmin = np.maximum((center - support + F(0.5)).astype(np.int32), 0)
    xsize = np.minimum((center + support + F(0.5)).astype(np.int32), n_in) - xmin
    j = np.arange(int(xsize.max()), dtype=np.int32)[None, :]
    live = j < xsize[:, None]
    raw = aa_filter(((xmin[:, None] + j).astype(F) - center[:, None] + F(0.5)) * invscale, bicubic)
    raw = np.where(live, raw, F(0))
    total = np.zeros(n_out, F)
    for k in range(raw.shape[1]):
        total = np.where(live[:, k], total + raw[:, k], total)
    w = np.where(total[:, None] != 0, raw / np.where(total == 0, F(1), total)[:, None], raw).astype(F)
    return xmin, xsize, np.where(live, w, F(0))


def _pass(p, xmin, xsize, w, axis):
    """Sum_j w_j * p[xmin + j] along `axis` (0: rows, 1: columns) of p [rows, columns, 3], ascending j, the first term a
    product."""
    p = np.moveaxis(p, axis, 0)
    acc = w[:, 0, None, None] * p[xmin]
    for j in range(1, w.shape[1]):
        live = (j < xsize)[:, None, None]
        acc = np.where(live, acc + w[:, j, None, None] * p[np.minimum(xmin + j, p.shape[0] - 1)], acc)
    return np.moveaxis(acc.astype(F), 0, axis)


def values(rgb, H, W, geom, crop=None, fill=(0.0, 0.0, 0.0), filt=BILINEAR_AA):
    """v: [3, H, W] float32 of an RGB picture [h, w, 3] (or the oracle's RGBA [h, w, 4]) under geometry `geom` =
    (rw, rh, px, py) of the crop (x, y, w, h) (None: the whole picture), resized with the antialiased filter `filt`."""
    p = np.asarray(rgb)[..., :3].astype(F)
    h, w = p.shape[:2]
    cx, cy, cw, ch = crop if crop is not None else (0, 0, w, h)
    p = p[cy:cy + ch, cx:cx + cw]
    rw, rh, px, py = geom
    v = np.empty((3, H, W), F)
    v[:] = np.asarray(fill, F).reshape(3, 1, 1)
    x0, x1, y0, y1 = max(0, px), min(W, px + rw), max(0, py), min(H, py + rh)
    if x0 >= x1 or y0 >= y1:
        return v
    bicubic = filt == BICUBIC_AA
    xm, xs, wx = (a[x0 - px:x1 - px] for a in aa_taps(cw, rw, bicubic))
    ym, ys, wy = (a[y0 - py:y1 - py] for a in aa_taps(ch, rh, bicubic))
    hor = _pass(p, xm, xs, wx, 1)      # [ch, x1 - x0, 3]
    ver = _pass(hor, ym, ys, wy, 0)    # [y1 - y0, x1 - x0, 3]
    v[:, y0:y1, x0:x1] = ver.transpose(2, 0, 1)
    return v


def store(v, mul=(1.0, 1.0, 1.0), add=(0.0, 0.0, 0.0), u8=False):
    """Step 4 for the filters: uint8 max(0, min(255, (int)(v + 0.5))), or float32 t = v * mul[c] + add[c] (to be cast
    to f16 / bf16 by the caller, round to nearest even), unclamped."""
    if u8:
        return np.clip((v + F(0.5)).astype(np.int32), 0, 255).astype(np.uint8)
    mul = np.asarray(mul, F)[:, None, None]
    add = np.asarray(add, F)[:, None, None]
    return (v * mul + add).astype(F)
