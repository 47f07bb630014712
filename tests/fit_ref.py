"""Restatement of h263cu_decode_step_device_tensor_fit (include/h263cu.h): the integer geometry of each fit, and the
values as numpy float32 operations in the header's order (resample_ref.py's arithmetic, at an offset index over a crop
box, with the fill outside the placed picture).  The GPU tests compare the kernel against it bit for bit; the CPU tests
pin it to torchvision."""
import numpy as np

import resample_ref as R

F = np.float32
STRETCH, LETTERBOX, CENTER_CROP = 0, 1, 2
MODES = {"stretch": STRETCH, "letterbox": LETTERBOX, "center_crop": CENTER_CROP}


def geometry(mode, short_side, cw, ch, W, H):
    """(rw, rh, px, py): the size a cw x ch crop is resized to and where its top-left lands in the W x H output."""
    if mode == STRETCH:
        return W, H, 0, 0
    if mode == LETTERBOX:
        if cw * H >= ch * W:
            rw, rh = W, max(1, (2 * ch * W + cw) // (2 * cw))
        else:
            rw, rh = max(1, (2 * cw * H + ch) // (2 * ch)), H
        return rw, rh, (W - rw) // 2, (H - rh) // 2
    S = short_side
    rw, rh = (S, S * ch // cw) if cw <= ch else (S * cw // ch, S)

    def place(r, o):
        if r < o:
            return (o - r) // 2
        d = r - o
        k = d // 2
        return -(k + (k & 1) if d & 1 else k)

    return rw, rh, place(rw, W), place(rh, H)


def values(rgb, H, W, geom, crop=None, fill=(0.0, 0.0, 0.0), taps=R.axis_taps):
    """v: [3, H, W] float32 of an RGB picture [h, w, 3] (or the oracle's RGBA [h, w, 4]) under geometry `geom` of the
    crop (x, y, w, h) (None: the whole picture).  `taps` as in resample_ref.resample."""
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
    xi0, xi1, lx0, lx1 = (a[x0 - px:x1 - px] for a in taps(cw, rw))
    yi0, yi1, ly0, ly1 = (a[y0 - py:y1 - py] for a in taps(ch, rh))
    lx0, lx1 = lx0[None, :, None], lx1[None, :, None]
    ly0, ly1 = ly0[:, None, None], ly1[:, None, None]
    top = lx0 * p[yi0][:, xi0] + lx1 * p[yi0][:, xi1]
    bottom = lx0 * p[yi1][:, xi0] + lx1 * p[yi1][:, xi1]
    v[:, y0:y1, x0:x1] = (ly0 * top + ly1 * bottom).transpose(2, 0, 1)
    return v
