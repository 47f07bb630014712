"""Host-side mirror of the reference's public API, backed by libh263cu.so.

Names, argument meaning and error behaviour follow the reference so that the parity
tests read like the reference's own tests:

    h263::H263State::{new, decode_next_picture, get_last_picture, is_sorenson}   state.rs:40-141
    h263::DecodedPicture::{as_yuv, as_luma, as_chroma_b, as_chroma_r, ...}         picture.rs:60-142
    yuv::bt601::yuv420_to_rgba(y, chroma_b, chroma_r, y_width) -> Vec<u8>          bt601.rs:105
    deblock::deblock::deblock(data, width, strength) -> Vec<u8>, QUANT_TO_STRENGTH deblock.rs:5-8,305

plus `BatchDecoder`, the batched form the GPU path is built for (one picture for each of
many independent streams per step).  All compute runs on the GPU through the C ABI; there
is no CPU fallback (errors surface as H263Error).
"""
import ctypes as C

import numpy as np

from . import _lib, frontend
from ._lib import H263Error, check

SORENSON_SPARK_BITSTREAM = _lib.OPT_SORENSON
USE_SCALABILITY_MODE = 2


def _quant_to_strength():
    arr = (C.c_uint8 * 32).in_dll(_lib.lib(), "h263cu_quant_to_strength")
    return [int(v) for v in arr]


class _LazyTable:
    def __init__(self):
        self._v = None

    def _get(self):
        if self._v is None:
            self._v = _quant_to_strength()
        return self._v

    def __getitem__(self, i):
        return self._get()[i]

    def __len__(self):
        return 32

    def __iter__(self):
        return iter(self._get())


QUANT_TO_STRENGTH = _LazyTable()


def yuv420_to_rgba(y, chroma_b, chroma_r, y_width):
    """yuv::bt601::yuv420_to_rgba: planar YUV 4:2:0 -> interleaved RGBA8888 (GPU)."""
    y = np.ascontiguousarray(y, np.uint8).reshape(-1)
    cb = np.ascontiguousarray(chroma_b, np.uint8).reshape(-1)
    cr = np.ascontiguousarray(chroma_r, np.uint8).reshape(-1)
    out = np.empty(y.size * 4, np.uint8)
    if y.size == 0:
        return out
    check(_lib.lib().h263cu_yuv420_to_rgba(y.ctypes.data, cb.ctypes.data, cr.ctypes.data, y.size, y_width,
                                           out.ctypes.data))
    return out


def deblock(data, width, strength):
    """deblock::deblock::deblock: Annex-J-style post filter on one plane (GPU)."""
    data = np.ascontiguousarray(data, np.uint8).reshape(-1)
    out = np.empty(data.size, np.uint8)
    if data.size == 0:
        return out
    check(_lib.lib().h263cu_deblock(data.ctypes.data, data.size, width, strength, out.ctypes.data))
    return out


def _device_rgba(out, n_slots, max_w, max_h, device):
    """The h263cu_device_rgba of a torch.uint8 CUDA tensor [slots, H, W, 4] on `device` (tight RGBA pixels; rows and
    slots may be padded), allocated as [n_slots, max_h, round_up(max_w, 4), 4] and returned as its [..., :max_w, :] view
    when `out` is None.  Raises ValueError when the tensor breaks a rule of the C ABI (include/h263cu.h), so that
    nothing is parsed.  The consumer stream is torch's current stream on the device."""
    import torch

    dev = torch.device("cuda", device)
    if out is None:
        out = torch.empty((n_slots, max_h, (max_w + 3) // 4 * 4, 4), dtype=torch.uint8, device=dev)[:, :, :max_w, :]
    if not isinstance(out, torch.Tensor) or out.dtype != torch.uint8 or out.device != dev:
        raise ValueError("out must be a torch.uint8 tensor on %s" % dev)
    if out.dim() != 4 or out.shape[3] != 4 or out.shape[0] < n_slots or out.shape[1] == 0 or out.shape[2] == 0:
        raise ValueError("out must have the shape [>= %d, H > 0, W > 0, 4], not %s" % (n_slots, tuple(out.shape)))
    slots, h, w, _ = out.shape
    s0, s1, s2, s3 = out.stride()
    if (w > 1 and s2 != 4) or s3 != 1:
        raise ValueError("out must hold tight R,G,B,A pixels (strides [..., 4, 1]), not %s" % (out.stride(),))
    # a dimension of size 1 has no stride of its own: take the tightest one the ABI allows
    row_pitch = s1 if h > 1 else (4 * w + 15) // 16 * 16
    pic_stride = s0 if slots > 1 else row_pitch * h
    base = out.data_ptr()
    if base % 16 or row_pitch % 16 or row_pitch < 4 * w or row_pitch >= 1 << 32:
        raise ValueError("out: base must be 16-byte aligned and the row stride a multiple of 16 bytes, >= 4 * W, < 2^32")
    if pic_stride % 16 or pic_stride < row_pitch * h or pic_stride >= 1 << 40:
        raise ValueError("out: the slot stride must be a multiple of 16 bytes, >= row stride * H, < 2^40")
    stream = torch.cuda.current_stream(dev).cuda_stream
    return out, _lib.DeviceRgba(base, row_pitch, pic_stride, w, h, stream or None)


_YUV_LAYOUTS = {"i420": _lib.YUV_I420, "nv12": _lib.YUV_NV12}


def _device_plane(t, name, n_slots, rows, cols, pair, dev):
    """The h263cu_device_plane of one plane tensor: [slots, rows, cols] uint8 with tight samples, or with `pair`
    [slots, rows, cols, 2] with tight CbCr pairs.  Raises ValueError for what the C ABI refuses."""
    import torch

    if not isinstance(t, torch.Tensor) or t.dtype != torch.uint8 or t.device != dev:
        raise ValueError("%s must be a torch.uint8 tensor on %s" % (name, dev))
    shape = (rows, cols, 2) if pair else (rows, cols)
    if t.dim() != 1 + len(shape) or t.shape[0] < n_slots or tuple(t.shape[1:]) != shape:
        raise ValueError("%s must have the shape [>= %d, %s], not %s" % (name, n_slots, ", ".join(map(str, shape)), tuple(t.shape)))
    st = t.stride()
    if pair and ((cols > 1 and st[2] != 2) or st[3] != 1):
        raise ValueError("%s must hold tight CbCr pairs (strides [..., 2, 1]), not %s" % (name, st))
    if not pair and cols > 1 and st[2] != 1:
        raise ValueError("%s must hold tight samples (last stride 1), not %s" % (name, st))
    row_bytes = cols * (2 if pair else 1)
    # a dimension of size 1 has no stride of its own: take the tightest one the ABI allows
    row_pitch = st[1] if rows > 1 else (row_bytes + 3) // 4 * 4
    pic_stride = st[0] if t.shape[0] > 1 else row_pitch * rows
    base = t.data_ptr()
    if base % 4 or row_pitch % 4 or row_pitch < row_bytes or row_pitch >= 1 << 32:
        raise ValueError("%s: base must be 4-byte aligned and the row stride a multiple of 4 bytes, >= %d, < 2^32" % (name, row_bytes))
    if pic_stride % 4 or pic_stride < row_pitch * rows or pic_stride >= 1 << 40:
        raise ValueError("%s: the slot stride must be a multiple of 4 bytes, >= row stride * %d, < 2^40" % (name, rows))
    return _lib.DevicePlane(base, row_pitch, pic_stride)


def _device_yuv(out, n_slots, max_w, max_h, device, layout):
    """The h263cu_device_yuv of torch.uint8 CUDA plane tensors on `device`: (y [slots, H, W], cb [slots, ch, cw],
    cr [slots, ch, cw]) for layout "i420", (y [slots, H, W], uv [slots, ch, cw, 2]) for "nv12", ch = ceil(H / 2),
    cw = ceil(W / 2); rows and slots may be padded.  out=None allocates n_slots slots of max_w x max_h with rows padded
    to multiples of 4 bytes and returns views of them.  Raises ValueError when a tensor breaks a rule of the C ABI
    (include/h263cu.h), so that nothing is parsed.  The consumer stream is torch's current stream on the device."""
    import torch

    if layout not in _YUV_LAYOUTS:
        raise ValueError("layout must be one of %s, not %r" % (sorted(_YUV_LAYOUTS), layout))
    nv12 = layout == "nv12"
    dev = torch.device("cuda", device)
    if out is None:
        ch, cw = (max_h + 1) // 2, (max_w + 1) // 2
        y = torch.empty((n_slots, max_h, (max_w + 3) // 4 * 4), dtype=torch.uint8, device=dev)[:, :, :max_w]
        if nv12:
            out = (y, torch.empty((n_slots, ch, (cw + 1) // 2 * 2, 2), dtype=torch.uint8, device=dev)[:, :, :cw, :])
        else:
            out = (y,) + tuple(torch.empty((n_slots, ch, (cw + 3) // 4 * 4), dtype=torch.uint8, device=dev)[:, :, :cw] for _ in range(2))
    out = tuple(out)
    if len(out) != (2 if nv12 else 3):
        raise ValueError("out must be (y, uv) for nv12 and (y, cb, cr) for i420")
    y = out[0]
    if not isinstance(y, torch.Tensor) or y.dim() != 3 or y.shape[1] == 0 or y.shape[2] == 0:
        raise ValueError("y must be a tensor [slots, H > 0, W > 0]")
    h, w = int(y.shape[1]), int(y.shape[2])
    ch, cw = (h + 1) // 2, (w + 1) // 2
    planes = [_device_plane(y, "y", n_slots, h, w, False, dev)]
    if nv12:
        planes += [_device_plane(out[1], "uv", n_slots, ch, cw, True, dev), _lib.DevicePlane(None, 0, 0)]
    else:
        planes += [_device_plane(out[1], "cb", n_slots, ch, cw, False, dev), _device_plane(out[2], "cr", n_slots, ch, cw, False, dev)]
    stream = torch.cuda.current_stream(dev).cuda_stream
    target = _lib.DeviceYuv((_lib.DevicePlane * 3)(*planes), w, h, _YUV_LAYOUTS[layout], 0, stream or None)
    return out, target


def _device_tensor(out, n_slots, size, dtype, mean, std, device):
    """The h263cu_device_tensor of a CUDA tensor [>= n_slots, 3, H, W] on `device` of dtype torch.uint8, float32,
    float16 or bfloat16, size = (H, W).  Any positive strides: contiguous, channels_last and padded or sliced views all
    pass.  out=None allocates a contiguous [n_slots, 3, H, W] tensor of `dtype` (None: float16).  mean / std (three
    values each, on the 0-1 scale as torchvision takes them) become mul = 1 / (255 * std) and add = -mean / std, computed
    in float64 and rounded once to float32; without either the values stay on the 0-255 scale.  Raises ValueError when
    an argument breaks a rule of the C ABI (include/h263cu.h), so that nothing is parsed.  The consumer stream is
    torch's current stream on the device."""
    import torch

    codes = {torch.uint8: _lib.TENSOR_U8, torch.float32: _lib.TENSOR_F32, torch.float16: _lib.TENSOR_F16,
             torch.bfloat16: _lib.TENSOR_BF16}
    dev = torch.device("cuda", device)
    try:
        h, w = (int(v) for v in size)
    except (TypeError, ValueError):
        raise ValueError("size must be (H, W), not %r" % (size,)) from None
    if not (1 <= h <= 16384 and 1 <= w <= 16384):
        raise ValueError("size must lie in 1..16384 on both axes, not %r" % ((h, w),))
    if dtype is not None and dtype not in codes:
        raise ValueError("dtype must be one of torch.uint8, float32, float16, bfloat16, not %s" % (dtype,))
    if out is None:
        out = torch.empty((n_slots, 3, h, w), dtype=dtype or torch.float16, device=dev)
    if not isinstance(out, torch.Tensor) or out.dtype not in codes or out.device != dev:
        raise ValueError("out must be a torch.uint8, float32, float16 or bfloat16 tensor on %s" % dev)
    if dtype is not None and out.dtype != dtype:
        raise ValueError("out is %s, not the dtype asked for (%s)" % (out.dtype, dtype))
    if out.dim() != 4 or out.shape[0] < n_slots or tuple(out.shape[1:]) != (3, h, w):
        raise ValueError("out must have the shape [>= %d, 3, %d, %d], not %s" % (n_slots, h, w, tuple(out.shape)))
    code = codes[out.dtype]
    if code == _lib.TENSOR_U8 and (mean is not None or std is not None):
        raise ValueError("mean / std need a float dtype: uint8 output holds the rounded RGB values")
    # a dimension of size 1 has no stride of its own: any positive one addresses it the same
    strides = [st if n > 1 else max(st, 1) for st, n in zip(out.stride(), out.shape)]
    if min(strides) <= 0:
        raise ValueError("out must have positive strides, not %s" % (out.stride(),))
    es = out.element_size()
    base = out.data_ptr()
    extent = ((w - 1) * strides[3] + (h - 1) * strides[2] + 2 * strides[1] + 1) * es
    if base % es or extent >= 1 << 40:
        raise ValueError("out: base must be aligned to the element size and a slot must span less than 2^40 bytes")
    mul, add = [1.0] * 3, [0.0] * 3
    if mean is not None or std is not None:
        m = [0.0] * 3 if mean is None else [float(v) for v in mean]
        sd = [1.0] * 3 if std is None else [float(v) for v in std]
        if len(m) != 3 or len(sd) != 3 or any(v == 0 for v in sd):
            raise ValueError("mean and std must hold three values each, std non-zero")
        mul = np.array([1.0 / (255.0 * v) for v in sd], np.float64).astype(np.float32)
        add = np.array([-a / b for a, b in zip(m, sd)], np.float64).astype(np.float32)
        if not (np.isfinite(mul).all() and np.isfinite(add).all()):
            raise ValueError("mean / std give a non-finite scale or offset")
        mul, add = [float(v) for v in mul], [float(v) for v in add]
    stream = torch.cuda.current_stream(dev).cuda_stream
    target = _lib.DeviceTensor(base, (C.c_int64 * 4)(*strides), w, h, code, 0, (C.c_float * 3)(*mul), (C.c_float * 3)(*add),
                               stream or None)
    return out, target


_FITS = {"stretch": _lib.FIT_STRETCH, "letterbox": _lib.FIT_LETTERBOX, "center_crop": _lib.FIT_CENTER_CROP}


def _tensor_fit(fit, short_side, fill, crops, n, always=False):
    """The h263cu_tensor_fit of the fit keywords of decode_step_device_tensor for n inputs, or None for the plain
    stretch of whole pictures (h263cu_decode_step_device_tensor, whatever the fill: nothing lies outside the picture)
    unless `always`.
    fit: "stretch", "letterbox" or "center_crop"; short_side: the resize of center_crop (1..16384), None otherwise;
    fill: one number or three, on the 0-255 scale; crops: None or [n, 4] boxes (x, y, w, h), one per input.  Raises
    ValueError for what the C ABI refuses, so that nothing is parsed.  The crop array stays alive as fit._crops."""
    if fit not in _FITS:
        raise ValueError("fit must be one of %s, not %r" % (sorted(_FITS), fit))
    if fit == "center_crop":
        if short_side is None or isinstance(short_side, bool) or int(short_side) != short_side or not 1 <= short_side <= 16384:
            raise ValueError("center_crop needs short_side, an integer in 1..16384, not %r" % (short_side,))
    elif short_side is not None:
        raise ValueError("short_side belongs to fit='center_crop' only")
    fill3 = np.asarray(fill, np.float64).reshape(-1)
    if fill3.size == 1:
        fill3 = np.repeat(fill3, 3)
    if fill3.size != 3 or not (np.isfinite(fill3).all() and (fill3 >= 0).all() and (fill3 <= 255).all()):
        raise ValueError("fill must be one number or three, finite, in 0..255, not %r" % (fill,))
    boxes = None
    if crops is not None:
        boxes = np.asarray(crops)
        if boxes.shape != (n, 4) or not (np.issubdtype(boxes.dtype, np.integer) or boxes.size == 0):
            raise ValueError("crops must be [%d, 4] integers (x, y, w, h), not %s of %s" % (n, boxes.shape, boxes.dtype))
        b = boxes.astype(np.int64)
        if (b < 0).any() or (b[:, 2:] == 0).any() or (b[:, :2] + b[:, 2:] >= 1 << 32).any():
            raise ValueError("crops: x, y >= 0, w, h > 0 and x + w, y + h < 2^32")
        boxes = np.ascontiguousarray(b, np.uint32)
    if fit == "stretch" and boxes is None and not always:
        return None
    f = _lib.TensorFit(_FITS[fit], int(short_side or 0), (C.c_float * 3)(*[float(v) for v in fill3]), 0,
                       None if boxes is None else boxes.ctypes.data_as(C.POINTER(_lib.TensorCrop)))
    f._crops = boxes
    return f


_FILTERS = {"bilinear": _lib.FILTER_BILINEAR_AA, "bicubic": _lib.FILTER_BICUBIC_AA}


def _tensor_filter(antialias, interpolation):
    """The H263CU_FILTER_* of decode_step_device_tensor's antialias / interpolation (torchvision's vocabulary: a string
    or an InterpolationMode), or None for the antialias=False bilinear of the plain and fit calls.  Raises ValueError
    for what is not offered, so that nothing is parsed: plain (antialias=False) bicubic is torch's a = -0.75 with
    clamped indices, a different function."""
    mode = getattr(interpolation, "value", interpolation)
    if mode not in _FILTERS:
        raise ValueError("interpolation must be 'bilinear' or 'bicubic', not %r" % (interpolation,))
    if not isinstance(antialias, (bool, np.bool_)):
        raise ValueError("antialias must be True or False, not %r" % (antialias,))
    if not antialias:
        if mode == "bicubic":
            raise ValueError("interpolation='bicubic' needs antialias=True: plain bicubic resizing is not offered")
        return None
    return _FILTERS[mode]


_PARSE = {"host": 0, "device": _lib.PARSE_ON_DEVICE}


def _parse_flag(parse):
    """The out_flags bit of decode_step*'s parse keyword: "host" (the threaded host parser) or "device" (the macroblock
    layer on the GPU, H263CU_PARSE_ON_DEVICE).  Anything else raises ValueError before any parser moves."""
    if not isinstance(parse, str) or parse not in _PARSE:
        raise ValueError("parse must be 'host' or 'device', not %r" % (parse,))
    return _PARSE[parse]


class DecodedPicture:
    """Mirror of h263::DecodedPicture: header fields + tight row-major u8 planes."""

    def __init__(self, width, height, picture_type, quantizer, temporal_reference, y, cb, cr):
        self.width, self.height = width, height
        self.picture_type = picture_type
        self.quantizer = quantizer
        self.temporal_reference = temporal_reference
        self._y, self._cb, self._cr = y, cb, cr

    def as_yuv(self):
        return self._y, self._cb, self._cr

    def as_luma(self):
        return self._y

    def as_chroma_b(self):
        return self._cb

    def as_chroma_r(self):
        return self._cr

    def format(self):
        """The picture's dimensions (DecodedPicture::format, picture.rs:60-66) as (width, height)."""
        return self.width, self.height

    def as_header(self):
        """The header fields the reference keeps with a decoded picture (DecodedPicture::as_header)."""
        return {"width": self.width, "height": self.height, "picture_type": self.picture_type,
                "quantizer": self.quantizer, "temporal_reference": self.temporal_reference}

    def luma_samples_per_row(self):
        return self.width

    def chroma_samples_per_row(self):
        return (self.width + 1) // 2


class Context:
    """Thin RAII wrapper of h263cu_ctx."""

    def __init__(self, device, max_streams, max_width, max_height, _borrowed=None):
        self.L = _lib.lib()
        self._owned = _borrowed is None
        if _borrowed is None:
            err = C.c_int(0)
            self.h = self.L.h263cu_create(device, max_streams, max_width, max_height, 0, C.byref(err))
            if not self.h:
                raise H263Error(err.value)
        else:
            self.h = _borrowed  # a context that belongs to a DeviceGroup
        self.device = device
        self.max_streams, self.max_width, self.max_height = max_streams, max_width, max_height

    def close(self):
        if getattr(self, "h", None):
            if self._owned:
                self.L.h263cu_destroy(self.h)
            self.h = None

    def readback_wait(self, age=0):
        check(self.L.h263cu_readback_wait(self.h, age))

    def __del__(self):
        self.close()

    def submit_step(self, pics, mbs, events, out_flags):
        check(self.L.h263cu_submit_step(self.h, pics.ctypes.data, len(pics), mbs.ctypes.data, len(mbs),
                                        events.ctypes.data if len(events) else None, len(events), out_flags))

    def step_upload(self, pics, mbs, events):
        err = C.c_int(0)
        s = self.L.h263cu_step_upload(self.h, pics.ctypes.data, len(pics), mbs.ctypes.data, len(mbs),
                                      events.ctypes.data if len(events) else None, len(events), C.byref(err))
        if not s:
            raise H263Error(err.value)
        return s

    def step_run(self, step, out_flags):
        check(self.L.h263cu_step_run(self.h, step, out_flags))

    def step_free(self, step):
        self.L.h263cu_step_free(self.h, step)

    def graph_build(self, steps, out_flags):
        """n resident steps as one CUDA graph (h263cu_graph_build); the steps must outlive it."""
        arr = (C.c_void_p * len(steps))(*steps)
        err = C.c_int(0)
        g = self.L.h263cu_graph_build(self.h, arr, len(steps), out_flags, C.byref(err))
        if not g:
            raise H263Error(err.value)
        return g

    def graph_launch(self, graph):
        check(self.L.h263cu_graph_launch(self.h, graph))

    def graph_free(self, graph):
        self.L.h263cu_graph_free(self.h, graph)

    def sync(self):
        check(self.L.h263cu_sync(self.h))

    def stream_info(self, stream):
        v = [C.c_uint32() for _ in range(5)]
        check(self.L.h263cu_stream_info(self.h, stream, *[C.byref(x) for x in v]))
        return dict(zip(("width", "height", "pic_type", "pquant", "tr"), [x.value for x in v]))

    def read_yuv(self, stream):
        i = self.stream_info(stream)
        w, h = i["width"], i["height"]
        cw, ch = (w + 1) // 2, (h + 1) // 2
        y = np.empty(w * h, np.uint8)
        cb = np.empty(cw * ch, np.uint8)
        cr = np.empty(cw * ch, np.uint8)
        check(self.L.h263cu_read_yuv(self.h, stream, y.ctypes.data, cb.ctypes.data, cr.ctypes.data))
        return y, cb, cr

    def read_rgba(self, stream):
        i = self.stream_info(stream)
        out = np.empty(i["width"] * i["height"] * 4, np.uint8)
        check(self.L.h263cu_read_rgba(self.h, stream, out.ctypes.data))
        return out

    def checksums(self, streams):
        s = np.ascontiguousarray(streams, np.uint32)
        out = np.zeros((len(s), 4), np.uint64)
        check(self.L.h263cu_checksums(self.h, s.ctypes.data, len(s), out.ctypes.data))
        return out

    def timer_start(self):
        check(self.L.h263cu_timer_start(self.h))

    def timer_stop(self):
        ms = C.c_float()
        check(self.L.h263cu_timer_stop(self.h, C.byref(ms)))
        return ms.value

    def launch_count(self):
        return int(self.L.h263cu_launch_count(self.h))

    def tiled_launch_count(self):
        return int(self.L.h263cu_tiled_launch_count(self.h))

    def profile_enable(self, on=True):
        check(self.L.h263cu_profile_enable(self.h, int(on)))

    def profile_read(self):
        ms = (C.c_double * 2)()
        n = (C.c_uint64 * 2)()
        check(self.L.h263cu_profile_read(self.h, ms, n))
        return dict(recon_ms=ms[0], recon_launches=int(n[0]), deblock_ms=ms[1], deblock_launches=int(n[1]))


class H263State:
    """Mirror of h263::H263State for ONE stream: host parse + GPU reconstruction.

    `decode_next_picture(packet)` takes the bytes of one picture (the reference reads them
    through `H263Reader::from_source(&packet[..])`; Sorenson pictures end at EOF, so one
    reader per packet is the only usable form, SURVEY.md T5)."""

    def __init__(self, decoder_options=SORENSON_SPARK_BITSTREAM, device=0, deblock=False, pipelined=False):
        """pipelined=True: decode_next_picture returns as soon as the picture is queued (parse done, upload + kernels +
        RGBA read-back in flight); get_last_rgba / get_last_picture wait for it.  A caller that hands in packet t + 1
        before it consumes picture t overlaps the host parse with the device work (two pinned RGBA buffers alternate)."""
        self.decoder_options = decoder_options
        self.device = device
        self.pipelined = pipelined
        self._ring, self._ring_size, self._ring_pos, self._pending = [None, None], 0, 0, False
        self._last_dims = (0, 0)
        self._views, self._views_size = [None, None], -1
        self.parser = frontend.Parser(decoder_options)
        self.ctx = None
        self.out_flags = _lib.OUT_RGBA | (_lib.OUT_DEBLOCK if deblock else 0)
        self._has_picture = False
        # the one-element argument arrays of h263cu_decode_step; the pinned RGBA ring is self._ring
        self._rgba_view = None
        self._one_parser = (C.c_void_p * 1)(self.parser.h)
        self._one_packet = (C.c_void_p * 1)()
        self._one_len = (C.c_size_t * 1)()
        self._one_id = np.zeros(1, np.uint32)
        self._one_err = np.zeros(1, np.int32)

    def is_sorenson(self):
        return bool(self.decoder_options & SORENSON_SPARK_BITSTREAM)

    def decode_next_picture(self, packet, _force_new_ctx=False):
        """One call into h263cu_decode_step for the one stream: parse into the context's pinned staging, upload,
        reconstruction and the RGBA read-back into this state's pinned buffer, then wait.  Transactional like the
        reference (state.rs:120-137): a packet that fails to parse raises and leaves parser and stream untouched."""
        data = packet if isinstance(packet, bytes) else bytes(packet)
        buf = np.frombuffer(data, np.uint8)
        # A picture larger than the context needs a bigger one.  It replaces the old context only once the packet has
        # decoded (a size change can only succeed on an I picture, which needs no reference planes): a packet that
        # fails leaves parser, context and last picture as they were (state.rs:120-137).  With a context in place the
        # header is not peeked first: decode_step reports a picture that does not fit (H263CU_ERR_CAPACITY) and the
        # call is repeated with a larger context.
        ctx = self.ctx
        if ctx is not None and not _force_new_ctx:
            w, h = self._last_dims
        else:
            hdr = frontend.peek_picture(data, self.decoder_options)
            w, h = int(hdr["width"]), int(hdr["height"])
            if w == 0 or h == 0:
                w = h = 16  # no usable size in the header: the parse inside decode_step reports the reference's error
            if ctx is None or w > ctx.max_width or h > ctx.max_height:
                ctx = Context(self.device, 1, max(w, 16), max(h, 16))
        L = _lib.lib()
        size = w * h * 4
        if size > self._ring_size:
            # both pinned buffers grow together; nothing may still be copying into the old ones
            if self.ctx is not None:
                self.ctx.sync()
            for k in range(2):
                if self._ring[k]:
                    L.h263cu_free_pinned(self._ring[k])
                self._ring[k] = L.h263cu_alloc_pinned(size)
                if not self._ring[k]:
                    self._ring_size = 0
                    raise MemoryError
            self._ring_size = size
            self._views_size = -1
        pos = self._ring_pos ^ 1  # the buffer that does not hold the last picture
        nd = C.c_uint32(0)
        self._one_packet[0], self._one_len[0], self._one_err[0] = buf.ctypes.data, buf.size, 0
        _lib.check(L.h263cu_decode_step(ctx.h, self._one_parser, self._one_packet, self._one_len, self._one_id.ctypes.data, 1, 1,
                                        self.out_flags, self._ring[pos], 0, self._one_err.ctypes.data, C.byref(nd)))
        if self._one_err[0]:
            if self._one_err[0] == _lib.ERR_CAPACITY and not _force_new_ctx:
                return self.decode_next_picture(data, _force_new_ctx=True)  # larger than the context: peek and grow
            raise _lib.H263Error(int(self._one_err[0]))
        d = L.h263cu_stream_dims(ctx.h, 0)  # the size the parser found (it may differ from the previous picture's)
        if d != (w << 16 | h):
            w, h = d >> 16, d & 0xFFFF
            size = w * h * 4
            assert size <= self._ring_size  # a picture that fits the context fits the buffers made with it
        self._last_dims = (w, h)
        if ctx is not self.ctx and self.ctx is not None:
            self.ctx.sync()  # the old context may still be copying the previous picture back
        self.ctx = ctx
        self._ring_pos = pos
        if self._views_size != size:  # numpy views of the two pinned buffers, made once per picture size
            self._views = [np.ctypeslib.as_array(C.cast(self._ring[k], C.POINTER(C.c_uint8)), shape=(size,)) for k in range(2)]
            self._views_size = size
        self._rgba_view = self._views[pos]
        self._has_picture = True
        self._pending = True
        if not self.pipelined:
            self._wait()

    def _wait(self):
        """Wait for the picture queued last: its planes are reconstructed and its RGBA has arrived in host memory."""
        if self._pending:
            self.ctx.readback_wait(0)
            self._pending = False

    def __del__(self):
        try:
            if getattr(self, "ctx", None) is not None:
                self.ctx.sync()
            for k in range(2):
                if self._ring[k]:
                    _lib.lib().h263cu_free_pinned(self._ring[k])
                    self._ring[k] = None
        except Exception:
            pass

    def get_last_picture(self):
        if not self._has_picture:
            return None
        self._wait()
        i = self.ctx.stream_info(0)
        y, cb, cr = self.ctx.read_yuv(0)
        return DecodedPicture(i["width"], i["height"], i["pic_type"], i["pquant"], i["tr"], y, cb, cr)

    def get_reference_picture(self):
        """state.rs:72-78.  The reference picture is the last non-disposable picture; disposable
        pictures do not decode in the reference (macroblock.rs:461-465), so it is the last picture."""
        return self.get_last_picture()

    def parse_picture(self, packet):
        """Header-only peek (H263State::parse_picture, state.rs:102-111): no decoder state changes."""
        return frontend.peek_picture(bytes(packet), self.decoder_options)

    def cleanup_buffers(self):
        """state.rs:81-98 drops every picture except the last and the reference one.  The device context
        never holds more than those two plane slots per stream, so there is nothing to free."""
        return None

    def get_last_rgba(self, copy=True):
        """RGBA of the last picture (fused yuv420_to_rgba, or deblock + yuv420_to_rgba).  copy=False returns a view of
        the pinned read-back buffer, valid until the picture after next is queued (two buffers alternate)."""
        if not self._has_picture:
            return None
        self._wait()
        return self._rgba_view.copy() if copy else self._rgba_view


class BatchDecoder:
    """n independent streams decoded in lock step: one picture per stream per step."""

    def __init__(self, n_streams, max_width, max_height, decoder_options=SORENSON_SPARK_BITSTREAM, device=0,
                 threads=0, ctx=None):
        self.n = n_streams
        self.parsers = [frontend.Parser(decoder_options) for _ in range(n_streams)]
        self.ctx = ctx if ctx is not None else Context(device, n_streams, max_width, max_height)
        self.threads = threads

    def parse_step(self, packets, stream_ids=None):
        ids = np.arange(self.n, dtype=np.uint32) if stream_ids is None else np.asarray(stream_ids, np.uint32)
        parsers = [self.parsers[int(s)] for s in ids]
        return frontend.parse_step(parsers, packets, ids, self.threads)

    def decode_step(self, packets, out_flags=_lib.OUT_RGBA, stream_ids=None, host_rgba=None, rgba_stride=0, parse="host"):
        """One decode_next_picture per stream through h263cu_decode_step: threaded parse into the
        context's pinned staging, asynchronous upload + reconstruction (+ RGBA read-back into the
        pinned buffer `host_rgba` when given).  Returns the per-picture error codes.

        parse="device" parses the macroblock layer on the GPU (H263CU_PARSE_ON_DEVICE): the same results, with the
        host left the picture headers; the call then waits for the parse kernel's per-picture results.  Every
        decode_step* method takes it."""
        flags = _parse_flag(parse)
        plan = self.plan_step(packets, stream_ids)
        return self.decode_planned(plan, out_flags | flags, host_rgba, rgba_stride)

    def plan_step(self, packets, stream_ids=None):
        """The pointer arrays h263cu_decode_step takes, built once for a list of packets (bytes or
        uint8 arrays, kept alive by the plan)."""
        n = len(packets)
        ids = np.arange(self.n, dtype=np.uint32)[:n] if stream_ids is None else np.ascontiguousarray(stream_ids, np.uint32)
        bufs = [np.frombuffer(pk, np.uint8) if not isinstance(pk, np.ndarray) else pk for pk in packets]
        return {
            "n": n, "bufs": bufs, "ids": ids,
            # an id beyond the decoder's streams is passed on as it is: the library refuses the step
            "parsers": (C.c_void_p * n)(*[self.parsers[min(int(s), self.n - 1)].h for s in ids]),
            "packets": (C.c_void_p * n)(*[b.ctypes.data for b in bufs]),
            "lens": (C.c_size_t * n)(*[b.size for b in bufs]),
            "errs": np.zeros(n, np.int32),
        }

    def decode_step_device(self, packets, out=None, out_flags=_lib.OUT_RGBA, stream_ids=None, parse="host"):
        """One decode_next_picture per stream with the RGBA left on the GPU (h263cu_decode_step_device): the picture of
        packet i goes to out[i], a torch.uint8 CUDA tensor [n, H, W, 4] on the context's device (a view with padded rows
        and slots is fine).  out=None allocates [n, max_h, round_up(max_w, 4), 4] and returns its [..., :max_w, :] view.
        The work is ordered on torch's current stream: what the caller queues there afterwards sees the pictures, with no
        host synchronisation.  Returns (out, per-picture error codes)."""
        flags = _parse_flag(parse)
        out, target = _device_rgba(out, len(packets), self.ctx.max_width, self.ctx.max_height, self.ctx.device)
        plan = self.plan_step(packets, stream_ids)
        nd = C.c_uint32(0)
        _lib.check(_lib.lib().h263cu_decode_step_device(
            self.ctx.h, plan["parsers"], plan["packets"], plan["lens"], plan["ids"].ctypes.data, plan["n"], self.threads,
            out_flags | flags, C.byref(target), plan["errs"].ctypes.data, C.byref(nd)))
        return out, plan["errs"]

    def decode_step_device_yuv(self, packets, out=None, layout="i420", deblock=False, stream_ids=None, parse="host"):
        """One decode_next_picture per stream with the decoded planes left on the GPU (h263cu_decode_step_device_yuv):
        the planes of packet i go to slot i of the tensors of `out`, torch.uint8 CUDA tensors on the context's device
        (views with padded rows and slots are fine): (y [n, H, W], cb [n, ch, cw], cr [n, ch, cw]) for layout "i420",
        (y [n, H, W], uv [n, ch, cw, 2]) for "nv12", ch = ceil(H / 2), cw = ceil(W / 2).  out=None allocates them for
        max_w x max_h with rows padded to multiples of 4 bytes and returns [..., :W] views.  deblock=True writes the
        deblocked planes.  No RGBA is produced.  The work is ordered on torch's current stream, with no host
        synchronisation.  Returns (planes, per-picture error codes)."""
        flags = _parse_flag(parse)
        out, target = _device_yuv(out, len(packets), self.ctx.max_width, self.ctx.max_height, self.ctx.device, layout)
        plan = self.plan_step(packets, stream_ids)
        nd = C.c_uint32(0)
        _lib.check(_lib.lib().h263cu_decode_step_device_yuv(
            self.ctx.h, plan["parsers"], plan["packets"], plan["lens"], plan["ids"].ctypes.data, plan["n"], self.threads,
            (_lib.OUT_DEBLOCK if deblock else 0) | flags, C.byref(target), plan["errs"].ctypes.data, C.byref(nd)))
        return out, plan["errs"]

    def decode_step_device_tensor(self, packets, size, out=None, dtype=None, mean=None, std=None, deblock=False, stream_ids=None,
                                  fit="stretch", short_side=None, fill=0, crops=None, antialias=False, interpolation="bilinear",
                                  parse="host"):
        """One decode_next_picture per stream with each picture bilinearly resized (torch's align_corners=False rule)
        to size = (H, W) and converted to normalised RGB on the GPU (h263cu_decode_step_device_tensor): packet i goes to
        out[i], a [>= n, 3, H, W] CUDA tensor on the context's device of torch.uint8, float32, float16 or bfloat16 with
        any positive strides (contiguous and channels_last both work).  out=None allocates a contiguous one of `dtype`
        (None: float16).  mean / std (0-1 scale, as torchvision takes them) normalise the float dtypes; without them the
        values are on the 0-255 scale.  deblock=True resamples the deblocked planes.  The work is ordered on torch's
        current stream, with no host synchronisation.  Returns (out, per-picture error codes).

        fit places each picture (h263cu_decode_step_device_tensor_fit): "stretch" (the default) resizes it to (H, W);
        "letterbox" keeps its aspect, fits it whole, centres it and sets the rest to `fill`; "center_crop" is
        torchvision's Resize(short_side, antialias=False) + CenterCrop((H, W)).  fill is one value or three on the 0-255
        scale (normalised like a pixel).  crops ([n, 4] of (x, y, w, h), one per packet) resizes that box of each picture
        instead of the whole: a box that does not fit its picture (h263_rs_b200.frontend.peek_picture gives the size) is
        that picture's H263CU_ERR_BAD_ARGUMENT, its stream untouched.

        antialias / interpolation choose the resize filter in torchvision's vocabulary
        (h263cu_decode_step_device_tensor_filter): antialias=True is torch's antialiased bilinear (torchvision Resize's
        default on tensors), with interpolation="bicubic" its antialiased bicubic (a = -0.5); bicubic without antialias
        is not offered.  Under every fit, "center_crop" with antialias=True is Resize(short_side) + CenterCrop."""
        flags = _parse_flag(parse)
        filt = _tensor_filter(antialias, interpolation)
        f = _tensor_fit(fit, short_side, fill, crops, len(packets), always=filt is not None)
        out, target = _device_tensor(out, len(packets), size, dtype, mean, std, self.ctx.device)
        plan = self.plan_step(packets, stream_ids)
        nd = C.c_uint32(0)
        L = _lib.lib()
        args = (self.ctx.h, plan["parsers"], plan["packets"], plan["lens"], plan["ids"].ctypes.data, plan["n"], self.threads,
                (_lib.OUT_DEBLOCK if deblock else 0) | flags, C.byref(target))
        if filt is not None:
            _lib.check(L.h263cu_decode_step_device_tensor_filter(*args, C.byref(f), filt, plan["errs"].ctypes.data, C.byref(nd)))
        elif f is None:
            _lib.check(L.h263cu_decode_step_device_tensor(*args, plan["errs"].ctypes.data, C.byref(nd)))
        else:
            _lib.check(L.h263cu_decode_step_device_tensor_fit(*args, C.byref(f), plan["errs"].ctypes.data, C.byref(nd)))
        return out, plan["errs"]

    def decode_planned(self, plan, out_flags=_lib.OUT_RGBA, host_rgba=None, rgba_stride=0):
        nd = C.c_uint32(0)
        _lib.check(_lib.lib().h263cu_decode_step(
            self.ctx.h, plan["parsers"], plan["packets"], plan["lens"], plan["ids"].ctypes.data, plan["n"], self.threads,
            out_flags, host_rgba, rgba_stride, plan["errs"].ctypes.data, C.byref(nd)))
        return plan["errs"]


class DeviceGroup:
    """Several GPUs driven from ONE process: one context per device, one shared pool of parser threads
    (h263cu_group_*, SURVEY.md 8e).  Global stream s lives on device s % n_devices, slot s // n_devices; with a host
    buffer the RGBA of stream s lands at index (s % n_devices) * streams_per_device + s // n_devices."""

    def __init__(self, devices, streams_per_device, max_width, max_height, decoder_options=SORENSON_SPARK_BITSTREAM, threads=0):
        self.L = _lib.lib()
        self.devices = list(devices)
        self.streams_per_device = streams_per_device
        dv = (C.c_int * len(self.devices))(*self.devices)
        err = C.c_int(0)
        self.h = self.L.h263cu_group_create(dv, len(self.devices), streams_per_device, max_width, max_height, threads, C.byref(err))
        if not self.h:
            raise H263Error(err.value)
        self.n = streams_per_device * len(self.devices)
        self.parsers = [frontend.Parser(decoder_options) for _ in range(self.n)]
        self.ctxs = [Context(d, streams_per_device, max_width, max_height, _borrowed=self.L.h263cu_group_ctx(self.h, k))
                     for k, d in enumerate(self.devices)]

    def close(self):
        if getattr(self, "h", None):
            for c in self.ctxs:
                c.close()
            self.L.h263cu_group_destroy(self.h)
            self.h = None

    def __del__(self):
        self.close()

    def position(self, stream):
        """Index of a global stream's picture in the host RGBA buffer (device-major)."""
        nd = len(self.devices)
        return (stream % nd) * self.streams_per_device + stream // nd

    def where(self, stream):
        """(context, local slot) of a global stream."""
        nd = len(self.devices)
        return self.ctxs[stream % nd], stream // nd

    def plan_step(self, packets, stream_ids=None):
        n = len(packets)
        ids = np.arange(n, dtype=np.uint32) if stream_ids is None else np.ascontiguousarray(stream_ids, np.uint32)
        bufs = [np.frombuffer(pk, np.uint8) if not isinstance(pk, np.ndarray) else pk for pk in packets]
        return {
            "n": n, "bufs": bufs, "ids": ids,
            "parsers": (C.c_void_p * n)(*[self.parsers[min(int(s), self.n - 1)].h for s in ids]),
            "packets": (C.c_void_p * n)(*[b.ctypes.data for b in bufs]),
            "lens": (C.c_size_t * n)(*[b.size for b in bufs]),
            "errs": np.zeros(n, np.int32),
        }

    def decode_planned(self, plan, out_flags=_lib.OUT_RGBA, host_rgba=None, rgba_stride=0):
        nd = C.c_uint32(0)
        _lib.check(self.L.h263cu_group_decode_step(self.h, plan["parsers"], plan["packets"], plan["lens"], plan["ids"].ctypes.data,
                                                   plan["n"], out_flags, host_rgba, rgba_stride, plan["errs"].ctypes.data, C.byref(nd)))
        return plan["errs"]

    def decode_step(self, packets, out_flags=_lib.OUT_RGBA, stream_ids=None, host_rgba=None, rgba_stride=0, parse="host"):
        """parse: "host" or "device", as BatchDecoder.decode_step's (every decode_step* method takes it)."""
        flags = _parse_flag(parse)
        return self.decode_planned(self.plan_step(packets, stream_ids), out_flags | flags, host_rgba, rgba_stride)

    def decode_step_device(self, packets, outs=None, out_flags=_lib.OUT_RGBA, stream_ids=None, parse="host"):
        """decode_step with the RGBA left on the GPUs (h263cu_group_decode_step_device): global stream s goes to slot
        s // n_devices of outs[s % n_devices], one torch.uint8 tensor [slots, H, W, 4] per device (see
        BatchDecoder.decode_step_device; None allocates streams_per_device slots on each).  Returns (outs, errors)."""
        flags = _parse_flag(parse)
        nd = len(self.devices)
        plan = self.plan_step(packets, stream_ids)
        need = [0] * nd
        for s in plan["ids"]:
            need[int(s) % nd] = max(need[int(s) % nd], int(s) // nd + 1)
        c0 = self.ctxs[0]
        pairs = [_device_rgba(None if outs is None else outs[k], need[k] if outs is not None else self.streams_per_device,
                              c0.max_width, c0.max_height, d) for k, d in enumerate(self.devices)]
        targets = (_lib.DeviceRgba * nd)(*[t for _, t in pairs])
        n_dec = C.c_uint32(0)
        _lib.check(self.L.h263cu_group_decode_step_device(self.h, plan["parsers"], plan["packets"], plan["lens"], plan["ids"].ctypes.data,
                                                          plan["n"], out_flags | flags, targets, plan["errs"].ctypes.data, C.byref(n_dec)))
        return [o for o, _ in pairs], plan["errs"]

    def decode_step_device_yuv(self, packets, outs=None, layout="i420", deblock=False, stream_ids=None, parse="host"):
        """decode_step with the decoded planes left on the GPUs (h263cu_group_decode_step_device_yuv): global stream s
        goes to slot s // n_devices of outs[s % n_devices], one tuple of plane tensors per device (see
        BatchDecoder.decode_step_device_yuv; None allocates streams_per_device slots on each).  Returns (outs, errors)."""
        flags = _parse_flag(parse)
        nd = len(self.devices)
        plan = self.plan_step(packets, stream_ids)
        need = [0] * nd
        for s in plan["ids"]:
            need[int(s) % nd] = max(need[int(s) % nd], int(s) // nd + 1)
        c0 = self.ctxs[0]
        pairs = [_device_yuv(None if outs is None else outs[k], need[k] if outs is not None else self.streams_per_device,
                             c0.max_width, c0.max_height, d, layout) for k, d in enumerate(self.devices)]
        targets = (_lib.DeviceYuv * nd)(*[t for _, t in pairs])
        n_dec = C.c_uint32(0)
        _lib.check(self.L.h263cu_group_decode_step_device_yuv(
            self.h, plan["parsers"], plan["packets"], plan["lens"], plan["ids"].ctypes.data, plan["n"],
            (_lib.OUT_DEBLOCK if deblock else 0) | flags, targets, plan["errs"].ctypes.data, C.byref(n_dec)))
        return [o for o, _ in pairs], plan["errs"]

    def decode_step_device_tensor(self, packets, size, outs=None, dtype=None, mean=None, std=None, deblock=False, stream_ids=None,
                                  fit="stretch", short_side=None, fill=0, crops=None, antialias=False, interpolation="bilinear",
                                  parse="host"):
        """decode_step with each picture resized and converted on the GPUs (h263cu_group_decode_step_device_tensor):
        global stream s goes to slot s // n_devices of outs[s % n_devices], one tensor per device (see
        BatchDecoder.decode_step_device_tensor; None allocates streams_per_device slots on each).  fit / short_side /
        fill / crops / antialias / interpolation as there; crops[i] belongs to packets[i].  Returns (outs, errors)."""
        flags = _parse_flag(parse)
        filt = _tensor_filter(antialias, interpolation)
        f = _tensor_fit(fit, short_side, fill, crops, len(packets), always=filt is not None)
        nd = len(self.devices)
        plan = self.plan_step(packets, stream_ids)
        need = [0] * nd
        for s in plan["ids"]:
            need[int(s) % nd] = max(need[int(s) % nd], int(s) // nd + 1)
        pairs = [_device_tensor(None if outs is None else outs[k], need[k] if outs is not None else self.streams_per_device,
                                size, dtype, mean, std, d) for k, d in enumerate(self.devices)]
        targets = (_lib.DeviceTensor * nd)(*[t for _, t in pairs])
        n_dec = C.c_uint32(0)
        args = (self.h, plan["parsers"], plan["packets"], plan["lens"], plan["ids"].ctypes.data, plan["n"],
                (_lib.OUT_DEBLOCK if deblock else 0) | flags, targets)
        if filt is not None:
            _lib.check(self.L.h263cu_group_decode_step_device_tensor_filter(*args, C.byref(f), filt, plan["errs"].ctypes.data,
                                                                            C.byref(n_dec)))
        elif f is None:
            _lib.check(self.L.h263cu_group_decode_step_device_tensor(*args, plan["errs"].ctypes.data, C.byref(n_dec)))
        else:
            _lib.check(self.L.h263cu_group_decode_step_device_tensor_fit(*args, C.byref(f), plan["errs"].ctypes.data, C.byref(n_dec)))
        return [o for o, _ in pairs], plan["errs"]

    def sync(self):
        check(self.L.h263cu_group_sync(self.h))
