"""ctypes loader for libh263cu.so (the C ABI declared in include/h263cu.h).

The library is built in-tree by `__graft_entry__.build()` / `h263_rs_b200.build`.
There is no CPU fallback: a missing library raises, and device entry points return
H263CU_ERR_NO_DEVICE / H263CU_ERR_CUDA without a GPU.
"""
import ctypes as C
import os

HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("H263CU_LIB", os.path.join(HERE, "libh263cu.so"))

OK = 0
ERR_INVALID_BITSTREAM = -12
ERR_UNHANDLED_IO_ERROR = -16
ERR_BAD_ARGUMENT = -100
ERR_CUDA = -101
ERR_NO_DEVICE = -102
ERR_CAPACITY = -103
ERR_REFERENCE_WOULD_ABORT = -104
ERR_NO_PICTURE = -105

OPT_SORENSON = 1
OUT_RGBA = 1
OUT_DEBLOCK = 2
PARSE_ON_DEVICE = 4  # H263CU_PARSE_ON_DEVICE: the macroblock layer is parsed on the GPU

PIC_I, PIC_P, PIC_DISPOSABLE_P, PIC_OTHER = 0, 1, 2, 3
MB_INTER, MB_WIDE, MB_FOURMV, MB_CODED = 1, 2, 4, 8


class Pic(C.Structure):
    _fields_ = [
        ("stream", C.c_uint32), ("width", C.c_uint16), ("height", C.c_uint16), ("mb_w", C.c_uint8),
        ("mb_h", C.c_uint8), ("pic_type", C.c_uint8), ("pquant", C.c_uint8), ("flags", C.c_uint8),
        ("version", C.c_uint8), ("temporal_reference", C.c_uint16), ("first_mb", C.c_uint32), ("n_mbs", C.c_uint32),
        ("first_event", C.c_uint32), ("n_event_units", C.c_uint32),
    ]


class MbUnion(C.Union):
    _fields_ = [("mv", (C.c_int8 * 2) * 4), ("intradc", C.c_uint8 * 6)]


class Mb(C.Structure):
    _fields_ = [
        ("ev_off", C.c_uint32), ("pic", C.c_uint16), ("mbx", C.c_uint8), ("mby", C.c_uint8), ("flags", C.c_uint8),
        ("quant", C.c_uint8), ("nev", C.c_uint8 * 6), ("u", MbUnion),
    ]


class DeviceRgba(C.Structure):
    """h263cu_device_rgba: where h263cu_decode_step_device writes RGBA (a caller-owned device buffer)."""
    _fields_ = [
        ("base", C.c_void_p), ("row_pitch", C.c_uint64), ("pic_stride", C.c_uint64), ("width", C.c_uint32),
        ("height", C.c_uint32), ("stream", C.c_void_p),
    ]


class DevicePlane(C.Structure):
    """h263cu_device_plane: one caller-owned device plane of h263cu_device_yuv."""
    _fields_ = [("base", C.c_void_p), ("row_pitch", C.c_uint64), ("pic_stride", C.c_uint64)]


class DeviceYuv(C.Structure):
    """h263cu_device_yuv: where h263cu_decode_step_device_yuv writes the Y, Cb and Cr planes (I420 or NV12)."""
    _fields_ = [
        ("plane", DevicePlane * 3), ("width", C.c_uint32), ("height", C.c_uint32), ("format", C.c_uint32),
        ("reserved", C.c_uint32), ("stream", C.c_void_p),
    ]


YUV_I420, YUV_NV12 = 0, 1  # H263CU_YUV_*


class DeviceTensor(C.Structure):
    """h263cu_device_tensor: where h263cu_decode_step_device_tensor writes the resized, normalised RGB pictures
    (element [slot][channel][row][column] at base + the dot product of the indices and `stride`, in elements)."""
    _fields_ = [
        ("base", C.c_void_p), ("stride", C.c_int64 * 4), ("width", C.c_uint32), ("height", C.c_uint32),
        ("dtype", C.c_uint32), ("reserved", C.c_uint32), ("mul", C.c_float * 3), ("add", C.c_float * 3),
        ("stream", C.c_void_p),
    ]


TENSOR_U8, TENSOR_F32, TENSOR_F16, TENSOR_BF16 = 0, 1, 2, 3  # H263CU_TENSOR_*


class TensorCrop(C.Structure):
    """h263cu_tensor_crop: the box (x, y, width, height) of a decoded picture that h263cu_tensor_fit resizes."""
    _fields_ = [("x", C.c_uint32), ("y", C.c_uint32), ("width", C.c_uint32), ("height", C.c_uint32)]


class TensorFit(C.Structure):
    """h263cu_tensor_fit: how h263cu_decode_step_device_tensor_fit places each picture (or its crop box) in the
    output: stretched, letterboxed with a fill, or resized by its short side and centre-cropped."""
    _fields_ = [
        ("mode", C.c_uint32), ("short_side", C.c_uint32), ("fill", C.c_float * 3), ("reserved", C.c_uint32),
        ("crops", C.POINTER(TensorCrop)),
    ]


FIT_STRETCH, FIT_LETTERBOX, FIT_CENTER_CROP = 0, 1, 2  # H263CU_FIT_*
FILTER_BILINEAR, FILTER_BILINEAR_AA, FILTER_BICUBIC_AA = 0, 1, 2  # H263CU_FILTER_*

class DeviceMotion(C.Structure):
    """h263cu_device_motion: where h263cu_decode_step_device_motion writes each picture's motion vectors
    ([slot][x, y][block row][block column], int16 half-pel), macroblock flags and quantisers ([slot][mb row][mb column],
    uint8); a NULL base is not written."""
    _fields_ = [
        ("mv", C.c_void_p), ("mv_stride", C.c_int64 * 4), ("mb_flags", C.c_void_p), ("flags_stride", C.c_int64 * 3),
        ("mb_quant", C.c_void_p), ("quant_stride", C.c_int64 * 3), ("mb_width", C.c_uint32), ("mb_height", C.c_uint32),
        ("stream", C.c_void_p),
    ]


class DeviceOutput(C.Structure):
    """h263cu_device_output: the one pixel output (RGBA, planes or tensor, with its fit and filter) that
    h263cu_decode_step_device_motion writes beside the motion fields."""
    _fields_ = [
        ("rgba", C.POINTER(DeviceRgba)), ("yuv", C.POINTER(DeviceYuv)), ("tensor", C.POINTER(DeviceTensor)),
        ("fit", C.POINTER(TensorFit)), ("filter", C.c_uint32), ("reserved", C.c_uint32),
    ]


MOTION_OUTSIDE = 0x80  # H263CU_MOTION_OUTSIDE


class DeviceResidual(C.Structure):
    """h263cu_device_residual: where h263cu_decode_step_device_residual writes each picture's prediction residual
    (int16 Y, Cb and Cr planes, element [slot][row][column]); a NULL base is not written."""
    _fields_ = [
        ("y", C.c_void_p), ("y_stride", C.c_int64 * 3), ("cb", C.c_void_p), ("cb_stride", C.c_int64 * 3), ("cr", C.c_void_p),
        ("cr_stride", C.c_int64 * 3), ("width", C.c_uint32), ("height", C.c_uint32), ("stream", C.c_void_p),
    ]

assert C.sizeof(Pic) == 32 and C.sizeof(Mb) == 24 and C.sizeof(DeviceRgba) == 40
assert C.sizeof(DevicePlane) == 24 and C.sizeof(DeviceYuv) == 96 and C.sizeof(DeviceTensor) == 88
assert C.sizeof(TensorCrop) == 16 and C.sizeof(TensorFit) == 32
assert C.sizeof(DeviceMotion) == 120 and C.sizeof(DeviceOutput) == 40 and C.sizeof(DeviceResidual) == 112

# Every symbol include/h263cu.h declares; tests check that the library exports all of them.
SYMBOLS = [
    "h263cu_is_eof_error", "h263cu_is_macroblock_error", "h263cu_is_gob_error", "h263cu_strerror",
    "h263cu_version", "h263cu_parser_create", "h263cu_parser_destroy", "h263cu_parser_options", "h263cu_parser_reset",
    "h263cu_peek_picture", "h263cu_parse_picture", "h263cu_parse_step", "h263cu_device_count",
    "h263cu_create", "h263cu_destroy", "h263cu_device_of", "h263cu_alloc_pinned", "h263cu_free_pinned",
    "h263cu_step_upload", "h263cu_step_free", "h263cu_step_run", "h263cu_submit_step",
    "h263cu_submit_step_readback", "h263cu_decode_step", "h263cu_sync", "h263cu_stream_info", "h263cu_read_yuv", "h263cu_read_rgba",
    "h263cu_checksums", "h263cu_timer_start", "h263cu_timer_stop", "h263cu_launch_count", "h263cu_tiled_launch_count",
    "h263cu_profile_enable", "h263cu_profile_read", "h263cu_host_times",
    "h263cu_yuv420_to_rgba", "h263cu_deblock", "h263cu_quant_to_strength",
    "h263cu_flv_scan", "h263cu_flv_mux",
    "h263cu_test_read_bits", "h263cu_test_start_code", "h263cu_test_read_vlc", "h263cu_test_decode_block",
    "h263cu_readback_wait", "h263cu_stream_dims", "h263cu_graph_build", "h263cu_graph_launch", "h263cu_graph_free", "h263cu_group_create", "h263cu_group_destroy", "h263cu_group_size", "h263cu_group_ctx",
    "h263cu_group_decode_step", "h263cu_group_sync", "h263cu_decode_step_device", "h263cu_group_decode_step_device",
    "h263cu_decode_step_device_yuv", "h263cu_group_decode_step_device_yuv",
    "h263cu_decode_step_device_tensor", "h263cu_group_decode_step_device_tensor",
    "h263cu_decode_step_device_tensor_fit", "h263cu_group_decode_step_device_tensor_fit", "h263cu_test_fit_geometry",
    "h263cu_decode_step_device_tensor_filter", "h263cu_group_decode_step_device_tensor_filter",
    "h263cu_test_device_parse_step", "h263cu_decode_step_device_motion", "h263cu_group_decode_step_device_motion",
    "h263cu_decode_step_device_residual", "h263cu_group_decode_step_device_residual",
]

_lib = None


def lib():
    """Load libh263cu.so; raises if it has not been built (no fallback)."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise RuntimeError(
            "libh263cu.so is missing (%s): run `python -c 'import __graft_entry__ as g; g.build()'`; "
            "this package has no CPU fallback" % LIB_PATH
        )
    L = C.CDLL(LIB_PATH)
    vp, u32, u64, i32 = C.c_void_p, C.c_uint32, C.c_uint64, C.c_int
    L.h263cu_strerror.restype = C.c_char_p
    L.h263cu_strerror.argtypes = [i32]
    L.h263cu_parser_create.restype = vp
    L.h263cu_parser_create.argtypes = [u32]
    L.h263cu_parser_destroy.argtypes = [vp]
    L.h263cu_parser_options.restype = u32
    L.h263cu_parser_options.argtypes = [vp]
    L.h263cu_parser_destroy.restype = None
    L.h263cu_parser_reset.argtypes = [vp]
    L.h263cu_parser_reset.restype = None
    L.h263cu_peek_picture.argtypes = [u32, C.c_char_p, C.c_size_t, C.POINTER(Pic)]
    L.h263cu_parse_picture.argtypes = [vp, C.c_char_p, C.c_size_t, u32, C.c_uint16, u32, u32, C.POINTER(Pic), vp, u32,
                                       vp, u32]
    L.h263cu_parse_step.argtypes = [vp, vp, vp, vp, u32, i32, vp, vp, u32, vp, u32, C.POINTER(u32), C.POINTER(u32),
                                    C.POINTER(u32), vp, vp]
    if hasattr(L, "h263cu_create"):
        L.h263cu_create.restype = vp
        L.h263cu_create.argtypes = [i32, u32, u32, u32, u32, C.POINTER(i32)]
        L.h263cu_destroy.argtypes = [vp]
        L.h263cu_destroy.restype = None
        L.h263cu_device_of.argtypes = [vp]
        L.h263cu_alloc_pinned.restype = vp
        L.h263cu_alloc_pinned.argtypes = [C.c_size_t]
        L.h263cu_free_pinned.argtypes = [vp]
        L.h263cu_free_pinned.restype = None
        L.h263cu_step_upload.restype = vp
        L.h263cu_step_upload.argtypes = [vp, vp, u32, vp, u32, vp, u32, C.POINTER(i32)]
        L.h263cu_step_free.argtypes = [vp, vp]
        L.h263cu_step_free.restype = None
        L.h263cu_step_run.argtypes = [vp, vp, u32]
        L.h263cu_submit_step.argtypes = [vp, vp, u32, vp, u32, vp, u32, u32]
        L.h263cu_submit_step_readback.argtypes = [vp, vp, u32, vp, u32, vp, u32, u32, vp, vp]
        L.h263cu_decode_step.argtypes = [vp, vp, vp, vp, vp, u32, i32, u32, vp, u64, vp, C.POINTER(u32)]
        L.h263cu_decode_step_device.argtypes = [vp, vp, vp, vp, vp, u32, i32, u32, C.POINTER(DeviceRgba), vp, C.POINTER(u32)]
        L.h263cu_decode_step_device_yuv.argtypes = [vp, vp, vp, vp, vp, u32, i32, u32, C.POINTER(DeviceYuv), vp, C.POINTER(u32)]
        L.h263cu_decode_step_device_tensor.argtypes = [vp, vp, vp, vp, vp, u32, i32, u32, C.POINTER(DeviceTensor), vp, C.POINTER(u32)]
        L.h263cu_decode_step_device_tensor_fit.argtypes = [vp, vp, vp, vp, vp, u32, i32, u32, C.POINTER(DeviceTensor),
                                                           C.POINTER(TensorFit), vp, C.POINTER(u32)]
        L.h263cu_decode_step_device_tensor_filter.argtypes = [vp, vp, vp, vp, vp, u32, i32, u32, C.POINTER(DeviceTensor),
                                                              C.POINTER(TensorFit), u32, vp, C.POINTER(u32)]
        L.h263cu_decode_step_device_motion.argtypes = [vp, vp, vp, vp, vp, u32, i32, u32, C.POINTER(DeviceMotion),
                                                        C.POINTER(DeviceOutput), vp, C.POINTER(u32)]
        L.h263cu_decode_step_device_residual.argtypes = [vp, vp, vp, vp, vp, u32, i32, u32, C.POINTER(DeviceResidual),
                                                          C.POINTER(DeviceMotion), C.POINTER(DeviceOutput), vp, C.POINTER(u32)]
        L.h263cu_test_device_parse_step.argtypes = [vp, vp, vp, vp, vp, u32, i32, vp, vp, u32, vp, u32, C.POINTER(u32), C.POINTER(u32),
                                                    C.POINTER(u32), vp, vp]
        L.h263cu_sync.argtypes = [vp]
        L.h263cu_readback_wait.argtypes = [vp, u32]
        L.h263cu_graph_build.restype = vp
        L.h263cu_graph_build.argtypes = [vp, vp, u32, u32, C.POINTER(i32)]
        L.h263cu_graph_launch.argtypes = [vp, vp]
        L.h263cu_graph_free.argtypes = [vp, vp]
        L.h263cu_graph_free.restype = None
        L.h263cu_stream_dims.restype = u32
        L.h263cu_stream_dims.argtypes = [vp, u32]
        L.h263cu_group_create.restype = vp
        L.h263cu_group_create.argtypes = [vp, u32, u32, u32, u32, i32, C.POINTER(i32)]
        L.h263cu_group_destroy.argtypes = [vp]
        L.h263cu_group_destroy.restype = None
        L.h263cu_group_size.restype = u32
        L.h263cu_group_size.argtypes = [vp]
        L.h263cu_group_ctx.restype = vp
        L.h263cu_group_ctx.argtypes = [vp, u32]
        L.h263cu_group_decode_step.argtypes = [vp, vp, vp, vp, vp, u32, u32, vp, u64, vp, C.POINTER(u32)]
        L.h263cu_group_decode_step_device.argtypes = [vp, vp, vp, vp, vp, u32, u32, C.POINTER(DeviceRgba), vp, C.POINTER(u32)]
        L.h263cu_group_decode_step_device_yuv.argtypes = [vp, vp, vp, vp, vp, u32, u32, C.POINTER(DeviceYuv), vp, C.POINTER(u32)]
        L.h263cu_group_decode_step_device_tensor.argtypes = [vp, vp, vp, vp, vp, u32, u32, C.POINTER(DeviceTensor), vp, C.POINTER(u32)]
        L.h263cu_group_decode_step_device_tensor_fit.argtypes = [vp, vp, vp, vp, vp, u32, u32, C.POINTER(DeviceTensor),
                                                                 C.POINTER(TensorFit), vp, C.POINTER(u32)]
        L.h263cu_group_decode_step_device_tensor_filter.argtypes = [vp, vp, vp, vp, vp, u32, u32, C.POINTER(DeviceTensor),
                                                                    C.POINTER(TensorFit), u32, vp, C.POINTER(u32)]
        L.h263cu_group_decode_step_device_motion.argtypes = [vp, vp, vp, vp, vp, u32, u32, C.POINTER(DeviceMotion),
                                                              C.POINTER(DeviceOutput), vp, C.POINTER(u32)]
        L.h263cu_group_decode_step_device_residual.argtypes = [vp, vp, vp, vp, vp, u32, u32, C.POINTER(DeviceResidual),
                                                                C.POINTER(DeviceMotion), C.POINTER(DeviceOutput), vp, C.POINTER(u32)]
        L.h263cu_group_sync.argtypes = [vp]
        L.h263cu_stream_info.argtypes = [vp, u32] + [C.POINTER(u32)] * 5
        L.h263cu_read_yuv.argtypes = [vp, u32, vp, vp, vp]
        L.h263cu_read_rgba.argtypes = [vp, u32, vp]
        L.h263cu_checksums.argtypes = [vp, vp, u32, vp]
        L.h263cu_timer_start.argtypes = [vp]
        L.h263cu_timer_stop.argtypes = [vp, C.POINTER(C.c_float)]
        L.h263cu_launch_count.restype = u64
        L.h263cu_launch_count.argtypes = [vp]
        L.h263cu_tiled_launch_count.restype = u64
        L.h263cu_tiled_launch_count.argtypes = [vp]
        L.h263cu_profile_enable.argtypes = [vp, i32]
        L.h263cu_profile_read.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(u64)]
        L.h263cu_host_times.argtypes = [vp, C.POINTER(C.c_double), C.POINTER(C.c_double), C.POINTER(u64), i32]
        L.h263cu_yuv420_to_rgba.argtypes = [vp, vp, vp, C.c_size_t, C.c_size_t, vp]
        L.h263cu_deblock.argtypes = [vp, C.c_size_t, C.c_size_t, C.c_uint8, vp]
    L.h263cu_flv_scan.restype = C.c_int64
    L.h263cu_flv_scan.argtypes = [vp, C.c_size_t, vp, C.c_size_t, C.POINTER(u32)]
    L.h263cu_flv_mux.restype = C.c_int64
    L.h263cu_flv_mux.argtypes = [vp, vp, vp, vp, u32, u32, u32, vp, C.c_size_t]
    L.h263cu_test_read_bits.argtypes = [C.c_char_p, C.c_size_t, C.POINTER(C.c_size_t), i32, i32, i32, C.POINTER(C.c_int64)]
    L.h263cu_test_start_code.argtypes = [C.c_char_p, C.c_size_t, C.c_size_t, C.POINTER(i32)]
    L.h263cu_test_read_vlc.argtypes = [i32, C.c_char_p, C.c_size_t, C.POINTER(C.c_size_t), C.POINTER(i32)]
    L.h263cu_test_decode_block.argtypes = [C.c_char_p, C.c_size_t, C.POINTER(C.c_size_t), u32, i32, i32, i32, C.POINTER(i32),
                                           C.POINTER(i32), vp, vp, C.POINTER(i32)]
    L.h263cu_test_fit_geometry.argtypes = [u32, u32, u32, u32, u32, u32, C.POINTER(C.c_int32)]
    _lib = L
    return L


class H263Error(Exception):
    """Mirror of h263::Error (error.rs:6-57) plus the library's own failures."""

    def __init__(self, code):
        self.code = code
        super().__init__("%s (%d)" % (lib().h263cu_strerror(code).decode(), code))

    def is_eof_error(self):
        return bool(lib().h263cu_is_eof_error(self.code))

    def is_macroblock_error(self):
        return bool(lib().h263cu_is_macroblock_error(self.code))

    def is_gob_error(self):
        return bool(lib().h263cu_is_gob_error(self.code))


def check(code):
    if code < 0:
        raise H263Error(code)
    return code
