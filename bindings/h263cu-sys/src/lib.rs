//! Raw bindings of `libh263cu.so`, one declaration per symbol of `include/h263cu.h` (same order).
//! Each item names the reference interface it stands in for (paths relative to ruffle-rs/h263-rs).
#![allow(non_camel_case_types)]
use std::os::raw::{c_char, c_int, c_void};

// ---- error codes: -1..-17 = h263::Error in declaration order (h263/src/error.rs:6-57) ----
pub const H263CU_OK: c_int = 0;
pub const H263CU_ERR_INTERNAL_DECODER_ERROR: c_int = -1;
pub const H263CU_ERR_MIDDLE_OF_BITSTREAM: c_int = -2;
pub const H263CU_ERR_INVALID_MACROBLOCK_HEADER: c_int = -3;
pub const H263CU_ERR_INVALID_MACROBLOCK_CODED_BITS: c_int = -4;
pub const H263CU_ERR_INVALID_INTRA_DC: c_int = -5;
pub const H263CU_ERR_INVALID_SHORT_COEFFICIENT: c_int = -6;
pub const H263CU_ERR_INVALID_LONG_COEFFICIENT: c_int = -7;
pub const H263CU_ERR_INVALID_MVD: c_int = -8;
pub const H263CU_ERR_INVALID_PTYPE: c_int = -9;
pub const H263CU_ERR_INVALID_PLUSPTYPE: c_int = -10;
pub const H263CU_ERR_INVALID_GOB_HEADER: c_int = -11;
pub const H263CU_ERR_INVALID_BITSTREAM: c_int = -12;
pub const H263CU_ERR_PICTURE_FORMAT_MISSING: c_int = -13;
pub const H263CU_ERR_PICTURE_FORMAT_INVALID: c_int = -14;
pub const H263CU_ERR_UNCODED_IFRAME_BLOCKS: c_int = -15;
pub const H263CU_ERR_UNHANDLED_IO_ERROR: c_int = -16;
pub const H263CU_ERR_UNIMPLEMENTED_DECODING: c_int = -17;
pub const H263CU_ERR_BAD_ARGUMENT: c_int = -100;
pub const H263CU_ERR_CUDA: c_int = -101;
pub const H263CU_ERR_NO_DEVICE: c_int = -102;
pub const H263CU_ERR_CAPACITY: c_int = -103;
pub const H263CU_ERR_REFERENCE_WOULD_ABORT: c_int = -104;
pub const H263CU_ERR_NO_PICTURE: c_int = -105;
pub const H263CU_ERR_OUT_OF_MEMORY: c_int = -106;

/// DecoderOption bits (h263/src/decoder/types.rs:3-18)
pub const H263CU_OPT_SORENSON_SPARK_BITSTREAM: u32 = 1;
pub const H263CU_OPT_USE_SCALABILITY_MODE: u32 = 2;
/// EXTENSION beyond the reference: decode Sorenson disposable P pictures (macroblock.rs:461-465 fails them)
pub const H263CU_OPT_DECODE_DISPOSABLE: u32 = 0x100;

pub const H263CU_PIC_I: u8 = 0;
pub const H263CU_PIC_P: u8 = 1;
pub const H263CU_PIC_DISPOSABLE_P: u8 = 2;
pub const H263CU_PIC_OTHER: u8 = 3;
pub const H263CU_PICFLAG_DEBLOCK: u8 = 1;
pub const H263CU_PICFLAG_HAS_INTER: u8 = 2;
pub const H263CU_PICFLAG_MV_IN_RANGE: u8 = 4;
pub const H263CU_PICFLAG_DISPOSABLE: u8 = 8;
pub const H263CU_MB_INTER: u8 = 1;
pub const H263CU_MB_WIDE: u8 = 2;
pub const H263CU_MB_FOURMV: u8 = 4;
pub const H263CU_MB_CODED: u8 = 8;
pub const H263CU_OUT_RGBA: u32 = 1;
pub const H263CU_OUT_DEBLOCK: u32 = 2;
pub const H263CU_PARSE_ON_DEVICE: u32 = 4; // the macroblock layer parsed on the GPU (decode_step calls)
pub const H263CU_YUV_I420: u32 = 0; // plane[0] Y, plane[1] Cb, plane[2] Cr
pub const H263CU_YUV_NV12: u32 = 1; // plane[0] Y, plane[1] CbCr pairs (Cb first), plane[2] all zero
pub const H263CU_TENSOR_U8: u32 = 0;
pub const H263CU_TENSOR_F32: u32 = 1;
pub const H263CU_TENSOR_F16: u32 = 2;
pub const H263CU_TENSOR_BF16: u32 = 3;
pub const H263CU_FIT_STRETCH: u32 = 0; // the (cropped) picture resized to width x height
pub const H263CU_FIT_LETTERBOX: u32 = 1; // aspect kept, the whole (cropped) picture inside, centred, fill around it
pub const H263CU_FIT_CENTER_CROP: u32 = 2; // torchvision Resize(short_side) then CenterCrop((height, width))
pub const H263CU_FILTER_BILINEAR: u32 = 0; // torch's antialias=False bilinear: the fit call's output
pub const H263CU_FILTER_BILINEAR_AA: u32 = 1; // torch's bilinear with antialias=True (torchvision Resize's default)
pub const H263CU_FILTER_BICUBIC_AA: u32 = 2; // torch's bicubic with antialias=True (a = -0.5)

#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct h263cu_pic {
    // 32 bytes
    pub stream: u32,
    pub width: u16,
    pub height: u16,
    pub mb_w: u8,
    pub mb_h: u8,
    pub pic_type: u8,
    pub pquant: u8,
    pub flags: u8,
    pub version: u8,
    pub temporal_reference: u16,
    pub first_mb: u32,
    pub n_mbs: u32,
    pub first_event: u32,
    pub n_event_units: u32,
}

#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct h263cu_mb {
    // 24 bytes
    pub ev_off: u32,
    pub pic: u16,
    pub mbx: u8,
    pub mby: u8,
    pub flags: u8,
    pub quant: u8,
    pub nev: [u8; 6],
    /// union { mv: [[i8; 2]; 4], intradc: [u8; 6] }
    pub u: [u8; 8],
}

#[repr(C)]
#[derive(Clone, Copy, Debug, Default)]
pub struct h263cu_flv_packet {
    // 24 bytes
    pub offset: u64,
    pub size: u32,
    pub timestamp_ms: u32,
    pub frame_type: u8,
    pub codec_id: u8,
    pub reserved: u16,
    pub reserved2: u32,
}

pub type h263cu_event = u16;

/// Where h263cu_decode_step_device writes RGBA: caller-owned device memory (see include/h263cu.h for the rules).
#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct h263cu_device_rgba {
    // 40 bytes
    pub base: *mut u8,       // device (or managed) memory of the context's device, 16-byte aligned
    pub row_pitch: u64,      // multiple of 16, >= 4 * width, < 2^32
    pub pic_stride: u64,     // multiple of 16, >= row_pitch * height, < 2^40
    pub width: u32,          // slot size
    pub height: u32,
    pub stream: *mut c_void, // the consumer's CUstream / cudaStream_t; null = the legacy default stream
}

/// One caller-owned device plane of h263cu_device_yuv (see include/h263cu.h for the rules).
#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct h263cu_device_plane {
    // 24 bytes
    pub base: *mut u8,   // device (or managed) memory of the context's device, 4-byte aligned
    pub row_pitch: u64,  // multiple of 4, >= the plane's slot row bytes, < 2^32
    pub pic_stride: u64, // multiple of 4, >= row_pitch * the plane's slot rows, < 2^40
}

/// Where h263cu_decode_step_device_yuv writes the decoded planes: caller-owned device memory, I420 or NV12.
#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct h263cu_device_yuv {
    // 96 bytes
    pub plane: [h263cu_device_plane; 3],
    pub width: u32,          // luma slot size; the chroma slot is ceil(width / 2) x ceil(height / 2)
    pub height: u32,
    pub format: u32,         // H263CU_YUV_I420 or H263CU_YUV_NV12
    pub reserved: u32,       // 0
    pub stream: *mut c_void, // the consumer's CUstream / cudaStream_t; null = the legacy default stream
}

/// Where h263cu_decode_step_device_tensor writes the resized, normalised RGB pictures: a caller-owned device tensor
/// [slot][channel (R, G, B)][row][column] (see include/h263cu.h for the definition of the values and the rules).
#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct h263cu_device_tensor {
    // 88 bytes
    pub base: *mut c_void,   // element [0][0][0][0]; device (or managed) memory of the context's device, element-aligned
    pub stride: [i64; 4],    // in elements: slot, channel, row, column; every stride > 0
    pub width: u32,          // output size, 1..16384: every picture is resized to exactly this
    pub height: u32,
    pub dtype: u32,          // H263CU_TENSOR_*
    pub reserved: u32,       // 0
    pub mul: [f32; 3],       // per channel: out = v * mul[c] + add[c]; 1 and 0 for H263CU_TENSOR_U8
    pub add: [f32; 3],
    pub stream: *mut c_void, // the consumer's CUstream / cudaStream_t; null = the legacy default stream
}

/// The box of a decoded picture that h263cu_decode_step_device_tensor_fit resizes.
#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct h263cu_tensor_crop {
    // 16 bytes
    pub x: u32,
    pub y: u32,
    pub width: u32,
    pub height: u32,
}

/// How h263cu_decode_step_device_tensor_fit places each picture in the tensor (include/h263cu.h defines the geometry).
#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct h263cu_tensor_fit {
    // 32 bytes
    pub mode: u32,                        // H263CU_FIT_*
    pub short_side: u32,                  // H263CU_FIT_CENTER_CROP: 1..16384; other modes: 0
    pub fill: [f32; 3],                   // per channel, on the 0..255 scale; finite, 0 <= fill <= 255
    pub reserved: u32,                    // 0
    pub crops: *const h263cu_tensor_crop, // null: every whole picture; else one per input (host memory)
}

pub const H263CU_MOTION_OUTSIDE: u32 = 0x80; // mb_flags of a slot cell outside the picture's macroblock grid

/// Where h263cu_decode_step_device_motion writes each picture's motion fields (include/h263cu.h defines the values):
/// caller-owned device buffers, each NULL base not written.
#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct h263cu_device_motion {
    // 120 bytes
    pub mv: *mut i16,            // [slot][component: x, y][block row][block column], half-pel units
    pub mv_stride: [i64; 4],     // in elements, each > 0
    pub mb_flags: *mut u8,       // [slot][mb row][mb column]: H263CU_MB_INTER | _FOURMV | _CODED, or H263CU_MOTION_OUTSIDE
    pub flags_stride: [i64; 3],
    pub mb_quant: *mut u8,       // [slot][mb row][mb column]: the quantiser in force, 0 outside the picture
    pub quant_stride: [i64; 3],
    pub mb_width: u32,           // slot grid in macroblocks, 1..255; the mv grid is 2*mb_width x 2*mb_height blocks
    pub mb_height: u32,
    pub stream: *mut c_void,     // the consumer's CUstream / cudaStream_t; null = the legacy default stream
}

/// The one pixel output h263cu_decode_step_device_motion writes beside the motion fields (at most one of rgba / yuv /
/// tensor is not null; none: motion only).
#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct h263cu_device_output {
    // 40 bytes
    pub rgba: *const h263cu_device_rgba,
    pub yuv: *const h263cu_device_yuv,
    pub tensor: *const h263cu_device_tensor,
    pub fit: *const h263cu_tensor_fit, // tensor only: null = the plain tensor call, else the fit / filter call
    pub filter: u32,                   // tensor with fit: H263CU_FILTER_*; otherwise 0
    pub reserved: u32,                 // 0
}

/// Where h263cu_decode_step_device_residual writes each picture's prediction residual (include/h263cu.h defines the
/// values): caller-owned int16 device planes, each NULL base not written.
#[repr(C)]
#[derive(Clone, Copy, Debug)]
pub struct h263cu_device_residual {
    // 112 bytes
    pub y: *mut i16,             // [slot][row][column]
    pub y_stride: [i64; 3],      // in elements, each > 0
    pub cb: *mut i16,            // [slot][row][column]
    pub cb_stride: [i64; 3],
    pub cr: *mut i16,            // [slot][row][column]
    pub cr_stride: [i64; 3],
    pub width: u32,              // the luma slot, 1..16384; the chroma slot is ceil(width/2) x ceil(height/2)
    pub height: u32,
    pub stream: *mut c_void,     // the consumer's CUstream / cudaStream_t; null = the legacy default stream
}

#[repr(C)]
pub struct h263cu_parser {
    _private: [u8; 0],
}
#[repr(C)]
pub struct h263cu_ctx {
    _private: [u8; 0],
}
#[repr(C)]
pub struct h263cu_step {
    _private: [u8; 0],
}
#[repr(C)]
pub struct h263cu_graph {
    _private: [u8; 0],
}
#[repr(C)]
pub struct h263cu_group {
    _private: [u8; 0],
}

extern "C" {
    // error.rs:66-93
    pub fn h263cu_is_eof_error(err: c_int) -> c_int;
    pub fn h263cu_is_macroblock_error(err: c_int) -> c_int;
    pub fn h263cu_is_gob_error(err: c_int) -> c_int;
    pub fn h263cu_strerror(err: c_int) -> *const c_char;
    pub fn h263cu_version() -> c_int;

    // host front end: H263Reader + the serial loop of decode_next_picture (state.rs:142-427)
    pub fn h263cu_parser_create(decoder_options: u32) -> *mut h263cu_parser; // H263State::new, state.rs:42-50
    pub fn h263cu_parser_destroy(p: *mut h263cu_parser);
    pub fn h263cu_parser_options(p: *const h263cu_parser) -> u32;
    pub fn h263cu_parser_reset(p: *mut h263cu_parser); // seek: state.rs:134-137
    pub fn h263cu_peek_picture(decoder_options: u32, data: *const u8, len: usize, pic: *mut h263cu_pic) -> c_int; // state.rs:102-111
    pub fn h263cu_parse_picture(
        p: *mut h263cu_parser, data: *const u8, len: usize, stream: u32, pic_index: u16, mb_base: u32, ev_base: u32,
        pic: *mut h263cu_pic, mbs: *mut h263cu_mb, mb_cap: u32, events: *mut h263cu_event, ev_cap: u32,
    ) -> c_int;
    pub fn h263cu_parse_step(
        parsers: *const *mut h263cu_parser, packets: *const *const u8, lens: *const usize, stream_ids: *const u32, n: u32,
        threads: c_int, pics: *mut h263cu_pic, mbs: *mut h263cu_mb, mb_cap: u32, events: *mut h263cu_event, ev_cap: u32,
        n_pics_out: *mut u32, n_mbs_out: *mut u32, n_units_out: *mut u32, per_pic_err: *mut c_int, pic_of_input: *mut i32,
    ) -> c_int;

    // test hooks (reader.rs:448-559, macroblock.rs:551-1010, block.rs:757-2124 replayed on the product front end)
    pub fn h263cu_test_read_bits(data: *const u8, len: usize, bitpos: *mut usize, nbits: c_int, is_signed: c_int, peek: c_int, value: *mut i64) -> c_int;
    pub fn h263cu_test_start_code(data: *const u8, len: usize, bitpos: usize, skipped: *mut c_int) -> c_int;
    pub fn h263cu_test_read_vlc(table: c_int, data: *const u8, len: usize, bitpos: *mut usize, out4: *mut c_int) -> c_int;
    pub fn h263cu_test_decode_block(
        data: *const u8, len: usize, bitpos: *mut usize, decoder_options: u32, version: c_int, is_intra: c_int,
        tcoef_present: c_int, intradc_code: *mut c_int, n_events: *mut c_int, run: *mut u8, level: *mut i16, overflow: *mut c_int,
    ) -> c_int;
    /// The fit geometry {rw, rh, px, py} of a cw x ch crop (include/h263cu.h), as h263cu_decode_step_device_tensor_fit computes it
    pub fn h263cu_test_fit_geometry(mode: u32, short_side: u32, cw: u32, ch: u32, width: u32, height: u32, out4: *mut i32) -> c_int;
    /// h263cu_parse_step's outputs produced by the device parse of `ctx` (H263CU_PARSE_ON_DEVICE); the parsers stay
    pub fn h263cu_test_device_parse_step(
        ctx: *mut h263cu_ctx, parsers: *const *mut h263cu_parser, packets: *const *const u8, lens: *const usize, stream_ids: *const u32,
        n: u32, threads: c_int, pics: *mut h263cu_pic, mbs: *mut h263cu_mb, mb_cap: u32, events: *mut h263cu_event, ev_cap: u32,
        n_pics_out: *mut u32, n_mbs_out: *mut u32, n_units_out: *mut u32, per_pic_err: *mut c_int, pic_of_input: *mut i32,
    ) -> c_int;

    // device context: the recon tail of decode_next_picture (state.rs:419-485) + yuv + deblock
    pub fn h263cu_device_count() -> c_int;
    pub fn h263cu_create(device: c_int, max_streams: u32, max_width: u32, max_height: u32, flags: u32, err: *mut c_int) -> *mut h263cu_ctx;
    pub fn h263cu_destroy(c: *mut h263cu_ctx);
    pub fn h263cu_device_of(c: *mut h263cu_ctx) -> c_int;
    pub fn h263cu_alloc_pinned(bytes: usize) -> *mut u8;
    pub fn h263cu_free_pinned(p: *mut u8);
    pub fn h263cu_step_upload(
        c: *mut h263cu_ctx, pics: *const h263cu_pic, n_pics: u32, mbs: *const h263cu_mb, n_mbs: u32, events: *const h263cu_event,
        n_units: u32, err: *mut c_int,
    ) -> *mut h263cu_step;
    pub fn h263cu_step_free(c: *mut h263cu_ctx, s: *mut h263cu_step);
    pub fn h263cu_step_run(c: *mut h263cu_ctx, s: *mut h263cu_step, out_flags: u32) -> c_int;
    pub fn h263cu_graph_build(c: *mut h263cu_ctx, steps: *const *mut h263cu_step, n_steps: u32, out_flags: u32, err: *mut c_int) -> *mut h263cu_graph;
    pub fn h263cu_graph_launch(c: *mut h263cu_ctx, g: *mut h263cu_graph) -> c_int;
    pub fn h263cu_graph_free(c: *mut h263cu_ctx, g: *mut h263cu_graph);
    pub fn h263cu_submit_step(
        c: *mut h263cu_ctx, pics: *const h263cu_pic, n_pics: u32, mbs: *const h263cu_mb, n_mbs: u32, events: *const h263cu_event,
        n_units: u32, out_flags: u32,
    ) -> c_int;
    pub fn h263cu_submit_step_readback(
        c: *mut h263cu_ctx, pics: *const h263cu_pic, n_pics: u32, mbs: *const h263cu_mb, n_mbs: u32, events: *const h263cu_event,
        n_units: u32, out_flags: u32, host_rgba: *mut u8, rgba_offsets: *const u64,
    ) -> c_int;
    /// Batched H263State::decode_next_picture (state.rs:138-489) from the bitstream
    pub fn h263cu_decode_step(
        c: *mut h263cu_ctx, parsers: *const *mut h263cu_parser, packets: *const *const u8, lens: *const usize,
        stream_ids: *const u32, n: u32, threads: c_int, out_flags: u32, host_rgba: *mut u8, rgba_stride: u64,
        per_pic_err: *mut c_int, n_decoded: *mut u32,
    ) -> c_int;
    /// h263cu_decode_step with the RGBA of input i written to slot i of caller-owned device memory
    pub fn h263cu_decode_step_device(
        c: *mut h263cu_ctx, parsers: *const *mut h263cu_parser, packets: *const *const u8, lens: *const usize,
        stream_ids: *const u32, n: u32, threads: c_int, out_flags: u32, out: *const h263cu_device_rgba,
        per_pic_err: *mut c_int, n_decoded: *mut u32,
    ) -> c_int;
    /// h263cu_decode_step with the Y, Cb and Cr planes of input i written to slot i of caller-owned device planes
    pub fn h263cu_decode_step_device_yuv(
        c: *mut h263cu_ctx, parsers: *const *mut h263cu_parser, packets: *const *const u8, lens: *const usize,
        stream_ids: *const u32, n: u32, threads: c_int, out_flags: u32, out: *const h263cu_device_yuv,
        per_pic_err: *mut c_int, n_decoded: *mut u32,
    ) -> c_int;
    /// h263cu_decode_step with input i resized and converted into slot i of a caller-owned device tensor
    pub fn h263cu_decode_step_device_tensor(
        c: *mut h263cu_ctx, parsers: *const *mut h263cu_parser, packets: *const *const u8, lens: *const usize,
        stream_ids: *const u32, n: u32, threads: c_int, out_flags: u32, out: *const h263cu_device_tensor,
        per_pic_err: *mut c_int, n_decoded: *mut u32,
    ) -> c_int;
    /// h263cu_decode_step_device_tensor with each picture (or its crop box) letterboxed, centre-cropped or stretched
    pub fn h263cu_decode_step_device_tensor_fit(
        c: *mut h263cu_ctx, parsers: *const *mut h263cu_parser, packets: *const *const u8, lens: *const usize,
        stream_ids: *const u32, n: u32, threads: c_int, out_flags: u32, out: *const h263cu_device_tensor,
        fit: *const h263cu_tensor_fit, per_pic_err: *mut c_int, n_decoded: *mut u32,
    ) -> c_int;
    /// h263cu_decode_step_device_tensor_fit resized with an antialiased filter (H263CU_FILTER_*)
    pub fn h263cu_decode_step_device_tensor_filter(
        c: *mut h263cu_ctx, parsers: *const *mut h263cu_parser, packets: *const *const u8, lens: *const usize,
        stream_ids: *const u32, n: u32, threads: c_int, out_flags: u32, out: *const h263cu_device_tensor,
        fit: *const h263cu_tensor_fit, filter: u32, per_pic_err: *mut c_int, n_decoded: *mut u32,
    ) -> c_int;
    pub fn h263cu_sync(c: *mut h263cu_ctx) -> c_int;
    pub fn h263cu_readback_wait(c: *mut h263cu_ctx, age: u32) -> c_int;

    // one process, several GPUs
    pub fn h263cu_group_create(
        devices: *const c_int, n_devices: u32, streams_per_device: u32, max_width: u32, max_height: u32, threads: c_int, err: *mut c_int,
    ) -> *mut h263cu_group;
    pub fn h263cu_group_destroy(g: *mut h263cu_group);
    pub fn h263cu_group_size(g: *const h263cu_group) -> u32;
    pub fn h263cu_group_ctx(g: *mut h263cu_group, index: u32) -> *mut h263cu_ctx;
    pub fn h263cu_group_decode_step(
        g: *mut h263cu_group, parsers: *const *mut h263cu_parser, packets: *const *const u8, lens: *const usize,
        stream_ids: *const u32, n: u32, out_flags: u32, host_rgba: *mut u8, rgba_stride: u64, per_pic_err: *mut c_int,
        n_decoded: *mut u32,
    ) -> c_int;
    pub fn h263cu_group_decode_step_device(
        g: *mut h263cu_group, parsers: *const *mut h263cu_parser, packets: *const *const u8, lens: *const usize,
        stream_ids: *const u32, n: u32, out_flags: u32, outs: *const h263cu_device_rgba, per_pic_err: *mut c_int,
        n_decoded: *mut u32,
    ) -> c_int;
    pub fn h263cu_group_decode_step_device_yuv(
        g: *mut h263cu_group, parsers: *const *mut h263cu_parser, packets: *const *const u8, lens: *const usize,
        stream_ids: *const u32, n: u32, out_flags: u32, outs: *const h263cu_device_yuv, per_pic_err: *mut c_int,
        n_decoded: *mut u32,
    ) -> c_int;
    pub fn h263cu_group_decode_step_device_tensor(
        g: *mut h263cu_group, parsers: *const *mut h263cu_parser, packets: *const *const u8, lens: *const usize,
        stream_ids: *const u32, n: u32, out_flags: u32, outs: *const h263cu_device_tensor, per_pic_err: *mut c_int,
        n_decoded: *mut u32,
    ) -> c_int;
    pub fn h263cu_group_decode_step_device_tensor_fit(
        g: *mut h263cu_group, parsers: *const *mut h263cu_parser, packets: *const *const u8, lens: *const usize,
        stream_ids: *const u32, n: u32, out_flags: u32, outs: *const h263cu_device_tensor, fit: *const h263cu_tensor_fit,
        per_pic_err: *mut c_int, n_decoded: *mut u32,
    ) -> c_int;
    pub fn h263cu_group_decode_step_device_tensor_filter(
        g: *mut h263cu_group, parsers: *const *mut h263cu_parser, packets: *const *const u8, lens: *const usize,
        stream_ids: *const u32, n: u32, out_flags: u32, outs: *const h263cu_device_tensor, fit: *const h263cu_tensor_fit,
        filter: u32, per_pic_err: *mut c_int, n_decoded: *mut u32,
    ) -> c_int;
    /// h263cu_decode_step with each picture's motion fields, alone (pixels null) or beside one pixel output
    pub fn h263cu_decode_step_device_motion(
        c: *mut h263cu_ctx, parsers: *const *mut h263cu_parser, packets: *const *const u8, lens: *const usize,
        stream_ids: *const u32, n: u32, threads: c_int, out_flags: u32, motion: *const h263cu_device_motion,
        pixels: *const h263cu_device_output, per_pic_err: *mut c_int, n_decoded: *mut u32,
    ) -> c_int;
    /// h263cu_decode_step_device_motion for a group: one motion target (and pixel output) per device
    pub fn h263cu_group_decode_step_device_motion(
        g: *mut h263cu_group, parsers: *const *mut h263cu_parser, packets: *const *const u8, lens: *const usize,
        stream_ids: *const u32, n: u32, out_flags: u32, motions: *const h263cu_device_motion,
        pixels: *const h263cu_device_output, per_pic_err: *mut c_int, n_decoded: *mut u32,
    ) -> c_int;
    /// h263cu_decode_step with each picture's prediction residual, alone or beside the motion fields (motion null:
    /// none) and / or one pixel output (pixels null: none)
    pub fn h263cu_decode_step_device_residual(
        c: *mut h263cu_ctx, parsers: *const *mut h263cu_parser, packets: *const *const u8, lens: *const usize,
        stream_ids: *const u32, n: u32, threads: c_int, out_flags: u32, residual: *const h263cu_device_residual,
        motion: *const h263cu_device_motion, pixels: *const h263cu_device_output, per_pic_err: *mut c_int,
        n_decoded: *mut u32,
    ) -> c_int;
    /// h263cu_decode_step_device_residual for a group: one residual target (and motion target, pixel output) per device
    pub fn h263cu_group_decode_step_device_residual(
        g: *mut h263cu_group, parsers: *const *mut h263cu_parser, packets: *const *const u8, lens: *const usize,
        stream_ids: *const u32, n: u32, out_flags: u32, residuals: *const h263cu_device_residual,
        motions: *const h263cu_device_motion, pixels: *const h263cu_device_output, per_pic_err: *mut c_int,
        n_decoded: *mut u32,
    ) -> c_int;
    pub fn h263cu_group_sync(g: *mut h263cu_group) -> c_int;

    // DecodedPicture accessors (h263/src/decoder/picture.rs:60-142)
    pub fn h263cu_stream_info(
        c: *mut h263cu_ctx, stream: u32, width: *mut u32, height: *mut u32, pic_type: *mut u32, pquant: *mut u32,
        temporal_reference: *mut u32,
    ) -> c_int;
    pub fn h263cu_stream_dims(c: *mut h263cu_ctx, stream: u32) -> u32;
    pub fn h263cu_read_yuv(c: *mut h263cu_ctx, stream: u32, y: *mut u8, cb: *mut u8, cr: *mut u8) -> c_int;
    pub fn h263cu_read_rgba(c: *mut h263cu_ctx, stream: u32, rgba: *mut u8) -> c_int;
    pub fn h263cu_checksums(c: *mut h263cu_ctx, streams: *const u32, n: u32, out4: *mut u64) -> c_int;

    pub fn h263cu_timer_start(c: *mut h263cu_ctx) -> c_int;
    pub fn h263cu_timer_stop(c: *mut h263cu_ctx, milliseconds: *mut f32) -> c_int;
    pub fn h263cu_launch_count(c: *mut h263cu_ctx) -> u64;
    pub fn h263cu_tiled_launch_count(c: *mut h263cu_ctx) -> u64;
    pub fn h263cu_host_times(c: *mut h263cu_ctx, parse_seconds: *mut f64, other_seconds: *mut f64, calls: *mut u64, reset: c_int) -> c_int;
    pub fn h263cu_profile_enable(c: *mut h263cu_ctx, enable: c_int) -> c_int;
    pub fn h263cu_profile_read(c: *mut h263cu_ctx, ms2: *mut f64, launches2: *mut u64) -> c_int;

    // sibling crates
    /// yuv::bt601::yuv420_to_rgba (yuv/src/bt601.rs:105-196)
    pub fn h263cu_yuv420_to_rgba(y: *const u8, chroma_b: *const u8, chroma_r: *const u8, y_len: usize, y_width: usize, rgba_out: *mut u8) -> c_int;
    /// deblock::deblock::deblock (deblock/src/deblock.rs:305-315)
    pub fn h263cu_deblock(data: *const u8, len: usize, width: usize, strength: u8, out: *mut u8) -> c_int;
    /// deblock::deblock::QUANT_TO_STRENGTH (deblock/src/deblock.rs:5-8)
    pub static h263cu_quant_to_strength: [u8; 32];

    // FLV container feed (one H263Reader::from_source(&packet[..]) per video tag)
    pub fn h263cu_flv_scan(data: *const u8, len: usize, out: *mut h263cu_flv_packet, cap: usize, n_other_tags: *mut u32) -> i64;
    pub fn h263cu_flv_mux(
        packets: *const u8, pkt_off: *const u64, pkt_len: *const u32, frame_types: *const u8, n: u32, ms_per_picture: u32,
        filler_every: u32, out: *mut u8, cap: usize,
    ) -> i64;
}

#[cfg(test)]
mod tests {
    use super::*;
    #[test]
    fn layouts_match_the_header() {
        assert_eq!(std::mem::size_of::<h263cu_pic>(), 32);
        assert_eq!(std::mem::size_of::<h263cu_mb>(), 24);
        assert_eq!(std::mem::size_of::<h263cu_flv_packet>(), 24);
        assert_eq!(std::mem::size_of::<h263cu_device_tensor>(), 88);
        assert_eq!(std::mem::size_of::<h263cu_tensor_crop>(), 16);
        assert_eq!(std::mem::size_of::<h263cu_tensor_fit>(), 32);
        assert_eq!(std::mem::size_of::<h263cu_device_motion>(), 120);
        assert_eq!(std::mem::size_of::<h263cu_device_output>(), 40);
        assert_eq!(std::mem::size_of::<h263cu_device_residual>(), 112);
    }
    #[test]
    fn library_answers() {
        unsafe {
            assert!(h263cu_version() >= 100);
            assert_eq!(h263cu_is_eof_error(H263CU_ERR_UNHANDLED_IO_ERROR), 1);
            assert_eq!(h263cu_quant_to_strength[31], 12);
        }
    }
}
