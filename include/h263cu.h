/*
 * h263cu.h -- C ABI of libh263cu.so, the B200-native reconstruction path for
 * ruffle-rs/h263-rs streams (H.263 / Sorenson Spark).
 *
 * The reference is a pure-Rust library without an FFI layer; the boundary it offers is
 * its public Rust API.  Each entry point below names the reference interface it stands
 * in for (paths relative to the reference repository).  A Rust `-sys` crate binds these
 * symbols 1:1 (see INTEGRATION.md); the façade crates on top keep the reference's own
 * names (`H263State::decode_next_picture`, `yuv::bt601::yuv420_to_rgba`,
 * `deblock::deblock::deblock`).
 *
 * Division of labour (BASELINE.json north_star):
 *   host  : serial bitstream / VLC parse, one parser per stream, threaded across streams
 *           (h263cu_parser_*, h263cu_parse_step).  Output = compact side info:
 *           h263cu_pic + h263cu_mb records + 16-bit run/level event units.
 *   device: everything after the parse -- inverse RLE + dequantisation, block
 *           classification, f32 IDCT (reference operation order, no FMA), motion
 *           compensation with edge clamping, residual add + clamp, optional deblocking
 *           post-filter, BT.601 YUV420 -> RGBA.  (h263cu_step_*, h263cu_submit_step)
 * There is no CPU fallback: device entry points fail with H263CU_ERR_NO_DEVICE /
 * H263CU_ERR_CUDA when no usable GPU is present.
 *
 * Threading: a context is externally synchronised (one submitting thread per context);
 * parsers are independent objects; h263cu_parse_step runs its own worker threads.
 * Ownership: the caller owns every host buffer; the context owns all device memory.
 * Errors: 0 = success, negative = failure, never aborts.
 */
#ifndef H263CU_H
#define H263CU_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

/* ---- error codes --------------------------------------------------------------------
 * -1..-17 are the reference's h263::Error variants in declaration order
 * (h263/src/error.rs:6-57). */
#define H263CU_OK 0
#define H263CU_ERR_INTERNAL_DECODER_ERROR (-1)
#define H263CU_ERR_MIDDLE_OF_BITSTREAM (-2)
#define H263CU_ERR_INVALID_MACROBLOCK_HEADER (-3)
#define H263CU_ERR_INVALID_MACROBLOCK_CODED_BITS (-4)
#define H263CU_ERR_INVALID_INTRA_DC (-5)
#define H263CU_ERR_INVALID_SHORT_COEFFICIENT (-6)
#define H263CU_ERR_INVALID_LONG_COEFFICIENT (-7)
#define H263CU_ERR_INVALID_MVD (-8)
#define H263CU_ERR_INVALID_PTYPE (-9)
#define H263CU_ERR_INVALID_PLUSPTYPE (-10)
#define H263CU_ERR_INVALID_GOB_HEADER (-11)
#define H263CU_ERR_INVALID_BITSTREAM (-12)
#define H263CU_ERR_PICTURE_FORMAT_MISSING (-13)
#define H263CU_ERR_PICTURE_FORMAT_INVALID (-14)
#define H263CU_ERR_UNCODED_IFRAME_BLOCKS (-15)
#define H263CU_ERR_UNHANDLED_IO_ERROR (-16) /* in-memory packets: UnexpectedEof */
#define H263CU_ERR_UNIMPLEMENTED_DECODING (-17)
/* library errors */
#define H263CU_ERR_BAD_ARGUMENT (-100)
#define H263CU_ERR_CUDA (-101)
#define H263CU_ERR_NO_DEVICE (-102)
#define H263CU_ERR_CAPACITY (-103)              /* stream / MB / event capacity exceeded */
#define H263CU_ERR_REFERENCE_WOULD_ABORT (-104) /* input on which the reference panics (abort) */
#define H263CU_ERR_NO_PICTURE (-105)            /* stream has not decoded a picture yet */
#define H263CU_ERR_OUT_OF_MEMORY (-106)

/* error.rs:66-93 classification helpers */
int h263cu_is_eof_error(int err);
int h263cu_is_macroblock_error(int err);
int h263cu_is_gob_error(int err);
const char* h263cu_strerror(int err);
int h263cu_version(void);

/* DecoderOption (h263/src/decoder/types.rs:3-18) */
#define H263CU_OPT_SORENSON_SPARK_BITSTREAM 1u
#define H263CU_OPT_USE_SCALABILITY_MODE 2u
/* EXTENSION, beyond the reference: decode Sorenson disposable P pictures (picture type 2, FLV frame type 3) like P
 * pictures that are shown but never become a reference.  The reference fails them with UnimplementedDecoding
 * (macroblock.rs:461-465), and so does this library unless the bit is set at h263cu_parser_create. */
#define H263CU_OPT_DECODE_DISPOSABLE 0x100u

/* ---- side-info format (host -> device) ------------------------------------------------
 * One time step = one picture for each of n streams.  All three arrays live in
 * caller-owned (ideally pinned) memory. */

#define H263CU_PIC_I 0
#define H263CU_PIC_P 1
#define H263CU_PIC_DISPOSABLE_P 2
#define H263CU_PIC_OTHER 3 /* PB / reserved types: only all-uncoded pictures decode */

#define H263CU_PICFLAG_DEBLOCK 1u   /* Sorenson DeblockingFlag (advisory, picture.rs:319-325) */
#define H263CU_PICFLAG_HAS_INTER 2u /* at least one MB needs the reference picture */
/* Every motion vector component of the picture lies in [-32, 31] half-pel units.  Always true for a stream decoded by
 * the front end: halfpel_decode (mvd_pred.rs:70-117) wraps into that range, and the extended range is unreachable
 * because the running options stay empty (state.rs:152-155).  When every picture of a step carries the flag the
 * device runs the reconstruction kernel without the clamped per-sample prediction path.  A producer that sets the
 * flag on a picture with longer vectors gets them clamped to the range. */
#define H263CU_PICFLAG_MV_IN_RANGE 4u
/* The picture is a disposable P picture decoded under H263CU_OPT_DECODE_DISPOSABLE: it becomes the stream's last
 * picture but not the reference of the next one (the previous reference stays in place). */
#define H263CU_PICFLAG_DISPOSABLE 8u

typedef struct h263cu_pic { /* 32 bytes */
    uint32_t stream;        /* stream slot inside the context, < max_streams */
    uint16_t width, height; /* true luma dimensions (not MB rounded) */
    uint8_t mb_w, mb_h;     /* ceil(width/16), ceil(height/16) (state.rs:173-174); <= 255 */
    uint8_t pic_type;       /* H263CU_PIC_* */
    uint8_t pquant;         /* PQUANT of the header; selects the deblock strength */
    uint8_t flags;          /* H263CU_PICFLAG_* */
    uint8_t version;        /* Sorenson version field (0xFF for baseline H.263) */
    uint16_t temporal_reference;
    uint32_t first_mb;      /* index of the picture's first record in the step's mb array */
    uint32_t n_mbs;         /* mb_w * mb_h */
    uint32_t first_event;   /* index of the picture's first unit in the step's event array */
    uint32_t n_event_units; /* 16-bit units used by this picture */
} h263cu_pic;

#define H263CU_MB_INTER 1u  /* motion compensated from the reference (MacroblockType::is_inter) */
#define H263CU_MB_WIDE 2u   /* this MB's events use the 2-unit wide form */
#define H263CU_MB_FOURMV 4u /* four motion vectors (informational; mv[] always holds 4) */
#define H263CU_MB_CODED 8u  /* COD=0 (informational) */

/* The flags, quantiser and vectors of these records reach the caller as dense per-picture grids through
 * h263cu_decode_step_device_motion below. */
typedef struct h263cu_mb { /* 24 bytes, raster order inside a picture */
    uint32_t ev_off;       /* first event unit of the MB, relative to pic.first_event */
    uint16_t pic;          /* index into the step's pic array */
    uint8_t mbx, mby;      /* macroblock coordinates */
    uint8_t flags;         /* H263CU_MB_* */
    uint8_t quant;         /* in-force quantiser 1..31 (state.rs:226-227) */
    uint8_t nev[6];        /* events per block, order Y0 Y1 Y2 Y3 Cb Cr (state.rs:287-381); at most 64
                              (INTRA: 63, and 0 under INTRADC code 0) */
    union {
        int8_t mv[4][2];    /* INTER: decoded half-pel vectors (x, y) per luma block */
        uint8_t intradc[6]; /* INTRA: raw 8-bit INTRADC codes (0xFF => 1024, else code*8);
                               0 = block dropped (zig-zag overflow, rle.rs:125-127), which then has nev 0 */
    } u;
} h263cu_mb;

/* Event unit, narrow form (default): bits 15..10 = RUN, bits 9..0 = LEVEL as a signed
 * 10-bit integer (never 0).  Wide form (H263CU_MB_WIDE, needed when some |LEVEL| of the MB
 * exceeds the 10-bit range, i.e. Sorenson 11-bit escapes): two units per event, first =
 * RUN, second = LEVEL as int16.  The device accumulates RUN into zig-zag positions,
 * dequantises and classifies (rle.rs:82-172).  The front end never emits a block whose
 * events push the zig-zag index past 63 (it drops such blocks, as the reference does);
 * in caller-built side info the device drops one the same way: the block stays Zero, the
 * intra DC included.  Caller-built side info is refused with H263CU_ERR_BAD_ARGUMENT when
 * a block holds more than 64 events (an intra block more than 63: the DC takes index 0),
 * or when an intra block with INTRADC code 0 (dropped) holds any event. */
typedef uint16_t h263cu_event;

/* ---- host front end (replaces H263Reader + the serial loop of
 *      H263State::decode_next_picture, h263/src/decoder/state.rs:142-427) ---------------- */
typedef struct h263cu_parser h263cu_parser;

/* H263State::new (state.rs:42-50): one parser per stream */
h263cu_parser* h263cu_parser_create(uint32_t decoder_options);
void h263cu_parser_destroy(h263cu_parser*);
/* The DecoderOption bits the parser was created with */
uint32_t h263cu_parser_options(const h263cu_parser*);
/* Seek: discard all stream state; the next picture must be an I picture (state.rs:134-137) */
void h263cu_parser_reset(h263cu_parser*);

/* H263State::parse_picture (state.rs:102-111): header only; fills width/height/mb_w/mb_h/
 * pic_type/pquant/flags/version/temporal_reference/n_mbs of *pic. Stateless. */
int h263cu_peek_picture(uint32_t decoder_options, const uint8_t* data, size_t len, h263cu_pic* pic);

/* Serial parse of one packet = one picture (one H263Reader::from_source(&packet[..]) per
 * picture).  Writes *pic, pic->n_mbs records to mbs[0..] and the event units to events[0..];
 * pic->first_mb / first_event are set to mb_base / ev_base and every record's `pic` field
 * to pic_index, so that many pictures can be packed into one step.  Transactional like the
 * reference (state.rs:120-137): on error the parser state is unchanged. */
int h263cu_parse_picture(h263cu_parser*, const uint8_t* data, size_t len, uint32_t stream,
                         uint16_t pic_index, uint32_t mb_base, uint32_t ev_base, h263cu_pic* pic,
                         h263cu_mb* mbs, uint32_t mb_cap, h263cu_event* events, uint32_t ev_cap);

/* Threaded parse of one time step: packet i belongs to parsers[i] / stream_ids[i] and
 * becomes picture i.  Pictures that fail to parse are reported in per_pic_err[i] (may be
 * NULL) and left out of the step (the remaining pictures are packed densely; *n_pics_out
 * counts them and pic_of_input[i] (may be NULL) gives the packed index or -1).
 * `threads` <= 0 selects std::thread::hardware_concurrency(). */
int h263cu_parse_step(h263cu_parser* const* parsers, const uint8_t* const* packets, const size_t* lens,
                      const uint32_t* stream_ids, uint32_t n, int threads, h263cu_pic* pics,
                      h263cu_mb* mbs, uint32_t mb_cap, h263cu_event* events, uint32_t ev_cap,
                      uint32_t* n_pics_out, uint32_t* n_mbs_out, uint32_t* n_units_out,
                      int* per_pic_err, int32_t* pic_of_input);

/* ---- test hooks: the front end's bit reader, VLC tables and block decoder as plain calls, so that the
 *      reference's own parser known-answer tests (reader.rs:448-559, macroblock.rs:551-1010, block.rs:757-2124)
 *      can be replayed on the product code.  Tables: 0 MCBPC_I, 1 MCBPC_P, 2 CBPY, 3 MVD, 4 TCOEF;
 *      out4 = {kind (0 valid, 1 stuffing, 2 invalid, 3 escape), a, b, c} as in csrc/vlc_codes.inc. ---- */
int h263cu_test_read_bits(const uint8_t* data, size_t len, size_t* bitpos, int nbits, int is_signed, int peek,
                          int64_t* value);
/* recognize_start_code (reader.rs:240-258): *skipped = stuffing bits before the code, -1 when there is none */
int h263cu_test_start_code(const uint8_t* data, size_t len, size_t bitpos, int* skipped);
int h263cu_test_read_vlc(int table, const uint8_t* data, size_t len, size_t* bitpos, int* out4);
/* decode_block (block.rs:670-755): *intradc_code = -1 when absent; run/level hold up to 64 events */
int h263cu_test_decode_block(const uint8_t* data, size_t len, size_t* bitpos, uint32_t decoder_options, int version,
                             int is_intra, int tcoef_present, int* intradc_code, int* n_events, uint8_t* run,
                             int16_t* level, int* overflow);

/* ---- device context ---------------------------------------------------------------- */
typedef struct h263cu_ctx h263cu_ctx;
typedef struct h263cu_step h263cu_step;

#define H263CU_OUT_RGBA 1u    /* produce RGBA (yuv::bt601::yuv420_to_rgba) for every picture */
#define H263CU_OUT_DEBLOCK 2u /* RGBA from deblocked planes: deblock::deblock(plane, width,
                                 QUANT_TO_STRENGTH[pquant]) per plane; the reference frames
                                 stay un-deblocked (deblock/src/lib.rs:1-2) */
/* Parse the macroblock layer on the GPU.  Accepted by h263cu_decode_step, h263cu_decode_step_device, _device_yuv,
 * _device_tensor, _device_tensor_fit, _device_tensor_filter and their h263cu_group_* forms; every other call that
 * takes out_flags ignores it.
 * - Split: the host keeps the stream state and the picture layer -- the picture header with the parser's previous
 *   format, the size, capacity and crop checks, and after the macroblock layer the reference checks of a picture with
 *   inter macroblocks (H263CU_ERR_UNCODED_IFRAME_BLOCKS, H263CU_ERR_REFERENCE_WOULD_ABORT).  The packets of the pictures
 *   that pass go to the device in one copy, and a kernel (one warp per picture) parses everything after each header:
 *   COD and stuffing, MCBPC, CBPY, DQUANT, MVD with median prediction, INTRADC, TCOEF with every escape form, the GOB
 *   resynchronisation stub, EOF and the uncoded padding after an early end.  Pictures that fail on the host never
 *   reach the device.
 * - Contract: the call's own, point for point -- the same per_pic_err codes, *n_decoded, transactional failure,
 *   capacity, crop and duplicate-id rules, and byte-identical outputs.  The records and events the kernels read are
 *   those h263cu_parse_step produces (h263cu_test_device_parse_step below checks this).
 * - The one difference: the call waits on the host for the parse kernel's per-picture results (16 bytes a picture),
 *   because the reference checks and the step's planning need each picture's outcome.  The parse writes into the side
 *   info ring slot once the kernels that read it two calls ago have finished, so the wait covers those kernels (and,
 *   through them, whatever they waited for on the caller's stream at that call) but never the previous call's
 *   kernels, nor work queued on the caller's stream since.  The pipeline is therefore one step shallower than with
 *   the host parse, whose upload waits for the same kernels on the copy stream without blocking the host.
 * - One capacity rule is stricter: a packet of 2^28 bytes or more fails the call with H263CU_ERR_CAPACITY before
 *   anything is parsed (bit positions are 32-bit on the device); with the host parse such a packet is parsed.
 * - Python: the decode_step* methods of BatchDecoder and DeviceGroup take parse="host" (the default) or
 *   parse="device" (this bit); any other value raises ValueError before any parser moves.
 * - The host parser still runs for calls without this bit; host and device steps may alternate on one context and
 *   one set of parsers. */
#define H263CU_PARSE_ON_DEVICE 4u

int h263cu_device_count(void);
/* Device memory for max_streams streams of up to max_width x max_height: two
 * reconstruction slots (current / reference) and two RGBA slots per stream. */
h263cu_ctx* h263cu_create(int device, uint32_t max_streams, uint32_t max_width, uint32_t max_height,
                          uint32_t flags, int* err);
void h263cu_destroy(h263cu_ctx*);
int h263cu_device_of(h263cu_ctx*);

/* Pinned host memory for side info / read-back buffers (cudaHostAlloc). */
void* h263cu_alloc_pinned(size_t bytes);
void h263cu_free_pinned(void* p);

/* Copy one step's side info into device memory (cudaMemcpyAsync on the context stream) and
 * keep it there: the "inputs resident in HBM" form used for kernel-only timing.
 * Side info handed in through h263cu_step_upload / h263cu_submit_step / h263cu_submit_step_readback need not come
 * from the library's parser, so it is checked on the host first: every record must lie in its picture's range, carry
 * that picture's index, sit at its raster position (mby * mb_w + mbx == index inside the picture) and keep its events
 * inside the picture's share of the event array, else H263CU_ERR_BAD_ARGUMENT.  H263CU_PICFLAG_HAS_INTER and
 * H263CU_PICFLAG_MV_IN_RANGE are derived from the records (set / cleared as needed), not taken on trust. */
h263cu_step* h263cu_step_upload(h263cu_ctx*, const h263cu_pic* pics, uint32_t n_pics, const h263cu_mb* mbs,
                                uint32_t n_mbs, const h263cu_event* events, uint32_t n_units, int* err);
void h263cu_step_free(h263cu_ctx*, h263cu_step*);
/* Reconstruct every picture of the step (async): the recon tail of decode_next_picture
 * (state.rs:419-485: gather + 3x idct_channel + reference bookkeeping) followed by the
 * requested outputs.  Each stream's "last picture" becomes the reference of its next one
 * (state.rs:72-78). */
int h263cu_step_run(h263cu_ctx*, h263cu_step*, uint32_t out_flags);
/* n resident steps as ONE CUDA graph.  A single stream's pictures are dependent launches of about ten microseconds
 * each (BASELINE.json configs[1]); captured into a graph they cost one launch call together.  The graph holds plane
 * addresses, so it is bound to the per-stream state it was built from: h263cu_graph_launch checks that every stream
 * the steps touch is where the capture assumed (plane slot, size, picture present), launches, and advances the
 * bookkeeping as the steps would have.  A graph over an even number of pictures per stream leaves the slots where they
 * started and can be launched again at once.  The steps must outlive the graph. */
typedef struct h263cu_graph h263cu_graph;
h263cu_graph* h263cu_graph_build(h263cu_ctx*, h263cu_step* const* steps, uint32_t n_steps, uint32_t out_flags, int* err);
int h263cu_graph_launch(h263cu_ctx*, h263cu_graph*);
void h263cu_graph_free(h263cu_ctx*, h263cu_graph*);
/* upload + run through an internal double-buffered ring (the streaming form) */
int h263cu_submit_step(h263cu_ctx*, const h263cu_pic* pics, uint32_t n_pics, const h263cu_mb* mbs,
                       uint32_t n_mbs, const h263cu_event* events, uint32_t n_units, uint32_t out_flags);
/* submit_step + asynchronous read-back of the RGBA pictures of this step into
 * host_rgba (pinned; picture i at i * 4*width*height when all pictures share one size,
 * else at rgba_offsets[i]); overlaps the copy with the next step's kernels.  Call
 * h263cu_sync before reading host_rgba. */
int h263cu_submit_step_readback(h263cu_ctx*, const h263cu_pic* pics, uint32_t n_pics, const h263cu_mb* mbs,
                                uint32_t n_mbs, const h263cu_event* events, uint32_t n_units,
                                uint32_t out_flags, uint8_t* host_rgba, const uint64_t* rgba_offsets);
/* Batched H263State::decode_next_picture (state.rs:138-489) from the bitstream: packet i is the next
 * picture of parsers[i] / stream_ids[i] (NULL: stream i).  The serial VLC parse runs on `threads`
 * host threads (h263cu_parse_step) into pinned staging owned by the context, the side info goes to
 * the device through the double-buffered ring, and the step is reconstructed asynchronously -- the
 * call returns as soon as the work is queued, so the parse of the next step overlaps this step's
 * kernels and copies.  Pictures that fail to parse are reported in per_pic_err[i] (may be NULL),
 * leave their stream untouched (the reference's transactional behaviour, state.rs:120-137) and are
 * left out of the step; *n_decoded (may be NULL) counts the rest.  A picture larger than the context is such a
 * per-picture error (H263CU_ERR_CAPACITY).  A stream id out of range or named twice fails the call as a whole
 * before anything is parsed, and the parsers advance only once the device stage has accepted the step: a call
 * that returns an error has changed no parser and no stream.  When host_rgba is not NULL the
 * RGBA picture of input i is copied to host_rgba + i * rgba_stride (tight rows of 4 * width bytes)
 * on the read-back stream; call h263cu_sync before reading it. */
int h263cu_decode_step(h263cu_ctx*, h263cu_parser* const* parsers, const uint8_t* const* packets, const size_t* lens,
                       const uint32_t* stream_ids, uint32_t n, int threads, uint32_t out_flags, uint8_t* host_rgba,
                       uint64_t rgba_stride, int* per_pic_err, uint32_t* n_decoded);

/* ---- device-resident output: RGBA straight into caller-owned device memory, no host read-back ----------------------
 * The recon kernel stores each macroblock's RGBA with one TMA tensor store; here the tensor map is a 3-D view of the
 * caller's buffer (bytes of a row, rows, slots) instead of the context's RGBA pool, and TMA's bounds clipping drops the
 * macroblock-rounded overhang at each slot's edge: the pictures land at their destination with no extra copy. */
typedef struct h263cu_device_rgba { /* 40 bytes */
    uint8_t* base;       /* device (or managed) memory of the context's device, 16-byte aligned */
    uint64_t row_pitch;  /* bytes between rows; multiple of 16, >= 4 * width, < 2^32 */
    uint64_t pic_stride; /* bytes between slots; multiple of 16, >= row_pitch * height, < 2^40 */
    uint32_t width, height; /* slot size: every picture of the call must fit in it */
    void* stream;        /* cudaStream_t of the consumer; NULL = the legacy default stream */
} h263cu_device_rgba;
/* h263cu_decode_step with the RGBA written into the caller's device buffer `out` instead of host memory.
 * - Behaviour is that of h263cu_decode_step: threaded parse, transactional failure, per-picture errors, duplicate and
 *   out-of-range stream ids, parsers that advance only once the device stage has accepted the step.  The one
 *   difference is where RGBA goes.  H263CU_OUT_RGBA is implied; out_flags may add H263CU_OUT_DEBLOCK.
 * - Layout: the RGBA of input i goes to slot i, base + i * pic_stride: rows of row_pitch bytes, tight R,G,B,A pixels,
 *   the picture at the slot's top-left.
 * - What is written: each picture's 4*w x h byte rectangle gets its RGBA, bit-exact.  Bytes inside the slot's
 *   4*width x height rectangle but outside the picture's own rectangle may be written.  Nothing else is ever written:
 *   not the row padding beyond 4*width, not the gap between slots, not the slot of an input that failed to parse.
 * - A picture larger than the slot is a per-picture H263CU_ERR_CAPACITY: left out, its stream untouched.
 * - Argument errors return H263CU_ERR_BAD_ARGUMENT before anything is parsed: a NULL out, a base that is not 16-byte
 *   aligned or that cudaPointerGetAttributes does not report as device or managed memory of the context's device,
 *   pitch or stride outside the rules above, a zero slot size.  A build without TMA RGBA stores (H263_RGBA_TMA=0, an
 *   A/B measurement variant) refuses every call the same way.
 * - Stream ordering, with no host synchronisation: the library's writes wait for all work queued on out->stream before
 *   the call (a buffer that earlier work still reads may be reused), and work queued on out->stream after the call
 *   sees the pictures.
 * - Context state: planes and reference bookkeeping advance as in h263cu_decode_step, so h263cu_read_yuv and the plane
 *   checksums keep working.  The context's RGBA ring is neither written nor waited on: h263cu_read_rgba returns
 *   H263CU_ERR_NO_PICTURE for the streams of such a step, as after a step without H263CU_OUT_RGBA.  Device and
 *   host read-back steps may alternate freely on one context. */
int h263cu_decode_step_device(h263cu_ctx*, h263cu_parser* const* parsers, const uint8_t* const* packets, const size_t* lens,
                              const uint32_t* stream_ids, uint32_t n, int threads, uint32_t out_flags, const h263cu_device_rgba* out,
                              int* per_pic_err, uint32_t* n_decoded);

/* ---- device-resident output: the decoded Y, Cb and Cr planes straight into caller-owned device memory ---------------
 * The planes DecodedPicture::as_luma / as_chroma_b / as_chroma_r hold (1.5 bytes per pixel, against 4 for RGBA), in
 * one of two layouts: I420 (three planes) or NV12 (a Y plane and one plane of interleaved CbCr pairs, the layout GPU
 * encoders take).  The recon kernel stores the plane words it already holds in registers; there is no colour
 * conversion and no TMA store, so any 4-byte aligned layout is accepted. */
#define H263CU_YUV_I420 0u /* plane[0] Y, plane[1] Cb, plane[2] Cr: DecodedPicture::as_luma / as_chroma_b / as_chroma_r */
#define H263CU_YUV_NV12 1u /* plane[0] Y, plane[1] CbCr pairs (Cb first); plane[2] must be all zero */
typedef struct h263cu_device_plane { /* 24 bytes */
    uint8_t* base;       /* device (or managed) memory of the context's device, 4-byte aligned */
    uint64_t row_pitch;  /* bytes between rows; multiple of 4, >= the plane's slot row bytes (below), < 2^32 */
    uint64_t pic_stride; /* bytes between slots; multiple of 4, >= row_pitch * the plane's slot rows, < 2^40 */
} h263cu_device_plane;
typedef struct h263cu_device_yuv { /* 96 bytes */
    h263cu_device_plane plane[3];
    uint32_t width, height; /* luma slot size: every picture of the call must fit in it; the chroma slot is
                               ceil(width / 2) x ceil(height / 2) samples */
    uint32_t format;        /* H263CU_YUV_I420 or H263CU_YUV_NV12 */
    uint32_t reserved;      /* 0 */
    void* stream;           /* cudaStream_t of the consumer; NULL = the legacy default stream */
} h263cu_device_yuv;
/* h263cu_decode_step with each decoded picture's planes written into the caller's device buffers `out`.
 * - Behaviour is that of h263cu_decode_step: threaded parse, transactional failure, per-picture errors, duplicate and
 *   out-of-range stream ids refused before the parse, parsers that advance only once the device stage has accepted the
 *   step.  No RGBA is produced: H263CU_OUT_RGBA is ignored.
 * - Layout: input i goes to slot i of each plane, plane[k].base + i * plane[k].pic_stride: rows of row_pitch bytes, the
 *   picture at the slot's top-left.  Slot row bytes: width (Y), ceil(width / 2) (I420 Cb and Cr), 2 * ceil(width / 2)
 *   (NV12 CbCr); slot rows: height (Y), ceil(height / 2) (chroma).  A picture of w x h samples fills w (Y),
 *   ceil(w / 2) (I420 chroma) or 2 * ceil(w / 2) (NV12 CbCr) bytes of each of its h (Y) or ceil(h / 2) (chroma) rows.
 * - What is written: each plane's picture rectangle, bit-exact.  Bytes inside the plane's slot rectangle but outside the
 *   picture may be written.  Nothing else is ever written: not the row padding, not the gaps between slots, not the
 *   slots of an input that failed.
 * - H263CU_OUT_DEBLOCK in out_flags: the planes written are deblock::deblock(plane, plane_width,
 *   QUANT_TO_STRENGTH[pquant]) of each plane, the planes the deblocked RGBA is converted from.  The context's reference
 *   planes stay un-deblocked.
 * - A picture larger than the slot is a per-picture H263CU_ERR_CAPACITY: left out, its stream untouched.
 * - Argument errors return H263CU_ERR_BAD_ARGUMENT before anything is parsed: a NULL out; an unknown format or a
 *   non-zero reserved; NV12 with a plane[2] that is not all zero; a zero slot size; a plane base, row pitch or slot
 *   stride that is not a multiple of 4 bytes; a pitch below the plane's slot row bytes or at or above 2^32; a stride
 *   below pitch * the plane's slot rows or at or above 2^40; a base that cudaPointerGetAttributes does not report as
 *   device or managed memory of the context's device.  Overlapping planes are not checked: they are the caller's error.
 * - Stream ordering and context state are those of h263cu_decode_step_device: the library's writes wait for the work
 *   queued on out->stream before the call, work queued on it after the call sees the planes, with no host
 *   synchronisation; planes and reference bookkeeping advance (h263cu_read_yuv and the checksums keep working); the
 *   RGBA ring is neither written nor waited on (h263cu_read_rgba returns H263CU_ERR_NO_PICTURE for the step's streams).
 *   Host, device RGBA and device plane steps may alternate freely on one context. */
int h263cu_decode_step_device_yuv(h263cu_ctx*, h263cu_parser* const* parsers, const uint8_t* const* packets, const size_t* lens,
                                  const uint32_t* stream_ids, uint32_t n, int threads, uint32_t out_flags, const h263cu_device_yuv* out,
                                  int* per_pic_err, uint32_t* n_decoded);

/* ---- device-resident output: resized, normalised RGB tensors [slot][channel][row][column] ---------------------------
 * The batch an ML pipeline takes: every picture of the call bilinearly resized to one width x height, as three channel
 * planes (R, G, B) of uint8, float32, float16 or bfloat16, each channel mapped by out = v * mul[c] + add[c].  One
 * kernel reads the just-reconstructed planes and writes the finished tensor; there is no RGBA and no intermediate.
 *
 * The output is defined exactly (IEEE fp32, round to nearest, no contraction).  For a decoded picture of w x h with
 * planes Y, Cb, Cr (deblocked on request) and an output of W x H:
 *  1. P_c(x, y) = channel c of yuv::bt601 of (Y[y][x], Cb[y/2][x/2], Cr[y/2][x/2]): an integer 0..255, exactly what
 *     yuv420_to_rgba produces at (x, y).
 *  2. per axis (x with w and W shown; y with h and H alike), torch's align_corners=False rule:
 *     scale = (float)w / (float)W;  s = max(0, scale * (X + 0.5f) - 0.5f);  x0 = (int)s;  x1 = x0 + (x0 < w - 1);
 *     l1 = s - (float)x0;  l0 = 1 - l1.
 *  3. v = ly0 * (lx0 * P(x0, y0) + lx1 * P(x1, y0)) + ly1 * (lx0 * P(x0, y1) + lx1 * P(x1, y1)), in that order.
 *  4. float dtypes: t = v * mul[c] + add[c] (two roundings), stored as f32 or converted round-to-nearest-even to f16 /
 *     bf16.  U8: min(255, (int)(v + 0.5f)).
 * At W = w and H = h every weight is 0 or 1: U8 is the RGB of yuv420_to_rgba exactly, floats are P * mul + add. */
#define H263CU_TENSOR_U8 0u
#define H263CU_TENSOR_F32 1u
#define H263CU_TENSOR_F16 2u
#define H263CU_TENSOR_BF16 3u
typedef struct h263cu_device_tensor { /* 88 bytes */
    void* base;             /* element [0][0][0][0]: device (or managed) memory of the context's device, aligned to the
                               element size */
    int64_t stride[4];      /* in elements: slot, channel (R, G, B), row, column; every stride > 0 */
    uint32_t width, height; /* output size, 1..16384: every picture of the call is resized to exactly this */
    uint32_t dtype;         /* H263CU_TENSOR_* */
    uint32_t reserved;      /* 0 */
    float mul[3], add[3];   /* per channel: out = v * mul[c] + add[c]; for U8 they must be 1 and 0 */
    void* stream;           /* cudaStream_t of the consumer; NULL = the legacy default stream */
} h263cu_device_tensor;
/* h263cu_decode_step with each decoded picture resized and converted into the caller's tensor `out`.
 * - Behaviour is that of h263cu_decode_step: threaded parse, transactional failure, per-picture errors, duplicate and
 *   out-of-range stream ids refused before the parse, parsers that advance only once the device stage has accepted the
 *   step.  No RGBA is produced: H263CU_OUT_RGBA is ignored.
 * - Layout: input i goes to slot i, element [i][c][y][x] at base + i * stride[0] + c * stride[1] + y * stride[2] +
 *   x * stride[3] elements.  Contiguous NCHW, channels-last (NHWC memory) and padded or sliced views are all strides.
 * - What is written: every element [slot][c][y][x] with c < 3, y < height, x < width of the slot of each decoded input.
 *   Nothing else is ever written: not the slots of inputs that failed, not any element outside those ranges.
 * - H263CU_OUT_DEBLOCK in out_flags: the planes resampled are the deblocked ones, those the deblocked RGBA is converted
 *   from.  The context's reference planes stay un-deblocked.
 * - There is no slot capacity: any picture size resizes to width x height.  A picture larger than the context is still
 *   a per-picture H263CU_ERR_CAPACITY.
 * - Argument errors return H263CU_ERR_BAD_ARGUMENT before anything is parsed: a NULL out; an unknown dtype or a non-zero
 *   reserved; a width or height of 0 or above 16384; a stride <= 0; a base not aligned to the element size; a slot
 *   extent ((width - 1) * stride[3] + (height - 1) * stride[2] + 2 * stride[1] + 1 elements) at or above 2^40 bytes; a
 *   non-finite mul or add, or U8 with a mul other than 1 or an add other than 0; a base that cudaPointerGetAttributes
 *   does not report as device or managed memory of the context's device.  Strides under which elements alias are not
 *   checked: they are the caller's error.
 * - Stream ordering and context state are those of h263cu_decode_step_device: the library's writes wait for the work
 *   queued on out->stream before the call, work queued on it after the call sees the tensor, with no host
 *   synchronisation; planes and reference bookkeeping advance; the RGBA ring is neither written nor waited on.  Host,
 *   device RGBA, device plane and device tensor steps may alternate freely on one context. */
int h263cu_decode_step_device_tensor(h263cu_ctx*, h263cu_parser* const* parsers, const uint8_t* const* packets, const size_t* lens,
                                     const uint32_t* stream_ids, uint32_t n, int threads, uint32_t out_flags,
                                     const h263cu_device_tensor* out, int* per_pic_err, uint32_t* n_decoded);

/* ---- device tensors with a fit: letterbox, resize-and-centre-crop, per-picture crop boxes ----------------------------
 * The geometry vision pipelines use instead of a stretch: torchvision's Resize(S) + CenterCrop((H, W)) (classifier
 * evaluation), a letterbox (detectors), and a crop box per picture resized to the output (RandomResizedCrop).  Each is
 * an integer crop, the resize of steps 2-3 above, then an integer pad or crop; the library works the geometry out per
 * picture from its decoded size.
 *
 * The definition, for input i with a decoded picture of w x h, its crop (cx, cy, cw, ch) (without crops: (0, 0, w, h))
 * and an output of W x H.  Geometry (64-bit integers, once per picture): a resized size (rw, rh) and a placement
 * (px, py), which may be negative:
 *  - STRETCH: rw = W, rh = H, px = py = 0.
 *  - LETTERBOX: when cw * H >= ch * W, rw = W and rh = max(1, (2 * ch * W + cw) / (2 * cw)) (ch * W / cw rounded half
 *    up); otherwise rh = H and rw = max(1, (2 * cw * H + ch) / (2 * ch)).  px = (W - rw) / 2, py = (H - rh) / 2, both
 *    floored: where ultralytics' LetterBox puts the picture.
 *  - CENTER_CROP with S = short_side: when cw <= ch, rw = S and rh = floor(S * ch / cw); otherwise rh = S and
 *    rw = floor(S * cw / ch) (torchvision's int(S * long / short)).  Per axis (x shown, y alike): if rw >= W,
 *    px = -anchor(rw - W) where anchor(d) is d / 2 rounded half to even (Python's round, as torchvision's centre crop
 *    anchors); otherwise px = (W - rw) / 2, floored (torchvision's left padding).
 * Value of output element (X, Y), with X' = X - px and Y' = Y - py:
 *  - inside the placed picture (0 <= X' < rw, 0 <= Y' < rh): v is steps 2-3 above at index (X', Y') with in = (cw, ch)
 *    and out = (rw, rh), so scale = (float)cw / (float)rw and x1 = x0 + (x0 < cw - 1), the samples read at
 *    P(cx + x, cy + y);
 *  - outside it: v = fill[c].
 *  Step 4 is unchanged for both: fill goes through mul / add like a pixel (U8: (int)(fill + 0.5f)).
 * So STRETCH without crops is exactly h263cu_decode_step_device_tensor's output, and for the float dtypes CENTER_CROP is
 * torchvision v2's resize(S, antialias=False) -> center_crop((H, W)) -> normalize on the 0-255 float RGB, with the
 * FMA-contracted coordinate caveat of step 2.  torchvision's Resize defaults to antialias=True, which this output does
 * not reproduce: h263cu_decode_step_device_tensor_filter below does. */
#define H263CU_FIT_STRETCH 0u     /* the (cropped) picture resized to width x height: h263cu_decode_step_device_tensor */
#define H263CU_FIT_LETTERBOX 1u   /* aspect kept, the whole (cropped) picture inside, centred, fill around it */
#define H263CU_FIT_CENTER_CROP 2u /* torchvision Resize(short_side) then CenterCrop((height, width)) */
typedef struct h263cu_tensor_crop { /* 16 bytes */
    uint32_t x, y, width, height;
} h263cu_tensor_crop;
typedef struct h263cu_tensor_fit { /* 32 bytes */
    uint32_t mode;                   /* H263CU_FIT_* */
    uint32_t short_side;             /* CENTER_CROP: 1..16384; other modes: 0 */
    float fill[3];                   /* per channel, on the 0..255 scale of P: finite, 0 <= fill <= 255 */
    uint32_t reserved;               /* 0 */
    const h263cu_tensor_crop* crops; /* NULL: every whole picture; else one per input, in the caller's order (host memory) */
} h263cu_tensor_fit;
/* h263cu_decode_step_device_tensor with the fit `fit`.
 * - What is written is unchanged: every element [slot][c][y][x] of each decoded input's slot, fill included, and
 *   nothing else ever.
 * - Argument errors return H263CU_ERR_BAD_ARGUMENT before anything is parsed: every rule of `out`; a NULL fit; an
 *   unknown mode; a non-zero reserved; a short_side outside 1..16384 with CENTER_CROP or non-zero without it; a fill
 *   that is not finite or lies outside [0, 255]; a crop of width or height 0; a crop whose x + width or y + height
 *   overflows 32 bits.
 * - A crop that does not lie inside its decoded picture (x + width > w or y + height > h) is a per-picture
 *   H263CU_ERR_BAD_ARGUMENT: the picture is left out, its stream untouched and its slot unwritten.  h263cu_peek_picture
 *   gives a packet's picture size before the call. */
int h263cu_decode_step_device_tensor_fit(h263cu_ctx*, h263cu_parser* const* parsers, const uint8_t* const* packets,
                                         const size_t* lens, const uint32_t* stream_ids, uint32_t n, int threads, uint32_t out_flags,
                                         const h263cu_device_tensor* out, const h263cu_tensor_fit* fit, int* per_pic_err,
                                         uint32_t* n_decoded);
/* The geometry above for one picture, as the library computes it: out4 = {rw, rh, px, py} of a crop of cw x ch under
 * `mode` / `short_side` into an output of width x height.  Not on any decode path (a test hook: tests pin it against
 * torchvision without a GPU).  Takes the same argument ranges as the call and returns H263CU_ERR_BAD_ARGUMENT outside
 * them. */
int h263cu_test_fit_geometry(uint32_t mode, uint32_t short_side, uint32_t cw, uint32_t ch, uint32_t width, uint32_t height,
                             int32_t* out4);
/* Test hook of H263CU_PARSE_ON_DEVICE: h263cu_parse_step's arguments and outputs (pics, records, events packed in
 * input order, per_pic_err, pic_of_input), produced by the device path of ctx -- host header parse, parse_mb kernel,
 * host finish -- instead of the host parser.  The parsers do not advance.  Not on any decode path. */
int h263cu_test_device_parse_step(h263cu_ctx* ctx, h263cu_parser* const* parsers, const uint8_t* const* packets, const size_t* lens,
                                  const uint32_t* stream_ids, uint32_t n, int threads, h263cu_pic* pics, h263cu_mb* mbs, uint32_t mb_cap,
                                  h263cu_event* events, uint32_t ev_cap, uint32_t* n_pics_out, uint32_t* n_mbs_out, uint32_t* n_units_out,
                                  int* per_pic_err, int32_t* pic_of_input);

/* ---- device tensors with a fit and an antialiased filter: torchvision's Resize defaults ------------------------------
 * torchvision's Resize(S) defaults to antialias=True on tensors, and timm / HF checkpoints often to bicubic, also
 * antialiased: a downscale reads every source sample under the filter widened by the scale, not just the two nearest.
 * A filter replaces steps 2-3 of the definition for the output elements inside the placed picture; step 1, the fit
 * geometry (rw, rh, px, py, crops, fill) and step 4 are those of h263cu_decode_step_device_tensor_fit.  The crop acts
 * as the whole picture, so taps are cut and renormalised at its edge (torchvision's resized_crop).
 *
 * Per axis (x with cw, rw and X' shown; y alike with ch, rh and Y'), IEEE fp32, round to nearest, no contraction, r = 1
 * for bilinear and 2 for bicubic:
 *   scale = (float)cw / (float)rw;  support = scale >= 1 ? (float)r * scale : (float)r;
 *   invscale = scale >= 1 ? 1 / scale : 1;  center = scale * ((float)X' + 0.5f);
 *   xmin = max((int)((center - support) + 0.5f), 0);  xsize = min((int)((center + support) + 0.5f), cw) - xmin;
 *   raw_j = filter((((float)(xmin + j) - center) + 0.5f) * invscale) for j < xsize;
 *   total = raw_0 + raw_1 + ... in ascending j, from 0;  w_j = total != 0 ? raw_j / total : raw_j.
 * ((int) truncates toward zero.)  filter is the triangle max(0, 1 - |t|) (computed as |t| < 1 ? 1 - |t| : 0) for
 * bilinear, and for bicubic Keys' cubic with a = -0.5 in torch's cubic_convolution1 / 2 order, x = |t|:
 *   x < 1: ((1.5 * x - 2.5) * x) * x + 1;  1 <= x < 2: ((-0.5 * x + 2.5) * x - 4) * x + 2;  else 0.
 * Separable, horizontal first, for each channel c:
 *   h(y) = wx_0 * P(cx + xmin + 0, cy + y) + wx_1 * P(cx + xmin + 1, cy + y) + ...  (ascending j: the first term is a
 *          product, every later step one multiply and one add);
 *   v = wy_0 * h(ymin + 0) + wy_1 * h(ymin + 1) + ...  (ascending k, alike).
 * Step 4 for these filters: U8 is max(0, min(255, (int)(v + 0.5f))) (bicubic overshoots: v may leave [0, 255]; for
 * v >= 0 this is the rule above); the float dtypes are not clamped, as torch's float path does not clamp.
 * Properties: at rw = cw every weight is exactly 0 or 1, so the filter is the identity on P, as steps 2-3 are (the AA
 * filters equal H263CU_FILTER_BILINEAR there); H263CU_FILTER_BILINEAR through this call is the fit call's output byte
 * for byte.
 *
 * Sources: ATen/native/cuda/UpSample.cuh (_compute_weights_span, _compute_weights, interpolate_aa_single_dim,
 * BilinearFilterFunctor, BicubicFilterFunctor) and ATen/native/UpSample.h (cubic_convolution1 / 2, aa_filter in the
 * CPU kernel).  torch's own CPU and CUDA kernels differ from each other in the last bits (the CPU kernel computes the
 * center and tap coordinate in double, the CUDA kernel associates the tap coordinate differently); on the 0-255 float
 * RGB this definition is within 8 ulp of 255 of torch's CPU F.interpolate(antialias=True) for bilinear and 32 for
 * bicubic (whose intermediates reach about 300), so the float dtypes are torchvision v2's resize(S, antialias=True) ->
 * center_crop -> normalize to that precision.  torch's uint8 antialias path is a different function (it clamps the
 * horizontal pass to bytes) and is not reproduced. */
#define H263CU_FILTER_BILINEAR 0u    /* steps 2-3: torch's antialias=False bilinear (the fit call's output) */
#define H263CU_FILTER_BILINEAR_AA 1u /* torch's bilinear with antialias=True (torchvision Resize's default) */
#define H263CU_FILTER_BICUBIC_AA 2u  /* torch's bicubic with antialias=True (a = -0.5) */
/* h263cu_decode_step_device_tensor_fit with the filter `filter` (H263CU_FILTER_*).  The contract is the fit call's
 * point for point (what is written, per-picture errors, a crop outside its picture as a per-picture
 * H263CU_ERR_BAD_ARGUMENT, stream ordering, context state); one more argument error is refused before the parse: an
 * unknown filter. */
int h263cu_decode_step_device_tensor_filter(h263cu_ctx*, h263cu_parser* const* parsers, const uint8_t* const* packets,
                                            const size_t* lens, const uint32_t* stream_ids, uint32_t n, int threads, uint32_t out_flags,
                                            const h263cu_device_tensor* out, const h263cu_tensor_fit* fit, uint32_t filter,
                                            int* per_pic_err, uint32_t* n_decoded);

/* ---- device motion fields: each picture's motion vectors, macroblock types and quantisers ---------------------------
 * The compressed-domain side information a model can use beside (or instead of) the pixels: motion vectors as cheap
 * optical flow, masks of skipped / intra macroblocks, quantiser maps.  One small kernel (motion_field_kernel) reads the
 * step's h263cu_mb records, already in device memory, and writes three dense grids per picture.
 *
 * Definition.  For decoded input i in slot s, let its picture have a macroblock grid of mb_w x mb_h and records
 * r[y][x] (raster order, h263cu_mb above).  For every slot cell (X, Y) with X < mb_width and Y < mb_height:
 *  - inside the picture (X < mb_w and Y < mb_h):
 *      mb_flags = r.flags & (H263CU_MB_INTER | H263CU_MB_FOURMV | H263CU_MB_CODED).  INTER is motion compensated,
 *        which includes COD=1 skipped macroblocks and the uncoded padding after an early end of the picture; CODED is
 *        COD=0; FOURMV is a coded INTER4V / INTER4V+Q macroblock.  H263CU_MB_WIDE is never exported.
 *      mb_quant = r.quant, the quantiser in force (state.rs:226-227); for an uncoded macroblock the one in force when
 *        it was reached.
 *      for k = 0..3 (Y0 Y1 Y2 Y3) the block (2X + (k & 1), 2Y + (k >> 1)) gets mv = r.mv[k] when INTER, else (0, 0):
 *        the decoded half-pel luma vectors after median prediction and wrap, the ones gather uses.
 *  - outside the picture (a smaller picture's remainder of the slot grid): mb_flags = H263CU_MOTION_OUTSIDE,
 *    mb_quant = 0, mv = (0, 0).
 * Sign convention: a vector points into the reference picture; for a disposable P picture that is the last
 * non-disposable picture of the stream.  Chroma vectors follow from the luma ones (average_sum_of_mvs). */
#define H263CU_MOTION_OUTSIDE 0x80u /* mb_flags of a slot cell outside the picture's macroblock grid */
typedef struct h263cu_device_motion { /* 120 bytes */
    int16_t* mv;              /* [slot][component: x, y][block row][block column], half-pel units; NULL: not written */
    int64_t mv_stride[4];     /* in elements, each > 0 */
    uint8_t* mb_flags;        /* [slot][mb row][mb column]; NULL: not written */
    int64_t flags_stride[3];  /* in elements, each > 0 */
    uint8_t* mb_quant;        /* [slot][mb row][mb column]; NULL: not written */
    int64_t quant_stride[3];  /* in elements, each > 0 */
    uint32_t mb_width, mb_height; /* slot grid in macroblocks, 1..255; the mv grid is 2*mb_width x 2*mb_height blocks */
    void* stream;             /* cudaStream_t of the consumer; NULL = the legacy default stream */
} h263cu_device_motion;
/* One pixel output to produce beside the motion fields: at most one of rgba / yuv / tensor is not NULL (none: motion
 * only).  rgba is h263cu_decode_step_device's output, yuv _device_yuv's, tensor _device_tensor's; with fit, tensor is
 * _device_tensor_fit's (filter 0) or _device_tensor_filter's (filter H263CU_FILTER_*). */
typedef struct h263cu_device_output { /* 40 bytes */
    const h263cu_device_rgba* rgba;
    const h263cu_device_yuv* yuv;
    const h263cu_device_tensor* tensor;
    const h263cu_tensor_fit* fit;  /* tensor only: NULL = the plain tensor call, else the fit / filter call */
    uint32_t filter;               /* tensor with fit: H263CU_FILTER_*; otherwise 0 */
    uint32_t reserved;             /* 0 */
} h263cu_device_output;
/* h263cu_decode_step with the motion fields of every decoded picture written into the caller's device buffers
 * `motion`, alone (pixels NULL) or beside one pixel output (pixels).
 * - Behaviour is that of h263cu_decode_step_device_tensor, point for point: threaded parse, transactional failure,
 *   per-picture errors, duplicate and out-of-range stream ids refused before the parse, parsers that advance only once
 *   the device stage has accepted the step.  H263CU_PARSE_ON_DEVICE is accepted.
 * - Layout: input i goes to slot i: mv element [i][c][by][bx] at mv + i * mv_stride[0] + c * mv_stride[1] +
 *   by * mv_stride[2] + bx * mv_stride[3] elements, mb_flags / mb_quant element [i][Y][X] alike with their strides.
 * - What is written: every element of each decoded input's slot grid (2 x 2*mb_height x 2*mb_width vectors,
 *   mb_height x mb_width flags and quantisers) of each output whose base is not NULL.  Nothing else is ever written: no
 *   stride padding, no gaps between slots, not the slot of an input that failed.
 * - A picture whose macroblock grid exceeds mb_width x mb_height is a per-picture H263CU_ERR_CAPACITY: left out, its
 *   stream untouched.  With a pixel output the capacity is the smaller of the two outputs' limits.
 * - With a pixel output, that output is byte-identical to the same call without motion, and out_flags means what it
 *   means for that call.  With pixels == NULL the step reconstructs as a step without outputs: H263CU_OUT_RGBA and
 *   H263CU_OUT_DEBLOCK are ignored.
 * - Stream ordering, with no host synchronisation: the library's writes wait for the work queued on motion->stream
 *   (and on the pixel output's stream) before the call, and work queued on either stream after the call sees every
 *   output.  Planes and reference bookkeeping advance as in h263cu_decode_step_device.
 * - Argument errors return H263CU_ERR_BAD_ARGUMENT before anything is parsed: a NULL motion; all three bases NULL; an
 *   mb_width or mb_height of 0 or above 255; a stride <= 0 of an output that is written; an mv base that is not 2-byte
 *   aligned; a slot extent at or above 2^40 bytes (mv: ((2*mb_width - 1) * mv_stride[3] + (2*mb_height - 1) *
 *   mv_stride[2] + mv_stride[1] + 1) * 2 bytes; flags and quant: (mb_width - 1) * stride[2] + (mb_height - 1) *
 *   stride[1] + 1 bytes); a base that cudaPointerGetAttributes does not report as device or managed memory of the
 *   context's device; in pixels: more than one output, a fit or a non-zero filter without tensor, a non-zero filter
 *   without fit, a non-zero reserved, an unknown filter, and every rule of the chosen output.  Strides under which
 *   elements alias, and outputs that overlap, are the caller's error.
 * - Not offered: motion output for H263State, graphs and caller-built side info.  The prediction residual comes from
 *   h263cu_decode_step_device_residual below, beside these fields or alone. */
int h263cu_decode_step_device_motion(h263cu_ctx*, h263cu_parser* const* parsers, const uint8_t* const* packets, const size_t* lens,
                                     const uint32_t* stream_ids, uint32_t n, int threads, uint32_t out_flags,
                                     const h263cu_device_motion* motion, const h263cu_device_output* pixels, int* per_pic_err,
                                     uint32_t* n_decoded);

/* ---- device prediction residuals: each picture's planes minus its motion-compensated prediction --------------------
 * The third input of compressed-domain video models (CoViAR and its descendants) beside the I picture's pixels and the
 * motion vectors.  One kernel (residual_kernel) reads the step's decoded planes, the stream's reference planes and the
 * step's h263cu_mb records, all still in device memory after the step, and writes three int16 planes per picture.
 *
 * Definition.  For decoded input i in slot s, let its picture be w x h, cw = ceil(w/2), ch = ceil(h/2), and cur its
 * decoded planes BEFORE any deblocking (the planes h263cu_read_yuv and h263cu_decode_step_device_yuv without
 * H263CU_OUT_DEBLOCK return; references are never deblocked either).  pred is what the reference's gather
 * (gather.rs:140-204) writes into the new picture before the inverse transform adds to it:
 *  - inside an INTER macroblock (r.flags & H263CU_MB_INTER: this includes COD=1 skips and the uncoded padding after an
 *    early end of the picture): luma sample (x, y) is gather_block (gather.rs:47-126) of the reference luma with vector
 *    r.mv[k], k = 2 * ((y & 15) >= 8) + ((x & 15) >= 8); chroma sample (x, y) is gather_block of the reference Cb / Cr
 *    with the vector (average_sum_of_mvs(sum of the four mv.x), average_sum_of_mvs(sum of the four mv.y))
 *    (types.rs:759-768).  Every reference read is clamped to the reference's true w x h (cw x ch) as read_sample does
 *    (gather.rs:16-31); half-pel samples are (a + b + 1) / 2 and (s00 + s10 + s01 + s11 + 2) / 4.  The reference is the
 *    stream's last non-disposable picture, the one the picture is predicted from.
 *  - everywhere else (intra macroblocks, every macroblock of an I picture) pred is 0: the reference zero-fills the new
 *    picture (picture.rs:39-58) and gather skips those macroblocks.
 * Output (int16): Y[s][y][x] = cur_Y(x, y) - pred_Y(x, y) for x < w, y < h; Cb and Cr alike for x < cw, y < ch; 0 for
 * every other element of the slot rectangle (width x height for Y, ceil(width/2) x ceil(height/2) for Cb and Cr).
 * Hence: values lie in [-255, 255]; cur = pred + residual exactly; the residual is 0 on every uncoded INTER macroblock
 * and equals the samples on intra macroblocks and I pictures.  It is the effective residual, the inverse transform's
 * output after both of the reference's clamps, not the raw transform output. */
typedef struct h263cu_device_residual { /* 112 bytes */
    int16_t* y;            /* [slot][row][column]; NULL: not written */
    int64_t y_stride[3];   /* in elements, each > 0 */
    int16_t* cb;           /* [slot][row][column]; NULL: not written */
    int64_t cb_stride[3];  /* in elements, each > 0 */
    int16_t* cr;           /* [slot][row][column]; NULL: not written */
    int64_t cr_stride[3];  /* in elements, each > 0 */
    uint32_t width, height; /* the luma slot, 1..16384; the chroma slot is ceil(width/2) x ceil(height/2) */
    void* stream;          /* cudaStream_t of the consumer; NULL = the legacy default stream */
} h263cu_device_residual;
/* h263cu_decode_step with the prediction residual of every decoded picture written into the caller's device planes
 * `residual`, alone or beside the motion fields (motion, NULL: none) and / or one pixel output (pixels, NULL: none):
 * the pixels, the motion vectors and the residual of one parse.
 * - Behaviour is that of h263cu_decode_step_device_motion, point for point: threaded parse, transactional failure,
 *   per-picture errors, parsers that advance only once the device stage has accepted the step; H263CU_PARSE_ON_DEVICE
 *   is accepted.
 * - Layout: input i goes to slot i: Y element [i][y][x] at y + i * y_stride[0] + y * y_stride[1] + x * y_stride[2]
 *   elements, Cb and Cr alike with their strides.  The motion fields and the pixel output use the same slots.
 * - What is written: every element of each decoded input's slot rectangles of each plane whose base is not NULL.
 *   Nothing else is ever written: no stride padding, no gaps between slots, not the slot of an input that failed.
 * - A picture larger than width x height is a per-picture H263CU_ERR_CAPACITY: left out, its stream untouched.  With
 *   motion and / or pixels the capacity is the smallest of the outputs' limits.
 * - The pixel output and the motion fields are byte-identical to the same call without residual, and out_flags means
 *   what it means for that call; with pixels == NULL the step reconstructs as a step without outputs (H263CU_OUT_RGBA
 *   and H263CU_OUT_DEBLOCK are ignored).
 * - Stream ordering, with no host synchronisation: the library's writes wait for the work queued on residual->stream
 *   (and on the motion and pixel output's streams) before the call, and work queued on any of them after the call sees
 *   every output.
 * - Argument errors return H263CU_ERR_BAD_ARGUMENT before anything is parsed: the rules of
 *   h263cu_decode_step_device_motion for motion (when not NULL) and pixels, and a NULL residual; all three bases NULL;
 *   a width or height of 0 or above 16384; a stride <= 0 of a plane that is written; a base that is not 2-byte aligned;
 *   a slot extent at or above 2^40 bytes (((W - 1) * stride[2] + (H - 1) * stride[1] + 1) * 2 bytes, W x H the plane's
 *   slot); a base that cudaPointerGetAttributes does not report as device or managed memory of the context's device.
 *   Strides under which elements alias, and outputs that overlap, are the caller's error.
 * - Not offered: residual output for H263State, graphs and caller-built side info; the raw inverse transform output;
 *   residuals accumulated over several pictures; other element types. */
int h263cu_decode_step_device_residual(h263cu_ctx*, h263cu_parser* const* parsers, const uint8_t* const* packets, const size_t* lens,
                                       const uint32_t* stream_ids, uint32_t n, int threads, uint32_t out_flags,
                                       const h263cu_device_residual* residual, const h263cu_device_motion* motion,
                                       const h263cu_device_output* pixels, int* per_pic_err, uint32_t* n_decoded);
int h263cu_sync(h263cu_ctx*);
/* Waits for the RGBA read-back of an earlier step only: age 0 = the step submitted last with a read-back, 1 = the one
 * before it (the read-back ring is two deep).  Lets a caller consume picture t while picture t + 1 is in flight: the
 * pipelined form of decode_next_picture + yuv420_to_rgba for ONE stream (api.H263State(pipelined=True)). */
int h263cu_readback_wait(h263cu_ctx*, uint32_t age);

/* ---- one process, several GPUs (streams shard by stream, no exchange between devices) ------------------------------
 * A group owns one context per listed device and feeds them all from ONE shared pool of parser threads: the pictures
 * of device d are parsed on all threads and queued on d, then the threads move on to d + 1 while d reconstructs and
 * copies back.  Global stream s lives on device s % n_devices in slot s / n_devices.  With host_rgba != NULL the RGBA
 * of stream s lands at host_rgba + ((s % n_devices) * streams_per_device + s / n_devices) * rgba_stride (device-major:
 * each device's pictures are contiguous).  Errors and the transactional behaviour are those of h263cu_decode_step. */
typedef struct h263cu_group h263cu_group;
h263cu_group* h263cu_group_create(const int* devices, uint32_t n_devices, uint32_t streams_per_device, uint32_t max_width,
                                  uint32_t max_height, int threads, int* err);
void h263cu_group_destroy(h263cu_group*);
uint32_t h263cu_group_size(const h263cu_group*);
h263cu_ctx* h263cu_group_ctx(h263cu_group*, uint32_t index);
int h263cu_group_decode_step(h263cu_group*, h263cu_parser* const* parsers, const uint8_t* const* packets, const size_t* lens,
                             const uint32_t* stream_ids, uint32_t n, uint32_t out_flags, uint8_t* host_rgba, uint64_t rgba_stride,
                             int* per_pic_err, uint32_t* n_decoded);
/* h263cu_decode_step_device for a group: outs holds one buffer per device (outs[d] on the group's device d), and
 * global stream s goes to slot s / n_devices of outs[s % n_devices] (the device-major placement above).  Every
 * buffer is checked before any device parses. */
int h263cu_group_decode_step_device(h263cu_group*, h263cu_parser* const* parsers, const uint8_t* const* packets, const size_t* lens,
                                    const uint32_t* stream_ids, uint32_t n, uint32_t out_flags, const h263cu_device_rgba* outs,
                                    int* per_pic_err, uint32_t* n_decoded);
/* h263cu_decode_step_device_yuv for a group, with the placement of h263cu_group_decode_step_device: outs holds one
 * set of planes per device, global stream s goes to slot s / n_devices of outs[s % n_devices], and every device's
 * planes are checked before any device parses. */
int h263cu_group_decode_step_device_yuv(h263cu_group*, h263cu_parser* const* parsers, const uint8_t* const* packets, const size_t* lens,
                                        const uint32_t* stream_ids, uint32_t n, uint32_t out_flags, const h263cu_device_yuv* outs,
                                        int* per_pic_err, uint32_t* n_decoded);
/* h263cu_decode_step_device_tensor for a group, with the placement of h263cu_group_decode_step_device: outs holds one
 * tensor per device, global stream s goes to slot s / n_devices of outs[s % n_devices], and every device's tensor is
 * checked before any device parses. */
int h263cu_group_decode_step_device_tensor(h263cu_group*, h263cu_parser* const* parsers, const uint8_t* const* packets,
                                           const size_t* lens, const uint32_t* stream_ids, uint32_t n, uint32_t out_flags,
                                           const h263cu_device_tensor* outs, int* per_pic_err, uint32_t* n_decoded);
/* h263cu_decode_step_device_tensor_fit for a group, with the placement of h263cu_group_decode_step_device_tensor:
 * fit->crops[i] (when not NULL) belongs to input i as passed, whichever device its stream lives on. */
int h263cu_group_decode_step_device_tensor_fit(h263cu_group*, h263cu_parser* const* parsers, const uint8_t* const* packets,
                                               const size_t* lens, const uint32_t* stream_ids, uint32_t n, uint32_t out_flags,
                                               const h263cu_device_tensor* outs, const h263cu_tensor_fit* fit, int* per_pic_err,
                                               uint32_t* n_decoded);
/* h263cu_decode_step_device_tensor_filter for a group, with the placement and crops of
 * h263cu_group_decode_step_device_tensor_fit. */
int h263cu_group_decode_step_device_tensor_filter(h263cu_group*, h263cu_parser* const* parsers, const uint8_t* const* packets,
                                                  const size_t* lens, const uint32_t* stream_ids, uint32_t n, uint32_t out_flags,
                                                  const h263cu_device_tensor* outs, const h263cu_tensor_fit* fit, uint32_t filter,
                                                  int* per_pic_err, uint32_t* n_decoded);
/* h263cu_decode_step_device_motion for a group, with the placement of h263cu_group_decode_step_device: motions holds
 * one set of motion buffers per device, pixels (NULL: motion only) one pixel output per device, and global stream s
 * goes to slot s / n_devices of both on device s % n_devices.  Every pixels[d] names the same kind of output with the
 * same fit pointer and filter; fit->crops[i] (when not NULL) belongs to input i as passed.  Every device's buffers are
 * checked before any device parses. */
int h263cu_group_decode_step_device_motion(h263cu_group*, h263cu_parser* const* parsers, const uint8_t* const* packets,
                                           const size_t* lens, const uint32_t* stream_ids, uint32_t n, uint32_t out_flags,
                                           const h263cu_device_motion* motions, const h263cu_device_output* pixels,
                                           int* per_pic_err, uint32_t* n_decoded);
/* h263cu_decode_step_device_residual for a group, with the placement and checks of
 * h263cu_group_decode_step_device_motion: residuals holds one set of residual planes per device, motions (NULL: none)
 * one set of motion buffers per device, pixels (NULL: none) one pixel output per device. */
int h263cu_group_decode_step_device_residual(h263cu_group*, h263cu_parser* const* parsers, const uint8_t* const* packets,
                                             const size_t* lens, const uint32_t* stream_ids, uint32_t n, uint32_t out_flags,
                                             const h263cu_device_residual* residuals, const h263cu_device_motion* motions,
                                             const h263cu_device_output* pixels, int* per_pic_err, uint32_t* n_decoded);
int h263cu_group_sync(h263cu_group*);

/* DecodedPicture accessors (h263/src/decoder/picture.rs:60-142): tight row-major planes,
 * chroma = ceil(w/2) x ceil(h/2).  Synchronise the context first. */
int h263cu_stream_info(h263cu_ctx*, uint32_t stream, uint32_t* width, uint32_t* height, uint32_t* pic_type,
                       uint32_t* pquant, uint32_t* temporal_reference);
/* width << 16 | height of the stream's last picture, 0 when it has none: the cheap form of h263cu_stream_info */
uint32_t h263cu_stream_dims(h263cu_ctx*, uint32_t stream);
int h263cu_read_yuv(h263cu_ctx*, uint32_t stream, uint8_t* y, uint8_t* cb, uint8_t* cr);
/* RGBA of the stream's last picture (4*width*height bytes, R,G,B,A); requires that the
 * last step ran with H263CU_OUT_RGBA. */
int h263cu_read_rgba(h263cu_ctx*, uint32_t stream, uint8_t* rgba);
/* Position-weighted 64-bit checksums computed on the device over the tight planes /
 * RGBA of the last picture of each listed stream:
 *   sum_i (byte[i] + 1) * ((uint32)(i * 2654435761) | 1)   (mod 2^64)
 * out = n x {y, cb, cr, rgba}. */
int h263cu_checksums(h263cu_ctx*, const uint32_t* streams, uint32_t n, uint64_t* out4);

/* CUDA-event timing on the context stream (used by bench.py). */
int h263cu_timer_start(h263cu_ctx*);
int h263cu_timer_stop(h263cu_ctx*, float* milliseconds);
/* Number of kernel launches issued by this context so far. */
uint64_t h263cu_launch_count(h263cu_ctx*);
/* How many of the reconstruction launches took the tiled kernel (the fast path: references with a
 * replicated border; any picture size) rather than the generic warp-per-macroblock kernel. */
uint64_t h263cu_tiled_launch_count(h263cu_ctx*);
/* Host time spent inside h263cu_decode_step since the last reset: the bitstream parse, and everything else (staging,
 * driver calls).  Reported beside the device time (the parse is the host's share of decode_next_picture). */
int h263cu_host_times(h263cu_ctx*, double* parse_seconds, double* other_seconds, uint64_t* calls, int reset);
/* Per-kernel timing: when enabled, every recon / deblock launch is bracketed by CUDA events
 * on the launching stream.  h263cu_profile_read synchronises, accumulates the elapsed times
 * since the last read into ms[0] (recon) / ms[1] (deblock+rgba) and the launch counts into
 * launches[0..1], and resets. */
int h263cu_profile_enable(h263cu_ctx*, int enable);
int h263cu_profile_read(h263cu_ctx*, double* ms2, uint64_t* launches2);

/* ---- stateless drop-ins for the sibling crates (host buffers in, host buffers out) ---- */
/* yuv::bt601::yuv420_to_rgba(y, chroma_b, chroma_r, y_width) -> Vec<u8>
 * (yuv/src/bt601.rs:105-196).  rgba_out holds 4*y_len bytes. y_len == 0 is a no-op. */
int h263cu_yuv420_to_rgba(const uint8_t* y, const uint8_t* chroma_b, const uint8_t* chroma_r, size_t y_len,
                          size_t y_width, uint8_t* rgba_out);
/* deblock::deblock::deblock(data, width, strength) -> Vec<u8> (deblock/src/deblock.rs:305-315) */
int h263cu_deblock(const uint8_t* data, size_t len, size_t width, uint8_t strength, uint8_t* out);
/* deblock::deblock::QUANT_TO_STRENGTH (deblock/src/deblock.rs:5-8) */
extern const uint8_t h263cu_quant_to_strength[32];

/* ---- FLV container feed (the caller side of H263Reader::from_source(&packet[..]): one reader per FLV
 *      video tag; Sorenson Spark is FLV video codec 2, one picture per tag) ------------------------- */
typedef struct h263cu_flv_packet { /* 24 bytes */
    uint64_t offset;       /* of the picture packet inside the FLV buffer (past the 1-byte video header) */
    uint32_t size;         /* bytes of the picture packet */
    uint32_t timestamp_ms; /* 32-bit tag timestamp (extended byte included) */
    uint8_t frame_type;    /* 1 key, 2 inter, 3 disposable inter */
    uint8_t codec_id;      /* always 2 (Sorenson H.263): other video codecs are skipped */
    uint16_t reserved;
    uint32_t reserved2;
} h263cu_flv_packet;

/* Zero-copy scan of an FLV byte stream: lists its H.263 video packets in file order.  Returns how many
 * there are (fill up to `cap` of them; call with cap = 0 to count) or a negative error when the buffer
 * is not FLV.  A buffer that ends inside a tag (streaming input) ends the scan at the last complete tag.
 * Audio, script, other-codec and video-info tags are skipped and counted in *n_other_tags (may be NULL). */
int64_t h263cu_flv_scan(const uint8_t* data, size_t len, h263cu_flv_packet* out, size_t cap, uint32_t* n_other_tags);
/* The matching muxer for generated streams (tests, examples): wraps n picture packets (as laid out by
 * h263cu_synth_stream) into an FLV byte stream, one video tag per picture at i * ms_per_picture;
 * frame_types may be NULL (first = key, rest = inter); filler_every > 0 adds an audio and a script tag
 * before every filler_every-th picture.  Returns the bytes needed / written, or a negative error. */
int64_t h263cu_flv_mux(const uint8_t* packets, const uint64_t* pkt_off, const uint32_t* pkt_len, const uint8_t* frame_types,
                       uint32_t n, uint32_t ms_per_picture, uint32_t filler_every, uint8_t* out, size_t cap);

/* The synthetic stream generator lives in its own library (include/h263synth.h, libh263synth.so): it is test and
 * benchmark tooling, not part of the decode path. */

#ifdef __cplusplus
}
#endif
#endif /* H263CU_H */
