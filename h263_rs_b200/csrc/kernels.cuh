// kernels.cuh -- device-side data structures and launch wrappers shared by kernels.cu
// and context.cu.
#pragma once
#include <cuda.h>  // CUtensorMap (types only: the driver is reached through cudaGetDriverEntryPoint)
#include <cuda_runtime.h>
#include <stdint.h>

#include "../../include/h263cu.h"
#include "parse_mb.h"

namespace h263dev {

// Device-side picture descriptor, built by the host for every picture of a step when the
// step is run (plane slots toggle per stream, so pointers are only known then).
// The two chroma planes of a picture are stored INTERLEAVED (CbCr pairs, like NV12): sample
// (x, y) of Cb sits at cur[1][y * pitch_c + 2 * x], of Cr one byte further (cur[2] == cur[1] + 1).
struct PicDev {
    uint8_t* cur[3];        // Y, Cb, Cr planes being reconstructed (Cb / Cr: element step CHROMA_STEP)
    const uint8_t* ref[3];  // reference planes (previous picture of the stream); may be null
    uint8_t* rgba;          // RGBA output (null when not requested)
    uint32_t first_event;   // offset of the picture's events in the step's event array
    uint32_t rgba_pitch;    // bytes
    uint16_t w, h;          // true luma dimensions
    uint16_t cw, ch;        // true chroma dimensions = ceil(w/2), ceil(h/2)
    uint16_t pitch_y, pitch_c;  // bytes per row of the luma plane / of the interleaved chroma plane
    uint8_t strength;       // QUANT_TO_STRENGTH[pquant]
    uint8_t flags;
    uint8_t pad[2];
    // the same planes as 32-bit offsets from the context's pools (tiled kernel): interior origin
    // of the Y plane in 4-byte units from y_pool, of the CbCr plane in 4-byte units from c_pool;
    // rgba_row0 = first row of the RGBA picture in the RGBA pool (rows of rgba_pitch bytes); with output into a
    // caller-owned buffer (OUT_DEV_RGBA / OUT_YUV below) it is the picture's slot << 12 instead
    uint32_t cur_y4, cur_c4, ref_y4, ref_c4, rgba_row0;
    uint32_t out_slot;  // OUT_TENSOR: the picture's slot in the caller's tensor (rgba_row0 >> 12 is its scratch slot)
};
constexpr int CHROMA_STEP = 2;  // bytes between horizontally adjacent samples of one chroma plane

// Pool base pointers of a context: kernel parameters of the tiled kernel (uniform registers),
// so that per-macroblock state in shared memory can be 32-bit offsets instead of pointers.
struct Pools {
    uint8_t* y;
    uint8_t* c;  // interleaved CbCr planes
    uint8_t* rgba;
    uint32_t pitch_y, pitch_c, rgba_pitch;  // row pitches shared by every plane of the context (bytes)
};

// Where the output of a step goes: the context's RGBA pool, RGBA into a caller-owned buffer, or the picture's planes
// into caller-owned buffers (h263cu_decode_step_device_yuv; no RGBA at all).  OUT_TENSOR (h263cu_decode_step_device_tensor)
// is a context-side mode only: the recon kernel runs as for a step without RGBA and resample_rgb_kernel writes the output.
enum { OUT_POOL = 0, OUT_DEV_RGBA = 1, OUT_YUV = 2, OUT_TENSOR = 3 };
// The caller's planes of OUT_YUV (a kernel parameter, the same for every picture of a step): the planes of the picture
// in slot s start at base[k] + s * stride[k], rows pitch[k] bytes apart.  nv12: base[1] holds CbCr pairs and base[2] is
// unused; else base[1] / base[2] hold Cb / Cr.  All bases, pitches and strides are multiples of 4 bytes.
struct YuvDst {
    uint8_t* base[3];
    uint64_t stride[3];
    uint32_t pitch[3];
    uint32_t nv12;
};
// Y / chroma rows of plane k of slot `slot`
__host__ __device__ __forceinline__ uint8_t* yuv_row(const YuvDst& d, int k, uint32_t slot, uint32_t row) {
    return d.base[k] + (size_t)slot * d.stride[k] + (size_t)row * d.pitch[k];
}

// Fused reconstruction of every macroblock of a step: inverse RLE + dequant + classify +
// IDCT + motion compensation + add/clamp -> planes, and BT.601 RGBA when `emit_rgba`.
// tiled != 0 selects recon_tile_kernel (padded reference planes), else the generic warp-per-macroblock
// recon_mb_kernel.
// tiled: 1 = every picture is a multiple of 16 in size, 2 = some are not (edge fix-up instantiation).
// wide_mv: some picture of the step may hold vectors beyond [-32, 31] half-pel units (no H263CU_PICFLAG_MV_IN_RANGE).
// rgba_map: TMA tensor map the tiled kernel stores RGBA through.  out = OUT_POOL: the context's RGBA pool (2-D, rows of
// rgba_pitch bytes, box 64 bytes x 16 rows); out = OUT_DEV_RGBA: a caller-owned buffer (3-D: bytes, rows, slots; box
// 64 x 16 x 1), the PicDev.rgba_row0 of each picture holding its slot << 12.
// out = OUT_YUV: with emit_rgba, the planes of every picture whose PicDev.rgba is not null also go to `yuv` (slot in
// PicDev.rgba_row0 >> 12), cut to the picture; rgba_map is unused.  yuv may be null for the other modes.
void launch_recon(const PicDev* pics, const h263cu_mb* mbs, const h263cu_event* events, uint32_t n_mbs,
                  int emit_rgba, int tiled, int wide_mv, const Pools& pools, const CUtensorMap* rgba_map, int out,
                  const YuvDst* yuv, cudaStream_t stream);
// recon_tile.cu
void launch_recon_tile(const PicDev* pics, const h263cu_mb* mbs, const h263cu_event* events, uint32_t n_mbs,
                       int emit_rgba, int unaligned, int wide_mv, const Pools& pools, const CUtensorMap* rgba_map,
                       int out, const YuvDst* yuv, cudaStream_t stream);
// how the tiled kernel stores RGBA: 1 = TMA tensor stores from a shared-memory tile (the build default),
// 0 = direct global stores (build variant for A/B measurements)
int recon_tile_uses_tma();

// Plane padding (bytes / rows) reserved around every reconstruction plane: the tiled kernel
// replicates 16 luma pixels / 8 CbCr pairs (16 bytes either way) into it; the extra columns keep
// the interior origin 32 B aligned and absorb aligned-word over-reads.
constexpr int PAD_Y_COLS = 32, PAD_Y_ROWS = 16, PAD_C_COLS = 32, PAD_C_ROWS = 8;

// Deblocking post-filter (per plane, per picture) fused with the RGBA conversion, or with yuv != null the plane-output
// form: the deblocked planes of every picture whose PicDev.rgba is not null go to `yuv` (slot in PicDev.rgba_row0 >> 12)
// instead, cut to the picture.  grid = (max tiles per picture, n_pics).
void launch_deblock_rgba(const PicDev* pics, uint32_t n_pics, uint32_t max_w, uint32_t max_h, const YuvDst* yuv,
                         cudaStream_t stream);
// deblock_tile.cu: the register-resident form for pictures whose sizes are multiples of 16
void launch_deblock_rgba_tile(const PicDev* pics, uint32_t n_pics, uint32_t max_w, uint32_t max_h, const YuvDst* yuv,
                              cudaStream_t stream);

// The caller's tensor of OUT_TENSOR (h263cu_device_tensor, checked): element [slot][c][y][x] at
// base + slot * stride[0] + c * stride[1] + y * stride[2] + x * stride[3] elements of `dtype` (H263CU_TENSOR_*).
struct TensorDst {
    void* base;
    int64_t stride[4];
    uint32_t width, height;
    float mul[3], add[3];
};
// Bilinear resize + BT.601 + per-channel affine map of every picture of a step into `dst`: picture i (pics[i]) goes to
// slot pics[i].out_slot.  It reads the picture's planes cur[0] / cur[1] (pitch_y / pitch_c), or with src != null the
// NV12 planes of slot i of `src` (the deblocked copies).  grid = (output tiles, n_pics).
// fit != null: the fit form (h263cu_decode_step_device_tensor_fit): picture i is read from its crop box and placed by
// fit->geo[i] (device memory, one record per picture of the step), fill outside the placed picture.
struct FitGeom {  // include/h263cu.h: crop (cx, cy, cw, ch), resized size (rw, rh), placement (px, py)
    int32_t cx, cy, cw, ch, rw, rh, px, py;
};
struct FitArgs {
    const FitGeom* geo;
    float fill[3];
};
void launch_resample_rgb(const PicDev* pics, uint32_t n_pics, const YuvDst* src, const TensorDst& dst, uint32_t dtype,
                         const FitArgs* fit, cudaStream_t stream);
// resample_filter.cu: the fit form with an antialiased filter (h263cu_decode_step_device_tensor_filter, `filter` =
// H263CU_FILTER_BILINEAR_AA or H263CU_FILTER_BICUBIC_AA), same arguments and placement as launch_resample_rgb's fit form.
void launch_resample_filter(const PicDev* pics, uint32_t n_pics, const YuvDst* src, const TensorDst& dst, uint32_t dtype,
                            uint32_t filter, const FitArgs& fit, cudaStream_t stream);

// Stateless kernels behind h263cu_yuv420_to_rgba / h263cu_deblock (tight planes).
void launch_yuv420_to_rgba(const uint8_t* y, const uint8_t* cb, const uint8_t* cr, uint32_t w, uint32_t h,
                           uint8_t* rgba, cudaStream_t stream);
void launch_deblock_plane(const uint8_t* in, uint8_t* out, uint32_t w, uint32_t h, int strength, cudaStream_t stream);

// Position-weighted checksums of the tight w x h window of a pitched plane:
// out[k] += sum_i (byte[i]+1) * ((uint32)(i*2654435761) | 1), i = y*row_bytes + x.
struct ChecksumJob {
    const uint8_t* base;
    uint32_t row_bytes;  // samples per row that count
    uint32_t rows;
    uint32_t pitch;
    uint32_t out_index;
    uint32_t step;       // bytes between samples (2 for a plane of the interleaved chroma pair)
    uint32_t pad;
};
void launch_checksums(const ChecksumJob* jobs, uint32_t n_jobs, unsigned long long* out, cudaStream_t stream);

// parse_mb.cu (H263CU_PARSE_ON_DEVICE): the macroblock layer of n_jobs pictures, their packets in `words`, the VLC
// tables (PT_WORDS words) in `tables`; one result per job.  The kernel takes 126.25 KiB of dynamic shared memory.
cudaError_t launch_parse_mb(const ParseJob* jobs, uint32_t n_jobs, const uint32_t* tables, const uint32_t* words, h263cu_mb* mbs,
                            h263cu_event* events, ParseResult* results, cudaStream_t stream);
// The records of the pictures that survived a device-parse step, compacted from src into dst with their packed index
void launch_pack_mbs(const h263cu_mb* src, h263cu_mb* dst, const PackMove* moves, uint32_t n_moves, cudaStream_t stream);

}  // namespace h263dev
