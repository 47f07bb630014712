// recon_tile.cu -- the hot kernel: fused reconstruction, one WARP per 4 consecutive macroblocks,
// for reference planes that carry the replicated border (DESIGN.md section 3).  Warps are
// autonomous: there is no CTA-wide barrier, only __syncwarp(), so a warp waiting on memory never
// holds up others.
//
//   phase 0  lanes 0..23 = the 24 blocks of the 4 macroblocks: event counts, motion vectors ->
//            source offsets / alignment / half-pel flags (gather.rs:140-204, types.rs:721-729,
//            759-768); coded blocks are compacted into slots
//   phase 1  lane = event: a segmented prefix sum gives the zig-zag index, dequantise, scatter,
//            classify (rle.rs:82-172)
//   phase 2  8 lanes per slot, 4 slots per pass: per row that holds a coefficient a row pass and
//            a column-pass update, then rounding (idct.rs:52-65,170-198); s16 residuals go to the
//            slot's rows
//   phase 3  lane = 4 luma columns x 8 rows (half of one 8x8 luma block) + the 2 x 4 chroma
//            samples of BOTH planes under them.  The chroma planes are stored interleaved (CbCr
//            pairs, like NV12), so a chroma row of a lane is one 32-bit word and runs through the
//            same code as a luma row: two aligned words per prediction row, half-pel
//            interpolation in 16-bit lanes (gather.rs:34-40,103-113), saturating residual add,
//            plane stores, border replication, BT.601 RGBA (bt601.rs:12-59).  RGBA leaves through
//            a shared-memory tile and one TMA tensor store per macroblock
//            (cp.async.bulk.tensor.2d into the context's pool, .3d into a caller's buffer), which takes the
//            415 MB per step of RGBA off the LSU pipe.
//
// Four lanes side by side cover a macroblock row, so a prediction pass touches the sectors of 8
// macroblock rows (v13: 16-20 luma, 32 chroma) -- the L1 look-ups that bounded v13 (DESIGN.md 4.1).
// Everything a lane needs per block sits in shared memory as 32-bit offsets from the context's
// pool bases (kernel parameters), so the epilogue does no 64-bit pointer chasing.
//
// v15 / v16 (DESIGN.md 4.1, profiles/r02_variants.txt): the kernel is bound by the ALU pipe and the issue slots, so
// integer work sits on the multiply pipe where it costs the same number of instructions (byte extraction and vector
// sums as IDP.4A dot products, plane words and even lanes as multiply-adds), BT.601 runs on complemented terms (one
// clamp instruction per channel), the RGBA tile is handed to the TMA unit before the plane stores, and the standard
// instantiations keep 5.4 KB of shared memory per warp so that 35 warps fit an SM beside the L1.
#include "recon_common.cuh"

namespace h263dev {

namespace {

constexpr int WARP_MBS = 4;  // macroblocks per warp
// Warps per CTA and CTAs per SM.  Without a CTA barrier a CTA is just a group of warps.  The instantiations for the
// standard picture formats (compile-time pitches, no edge fix-up, no clamped prediction) keep less per warp in shared
// memory (WarpTailT<true>) and compile to 56 registers: 7 CTAs of 5 warps = 35 warps per SM inside the 196 KB
// carve-out, which leaves the L1 in place; the others run 8 CTAs of 4 warps at 64 registers.  The kernel gains about 5 %
// per extra CTA of 4 warps (profiles/r02_variants.txt); 4 warps beat 8 by 2 % (shorter tails).
#ifndef H263_STD_WARPS
#define H263_STD_WARPS 5
#endif
#ifndef H263_STD_CTAS
#define H263_STD_CTAS 7
#endif
constexpr int GEN_WARPS = 4, GEN_CTAS = 8;
// Ablation builds for time attribution (results are wrong by design): 1 = no event walk / transform,
// 2 = no prediction loads (every macroblock treated as intra), 4 = no RGBA, 8 = no plane stores,
// 16 = RGBA computed but not stored.
#ifndef H263_ABLATE
#define H263_ABLATE 0
#endif
// 1 = RGBA through the shared-memory tile + TMA tensor stores, 0 = one 128-bit global store per lane and row
#ifndef H263_RGBA_TMA
#define H263_RGBA_TMA 1
#endif
// BT.601 arithmetic: 0 = multiply-add + shift + saturating packs (v14), 1 = complemented terms, one clamp per channel,
// 2 = 1 with the sample extraction as a dot product, 3 = 0 with extraction and shifts as dot products, 4 = 2 with green
// and blue as differences from red added inside the clamp instruction (profiles/r02_variants.txt)
#ifndef H263_RGBA_MODE
#define H263_RGBA_MODE 4
#endif
constexpr int WARP_BLOCKS = WARP_MBS * 6;
constexpr int RES_WORDS = 36;    // per slot: 8 residual rows of 8 x s16 (16 bytes) + 4 words of padding, which put
                                 // the four slots of a pass on different banks
constexpr int EV_CAP = 64;       // events walked at once (one slot has at most 64); more are walked in chunks (1.4 % of
                                 // the benchmark's tiles hold more than 64 events)
constexpr int SLOT_FLOATS = 68;  // 64 + 4 pad: 16 B aligned, the four slots of a pass start 4 banks apart
constexpr int STAGE_BYTES = 4096;  // RGBA of the warp's four macroblocks: 4 x (16 rows x 64 bytes)

// per-macroblock flags (WarpTail.mba[].w, low byte; mbx sits above them)
constexpr uint32_t MBF_INTER = 1u << 0;
constexpr uint32_t MBF_LEFT = 1u << 2, MBF_RIGHT = 1u << 3, MBF_TOP = 1u << 4, MBF_BOTTOM = 1u << 5;
constexpr uint32_t MBF_RGBA = 1u << 6;
// per-block flags (WarpTail.bf[]): byte alignment of the first source sample (2 bits) | ix | iy | slow
constexpr uint32_t BF_SLOW = 1u << 4;  // the vector leaves the replicated border: clamped per-sample path

// The part of a warp's shared memory that is dead by the time RGBA is produced: the RGBA tile aliases it.
struct __align__(16) WarpStage {
    uint32_t res[WARP_BLOCKS][RES_WORDS];  // per slot: residual rows, s16 row-major (row j = words 4j..4j+3)
    uint32_t evbuf[EV_CAP];                // walked events of the slots in flight: lin[5:0] | dropped[15] | value[31:16]
    uint2 slotdesc[WARP_BLOCKS];           // x = first event unit (absolute), y = nev | quant<<8 | wide<<13 | inter<<14 | chroma<<15 | block<<16 | dc<<24
    uint32_t sstart[WARP_BLOCKS];          // per slot: index of its first event among the warp's events
    uint32_t slotinfo[WARP_BLOCKS];        // per slot, gathered by the walk: rows[7:0] | column > 0 [8] | overflow [9]; after
                                           // the classification: the pass descriptors of the slots that need the
                                           // transform, sorted by rows to transform (most first)
};
static_assert(sizeof(WarpStage) == STAGE_BYTES, "the RGBA tile aliases exactly this");

// What lives from phase 0 to the end, plus the coefficient slots.  COMPACT (standard formats): the macroblock records are
// dead after phase 0 and sit in the coefficient slots; pitches, picture index and edge info are not kept at all.
template <bool COMPACT>
struct WarpTailT;
template <>
struct __align__(16) WarpTailT<true> {
    float coef[4][SLOT_FLOATS];     // coefficients of the four slots in flight
    uint4 mba[WARP_MBS];            // ydst4, cdst4, rgba row, flags[7:0] | mbx[15:8]
    uint32_t bd[WARP_BLOCKS];       // per block: 4-byte offset (from the y or c pool) of the aligned word that holds
                                    // the first source sample of the block's row 0 (blocks 4 and 5 share one)
    uint32_t meta[WARP_BLOCKS];     // per block: cls[2:0] | slot[7:3] | dcres[31:16]
    uint8_t bf[WARP_BLOCKS];        // per block: BF_* flags
    __device__ __forceinline__ uint32_t* mbrec() { return reinterpret_cast<uint32_t*>(&coef[0][0]); }
};
template <>
struct __align__(16) WarpTailT<false> {
    float coef[4][SLOT_FLOATS];
    uint4 mba[WARP_MBS];
    uint4 mbb[WARP_MBS];            // pitches (y | c << 16), -, picture index, edge info
    uint32_t bd[WARP_BLOCKS];
    uint32_t meta[WARP_BLOCKS];
    uint32_t mbrec_[WARP_BLOCKS];   // the four macroblock records (the clamped prediction path reads them again)
    uint8_t bf[WARP_BLOCKS];
    __device__ __forceinline__ uint32_t* mbrec() { return mbrec_; }
};

template <bool COMPACT, int NW>
struct TileSmemT {
    WarpStage stage[NW];  // first: TMA store sources must be 128-byte aligned
    WarpTailT<COMPACT> tail[NW];
};
// the 196 KB carve-out holds 200 704 bytes, of which every resident CTA takes 1 KB besides its own shared memory
static_assert(sizeof(TileSmemT<true, H263_STD_WARPS>) <= 200704 / H263_STD_CTAS - 1024, "shared memory budget of the standard instantiations");
static_assert(sizeof(TileSmemT<false, GEN_WARPS>) <= 200704 / GEN_CTAS - 1024, "shared memory budget of the generic instantiations");

__device__ const float g_basis[8][8] = H263_BASIS_TABLE;
__device__ const uint8_t g_dezigzag[64] = H263_DEZIGZAG_LINEAR;

// compile-time copy of BASIS_TABLE: with y and j unrolled these fold into immediates of the column pass
__device__ __forceinline__ constexpr float k_basis(int y, int j) {
    constexpr float T[8][8] = H263_BASIS_TABLE;
    return T[y][j];
}

// H.263 dequantisation of a narrow (10-bit) level: |level| <= 512, so QP*(2|level|+1) stays below
// 2^15 and the wrapping-i16 arithmetic of rle.rs:130-133 cannot wrap. q2 = 2*QP, qc = QP - (QP even).
__device__ __forceinline__ int dequant_narrow(int level, int q2, int qc) {
    const int mag = q2 * abs(level) + qc;
    const int v = level < 0 ? -mag : mag;
    return max(min(v, 2047), -2048);
}

// rounding of the (already /4) transform output q: trunc(q * m + copysign(0.5, q)) with m = 1 for
// Full / Horiz blocks (x * 1 == x) and m = BASIS_TABLE[0][0] for Vert blocks, where
// (v * B00) / 4 == (v / 4) * B00 exactly (power-of-two scaling) -- idct.rs:143-145,161-163,189-190
__device__ __forceinline__ int round_q(float q, float m) { return __float2int_rz(fadd(fmul(q, m), copysign_half(q))); }

// ---- half-pel interpolation in 16-bit lanes -------------------------------------------------
// A prediction row of a lane is 4 samples (luma: 4 pixels; chroma: the CbCr pairs of 2 samples) that start `sh`
// bits into the aligned word pair (w0, w1); the horizontal neighbours start `shb` bits in (sh, or sh + one sample).
// Returns a + b per sample in two words of two 16-bit lanes.  With shb == sh this is 2a.
struct RowSum {
    uint32_t lo, hi;
};
// lo = the even samples (bytes 0 and 2 of the four), hi = the odd ones: luma (p0, p2) (p1, p3), chroma (cb0, cb1) (cr0, cr1).
// Only the odd samples are unpacked: a word is E + 256 O in terms of its even / odd lane words, so the even lanes of
// a + b are (a + b) - 256 (O_a + O_b) -- exact modulo 2^32, the true lane sums are below 2^32 -- one multiply-add on
// the multiply pipe instead of two byte permutes on the ALU.
__device__ __forceinline__ RowSum row_sum4(uint32_t w0, uint32_t w1, int sh, int shb) {
    const uint32_t a = __funnelshift_r(w0, w1, sh), b = __funnelshift_rc(w0, w1, shb);
    RowSum h;
    h.hi = __byte_perm(a, 0, 0x4341) + __byte_perm(b, 0, 0x4341);
    h.lo = (a + b) - 256u * h.hi;
    return h;
}
// (top * (2 - iy) + bottom * iy + 2) >> 2 per 16-bit lane: with iy == 0 and ix == 0 this is exactly the sample,
// with one of them it is (a + b + 1) >> 1 -- one form covers the four modes of gather.rs:34-40,103-113.
// The weights arrive scaled by 64 (wt = 64 * (2 - iy), wb = 64 * iy), so the sum lands in bits 8..15 of each lane
// (at most 510 * 128 + 128 < 2^16: no carry into the upper lane) and one byte permute both shifts and masks.
__device__ __forceinline__ uint32_t vmix(uint32_t top, uint32_t bottom, uint32_t wt, uint32_t wb) {
    return __byte_perm(top * wt + (bottom * wb + 0x00800080u), 0, 0x4341);
}

// ---- BT.601 (bt601.rs:12-59) ----------------------------------------------------------------
#if H263_RGBA_MODE == 0 || H263_RGBA_MODE == 3
__device__ __forceinline__ uint32_t pack_sat(int a, int b, uint32_t c) {
    uint32_t d;  // d = c[15:0] << 16 | sat_u8(a) << 8 | sat_u8(b)
    asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(a), "r"(b), "r"(c));
    return d;
}
#endif
struct CT {
    int r, g, b;
};
// chroma terms with the -16 luma offset and the rounding constant folded in:
//   R = (76309*y + r) >> 16 with r = 104597*(cr-128) + 32768 - 16*76309, etc.
// The multipliers are passed in registers (see opaque()): a product with an immediate multiplier
// AND an immediate addend does not encode, and the compiler would otherwise materialise the
// multiplier once per use.
__device__ __forceinline__ int opaque(int v) {
    asm("" : "+r"(v));
    return v;
}
#if H263_RGBA_MODE == 0 || H263_RGBA_MODE == 3
__device__ __forceinline__ CT chroma_terms_folded(int cb, int cr, int kr, int kg, int kb) {
    CT t;
    t.r = cr * kr + (32768 - 128 * 104597 - 16 * 76309);
    t.g = cr * kg + (cb * -25675 + (32768 + 128 * 53279 + 128 * 25675 - 16 * 76309));
    t.b = cb * kb + (32768 - 128 * 132201 - 16 * 76309);
    return t;
}
#else
// The same terms complemented, t' = 0xFFFFFF - t (kr, kg, kb arrive negated): with w = t' - 76309*y = 0xFFFFFF - x the
// clamp of w to [0, 0xFFFFFF] carries 255 - clamp(x >> 16, 0, 255) in byte 2 and zero in byte 3 (rgba_px below).
__device__ __forceinline__ CT chroma_terms_folded(int cb, int cr, int kr, int kg, int kb) {
    CT t;
    t.r = cr * kr + (0xFFFFFF - (32768 - 128 * 104597 - 16 * 76309));
    t.g = cr * kg + (cb * 25675 + (0xFFFFFF - (32768 + 128 * 53279 + 128 * 25675 - 16 * 76309)));
    t.b = cb * kb + (0xFFFFFF - (32768 - 128 * 132201 - 16 * 76309));
#if H263_RGBA_MODE == 4
    // green and blue as differences from red: the pixel's multiply-add then happens once (red) and the other two
    // channels add their difference inside the clamp instruction (VIADDMNMX.RELU)
    t.g = cr * (kg - kr) + (cb * 25675 + ((32768 - 128 * 104597) - (32768 + 128 * 53279 + 128 * 25675)));
    t.b = cb * kb + (cr * -kr + ((32768 - 128 * 104597) - (32768 - 128 * 132201)));
#endif
    return t;
}
#endif
#if H263_RGBA_MODE == 0
// yw = the four luma samples of the row as bytes, k = which one
__device__ __forceinline__ uint32_t rgba_px(uint32_t yw, int k, int ky, const CT& t) {
    const int y = (int)(__byte_perm(yw, 0, 0x4440 + k));
    const int r = (y * ky + t.r) >> 16, g = (y * ky + t.g) >> 16, b = (y * ky + t.b) >> 16;
    return pack_sat(g, r, pack_sat(255, b, 0));
}
#elif H263_RGBA_MODE == 3
// everything but the saturating packs on the multiply pipe: sample extraction and the >> 16 are dot products
// (IDP.4A with a one-hot selector, IDP.2A picking the signed upper half)
__device__ __forceinline__ uint32_t rgba_px(uint32_t yw, int k, int ky, const CT& t) {
    const int y = (int)__dp4a(yw, 1u << (8 * k), 0u);
    const int r = __dp2a_hi(y * ky + t.r, 0x01000000, 0), g = __dp2a_hi(y * ky + t.g, 0x01000000, 0), b = __dp2a_hi(y * ky + t.b, 0x01000000, 0);
    return pack_sat(g, r, pack_sat(255, b, 0));
}
#else
// Complemented form: w_c = clamp(t'_c - 76309*y, 0, 0xFFFFFF) = clamp(0xFFFFFF - x_c) is ONE instruction per channel
// (VIADDMNMX.RELU) and holds 255 - C in byte 2, 0 in byte 3: for x < 0 it is 0xFFFFFF (C = 0), for x > 0xFFFFFF it is
// 0 (C = 255), and in between 0xFFFFFF - x is the 24-bit complement of x.  One byte permute gathers (~R, ~G, 0, 0), one
// LOP3 merges ~B and inverts: (R, G, B, 0xFF).  ky arrives negated.
__device__ __forceinline__ uint32_t rgba_px(uint32_t yw, int k, int ky, const CT& t) {
#if H263_RGBA_MODE == 1
    const int y = (int)(__byte_perm(yw, 0, 0x4440 + k));
#else
    const int y = (int)__dp4a(yw, 1u << (8 * k), 0u);  // sample extraction on the multiply pipe
#endif
#if H263_RGBA_MODE == 4
    const int xr = y * ky + t.r;
    const uint32_t wr = (uint32_t)__vimin_s32_relu(xr, 0xFFFFFF), wg = (uint32_t)__viaddmin_s32_relu(xr, t.g, 0xFFFFFF),
                   wb = (uint32_t)__viaddmin_s32_relu(xr, t.b, 0xFFFFFF);
#else
    const int nyk = opaque(y * ky);  // the compiler folds the additions into three multiply-adds + three clamps
    const uint32_t wr = (uint32_t)__viaddmin_s32_relu(nyk, t.r, 0xFFFFFF), wg = (uint32_t)__viaddmin_s32_relu(nyk, t.g, 0xFFFFFF),
                   wb = (uint32_t)__viaddmin_s32_relu(nyk, t.b, 0xFFFFFF);
#endif
    const uint32_t rg = __byte_perm(wr, wg, 0x3362);
    uint32_t px;  // ~(rg | (wb & 0xFFFF0000)) as ONE LOP3 (the compiler splits the inversion off)
    asm("lop3.b32 %0, %1, %2, 0xFFFF0000, 0x07;" : "=r"(px) : "r"(rg), "r"(wb));
    return px;
}
#endif

// One step of an inclusive warp prefix sum: v += v of the lane d below, where there is one.  The shuffle's own
// predicate (source lane in range) guards the addition: two instructions per step instead of shuffle + compare +
// select + add.
__device__ __forceinline__ uint32_t scan_up_step(uint32_t v, int d) {
    asm volatile("{ .reg .pred p; .reg .b32 t; shfl.sync.up.b32 t|p, %0, %1, 0, 0xffffffff; @p add.u32 %0, %0, t; }" : "+r"(v) : "r"(d));
    return v;
}
// The same for a segmented sum: the addition happens when the lane d below belongs to the same segment (dist = lanes
// between this lane and the head of its segment).
__device__ __forceinline__ int seg_scan_up_step(int v, int d, int dist) {
    asm volatile("{ .reg .pred p; .reg .b32 t; shfl.sync.up.b32 t, %0, %1, 0, 0xffffffff; setp.ge.s32 p, %2, %1; @p add.s32 %0, %0, t; }"
                 : "+r"(v)
                 : "r"(d), "r"(dist));
    return v;
}

// Two words of two 16-bit lanes holding bytes (e0, e1) and (o0, o1) -> the bytes (e0, o0, e1, o1): o * 256 + e
__device__ __forceinline__ uint32_t mad_pack(uint32_t o, uint32_t e) { return o * 256u + e; }

// keep the low `keep` bytes (0..4) of a, take the rest from b
__device__ __forceinline__ uint32_t merge_bytes(uint32_t a, uint32_t b, int keep) {
    const uint32_t m = keep >= 4 ? 0xFFFFFFFFu : ((1u << (8 * keep)) - 1u);
    return (a & m) | (b & ~m);
}

// Byte offset of (macroblock q, row, 16-byte chunk c) inside the warp's RGBA tile.  Each macroblock is a dense
// 16-row x 64-byte box of a TMA store.  The two row groups of a macroblock write the same banks (rows 8 apart): a 2-way
// conflict on the eight 128-bit shared stores of a lane.  No TMA swizzle mode removes it for a 64-byte box -- 64B
// XORs address bits 7..8 only, and 128B pads every 64-byte row to 128 bytes (tools/tma_swizzle_probe.cu,
// profiles/r02_tma_swizzle_probe.txt) -- and the kernel is not bound by it (direct 128-bit global stores, the dense
// tile and a conflict-free layout run within 0.5 % of each other, profiles/r02_variants.txt).
__device__ __forceinline__ uint32_t stage_offset(int q, int row, int c) { return (uint32_t)(q * 1024 + row * 64 + c * 16); }

}  // namespace


// PY / PC / PR: luma, chroma and RGBA row pitches in bytes when they are known at compile time (the
// standard picture formats; all planes of a context share them), 0 = read them from the descriptors.
// Constant pitches turn every row address of the epilogue into an immediate offset.
// EDGE: pictures whose size is not a multiple of 16.  The planes are macroblock-rounded; the part of the last
// macroblock column / row that lies outside the picture is overwritten with the picture's edge pixels before the
// stores (and the border replication continues from there), so that prediction reads beyond the true edge see
// read_sample's clamp (gather.rs:16-31).  Compiled out of the instantiations for aligned pictures.
// WIDE_MV: some vector of the step may leave the replicated border (no H263CU_PICFLAG_MV_IN_RANGE; unreachable from a
// parsed stream, mvd_pred.rs:70-117): the instantiation with the clamped per-sample path.  Without it every vector of
// the step lies in the range (the parser cannot leave it, caller-built side info is checked on the host), nothing is
// clamped, and that path does not weigh on the register allocation.
// NW / NCTAS: warps per CTA and CTAs per SM (5 x 7 for the standard formats, 4 x 8 otherwise).
// OUT: where the output goes (kernels.cuh).  OUT_POOL: RGBA into the context's pool.
// OUT_DEV_RGBA: RGBA goes to a caller-owned device buffer (h263cu_decode_step_device) through a 3-D tensor map of
// (bytes, rows, slots); PicDev.rgba_row0 carries slot << 12 (16 * mby < 4096 fills the low bits, so phase 0 is
// unchanged).  The map's bounds are the slot's, and TMA drops the rows of a macroblock box below them; the right-edge
// macroblocks of pictures whose width is not a multiple of 16 (EDGE) are stored directly, cut to the picture.
// OUT_YUV: no RGBA (the BT.601 conversion, the tile and the TMA store are compiled out); each lane stores the plane
// words it holds into the caller's planes `yuv` as well (h263cu_decode_step_device_yuv), slot << 12 in rgba_row0 as
// above.  Plain stores, cut to the picture in the right-edge and bottom-edge macroblocks of EDGE instantiations.
template <int PY, int PC, int PR, bool EDGE, bool WIDE_MV, int NW, int NCTAS, int OUT>
__global__ void __launch_bounds__(NW * 32, NCTAS)
    recon_tile_kernel(const PicDev* __restrict__ pics, const h263cu_mb* __restrict__ mbs,
                      const h263cu_event* __restrict__ events, uint32_t n_mbs, int emit_rgba, const Pools pools,
                      const __grid_constant__ CUtensorMap rgba_map, const YuvDst yuv) {
    constexpr bool COMPACT = PY != 0 && !EDGE && !WIDE_MV;
    constexpr int CTA_WARPS = NW;
    __shared__ __align__(1024) TileSmemT<COMPACT, NW> S;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    WarpStage& G = S.stage[warp];
    WarpTailT<COMPACT>& W = S.tail[warp];
    uint32_t* const mbrec = W.mbrec();
    const int g = lane >> 3, t = lane & 7;
    const uint32_t lt_mask = (1u << lane) - 1u;

    const uint32_t n_tiles = (n_mbs + WARP_MBS - 1) / WARP_MBS;
    const uint32_t tile = blockIdx.x * CTA_WARPS + warp;
    if (tile >= n_tiles) return;  // warp-uniform; no CTA barrier follows
    const uint32_t mb0 = tile * WARP_MBS;
    const int n_w = (int)min((uint32_t)WARP_MBS, n_mbs - mb0);

    // ================= phase 0: lane = block (macroblock lane / 6, block lane % 6) ==============
    if (lane < n_w * 6) mbrec[lane] = __ldg(reinterpret_cast<const uint32_t*>(mbs) + (size_t)tile * WARP_BLOCKS + lane);
    __syncwarp();
    int n_slots;
    {
        const bool bvalid = lane < n_w * 6;
        const int bm = bvalid ? (lane * 43) >> 8 : 0, bb = bvalid ? lane - bm * 6 : 0;
        const uint32_t* r = &mbrec[bm * 6];
        const uint32_t w0 = r[0], w1 = r[1], w2 = r[2], w3 = r[3], w4 = r[4], w5 = r[5];
        const uint32_t pic = w1 & 0xFFFFu;
        const PicDev& P = pics[pic];
        const int mbx = (w1 >> 16) & 0xFF, mby = w1 >> 24;
        const bool inter = (w2 & H263CU_MB_INTER) != 0, wide = (w2 & H263CU_MB_WIDE) != 0;
        // nev[6] = bytes 2..7 of (w2, w3); intradc[6] = bytes 0..5 of (w4, w5)
        const uint32_t nev = bvalid ? __byte_perm(w2, w3, 0x4440u + (uint32_t)bb + 2u) & 0xFFu : 0u;
        const uint32_t code = inter ? 0u : __byte_perm(w4, w5, 0x4440u + (uint32_t)bb) & 0xFFu;

        // motion: source offset, alignment and half-pel flags of this block
        uint32_t boff = 0, bflags = 0;
        if (inter) {
            int mvx, mvy, bx, sy, pitch;
            uint32_t base;
            bool in_range;
            // Vectors of a step that runs this instantiation lie in [-32, 31] (the parser's halfpel_decode wraps into
            // that range, mvd_pred.rs:70-117; caller-built side info is checked on the host and a picture with a longer
            // vector takes the WIDE_MV instantiation), so nothing is clamped here.  Signed bytes come out of the record
            // words as dot products with a one-hot selector (IDP.4A on the multiply pipe, not the ALU).
            if (bb < 4) {
                // mv[bb] = bytes 2bb, 2bb+1 of (w4, w5)
                const int m = (int)((bb < 2 ? w4 : w5) >> (16 * (bb & 1)));
                mvx = __dp4a(m, 0x00000001, 0), mvy = __dp4a(m, 0x00000100, 0);
                in_range = mvx >= -32 && mvx <= 31 && mvy >= -32 && mvy <= 31;
                bx = mbx * 16 + (bb & 1) * 8 + (mvx >> 1), sy = mby * 16 + (bb >> 1) * 8 + (mvy >> 1);
                pitch = PY ? PY : P.pitch_y, base = P.ref_y4;
            } else {
                // both chroma blocks use the average of the four luma vectors (gather.rs:182, types.rs:759-768):
                // average_sum_of_mvs(s) = 2 (s >> 4) + [s & 15 > 2] + [s & 15 >= 14] = ((s + 13) >> 4) + ((s + 2) >> 4);
                // the chroma planes are interleaved: sample x of a row sits at byte 2x (Cb) and 2x + 1 (Cr)
                const int sx = __dp4a((int)w5, 0x00010001, __dp4a((int)w4, 0x00010001, 13));
                const int sy13 = __dp4a((int)w5, 0x01000100, __dp4a((int)w4, 0x01000100, 13));
                mvx = (sx >> 4) + ((sx - 11) >> 4), mvy = (sy13 >> 4) + ((sy13 - 11) >> 4);
                in_range = mvx >= -16 && mvx <= 15 && mvy >= -16 && mvy <= 15;
                bx = 2 * (mbx * 8 + (mvx >> 1)), sy = mby * 8 + (mvy >> 1);
                pitch = PC ? PC : P.pitch_c, base = P.ref_c4;
            }
            const int a = bx & 3;
            boff = base + (uint32_t)((sy * pitch + (bx - a)) >> 2);
            bflags = (uint32_t)(a | ((mvx & 1) << 2) | ((mvy & 1) << 3)) | (!WIDE_MV || in_range ? 0u : BF_SLOW);
        }
        if (bvalid) {
            W.bd[lane] = boff;
            W.bf[lane] = (uint8_t)bflags;
            if (bb == 0) {
                const int pitch_y = PY ? PY : P.pitch_y, pitch_c = PC ? PC : P.pitch_c;
                const int mbw = (P.w + 15) >> 4, mbh = (P.h + 15) >> 4;
                // valid luma columns / rows of the last macroblock column / row (0 = all 16) and the same for
                // chroma (0 = all 8)
                const uint32_t ed = EDGE ? ((uint32_t)(P.w & 15) | ((uint32_t)(P.h & 15) << 4) | ((uint32_t)(P.cw & 7) << 8) |
                                            ((uint32_t)(P.ch & 7) << 12))
                                         : 0u;
                uint32_t flags = inter ? MBF_INTER : 0u;
                if (mbx == 0) flags |= MBF_LEFT;
                if (mbx == mbw - 1) flags |= MBF_RIGHT;
                if (mby == 0) flags |= MBF_TOP;
                if (mby == mbh - 1) flags |= MBF_BOTTOM;
                if (emit_rgba && P.rgba) flags |= MBF_RGBA;
                W.mba[bm] = make_uint4(P.cur_y4 + (uint32_t)((mby * 16 * pitch_y + mbx * 16) >> 2),
                                       P.cur_c4 + (uint32_t)((mby * 8 * pitch_c + mbx * 16) >> 2), P.rgba_row0 + (uint32_t)(mby * 16),
                                       flags | ((uint32_t)mbx << 8));
                if constexpr (!COMPACT) W.mbb[bm] = make_uint4((uint32_t)pitch_y | ((uint32_t)pitch_c << 16), 0u, pic, ed);
            }
        }

        // coded blocks -> slots (block order); their events form one sequence per warp
        const bool coded = nev > 0;
        const uint32_t coded_mask = __ballot_sync(FULL, coded);
        const int pos = __popc(coded_mask & lt_mask);
        n_slots = __popc(coded_mask);
        uint32_t ev_incl = nev;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) ev_incl = scan_up_step(ev_incl, d);
        // events of the blocks before this one inside the macroblock
        const uint32_t before = (ev_incl - nev) - __shfl_sync(FULL, ev_incl - nev, bm * 6);
        if (coded) {
            G.sstart[pos] = ev_incl - nev;
            const uint32_t first = P.first_event + w0 + (wide ? 2 * before : before);
            const uint32_t quant = (w2 >> 8) & 31u;
            G.slotdesc[pos] = make_uint2(first, nev | (quant << 8) | (wide ? 1u << 13 : 0u) | (inter ? 1u << 14 : 0u) |
                                                    (bb >= 4 ? 1u << 15 : 0u) | ((uint32_t)lane << 16) | (code << 24));
            asm volatile("prefetch.global.L1 [%0];" ::"l"(events + first));
        } else if (bvalid) {
            // no coefficients: Dc(level) when an intra DC is present, else Zero (rle.rs:94-104)
            const bool has_dc = code != 0;
            const int dcres = has_dc ? round_residual_dc((float)intradc_level((int)code)) : 0;
            W.meta[lane] = (uint32_t)(has_dc ? CLS_DC : CLS_ZERO) | ((uint32_t)dcres << 16);
        }
    }
    __syncwarp();


    // ================= phases 1 + 2, per chunk of slots whose events fit the event buffer ==========
    // (one chunk unless the four macroblocks hold more than EV_CAP events)
    {
        const float* const basis = &g_basis[0][0];
        const float bt0 = basis[0 * 8 + t], bt1 = basis[1 * 8 + t], bt2 = basis[2 * 8 + t], bt3 = basis[3 * 8 + t],
                    bt4 = basis[4 * 8 + t], bt5 = basis[5 * 8 + t], bt6 = basis[6 * 8 + t], bt7 = basis[7 * 8 + t];
        float* c = W.coef[g];
        const int tperm = (t & 4) | ((t & 1) << 1) | ((t >> 1) & 1);
        // lane = slot for the per-slot steps
        if (H263_ABLATE & 1) n_slots = 0;
        const bool is_slot = lane < n_slots;
        const uint2 my_sd = is_slot ? G.slotdesc[lane] : make_uint2(0u, 0u);
        const uint32_t my_start = is_slot ? G.sstart[lane] : 0xFFFFFFFFu;
        const uint32_t my_end = my_start + (my_sd.y & 0xFFu);
        int s_lo = 0;
        uint32_t e_lo = 0;
        while (s_lo < n_slots) {
            // slots of this chunk: the longest run starting at s_lo whose events fit the buffer
            // (a slot with more events than the buffer holds -- a malformed record, real blocks have at most
            // 64 -- is walked as far as the buffer goes: its index is past 63 by then and it is dropped)
            const int s_hi = max(s_lo + 1, s_lo + __popc(__ballot_sync(FULL, is_slot && lane >= s_lo && my_end - e_lo <= (uint32_t)EV_CAP)));
            const bool in_chunk = lane >= s_lo && lane < s_hi;
            const uint32_t e_end = __shfl_sync(FULL, my_end, s_hi - 1);
            const uint32_t e_hi = min(e_end, e_lo + (uint32_t)EV_CAP);
            if (in_chunk) G.slotinfo[lane] = 0u;
            __syncwarp();

            // ---- phase 1: lane = event.  The zig-zag index is a segmented prefix sum of run + 1 over the
            // events of a slot (rle.rs:117-135); dequantise and park (position, value) in the event buffer.
            uint32_t carry = 0;  // running sum of the slot that continues from the previous round
            for (uint32_t eb = e_lo; eb < e_hi; eb += 32) {
                const uint32_t e = eb + lane;
                const bool act = e < e_hi;
                // which slot: slots whose first event lies in this round mark their head
                const bool head = in_chunk && my_start >= eb && my_start < eb + 32;
                const uint32_t heads = __reduce_or_sync(FULL, head ? 1u << (my_start - eb) : 0u);
                const int n_before = __popc(__ballot_sync(FULL, in_chunk && my_start < eb));
                const uint32_t below = heads & (0xFFFFFFFFu >> (31 - lane));
                const int slot = s_lo + n_before - 1 + __popc(below);
                const int seg = below ? 31 - __clz(below) : -1;  // lane where my slot's events start in this round
                int v = 0, val = 0;
                bool inter = false;
                if (act) {
                    const uint2 sd = G.slotdesc[slot];
                    const uint32_t k = e - G.sstart[slot];
                    const int quant = (int)((sd.y >> 8) & 31u);
                    inter = (sd.y >> 14) & 1u;
                    int run;
                    if (!((sd.y >> 13) & 1u)) {
                        const uint32_t u = __ldg(events + sd.x + k);
                        run = (int)(u >> 10);
                        val = dequant_narrow(((int)(u << 22)) >> 22, 2 * quant, quant - 1 + (quant & 1));
                    } else {
                        run = __ldg(events + sd.x + 2 * k) & 63;
                        val = dequant((int16_t)__ldg(events + sd.x + 2 * k + 1), quant);
                    }
                    v = run + 1;
                }
                const int dist = lane - max(seg, 0);
#pragma unroll
                for (int d = 1; d < 32; d <<= 1) v = seg_scan_up_step(v, d, dist);
                if (seg < 0) v += (int)carry;
                carry = (uint32_t)__shfl_sync(FULL, v, 31);
                if (act) {
                    const int idx = (inter ? 0 : 1) + v - 1;  // intra: the DC occupies zig-zag index 0 (rle.rs:117-121)
                    uint32_t bits, ent;
                    if (idx < 64) {
                        const int lin = g_dezigzag[idx];
                        ent = (uint32_t)lin | ((uint32_t)val << 16);
                        bits = (1u << (lin >> 3)) | ((lin & 7) ? 0x100u : 0u);
                    } else {
                        ent = 0x8000u;  // the whole block stays Zero, DC included (rle.rs:125-127)
                        bits = 0x200u;
                    }
                    G.evbuf[e - e_lo] = ent;
                    atomicOr(&G.slotinfo[slot], bits);
                }
            }
            __syncwarp();

            // ---- classification, lane = slot (rle.rs:94-171) ----
            int key = 4;
            uint32_t pd = 0u;
            if (in_chunk) {
                const uint32_t info = G.slotinfo[lane];
                const bool inter = (my_sd.y >> 14) & 1u;
                const uint32_t blk = (my_sd.y >> 16) & 0xFFu, code = my_sd.y >> 24;
                const bool ovf = (info & 0x200u) != 0, col = (info & 0x100u) != 0;
                const uint32_t rows = info & 0xFFu;
                const bool has_dc = !inter && code != 0 && !ovf;
                int cls, dcres = 0;
                uint32_t R = 0;
                if (ovf || (!rows && !has_dc)) {
                    cls = CLS_ZERO;
                } else if (!(rows & 0xFEu) && !col) {
                    cls = CLS_DC;
                    // Dc(level): the intra DC, or the one coefficient an inter block put on index 0
                    const int dc = has_dc ? intradc_level((int)code) : (int)G.evbuf[my_start - e_lo] >> 16;
                    dcres = round_residual_dc((float)dc);
                } else {
                    cls = col ? CLS_FULL : CLS_VERT;
                    R = rows | (has_dc ? 1u : 0u);
                }
                W.meta[blk] = (uint32_t)cls | ((uint32_t)lane << 3) | ((uint32_t)dcres << 16);
                // everything a pass needs to know about the slot, in one word: slot[4:0] | rows to transform[12:5] |
                // Vert[13] | intra DC present[14] | first event inside the chunk[21:15] | events[29:22] | chroma[30]
                pd = (uint32_t)lane | (R << 5) | (cls == CLS_VERT ? 1u << 13 : 0u) | (has_dc ? 1u << 14 : 0u) | ((my_start - e_lo) << 15) |
                     ((my_sd.y & 0xFFu) << 22) | ((my_sd.y & 0x8000u) << 15);
                const int n = __popc(R);
                key = n >= 4 ? 0 : (n >= 2 ? 1 : (n == 1 ? 2 : 3));
            }
            // slots that need the transform first, those with many rows before those with few, so that the
            // four slots of a pass cost about the same
            int pos = s_lo, n_need = 0;
#pragma unroll
            for (int j = 0; j < 3; j++) {
                const uint32_t b = __ballot_sync(FULL, key == j);
                if (j < key) pos += __popc(b);
                if (j == key) pos += __popc(b & lt_mask);
                n_need += __popc(b);
            }
            __syncwarp();  // every lane has read the walk's word of its slot: the sorted descriptors replace them
            if (key < 3) G.slotinfo[pos] = pd;
            __syncwarp();

            // ---- phase 2: 4 slots per pass, 8 lanes per slot, lane t = column i of the block ---------
            for (int si0 = s_lo; si0 < s_lo + n_need; si0 += 4) {
                const int si = si0 + g;
                const bool valid = si < s_lo + n_need;
                const uint32_t pd = valid ? G.slotinfo[si] : 0u;
                const int sl = (int)(pd & 31u);
                const uint32_t R = (pd >> 5) & 0xFFu;
                const bool vert = (pd >> 13) & 1u;
                const int nev = (int)((pd >> 22) & 0xFFu);
                const uint32_t first = (pd >> 15) & 127u;
                // lane t clears row t of the slot, then the slot's events are scattered into it
                *reinterpret_cast<float4*>(c + t * 8) = make_float4(0.f, 0.f, 0.f, 0.f);
                *reinterpret_cast<float4*>(c + t * 8 + 4) = make_float4(0.f, 0.f, 0.f, 0.f);
                const int nevmax = __reduce_max_sync(FULL, nev);
                __syncwarp();
                if (t < nev) {
                    const uint32_t ent = G.evbuf[first + t];
                    c[ent & 63u] = (float)((int)ent >> 16);
                }
                if (nevmax > 8) {  // rare: more than 8 events in a slot of this pass
                    for (int k = t + 8; k < nev; k += 8) {
                        const uint32_t ent = G.evbuf[first + k];
                        c[ent & 63u] = (float)((int)ent >> 16);
                    }
                }
                if (pd & 0x4000u) {
                    if (t == 0) c[0] = (float)intradc_level((int)(G.slotdesc[sl].y >> 24));
                }
                // Per row y that holds a coefficient in ANY of the four slots (warp-uniform skip otherwise):
                //   row pass    t[y][i] = sum_x c[y][x] * B[x][i], ascending x (idct_1d, idct.rs:52-65), pre-divided
                //               by 4 (exact), which takes the /4 of idct.rs:189 out of the 64-output rounding
                //   column pass out[i][j] += t[y][i] * B[y][j] for the 8 pixel rows j, ascending y; B[y][j] are
                //               compile-time constants, t[y][i] never leaves the register
                // A slot that has no coefficient in row y reads zeros there (the slot was cleared), so its terms
                // are +-0 and change nothing -- skipping all-zero rows is exact, computing them is too.
                const uint32_t U = __reduce_or_sync(FULL, R);
                __syncwarp();
                float acc[8] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
#pragma unroll
                for (int y = 0; y < 8; y++) {
                    if (!((U >> y) & 1u)) continue;  // warp-uniform
                    const float4 ca = *reinterpret_cast<const float4*>(c + y * 8);
                    const float4 cc = *reinterpret_cast<const float4*>(c + y * 8 + 4);
                    float a = fmul(ca.x, bt0);  // 0 + x == x
                    a = fadd(a, fmul(ca.y, bt1));
                    a = fadd(a, fmul(ca.z, bt2));
                    a = fadd(a, fmul(ca.w, bt3));
                    a = fadd(a, fmul(cc.x, bt4));
                    a = fadd(a, fmul(cc.y, bt5));
                    a = fadd(a, fmul(cc.z, bt6));
                    a = fadd(a, fmul(cc.w, bt7));
                    if (vert) a = ca.x;  // Vert: the first column feeds idct_1d directly (idct.rs:152-153)
                    a = fmul(a, 0.25f);
#pragma unroll
                    for (int j = 0; j < 8; j++) acc[j] = fadd(acc[j], fmul(a, k_basis(y, j)));
                }
                const bool any_vert = __any_sync(FULL, vert);  // warp-uniform, taken outside the lane-dependent branch below
                if (R) {
                    // pixel (x = t, y = j): residual row j of the slot, s16 row-major.  The reference clamps the rounded
                    // value to [-256, 255] (idct.rs:190) before it adds it to the prediction and clamps to [0, 255]
                    // (idct.rs:191-194); the first clamp cannot change the result of the second (prediction in
                    // [0, 255]), and |value| <= 2048 * (sum_x |B[x][i]|)^2 / 4 < 14300 fits the s16 that carries it,
                    // so only the saturating add of phase 3 clamps.
                    // luma slots keep the columns of each group of four as (0, 2, 1, 3): the two words a lane of phase 3
                    // reads per row are then its even and its odd samples, the split its registers use
                    uint16_t* rrow = reinterpret_cast<uint16_t*>(&G.res[sl][0]) + ((pd & 0x40000000u) ? t : tperm);
                    if (any_vert) {  // rare: a block with coefficients in its first column only
                        const float m = vert ? H263_B00 : 1.0f;
#pragma unroll
                        for (int j = 0; j < 8; j++) rrow[j * 8] = (uint16_t)(int16_t)round_q(acc[j], m);
                    } else {
#pragma unroll
                        for (int j = 0; j < 8; j++) rrow[j * 8] = (uint16_t)(int16_t)__float2int_rz(fadd(acc[j], copysign_half(acc[j])));
                    }
                }
                __syncwarp();  // the coefficient slots are reused by the next pass
            }
            s_lo = s_hi;
            e_lo = e_end;
        }
    }

    // ================= phase 3: MC + add + clamp + stores + RGBA, all in registers ===============
    // lane = (macroblock, row group rgrp of 8 luma rows, column group cg of 4 luma columns): one half of the luma
    // block lb (its 8 rows, 4 of its columns) and the chroma samples under it -- columns 2cg, 2cg+1 and rows
    // 4rgrp..4rgrp+3 of Cb and Cr, which are one 32-bit word per row of the interleaved chroma plane.
    {
        const int mbq = lane >> 3, rgrp = (lane >> 2) & 1, cg = lane & 3;
        const bool unit_ok = mbq < n_w;
        const int mbi = unit_ok ? mbq : 0;
        const uint4 ma = W.mba[mbi];
        uint4 mv = make_uint4(0u, (ma.w >> 8) & 0xFFu, 0u, 0u);  // pitches, mbx, picture index, edge info
        if constexpr (!COMPACT) {
            const uint4 b = W.mbb[mbi];
            mv.x = b.x, mv.z = b.z, mv.w = b.w;
        }
        const uint32_t flags = (unit_ok ? ma.w : 0u) & ~((H263_ABLATE & 2) ? MBF_INTER : 0u) & ~((H263_ABLATE & 4) ? MBF_RGBA : 0u);
        const uint32_t pitch_y4 = PY ? PY / 4 : (mv.x & 0xFFFFu) >> 2, pitch_c4 = PC ? PC / 4 : mv.x >> 18;
        const int lb = rgrp * 2 + (cg >> 1);  // luma block of this lane
        const int bl = mbi * 6 + lb, bc = mbi * 6 + 4;

        uint32_t ylo[8], yhi[8];  // luma rows: samples (p0, p2) and (p1, p3) in 16-bit lanes (even / odd, like Cb / Cr below)
        uint32_t cbp[4], crp[4];  // chroma rows: (cb0, cb1) and (cr0, cr1)
        if (flags & MBF_INTER) {
            const uint32_t fl = W.bf[bl], fc = W.bf[bc];
            if (!WIDE_MV || !(fl & BF_SLOW)) {
                const int sh = (fl & 3u) * 8, shb = sh + ((fl & 4u) << 1);
                const uint32_t wb = ((fl >> 3) & 1u) * 64u, wt = 128u - wb;
                // the second word of a row is needed unless the block starts word-aligned with a full-pel x vector; the
                // ninth row only for vertical interpolation (its weight is 0 otherwise).  A load pass costs the L1 one
                // look-up per distinct sector it touches, so lanes that do not need a word stay out of the pass.
                const bool second = (fl & 7u) != 0;
                const uint32_t* src = reinterpret_cast<const uint32_t*>(pools.y) + W.bd[bl] + (uint32_t)(cg & 1);
                RowSum hs[9];
#pragma unroll
                for (int r = 0; r < 9; r++) {
                    const uint32_t* p = src + (uint32_t)r * pitch_y4;
                    uint32_t w0 = 0u, w1 = 0u;
                    if (r < 8 || wb != 0) {
                        w0 = __ldg(p);
                        if (second) w1 = __ldg(p + 1);
                    }
                    hs[r] = row_sum4(w0, w1, sh, shb);
                }
#pragma unroll
                for (int r = 0; r < 8; r++) {
                    ylo[r] = vmix(hs[r].lo, hs[r + 1].lo, wt, wb);
                    yhi[r] = vmix(hs[r].hi, hs[r + 1].hi, wt, wb);
                }
            } else {
                // vector beyond the replicated border: clamped per-sample fetch (read_sample, gather.rs:16-31)
                const PicDev& P = pics[mv.z];
                const uint32_t* rr = &mbrec[mbi * 6];
                const uint32_t w1 = rr[1];
                const uint32_t mvw = lb < 2 ? (rr[4] >> (16 * lb)) : (rr[5] >> (16 * (lb - 2)));
                const int mvx = (int8_t)(mvw & 0xFF), mvy = (int8_t)((mvw >> 8) & 0xFF);
                const int x0 = (int)((w1 >> 16) & 0xFF) * 16 + cg * 4, y0 = (int)(w1 >> 24) * 16 + rgrp * 8;
#pragma unroll
                for (int r = 0; r < 8; r++) {
                    uint32_t s[4];
#pragma unroll
                    for (int k = 0; k < 4; k++) s[k] = mc_fetch1(P.ref[0], P.pitch_y, 1, P.w, P.h, x0 + k, y0 + r, mvx, mvy);
                    ylo[r] = s[0] | (s[2] << 16), yhi[r] = s[1] | (s[3] << 16);
                }
            }
            if (!WIDE_MV || !(fc & BF_SLOW)) {
                const int sh = (fc & 3u) * 8, shb = sh + ((fc & 4u) << 2);  // a chroma sample is two bytes away
                const uint32_t wb = ((fc >> 3) & 1u) * 64u, wt = 128u - wb;
                const bool second = (fc & 7u) != 0;
                const uint32_t* src = reinterpret_cast<const uint32_t*>(pools.c) + W.bd[bc] + (uint32_t)cg + (uint32_t)(rgrp * 4) * pitch_c4;
                RowSum hs[5];
#pragma unroll
                for (int r = 0; r < 5; r++) {
                    const uint32_t* p = src + (uint32_t)r * pitch_c4;
                    uint32_t w0 = 0u, w1 = 0u;
                    if (r < 4 || wb != 0) {
                        w0 = __ldg(p);
                        if (second) w1 = __ldg(p + 1);
                    }
                    hs[r] = row_sum4(w0, w1, sh, shb);
                }
#pragma unroll
                for (int r = 0; r < 4; r++) {
                    cbp[r] = vmix(hs[r].lo, hs[r + 1].lo, wt, wb);
                    crp[r] = vmix(hs[r].hi, hs[r + 1].hi, wt, wb);
                }
            } else {
                const PicDev& P = pics[mv.z];
                const uint32_t* rr = &mbrec[mbi * 6];
                const uint32_t w1 = rr[1], w4 = rr[4], w5 = rr[5];
                const int sumx = (int8_t)byte_of(w4, 0) + (int8_t)byte_of(w4, 2) + (int8_t)byte_of(w5, 0) + (int8_t)byte_of(w5, 2);
                const int sumy = (int8_t)byte_of(w4, 1) + (int8_t)byte_of(w4, 3) + (int8_t)byte_of(w5, 1) + (int8_t)byte_of(w5, 3);
                const int mvx = average_sum_of_mvs(sumx), mvy = average_sum_of_mvs(sumy);
                const int x0 = (int)((w1 >> 16) & 0xFF) * 8 + cg * 2, y0 = (int)(w1 >> 24) * 8 + rgrp * 4;
#pragma unroll
                for (int r = 0; r < 4; r++) {
                    cbp[r] = mc_fetch1(P.ref[1], P.pitch_c, CHROMA_STEP, P.cw, P.ch, x0, y0 + r, mvx, mvy) |
                             (mc_fetch1(P.ref[1], P.pitch_c, CHROMA_STEP, P.cw, P.ch, x0 + 1, y0 + r, mvx, mvy) << 16);
                    crp[r] = mc_fetch1(P.ref[2], P.pitch_c, CHROMA_STEP, P.cw, P.ch, x0, y0 + r, mvx, mvy) |
                             (mc_fetch1(P.ref[2], P.pitch_c, CHROMA_STEP, P.cw, P.ch, x0 + 1, y0 + r, mvx, mvy) << 16);
                }
            }
        } else {
            // intra: the prediction is the zero-initialised plane (picture.rs:42-48)
#pragma unroll
            for (int r = 0; r < 8; r++) ylo[r] = yhi[r] = 0u;
#pragma unroll
            for (int r = 0; r < 4; r++) cbp[r] = crp[r] = 0u;
        }

        // ---- residuals: packed s16x2 add, saturate to [0, 255] (idct.rs:191-194) ----
        if (unit_ok) {
            const uint32_t m = W.meta[bl];
            const int cls = (int)(m & 7u);
            if (cls == CLS_DC) {
                const uint32_t dd = __byte_perm(m, 0, 0x3232);  // (dcres, dcres)
#pragma unroll
                for (int r = 0; r < 8; r++) {
                    ylo[r] = __viaddmin_s16x2_relu(ylo[r], dd, 0x00FF00FFu);
                    yhi[r] = __viaddmin_s16x2_relu(yhi[r], dd, 0x00FF00FFu);
                }
            } else if (cls != CLS_ZERO) {
                // columns 4(cg & 1) .. +3 of the slot's rows, stored as (0, 2), (1, 3): two words per row
                const uint2* c = reinterpret_cast<const uint2*>(&G.res[(m >> 3) & 31u][2 * (cg & 1)]);
#pragma unroll
                for (int r = 0; r < 8; r++) {
                    const uint2 rv = c[r * 2];
                    ylo[r] = __viaddmin_s16x2_relu(ylo[r], rv.x, 0x00FF00FFu);
                    yhi[r] = __viaddmin_s16x2_relu(yhi[r], rv.y, 0x00FF00FFu);
                }
            }
            // blocks 4 and 5 of a macroblock sit at an even index: one 64-bit load for both words
            const uint2 mcc = *reinterpret_cast<const uint2*>(&W.meta[bc]);
#pragma unroll
            for (int pl = 0; pl < 2; pl++) {
                uint32_t(&cc)[4] = pl ? crp : cbp;
                const uint32_t mc = pl ? mcc.y : mcc.x;
                const int ccls = (int)(mc & 7u);
                if (ccls == CLS_DC) {
                    const uint32_t dd = __byte_perm(mc, 0, 0x3232);
#pragma unroll
                    for (int r = 0; r < 4; r++) cc[r] = __viaddmin_s16x2_relu(cc[r], dd, 0x00FF00FFu);
                } else if (ccls != CLS_ZERO) {
                    // columns 2cg, 2cg+1 of rows 4rgrp..4rgrp+3: one word per row
                    const uint32_t* c = &G.res[(mc >> 3) & 31u][rgrp * 16 + cg];
#pragma unroll
                    for (int r = 0; r < 4; r++) cc[r] = __viaddmin_s16x2_relu(cc[r], c[r * 4], 0x00FF00FFu);
                }
            }
        }

        // ---- plane words: luma (p0 p1 p2 p3), chroma (cb0 cr0 cb1 cr1) ----
        uint32_t yw[8], cw[4];
#pragma unroll
        for (int r = 0; r < 8; r++) yw[r] = mad_pack(yhi[r], ylo[r]);
#pragma unroll
        for (int r = 0; r < 4; r++) cw[r] = mad_pack(crp[r], cbp[r]);
        if constexpr (EDGE) {
            const uint32_t ed = mv.w;
            const int vw = (int)(ed & 15u), vh = (int)((ed >> 4) & 15u), cvw = (int)((ed >> 8) & 7u), cvh = (int)((ed >> 12) & 7u);
            const bool fix_r = (flags & MBF_RIGHT) != 0, fix_b = (flags & MBF_BOTTOM) != 0;
            {
                // right edge, luma: the pixel of column vw - 1 lives in the lane with cg = (vw - 1) >> 2 of this row group
                const int e = (vw - 1) & 15, keep = min(max(vw - 4 * cg, 0), 4);
                const int from = (lane & ~3) | (e >> 2);
#pragma unroll
                for (int r = 0; r < 8; r++) {
                    const uint32_t mine = __byte_perm(yw[r], 0, (uint32_t)(e & 3)) & 0xFFu;
                    const uint32_t v = __shfl_sync(FULL, mine, from);
                    if (fix_r && vw) yw[r] = merge_bytes(yw[r], v * 0x01010101u, keep);
                }
            }
            {
                // right edge, chroma: the CbCr pair of sample cvw - 1
                const int e = (cvw - 1) & 7, keep = min(max(cvw - 2 * cg, 0), 2);
                const int from = (lane & ~3) | (e >> 1);
#pragma unroll
                for (int r = 0; r < 4; r++) {
                    const uint32_t mine = (e & 1) ? cw[r] >> 16 : cw[r] & 0xFFFFu;
                    const uint32_t v = __shfl_sync(FULL, mine, from);
                    if (fix_r && cvw) cw[r] = merge_bytes(cw[r], v | (v << 16), 2 * keep);
                }
            }
            {
                // bottom edge: rows below row vh - 1 (chroma cvh - 1) repeat it; its owner is the lane of the same
                // macroblock and column group with rgrp = (vh - 1) >> 3 (chroma (cvh - 1) >> 2)
                const int f = (vh - 1) & 15, rf = f & 7;
                uint32_t own = yw[0];
#pragma unroll
                for (int k = 1; k < 8; k++) own = rf == k ? yw[k] : own;
                const uint32_t s = __shfl_sync(FULL, own, (lane & ~4) | ((f >> 3) << 2));
                if (fix_b && vh) {
#pragma unroll
                    for (int r = 0; r < 8; r++)
                        if (rgrp * 8 + r > f) yw[r] = s;
                }
                const int cf = (cvh - 1) & 7, crf = cf & 3;
                uint32_t cown = cw[0];
#pragma unroll
                for (int k = 1; k < 4; k++) cown = crf == k ? cw[k] : cown;
                const uint32_t cs = __shfl_sync(FULL, cown, (lane & ~4) | ((cf >> 2) << 2));
                if (fix_b && cvh) {
#pragma unroll
                    for (int r = 0; r < 4; r++)
                        if (rgrp * 4 + r > cf) cw[r] = cs;
                }
            }
        }

        // ---- BT.601 RGBA (bt601.rs:12-59): 4 pixels per row = 16 bytes; chroma row r >> 1, sample 0 for pixels 0-1
        // and sample 1 for pixels 2-3, all in this lane's registers ----
#if H263_RGBA_TMA
        if constexpr (OUT != OUT_YUV) __syncwarp();  // every lane has read its residuals: the RGBA tile may overwrite them
#endif
        if (OUT != OUT_YUV && (flags & MBF_RGBA)) {
#if H263_RGBA_MODE == 0 || H263_RGBA_MODE == 3
            const int kr = opaque(104597), kg = opaque(-53279), kb = opaque(132201), ky = opaque(76309);
#else
            const int kr = opaque(-104597), kg = opaque(53279), kb = opaque(-132201), ky = opaque(-76309);
#endif
#if H263_RGBA_TMA
            uint8_t* const stage = reinterpret_cast<uint8_t*>(&G);
#else
            const uint32_t rgba_pitch = PR ? PR : pools.rgba_pitch;
            uint8_t* const o = pools.rgba + (size_t)(ma.z + (uint32_t)(rgrp * 8)) * rgba_pitch + (size_t)(mv.y * 64u + (uint32_t)cg * 16u);
#endif
#pragma unroll
            for (int c2 = 0; c2 < 4; c2++) {
#if H263_RGBA_MODE >= 2
                // cw = (cb0, cr0, cb1, cr1): the samples come out as dot products with a one-hot selector (multiply pipe)
                const CT t0 = chroma_terms_folded((int)__dp4a(cw[c2], 1u, 0u), (int)__dp4a(cw[c2], 1u << 8, 0u), kr, kg, kb);
                const CT t1 = chroma_terms_folded((int)__dp4a(cw[c2], 1u << 16, 0u), (int)__dp4a(cw[c2], 1u << 24, 0u), kr, kg, kb);
#else
                const CT t0 = chroma_terms_folded((int)(cbp[c2] & 0xFFFFu), (int)(crp[c2] & 0xFFFFu), kr, kg, kb);
                const CT t1 = chroma_terms_folded((int)(cbp[c2] >> 16), (int)(crp[c2] >> 16), kr, kg, kb);
#endif
#pragma unroll
                for (int rr = 0; rr < 2; rr++) {
                    const int r = c2 * 2 + rr;
                    uint4 px;
                    px.x = rgba_px(yw[r], 0, ky, t0);
                    px.y = rgba_px(yw[r], 1, ky, t0);
                    px.z = rgba_px(yw[r], 2, ky, t1);
                    px.w = rgba_px(yw[r], 3, ky, t1);
#if H263_RGBA_TMA
                    *reinterpret_cast<uint4*>(stage + stage_offset(mbq, rgrp * 8 + r, cg)) = px;
#else
                    if (H263_ABLATE & 16) {  // RGBA computed, store suppressed (kept alive by an impossible condition)
                        if ((px.x ^ px.y ^ px.z ^ px.w) == 0x12345678u) *reinterpret_cast<uint4*>(o + (size_t)r * rgba_pitch) = px;
                    } else
                        *reinterpret_cast<uint4*>(o + (size_t)r * rgba_pitch) = px;
#endif
                }
            }
        }
#if H263_RGBA_TMA
        // generic-proxy writes -> async-proxy reads; then one TMA tensor store per macroblock: box = 64 bytes x 16
        // rows at (x = 64 mbx, y = the macroblock's first RGBA row) of the context's RGBA pool
        if constexpr (OUT != OUT_YUV) {
            asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
            __syncwarp();
            if (lane < n_w) {
                const uint32_t f = W.mba[lane].w & ~((H263_ABLATE & (4 | 16)) ? MBF_RGBA : 0u);
                if ((f & MBF_RGBA) && !(OUT == OUT_DEV_RGBA && EDGE && (f & MBF_RIGHT))) {
                    const uint32_t src = (uint32_t)__cvta_generic_to_shared(&G) + (uint32_t)lane * 1024u;
                    if constexpr (OUT == OUT_DEV_RGBA) {
                        // caller-owned buffer: 3-D map (bytes, rows, slots); the row word is slot << 12 | 16 mby
                        const uint32_t z = W.mba[lane].z;
                        asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.bulk_group [%0, {%2, %3, %4}], [%1];" ::"l"(&rgba_map),
                                     "r"(src), "r"((int)((f >> 8 & 0xFFu) * 64u)), "r"((int)(z & 0xFFFu)), "r"((int)(z >> 12))
                                     : "memory");
                    } else {
                        asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];" ::"l"(&rgba_map), "r"(src),
                                     "r"((int)((f >> 8 & 0xFFu) * 64u)), "r"((int)W.mba[lane].z)
                                     : "memory");
                    }
                    asm volatile("cp.async.bulk.commit_group;" ::: "memory");
                }
            }
            if constexpr (OUT == OUT_DEV_RGBA && EDGE) {
                // A tensor store writes whole 16-byte chunks, also where the tensor's row ends inside one: at the right edge
                // of a picture whose width is not a multiple of 4 it would write past the slot.  The right-edge macroblocks
                // (the only boxes that reach beyond 16 * floor(w / 16) pixels) leave through plain stores cut to the picture.
                for (int q = 0; q < n_w; q++) {
                    const uint32_t f = W.mba[q].w;
                    if (!(f & MBF_RGBA) || !(f & MBF_RIGHT)) continue;  // warp-uniform
                    const PicDev& P = pics[W.mbb[q].z];
                    const int px0 = (int)(f >> 8 & 0xFFu) * 16, py0 = (int)(W.mba[q].z & 0xFFFu);
                    for (int k = lane; k < 64; k += 32) {
                        const int row = k >> 2, c = k & 3, px = px0 + c * 4, py = py0 + row;
                        if (px < P.w && py < P.h)
                            store_rgba_quad(P.rgba + (size_t)py * P.rgba_pitch + (size_t)px * 4,
                                            *reinterpret_cast<const uint4*>(reinterpret_cast<const uint8_t*>(&G) + stage_offset(q, row, c)), P.w - px);
                    }
                }
            }
        }
#endif

        // (the plane stores come after the RGBA tile has been handed to the TMA unit, so that the unit reads the tile
        // while the warp is still busy: a warp may not leave before that read is over)
        // ---- plane stores (+ border replication for the next picture's prediction) ----
        if (unit_ok && !(H263_ABLATE & 8)) {
            const uint32_t pitch_y = pitch_y4 * 4, pitch_c = pitch_c4 * 4;
            uint8_t* py = pools.y + (size_t)(ma.x + (uint32_t)(rgrp * 8) * pitch_y4 + (uint32_t)cg) * 4;
            uint8_t* pc = pools.c + (size_t)(ma.y + (uint32_t)(rgrp * 4) * pitch_c4 + (uint32_t)cg) * 4;
#pragma unroll
            for (int r = 0; r < 8; r++) *reinterpret_cast<uint32_t*>(py + r * pitch_y) = yw[r];
#pragma unroll
            for (int r = 0; r < 4; r++) *reinterpret_cast<uint32_t*>(pc + r * pitch_c) = cw[r];
            // edges this lane owns: left for cg = 0, right for cg = 3, top for rgrp = 0, bottom for rgrp = 1.
            // 16 luma pixels / 8 CbCr pairs (16 bytes) of extension on each side, 16 / 8 rows above and below.
            const bool e_left = (flags & MBF_LEFT) && cg == 0, e_right = (flags & MBF_RIGHT) && cg == 3;
            const bool e_top = (flags & MBF_TOP) && rgrp == 0, e_bot = (flags & MBF_BOTTOM) && rgrp == 1;
            if (e_left | e_right | e_top | e_bot) {
                const ptrdiff_t side = e_left ? -16 : 4;  // of the 16 border bytes, from the lane's word
                if (e_left | e_right) {
#pragma unroll
                    for (int r = 0; r < 8; r++) {
                        const uint32_t v = __byte_perm(yw[r], 0, e_left ? 0x0000 : 0x3333);
                        *reinterpret_cast<uint4*>(py + r * pitch_y + side) = make_uint4(v, v, v, v);
                    }
#pragma unroll
                    for (int r = 0; r < 4; r++) {
                        const uint32_t v = __byte_perm(cw[r], 0, e_left ? 0x1010 : 0x3232);
                        *reinterpret_cast<uint4*>(pc + r * pitch_c + side) = make_uint4(v, v, v, v);
                    }
                }
                if (e_top | e_bot) {
                    // vertical extension, including the corners when the lane also sits on a vertical edge
                    const bool corner = e_left | e_right;
                    const uint32_t v = e_top ? yw[0] : yw[7];
                    uint8_t* rowp = e_top ? py : py + 7 * pitch_y;
                    const ptrdiff_t dir = e_top ? -(ptrdiff_t)pitch_y : (ptrdiff_t)pitch_y;
                    const uint32_t vc = __byte_perm(v, 0, e_left ? 0x0000 : 0x3333);
                    for (int k = 1; k <= 16; k++) {
                        uint8_t* d = rowp + k * dir;
                        *reinterpret_cast<uint32_t*>(d) = v;
                        if (corner) *reinterpret_cast<uint4*>(d + side) = make_uint4(vc, vc, vc, vc);
                    }
                    const uint32_t c = e_top ? cw[0] : cw[3];
                    uint8_t* rc = e_top ? pc : pc + 3 * pitch_c;
                    const ptrdiff_t cdir = e_top ? -(ptrdiff_t)pitch_c : (ptrdiff_t)pitch_c;
                    const uint32_t cc = __byte_perm(c, 0, e_left ? 0x1010 : 0x3232);
                    for (int k = 1; k <= 8; k++) {
                        uint8_t* d = rc + k * cdir;
                        *reinterpret_cast<uint32_t*>(d) = c;
                        if (corner) *reinterpret_cast<uint4*>(d + side) = make_uint4(cc, cc, cc, cc);
                    }
                }
            }
        }

        // ---- plane output (OUT_YUV): the same words into the caller's planes, cut to the picture ----
        if constexpr (OUT == OUT_YUV) {
            if (flags & MBF_RGBA) {
                const uint32_t slot = ma.z >> 12, mrow = ma.z & 0xFFFu;  // slot << 12 | 16 mby
                // bytes (luma) / samples (chroma) and rows of the lane that lie inside the picture: all of them but in
                // the right-edge / bottom-edge macroblocks of a picture whose size is not a multiple of 16
                int yv = 4, yr = 8, cv = 2, cr = 4;
                if constexpr (EDGE) {
                    const uint32_t ed = mv.w;
                    const int vw = (int)(ed & 15u), vh = (int)((ed >> 4) & 15u), cvw = (int)((ed >> 8) & 7u), cvh = (int)((ed >> 12) & 7u);
                    if (flags & MBF_RIGHT) {
                        if (vw) yv = vw - 4 * cg;
                        if (cvw) cv = cvw - 2 * cg;
                    }
                    if (flags & MBF_BOTTOM) {
                        if (vh) yr = vh - 8 * rgrp;
                        if (cvh) cr = cvh - 4 * rgrp;
                    }
                }
                uint8_t* const yd = yuv_row(yuv, 0, slot, mrow + (uint32_t)(rgrp * 8)) + mv.y * 16u + (uint32_t)cg * 4u;
#pragma unroll
                for (int r = 0; r < 8; r++)
                    if (r < yr) store_word_cut(yd + (size_t)r * yuv.pitch[0], yw[r], yv);
                const uint32_t crow = (mrow >> 1) + (uint32_t)(rgrp * 4), cx = mv.y * 8u + (uint32_t)cg * 2u;
                if (yuv.nv12) {
                    // CbCr pairs: the lane's chroma word as it stands
                    uint8_t* const cd = yuv_row(yuv, 1, slot, crow) + 2u * cx;
#pragma unroll
                    for (int r = 0; r < 4; r++)
                        if (r < cr) store_word_cut(cd + (size_t)r * yuv.pitch[1], cw[r], 2 * cv);
                } else {
                    // I420: (cb0 cr0 cb1 cr1) -> (cb0 cb1), (cr0 cr1)
                    uint8_t* const bd = yuv_row(yuv, 1, slot, crow) + cx;
                    uint8_t* const rd = yuv_row(yuv, 2, slot, crow) + cx;
#pragma unroll
                    for (int r = 0; r < 4; r++)
                        if (r < cr) {
                            store_pair_cut(bd + (size_t)r * yuv.pitch[1], __byte_perm(cw[r], 0, 0x0020), cv);
                            store_pair_cut(rd + (size_t)r * yuv.pitch[2], __byte_perm(cw[r], 0, 0x0031), cv);
                        }
                }
            }
        }

#if H263_RGBA_TMA
        // the tile must stay in place until the stores have read it
        if constexpr (OUT != OUT_YUV) asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory");
#endif
    }
}

int recon_tile_uses_tma() { return H263_RGBA_TMA; }

void launch_recon_tile(const PicDev* pics, const h263cu_mb* mbs, const h263cu_event* events, uint32_t n_mbs, int emit_rgba,
                       int unaligned, int wide_mv, const Pools& pools, const CUtensorMap* rgba_map, int out, const YuvDst* yuv,
                       cudaStream_t stream) {
    if (n_mbs == 0) return;
    // pitches of the standard formats (context.cu: pitch_y = pitch_c = 16 * mbw + 64, rgba = 64 * mbw)
    const uint32_t py = pools.pitch_y, pc = pools.pitch_c, pr = pools.rgba_pitch;
    const CUtensorMap& tm = *rgba_map;
    YuvDst yd{};
    if (yuv) yd = *yuv;
#define H263_LAUNCH1(PY_, PC_, PR_, EDGE_, WIDE_, NW_, NCTAS_, OUT_)                                                               \
    recon_tile_kernel<PY_, PC_, PR_, EDGE_, WIDE_, NW_, NCTAS_, OUT_>                                                              \
        <<<(n_mbs + NW_ * WARP_MBS - 1) / (NW_ * WARP_MBS), NW_ * 32, 0, stream>>>(pics, mbs, events, n_mbs, emit_rgba, pools, tm, yd)
#define H263_LAUNCH(PY_, PC_, PR_, EDGE_, WIDE_, NW_, NCTAS_)                  \
    do {                                                                       \
        if (out == OUT_YUV)                                                    \
            H263_LAUNCH1(PY_, PC_, PR_, EDGE_, WIDE_, NW_, NCTAS_, OUT_YUV);   \
        else if (out == OUT_DEV_RGBA)                                          \
            H263_LAUNCH1(PY_, PC_, PR_, EDGE_, WIDE_, NW_, NCTAS_, OUT_DEV_RGBA); \
        else                                                                   \
            H263_LAUNCH1(PY_, PC_, PR_, EDGE_, WIDE_, NW_, NCTAS_, OUT_POOL);  \
    } while (0)
    if (wide_mv) {  // hand-built side info with vectors beyond the range: clamped per-sample path, run-time pitches
        if (unaligned)
            H263_LAUNCH(0, 0, 0, true, true, GEN_WARPS, GEN_CTAS);
        else
            H263_LAUNCH(0, 0, 0, false, true, GEN_WARPS, GEN_CTAS);
    } else if (unaligned)  // some picture of the step is not a multiple of 16 in size: edge fix-up, run-time pitches
        H263_LAUNCH(0, 0, 0, true, false, GEN_WARPS, GEN_CTAS);
    else if (py == 416 && pc == 416 && pr == 1408)  // CIF 352x288
        H263_LAUNCH(416, 416, 1408, false, false, H263_STD_WARPS, H263_STD_CTAS);
    else if (py == 240 && pc == 240 && pr == 704)  // QCIF 176x144
        H263_LAUNCH(240, 240, 704, false, false, H263_STD_WARPS, H263_STD_CTAS);
    else if (py == 768 && pc == 768 && pr == 2816)  // 4CIF 704x576
        H263_LAUNCH(768, 768, 2816, false, false, H263_STD_WARPS, H263_STD_CTAS);
    else
        H263_LAUNCH(0, 0, 0, false, false, GEN_WARPS, GEN_CTAS);
#undef H263_LAUNCH
#undef H263_LAUNCH1
}

}  // namespace h263dev
