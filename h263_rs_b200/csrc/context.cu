// context.cu -- device context, step objects and the device half of the C ABI
// (include/h263cu.h).  The context owns all device memory: per stream two reconstruction
// slots (current / reference, ping-pong) for Y and the interleaved CbCr plane and a two-deep RGBA ring; side
// info arrives through pinned cudaMemcpyAsync.  Everything here is plumbing around the
// kernels in kernels.cu -- there is no CPU fallback: without a usable device the entry
// points return H263CU_ERR_NO_DEVICE / H263CU_ERR_CUDA.
#include <cuda_runtime.h>

#include <algorithm>
#include <chrono>
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <vector>

#include "device_math.cuh"
#include "kernels.cuh"

using namespace h263dev;

// frontend.cpp: the threaded parse with the parsers' state change held back until parse_step_finish(accept)
namespace h263fe {
int parse_step_deferred(h263cu_parser* const* parsers, const uint8_t* const* packets, const size_t* lens,
                        const uint32_t* stream_ids, uint32_t n, int threads, h263cu_pic* pics, h263cu_mb* mbs, uint32_t mb_cap,
                        h263cu_event* events, uint32_t ev_cap, uint32_t* n_pics_out, uint32_t* n_mbs_out, uint32_t* n_units_out,
                        int* per_pic_err, int32_t* pic_of_input, uint32_t max_w, uint32_t max_h, const uint32_t* min_size);
void parse_step_finish(h263cu_parser* const* parsers, uint32_t n, bool accept);
// ... and its device form (H263CU_PARSE_ON_DEVICE): the picture layer before and after parse_mb.cu's kernel
int device_parse_tables(uint32_t* out);
int device_parse_prepare(h263cu_parser* const* parsers, const uint8_t* const* packets, const size_t* lens, const uint32_t* stream_ids,
                         uint32_t n, int threads, uint32_t max_w, uint32_t max_h, const uint32_t* min_size, const uint64_t* pkt_off,
                         uint8_t* stage, h263cu_pic* pics, int* errs, h263dev::ParseJob* jobs, int32_t* job_of_input, uint32_t* n_jobs_out,
                         uint32_t* n_mbs_out, uint32_t* n_units_out);
void device_parse_finish(h263cu_parser* const* parsers, uint32_t n, const int32_t* job_of_input, const h263dev::ParseResult* res,
                         h263cu_pic* pics, int* errs);
}  // namespace h263fe

extern "C" const uint8_t h263cu_quant_to_strength[32] = H263_QUANT_TO_STRENGTH;

namespace {

#define CU_TRY(expr)                      \
    do {                                  \
        cudaError_t _e = (expr);          \
        if (_e != cudaSuccess) return map_cuda_error(_e); \
    } while (0)

int map_cuda_error(cudaError_t e) {
    switch (e) {
        case cudaErrorNoDevice:
        case cudaErrorInsufficientDriver:
        case cudaErrorInvalidDevice: return H263CU_ERR_NO_DEVICE;
        case cudaErrorMemoryAllocation: return H263CU_ERR_OUT_OF_MEMORY;
        default: return H263CU_ERR_CUDA;
    }
}

inline size_t round_up(size_t v, size_t a) { return (v + a - 1) / a * a; }

struct StreamState {
    bool has_pic = false;
    uint8_t cur_slot = 0;  // slot that holds the last decoded picture
    int8_t rgba_slot = -1; // ring slot that holds the last picture's RGBA (-1 = none)
    uint16_t w = 0, h = 0;
    uint8_t pic_type = 0, pquant = 0;
    uint16_t tr = 0;
    uint32_t stamp = 0;
    uint32_t seen = 0;    // epoch of the last h263cu_decode_step that named this stream (duplicate check)
    // the prediction source of the next picture: the last NON-disposable picture.  Identical to the last picture unless
    // the stream carries disposable P pictures (H263CU_PICFLAG_DISPOSABLE), which are shown but never predicted from.
    bool has_ref = false;
    uint8_t ref_slot = 0;
    uint16_t ref_w = 0, ref_h = 0;
    bool padded = false;  // the reference picture's planes carry the replicated border (tiled kernel)
};

// where the next picture of a stream is reconstructed: never over its prediction source
inline int next_slot(const StreamState& st) { return st.has_ref ? (st.ref_slot ^ 1) : (st.has_pic ? (st.cur_slot ^ 1) : 0); }

// state.rs:464-483 on the device side: the picture becomes the stream's last picture and, unless it is disposable,
// the reference of the next one
inline void advance_stream(StreamState& st, const h263cu_pic& p, bool want_rgba, int rgba_ring, bool tiled) {
    const int slot = next_slot(st);
    st.cur_slot = (uint8_t)slot;
    st.has_pic = true;
    st.w = p.width, st.h = p.height;
    st.pic_type = p.pic_type, st.pquant = p.pquant, st.tr = p.temporal_reference;
    st.rgba_slot = want_rgba ? (int8_t)rgba_ring : (int8_t)-1;
    if (!(p.flags & H263CU_PICFLAG_DISPOSABLE)) {
        st.has_ref = true;
        st.ref_slot = (uint8_t)slot;
        st.ref_w = p.width, st.ref_h = p.height;
        st.padded = tiled;
    }
}

}  // namespace

struct h263cu_step {
    std::vector<h263cu_pic> pics;
    h263cu_mb* d_mbs = nullptr;
    h263cu_event* d_events = nullptr;
    uint32_t n_mbs = 0, n_units = 0;
    size_t mb_cap = 0, ev_cap = 0;  // capacities in elements (ring reuse)
    uint32_t max_w = 0, max_h = 0;
};

struct h263cu_ctx {
    int device = 0;
    uint32_t max_streams = 0, max_w = 0, max_h = 0;
    uint32_t mbw = 0, mbh = 0;
    uint32_t pitch_y = 0, pitch_c = 0, rgba_pitch = 0;
    size_t y_slot = 0, c_slot = 0, rgba_slot = 0;
    uint8_t *y_pool = nullptr, *c_pool = nullptr, *rgba_pool = nullptr;  // c_pool: interleaved CbCr planes
    CUtensorMap rgba_map;  // TMA view of rgba_pool: rows of rgba_pitch bytes, box 64 bytes x 16 rows (one macroblock)
    std::vector<StreamState> streams;
    uint32_t stamp = 0, decode_epoch = 0;
    uint32_t rgba_parity = 0;

    cudaStream_t s_main = nullptr, s_h2d = nullptr, s_d2h = nullptr;
    cudaStream_t s_pics = nullptr;  // descriptor uploads: overlap the previous step's kernels
    // PicDev staging ring (pinned host + device)
    static constexpr int PIC_RING = 4;
    PicDev* h_pics[PIC_RING] = {};
    PicDev* d_pics[PIC_RING] = {};
    cudaEvent_t pics_done[PIC_RING] = {};  // the kernels that read d_pics[i] have finished
    cudaEvent_t pics_up[PIC_RING] = {};    // d_pics[i] is uploaded
    // the fit geometry of h263cu_decode_step_device_tensor_fit, one record per picture beside h_pics / d_pics (the same
    // capacity, the same events)
    FitGeom* h_geo[PIC_RING] = {};
    FitGeom* d_geo[PIC_RING] = {};
    size_t pics_cap = 0;
    int pic_ring_pos = 0;
    // side-info ring used by h263cu_submit_step*
    h263cu_step ring[2];
    cudaEvent_t ring_h2d_done[2] = {}, ring_run_done[2] = {};
    int ring_pos = 0;
    // pinned staging of h263cu_decode_step, one set per side-info ring slot (grow only)
    struct Staging {
        h263cu_pic* pics = nullptr;
        h263cu_mb* mbs = nullptr;
        h263cu_event* events = nullptr;
        size_t pic_cap = 0, mb_cap = 0, ev_cap = 0;
    } staging[2];
    std::vector<int32_t> pic_of_input;
    // H263CU_PARSE_ON_DEVICE: the VLC tables (uploaded on first use), the step's packets, jobs and results.  One set:
    // the call waits for the parse's results, and the next call's copies are queued behind this call's on s_parse.
    cudaStream_t s_parse = nullptr;
    cudaEvent_t parse_done = nullptr;  // the step's records and events are in the ring slot (compacted if needed)
    uint32_t* d_tables = nullptr;
    uint8_t *h_pkts = nullptr, *d_pkts = nullptr;
    size_t pkts_cap = 0, d_pkts_cap = 0;
    ParseJob *h_pjobs = nullptr, *d_pjobs = nullptr;
    ParseResult *h_res = nullptr, *d_res = nullptr;
    PackMove *h_moves = nullptr, *d_moves = nullptr;
    size_t pjobs_cap = 0, d_pjobs_cap = 0, res_cap = 0, d_res_cap = 0, moves_cap = 0, d_moves_cap = 0;
    h263cu_mb* d_mbs_tmp = nullptr;  // the records before compaction, when a picture of the step failed
    size_t mbs_tmp_cap = 0;
    std::vector<uint64_t> dp_pkt_off;  // per input (+ 1): the packet's offset in h_pkts / d_pkts
    std::vector<h263cu_pic> dp_pics;   // per input: the picture once the host has parsed its header
    std::vector<int> dp_errs;
    std::vector<int32_t> dp_job;       // per input: its job, or -1
    std::vector<PackMove> dp_moves;    // per decoded picture: where its records are and where they go
    uint32_t dp_mb_total = 0, dp_ev_total = 0;  // the ring slot's records and event units the kernel wrote
    std::vector<uint64_t> rgba_offsets;
    std::vector<uint32_t> dev_slots;  // h263cu_decode_step_device: slot of each packed picture in the caller's buffer
    std::vector<uint32_t> fit_min;    // h263cu_decode_step_device_tensor_fit: per input, the picture size its crop needs
    std::vector<FitGeom> fit_geo;     // ... and the geometry of each packed picture
    // h263cu_decode_step_device: the consumer stream's earlier work -> s_main, the step's RGBA -> the consumer stream
    cudaEvent_t dev_ready = nullptr, dev_done = nullptr;
    // h263cu_decode_step_device_tensor with H263CU_OUT_DEBLOCK: NV12 planes the deblock kernels write and the resample
    // kernel reads, picture i of a step in slot i (allocated on first use, grown as needed)
    uint8_t* tensor_scratch = nullptr;
    size_t tensor_scratch_slots = 0;
    // RGBA ring read-back tracking
    cudaEvent_t rgba_written[2] = {}, rgba_read[2] = {};
    // timing
    cudaEvent_t t0 = nullptr, t1 = nullptr;
    uint64_t launches = 0, tiled_launches = 0;
    // optional per-kernel timing (h263cu_profile_*): event pairs, kind 0 = recon, 1 = deblock
    bool profiling = false;
    std::vector<cudaEvent_t> prof_free;
    struct ProfSpan {
        cudaEvent_t a, b;
        int kind;
    };
    std::vector<ProfSpan> prof_spans;
    // checksum scratch
    ChecksumJob* d_jobs = nullptr;
    unsigned long long* d_sums = nullptr;
    size_t jobs_cap = 0;

    int force_kernel = 0;  // H263CU_KERNEL=mb|tile overrides the per-step choice (A/B checks)
    // host time spent inside h263cu_decode_step, split into the bitstream parse and everything else (staging, driver
    // calls): the north-star asks for the host parse time beside the device time
    double host_parse_s = 0.0, host_other_s = 0.0;
    uint64_t host_calls = 0;
    // interior origin (pixel 0,0) of a plane; the padding lies at negative offsets
    uint8_t* plane(int p, uint32_t stream, int slot) const {
        const size_t idx = (size_t)stream * 2 + (size_t)slot;
        if (p == 0) return y_pool + idx * y_slot + (size_t)PAD_Y_ROWS * pitch_y + PAD_Y_COLS;
        // Cb and Cr share one interleaved plane: Cr starts one byte after Cb, samples are CHROMA_STEP bytes apart
        return c_pool + idx * c_slot + (size_t)PAD_C_ROWS * pitch_c + PAD_C_COLS + (p == 2 ? 1 : 0);
    }
    uint8_t* rgba(uint32_t stream, int slot) const { return rgba_pool + ((size_t)slot * max_streams + stream) * rgba_slot; }
};

namespace {

int ensure_pic_ring(h263cu_ctx* c, size_t n) {
    if (n <= c->pics_cap) return 0;
    CU_TRY(cudaStreamSynchronize(c->s_main));
    size_t cap = std::max<size_t>(n, 256);
    for (int i = 0; i < h263cu_ctx::PIC_RING; i++) {
        if (c->h_pics[i]) cudaFreeHost(c->h_pics[i]);
        if (c->d_pics[i]) cudaFree(c->d_pics[i]);
        if (c->h_geo[i]) cudaFreeHost(c->h_geo[i]);
        if (c->d_geo[i]) cudaFree(c->d_geo[i]);
        c->h_pics[i] = nullptr, c->d_pics[i] = nullptr, c->h_geo[i] = nullptr, c->d_geo[i] = nullptr;
        CU_TRY(cudaHostAlloc((void**)&c->h_pics[i], cap * sizeof(PicDev), cudaHostAllocDefault));
        CU_TRY(cudaMalloc((void**)&c->d_pics[i], cap * sizeof(PicDev)));
        CU_TRY(cudaHostAlloc((void**)&c->h_geo[i], cap * sizeof(FitGeom), cudaHostAllocDefault));
        CU_TRY(cudaMalloc((void**)&c->d_geo[i], cap * sizeof(FitGeom)));
    }
    c->pics_cap = cap;
    return 0;
}

int step_reserve(h263cu_step* s, size_t n_mbs, size_t n_units) {
    if (n_mbs > s->mb_cap) {
        if (s->d_mbs) cudaFree(s->d_mbs);
        s->d_mbs = nullptr;
        size_t cap = n_mbs + n_mbs / 8 + 64;
        CU_TRY(cudaMalloc((void**)&s->d_mbs, cap * sizeof(h263cu_mb)));
        s->mb_cap = cap;
    }
    if (n_units + 8 > s->ev_cap) {
        if (s->d_events) cudaFree(s->d_events);
        s->d_events = nullptr;
        size_t cap = n_units + n_units / 8 + 64;
        CU_TRY(cudaMalloc((void**)&s->d_events, cap * sizeof(h263cu_event)));
        s->ev_cap = cap;
    }
    return 0;
}

int prof_take(h263cu_ctx* c, cudaEvent_t* a, cudaEvent_t* b) {
    for (cudaEvent_t* e : {a, b}) {
        if (!c->prof_free.empty()) {
            *e = c->prof_free.back();
            c->prof_free.pop_back();
        } else {
            CU_TRY(cudaEventCreate(e));
        }
    }
    return 0;
}
void prof_end(h263cu_ctx* c, cudaEvent_t a, cudaEvent_t b, int kind) {
    cudaEventRecord(b, c->s_main);
    c->prof_spans.push_back({a, b, kind});
}

// The device-side descriptor of one picture, given the state of its stream BEFORE the picture (run_step and the graph
// builder, which walks a simulated copy of the state, share it).
PicDev make_picdev(const h263cu_ctx* c, const h263cu_pic& p, const StreamState& st, bool want_rgba, int rgba_ring) {
    const int ref_slot = st.ref_slot, new_slot = next_slot(st);
    PicDev d;
    std::memset(&d, 0, sizeof(d));
    for (int k = 0; k < 3; k++) {
        d.cur[k] = c->plane(k, p.stream, new_slot);
        d.ref[k] = st.has_ref ? c->plane(k, p.stream, ref_slot) : nullptr;
    }
    d.rgba = want_rgba ? c->rgba(p.stream, rgba_ring) : nullptr;
    d.cur_y4 = (uint32_t)((d.cur[0] - c->y_pool) >> 2);
    d.cur_c4 = (uint32_t)((d.cur[1] - c->c_pool) >> 2);
    d.ref_y4 = st.has_ref ? (uint32_t)((d.ref[0] - c->y_pool) >> 2) : 0u;
    d.ref_c4 = st.has_ref ? (uint32_t)((d.ref[1] - c->c_pool) >> 2) : 0u;
    d.rgba_row0 = want_rgba ? (uint32_t)((size_t)(d.rgba - c->rgba_pool) / c->rgba_pitch) : 0u;
    d.first_event = p.first_event;
    d.rgba_pitch = c->rgba_pitch;
    d.w = p.width, d.h = p.height;
    d.cw = (uint16_t)((p.width + 1) / 2), d.ch = (uint16_t)((p.height + 1) / 2);
    d.pitch_y = (uint16_t)c->pitch_y, d.pitch_c = (uint16_t)c->pitch_c;
    d.strength = h263cu_quant_to_strength[p.pquant & 31];
    d.flags = p.flags;
    return d;
}

// Output into caller-owned device memory: RGBA (h263cu_decode_step_device: the tensor map over the buffer, its base,
// pitch and stride) or the planes (h263cu_decode_step_device_yuv: `yuv`), the slot of every picture of the step and
// the consumer stream to order against.
struct DeviceTarget {
    int out;  // OUT_DEV_RGBA, OUT_YUV or OUT_TENSOR
    CUtensorMap map;
    uint8_t* base;
    uint64_t row_pitch, pic_stride;
    YuvDst yuv;
    TensorDst tensor;  // OUT_TENSOR (h263cu_decode_step_device_tensor)
    uint32_t dtype;
    const FitGeom* geo;  // OUT_TENSOR with a fit: the geometry of every picture of the step (host), else null
    float fill[3];
    uint32_t filter;     // OUT_TENSOR with a fit: H263CU_FILTER_* (resample_filter_kernel for the antialiased ones)
    const uint32_t* slots;
    cudaStream_t stream;
};

// The NV12 scratch planes of OUT_TENSOR with deblocking, `n` slots of the context's largest picture: the deblock
// kernels' plane-output form writes slot i of them for picture i, resample_rgb_kernel reads them.  Grown on demand
// (after the kernels that read the old allocation have finished); nothing is enqueued.
int ensure_tensor_scratch(h263cu_ctx* c, uint32_t n, YuvDst* d) {
    const size_t pitch = (size_t)c->mbw * 16, y_bytes = pitch * c->mbh * 16, c_bytes = pitch * c->mbh * 8;
    if (n > c->tensor_scratch_slots) {
        CU_TRY(cudaStreamSynchronize(c->s_main));
        if (c->tensor_scratch) cudaFree(c->tensor_scratch);
        c->tensor_scratch = nullptr, c->tensor_scratch_slots = 0;
        const size_t slots = std::max<size_t>(n, 64);
        CU_TRY(cudaMalloc((void**)&c->tensor_scratch, slots * (y_bytes + c_bytes)));
        c->tensor_scratch_slots = slots;
    }
    std::memset(d, 0, sizeof(*d));
    d->base[0] = c->tensor_scratch, d->base[1] = c->tensor_scratch + c->tensor_scratch_slots * y_bytes;
    d->stride[0] = y_bytes, d->stride[1] = c_bytes;
    d->pitch[0] = d->pitch[1] = (uint32_t)pitch;
    d->nv12 = 1;
    return 0;
}

// Validates a step against the context and the per-stream state, builds the PicDev array,
// enqueues the kernels on s_main and advances the per-stream reference bookkeeping
// (state.rs:464-483: the picture just decoded becomes the reference of the next one).
// Nothing of the per-stream state changes unless the kernels have been enqueued: a step that is
// refused, or that fails on the way to the launch, leaves every stream as it was.
// With `dev` the RGBA (or with dev->out == OUT_YUV, the planes and no RGBA; with OUT_TENSOR, the resampled tensor and
// no RGBA) goes to the caller's buffers instead of the pool ring, which is neither written nor waited on.
int run_step(h263cu_ctx* c, h263cu_step* s, uint32_t out_flags, bool lean = false, const DeviceTarget* dev = nullptr) {
    const uint32_t n = (uint32_t)s->pics.size();
    if (n == 0) return 0;
    if (n > 65535) return H263CU_ERR_CAPACITY;  // h263cu_mb.pic is 16 bits wide
    const bool want_rgba = dev || (out_flags & H263CU_OUT_RGBA) != 0;
    const bool pool_rgba = want_rgba && !dev;
    const bool want_deblock = want_rgba && (out_flags & H263CU_OUT_DEBLOCK) != 0;
    const bool tensor = dev && dev->out == OUT_TENSOR;
    const uint32_t stamp = ++c->stamp;  // marks the streams named by this step (duplicate check only)
    uint32_t max_w = 0, max_h = 0;
    bool tiled = true, aligned16 = true, wide_mv = false;
    for (uint32_t i = 0; i < n; i++) {
        const h263cu_pic& p = s->pics[i];
        if (p.stream >= c->max_streams) return H263CU_ERR_CAPACITY;
        if (p.width == 0 || p.height == 0 || p.width > c->max_w || p.height > c->max_h) return H263CU_ERR_CAPACITY;
        if ((uint32_t)p.mb_w * 16 < p.width || (uint32_t)p.mb_h * 16 < p.height ||
            (uint32_t)p.mb_w > c->mbw || (uint32_t)p.mb_h > c->mbh)
            return H263CU_ERR_BAD_ARGUMENT;
        if ((uint64_t)p.first_mb + p.n_mbs > s->n_mbs || (uint64_t)p.first_event + p.n_event_units > s->n_units ||
            p.n_mbs != (uint32_t)p.mb_w * p.mb_h)
            return H263CU_ERR_BAD_ARGUMENT;
        StreamState& st = c->streams[p.stream];
        if (st.stamp == stamp) return H263CU_ERR_BAD_ARGUMENT;  // a stream appears once per step
        st.stamp = stamp;
        if (p.flags & H263CU_PICFLAG_HAS_INTER) {
            if (!st.has_ref) return H263CU_ERR_UNCODED_IFRAME_BLOCKS;             // gather.rs:149
            if (st.ref_w != p.width || st.ref_h != p.height) return H263CU_ERR_REFERENCE_WOULD_ABORT;
        }
        max_w = std::max<uint32_t>(max_w, p.width);
        max_h = std::max<uint32_t>(max_h, p.height);
        // the tiled kernel needs references with a replicated border; sizes that are not multiples of 16 take its
        // edge fix-up instantiation, and the register-resident deblock kernel needs aligned pictures
        if ((p.width | p.height) & 15) aligned16 = false;
        if ((p.flags & H263CU_PICFLAG_HAS_INTER) && !(p.flags & H263CU_PICFLAG_MV_IN_RANGE)) wide_mv = true;
        if ((p.flags & H263CU_PICFLAG_HAS_INTER) && !st.padded) tiled = false;
    }
    if (c->force_kernel == 1) tiled = false;
    int e = ensure_pic_ring(c, n);
    if (e) return e;
    YuvDst scratch{};
    if (tensor && want_deblock && (e = ensure_tensor_scratch(c, n, &scratch))) return e;
    const int slot = c->pic_ring_pos;
    CU_TRY(cudaEventSynchronize(c->pics_done[slot]));
    const int rgba_ring = (int)(c->rgba_parity & 1u);
    PicDev* hp = c->h_pics[slot];
    const bool fit = tensor && dev->geo;
    if (fit) std::memcpy(c->h_geo[slot], dev->geo, n * sizeof(FitGeom));
    for (uint32_t i = 0; i < n; i++) {
        const h263cu_pic& p = s->pics[i];
        PicDev d = make_picdev(c, p, c->streams[p.stream], pool_rgba, rgba_ring);
        if (tensor) {
            // the deblock kernels write slot i of the scratch planes for every picture whose rgba is set
            d.rgba = want_deblock ? yuv_row(scratch, 0, i, 0) : nullptr;
            d.rgba_row0 = i << 12;
            d.out_slot = dev->slots[i];
        } else if (dev) {
            if (dev->out == OUT_YUV) {  // the kernels take the destination from dev->yuv; rgba marks the picture as output
                d.rgba = yuv_row(dev->yuv, 0, dev->slots[i], 0);
                d.rgba_pitch = dev->yuv.pitch[0];
            } else {
                d.rgba = dev->base + (size_t)dev->slots[i] * dev->pic_stride;
                d.rgba_pitch = (uint32_t)dev->row_pitch;
            }
            d.rgba_row0 = dev->slots[i] << 12;
        }
        hp[i] = d;
    }
    cudaEvent_t pa = nullptr, pb = nullptr, qa = nullptr, qb = nullptr;
    if (c->profiling) {
        // the event pairs are taken before anything is enqueued: a failure here leaves no trace
        if ((e = prof_take(c, &pa, &pb))) return e;
        if (want_deblock && (e = prof_take(c, &qa, &qb))) {
            c->prof_free.push_back(pa), c->prof_free.push_back(pb);
            return e;
        }
    }
    // the descriptors travel on their own stream, so the copy overlaps the previous step's kernels
    // (pics_done[slot] was waited for above: the kernels that read this ring slot four steps ago are done).
    // Lean form (one small step, e.g. a single stream's picture): everything goes to s_main in order -- there is
    // nothing to overlap, and every driver call saved is a microsecond or two of the caller's time per picture.
    if (lean) {
        CU_TRY(cudaMemcpyAsync(c->d_pics[slot], hp, n * sizeof(PicDev), cudaMemcpyHostToDevice, c->s_main));
        if (fit) CU_TRY(cudaMemcpyAsync(c->d_geo[slot], c->h_geo[slot], n * sizeof(FitGeom), cudaMemcpyHostToDevice, c->s_main));
    } else {
        CU_TRY(cudaMemcpyAsync(c->d_pics[slot], hp, n * sizeof(PicDev), cudaMemcpyHostToDevice, c->s_pics));
        if (fit) CU_TRY(cudaMemcpyAsync(c->d_geo[slot], c->h_geo[slot], n * sizeof(FitGeom), cudaMemcpyHostToDevice, c->s_pics));
        CU_TRY(cudaEventRecord(c->pics_up[slot], c->s_pics));
        CU_TRY(cudaStreamWaitEvent(c->s_main, c->pics_up[slot], 0));
    }
    if (pool_rgba) {
        // do not overwrite an RGBA ring slot that is still being read back
        CU_TRY(cudaStreamWaitEvent(c->s_main, c->rgba_read[rgba_ring], 0));
    }
    if (dev) {
        // the caller's buffer is written only after everything queued on its stream so far (which may still read it)
        CU_TRY(cudaEventRecord(c->dev_ready, dev->stream));
        CU_TRY(cudaStreamWaitEvent(c->s_main, c->dev_ready, 0));
    }
    if (pa) cudaEventRecord(pa, c->s_main);
    const Pools pools{c->y_pool, c->c_pool, c->rgba_pool, c->pitch_y, c->pitch_c, c->rgba_pitch};
    // OUT_TENSOR: the recon kernel runs as for a step without RGBA, the deblock kernels write the scratch planes
    const YuvDst* yuv = dev && dev->out == OUT_YUV ? &dev->yuv : tensor && want_deblock ? &scratch : nullptr;
    const bool dev_out = dev && !tensor;
    launch_recon(c->d_pics[slot], s->d_mbs, s->d_events, s->n_mbs, want_rgba && !want_deblock && !tensor, tiled ? (aligned16 ? 1 : 2) : 0,
                 wide_mv, pools, dev_out ? &dev->map : &c->rgba_map, dev_out ? dev->out : OUT_POOL, yuv, c->s_main);
    if (pa) prof_end(c, pa, pb, 0);
    if (want_deblock) {
        if (qa) cudaEventRecord(qa, c->s_main);
        if (aligned16 && c->force_kernel != 1)
            launch_deblock_rgba_tile(c->d_pics[slot], n, max_w, max_h, yuv, c->s_main);
        else
            launch_deblock_rgba(c->d_pics[slot], n, max_w, max_h, yuv, c->s_main);
        if (qa) prof_end(c, qa, qb, 1);
    }
    if (tensor) {
        const FitArgs fa{c->d_geo[slot], {dev->fill[0], dev->fill[1], dev->fill[2]}};
        if (fit && dev->filter != H263CU_FILTER_BILINEAR)
            launch_resample_filter(c->d_pics[slot], n, want_deblock ? &scratch : nullptr, dev->tensor, dev->dtype, dev->filter, fa,
                                   c->s_main);
        else
            launch_resample_rgb(c->d_pics[slot], n, want_deblock ? &scratch : nullptr, dev->tensor, dev->dtype, fit ? &fa : nullptr,
                                c->s_main);
    }
    CU_TRY(cudaGetLastError());
    // ---- the step is on the device: commit the bookkeeping ----
    c->pic_ring_pos = (c->pic_ring_pos + 1) % h263cu_ctx::PIC_RING;
    c->launches += (want_deblock ? 2 : 1) + (tensor ? 1 : 0);
    if (tiled) c->tiled_launches++;
    for (uint32_t i = 0; i < n; i++) advance_stream(c->streams[s->pics[i].stream], s->pics[i], pool_rgba, rgba_ring, tiled);
    CU_TRY(cudaEventRecord(c->pics_done[slot], c->s_main));
    if (dev) {
        // work the caller queues on its stream from now on sees the pictures
        CU_TRY(cudaEventRecord(c->dev_done, c->s_main));
        CU_TRY(cudaStreamWaitEvent(dev->stream, c->dev_done, 0));
    }
    if (pool_rgba) {
        if (!lean) CU_TRY(cudaEventRecord(c->rgba_written[rgba_ring], c->s_main));  // lean: the read-back follows on s_main
        c->rgba_parity++;
    }
    return 0;
}

// Checks caller-built side info before it goes to the device, where the kernels index with it unchecked: every
// record belongs to the picture whose range it lies in and sits at its raster position, its events stay inside the
// picture's share of the event array, no block holds more events than a block can (64, intra 63) or events under a
// dropped intra DC.  HAS_INTER / MV_IN_RANGE are derived from the records, not taken on trust: a
// picture with an inter macroblock gets HAS_INTER, one with a vector beyond [-32, 31] loses MV_IN_RANGE (and takes
// the clamped-fetch instantiation).  Side info produced by the library's own parser skips this pass.
int validate_side_info(std::vector<h263cu_pic>& pics, const h263cu_mb* mbs, uint32_t n_mbs, uint32_t n_units) {
    for (size_t i = 0; i < pics.size(); i++) {
        h263cu_pic& p = pics[i];
        if ((uint64_t)p.first_mb + p.n_mbs > n_mbs || (uint64_t)p.first_event + p.n_event_units > n_units ||
            p.n_mbs != (uint32_t)p.mb_w * p.mb_h || p.mb_w == 0)
            return H263CU_ERR_BAD_ARGUMENT;
        bool any_inter = false, in_range = true;
        const h263cu_mb* m = mbs + p.first_mb;
        for (uint32_t k = 0; k < p.n_mbs; k++, m++) {
            if (m->pic != i || (uint32_t)m->mby * p.mb_w + m->mbx != k || m->mbx >= p.mb_w) return H263CU_ERR_BAD_ARGUMENT;
            // Per block: at most 64 events (63 for intra, whose DC takes zig-zag index 0), and none under an intra DC
            // code 0 (a dropped block).  The tiled kernel walks 64 events of a block at most and would read the rest
            // from past its event buffer; a dropped intra block would be transformed without its DC.
            const bool intra = !(m->flags & H263CU_MB_INTER);
            uint32_t ev = 0;
            for (int b = 0; b < 6; b++) {
                if (m->nev[b] > (intra ? 63 : 64) || (intra && m->nev[b] && m->u.intradc[b] == 0)) return H263CU_ERR_BAD_ARGUMENT;
                ev += m->nev[b];
            }
            if (m->flags & H263CU_MB_WIDE) ev *= 2;
            if ((uint64_t)m->ev_off + ev > p.n_event_units) return H263CU_ERR_BAD_ARGUMENT;
            if (m->flags & H263CU_MB_INTER) {
                any_inter = true;
                for (int b = 0; b < 4; b++)
                    in_range &= m->u.mv[b][0] >= -32 && m->u.mv[b][0] <= 31 && m->u.mv[b][1] >= -32 && m->u.mv[b][1] <= 31;
            }
        }
        if (any_inter) p.flags |= H263CU_PICFLAG_HAS_INTER;
        if (!in_range) p.flags &= (uint8_t)~H263CU_PICFLAG_MV_IN_RANGE;
    }
    return 0;
}

int upload_into(h263cu_ctx* c, h263cu_step* s, const h263cu_pic* pics, uint32_t n_pics, const h263cu_mb* mbs,
                uint32_t n_mbs, const h263cu_event* events, uint32_t n_units, cudaStream_t stream, bool trusted) {
    int e = step_reserve(s, n_mbs, n_units);
    if (e) return e;
    try {
        s->pics.assign(pics, pics + n_pics);
    } catch (const std::bad_alloc&) {
        return H263CU_ERR_OUT_OF_MEMORY;
    }
    s->n_mbs = n_mbs, s->n_units = n_units;
    if (!trusted && (e = validate_side_info(s->pics, mbs, n_mbs, n_units))) {
        s->pics.clear();
        return e;
    }
    if (n_mbs) CU_TRY(cudaMemcpyAsync(s->d_mbs, mbs, (size_t)n_mbs * sizeof(h263cu_mb), cudaMemcpyHostToDevice, stream));
    if (n_units)
        CU_TRY(cudaMemcpyAsync(s->d_events, events, (size_t)n_units * sizeof(h263cu_event), cudaMemcpyHostToDevice, stream));
    (void)c;
    return 0;
}

template <typename T>
int grow_pinned(T** p, size_t* cap, size_t need) {
    if (need <= *cap) return 0;
    if (*p) cudaFreeHost(*p);
    *p = nullptr, *cap = 0;
    const size_t n = need + need / 4 + 64;
    CU_TRY(cudaHostAlloc((void**)p, n * sizeof(T), cudaHostAllocDefault));
    *cap = n;
    return 0;
}
// device memory, grown like grow_pinned (nothing may be using the old allocation)
template <typename T>
int grow_device(T** p, size_t* cap, size_t need) {
    if (need <= *cap) return 0;
    if (*p) cudaFree(*p);
    *p = nullptr, *cap = 0;
    const size_t n = need + need / 4 + 64;
    CU_TRY(cudaMalloc((void**)p, n * sizeof(T)));
    *cap = n;
    return 0;
}

// cuTensorMapEncodeTiled through the runtime's driver entry point (the library does not link libcuda), looked up once
typedef CUresult (*EncodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiled encode_tiled() {
    static const EncodeTiled fn = [] {
        EncodeTiled enc = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", (void**)&enc, cudaEnableDefault, &q) != cudaSuccess) {
            cudaGetLastError();
            enc = nullptr;
        }
        return enc;
    }();
    return fn;
}
// RGBA byte maps with a box of one macroblock (64 bytes x 16 rows): rank 2 over the pool (dims = {pitch, rows}), rank 3
// over a caller's buffer (dims = {bytes per row, rows, slots}); strides[] holds the rank - 1 byte strides
int encode_rgba_map(CUtensorMap* map, void* base, uint32_t rank, const cuuint64_t* dims, const cuuint64_t* strides) {
    const EncodeTiled enc = encode_tiled();
    if (!enc) return H263CU_ERR_CUDA;
    const cuuint32_t box[3] = {64, 16, 1}, es[3] = {1, 1, 1};
    if (enc(map, CU_TENSOR_MAP_DATA_TYPE_UINT8, rank, base, dims, strides, box, es, CU_TENSOR_MAP_INTERLEAVE_NONE,
            CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
        return H263CU_ERR_CUDA;
    return 0;
}
int make_rgba_map(CUtensorMap* map, void* base, uint64_t pitch, uint64_t rows) {
    std::memset(map, 0, sizeof(*map));
    if (!recon_tile_uses_tma()) return 0;
    const cuuint64_t dims[2] = {pitch, rows}, strides[1] = {pitch};
    return encode_rgba_map(map, base, 2, dims, strides);
}
// 0 when cudaPointerGetAttributes reports `p` as device or managed memory of the context's device
int check_device_memory(const h263cu_ctx* c, const void* p) {
    cudaPointerAttributes a;
    if (cudaPointerGetAttributes(&a, p) != cudaSuccess) {
        cudaGetLastError();
        return H263CU_ERR_BAD_ARGUMENT;
    }
    if ((a.type != cudaMemoryTypeDevice && a.type != cudaMemoryTypeManaged) || a.device != c->device) return H263CU_ERR_BAD_ARGUMENT;
    return 0;
}
// The argument rules of h263cu_decode_step_device (include/h263cu.h), checked before anything is parsed
int check_device_rgba(const h263cu_ctx* c, const h263cu_device_rgba* o) {
    if (!o || !recon_tile_uses_tma()) return H263CU_ERR_BAD_ARGUMENT;
    if (!o->base || ((uintptr_t)o->base & 15u) || o->width == 0 || o->height == 0) return H263CU_ERR_BAD_ARGUMENT;
    if (o->row_pitch % 16 || o->row_pitch < 4ull * o->width || o->row_pitch >= (1ull << 32)) return H263CU_ERR_BAD_ARGUMENT;
    // TMA strides are below 2^40 bytes
    if (o->pic_stride % 16 || o->pic_stride < o->row_pitch * o->height || o->pic_stride >= (1ull << 40)) return H263CU_ERR_BAD_ARGUMENT;
    return check_device_memory(c, o->base);
}
// The argument rules of h263cu_decode_step_device_yuv (include/h263cu.h), checked before anything is parsed.  Plain
// stores of 4-byte words (16-bit and bytes at a row's end) need 4-byte alignment only; the 2^40 bound on strides is
// the RGBA form's.
int check_device_yuv(const h263cu_ctx* c, const h263cu_device_yuv* o) {
    if (!o || o->format > H263CU_YUV_NV12 || o->reserved != 0 || o->width == 0 || o->height == 0) return H263CU_ERR_BAD_ARGUMENT;
    const bool nv12 = o->format == H263CU_YUV_NV12;
    const uint64_t cw = (o->width + 1ull) / 2, ch = (o->height + 1ull) / 2;
    const uint64_t row_bytes[3] = {o->width, nv12 ? 2 * cw : cw, cw}, rows[3] = {o->height, ch, ch};
    if (nv12 && (o->plane[2].base || o->plane[2].row_pitch || o->plane[2].pic_stride)) return H263CU_ERR_BAD_ARGUMENT;
    for (int k = 0; k < (nv12 ? 2 : 3); k++) {
        const h263cu_device_plane& p = o->plane[k];
        if (!p.base || ((uintptr_t)p.base & 3u) || p.row_pitch % 4 || p.pic_stride % 4) return H263CU_ERR_BAD_ARGUMENT;
        if (p.row_pitch < row_bytes[k] || p.row_pitch >= (1ull << 32)) return H263CU_ERR_BAD_ARGUMENT;
        if (p.pic_stride < p.row_pitch * rows[k] || p.pic_stride >= (1ull << 40)) return H263CU_ERR_BAD_ARGUMENT;
    }
    for (int k = 0; k < (nv12 ? 2 : 3); k++)
        if (int e = check_device_memory(c, o->plane[k].base)) return e;
    return 0;
}
// The argument rules of h263cu_decode_step_device_tensor (include/h263cu.h), checked before anything is parsed
int check_device_tensor(const h263cu_ctx* c, const h263cu_device_tensor* o) {
    if (!o || o->dtype > H263CU_TENSOR_BF16 || o->reserved != 0) return H263CU_ERR_BAD_ARGUMENT;
    if (o->width == 0 || o->height == 0 || o->width > 16384 || o->height > 16384) return H263CU_ERR_BAD_ARGUMENT;
    static const uint32_t elem_bytes[4] = {1, 4, 2, 2};
    const uint32_t es = elem_bytes[o->dtype];
    if (!o->base || (uintptr_t)o->base % es) return H263CU_ERR_BAD_ARGUMENT;
    for (int k = 0; k < 4; k++)
        if (o->stride[k] <= 0) return H263CU_ERR_BAD_ARGUMENT;
    // bytes from element [s][0][0][0] to one past [s][2][height - 1][width - 1]; 128-bit: a stride may be up to 2^63
    const unsigned __int128 extent = ((unsigned __int128)(o->width - 1) * (uint64_t)o->stride[3] +
                                      (unsigned __int128)(o->height - 1) * (uint64_t)o->stride[2] +
                                      (unsigned __int128)2 * (uint64_t)o->stride[1] + 1) * es;
    if (extent >= ((unsigned __int128)1 << 40)) return H263CU_ERR_BAD_ARGUMENT;
    for (int k = 0; k < 3; k++) {
        if (!std::isfinite(o->mul[k]) || !std::isfinite(o->add[k])) return H263CU_ERR_BAD_ARGUMENT;
        if (o->dtype == H263CU_TENSOR_U8 && (o->mul[k] != 1.0f || o->add[k] != 0.0f)) return H263CU_ERR_BAD_ARGUMENT;
    }
    return check_device_memory(c, o->base);
}
// The argument rules of h263cu_decode_step_device_tensor_fit (include/h263cu.h) for n inputs, before anything is parsed
int check_tensor_fit(const h263cu_tensor_fit* f, uint32_t n) {
    if (!f || f->mode > H263CU_FIT_CENTER_CROP || f->reserved != 0) return H263CU_ERR_BAD_ARGUMENT;
    if (f->mode == H263CU_FIT_CENTER_CROP ? f->short_side < 1 || f->short_side > 16384 : f->short_side != 0)
        return H263CU_ERR_BAD_ARGUMENT;
    for (int k = 0; k < 3; k++)
        if (!(f->fill[k] >= 0.0f && f->fill[k] <= 255.0f)) return H263CU_ERR_BAD_ARGUMENT;  // NaN fails too
    if (f->crops)
        for (uint32_t i = 0; i < n; i++) {
            const h263cu_tensor_crop& b = f->crops[i];
            if (b.width == 0 || b.height == 0 || (uint64_t)b.x + b.width > 0xFFFFFFFFull || (uint64_t)b.y + b.height > 0xFFFFFFFFull)
                return H263CU_ERR_BAD_ARGUMENT;
        }
    return 0;
}
// The fit geometry of include/h263cu.h: resized size and placement {rw, rh, px, py} of a cw x ch crop in a W x H output
// (arguments within the ranges check_tensor_fit and check_device_tensor enforce; cw, ch < 2^16)
void fit_geometry(uint32_t mode, uint32_t short_side, uint32_t cw, uint32_t ch, uint32_t W, uint32_t H, int32_t* out4) {
    const int64_t w = cw, h = ch, ow = W, oh = H, S = short_side;
    int64_t rw = ow, rh = oh, px = 0, py = 0;
    if (mode == H263CU_FIT_LETTERBOX) {
        if (w * oh >= h * ow)
            rh = std::max<int64_t>(1, (2 * h * ow + w) / (2 * w));
        else
            rw = std::max<int64_t>(1, (2 * w * oh + h) / (2 * h));
        px = (ow - rw) / 2, py = (oh - rh) / 2;  // rw <= W and rh <= H: floored
    } else if (mode == H263CU_FIT_CENTER_CROP) {
        if (w <= h)
            rw = S, rh = S * h / w;
        else
            rh = S, rw = S * w / h;
        // torchvision: padding (o - r) // 2 on the left of a short axis, crop anchor round((r - o) / 2) (half to even)
        const auto place = [](int64_t r, int64_t o) -> int64_t {
            if (r < o) return (o - r) / 2;
            const int64_t d = r - o, k = d / 2;
            return -((d & 1) ? k + (k & 1) : k);
        };
        px = place(rw, ow), py = place(rh, oh);
    }
    out4[0] = (int32_t)rw, out4[1] = (int32_t)rh, out4[2] = (int32_t)px, out4[3] = (int32_t)py;
}
void free_step_buffers(h263cu_step* s) {
    if (s->d_mbs) cudaFree(s->d_mbs);
    if (s->d_events) cudaFree(s->d_events);
    s->d_mbs = nullptr, s->d_events = nullptr;
    s->mb_cap = s->ev_cap = 0;
}

}  // namespace

extern "C" {

int h263cu_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    return n;
}

h263cu_ctx* h263cu_create(int device, uint32_t max_streams, uint32_t max_width, uint32_t max_height, uint32_t flags,
                          int* err) {
    (void)flags;
    int dummy;
    if (!err) err = &dummy;
    *err = 0;
    if (max_streams == 0 || max_width == 0 || max_height == 0 || max_width > 4080 || max_height > 4080) {
        *err = H263CU_ERR_BAD_ARGUMENT;
        return nullptr;
    }
    int ndev = 0;
    cudaError_t ce = cudaGetDeviceCount(&ndev);
    if (ce != cudaSuccess || ndev == 0) {
        cudaGetLastError();
        *err = H263CU_ERR_NO_DEVICE;
        return nullptr;
    }
    if (device < 0 || device >= ndev) {
        *err = H263CU_ERR_NO_DEVICE;
        return nullptr;
    }
    if (cudaSetDevice(device) != cudaSuccess) {
        *err = H263CU_ERR_CUDA;
        return nullptr;
    }
    h263cu_ctx* c = new (std::nothrow) h263cu_ctx();
    if (!c) {
        *err = H263CU_ERR_OUT_OF_MEMORY;
        return nullptr;
    }
    c->device = device;
    c->max_streams = max_streams, c->max_w = max_width, c->max_h = max_height;
    c->mbw = (max_width + 15) / 16, c->mbh = (max_height + 15) / 16;
    // planes are MB-rounded so that whole-macroblock stores never need predication; the
    // padding is never read as picture content (sample coordinates clamp to the true size)
    // plus a border (PAD_*) into which the tiled kernel replicates the edge pixels, so that
    // motion compensation needs no per-sample clamping (unrestricted-MV extension)
    c->pitch_y = c->mbw * 16 + 2 * PAD_Y_COLS;
    c->pitch_c = c->mbw * 8 * CHROMA_STEP + 2 * PAD_C_COLS;  // interleaved CbCr rows: the same pitch as luma
    c->rgba_pitch = c->mbw * 16 * 4;
    c->y_slot = (size_t)c->pitch_y * (c->mbh * 16 + 2 * PAD_Y_ROWS);
    c->c_slot = (size_t)c->pitch_c * (c->mbh * 8 + 2 * PAD_C_ROWS);
    if (const char* k = getenv("H263CU_KERNEL")) c->force_kernel = !strcmp(k, "mb") ? 1 : (!strcmp(k, "tile") ? 2 : 0);
    c->rgba_slot = (size_t)c->rgba_pitch * c->mbh * 16;
    c->streams.resize(max_streams);
    auto fail = [&](int code) {
        *err = code;
        h263cu_destroy(c);
        return (h263cu_ctx*)nullptr;
    };
    const size_t pad = 256;  // aligned-word prediction loads may run a few bytes past a row
    // the tiled kernel addresses the pools through 32-bit offsets: 4-byte units for the planes,
    // 16-byte units for RGBA
    if (c->y_slot * 2 * max_streams + pad >= (16ull << 30) || c->rgba_slot * 2 * max_streams + pad >= (64ull << 30)) return fail(H263CU_ERR_CAPACITY);
    if (cudaMalloc((void**)&c->y_pool, c->y_slot * 2 * max_streams + pad) != cudaSuccess) return fail(H263CU_ERR_OUT_OF_MEMORY);
    if (cudaMalloc((void**)&c->c_pool, c->c_slot * 2 * max_streams + pad) != cudaSuccess) return fail(H263CU_ERR_OUT_OF_MEMORY);
    if (cudaMalloc((void**)&c->rgba_pool, c->rgba_slot * 2 * max_streams + pad) != cudaSuccess) return fail(H263CU_ERR_OUT_OF_MEMORY);
    {
        // TMA tensor map over the RGBA pool: the reconstruction kernel stores one 64-byte x 16-row box per macroblock
        // (cp.async.bulk.tensor.2d) from a shared-memory tile
        const int e = make_rgba_map(&c->rgba_map, c->rgba_pool, c->rgba_pitch, (uint64_t)2 * max_streams * c->mbh * 16);
        if (e) return fail(e);
    }
    if (cudaStreamCreateWithFlags(&c->s_main, cudaStreamNonBlocking) != cudaSuccess) return fail(H263CU_ERR_CUDA);
    if (cudaStreamCreateWithFlags(&c->s_h2d, cudaStreamNonBlocking) != cudaSuccess) return fail(H263CU_ERR_CUDA);
    if (cudaStreamCreateWithFlags(&c->s_d2h, cudaStreamNonBlocking) != cudaSuccess) return fail(H263CU_ERR_CUDA);
    if (cudaStreamCreateWithFlags(&c->s_pics, cudaStreamNonBlocking) != cudaSuccess) return fail(H263CU_ERR_CUDA);
    if (cudaStreamCreateWithFlags(&c->s_parse, cudaStreamNonBlocking) != cudaSuccess) return fail(H263CU_ERR_CUDA);
    if (cudaEventCreateWithFlags(&c->parse_done, cudaEventDisableTiming) != cudaSuccess) return fail(H263CU_ERR_CUDA);
    for (int i = 0; i < h263cu_ctx::PIC_RING; i++)
        if (cudaEventCreateWithFlags(&c->pics_done[i], cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&c->pics_up[i], cudaEventDisableTiming) != cudaSuccess)
            return fail(H263CU_ERR_CUDA);
    for (int i = 0; i < 2; i++) {
        if (cudaEventCreateWithFlags(&c->ring_h2d_done[i], cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&c->ring_run_done[i], cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&c->rgba_written[i], cudaEventDisableTiming) != cudaSuccess ||
            cudaEventCreateWithFlags(&c->rgba_read[i], cudaEventDisableTiming) != cudaSuccess)
            return fail(H263CU_ERR_CUDA);
    }
    if (cudaEventCreateWithFlags(&c->dev_ready, cudaEventDisableTiming) != cudaSuccess ||
        cudaEventCreateWithFlags(&c->dev_done, cudaEventDisableTiming) != cudaSuccess)
        return fail(H263CU_ERR_CUDA);
    if (cudaEventCreate(&c->t0) != cudaSuccess || cudaEventCreate(&c->t1) != cudaSuccess) return fail(H263CU_ERR_CUDA);
    // planes start out zeroed (DecodedPicture::new, picture.rs:39-58); every macroblock of a
    // picture is rewritten by the kernel, so this only matters for defensive reads
    cudaMemsetAsync(c->y_pool, 0, c->y_slot * 2 * max_streams + pad, c->s_main);
    cudaMemsetAsync(c->c_pool, 0, c->c_slot * 2 * max_streams + pad, c->s_main);
    if (cudaStreamSynchronize(c->s_main) != cudaSuccess) return fail(H263CU_ERR_CUDA);
    return c;
}

void h263cu_destroy(h263cu_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->s_main) cudaStreamSynchronize(c->s_main);
    if (c->s_h2d) cudaStreamSynchronize(c->s_h2d);
    if (c->s_d2h) cudaStreamSynchronize(c->s_d2h);
    if (c->s_pics) cudaStreamSynchronize(c->s_pics);
    if (c->s_parse) cudaStreamSynchronize(c->s_parse);
    for (int i = 0; i < 2; i++) free_step_buffers(&c->ring[i]);
    for (void* p : {(void*)c->h_pkts, (void*)c->h_pjobs, (void*)c->h_res, (void*)c->h_moves})
        if (p) cudaFreeHost(p);
    for (void* p : {(void*)c->d_tables, (void*)c->d_pkts, (void*)c->d_pjobs, (void*)c->d_res, (void*)c->d_moves, (void*)c->d_mbs_tmp})
        if (p) cudaFree(p);
    if (c->parse_done) cudaEventDestroy(c->parse_done);
    for (auto& st : c->staging) {
        if (st.pics) cudaFreeHost(st.pics);
        if (st.mbs) cudaFreeHost(st.mbs);
        if (st.events) cudaFreeHost(st.events);
    }
    for (int i = 0; i < h263cu_ctx::PIC_RING; i++) {
        if (c->h_pics[i]) cudaFreeHost(c->h_pics[i]);
        if (c->d_pics[i]) cudaFree(c->d_pics[i]);
        if (c->h_geo[i]) cudaFreeHost(c->h_geo[i]);
        if (c->d_geo[i]) cudaFree(c->d_geo[i]);
        if (c->pics_done[i]) cudaEventDestroy(c->pics_done[i]);
        if (c->pics_up[i]) cudaEventDestroy(c->pics_up[i]);
    }
    for (int i = 0; i < 2; i++) {
        if (c->ring_h2d_done[i]) cudaEventDestroy(c->ring_h2d_done[i]);
        if (c->ring_run_done[i]) cudaEventDestroy(c->ring_run_done[i]);
        if (c->rgba_written[i]) cudaEventDestroy(c->rgba_written[i]);
        if (c->rgba_read[i]) cudaEventDestroy(c->rgba_read[i]);
    }
    if (c->t0) cudaEventDestroy(c->t0);
    if (c->t1) cudaEventDestroy(c->t1);
    if (c->dev_ready) cudaEventDestroy(c->dev_ready);
    if (c->dev_done) cudaEventDestroy(c->dev_done);
    if (c->tensor_scratch) cudaFree(c->tensor_scratch);
    for (auto& sp : c->prof_spans) {
        cudaEventDestroy(sp.a);
        cudaEventDestroy(sp.b);
    }
    for (auto e : c->prof_free) cudaEventDestroy(e);
    if (c->d_jobs) cudaFree(c->d_jobs);
    if (c->d_sums) cudaFree(c->d_sums);
    if (c->y_pool) cudaFree(c->y_pool);
    if (c->c_pool) cudaFree(c->c_pool);
    if (c->rgba_pool) cudaFree(c->rgba_pool);
    if (c->s_main) cudaStreamDestroy(c->s_main);
    if (c->s_h2d) cudaStreamDestroy(c->s_h2d);
    if (c->s_d2h) cudaStreamDestroy(c->s_d2h);
    if (c->s_pics) cudaStreamDestroy(c->s_pics);
    if (c->s_parse) cudaStreamDestroy(c->s_parse);
    delete c;
}

int h263cu_device_of(h263cu_ctx* c) { return c ? c->device : -1; }

void* h263cu_alloc_pinned(size_t bytes) {
    void* p = nullptr;
    if (cudaHostAlloc(&p, bytes ? bytes : 1, cudaHostAllocDefault) != cudaSuccess) {
        cudaGetLastError();
        return nullptr;
    }
    return p;
}
void h263cu_free_pinned(void* p) {
    if (p) cudaFreeHost(p);
}

h263cu_step* h263cu_step_upload(h263cu_ctx* c, const h263cu_pic* pics, uint32_t n_pics, const h263cu_mb* mbs,
                                uint32_t n_mbs, const h263cu_event* events, uint32_t n_units, int* err) {
    int dummy;
    if (!err) err = &dummy;
    *err = 0;
    if (!c || !pics || (!mbs && n_mbs) || (!events && n_units)) {
        *err = H263CU_ERR_BAD_ARGUMENT;
        return nullptr;
    }
    cudaSetDevice(c->device);
    h263cu_step* s = new (std::nothrow) h263cu_step();
    if (!s) {
        *err = H263CU_ERR_OUT_OF_MEMORY;
        return nullptr;
    }
    int e = upload_into(c, s, pics, n_pics, mbs, n_mbs, events, n_units, c->s_main, false);
    if (e) {
        free_step_buffers(s);
        delete s;
        *err = e;
        return nullptr;
    }
    return s;
}

void h263cu_step_free(h263cu_ctx* c, h263cu_step* s) {
    if (!s) return;
    if (c) {
        cudaSetDevice(c->device);
        cudaStreamSynchronize(c->s_main);
    }
    free_step_buffers(s);
    delete s;
}

int h263cu_step_run(h263cu_ctx* c, h263cu_step* s, uint32_t out_flags) {
    if (!c || !s) return H263CU_ERR_BAD_ARGUMENT;
    cudaSetDevice(c->device);
    return run_step(c, s, out_flags);
}

// `resident`: the side info is already in the ring slot, written by the device parse (device_parse); mbs / events are
// not read, and the kernels wait for parse_done instead of an upload.
static int submit_common(h263cu_ctx* c, const h263cu_pic* pics, uint32_t n_pics, const h263cu_mb* mbs, uint32_t n_mbs,
                         const h263cu_event* events, uint32_t n_units, uint32_t out_flags, bool trusted = false, bool lean = false,
                         const DeviceTarget* dev = nullptr, bool resident = false) {
    if (!c || !pics || (!resident && ((!mbs && n_mbs) || (!events && n_units)))) return H263CU_ERR_BAD_ARGUMENT;
    cudaSetDevice(c->device);
    const int slot = c->ring_pos;
    h263cu_step* s = &c->ring[slot];
    if (n_mbs > s->mb_cap || (size_t)n_units + 8 > s->ev_cap) CU_TRY(cudaEventSynchronize(c->ring_run_done[slot]));
    int e;
    if (resident) {
        try {
            s->pics.assign(pics, pics + n_pics);
        } catch (const std::bad_alloc&) {
            return H263CU_ERR_OUT_OF_MEMORY;
        }
        s->n_mbs = n_mbs, s->n_units = n_units;
        CU_TRY(cudaStreamWaitEvent(c->s_main, c->parse_done, 0));
    } else if (lean) {
        // in-order on s_main: the kernels that read this ring slot two submits ago precede these copies on the stream
        if ((e = upload_into(c, s, pics, n_pics, mbs, n_mbs, events, n_units, c->s_main, trusted))) return e;
        CU_TRY(cudaEventRecord(c->ring_h2d_done[slot], c->s_main));
    } else {
        // the copy engine may not overwrite side info that a kernel is still reading
        CU_TRY(cudaStreamWaitEvent(c->s_h2d, c->ring_run_done[slot], 0));
        if ((e = upload_into(c, s, pics, n_pics, mbs, n_mbs, events, n_units, c->s_h2d, trusted))) return e;
        CU_TRY(cudaEventRecord(c->ring_h2d_done[slot], c->s_h2d));
        CU_TRY(cudaStreamWaitEvent(c->s_main, c->ring_h2d_done[slot], 0));
    }
    e = run_step(c, s, out_flags, lean, dev);
    if (e) return e;
    c->ring_pos ^= 1;  // the ring slot is taken only by a step that runs
    CU_TRY(cudaEventRecord(c->ring_run_done[slot], c->s_main));
    return 0;
}

int h263cu_submit_step(h263cu_ctx* c, const h263cu_pic* pics, uint32_t n_pics, const h263cu_mb* mbs, uint32_t n_mbs,
                       const h263cu_event* events, uint32_t n_units, uint32_t out_flags) {
    return submit_common(c, pics, n_pics, mbs, n_mbs, events, n_units, out_flags);
}

static int submit_readback(h263cu_ctx* c, const h263cu_pic* pics, uint32_t n_pics, const h263cu_mb* mbs, uint32_t n_mbs,
                           const h263cu_event* events, uint32_t n_units, uint32_t out_flags, uint8_t* host_rgba,
                           const uint64_t* rgba_offsets, bool trusted, bool lean = false, bool resident = false) {
    if (!host_rgba) return H263CU_ERR_BAD_ARGUMENT;
    out_flags |= H263CU_OUT_RGBA;
    int e = submit_common(c, pics, n_pics, mbs, n_mbs, events, n_units, out_flags, trusted, lean, nullptr, resident);
    if (e) return e;
    const int ring = (int)((c->rgba_parity - 1) & 1u);  // the slot run_step just wrote
    const cudaStream_t s_d2h = lean ? c->s_main : c->s_d2h;
    if (!lean) CU_TRY(cudaStreamWaitEvent(c->s_d2h, c->rgba_written[ring], 0));
    uint64_t off = 0;
    uint32_t i = 0;
    while (i < n_pics) {
        const h263cu_pic& p = pics[i];
        const uint64_t dst = rgba_offsets ? rgba_offsets[i] : off;
        const size_t tight = (size_t)p.width * 4;
        const bool dense = tight == c->rgba_pitch && (size_t)p.height * c->rgba_pitch == c->rgba_slot;
        if (dense) {
            // coalesce runs of consecutive streams with contiguous destinations into one copy
            uint32_t j = i + 1;
            while (j < n_pics && pics[j].stream == pics[j - 1].stream + 1 && pics[j].width == p.width &&
                   pics[j].height == p.height &&
                   (!rgba_offsets || rgba_offsets[j] == rgba_offsets[j - 1] + c->rgba_slot))
                j++;
            CU_TRY(cudaMemcpyAsync(host_rgba + dst, c->rgba(p.stream, ring), (size_t)(j - i) * c->rgba_slot,
                                   cudaMemcpyDeviceToHost, s_d2h));
            off = dst + (uint64_t)(j - i) * c->rgba_slot;
            i = j;
        } else {
            CU_TRY(cudaMemcpy2DAsync(host_rgba + dst, tight, c->rgba(p.stream, ring), c->rgba_pitch, tight, p.height,
                                     cudaMemcpyDeviceToHost, s_d2h));
            off = dst + (uint64_t)tight * p.height;
            i++;
        }
    }
    CU_TRY(cudaEventRecord(c->rgba_read[ring], s_d2h));
    return 0;
}

int h263cu_submit_step_readback(h263cu_ctx* c, const h263cu_pic* pics, uint32_t n_pics, const h263cu_mb* mbs,
                                uint32_t n_mbs, const h263cu_event* events, uint32_t n_units, uint32_t out_flags,
                                uint8_t* host_rgba, const uint64_t* rgba_offsets) {
    return submit_readback(c, pics, n_pics, mbs, n_mbs, events, n_units, out_flags, host_rgba, rgba_offsets, false);
}

// The parse of a step with H263CU_PARSE_ON_DEVICE, into ring slot `slot`: the host parses the picture headers
// (h263fe::device_parse_prepare), the packets of the pictures that pass go up in one copy, parse_mb_kernel parses their
// macroblock layer on s_parse into the slot's records and events -- after the kernels that read the slot last -- and
// the host waits for the per-picture results alone (never for s_main or the caller's stream) and finishes the pictures
// (h263fe::device_parse_finish).  Output as h263fe::parse_step_deferred's: the decoded pictures packed in input order
// into pics (first_mb dense; first_event is the picture's event region, so *n_units is the regions' total), per_pic_err
// and pic_of_input per input, the parsers' pending states.  When a picture failed after its records were written and
// `compact`, the survivors' records are moved to their packed positions on s_parse.  parse_done marks the side info
// complete.  On an error return the caller drops the pending states (parse_step_finish(.., false)).
static int device_parse(h263cu_ctx* c, int slot, h263cu_parser* const* parsers, const uint8_t* const* packets, const size_t* lens,
                        const uint32_t* stream_ids, uint32_t n, int threads, uint32_t max_w, uint32_t max_h, const uint32_t* min_size,
                        h263cu_pic* pics, uint32_t* n_pics_out, uint32_t* n_mbs_out, uint32_t* n_units_out, int* per_pic_err,
                        int32_t* pic_of_input, bool compact) {
    if (!parsers || !packets || !lens) return H263CU_ERR_BAD_ARGUMENT;
    int e;
    try {
        c->dp_pkt_off.resize((size_t)n + 1);
        c->dp_pics.resize(n);
        c->dp_errs.resize(n);
        c->dp_job.resize(n);
        c->dp_moves.clear();
        c->dp_moves.reserve(n);
    } catch (const std::bad_alloc&) {
        return H263CU_ERR_OUT_OF_MEMORY;
    }
    // every packet 4-byte aligned and followed by >= 12 zero bytes (parse_mb.cu's reader); bit positions are 32-bit
    uint64_t off = 0;
    for (uint32_t i = 0; i < n; i++) {
        if (lens[i] >= (1u << 28)) return H263CU_ERR_CAPACITY;
        c->dp_pkt_off[i] = off;
        off += round_up(lens[i] + 12, 16);
    }
    c->dp_pkt_off[n] = off;
    if (off / 4 > 0xFFFFFFFFull) return H263CU_ERR_CAPACITY;
    if (!c->d_tables) {
        std::vector<uint32_t> t(PT_WORDS);
        if ((e = h263fe::device_parse_tables(t.data()))) return e;
        CU_TRY(cudaMalloc((void**)&c->d_tables, PT_WORDS * sizeof(uint32_t)));
        CU_TRY(cudaMemcpy(c->d_tables, t.data(), PT_WORDS * sizeof(uint32_t), cudaMemcpyHostToDevice));
    }
    // the pinned sets were last read by copies that precede the previous call's result read-back, which it waited for
    if ((e = grow_pinned(&c->h_pkts, &c->pkts_cap, off)) || (e = grow_pinned(&c->h_pjobs, &c->pjobs_cap, n)) ||
        (e = grow_pinned(&c->h_res, &c->res_cap, n)))
        return e;
    uint32_t nj = 0, mb_total = 0, ev_total = 0;
    e = h263fe::device_parse_prepare(parsers, packets, lens, stream_ids, n, threads, max_w, max_h, min_size, c->dp_pkt_off.data(),
                                     c->h_pkts, c->dp_pics.data(), c->dp_errs.data(), c->h_pjobs, c->dp_job.data(), &nj, &mb_total,
                                     &ev_total);
    if (e) return e;
    h263cu_step* s = &c->ring[slot];
    if (nj) {
        if (mb_total > s->mb_cap || (size_t)ev_total + 8 > s->ev_cap) {
            CU_TRY(cudaEventSynchronize(c->ring_run_done[slot]));
            if ((e = step_reserve(s, mb_total, ev_total))) return e;
        }
        CU_TRY(cudaStreamSynchronize(c->s_parse));  // a compaction of the previous call may still read d_moves
        if ((e = grow_device(&c->d_pkts, &c->d_pkts_cap, off)) || (e = grow_device(&c->d_pjobs, &c->d_pjobs_cap, nj)) ||
            (e = grow_device(&c->d_res, &c->d_res_cap, nj)))
            return e;
        // the records and events may be overwritten once the kernels that read this ring slot last have finished
        CU_TRY(cudaStreamWaitEvent(c->s_parse, c->ring_run_done[slot], 0));
        CU_TRY(cudaMemcpyAsync(c->d_pkts, c->h_pkts, off, cudaMemcpyHostToDevice, c->s_parse));
        CU_TRY(cudaMemcpyAsync(c->d_pjobs, c->h_pjobs, nj * sizeof(ParseJob), cudaMemcpyHostToDevice, c->s_parse));
        CU_TRY(launch_parse_mb(c->d_pjobs, nj, c->d_tables, reinterpret_cast<const uint32_t*>(c->d_pkts), s->d_mbs, s->d_events, c->d_res,
                               c->s_parse));
        CU_TRY(cudaMemcpyAsync(c->h_res, c->d_res, nj * sizeof(ParseResult), cudaMemcpyDeviceToHost, c->s_parse));
        CU_TRY(cudaEventRecord(c->parse_done, c->s_parse));
        CU_TRY(cudaEventSynchronize(c->parse_done));
        h263fe::device_parse_finish(parsers, n, c->dp_job.data(), c->h_res, c->dp_pics.data(), c->dp_errs.data());
    }
    c->dp_mb_total = mb_total, c->dp_ev_total = ev_total;
    uint32_t np = 0, nm = 0;
    for (uint32_t i = 0; i < n; i++) {
        if (per_pic_err) per_pic_err[i] = c->dp_errs[i];
        pic_of_input[i] = -1;
        if (c->dp_errs[i]) continue;
        const ParseJob& J = c->h_pjobs[c->dp_job[i]];
        h263cu_pic pc = c->dp_pics[i];
        pc.first_mb = nm;
        pc.first_event = J.first_event;
        c->dp_moves.push_back(PackMove{J.first_mb, nm, pc.n_mbs, np});
        pics[np] = pc;
        pic_of_input[i] = (int32_t)np++;
        nm += pc.n_mbs;
    }
    if (compact && np && np < nj) {
        // a picture failed after the kernel wrote its records: move the survivors' records to their packed positions
        // and indices (the events stay where they are: each record points into its picture's region)
        if ((e = grow_device(&c->d_mbs_tmp, &c->mbs_tmp_cap, mb_total)) || (e = grow_pinned(&c->h_moves, &c->moves_cap, np)) ||
            (e = grow_device(&c->d_moves, &c->d_moves_cap, np)))
            return e;
        std::memcpy(c->h_moves, c->dp_moves.data(), np * sizeof(PackMove));
        CU_TRY(cudaMemcpyAsync(c->d_mbs_tmp, s->d_mbs, (size_t)mb_total * sizeof(h263cu_mb), cudaMemcpyDeviceToDevice, c->s_parse));
        CU_TRY(cudaMemcpyAsync(c->d_moves, c->h_moves, np * sizeof(PackMove), cudaMemcpyHostToDevice, c->s_parse));
        launch_pack_mbs(c->d_mbs_tmp, s->d_mbs, c->d_moves, np, c->s_parse);
        CU_TRY(cudaGetLastError());
        CU_TRY(cudaEventRecord(c->parse_done, c->s_parse));
    }
    *n_pics_out = np;
    *n_mbs_out = nm;
    *n_units_out = ev_total;
    return 0;
}

// The body of h263cu_decode_step, h263cu_decode_step_device, h263cu_decode_step_device_yuv and
// h263cu_decode_step_device_tensor; `positions` (may be NULL: input i sits at position i) says where input i's output
// goes: in host_rgba, in units of rgba_stride (the group form scatters the pictures of one device over a buffer shared
// by all), or the slot in the caller's device buffer `dev_out` (not NULL: device RGBA), device planes `yuv_out` (not
// NULL: device planes, no RGBA) or device tensor `tensor_out` (not NULL: resampled RGB, no RGBA), the latter placed by
// `fit` when not NULL (h263cu_decode_step_device_tensor_fit; fit->crops indexed like the inputs here) and resized
// with `filter` (H263CU_FILTER_*, h263cu_decode_step_device_tensor_filter; checked by the caller).
static int decode_step_scattered(h263cu_ctx* c, h263cu_parser* const* parsers, const uint8_t* const* packets, const size_t* lens,
                                 const uint32_t* stream_ids, uint32_t n, int threads, uint32_t out_flags, uint8_t* host_rgba,
                                 uint64_t rgba_stride, const uint32_t* positions, const h263cu_device_rgba* dev_out,
                                 const h263cu_device_yuv* yuv_out, const h263cu_device_tensor* tensor_out,
                                 const h263cu_tensor_fit* fit, int* per_pic_err, uint32_t* n_decoded,
                                 uint32_t filter = H263CU_FILTER_BILINEAR) {
    if (!c || !parsers || !packets || !lens) return H263CU_ERR_BAD_ARGUMENT;
    if (n_decoded) *n_decoded = 0;
    const auto t_enter = std::chrono::steady_clock::now();
    cudaSetDevice(c->device);
    int e;
    if (dev_out && (e = check_device_rgba(c, dev_out))) return e;
    if (yuv_out && (e = check_device_yuv(c, yuv_out))) return e;
    if (tensor_out && (e = check_device_tensor(c, tensor_out))) return e;
    if (fit && (e = check_tensor_fit(fit, n))) return e;
    if (n == 0) return 0;
    // capacities: a picture holds at most mbw * mbh macroblocks of this context; every event costs at least
    // 3 bits of bitstream and takes at most 2 units
    size_t bytes = 0;
    for (uint32_t i = 0; i < n; i++) bytes += lens[i];
    const size_t mb_need = (size_t)n * c->mbw * c->mbh, ev_need = bytes * 16 / 3 + 16 * (size_t)n;
    if (mb_need > 0xFFFFFFFFull || ev_need > 0xFFFFFFFFull) return H263CU_ERR_CAPACITY;
    // Stream ids are checked before anything is parsed; a picture larger than the context fails as that picture's
    // error inside the parse.  The parsers advance only when the device stage has accepted the step, so a failing
    // call leaves every stream as it was (decode_next_picture is a transaction, state.rs:120-137).
    c->decode_epoch++;
    for (uint32_t i = 0; i < n; i++) {
        const uint32_t sid = stream_ids ? stream_ids[i] : i;
        if (sid >= c->max_streams) return H263CU_ERR_CAPACITY;
        if (c->streams[sid].seen == c->decode_epoch) return H263CU_ERR_BAD_ARGUMENT;
        c->streams[sid].seen = c->decode_epoch;
    }
    const int slot = c->ring_pos;  // the ring slot submit_common is about to use
    h263cu_ctx::Staging& st = c->staging[slot];
    // the copy engine has finished with this staging set (it was read two submits ago)
    CU_TRY(cudaEventSynchronize(c->ring_h2d_done[slot]));
    // with the parse on the device the records and events never pass through the host
    const bool on_device = (out_flags & H263CU_PARSE_ON_DEVICE) != 0;
    if ((e = grow_pinned(&st.pics, &st.pic_cap, n)) || (!on_device && (e = grow_pinned(&st.mbs, &st.mb_cap, mb_need))) ||
        (!on_device && (e = grow_pinned(&st.events, &st.ev_cap, ev_need))))
        return e;
    const uint32_t* min_size = nullptr;  // a crop box must lie inside its picture: a per-picture error of the parse
    try {
        c->pic_of_input.resize(n);
        if (fit && fit->crops) {
            c->fit_min.resize(2 * (size_t)n);
            for (uint32_t i = 0; i < n; i++)
                c->fit_min[2 * i] = fit->crops[i].x + fit->crops[i].width, c->fit_min[2 * i + 1] = fit->crops[i].y + fit->crops[i].height;
            min_size = c->fit_min.data();
        }
    } catch (const std::bad_alloc&) {
        return H263CU_ERR_OUT_OF_MEMORY;
    }
    uint32_t np = 0, nm = 0, nu = 0;
    const auto t_parse0 = std::chrono::steady_clock::now();
    // device output: a picture larger than the caller's slot fails like one larger than the context (a tensor has no
    // slot size: every picture is resized to it)
    const uint32_t max_w = dev_out ? std::min(c->max_w, dev_out->width) : yuv_out ? std::min(c->max_w, yuv_out->width) : c->max_w;
    const uint32_t max_h = dev_out ? std::min(c->max_h, dev_out->height) : yuv_out ? std::min(c->max_h, yuv_out->height) : c->max_h;
    if (on_device)
        e = device_parse(c, slot, parsers, packets, lens, stream_ids, n, threads, max_w, max_h, min_size, st.pics, &np, &nm, &nu, per_pic_err,
                         c->pic_of_input.data(), true);
    else
        e = h263fe::parse_step_deferred(parsers, packets, lens, stream_ids, n, threads, st.pics, st.mbs, (uint32_t)st.mb_cap, st.events,
                                        (uint32_t)st.ev_cap, &np, &nm, &nu, per_pic_err, c->pic_of_input.data(), max_w, max_h, min_size);
    const auto t_parse1 = std::chrono::steady_clock::now();
    c->host_parse_s += std::chrono::duration<double>(t_parse1 - t_parse0).count();
    c->host_other_s += std::chrono::duration<double>(t_parse0 - t_enter).count();
    c->host_calls++;
    struct Tail {  // whatever follows the parse on any return path counts as "other"
        h263cu_ctx* c;
        std::chrono::steady_clock::time_point t;
        ~Tail() { c->host_other_s += std::chrono::duration<double>(std::chrono::steady_clock::now() - t).count(); }
    } tail{c, t_parse1};
    if (e) {
        if (on_device) cudaStreamSynchronize(c->s_parse);  // see below: nothing of a refused step stays queued
        h263fe::parse_step_finish(parsers, n, false);
        return e;
    }
    if (n_decoded) *n_decoded = np;
    if (np == 0) return 0;
    // one picture of at most a 4CIF's macroblocks: the single-stream case (H263State), latency bound on driver calls
    const bool lean = np == 1 && nm <= 1584;
    if (dev_out || yuv_out || tensor_out) {
        DeviceTarget dt;
        std::memset(&dt, 0, sizeof(dt));
        dt.out = dev_out ? OUT_DEV_RGBA : yuv_out ? OUT_YUV : OUT_TENSOR;
        if (dev_out) {
            dt.base = dev_out->base, dt.row_pitch = dev_out->row_pitch, dt.pic_stride = dev_out->pic_stride;
            dt.stream = (cudaStream_t)dev_out->stream;
        } else if (tensor_out) {
            dt.tensor.base = tensor_out->base;
            for (int k = 0; k < 4; k++) dt.tensor.stride[k] = tensor_out->stride[k];
            dt.tensor.width = tensor_out->width, dt.tensor.height = tensor_out->height;
            for (int k = 0; k < 3; k++) dt.tensor.mul[k] = tensor_out->mul[k], dt.tensor.add[k] = tensor_out->add[k];
            dt.dtype = tensor_out->dtype;
            dt.stream = (cudaStream_t)tensor_out->stream;
        } else {
            for (int k = 0; k < 3; k++) {
                dt.yuv.base[k] = yuv_out->plane[k].base;
                dt.yuv.stride[k] = yuv_out->plane[k].pic_stride;
                dt.yuv.pitch[k] = (uint32_t)yuv_out->plane[k].row_pitch;
            }
            dt.yuv.nv12 = yuv_out->format == H263CU_YUV_NV12;
            dt.stream = (cudaStream_t)yuv_out->stream;
        }
        uint32_t n_slots = 0;
        try {
            c->dev_slots.resize(np);
            if (fit) c->fit_geo.resize(np);
        } catch (const std::bad_alloc&) {
            if (on_device) cudaStreamSynchronize(c->s_parse);  // see below: nothing of a refused step stays queued
            h263fe::parse_step_finish(parsers, n, false);
            return H263CU_ERR_OUT_OF_MEMORY;
        }
        if (fit) {  // the geometry of every decoded picture, from its size now that the parse knows it
            for (uint32_t i = 0; i < n; i++) {
                const int32_t k = c->pic_of_input[i];
                if (k < 0) continue;
                const h263cu_pic& p = st.pics[k];
                const h263cu_tensor_crop b = fit->crops ? fit->crops[i] : h263cu_tensor_crop{0, 0, p.width, p.height};
                FitGeom& g = c->fit_geo[(size_t)k];
                g.cx = (int32_t)b.x, g.cy = (int32_t)b.y, g.cw = (int32_t)b.width, g.ch = (int32_t)b.height;
                int32_t r[4];
                fit_geometry(fit->mode, fit->short_side, b.width, b.height, tensor_out->width, tensor_out->height, r);
                g.rw = r[0], g.rh = r[1], g.px = r[2], g.py = r[3];
            }
            dt.geo = c->fit_geo.data();
            for (int k = 0; k < 3; k++) dt.fill[k] = fit->fill[k];
            dt.filter = filter;
        }
        for (uint32_t i = 0; i < n; i++)
            if (c->pic_of_input[i] >= 0) {
                const uint32_t k = positions ? positions[i] : i;
                c->dev_slots[(size_t)c->pic_of_input[i]] = k;
                n_slots = std::max(n_slots, k + 1);
            }
        dt.slots = c->dev_slots.data();
        if (dev_out) {
            const cuuint64_t dims[3] = {4ull * dev_out->width, dev_out->height, n_slots}, strides[2] = {dev_out->row_pitch, dev_out->pic_stride};
            e = encode_rgba_map(&dt.map, dev_out->base, 3, dims, strides);
        }
        if (!e) e = submit_common(c, st.pics, np, st.mbs, nm, st.events, nu, out_flags | H263CU_OUT_RGBA, true, lean, &dt, on_device);
    } else if (!host_rgba) {
        e = submit_common(c, st.pics, np, st.mbs, nm, st.events, nu, out_flags, true, lean, nullptr, on_device);
    } else {
        try {
            c->rgba_offsets.resize(np);
        } catch (const std::bad_alloc&) {
            if (on_device) cudaStreamSynchronize(c->s_parse);  // see below: nothing of a refused step stays queued
            h263fe::parse_step_finish(parsers, n, false);
            return H263CU_ERR_OUT_OF_MEMORY;
        }
        for (uint32_t i = 0; i < n; i++)
            if (c->pic_of_input[i] >= 0) c->rgba_offsets[(size_t)c->pic_of_input[i]] = (uint64_t)(positions ? positions[i] : i) * rgba_stride;
        e = submit_readback(c, st.pics, np, st.mbs, nm, st.events, nu, out_flags, host_rgba, c->rgba_offsets.data(), true, lean, on_device);
    }
    // a refused step leaves no device-parse work behind that a later upload into this ring slot could overtake (the
    // slot's ring_run_done is recorded only by a step that runs)
    if (e && on_device) cudaStreamSynchronize(c->s_parse);
    // the device stage has the step (or refused it): only now do the parsers move on
    h263fe::parse_step_finish(parsers, n, e == 0);
    return e;
}

int h263cu_decode_step(h263cu_ctx* c, h263cu_parser* const* parsers, const uint8_t* const* packets, const size_t* lens,
                       const uint32_t* stream_ids, uint32_t n, int threads, uint32_t out_flags, uint8_t* host_rgba,
                       uint64_t rgba_stride, int* per_pic_err, uint32_t* n_decoded) {
    return decode_step_scattered(c, parsers, packets, lens, stream_ids, n, threads, out_flags, host_rgba, rgba_stride, nullptr, nullptr,
                                 nullptr, nullptr, nullptr, per_pic_err, n_decoded);
}

int h263cu_decode_step_device(h263cu_ctx* c, h263cu_parser* const* parsers, const uint8_t* const* packets, const size_t* lens,
                              const uint32_t* stream_ids, uint32_t n, int threads, uint32_t out_flags, const h263cu_device_rgba* out,
                              int* per_pic_err, uint32_t* n_decoded) {
    if (!out) return H263CU_ERR_BAD_ARGUMENT;
    return decode_step_scattered(c, parsers, packets, lens, stream_ids, n, threads, out_flags, nullptr, 0, nullptr, out, nullptr,
                                 nullptr, nullptr, per_pic_err, n_decoded);
}

int h263cu_decode_step_device_yuv(h263cu_ctx* c, h263cu_parser* const* parsers, const uint8_t* const* packets, const size_t* lens,
                                  const uint32_t* stream_ids, uint32_t n, int threads, uint32_t out_flags, const h263cu_device_yuv* out,
                                  int* per_pic_err, uint32_t* n_decoded) {
    if (!out) return H263CU_ERR_BAD_ARGUMENT;
    return decode_step_scattered(c, parsers, packets, lens, stream_ids, n, threads, out_flags, nullptr, 0, nullptr, nullptr, out,
                                 nullptr, nullptr, per_pic_err, n_decoded);
}

int h263cu_decode_step_device_tensor(h263cu_ctx* c, h263cu_parser* const* parsers, const uint8_t* const* packets, const size_t* lens,
                                     const uint32_t* stream_ids, uint32_t n, int threads, uint32_t out_flags,
                                     const h263cu_device_tensor* out, int* per_pic_err, uint32_t* n_decoded) {
    if (!out) return H263CU_ERR_BAD_ARGUMENT;
    return decode_step_scattered(c, parsers, packets, lens, stream_ids, n, threads, out_flags, nullptr, 0, nullptr, nullptr, nullptr,
                                 out, nullptr, per_pic_err, n_decoded);
}

int h263cu_decode_step_device_tensor_fit(h263cu_ctx* c, h263cu_parser* const* parsers, const uint8_t* const* packets,
                                         const size_t* lens, const uint32_t* stream_ids, uint32_t n, int threads, uint32_t out_flags,
                                         const h263cu_device_tensor* out, const h263cu_tensor_fit* fit, int* per_pic_err,
                                         uint32_t* n_decoded) {
    if (!out || !fit) return H263CU_ERR_BAD_ARGUMENT;
    return decode_step_scattered(c, parsers, packets, lens, stream_ids, n, threads, out_flags, nullptr, 0, nullptr, nullptr, nullptr,
                                 out, fit, per_pic_err, n_decoded);
}

int h263cu_decode_step_device_tensor_filter(h263cu_ctx* c, h263cu_parser* const* parsers, const uint8_t* const* packets,
                                            const size_t* lens, const uint32_t* stream_ids, uint32_t n, int threads, uint32_t out_flags,
                                            const h263cu_device_tensor* out, const h263cu_tensor_fit* fit, uint32_t filter,
                                            int* per_pic_err, uint32_t* n_decoded) {
    if (!out || !fit || filter > H263CU_FILTER_BICUBIC_AA) return H263CU_ERR_BAD_ARGUMENT;
    return decode_step_scattered(c, parsers, packets, lens, stream_ids, n, threads, out_flags, nullptr, 0, nullptr, nullptr, nullptr,
                                 out, fit, per_pic_err, n_decoded, filter);
}

int h263cu_test_fit_geometry(uint32_t mode, uint32_t short_side, uint32_t cw, uint32_t ch, uint32_t width, uint32_t height,
                             int32_t* out4) {
    const h263cu_tensor_fit f{mode, short_side, {0.0f, 0.0f, 0.0f}, 0, nullptr};
    if (!out4 || check_tensor_fit(&f, 0) || cw == 0 || ch == 0 || cw > 65535 || ch > 65535 || width == 0 || height == 0 ||
        width > 16384 || height > 16384)
        return H263CU_ERR_BAD_ARGUMENT;
    fit_geometry(mode, short_side, cw, ch, width, height, out4);
    return 0;
}

int h263cu_test_device_parse_step(h263cu_ctx* c, h263cu_parser* const* parsers, const uint8_t* const* packets, const size_t* lens,
                                  const uint32_t* stream_ids, uint32_t n, int threads, h263cu_pic* pics, h263cu_mb* mbs, uint32_t mb_cap,
                                  h263cu_event* events, uint32_t ev_cap, uint32_t* n_pics_out, uint32_t* n_mbs_out, uint32_t* n_units_out,
                                  int* per_pic_err, int32_t* pic_of_input) {
    if (!c || !parsers || !packets || !lens || !pics || !mbs || !n_pics_out || !n_mbs_out || !n_units_out) return H263CU_ERR_BAD_ARGUMENT;
    cudaSetDevice(c->device);
    std::vector<h263cu_pic> dpics;
    std::vector<int> errs;
    std::vector<int32_t> packed;
    std::vector<h263cu_mb> raw_mbs;
    std::vector<h263cu_event> raw_events;
    uint32_t np = 0, nm = 0, nu = 0;
    int e = 0;
    try {
        dpics.resize(n), errs.resize(n), packed.resize(n);
        e = device_parse(c, c->ring_pos, parsers, packets, lens, stream_ids, n, threads, 0, 0, nullptr, dpics.data(), &np, &nm, &nu,
                         errs.data(), packed.data(), false);
        if (!e && np) {
            // what the kernel wrote, as it lies in the ring slot
            const h263cu_step& s = c->ring[c->ring_pos];
            raw_mbs.resize(c->dp_mb_total), raw_events.resize(c->dp_ev_total);
            cudaError_t ce = cudaMemcpyAsync(raw_mbs.data(), s.d_mbs, raw_mbs.size() * sizeof(h263cu_mb), cudaMemcpyDeviceToHost, c->s_parse);
            if (ce == cudaSuccess && nu)
                ce = cudaMemcpyAsync(raw_events.data(), s.d_events, raw_events.size() * sizeof(h263cu_event), cudaMemcpyDeviceToHost, c->s_parse);
            if (ce == cudaSuccess) ce = cudaStreamSynchronize(c->s_parse);
            if (ce != cudaSuccess) e = map_cuda_error(ce);
        }
    } catch (const std::bad_alloc&) {
        e = H263CU_ERR_OUT_OF_MEMORY;
    }
    h263fe::parse_step_finish(parsers, n, false);  // the parsers stay where they were
    if (e) return e;
    // packed as h263cu_parse_step packs: records and events dense, in input order
    uint32_t pm = 0, pu = 0;
    for (uint32_t i = 0; i < n; i++) {
        if (per_pic_err) per_pic_err[i] = errs[i];
        if (packed[i] < 0) continue;
        const uint32_t k = (uint32_t)packed[i];
        h263cu_pic pc = dpics[k];
        if ((uint64_t)pm + pc.n_mbs > mb_cap || (uint64_t)pu + pc.n_event_units > ev_cap) return H263CU_ERR_CAPACITY;
        const PackMove& mv = c->dp_moves[k];
        for (uint32_t j = 0; j < pc.n_mbs; j++) {
            mbs[pm + j] = raw_mbs[mv.src_first + j];
            mbs[pm + j].pic = (uint16_t)k;
        }
        if (pc.n_event_units) std::memcpy(events + pu, raw_events.data() + pc.first_event, pc.n_event_units * sizeof(h263cu_event));
        pc.first_mb = pm, pc.first_event = pu;
        pics[k] = pc;
        pm += pc.n_mbs, pu += pc.n_event_units;
    }
    if (pic_of_input) std::memcpy(pic_of_input, packed.data(), n * sizeof(int32_t));
    *n_pics_out = np;
    *n_mbs_out = pm;
    *n_units_out = pu;
    return 0;
}

int h263cu_sync(h263cu_ctx* c) {
    if (!c) return H263CU_ERR_BAD_ARGUMENT;
    cudaSetDevice(c->device);
    CU_TRY(cudaStreamSynchronize(c->s_h2d));
    CU_TRY(cudaStreamSynchronize(c->s_main));
    CU_TRY(cudaStreamSynchronize(c->s_d2h));
    return 0;
}

int h263cu_stream_info(h263cu_ctx* c, uint32_t stream, uint32_t* width, uint32_t* height, uint32_t* pic_type,
                       uint32_t* pquant, uint32_t* temporal_reference) {
    if (!c || stream >= c->max_streams) return H263CU_ERR_BAD_ARGUMENT;
    const StreamState& st = c->streams[stream];
    if (!st.has_pic) return H263CU_ERR_NO_PICTURE;
    if (width) *width = st.w;
    if (height) *height = st.h;
    if (pic_type) *pic_type = st.pic_type;
    if (pquant) *pquant = st.pquant;
    if (temporal_reference) *temporal_reference = st.tr;
    return 0;
}

uint32_t h263cu_stream_dims(h263cu_ctx* c, uint32_t stream) {
    if (!c || stream >= c->max_streams || !c->streams[stream].has_pic) return 0u;
    return ((uint32_t)c->streams[stream].w << 16) | c->streams[stream].h;
}

int h263cu_read_yuv(h263cu_ctx* c, uint32_t stream, uint8_t* y, uint8_t* cb, uint8_t* cr) {
    if (!c || stream >= c->max_streams || !y || !cb || !cr) return H263CU_ERR_BAD_ARGUMENT;
    cudaSetDevice(c->device);
    const StreamState& st = c->streams[stream];
    if (!st.has_pic) return H263CU_ERR_NO_PICTURE;
    CU_TRY(cudaStreamSynchronize(c->s_main));
    const size_t cw = (st.w + 1) / 2, ch = (st.h + 1) / 2;
    CU_TRY(cudaMemcpy2D(y, st.w, c->plane(0, stream, st.cur_slot), c->pitch_y, st.w, st.h, cudaMemcpyDeviceToHost));
    // the chroma planes live interleaved on the device: copy the CbCr rows and split them here
    std::vector<uint8_t> pairs;
    try {
        pairs.resize(cw * ch * CHROMA_STEP);
    } catch (const std::bad_alloc&) {
        return H263CU_ERR_OUT_OF_MEMORY;
    }
    CU_TRY(cudaMemcpy2D(pairs.data(), cw * CHROMA_STEP, c->plane(1, stream, st.cur_slot), c->pitch_c, cw * CHROMA_STEP, ch,
                        cudaMemcpyDeviceToHost));
    for (size_t i = 0; i < cw * ch; i++) cb[i] = pairs[2 * i], cr[i] = pairs[2 * i + 1];
    return 0;
}

int h263cu_read_rgba(h263cu_ctx* c, uint32_t stream, uint8_t* rgba) {
    if (!c || stream >= c->max_streams || !rgba) return H263CU_ERR_BAD_ARGUMENT;
    cudaSetDevice(c->device);
    const StreamState& st = c->streams[stream];
    if (!st.has_pic || st.rgba_slot < 0) return H263CU_ERR_NO_PICTURE;
    CU_TRY(cudaStreamSynchronize(c->s_main));
    CU_TRY(cudaMemcpy2D(rgba, (size_t)st.w * 4, c->rgba(stream, st.rgba_slot), c->rgba_pitch, (size_t)st.w * 4, st.h,
                        cudaMemcpyDeviceToHost));
    return 0;
}

int h263cu_checksums(h263cu_ctx* c, const uint32_t* streams, uint32_t n, uint64_t* out4) {
    if (!c || !streams || !out4) return H263CU_ERR_BAD_ARGUMENT;
    if (n == 0) return 0;
    cudaSetDevice(c->device);
    std::vector<ChecksumJob> jobs;
    jobs.reserve((size_t)n * 4);
    for (uint32_t i = 0; i < n; i++) {
        if (streams[i] >= c->max_streams) return H263CU_ERR_BAD_ARGUMENT;
        const StreamState& st = c->streams[streams[i]];
        if (!st.has_pic) return H263CU_ERR_NO_PICTURE;
        const uint32_t cw = (st.w + 1u) / 2u, ch = (st.h + 1u) / 2u;
        jobs.push_back({c->plane(0, streams[i], st.cur_slot), st.w, st.h, c->pitch_y, i * 4 + 0, 1u, 0u});
        jobs.push_back({c->plane(1, streams[i], st.cur_slot), cw, ch, c->pitch_c, i * 4 + 1, (uint32_t)CHROMA_STEP, 0u});
        jobs.push_back({c->plane(2, streams[i], st.cur_slot), cw, ch, c->pitch_c, i * 4 + 2, (uint32_t)CHROMA_STEP, 0u});
        if (st.rgba_slot >= 0)
            jobs.push_back({c->rgba(streams[i], st.rgba_slot), (uint32_t)st.w * 4u, st.h, c->rgba_pitch, i * 4 + 3, 1u, 0u});
    }
    if (jobs.size() > c->jobs_cap) {
        if (c->d_jobs) cudaFree(c->d_jobs);
        if (c->d_sums) cudaFree(c->d_sums);
        c->d_jobs = nullptr, c->d_sums = nullptr;
        c->jobs_cap = 0;
        const size_t cap = (size_t)n * 4 + 64;
        CU_TRY(cudaMalloc((void**)&c->d_jobs, cap * sizeof(ChecksumJob)));
        CU_TRY(cudaMalloc((void**)&c->d_sums, cap * sizeof(unsigned long long)));
        c->jobs_cap = cap;
    }
    CU_TRY(cudaMemcpyAsync(c->d_jobs, jobs.data(), jobs.size() * sizeof(ChecksumJob), cudaMemcpyHostToDevice, c->s_main));
    CU_TRY(cudaMemsetAsync(c->d_sums, 0, (size_t)n * 4 * sizeof(unsigned long long), c->s_main));
    // grid.y is limited to 65535 jobs per launch
    for (size_t first = 0; first < jobs.size(); first += 60000) {
        const uint32_t cnt = (uint32_t)std::min<size_t>(60000, jobs.size() - first);
        launch_checksums(c->d_jobs + first, cnt, c->d_sums, c->s_main);
        c->launches++;
    }
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaMemcpyAsync(out4, c->d_sums, (size_t)n * 4 * sizeof(unsigned long long), cudaMemcpyDeviceToHost, c->s_main));
    CU_TRY(cudaStreamSynchronize(c->s_main));
    return 0;
}

int h263cu_timer_start(h263cu_ctx* c) {
    if (!c) return H263CU_ERR_BAD_ARGUMENT;
    cudaSetDevice(c->device);
    CU_TRY(cudaEventRecord(c->t0, c->s_main));
    return 0;
}
int h263cu_timer_stop(h263cu_ctx* c, float* ms) {
    if (!c || !ms) return H263CU_ERR_BAD_ARGUMENT;
    cudaSetDevice(c->device);
    CU_TRY(cudaEventRecord(c->t1, c->s_main));
    CU_TRY(cudaEventSynchronize(c->t1));
    CU_TRY(cudaEventElapsedTime(ms, c->t0, c->t1));
    return 0;
}
uint64_t h263cu_launch_count(h263cu_ctx* c) { return c ? c->launches : 0; }
uint64_t h263cu_tiled_launch_count(h263cu_ctx* c) { return c ? c->tiled_launches : 0; }

int h263cu_host_times(h263cu_ctx* c, double* parse_seconds, double* other_seconds, uint64_t* calls, int reset) {
    if (!c) return H263CU_ERR_BAD_ARGUMENT;
    if (parse_seconds) *parse_seconds = c->host_parse_s;
    if (other_seconds) *other_seconds = c->host_other_s;
    if (calls) *calls = c->host_calls;
    if (reset) c->host_parse_s = c->host_other_s = 0.0, c->host_calls = 0;
    return 0;
}

int h263cu_profile_enable(h263cu_ctx* c, int enable) {
    if (!c) return H263CU_ERR_BAD_ARGUMENT;
    c->profiling = enable != 0;
    return 0;
}
int h263cu_profile_read(h263cu_ctx* c, double* ms2, uint64_t* launches2) {
    if (!c || !ms2 || !launches2) return H263CU_ERR_BAD_ARGUMENT;
    cudaSetDevice(c->device);
    CU_TRY(cudaStreamSynchronize(c->s_main));
    ms2[0] = ms2[1] = 0.0;
    launches2[0] = launches2[1] = 0;
    for (const auto& sp : c->prof_spans) {
        float ms = 0.f;
        CU_TRY(cudaEventElapsedTime(&ms, sp.a, sp.b));
        ms2[sp.kind] += ms;
        launches2[sp.kind]++;
        c->prof_free.push_back(sp.a);
        c->prof_free.push_back(sp.b);
    }
    c->prof_spans.clear();
    return 0;
}

int h263cu_readback_wait(h263cu_ctx* c, uint32_t age) {
    if (!c || age > 1) return H263CU_ERR_BAD_ARGUMENT;
    cudaSetDevice(c->device);
    if (c->rgba_parity <= age) return H263CU_ERR_NO_PICTURE;  // no such step yet
    const int ring = (int)((c->rgba_parity - 1u - age) & 1u);
    CU_TRY(cudaEventSynchronize(c->rgba_read[ring]));
    return 0;
}

// ---- resident steps as ONE CUDA graph ---------------------------------------------------------------------------
// A single stream's pictures are dependent launches of ~10 us each: issuing them one by one is bound by the launch
// path.  h263cu_graph_build captures the launches of n resident steps into one graph; the descriptors of all their
// pictures are computed once from a simulated walk of the per-stream state and live in their own device array.
struct h263cu_graph {
    cudaGraph_t graph = nullptr;
    cudaGraphExec_t exec = nullptr;
    PicDev* d_pics = nullptr;
    uint32_t out_flags = 0;
    uint64_t launches = 0, tiled_launches = 0;
    uint32_t rgba_steps = 0;
    uint32_t rgba_parity0 = 0;  // parity of the RGBA ring the capture assumed
    std::vector<uint32_t> streams;        // streams the graph touches
    std::vector<StreamState> before, after;  // their state the capture assumed / leaves behind
};

h263cu_graph* h263cu_graph_build(h263cu_ctx* c, h263cu_step* const* steps, uint32_t n_steps, uint32_t out_flags, int* err) {
    int dummy;
    if (!err) err = &dummy;
    *err = 0;
    if (!c || !steps || n_steps == 0) {
        *err = H263CU_ERR_BAD_ARGUMENT;
        return nullptr;
    }
    cudaSetDevice(c->device);
    const bool want_rgba = (out_flags & H263CU_OUT_RGBA) != 0;
    const bool want_deblock = want_rgba && (out_flags & H263CU_OUT_DEBLOCK) != 0;
    h263cu_graph* g = new (std::nothrow) h263cu_graph();
    if (!g) {
        *err = H263CU_ERR_OUT_OF_MEMORY;
        return nullptr;
    }
    auto fail = [&](int code) {
        *err = code;
        h263cu_graph_free(c, g);
        return (h263cu_graph*)nullptr;
    };
    g->out_flags = out_flags;
    g->rgba_parity0 = c->rgba_parity & 1u;
    // ---- walk the steps over a copy of the stream state: the checks of run_step, the descriptors, the end state ----
    std::vector<StreamState> sim;
    std::vector<PicDev> picdev;
    struct StepPlan {
        size_t first_pic;
        uint32_t max_w, max_h;
        bool tiled, aligned16, wide_mv;
    };
    std::vector<StepPlan> plan;
    try {
        sim = c->streams;
        std::vector<uint8_t> touched(c->max_streams, 0);
        uint32_t parity = c->rgba_parity;
        for (uint32_t k = 0; k < n_steps; k++) {
            const h263cu_step* s = steps[k];
            if (!s || s->pics.empty()) return fail(H263CU_ERR_BAD_ARGUMENT);
            StepPlan sp{picdev.size(), 0, 0, true, true, false};
            const uint32_t stamp = ++c->stamp;
            for (const h263cu_pic& p : s->pics) {
                if (p.stream >= c->max_streams || p.width == 0 || p.height == 0 || p.width > c->max_w || p.height > c->max_h)
                    return fail(H263CU_ERR_CAPACITY);
                if ((uint32_t)p.mb_w * 16 < p.width || (uint32_t)p.mb_h * 16 < p.height || (uint32_t)p.mb_w > c->mbw ||
                    (uint32_t)p.mb_h > c->mbh || (uint64_t)p.first_mb + p.n_mbs > s->n_mbs ||
                    (uint64_t)p.first_event + p.n_event_units > s->n_units || p.n_mbs != (uint32_t)p.mb_w * p.mb_h)
                    return fail(H263CU_ERR_BAD_ARGUMENT);
                StreamState& st = sim[p.stream];
                if (st.stamp == stamp) return fail(H263CU_ERR_BAD_ARGUMENT);
                st.stamp = stamp;
                if (p.flags & H263CU_PICFLAG_HAS_INTER) {
                    if (!st.has_ref) return fail(H263CU_ERR_UNCODED_IFRAME_BLOCKS);
                    if (st.ref_w != p.width || st.ref_h != p.height) return fail(H263CU_ERR_REFERENCE_WOULD_ABORT);
                    if (!(p.flags & H263CU_PICFLAG_MV_IN_RANGE)) sp.wide_mv = true;
                    if (!st.padded) sp.tiled = false;
                }
                if ((p.width | p.height) & 15) sp.aligned16 = false;
                sp.max_w = std::max<uint32_t>(sp.max_w, p.width), sp.max_h = std::max<uint32_t>(sp.max_h, p.height);
                if (!touched[p.stream]) touched[p.stream] = 1, g->streams.push_back(p.stream);
            }
            if (c->force_kernel == 1) sp.tiled = false;
            const int ring = (int)(parity & 1u);
            for (const h263cu_pic& p : s->pics) {
                StreamState& st = sim[p.stream];
                picdev.push_back(make_picdev(c, p, st, want_rgba, ring));
                advance_stream(st, p, want_rgba, ring, sp.tiled);
            }
            if (want_rgba) parity++, g->rgba_steps++;
            g->launches += want_deblock ? 2 : 1;
            if (sp.tiled) g->tiled_launches++;
            plan.push_back(sp);
        }
        for (uint32_t sid : g->streams) g->before.push_back(c->streams[sid]), g->after.push_back(sim[sid]);
    } catch (const std::bad_alloc&) {
        return fail(H263CU_ERR_OUT_OF_MEMORY);
    }
    if (cudaMalloc((void**)&g->d_pics, picdev.size() * sizeof(PicDev)) != cudaSuccess) return fail(H263CU_ERR_OUT_OF_MEMORY);
    if (cudaMemcpy(g->d_pics, picdev.data(), picdev.size() * sizeof(PicDev), cudaMemcpyHostToDevice) != cudaSuccess)
        return fail(H263CU_ERR_CUDA);
    // ---- capture ----
    if (cudaStreamSynchronize(c->s_main) != cudaSuccess) return fail(H263CU_ERR_CUDA);
    if (cudaStreamBeginCapture(c->s_main, cudaStreamCaptureModeThreadLocal) != cudaSuccess) return fail(H263CU_ERR_CUDA);
    const Pools pools{c->y_pool, c->c_pool, c->rgba_pool, c->pitch_y, c->pitch_c, c->rgba_pitch};
    for (uint32_t k = 0; k < n_steps; k++) {
        const h263cu_step* s = steps[k];
        const StepPlan& sp = plan[k];
        const PicDev* dp = g->d_pics + sp.first_pic;
        launch_recon(dp, s->d_mbs, s->d_events, s->n_mbs, want_rgba && !want_deblock, sp.tiled ? (sp.aligned16 ? 1 : 2) : 0, sp.wide_mv, pools,
                     &c->rgba_map, OUT_POOL, nullptr, c->s_main);
        if (want_deblock) {
            if (sp.aligned16 && c->force_kernel != 1)
                launch_deblock_rgba_tile(dp, (uint32_t)s->pics.size(), sp.max_w, sp.max_h, nullptr, c->s_main);
            else
                launch_deblock_rgba(dp, (uint32_t)s->pics.size(), sp.max_w, sp.max_h, nullptr, c->s_main);
        }
    }
    if (cudaStreamEndCapture(c->s_main, &g->graph) != cudaSuccess || !g->graph) {
        cudaGetLastError();
        return fail(H263CU_ERR_CUDA);
    }
    if (cudaGraphInstantiate(&g->exec, g->graph, 0) != cudaSuccess) {
        cudaGetLastError();
        return fail(H263CU_ERR_CUDA);
    }
    return g;
}

int h263cu_graph_launch(h263cu_ctx* c, h263cu_graph* g) {
    if (!c || !g || !g->exec) return H263CU_ERR_BAD_ARGUMENT;
    cudaSetDevice(c->device);
    // the graph holds plane addresses: it runs only from the state it was captured for
    if (g->rgba_steps && (c->rgba_parity & 1u) != g->rgba_parity0) return H263CU_ERR_BAD_ARGUMENT;
    for (size_t i = 0; i < g->streams.size(); i++) {
        const StreamState &a = c->streams[g->streams[i]], &b = g->before[i];
        if (a.has_pic != b.has_pic || (a.has_pic && a.cur_slot != b.cur_slot) || a.has_ref != b.has_ref ||
            (a.has_ref && (a.ref_slot != b.ref_slot || a.ref_w != b.ref_w || a.ref_h != b.ref_h || a.padded != b.padded)))
            return H263CU_ERR_BAD_ARGUMENT;
    }
    if (g->rgba_steps) {  // read-backs of earlier steps may still hold the RGBA ring
        CU_TRY(cudaStreamWaitEvent(c->s_main, c->rgba_read[0], 0));
        CU_TRY(cudaStreamWaitEvent(c->s_main, c->rgba_read[1], 0));
    }
    CU_TRY(cudaGraphLaunch(g->exec, c->s_main));
    for (size_t i = 0; i < g->streams.size(); i++) {
        StreamState& st = c->streams[g->streams[i]];
        const uint32_t seen = st.seen, stamp = st.stamp;
        st = g->after[i];
        st.seen = seen, st.stamp = stamp;
    }
    c->rgba_parity += g->rgba_steps;
    c->launches += g->launches;
    c->tiled_launches += g->tiled_launches;
    if (g->rgba_steps) {
        CU_TRY(cudaEventRecord(c->rgba_written[0], c->s_main));
        CU_TRY(cudaEventRecord(c->rgba_written[1], c->s_main));
    }
    return 0;
}

void h263cu_graph_free(h263cu_ctx* c, h263cu_graph* g) {
    if (!g) return;
    if (c) {
        cudaSetDevice(c->device);
        cudaStreamSynchronize(c->s_main);
    }
    if (g->exec) cudaGraphExecDestroy(g->exec);
    if (g->graph) cudaGraphDestroy(g->graph);
    if (g->d_pics) cudaFree(g->d_pics);
    delete g;
}

// ---- one process, several GPUs: a group of contexts fed by ONE shared pool of parser threads (SURVEY.md 8e) ----
struct h263cu_group {
    std::vector<h263cu_ctx*> ctx;
    uint32_t streams_per_device = 0;
    int threads = 0;
    // per-device argument slices of the current step (reused)
    struct Slice {
        std::vector<h263cu_parser*> parsers;
        std::vector<const uint8_t*> packets;
        std::vector<size_t> lens;
        std::vector<uint32_t> ids, input, pos;
        std::vector<h263cu_tensor_crop> crops;  // the fit's crop boxes of the slice's inputs
        std::vector<int> errs;
    };
    std::vector<Slice> slice;
};

h263cu_group* h263cu_group_create(const int* devices, uint32_t n_devices, uint32_t streams_per_device, uint32_t max_width,
                                  uint32_t max_height, int threads, int* err) {
    int dummy;
    if (!err) err = &dummy;
    *err = 0;
    if (!devices || n_devices == 0 || n_devices > 64 || streams_per_device == 0) {
        *err = H263CU_ERR_BAD_ARGUMENT;
        return nullptr;
    }
    h263cu_group* g = new (std::nothrow) h263cu_group();
    if (!g) {
        *err = H263CU_ERR_OUT_OF_MEMORY;
        return nullptr;
    }
    g->streams_per_device = streams_per_device, g->threads = threads;
    try {
        g->slice.resize(n_devices);
    } catch (const std::bad_alloc&) {
        delete g;
        *err = H263CU_ERR_OUT_OF_MEMORY;
        return nullptr;
    }
    for (uint32_t d = 0; d < n_devices; d++) {
        h263cu_ctx* c = h263cu_create(devices[d], streams_per_device, max_width, max_height, 0, err);
        if (!c) {
            h263cu_group_destroy(g);
            return nullptr;
        }
        g->ctx.push_back(c);
    }
    return g;
}

void h263cu_group_destroy(h263cu_group* g) {
    if (!g) return;
    for (h263cu_ctx* c : g->ctx) h263cu_destroy(c);
    delete g;
}

uint32_t h263cu_group_size(const h263cu_group* g) { return g ? (uint32_t)g->ctx.size() : 0u; }
h263cu_ctx* h263cu_group_ctx(h263cu_group* g, uint32_t index) { return g && index < g->ctx.size() ? g->ctx[index] : nullptr; }

// The body of h263cu_group_decode_step (outs == yuv_outs == tensor_outs == NULL), h263cu_group_decode_step_device (outs:
// one per device), h263cu_group_decode_step_device_yuv (yuv_outs: one per device) and
// h263cu_group_decode_step_device_tensor (tensor_outs: one per device), with `fit` h263cu_group_decode_step_device_tensor_fit
// and with `filter` too h263cu_group_decode_step_device_tensor_filter.
static int group_decode(h263cu_group* g, h263cu_parser* const* parsers, const uint8_t* const* packets, const size_t* lens,
                        const uint32_t* stream_ids, uint32_t n, uint32_t out_flags, uint8_t* host_rgba, uint64_t rgba_stride,
                        const h263cu_device_rgba* outs, const h263cu_device_yuv* yuv_outs, const h263cu_device_tensor* tensor_outs,
                        const h263cu_tensor_fit* fit, int* per_pic_err, uint32_t* n_decoded,
                        uint32_t filter = H263CU_FILTER_BILINEAR) {
    if (!g || !parsers || !packets || !lens) return H263CU_ERR_BAD_ARGUMENT;
    if (n_decoded) *n_decoded = 0;
    const uint32_t nd = (uint32_t)g->ctx.size();
    if (fit && check_tensor_fit(fit, n)) return H263CU_ERR_BAD_ARGUMENT;
    if (outs || yuv_outs || tensor_outs)  // every device's buffer is checked before any device parses
        for (uint32_t d = 0; d < nd; d++) {
            cudaSetDevice(g->ctx[d]->device);
            const int e = outs ? check_device_rgba(g->ctx[d], &outs[d])
                               : yuv_outs ? check_device_yuv(g->ctx[d], &yuv_outs[d]) : check_device_tensor(g->ctx[d], &tensor_outs[d]);
            if (e) return e;
        }
    try {
        for (auto& sl : g->slice)
            sl.parsers.clear(), sl.packets.clear(), sl.lens.clear(), sl.ids.clear(), sl.input.clear(), sl.pos.clear(), sl.crops.clear();
        for (uint32_t i = 0; i < n; i++) {
            const uint32_t sid = stream_ids ? stream_ids[i] : i;
            const uint32_t d = sid % nd, local = sid / nd;
            if (local >= g->streams_per_device) return H263CU_ERR_CAPACITY;
            h263cu_group::Slice& sl = g->slice[d];
            sl.parsers.push_back(parsers[i]), sl.packets.push_back(packets[i]), sl.lens.push_back(lens[i]);
            sl.ids.push_back(local), sl.input.push_back(i), sl.pos.push_back(d * g->streams_per_device + local);
            if (fit && fit->crops) sl.crops.push_back(fit->crops[i]);
        }
        for (auto& sl : g->slice) sl.errs.assign(sl.ids.size(), 0);
    } catch (const std::bad_alloc&) {
        return H263CU_ERR_OUT_OF_MEMORY;
    }
    // Device by device: the pictures of device d are parsed on ALL of the group's parser threads and queued on d (upload,
    // kernels and read-back are asynchronous), then the threads move on to device d + 1 while d works and copies back.
    // No core is tied to a GPU: a device with fewer or cheaper pictures just takes less of the pool's time.
    int first_err = 0;
    uint32_t total = 0;
    for (uint32_t d = 0; d < nd; d++) {
        h263cu_group::Slice& sl = g->slice[d];
        const uint32_t m = (uint32_t)sl.ids.size();
        if (m == 0) continue;
        uint32_t got = 0;
        // RGBA of global stream s goes to host_rgba + ((s % n_devices) * streams_per_device + s / n_devices) * rgba_stride:
        // device-major, so that the pictures of one device are contiguous and leave in few large copies
        int e;
        if (outs || yuv_outs || tensor_outs) {
            // device output: the local slot of the stream is its slot in the device's buffer
            h263cu_tensor_fit dfit{};
            if (fit) dfit = *fit, dfit.crops = fit->crops ? sl.crops.data() : nullptr;
            e = decode_step_scattered(g->ctx[d], sl.parsers.data(), sl.packets.data(), sl.lens.data(), sl.ids.data(), m, g->threads,
                                      out_flags, nullptr, 0, sl.ids.data(), outs ? &outs[d] : nullptr, yuv_outs ? &yuv_outs[d] : nullptr,
                                      tensor_outs ? &tensor_outs[d] : nullptr, fit ? &dfit : nullptr, sl.errs.data(), &got, filter);
        } else if (host_rgba) {
            e = decode_step_scattered(g->ctx[d], sl.parsers.data(), sl.packets.data(), sl.lens.data(), sl.ids.data(), m, g->threads,
                                      out_flags, host_rgba, rgba_stride, sl.pos.data(), nullptr, nullptr, nullptr, nullptr, sl.errs.data(),
                                      &got);
        } else {
            e = h263cu_decode_step(g->ctx[d], sl.parsers.data(), sl.packets.data(), sl.lens.data(), sl.ids.data(), m, g->threads, out_flags,
                                   nullptr, 0, sl.errs.data(), &got);
        }
        if (e && !first_err) first_err = e;
        total += got;
        if (per_pic_err)
            for (uint32_t k = 0; k < m; k++) per_pic_err[sl.input[k]] = e ? e : sl.errs[k];
    }
    if (n_decoded) *n_decoded = total;
    return first_err;
}

int h263cu_group_decode_step(h263cu_group* g, h263cu_parser* const* parsers, const uint8_t* const* packets, const size_t* lens,
                             const uint32_t* stream_ids, uint32_t n, uint32_t out_flags, uint8_t* host_rgba, uint64_t rgba_stride,
                             int* per_pic_err, uint32_t* n_decoded) {
    return group_decode(g, parsers, packets, lens, stream_ids, n, out_flags, host_rgba, rgba_stride, nullptr, nullptr, nullptr, nullptr,
                        per_pic_err, n_decoded);
}

int h263cu_group_decode_step_device(h263cu_group* g, h263cu_parser* const* parsers, const uint8_t* const* packets, const size_t* lens,
                                    const uint32_t* stream_ids, uint32_t n, uint32_t out_flags, const h263cu_device_rgba* outs,
                                    int* per_pic_err, uint32_t* n_decoded) {
    if (!outs) return H263CU_ERR_BAD_ARGUMENT;
    return group_decode(g, parsers, packets, lens, stream_ids, n, out_flags, nullptr, 0, outs, nullptr, nullptr, nullptr, per_pic_err,
                        n_decoded);
}

int h263cu_group_decode_step_device_yuv(h263cu_group* g, h263cu_parser* const* parsers, const uint8_t* const* packets, const size_t* lens,
                                        const uint32_t* stream_ids, uint32_t n, uint32_t out_flags, const h263cu_device_yuv* outs,
                                        int* per_pic_err, uint32_t* n_decoded) {
    if (!outs) return H263CU_ERR_BAD_ARGUMENT;
    return group_decode(g, parsers, packets, lens, stream_ids, n, out_flags, nullptr, 0, nullptr, outs, nullptr, nullptr, per_pic_err,
                        n_decoded);
}

int h263cu_group_decode_step_device_tensor(h263cu_group* g, h263cu_parser* const* parsers, const uint8_t* const* packets,
                                           const size_t* lens, const uint32_t* stream_ids, uint32_t n, uint32_t out_flags,
                                           const h263cu_device_tensor* outs, int* per_pic_err, uint32_t* n_decoded) {
    if (!outs) return H263CU_ERR_BAD_ARGUMENT;
    return group_decode(g, parsers, packets, lens, stream_ids, n, out_flags, nullptr, 0, nullptr, nullptr, outs, nullptr, per_pic_err,
                        n_decoded);
}

int h263cu_group_decode_step_device_tensor_fit(h263cu_group* g, h263cu_parser* const* parsers, const uint8_t* const* packets,
                                               const size_t* lens, const uint32_t* stream_ids, uint32_t n, uint32_t out_flags,
                                               const h263cu_device_tensor* outs, const h263cu_tensor_fit* fit, int* per_pic_err,
                                               uint32_t* n_decoded) {
    if (!outs || !fit) return H263CU_ERR_BAD_ARGUMENT;
    return group_decode(g, parsers, packets, lens, stream_ids, n, out_flags, nullptr, 0, nullptr, nullptr, outs, fit, per_pic_err,
                        n_decoded);
}

int h263cu_group_decode_step_device_tensor_filter(h263cu_group* g, h263cu_parser* const* parsers, const uint8_t* const* packets,
                                                  const size_t* lens, const uint32_t* stream_ids, uint32_t n, uint32_t out_flags,
                                                  const h263cu_device_tensor* outs, const h263cu_tensor_fit* fit, uint32_t filter,
                                                  int* per_pic_err, uint32_t* n_decoded) {
    if (!outs || !fit || filter > H263CU_FILTER_BICUBIC_AA) return H263CU_ERR_BAD_ARGUMENT;
    return group_decode(g, parsers, packets, lens, stream_ids, n, out_flags, nullptr, 0, nullptr, nullptr, outs, fit, per_pic_err,
                        n_decoded, filter);
}

int h263cu_group_sync(h263cu_group* g) {
    if (!g) return H263CU_ERR_BAD_ARGUMENT;
    int first = 0;
    for (h263cu_ctx* c : g->ctx) {
        const int e = h263cu_sync(c);
        if (e && !first) first = e;
    }
    return first;
}

// ---- stateless drop-ins: host buffers in, host buffers out ---------------------------------
// One scratch set per device (device buffer, pinned staging, stream), used under one lock: the calls run on the
// device that is current on the calling thread, like any CUDA runtime call.
namespace {
struct DropInScratch {
    uint8_t* dev = nullptr;
    size_t dev_cap = 0;
    uint8_t* pinned = nullptr;
    size_t pinned_cap = 0;
    cudaStream_t stream = nullptr;
};
std::mutex g_scratch_mutex;
DropInScratch g_scratch[64];

int scratch_get(size_t dev_bytes, size_t pinned_bytes, DropInScratch** out) {
    int device = 0;
    CU_TRY(cudaGetDevice(&device));
    if (device < 0 || device >= 64) return H263CU_ERR_NO_DEVICE;
    DropInScratch& sc = g_scratch[device];
    if (!sc.stream) CU_TRY(cudaStreamCreateWithFlags(&sc.stream, cudaStreamNonBlocking));
    if (dev_bytes > sc.dev_cap) {
        if (sc.dev) cudaFree(sc.dev);
        sc.dev = nullptr, sc.dev_cap = 0;
        CU_TRY(cudaMalloc((void**)&sc.dev, dev_bytes + dev_bytes / 4));
        sc.dev_cap = dev_bytes + dev_bytes / 4;
    }
    if (pinned_bytes > sc.pinned_cap) {
        if (sc.pinned) cudaFreeHost(sc.pinned);
        sc.pinned = nullptr, sc.pinned_cap = 0;
        CU_TRY(cudaHostAlloc((void**)&sc.pinned, pinned_bytes + pinned_bytes / 4, cudaHostAllocDefault));
        sc.pinned_cap = pinned_bytes + pinned_bytes / 4;
    }
    *out = &sc;
    return 0;
}
}  // namespace

int h263cu_yuv420_to_rgba(const uint8_t* y, const uint8_t* chroma_b, const uint8_t* chroma_r, size_t y_len,
                          size_t y_width, uint8_t* rgba_out) {
    if (y_len == 0) return 0;  // bt601.rs:106-112
    if (!y || !chroma_b || !chroma_r || !rgba_out || y_width == 0 || y_len % y_width != 0 || y_width > 65535)
        return H263CU_ERR_BAD_ARGUMENT;
    if (h263cu_device_count() == 0) return H263CU_ERR_NO_DEVICE;
    std::lock_guard<std::mutex> lock(g_scratch_mutex);
    const size_t h = y_len / y_width, cw = (y_width + 1) / 2, ch = (h + 1) / 2, clen = cw * ch;
    const size_t o_cb = round_up(y_len, 256), o_cr = o_cb + round_up(clen, 256), o_out = o_cr + round_up(clen, 256);
    DropInScratch* sc;
    int e = scratch_get(o_out + y_len * 4, o_out + y_len * 4, &sc);
    if (e) return e;
    // pinned staging in both directions: one asynchronous copy each way on the drop-ins' own stream
    std::memcpy(sc->pinned, y, y_len);
    std::memcpy(sc->pinned + o_cb, chroma_b, clen);
    std::memcpy(sc->pinned + o_cr, chroma_r, clen);
    CU_TRY(cudaMemcpyAsync(sc->dev, sc->pinned, o_cr + clen, cudaMemcpyHostToDevice, sc->stream));
    launch_yuv420_to_rgba(sc->dev, sc->dev + o_cb, sc->dev + o_cr, (uint32_t)y_width, (uint32_t)h, sc->dev + o_out, sc->stream);
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaMemcpyAsync(sc->pinned + o_out, sc->dev + o_out, y_len * 4, cudaMemcpyDeviceToHost, sc->stream));
    CU_TRY(cudaStreamSynchronize(sc->stream));
    std::memcpy(rgba_out, sc->pinned + o_out, y_len * 4);
    return 0;
}

int h263cu_deblock(const uint8_t* data, size_t len, size_t width, uint8_t strength, uint8_t* out) {
    if (len == 0) return 0;
    if (!data || !out || width == 0 || len % width != 0 || width > 65535) return H263CU_ERR_BAD_ARGUMENT;
    if (h263cu_device_count() == 0) return H263CU_ERR_NO_DEVICE;
    std::lock_guard<std::mutex> lock(g_scratch_mutex);
    const size_t h = len / width;
    const size_t o_out = round_up(len, 256);
    DropInScratch* sc;
    int e = scratch_get(o_out + len, o_out + len, &sc);
    if (e) return e;
    std::memcpy(sc->pinned, data, len);
    CU_TRY(cudaMemcpyAsync(sc->dev, sc->pinned, len, cudaMemcpyHostToDevice, sc->stream));
    launch_deblock_plane(sc->dev, sc->dev + o_out, (uint32_t)width, (uint32_t)h, strength, sc->stream);
    CU_TRY(cudaGetLastError());
    CU_TRY(cudaMemcpyAsync(sc->pinned + o_out, sc->dev + o_out, len, cudaMemcpyDeviceToHost, sc->stream));
    CU_TRY(cudaStreamSynchronize(sc->stream));
    std::memcpy(out, sc->pinned + o_out, len);
    return 0;
}

}  // extern "C"
