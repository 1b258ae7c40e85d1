// Shared declarations for the sm_100a JPEG encode path (kernels + C-ABI).
#pragma once

#include <cuda.h>
#include <cuda_runtime.h>

#include <cstdint>
#include <exception>
#include <cstdio>
#include <string>
#include <vector>

#include "../../include/jpgenc_b200.h"

namespace jpgenc {

constexpr int kBlocksPerMcu = 6;          // Y00 Y01 Y10 Y11 Cb Cr  (src/Image.cpp:959-967)
constexpr int kCoefPerBlock = 64;
constexpr int kBlockBytes = 128;          // 64 x int16

// zigzag scan: natural index (v*8+u) of the i-th coefficient (include/Coding.hpp:57-81)
#define JPGENC_ZIGZAG_LIST                                                                            \
    0, 1, 8, 16, 9, 2, 3, 10, 17, 24, 32, 25, 18, 11, 4, 5, 12, 19, 26, 33, 40, 48, 41, 34, 27, 20, 13, 6, \
    7, 14, 21, 28, 35, 42, 49, 56, 57, 50, 43, 36, 29, 22, 15, 23, 30, 37, 44, 51, 58, 59, 52, 45, 38, \
    31, 39, 46, 53, 60, 61, 54, 47, 55, 62, 63

// Per-table constants of the FP32 fast path, natural order.
//   mul[i] = s_v * s_u / q[i]   (AAN output scales folded with the quantiser; Dct.hpp:36-43, Coding.hpp:92-94)
//   thr[i] = 0.5 - delta_i      a quotient whose distance to the nearest integer exceeds thr is "on a rounding
//                               boundary" as far as FP32 can tell; such blocks are redone in exact FP64
struct QuantConsts {
    float mul[64];
    float thr[64];
};
// the same constants in the pair order of the packed (FP32x2) transform: entry [u*4+q] holds natural indices
// ((2q)*8+u, (2q+1)*8+u)
struct QuantConsts2 {
    float2 mul[32];
    float2 thr[32];
};

// Constants of the exact path: the reference's own doubles (Dct.hpp:21-43) and integer quantisers.
struct ExactConsts {
    double a1, a2, a3, a4, a5;
    double s[8];
    double scale;                         // 255. / maxval  (src/Image.cpp:465)
    uint8_t qy[64];
    uint8_t qc[64];
};

struct ColorConsts {                      // FP32 fast path; sample scale folded in, chroma rows also carry the /4
    float y[3], cb[3], cr[3];
};

// Planar RGB: three planes of one byte per pixel, one row pitch.  It has no JPGENC_PIXEL_* code (the calls take three plane
// pointers); inside the library it is this format.
constexpr int kPixelPlanar = 17;
// YUV 4:2:0 frames (jpgenc_*_yuv420; JPGENC_YUV_I420 / JPGENC_YUV_NV12 inside the library): a Y plane of one byte per pixel and
// chroma planes of ceil(w/2) x ceil(h/2) samples -- U and V apart (I420) or interleaved U, V pairs (NV12)
constexpr int kPixelI420 = 18;
constexpr int kPixelNV12 = 19;
// YUV 4:2:2 and 4:4:4 frames (jpgenc_*_yuv; JPGENC_YUV_I422 .. JPGENC_YUV_UYVY): chroma of ceil(w/2) x h samples -- U and V apart
// (I422) or interleaved U, V pairs (NV16) --, of w x h samples (I444), or 4:2:2 packed into the Y plane as groups of two pixels
// Y0 U Y1 V (YUYV) or U Y0 V Y1 (UYVY)
constexpr int kPixelI422 = 20;
constexpr int kPixelNV16 = 21;
constexpr int kPixelI444 = 22;
constexpr int kPixelYUYV = 23;
constexpr int kPixelUYVY = 24;
__host__ __device__ constexpr bool is_yuv(int format) { return format >= kPixelI420 && format <= kPixelUYVY; }
__host__ __device__ constexpr bool is_packed_yuv(int format) { return format == kPixelYUYV || format == kPixelUYVY; }
// chroma subsampling of a YUV format: vertical (4:2:0) and horizontal (all but 4:4:4), as shifts
__host__ __device__ constexpr uint32_t chroma_vsub(int format) { return format == kPixelI420 || format == kPixelNV12 ? 1u : 0u; }
__host__ __device__ constexpr uint32_t chroma_hsub(int format) { return format == kPixelI444 ? 0u : 1u; }

// bytes of one chroma row of a YUV image w pixels wide (NV12 / NV16: U, V pairs; packed formats have no chroma plane)
__host__ __device__ constexpr uint32_t chroma_row_bytes(int format, uint32_t w) {
    return is_packed_yuv(format) ? 0u : format == kPixelI444 ? w : (w + 1) / 2 * (format == kPixelNV12 || format == kPixelNV16 ? 2u : 1u);
}

// bytes per pixel of a JPGENC_PIXEL_* format (planar: of one plane; YUV: of the Y plane, 2 for packed 4:2:2)
__host__ __device__ constexpr uint32_t pixel_bytes(int format) {
    return is_packed_yuv(format) ? 2u : format >= JPGENC_PIXEL_GRAY ? 1u : format >= JPGENC_PIXEL_RGBA ? 4u : 3u;
}
// bytes of one row of the first plane (packed 4:2:2: whole groups of two pixels, 4 ceil(w/2))
__host__ __device__ constexpr uint32_t row_bytes(int format, uint32_t w) { return is_packed_yuv(format) ? (w + 1) / 2 * 4 : w * pixel_bytes(format); }

// Where an image's bytes are and how they are laid out: up to three planes, the format, the row pitch of the first plane and
// a second pitch (YUV: of the chroma planes; planar RGB: equal to `pitch`; unused otherwise).  Tight RGB is {{p}, RGB, w * 3,
// 0}.  Planar RGB: planes R, G, B; YUV: Y, U, V (NV12 / NV16: Y, UV, null; YUYV / UYVY: the packed plane, null, null).
struct PixelSource {
    const uint8_t* plane[3] = {nullptr, nullptr, nullptr};
    int format = JPGENC_PIXEL_RGB;        // JPGENC_PIXEL_*, kPixelPlanar or kPixelI420 .. kPixelUYVY
    uint32_t pitch = 0;
    uint32_t pitch2 = 0;
};
// pointers (= planes) a caller passes for an image of this format
__host__ __device__ constexpr uint32_t source_planes(int format) {
    return format == kPixelPlanar || (is_yuv(format) && !is_packed_yuv(format)) ? 3u : 1u;
}

// the second and third plane of one image of a pass and its second pitch: one entry per image follows the FrameGeom array in
// the same copy for the formats of several planes (planar RGB, YUV)
struct ExtraPlanes {
    const uint8_t* plane[2];
    uint64_t pitch2;
};

// ---- a pass of images of individual sizes (jpgenc_encode_images_packed), device resident -------------------------
// One entry per image of the pass and one behind the last, whose prefix fields hold the pass totals: the images' work
// units are numbered through the whole pass, and a CTA finds its image by a search over the prefix of its own unit.
// All prefixes fit 32 bits: a pass has fewer than 2^31 coefficient blocks.
struct FrameGeom {
    const uint8_t* rgb;
    uint32_t real_w, real_h, mcu_w, mcu_h;
    uint32_t block0;                      // first coefficient block (blocks are numbered through the pass)
    uint32_t strip0;                      // first K1 strip (a CTA: kMcus MCUs of one MCU row)
    uint32_t tile0;                       // first K2 tile = item slab; its K3 ranges start at tile0 * split
    uint32_t group0;                      // first K3 group (a CTA of K3a / K3b)
    uint32_t super0;                      // first K3 super-group (256 groups)
    uint32_t pitch;                       // bytes from one pixel row to the next (read only by the kernels of other pixel layouts)
};
static_assert(sizeof(FrameGeom) == 48, "FrameGeom is copied as an array");

// the image f (0 <= f < F) whose units [geom[f].*key, geom[f + 1].*key) contain unit x, found by a whole warp in two rounds of
// 32 parallel probes for F <= 1024 (every lane must take part; every lane returns f)
__device__ __forceinline__ uint32_t geom_find_warp(const FrameGeom* geom, uint32_t F, uint32_t x, uint32_t FrameGeom::*key) {
    const uint32_t lane = threadIdx.x & 31;
    uint32_t lo = 0, n = F;                                   // the answer lies in [lo, lo + n)
    while (n > 1) {
        const uint32_t step = (n + 31) / 32, i = lo + lane * step;
        const unsigned le = __ballot_sync(0xffffffffu, i < lo + n && geom[i].*key <= x);   // lane 0 always holds
        const uint32_t k = 31 - __clz(le);
        lo += k * step;
        n = min(step, n - k * step);
    }
    return lo;
}

struct ForwardParams {
    const uint8_t* rgb;                   // src.plane[0] of one image (K1 reads it here: at this offset the tight-RGB kernels compile
                                          // to the code they were measured with) ...
    const uint8_t* const* frames;         // ... or (non-null) one device pointer per frame of a batch of equally sized frames
    uint32_t blocks_per_frame;            // frame f owns coefficient blocks [f * blocks_per_frame, (f + 1) * blocks_per_frame)
    int16_t* coef;
    uint32_t* refine_list;                // block ids (mcu*6+k) that need the exact path
    uint32_t* refine_count;
    uint32_t refine_cap;
    uint32_t real_w, real_h;
    uint32_t mcu_w, mcu_h;
    uint32_t mcu_y0;                      // first MCU row of this launch (band-wise launches behind the H2D copies)
    uint32_t prefetch_ahead;              // > 0: every CTA pulls the strip of the CTA this many positions later into L2
    ColorConsts color;
    QuantConsts2 luma;
    QuantConsts2 chroma;
    alignas(64) CUtensorMap coef_map;     // coefficient array as rows of 128 bytes, for the tensor store of full strips
    // images of individual sizes (forward_mixed_kernel): geom[nframes + 1], `strips` CTAs in all; the fields above that
    // describe one size (frames, blocks_per_frame, real_w .. mcu_y0) and `src` are unused there
    const FrameGeom* geom;
    uint32_t nframes;
    uint32_t strips;
    PixelSource src;                      // the single image: its other planes and pitches (the format is the kernels' template parameter)
    // images of individual sizes in a format of several planes: extra[f] (plane 0 and `pitch` are in FrameGeom)
    const ExtraPlanes* extra;
};

// host side: the totals of the pass of images of individual sizes bound to a context (the device reads them from the
// entry behind the last image of FrameGeom)
struct MixedPass {
    bool on = false;
    bool aligned = false;                 // every image has real_w % 16 == 0 and a 16-byte aligned pointer (K1's bulk copies)
    int format = -1;                      // JPGENC_PIXEL_*, kPixelPlanar or kPixelI420 .. kPixelUYVY: the pixel-layout kernels (with
                                          // FrameGeom::pitch and, for several planes, ExtraPlanes); -1 tight RGB
    uint32_t blocks = 0, strips = 0, tiles = 0, groups = 0, supers = 0;
    uint32_t split = 1;                   // K3 ranges per K2 tile, one choice for the whole pass (launch_entropy)
};

__host__ __device__ inline uint64_t umin64(uint64_t a, uint64_t b) { return a < b ? a : b; }

// device-side Huffman tables, indexed [table][symbol]:
//   entry  (length << 16) | right-aligned code; 0 = absent
//   fast   ((length + cat) << 27) | (code << cat) with cat = symbol & 15: OR the magnitude bits in and the word is the
//          complete (bit count, bits) pair of the symbol; 0 where that does not fit in 27 bits (or the symbol is absent)
struct DeviceTables {
    uint32_t entry[4][256];
    uint32_t fast[4][256];
};

// ---- entropy-stage geometry of a pass (one image = a pass of one frame), device resident -------------------------
// Produced either by the host (single image: the tables are built on the host, so the sizes are known there) or by
// finalize_tables_kernel (batches: tables, sizes and offsets never leave the device); K3a/K3b/K4 read it from device
// memory and take no size from the host.  One block of memory, in this order:
//   PassHeader | raw_off u64[F] | raw_bytes u64[F] | frame_bits u64[F] | file_base u64[F] | k4_tile0 u32[F+1] | hdr_len u32[F]
//   | (8-byte aligned) total_bits u64[F] | ff_incl u64[F]
// The part up to hdr_len is input of K3/K4; total_bits (K3b) and ff_incl (K4) are their results.
struct PassHeader {
    unsigned long long raw_total;    // bytes of `raw` in use: every frame's scan padded to 16 bytes, plus slack
    unsigned long long out_total;    // bytes of the pass's output before byte stuffing: sum of hdr_len + raw_bytes + tail
    unsigned long long raw_sum;      // sum of raw_bytes (an upper bound of the FF bytes K4 can stuff)
    uint32_t k4_tiles;               // K4 tiles of all frames
    uint32_t error;                  // kPass* below; when set, K3a/K3b/K4 return at once
    uint32_t error_frame;
    uint32_t nframes;
    unsigned long long pad[3];
};
static_assert(sizeof(PassHeader) == 64, "PassHeader is copied as 64 bytes");
constexpr uint32_t kPassOk = 0, kPassMissingSymbol = 1, kPassNoSymbols = 2, kPassRawOverflow = 4, kPassOutOverflow = 8;

struct PassMeta {
    PassHeader* hdr;
    unsigned long long *raw_off, *raw_bytes, *frame_bits, *file_base;
    uint32_t *k4_tile0, *hdr_len;
    unsigned long long *total_bits, *ff_incl;
};
__host__ __device__ inline size_t pass_meta_input_bytes(uint32_t F) {
    return (sizeof(PassHeader) + static_cast<size_t>(F) * 32 + (static_cast<size_t>(F) + 1) * 4 + static_cast<size_t>(F) * 4 + 7) & ~static_cast<size_t>(7);
}
__host__ __device__ inline size_t pass_meta_bytes(uint32_t F) { return pass_meta_input_bytes(F) + static_cast<size_t>(F) * 16; }
__host__ __device__ inline PassMeta pass_meta_view(void* base, uint32_t F) {
    uint8_t* b = static_cast<uint8_t*>(base);
    PassMeta m;
    m.hdr = reinterpret_cast<PassHeader*>(b);
    m.raw_off = reinterpret_cast<unsigned long long*>(b + sizeof(PassHeader));
    m.raw_bytes = m.raw_off + F;
    m.frame_bits = m.raw_bytes + F;
    m.file_base = m.frame_bits + F;
    m.k4_tile0 = reinterpret_cast<uint32_t*>(m.file_base + F);
    m.hdr_len = m.k4_tile0 + F + 1;
    m.total_bits = reinterpret_cast<unsigned long long*>(b + pass_meta_input_bytes(F));
    m.ff_incl = m.total_bits + F;
    return m;
}
// a frame's raw (un-stuffed) scan occupies its bytes rounded up to 16, plus slack for the last words K3b touches
__host__ __device__ inline unsigned long long raw_slot_bytes(unsigned long long nbytes) { return ((nbytes + 15) & ~15ull) + 64; }

}  // namespace jpgenc

namespace jpgenc { class TablePool; class HostPool; }

constexpr int kGraphKeyWords = 8;         // jpgenc_ctx::PhaseGraph: what a captured encode phase depends on

struct jpgenc_ctx {
    int device = 0;
    jpgenc::TablePool* pool = nullptr;    // host worker threads that build the four Huffman tables side by side
    jpgenc::HostPool* host_pool = nullptr;   // parallel table builds of a batch of frames
    bool owns_host_pool = false;             // pipeline lanes share their parent context's pool
    bool parallel_tables = true;          // false inside a batch: there the frames run in parallel instead
    std::vector<jpgenc_ctx*> lanes;       // further pipeline lanes of the batched-frame calls (contexts on the same device with their own
                                          // stream and buffers): while one lane's pass waits for its Huffman tables on the host, the
                                          // other lanes' kernels run
    cudaStream_t stream = nullptr;
    cudaStream_t copy_stream = nullptr;   // host-to-device copies of jpgenc_encode_rgb, overlapped with K1 band by band
    cudaEvent_t ev_band[16] = {};
    cudaEvent_t ev_a = nullptr, ev_b = nullptr, ev_t0 = nullptr, ev_t1 = nullptr, ev_u0 = nullptr, ev_u1 = nullptr, ev_k0 = nullptr, ev_k1 = nullptr;
    // K3/K4 of one image: the time of encode N is read while K2 of encode N + 1 runs (or by jpgenc_get_stats)
    cudaEvent_t ev_e0 = nullptr, ev_e1 = nullptr;
    bool ent_pending = false, stats_pending = false, last_whole = false;
    // Event records between the kernels of an image (jpgenc_set_stage_timing): 0 none -- inside the replayed graphs every
    // record is a node of its own, ~3 us each, 22 us per image with all eight --, 1 around the K1 fast kernel alone (the
    // roofline kernel), 2 around every stage.  *_timed: the level the events of the encode in flight were recorded at.
    int stage_timing = 0, fwd_timed = 0, stats_timed = 0, ent_timed = 0;
    uint32_t k4_grid_hint = 0;            // single image: the grid K4a / K4 are captured with (run_pipeline)
    float last_k1 = 0, last_fwd = 0, last_st = 0;
    std::string error;
    int sm_count = 148;
    uint64_t launches = 0;
    bool capturing = false;               // the stream is being captured into a graph (run_phase): events are recorded as external event nodes
    uint64_t alloc_gen = 0;               // bumped whenever a buffer of the context is (re)allocated or a parameter changes: captured graphs are stale then
    // whole-image encodes of pixels that stay bound: the two GPU phases (K1 .. K2 + publish; tables upload .. K4 + publish) as
    // CUDA graphs, captured when the same configuration is encoded a second time
    struct PhaseGraph {
        cudaGraphExec_t exec = nullptr;
        uint64_t key[kGraphKeyWords] = {};
        uint64_t seen[kGraphKeyWords] = {};   // key of the previous encode (a graph is captured when it repeats)
        uint32_t launches = 0;                // kernels per replay
        uint32_t publishes = 0;               // mailbox announcements per replay
    } graph_a, graph_b;

    // parameters
    uint8_t qy[64], qc[64];
    double dct_a[5], dct_s[8];

    // image state
    uint32_t nframes = 1;                 // > 1: a batch of equally sized frames goes through every kernel at once
    const uint8_t** d_frame_ptrs = nullptr;   // [nframes] device pointers of the frames (batches only)
    size_t frame_ptrs_cap = 0;
    bool frames_aligned = false;          // every frame pointer is 16-byte aligned (bulk-copy path of K1)
    jpgenc::MixedPass mixed;              // on: the frames bound are images of individual sizes, described by d_geom
    jpgenc::FrameGeom* d_geom = nullptr;  // [nframes + 1]
    size_t geom_cap = 0;
    jpgenc::PixelSource src;              // the single image bound (set whole by every bind; plane 0 is also a batch's first frame)
    uint8_t* d_rgb_owned = nullptr;
    size_t rgb_cap = 0;
    uint32_t real_w = 0, real_h = 0, maxval = 255, mcu_w = 0, mcu_h = 0;
    bool have_pixels = false, have_coef = false, have_scan = false, forward_pending = false, upload_pending = false;

    int16_t* d_coef = nullptr;
    size_t coef_cap = 0;
    uint32_t* d_refine_list = nullptr;
    size_t refine_cap = 0;
    uint32_t* d_counters = nullptr;       // kCounterWords words, see kCnt* below
    uint8_t* d_stats = nullptr;           // per frame: hist u32[4][256] + first-occurrence keys u64[4][256]; then a copy of the refine counter
    size_t stats_cap = 0;
    uint8_t* d_meta = nullptr;            // PassMeta block of the frames bound to the context (lives behind d_tables, same allocation)
    uint32_t entropy_runs = 0;            // K3/K4 passes over the current symbol items (reset by K2)
    bool file_mode = false;               // K4 writes complete files (header + scan + EOI per frame) instead of bare scans
    uint8_t* d_hdr_prefix = nullptr;      // SOI .. SOF0 of the frames of a batch (identical for all of them)
    uint32_t hdr_prefix_len = 0;
    uint64_t raw_limit = 0, out_limit = 0;   // what finalize_tables_kernel may use of d_raw / d_scan
    uint64_t batch_raw_per_frame = 0;     // batched calls: raw-scan bytes reserved per frame (1.5 x the largest seen so far; 0 = nothing seen yet)
    uint32_t batch_geom_w = 0, batch_geom_h = 0;   // ... the frame size that figure was learnt on (kept across calls of one size)
    cudaEvent_t ev_done = nullptr;        // batched calls: end of the slot's current pass
    cudaEvent_t ev_k4 = nullptr;          // ... its K4 is through (the next pass's K3 waits for it: passes finish one after the other)
    cudaEvent_t ev_fwd = nullptr;         // ... its K1/refinement are through (a call of two passes: the next pass's K1 waits for it)
    cudaEvent_t ev_copied = nullptr;      // ... its files have left d_scan (recorded on out_stream)
    cudaStream_t out_stream = nullptr;    // device-to-host copies of finished passes, beside the slot's kernels
    bool copy_pending = false;
    uint8_t hdr_prefix_host[256] = {};    // what d_hdr_prefix holds
    uint32_t* d_items = nullptr;          // K2's symbol stream (blockwalk.cuh), consumed by K3
    size_t items_cap = 0;
    uint32_t* d_tile_cnt = nullptr;             // per K2 tile: number of items in its slab
    size_t tile_cnt_cap = 0;
    uint32_t* d_range_bits = nullptr;           // per K2 tile: bits its items encode to (K3a)
    size_t range_bits_cap = 0;
    unsigned long long* d_range_base = nullptr; // bits per group of 8 tiles, then per 256 groups (K3a); K3b derives offsets from them
    size_t range_base_cap = 0;
    bool have_items = false;
    uint32_t k2_tiles_done = 0;           // K2 tiles already processed behind the bands of an upload (jpgenc_encode_rgb)
    std::vector<uint32_t> host_hist;      // K2's histograms as last read back, [nframes][4][256]
    std::vector<uint64_t> frame_bits;     // per frame: scan bits the statistics predict (checked against K3's count)
    bool k2_configured = false;
    // launch_forward_rows(first) clears K1's counters AND what K2 / K3a accumulate into in one kernel; launch_symbol_stats(first)
    // then skips its own clears -- valid while no buffer was reallocated and the frame count is the same
    bool stats_clear_valid = false;
    uint64_t stats_clear_gen = 0;
    uint32_t stats_clear_frames = 0;
    void* d_tab_scratch = nullptr;        // device-side table build (tables_device.cu): work space, one slab per table
    size_t tab_scratch_cap = 0;
    jpgenc_huff_table* d_built_tables = nullptr;   // ... its results [4 * nframes], and one status word per table behind them
    size_t built_tables_cap = 0;
    jpgenc::DeviceTables* d_tables = nullptr;   // [nframes]
    size_t tables_cap = 0;
    unsigned long long* d_lookback = nullptr;  // one look-back word per K4 tile
    size_t lookback_cap = 0;
    uint32_t* d_raw = nullptr;            // un-stuffed scan, 32-bit words, bytes in stream order
    size_t raw_cap = 0;
    uint8_t* d_scan = nullptr;            // K4's output: the stuffed scan, or (file_mode) the complete files of a pass back to back
    size_t scan_cap = 0;
    void* d_flush = nullptr;              // L2 eviction scratch
    size_t flush_bytes = 0;
    void* h_file_pinned = nullptr;        // two band-sized pinned buffers for streamed inputs (jpgenc_encode_ppm_file)
    size_t file_pinned_bytes = 0;
    // mailbox: mapped pinned memory the kernels of ONE image write their results into (the host polls it instead of
    // synchronising the stream); layout: kMail* below
    unsigned long long* h_mailbox = nullptr;   // host view
    unsigned long long* d_mailbox = nullptr;   // device view of the same memory
    uint32_t stat_count[4][256];          // K2's statistics of the current image as last received
    uint64_t stat_first[4][256];
    uint32_t mailbox_seq = 0;             // announced by K2 / K4 of the current encode
    void* h_pinned = nullptr;             // small pinned staging (stats, totals)
    size_t pinned_bytes = 0;

    jpgenc_stats stats{};
    jpgenc_huff_table last_tables[4];     // tables of the last whole-image run (for jpgenc_assemble_last)
    bool have_tables = false;
};

// event on the context's stream; inside a stream capture it becomes an event-record NODE of the graph (a plain record there
// only marks a dependency and leaves an event that cannot be waited for or timed)
inline cudaError_t jpgenc_record(jpgenc_ctx* c, cudaEvent_t ev) {
    return cudaEventRecordWithFlags(ev, c->stream, c->capturing ? cudaEventRecordExternal : cudaEventRecordDefault);
}

// an event of the per-stage timing: recorded only when stage timing is on at `level` or above
inline cudaError_t stage_record(jpgenc_ctx* c, cudaEvent_t ev, int level) {
    return c->stage_timing >= level ? jpgenc_record(c, ev) : cudaSuccess;
}

#define JPGENC_CUDA(ctx, expr)                                                                       \
    do {                                                                                             \
        cudaError_t e__ = (expr);                                                                    \
        if (e__ != cudaSuccess) {                                                                    \
            (ctx)->error = std::string(#expr) + ": " + cudaGetErrorString(e__);                      \
            return JPGENC_ERR_CUDA;                                                                  \
        }                                                                                            \
    } while (0)

// No exception crosses the C boundary (include/jpgenc_b200.h): every entry point that takes a context is a function-try-block
// closed by this.  What can arrive here is std::bad_alloc / std::length_error from a host container.
#define JPGENC_CATCH(ctx)                                                                            \
    catch (const std::exception& ex__) {                                                             \
        if (ctx) (ctx)->error = std::string("host exception: ") + ex__.what();                      \
        return JPGENC_ERR_NOMEM;                                                                     \
    } catch (...) {                                                                                  \
        if (ctx) (ctx)->error = "host exception";                                                   \
        return JPGENC_ERR_NOMEM;                                                                     \
    }

// launchers implemented in the kernel translation units
namespace jpgenc {
// words of jpgenc_ctx::d_counters
constexpr int kCntRefine = 0;      // entries in the refinement list (K1)
constexpr int kCntRefined = 3;     // list entries already refined (band-wise encodes)
constexpr int kCntFinalize = 4;    // finalize_tables_kernel's CTA ticket (resets itself)
constexpr int kCntK3Redo = 6;     // chunks K3b packed the slow way (zeroed by K3a; read by tests through jpgenc_debug_counter)
constexpr int kCntSeq = 5;         // mailbox sequence number (mailbox_publish_kernel increments it; never cleared)
constexpr int kCounterWords = 16;
// The host mailbox (jpgenc_ctx::h_mailbox, mapped pinned memory) as 64-bit words.  Every word carries its own validity: value
// (42 bits) | tag << 42, tag = mail_tag(sequence number of the publishing kernel) != 0 -- an aligned 8-byte store arrives
// whole, so the host needs no flag behind the data and the kernel no system-wide fence in front of one; the host zeroes what
// it has consumed, so a tag is never met again.
//   [kMailStatsHead]           n present symbols (11 bits) | K1's refinement counter << 11
//   [kMailStatsHead + 1 + 2k]  record k: count (32 bits) | (table * 256 + symbol) << 32
//   [kMailStatsHead + 2 + 2k]            first-occurrence key
//   [kMailTotals], [+1]        scan bits, stuffed FF bytes (K4)
constexpr int kMailStatsHead = 0;
constexpr int kMailTotals = 2064;
constexpr int kMailWords64 = 2080;
constexpr int kMailTagShift = 42;
__host__ __device__ inline unsigned long long mail_tag(uint32_t seq) { return static_cast<unsigned long long>(seq % 0x1FFFFFu + 1u); }
__host__ __device__ inline unsigned long long mail_word(unsigned long long value, uint32_t seq) { return value | (mail_tag(seq) << kMailTagShift); }
int launch_forward(jpgenc_ctx* c);
int launch_forward_rows(jpgenc_ctx* c, uint32_t y0, uint32_t rows, bool first, bool last);
// K1 + exact refinement over a pass of images of individual sizes (c->mixed, c->d_geom)
int launch_forward_mixed(jpgenc_ctx* c);
int launch_dct_quant_blocks(jpgenc_ctx* c, const float* in, int16_t* out, uint64_t nblocks, const uint8_t q[64],
                            uint64_t* refined);
int launch_planes_to_mcu(jpgenc_ctx* c, const int32_t* d_qy, const int32_t* d_qcb, const int32_t* d_qcr);
int launch_refine_pending(jpgenc_ctx* c);
int launch_planes_exact(jpgenc_ctx* c, const double* d_planes, bool ycbcr);
// K2 over the tiles [tile0, tile0 + ntiles) of the bound image(s); `first` also clears the statistics
int launch_symbol_stats(jpgenc_ctx* c, uint32_t tile0, uint32_t ntiles, bool first);
// K1's counters, the statistics of all frames bound and K3a's sums in one launch (false: the statistics' buffers do not exist yet)
bool launch_encode_clear(jpgenc_ctx* c);
int launch_entropy(jpgenc_ctx* c, uint32_t k4_grid);
int launch_publish_stats(jpgenc_ctx* c);
// batches: built tables + K2's histograms -> DeviceTables and the PassMeta block, all on the device
int launch_finalize_tables(jpgenc_ctx* c);
constexpr uint32_t kK4Threads = 256;
constexpr uint32_t kK4TileBytes = kK4Threads * 16;   // input bytes per K4 tile: 16 per thread (entropy.cu)
size_t table_scratch_bytes();
int build_table_arrays_host(const uint32_t count[256], const uint64_t first_pos[256], jpgenc_huff_table* out);
int launch_build_tables(jpgenc_ctx* c, const uint8_t* d_stats, uint32_t stats_stride, uint32_t ntables, void* d_scratch,
                        jpgenc_huff_table* d_out, uint32_t* d_status);
int launch_synth_rgb(jpgenc_ctx* c, uint8_t* d, uint32_t w, uint32_t h, uint32_t seed);
int launch_synth_blocks(jpgenc_ctx* c, float* d, uint64_t nblocks);
int launch_flush(jpgenc_ctx* c);
void fill_quant_consts(const uint8_t q[64], const double s[8], QuantConsts* out, double input_err);
void default_dct_constants(double a[5], double s[8]);
}  // namespace jpgenc
