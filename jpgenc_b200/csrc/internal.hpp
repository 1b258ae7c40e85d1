// Helpers shared by the translation units of the C-ABI layer (capi.cu: context, stage calls, one image; pipeline.cu:
// batches of frames).  Not part of the boundary: include/jpgenc_b200.h is.
#pragma once

#include "common.cuh"

namespace jpgenc { namespace detail {

constexpr size_t kStatsBytes = 4096 + 8192;   // per frame: symbol histogram u32[4][256] + first-occurrence keys u64[4][256] (stats.cu)

int fail(jpgenc_ctx* c, int code, const char* what);

// device buffer of at least need_bytes, grown on demand.  `headroom`: for buffers whose size follows the data (scan sizes
// differ from pass to pass): a reallocation frees device memory, which synchronises the whole device, so it should happen
// a few times, not whenever a pass is slightly larger than the last one
int ensure_bytes(jpgenc_ctx* c, void** ptr, size_t* cap, size_t need_bytes, bool headroom);
template <class T>
int ensure(jpgenc_ctx* c, T** ptr, size_t* cap, size_t need_bytes, bool headroom = false) {
    void* p = *ptr;
    const int rc = ensure_bytes(c, &p, cap, need_bytes, headroom);
    *ptr = static_cast<T*>(p);
    return rc;
}

int set_geometry(jpgenc_ctx* c, uint32_t w, uint32_t h, uint32_t maxval);
// A caller's image: a known format, its planes (NV12 / NV16: v must be NULL; YUYV / UYVY: u and v NULL, pitch2 0), sides 1..65535
// and pitches that hold a row (0 -> the row size, filled in; planar RGB: pitch2 = pitch); JPGENC_ERR_ARG otherwise
int check_source(jpgenc_ctx* c, PixelSource* s, uint32_t w, uint32_t h);
// every colour sample of a host source is <= maxval (maxval 0 or 255: true): a 4th byte and the bytes between rows are not read;
// planar RGB: all three planes; YUV frames have no maxval
bool source_within_maxval(const PixelSource& s, uint32_t w, uint32_t h, uint32_t maxval);
// the sources of the C entry points (a format code they do not take becomes -1, which check_source refuses)
PixelSource image_source(const void* px, uint32_t pitch, int format);
PixelSource planar_source(const void* r, const void* g, const void* b, uint32_t pitch);
PixelSource yuv_source(const void* y, const void* u, const void* v, uint32_t y_pitch, uint32_t c_pitch, int layout);
// the layouts the jpgenc_*_yuv420 calls take
inline bool is_yuv420_layout(int layout) { return layout == JPGENC_YUV_I420 || layout == JPGENC_YUV_NV12; }

// One plane of a checked host source as it is uploaded: `rows` host rows of `row` bytes, `pitch` bytes apart (vsub 1: the chroma
// planes of YUV 4:2:0, half the image's rows rounded up), staged as tight rows at `dev_off` of the device copy; YUV planes start
// on 256 bytes
struct StagedPlane {
    const uint8_t* host;
    size_t pitch, row, rows, dev_off;
    uint32_t vsub;
};
uint32_t staged_planes(const PixelSource& s, uint32_t w, uint32_t h, StagedPlane pl[3]);   // the number of planes
size_t staged_bytes(const StagedPlane* pl, uint32_t np);
// the three planes of planar RGB lie equally spaced in host memory with tight rows: their spacing (one strided copy moves them
// all); 0 otherwise
size_t planes_gap(const StagedPlane* pl, uint32_t np);
int ensure_pinned(jpgenc_ctx* c, size_t bytes);                 // c->h_pinned, grown on demand
int ensure_coef(jpgenc_ctx* c);                                  // coefficients + refinement list of the bound frames
int ensure_stats_buffers(jpgenc_ctx* c);                         // K2's outputs for the bound frames (+ pinned staging)
int ensure_entropy_buffers(jpgenc_ctx* c, uint64_t raw_total, uint64_t out_total, uint64_t k4_tiles);
void ensure_host_pool(jpgenc_ctx* c);
void leave_batch_state(jpgenc_ctx* c);
int flush_entropy_time(jpgenc_ctx* c);
int poll_mailbox(jpgenc_ctx* c, int word, unsigned long long* value);

// pinned staging of a context: [statistics F * kStatsBytes + 16][device tables F * 8 KB][PassMeta block (common.cuh)]
size_t stage_tables_off(uint32_t F);
size_t stage_meta_off(uint32_t F);
size_t stage_bytes(uint32_t F);

uint32_t env_u32(const char* name, uint32_t dflt);
double now_us();

}}  // namespace jpgenc::detail
