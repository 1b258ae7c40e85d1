// C-ABI of the encode path (include/jpgenc_b200.h): context, buffers, stage calls, whole-image driver.
#include <algorithm>
#include <atomic>
#include <chrono>
#include <condition_variable>
#include <deque>
#include <memory>
#include <functional>
#include <mutex>
#include <thread>
#include <cmath>
#include <cstdlib>
#include <cstring>
#include <vector>

#include <sched.h>
#include <unistd.h>
#include <cctype>

#include "common.cuh"
#include "../host/ppm_reader.hpp"

#include "host_pools.hpp"

#include "internal.hpp"

namespace jpgenc {
int launch_exact_all(jpgenc_ctx* c);
}

using namespace jpgenc;
using namespace jpgenc::detail;

namespace {
thread_local std::string g_create_error;
}

namespace jpgenc { namespace detail {

const uint8_t kAnnexKLuma[64] = {16, 11, 10, 16, 24,  40,  51,  61,  12, 12, 14, 19, 26,  58,  60,  55,
                                 14, 13, 16, 24, 40,  57,  69,  56,  14, 17, 22, 29, 51,  87,  80,  62,
                                 18, 22, 37, 56, 68,  109, 103, 77,  24, 35, 55, 64, 81,  104, 113, 92,
                                 49, 64, 78, 87, 103, 121, 120, 101, 72, 92, 95, 98, 112, 100, 103, 99};   // src/Image.cpp:850-859
const uint8_t kAnnexKChroma[64] = {17, 18, 24, 47, 99, 99, 99, 99, 18, 21, 26, 66, 99, 99, 99, 99,
                                   24, 26, 56, 99, 99, 99, 99, 99, 47, 66, 99, 99, 99, 99, 99, 99,
                                   99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99,
                                   99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99, 99};        // src/Image.cpp:860-869

int fail(jpgenc_ctx* c, int code, const char* what) {
    c->error = what;
    return code;
}

int ensure_bytes(jpgenc_ctx* c, void** ptr, size_t* cap, size_t need_bytes, bool headroom) {
    if (*ptr && *cap >= need_bytes) return JPGENC_OK;
    if (headroom) need_bytes += need_bytes / 4 + 4096;
    if (*ptr) JPGENC_CUDA(c, cudaFree(*ptr));
    *ptr = nullptr; *cap = 0;
    void* p = nullptr;
    const size_t bytes = (need_bytes + 255) & ~static_cast<size_t>(255);
    JPGENC_CUDA(c, cudaMalloc(&p, bytes));
    *ptr = p;
    *cap = bytes;
    ++c->alloc_gen;
    return JPGENC_OK;
}

int set_geometry(jpgenc_ctx* c, uint32_t w, uint32_t h, uint32_t maxval) {
    if (w == 0 || h == 0 || maxval == 0 || maxval > 255) return fail(c, JPGENC_ERR_ARG, "width/height/maxval out of range");
    c->real_w = w; c->real_h = h; c->maxval = maxval;
    c->mcu_w = (w + 15) / 16; c->mcu_h = (h + 15) / 16;        // src/Image.cpp:479-489
    c->src = PixelSource{};                                      // tight RGB until a bind sets its source
    c->src.pitch = w * 3;
    c->nframes = 1;
    c->mixed.on = false;
    c->have_pixels = false;                                      // whoever changes the geometry binds its pixels afterwards
    c->have_coef = c->have_scan = c->have_items = false; c->k2_tiles_done = 0;
    return JPGENC_OK;
}

int check_source(jpgenc_ctx* c, PixelSource* s, uint32_t w, uint32_t h) {
    const int f = s->format;
    if ((f < JPGENC_PIXEL_RGB || f > JPGENC_PIXEL_BGRA) && f != JPGENC_PIXEL_GRAY && f != kPixelPlanar && !is_yuv(f))
        return fail(c, JPGENC_ERR_ARG, "unknown pixel format");
    const bool semi = f == kPixelNV12 || f == kPixelNV16;
    for (uint32_t k = 0; k < source_planes(f); ++k)
        if (!s->plane[k] && !(semi && k == 2)) return fail(c, JPGENC_ERR_ARG, "null plane pointer");
    if (semi && s->plane[2]) return fail(c, JPGENC_ERR_ARG, "NV12 / NV16 take their UV plane as u; v must be NULL");
    if (is_packed_yuv(f) && (s->plane[1] || s->plane[2] || s->pitch2))
        return fail(c, JPGENC_ERR_ARG, "YUYV / UYVY take one packed plane as y; u and v must be NULL and c_pitch 0");
    if (w == 0 || h == 0 || w > 65535 || h > 65535) return fail(c, JPGENC_ERR_ARG, "image side out of range (1..65535)");
    const uint32_t row = row_bytes(f, w);
    if (s->pitch == 0) s->pitch = row;
    if (s->pitch < row) return fail(c, JPGENC_ERR_ARG, "row pitch below the row size");
    if (f == kPixelPlanar) s->pitch2 = s->pitch;
    if (is_yuv(f) && !is_packed_yuv(f)) {
        const uint32_t crow = chroma_row_bytes(f, w);
        if (s->pitch2 == 0) s->pitch2 = crow;
        if (s->pitch2 < crow) return fail(c, JPGENC_ERR_ARG, "chroma pitch below the chroma row size");
    }
    return JPGENC_OK;
}

bool source_within_maxval(const PixelSource& s, uint32_t w, uint32_t h, uint32_t maxval) {
    if (maxval == 0 || maxval >= 255 || is_yuv(s.format)) return true;
    for (uint32_t k = 0; k < source_planes(s.format); ++k)
        if (!samples_within_maxval(s.plane[k], w, h, s.pitch, pixel_bytes(s.format), maxval)) return false;
    return true;
}

PixelSource yuv_source(const void* y, const void* u, const void* v, uint32_t y_pitch, uint32_t c_pitch, int layout) {
    static_assert(kPixelI420 + JPGENC_YUV_UYVY == kPixelUYVY && kPixelI420 + JPGENC_YUV_NV16 == kPixelNV16, "JPGENC_YUV_* follow the formats");
    PixelSource s;
    s.format = layout >= JPGENC_YUV_I420 && layout <= JPGENC_YUV_UYVY ? kPixelI420 + layout : -1;
    s.pitch = y_pitch;
    s.pitch2 = c_pitch;
    s.plane[0] = static_cast<const uint8_t*>(y); s.plane[1] = static_cast<const uint8_t*>(u); s.plane[2] = static_cast<const uint8_t*>(v);
    return s;
}

PixelSource planar_source(const void* r, const void* g, const void* b, uint32_t pitch) {
    PixelSource s;
    s.format = kPixelPlanar;
    s.pitch = pitch;
    s.plane[0] = static_cast<const uint8_t*>(r); s.plane[1] = static_cast<const uint8_t*>(g); s.plane[2] = static_cast<const uint8_t*>(b);
    return s;
}

PixelSource image_source(const void* px, uint32_t pitch, int format) {
    PixelSource s;
    s.format = (format >= JPGENC_PIXEL_RGB && format <= JPGENC_PIXEL_BGRA) || format == JPGENC_PIXEL_GRAY ? format : -1;   // public codes only
    s.pitch = pitch;
    s.plane[0] = static_cast<const uint8_t*>(px);
    return s;
}

uint32_t staged_planes(const PixelSource& s, uint32_t w, uint32_t h, StagedPlane pl[3]) {
    const bool yuv = is_yuv(s.format);
    const uint32_t np = s.format == kPixelNV12 || s.format == kPixelNV16 ? 2u : source_planes(s.format);
    size_t off = 0;
    for (uint32_t k = 0; k < np; ++k) {
        const bool chroma = yuv && k > 0;
        pl[k].host = s.plane[k];
        pl[k].pitch = chroma ? s.pitch2 : s.pitch;
        pl[k].row = chroma ? chroma_row_bytes(s.format, w) : row_bytes(s.format, w);
        pl[k].vsub = chroma ? chroma_vsub(s.format) : 0u;
        pl[k].rows = (h + pl[k].vsub) >> pl[k].vsub;
        pl[k].dev_off = off;
        off += pl[k].row * pl[k].rows;
        if (yuv) off = (off + 255) & ~static_cast<size_t>(255);
    }
    return np;
}

size_t staged_bytes(const StagedPlane* pl, uint32_t np) { return pl[np - 1].dev_off + pl[np - 1].row * pl[np - 1].rows; }

size_t planes_gap(const StagedPlane* pl, uint32_t np) {
    // (planes of one row size, tight rows, and device planes as far apart as a plane is long: planar RGB and tight I444 planes)
    if (np != 3 || pl[1].vsub || pl[0].pitch != pl[0].row || pl[1].row != pl[0].row || pl[1].pitch != pl[1].row ||
        pl[1].dev_off != pl[0].row * pl[0].rows)
        return 0;
    const uintptr_t gap = reinterpret_cast<uintptr_t>(pl[1].host) - reinterpret_cast<uintptr_t>(pl[0].host);
    const bool equal = reinterpret_cast<uintptr_t>(pl[2].host) - reinterpret_cast<uintptr_t>(pl[1].host) == gap;
    return equal && gap >= pl[0].row * pl[0].rows && gap <= (uintptr_t{1} << 48) ? gap : 0;
}

// pinned host staging, grown on demand
int ensure_pinned(jpgenc_ctx* c, size_t bytes) {
    if (c->pinned_bytes >= bytes) return JPGENC_OK;
    if (c->h_pinned) JPGENC_CUDA(c, cudaFreeHost(c->h_pinned));
    c->h_pinned = nullptr; c->pinned_bytes = 0;
    JPGENC_CUDA(c, cudaMallocHost(&c->h_pinned, bytes));
    c->pinned_bytes = bytes;
    ++c->alloc_gen;
    return JPGENC_OK;
}

// after the stream has been synchronised past K1: event times and the refine counter
int refresh_forward_stats(jpgenc_ctx* c) {
    if (!c->forward_pending) return JPGENC_OK;
    c->stats.ms_forward = c->stats.ms_k1 = 0;
    if (c->fwd_timed >= 2) JPGENC_CUDA(c, cudaEventElapsedTime(&c->stats.ms_forward, c->ev_a, c->ev_b));
    if (c->fwd_timed >= 1) JPGENC_CUDA(c, cudaEventElapsedTime(&c->stats.ms_k1, c->ev_k0, c->ev_k1));
    c->forward_pending = false;
    return JPGENC_OK;
}

int ensure_coef(jpgenc_ctx* c) {
    const size_t nblocks = c->mixed.on ? c->mixed.blocks : static_cast<size_t>(c->mcu_w) * c->mcu_h * kBlocksPerMcu * c->nframes;
    if (nblocks * 64 > 0xFFFFFFFFull * 16) return fail(c, JPGENC_ERR_ARG, "image (or batch) too large");
    int rc = ensure(c, &c->d_coef, &c->coef_cap, nblocks * kBlockBytes);
    if (rc) return rc;
    size_t cap_bytes = c->refine_cap * sizeof(uint32_t);
    rc = ensure(c, &c->d_refine_list, &cap_bytes, nblocks * sizeof(uint32_t));
    c->refine_cap = cap_bytes / sizeof(uint32_t);
    return rc;
}

double now_us() {
    return std::chrono::duration<double, std::micro>(std::chrono::steady_clock::now().time_since_epoch()).count();
}

// device buffers of K2 / K3 for the frames bound to the context
int ensure_stats_buffers(jpgenc_ctx* c) {
    const uint32_t F = c->nframes;
    const size_t nblocks = static_cast<size_t>(c->mcu_w) * c->mcu_h * kBlocksPerMcu, tiles = (nblocks + 383) / 384;
    // images of individual sizes: the pass's own tiles, groups and super-groups (c->mixed)
    const size_t all_tiles = c->mixed.on ? c->mixed.tiles : F * tiles;
    const size_t range_words = c->mixed.on ? c->mixed.groups + c->mixed.supers : F * (tiles * 4 / 8 + tiles * 4 / 2048 + 4);
    int rc;
    // one fixed slab of item slots per tile, sized for the worst case (every coefficient non-zero); typical images
    // touch a few percent of it
    if ((rc = ensure(c, &c->d_items, &c->items_cap, all_tiles * 384 * 64 * sizeof(uint32_t)))) return rc;
    if ((rc = ensure(c, &c->d_tile_cnt, &c->tile_cnt_cap, all_tiles * sizeof(uint32_t)))) return rc;
    // K3 may cut a tile into four ranges (small images, launch_entropy): sized for that
    if ((rc = ensure(c, &c->d_range_bits, &c->range_bits_cap, all_tiles * 4 * sizeof(uint32_t)))) return rc;
    if ((rc = ensure(c, &c->d_range_base, &c->range_base_cap, range_words * sizeof(unsigned long long)))) return rc;
    if ((rc = ensure(c, &c->d_stats, &c->stats_cap, F * kStatsBytes + 16))) return rc;
    return ensure_pinned(c, stage_bytes(F));
}

// device buffers of K3 / K4 for `raw_total` bytes of raw scan, `out_total` bytes of output and `k4_tiles` K4 tiles
int ensure_entropy_buffers(jpgenc_ctx* c, uint64_t raw_total, uint64_t out_total, uint64_t k4_tiles) {
    const uint32_t F = c->nframes;
    int rc;
    if ((rc = ensure(c, &c->d_raw, &c->raw_cap, raw_total, true))) return rc;
    if ((rc = ensure(c, &c->d_scan, &c->scan_cap, out_total + 64, true))) return rc;
    // tables and frame geometry share one allocation, in the order of the staging buffer: one copy brings both
    if ((rc = ensure(c, &c->d_tables, &c->tables_cap, F * sizeof(DeviceTables) + pass_meta_bytes(F)))) return rc;
    c->d_meta = reinterpret_cast<uint8_t*>(c->d_tables) + F * sizeof(DeviceTables);
    size_t lb_bytes = c->lookback_cap;
    if ((rc = ensure(c, &c->d_lookback, &lb_bytes, (k4_tiles + 8) * sizeof(unsigned long long), true))) return rc;
    c->lookback_cap = lb_bytes;
    return JPGENC_OK;
}

uint32_t env_u32(const char* name, uint32_t dflt) {
    const char* v = std::getenv(name);
    return v && *v ? static_cast<uint32_t>(std::strtoul(v, nullptr, 10)) : dflt;
}

// the context's pool of host threads (HostPool): this process's share of the host -- the cores divided by the visible GPUs
// (one process per GPU is the deployment this library is written for); JPGENC_HOST_THREADS overrides
void ensure_host_pool(jpgenc_ctx* c) {
    if (c->host_pool) return;
    int ndev = 1;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev < 1) ndev = 1;
    const unsigned share = std::max(2u, std::thread::hardware_concurrency() / static_cast<unsigned>(ndev));
    const unsigned workers = std::min(15u, std::max(2u, env_u32("JPGENC_HOST_THREADS", share)) - 1);   // the caller works too
    c->host_pool = new HostPool(workers);
    c->owns_host_pool = true;
}

// threads beside the caller that build the four tables of a single image (TablePool): ONE -- it takes the two DC tables and
// chroma AC while the caller builds luma AC, which is about the same work (a photograph: 3 + 3 + 3 us against 10; noise: both AC
// tables are large and the same holds).  Measured against a thread per table (3840x2160 / 16384^2 / 2048^2 noise, all 16 cores
// and pinned to 4): 0.0887 / 0.6787 / 0.1529 ms against 0.0913 / 0.6806 / 0.1540 -- fewer threads to wake and to wait for, and
// a process that shares its host with seven other ranks keeps two of its four cores.
constexpr int kTableWorkers = 1;

// pinned staging: [statistics F * kStatsBytes + 16][device tables F * 8 KB][PassMeta block (common.cuh)]
size_t stage_tables_off(uint32_t F) { return ((F * kStatsBytes + 16 + 255) / 256) * 256; }
size_t stage_meta_off(uint32_t F) { return stage_tables_off(F) + F * sizeof(DeviceTables); }
size_t stage_bytes(uint32_t F) { return stage_meta_off(F) + pass_meta_bytes(F) + 64; }


// K3/K4 time of the last single-image encode (its events complete while the host is already elsewhere): read it now and,
// when that encode went through all four stages, add its stage times to the running sums
int flush_entropy_time(jpgenc_ctx* c) {
    if (!c->ent_pending) return JPGENC_OK;
    c->stats.ms_entropy = 0;
    if (c->ent_timed >= 2) {
        JPGENC_CUDA(c, cudaEventSynchronize(c->ev_e1));
        JPGENC_CUDA(c, cudaEventElapsedTime(&c->stats.ms_entropy, c->ev_e0, c->ev_e1));
    }
    c->ent_pending = false;
    if (c->last_whole) {
        c->stats.sum_ms_k1 += c->last_k1; c->stats.sum_ms_forward += c->last_fwd;
        c->stats.sum_ms_stats += c->last_st; c->stats.sum_ms_entropy += c->stats.ms_entropy;
        c->stats.timed_encodes += 1;
        c->last_whole = false;
    }
    return JPGENC_OK;
}

// Waits until mailbox word `word` carries the tag of the current encode's publishing kernel and returns its value.  The word
// is written over PCIe into page-locked host memory: polling it costs a microsecond where a device-to-host copy plus
// cudaStreamSynchronize cost 20-30.  The stream is queried every now and then so that a failed launch is reported instead
// of waited for; long waits (the pixels of a large image still crossing PCIe) yield the core.
int poll_mailbox(jpgenc_ctx* c, int word, unsigned long long* value) {
    volatile unsigned long long* w = c->h_mailbox + word;
    const unsigned long long tag = mail_tag(c->mailbox_seq);
    const double t0 = now_us();
    unsigned long long v = 0;
    for (uint32_t spins = 1;; ++spins) {
        v = *w;
        if ((v >> kMailTagShift) == tag) break;
#if defined(__x86_64__)
        __builtin_ia32_pause();
#endif
        if ((spins & 0x3FFu) == 0) {
            const cudaError_t e = cudaStreamQuery(c->stream);
            if (e == cudaSuccess) {
                v = *w;
                if ((v >> kMailTagShift) == tag) break;
                return fail(c, JPGENC_ERR_CUDA, "the kernels finished without delivering their result");
            }
            if (e != cudaErrorNotReady) { c->error = std::string("kernel failed: ") + cudaGetErrorString(e); return JPGENC_ERR_CUDA; }
            if (now_us() - t0 > 2000.0) usleep(50);
        }
    }
    std::atomic_thread_fence(std::memory_order_acquire);
    *value = v & ((1ull << kMailTagShift) - 1);
    *w = 0;                                                          // consumed: this tag is never met again in this word
    return JPGENC_OK;
}

void leave_batch_state(jpgenc_ctx* c) {
    c->nframes = 1;                                                  // the context goes back to single-image state
    c->mixed.on = false;
    c->have_pixels = c->have_coef = c->have_scan = c->have_items = false; c->k2_tiles_done = 0;
    c->file_mode = false;
    c->host_hist.clear();
}

}}  // namespace jpgenc::detail

extern "C" {

int jpgenc_create(int device, jpgenc_ctx** out) {
    if (!out) return JPGENC_ERR_ARG;
    *out = nullptr;
    int ndev = 0;
    cudaError_t e = cudaGetDeviceCount(&ndev);
    if (e != cudaSuccess || ndev == 0) {
        g_create_error = std::string("no CUDA device (") + cudaGetErrorString(e) + "); this library has no CPU fallback";
        return JPGENC_ERR_NO_DEVICE;
    }
    if (device < 0 || device >= ndev) {
        g_create_error = "device index out of range";
        return JPGENC_ERR_ARG;
    }
    jpgenc_ctx* c = new jpgenc_ctx();
    c->device = device;
    auto bail = [&](const char* what, cudaError_t err) {
        g_create_error = std::string(what) + ": " + cudaGetErrorString(err);
        jpgenc_destroy(c);                                         // null-safe on every member: releases what exists so far
        return JPGENC_ERR_CUDA;
    };
    if ((e = cudaSetDevice(device)) != cudaSuccess) return bail("cudaSetDevice", e);
    cudaDeviceProp prop;
    if ((e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) return bail("cudaGetDeviceProperties", e);
    if (prop.major < 10) {
        g_create_error = "device is not sm_100 (Blackwell); the kernels are built for sm_100a only";
        jpgenc_destroy(c);
        return JPGENC_ERR_NO_DEVICE;
    }
    c->sm_count = prop.multiProcessorCount;
    if ((e = cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking)) != cudaSuccess) return bail("cudaStreamCreate", e);
    if ((e = cudaStreamCreateWithFlags(&c->copy_stream, cudaStreamNonBlocking)) != cudaSuccess) return bail("cudaStreamCreate", e);
    for (cudaEvent_t& ev : c->ev_band)
        if ((e = cudaEventCreateWithFlags(&ev, cudaEventDisableTiming)) != cudaSuccess) return bail("cudaEventCreate", e);
    for (cudaEvent_t* ev : {&c->ev_a, &c->ev_b, &c->ev_t0, &c->ev_t1, &c->ev_u0, &c->ev_u1, &c->ev_k0, &c->ev_k1})
        if ((e = cudaEventCreate(ev)) != cudaSuccess) return bail("cudaEventCreate", e);
    std::memcpy(c->qy, kAnnexKLuma, 64);
    std::memcpy(c->qc, kAnnexKChroma, 64);
    default_dct_constants(c->dct_a, c->dct_s);
    void* p = nullptr;
    if ((e = cudaMalloc(&p, kCounterWords * sizeof(uint32_t))) != cudaSuccess) return bail("cudaMalloc", e);
    c->d_counters = static_cast<uint32_t*>(p);
    if ((e = cudaMemset(p, 0, kCounterWords * sizeof(uint32_t))) != cudaSuccess) return bail("cudaMemset", e);
    c->pinned_bytes = 64 * 1024;
    if ((e = cudaMallocHost(&c->h_pinned, c->pinned_bytes)) != cudaSuccess) return bail("cudaMallocHost", e);
    for (cudaEvent_t* ev : {&c->ev_e0, &c->ev_e1})
        if ((e = cudaEventCreate(ev)) != cudaSuccess) return bail("cudaEventCreate", e);
    // the mailbox: page-locked host memory the kernels write into directly (results of one image, a few KB)
    if ((e = cudaHostAlloc(reinterpret_cast<void**>(&c->h_mailbox), kMailWords64 * sizeof(unsigned long long), cudaHostAllocMapped)) != cudaSuccess) return bail("cudaHostAlloc", e);
    std::memset(c->h_mailbox, 0, kMailWords64 * sizeof(unsigned long long));
    if ((e = cudaHostGetDevicePointer(reinterpret_cast<void**>(&c->d_mailbox), c->h_mailbox, 0)) != cudaSuccess) return bail("cudaHostGetDevicePointer", e);
    *out = c;
    return JPGENC_OK;
}

void jpgenc_destroy(jpgenc_ctx* c) {
    if (!c) return;
    cudaSetDevice(c->device);
    if (c->stream) cudaStreamSynchronize(c->stream);
    if (c->copy_stream) cudaStreamSynchronize(c->copy_stream);
    for (jpgenc_ctx* l : c->lanes) jpgenc_destroy(l);
    delete c->pool;
    if (c->owns_host_pool) delete c->host_pool;
    cudaFree(c->d_rgb_owned); cudaFree(c->d_coef); cudaFree(c->d_refine_list); cudaFree(c->d_counters);
    cudaFree(c->d_stats); cudaFree(c->d_tables);   /* d_meta lives in the same allocation */ cudaFree(c->d_frame_ptrs); cudaFree(c->d_geom); cudaFree(c->d_lookback); cudaFree(c->d_raw);
    cudaFree(c->d_scan); cudaFree(c->d_hdr_prefix); cudaFree(c->d_flush);
    cudaFree(c->d_tab_scratch); cudaFree(c->d_built_tables);
    cudaFree(c->d_items); cudaFree(c->d_tile_cnt); cudaFree(c->d_range_bits); cudaFree(c->d_range_base);
    if (c->h_pinned) cudaFreeHost(c->h_pinned);
    if (c->h_mailbox) cudaFreeHost(c->h_mailbox);
    if (c->ev_e0) cudaEventDestroy(c->ev_e0);
    if (c->ev_e1) cudaEventDestroy(c->ev_e1);
    if (c->graph_a.exec) cudaGraphExecDestroy(c->graph_a.exec);
    if (c->graph_b.exec) cudaGraphExecDestroy(c->graph_b.exec);
    if (c->h_file_pinned) cudaFreeHost(c->h_file_pinned);
    for (cudaEvent_t ev : {c->ev_a, c->ev_b, c->ev_t0, c->ev_t1, c->ev_u0, c->ev_u1, c->ev_k0, c->ev_k1}) if (ev) cudaEventDestroy(ev);
    for (cudaEvent_t ev : c->ev_band) if (ev) cudaEventDestroy(ev);
    if (c->ev_done) cudaEventDestroy(c->ev_done);
    if (c->ev_fwd) cudaEventDestroy(c->ev_fwd);
    if (c->ev_k4) cudaEventDestroy(c->ev_k4);
    if (c->ev_copied) cudaEventDestroy(c->ev_copied);
    if (c->out_stream) { cudaStreamSynchronize(c->out_stream); cudaStreamDestroy(c->out_stream); }
    if (c->copy_stream) cudaStreamDestroy(c->copy_stream);
    if (c->stream) cudaStreamDestroy(c->stream);
    delete c;
}

const char* jpgenc_last_error(const jpgenc_ctx* c) { return c ? c->error.c_str() : g_create_error.c_str(); }
void* jpgenc_stream(jpgenc_ctx* c) { return c ? static_cast<void*>(c->stream) : nullptr; }
uint64_t jpgenc_launch_count(const jpgenc_ctx* c) { return c ? c->launches : 0; }

int jpgenc_synchronize(jpgenc_ctx* c) try {
    if (!c) return JPGENC_ERR_ARG;
    JPGENC_CUDA(c, cudaStreamSynchronize(c->stream));
    return JPGENC_OK;
} JPGENC_CATCH(c)

int jpgenc_get_stats(jpgenc_ctx* c, jpgenc_stats* out) try {
    if (!c || !out) return JPGENC_ERR_ARG;
    const int rf = flush_entropy_time(c);
    if (rf) return rf;
    c->stats.real_w = c->real_w; c->stats.real_h = c->real_h; c->stats.mcu_w = c->mcu_w; c->stats.mcu_h = c->mcu_h;
    c->stats.n_blocks = static_cast<uint64_t>(c->mcu_w) * c->mcu_h * kBlocksPerMcu;
    *out = c->stats;
    return JPGENC_OK;
} JPGENC_CATCH(c)

int jpgenc_set_stage_timing(jpgenc_ctx* c, int level) try {
    if (!c || level < 0 || level > 2) return JPGENC_ERR_ARG;
    c->stage_timing = level;                                     // part of the graph keys (run_pipeline): the phases are captured again
    return JPGENC_OK;
} JPGENC_CATCH(c)

int jpgenc_set_qtables(jpgenc_ctx* c, const uint8_t qy[64], const uint8_t qc[64]) try {
    if (!c || !qy || !qc) return JPGENC_ERR_ARG;
    for (int i = 0; i < 64; ++i)
        if (qy[i] == 0 || qc[i] == 0) return fail(c, JPGENC_ERR_ARG, "quantiser entries must be >= 1");
    std::memcpy(c->qy, qy, 64);
    std::memcpy(c->qc, qc, 64);
    ++c->alloc_gen;
    return JPGENC_OK;
} JPGENC_CATCH(c)

int jpgenc_set_dct_constants(jpgenc_ctx* c, const double a[5], const double s[8]) try {
    if (!c || !a || !s) return JPGENC_ERR_ARG;
    std::memcpy(c->dct_a, a, sizeof c->dct_a);
    std::memcpy(c->dct_s, s, sizeof c->dct_s);
    ++c->alloc_gen;
    return JPGENC_OK;
} JPGENC_CATCH(c)

// binds device pixels: the source is checked, then replaces whatever was bound
static int bind_source(jpgenc_ctx* c, PixelSource src, uint32_t w, uint32_t h, uint32_t maxval) {
    int rc = check_source(c, &src, w, h);
    if (rc || (rc = set_geometry(c, w, h, maxval))) return rc;
    c->src = src;
    c->have_pixels = true;
    return JPGENC_OK;
}

int jpgenc_upload_rgb(jpgenc_ctx* c, const uint8_t* host_rgb, uint32_t w, uint32_t h, uint32_t maxval) try {
    if (!c || !host_rgb) return JPGENC_ERR_ARG;
    if (!source_within_maxval(image_source(host_rgb, w * 3, JPGENC_PIXEL_RGB), w, h, maxval)) return fail(c, JPGENC_ERR_FORMAT, "a sample exceeds maxval");
    JPGENC_CUDA(c, cudaSetDevice(c->device));
    int rc = set_geometry(c, w, h, maxval);
    if (rc) return rc;
    const size_t bytes = static_cast<size_t>(w) * h * 3;
    if ((rc = ensure(c, &c->d_rgb_owned, &c->rgb_cap, bytes + 16))) return rc;
    JPGENC_CUDA(c, jpgenc_record(c, c->ev_a));
    JPGENC_CUDA(c, cudaMemcpyAsync(c->d_rgb_owned, host_rgb, bytes, cudaMemcpyHostToDevice, c->stream));
    JPGENC_CUDA(c, jpgenc_record(c, c->ev_b));
    JPGENC_CUDA(c, cudaStreamSynchronize(c->stream));            // the caller may reuse host_rgb as soon as we return
    JPGENC_CUDA(c, cudaEventElapsedTime(&c->stats.ms_h2d, c->ev_a, c->ev_b));
    c->src.plane[0] = c->d_rgb_owned;
    c->have_pixels = true;
    return JPGENC_OK;
} JPGENC_CATCH(c)

int jpgenc_bind_device_rgb(jpgenc_ctx* c, const void* dev_rgb, uint32_t w, uint32_t h, uint32_t maxval) try {
    if (!c || !dev_rgb) return JPGENC_ERR_ARG;
    const int rc = set_geometry(c, w, h, maxval);
    if (rc) return rc;
    c->src.plane[0] = static_cast<const uint8_t*>(dev_rgb);
    c->have_pixels = true;
    return JPGENC_OK;
} JPGENC_CATCH(c)

int jpgenc_bind_device_image(jpgenc_ctx* c, const void* dev, uint32_t w, uint32_t h, uint32_t row_pitch, int format, uint32_t maxval) try {
    if (!c) return JPGENC_ERR_ARG;
    return bind_source(c, image_source(dev, row_pitch, format), w, h, maxval);
} JPGENC_CATCH(c)

int jpgenc_bind_device_planar(jpgenc_ctx* c, const void* r, const void* g, const void* b, uint32_t w, uint32_t h, uint32_t row_pitch,
                              uint32_t maxval) try {
    if (!c) return JPGENC_ERR_ARG;
    return bind_source(c, planar_source(r, g, b, row_pitch), w, h, maxval);
} JPGENC_CATCH(c)

int jpgenc_bind_device_yuv(jpgenc_ctx* c, const void* y, const void* u, const void* v, uint32_t w, uint32_t h, uint32_t y_pitch,
                           uint32_t c_pitch, int layout) try {
    if (!c) return JPGENC_ERR_ARG;
    return bind_source(c, yuv_source(y, u, v, y_pitch, c_pitch, layout), w, h, 255);
} JPGENC_CATCH(c)

int jpgenc_bind_device_yuv420(jpgenc_ctx* c, const void* y, const void* u, const void* v, uint32_t w, uint32_t h, uint32_t y_pitch,
                              uint32_t c_pitch, int layout) try {
    if (!c) return JPGENC_ERR_ARG;
    if (!is_yuv420_layout(layout)) return fail(c, JPGENC_ERR_ARG, "unknown YUV 4:2:0 layout");
    return jpgenc_bind_device_yuv(c, y, u, v, w, h, y_pitch, c_pitch, layout);
} JPGENC_CATCH(c)

static int enqueue_forward(jpgenc_ctx* c);

int jpgenc_color_dct_quant(jpgenc_ctx* c) try {
    if (!c) return JPGENC_ERR_ARG;
    if (!c->have_pixels) return fail(c, JPGENC_ERR_ARG, "no pixels bound: call jpgenc_upload_rgb / jpgenc_bind_device_rgb first");
    JPGENC_CUDA(c, cudaSetDevice(c->device));
    int rc = ensure_coef(c);
    if (rc) return rc;
    if ((rc = flush_entropy_time(c))) return rc;
    if ((rc = enqueue_forward(c))) return rc;
    c->forward_pending = true;
    c->fwd_timed = c->stage_timing;
    c->have_coef = true;
    c->have_scan = c->have_items = false; c->k2_tiles_done = 0;
    return JPGENC_OK;
} JPGENC_CATCH(c)

int jpgenc_get_coefficients(jpgenc_ctx* c, int16_t* dst) try {
    if (!c || !dst) return JPGENC_ERR_ARG;
    if (!c->have_coef) return fail(c, JPGENC_ERR_ARG, "no coefficients yet");
    const size_t bytes = static_cast<size_t>(c->mcu_w) * c->mcu_h * kBlocksPerMcu * kBlockBytes;
    JPGENC_CUDA(c, cudaMemcpyAsync(dst, c->d_coef, bytes, cudaMemcpyDeviceToHost, c->stream));
    JPGENC_CUDA(c, cudaStreamSynchronize(c->stream));
    uint32_t refined = 0;
    JPGENC_CUDA(c, cudaMemcpy(&refined, c->d_counters, sizeof refined, cudaMemcpyDeviceToHost));
    c->stats.refined_blocks = refined;
    return refresh_forward_stats(c);
} JPGENC_CATCH(c)

int jpgenc_set_coefficients_mcu(jpgenc_ctx* c, const int16_t* coef, uint32_t mcu_w, uint32_t mcu_h) try {
    if (!c || !coef || !mcu_w || !mcu_h) return JPGENC_ERR_ARG;
    JPGENC_CUDA(c, cudaSetDevice(c->device));
    if (c->real_w == 0 || (c->real_w + 15) / 16 != mcu_w || (c->real_h + 15) / 16 != mcu_h) {
        c->real_w = mcu_w * 16; c->real_h = mcu_h * 16; c->maxval = 255;
        c->have_pixels = false;                                   // pixels bound earlier belong to another geometry: K1 must not read them with this one
    }
    c->mcu_w = mcu_w; c->mcu_h = mcu_h;
    int rc = ensure_coef(c);
    if (rc) return rc;
    const size_t bytes = static_cast<size_t>(mcu_w) * mcu_h * kBlocksPerMcu * kBlockBytes;
    JPGENC_CUDA(c, cudaMemcpyAsync(c->d_coef, coef, bytes, cudaMemcpyHostToDevice, c->stream));
    JPGENC_CUDA(c, cudaStreamSynchronize(c->stream));
    c->have_coef = true;
    c->have_scan = c->have_items = false; c->k2_tiles_done = 0;
    return JPGENC_OK;
} JPGENC_CATCH(c)

int jpgenc_set_coefficients(jpgenc_ctx* c, const int32_t* q_y, const int32_t* q_cb, const int32_t* q_cr, uint32_t mcu_w,
                            uint32_t mcu_h) try {
    if (!c || !q_y || !q_cb || !q_cr || !mcu_w || !mcu_h) return JPGENC_ERR_ARG;
    JPGENC_CUDA(c, cudaSetDevice(c->device));
    if (c->real_w == 0 || (c->real_w + 15) / 16 != mcu_w || (c->real_h + 15) / 16 != mcu_h) {
        c->real_w = mcu_w * 16; c->real_h = mcu_h * 16; c->maxval = 255;
        c->have_pixels = false;                                   // pixels bound earlier belong to another geometry: K1 must not read them with this one
    }
    c->mcu_w = mcu_w; c->mcu_h = mcu_h;
    int rc = ensure_coef(c);
    if (rc) return rc;
    const size_t ny = static_cast<size_t>(mcu_w) * mcu_h * 256, nc = ny / 4;
    int32_t* d = nullptr;
    JPGENC_CUDA(c, cudaMalloc(reinterpret_cast<void**>(&d), (ny + 2 * nc) * sizeof(int32_t)));
    cudaError_t e = cudaMemcpyAsync(d, q_y, ny * 4, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d + ny, q_cb, nc * 4, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) e = cudaMemcpyAsync(d + ny + nc, q_cr, nc * 4, cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) rc = launch_planes_to_mcu(c, d, d + ny, d + ny + nc);
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    cudaFree(d);
    if (e != cudaSuccess) { c->error = cudaGetErrorString(e); return JPGENC_ERR_CUDA; }
    if (rc) return rc;
    c->have_coef = true;
    c->have_scan = c->have_items = false; c->k2_tiles_done = 0;
    return JPGENC_OK;
} JPGENC_CATCH(c)

// ---- K2 and K3/K4 for all frames bound to the context (one image = one frame) ------------------------------------
// ---- one image: the GPU work of an encode as two enqueue-only phases (no host waits inside: they can be captured) ----
// K1 + exact refinement, between the forward-stage events
static int enqueue_forward(jpgenc_ctx* c) {
    JPGENC_CUDA(c, stage_record(c, c->ev_a, 2));
    const int rc = launch_forward(c);
    if (rc) return rc;
    JPGENC_CUDA(c, stage_record(c, c->ev_b, 2));
    return JPGENC_OK;
}
// K2 over the tiles [done, tiles) and the hand-over of the statistics to the host's mailbox
static int enqueue_stats(jpgenc_ctx* c, uint32_t done) {
    const size_t nblocks = static_cast<size_t>(c->mcu_w) * c->mcu_h * kBlocksPerMcu, tiles = (nblocks + 383) / 384;
    JPGENC_CUDA(c, stage_record(c, c->ev_t0, 2));
    int rc = launch_symbol_stats(c, done, static_cast<uint32_t>(tiles) - done, done == 0);
    if (rc) return rc;
    JPGENC_CUDA(c, stage_record(c, c->ev_t1, 2));
    return launch_publish_stats(c);
}
// the host's half: wait for the mailbox, take the histogram
static int wait_stats(jpgenc_ctx* c) {
    c->have_items = true;
    int rc = flush_entropy_time(c);                               // the previous encode's K3/K4 time, while K2 runs
    if (rc) return rc;
    unsigned long long head = 0;
    if ((rc = poll_mailbox(c, kMailStatsHead, &head))) return rc;   // the statistics are in the mailbox
    const uint32_t present = static_cast<uint32_t>(head & 0x7FFu);
    std::memset(c->stat_count, 0, sizeof c->stat_count);
    std::memset(c->stat_first, 0xFF, sizeof c->stat_first);
    for (uint32_t k = 0; k < present; ++k) {
        unsigned long long a = 0, b = 0;
        if ((rc = poll_mailbox(c, kMailStatsHead + 1 + 2 * k, &a))) return rc;
        if ((rc = poll_mailbox(c, kMailStatsHead + 2 + 2 * k, &b))) return rc;
        const uint32_t e = static_cast<uint32_t>(a >> 32) & 1023u;
        (&c->stat_count[0][0])[e] = static_cast<uint32_t>(a);
        (&c->stat_first[0][0])[e] = b;
    }
    c->host_hist.assign(&c->stat_count[0][0], &c->stat_count[0][0] + 1024);
    if (c->upload_pending || c->forward_pending) c->stats.refined_blocks = static_cast<uint32_t>(head >> 11);
    c->stats_pending = true;
    c->stats_timed = c->stage_timing;
    return JPGENC_OK;
}

// K2 for the image bound to the context; the statistics arrive in the host mailbox
static int stats_frames(jpgenc_ctx* c) {
    JPGENC_CUDA(c, cudaSetDevice(c->device));
    if (c->nframes != 1) return fail(c, JPGENC_ERR_ARG, "stage calls work on one image; a batch is bound");
    const size_t nblocks = static_cast<size_t>(c->mcu_w) * c->mcu_h * kBlocksPerMcu, tiles = (nblocks + 383) / 384;
    int rc;
    if ((rc = ensure_stats_buffers(c))) return rc;
    // a band-wise upload has already taken the first k2_tiles_done tiles through K2
    const uint32_t done = std::min<uint32_t>(c->k2_tiles_done, static_cast<uint32_t>(tiles));
    c->k2_tiles_done = 0;
    if ((rc = enqueue_stats(c, done))) return rc;
    return wait_stats(c);
}

// stage times whose events are complete once K3/K4 have been enqueued (called while those run): K1 and refinement, the
// upload, K2 of the current encode, K3/K4 of the previous one
static int read_completed_times(jpgenc_ctx* c) {
    int rc = flush_entropy_time(c);
    if (rc) return rc;
    const bool whole = c->forward_pending && c->stats_pending;
    if (c->upload_pending) {          // banded upload of jpgenc_encode_rgb: ev_b was recorded on the copy stream behind the last band
        JPGENC_CUDA(c, cudaEventSynchronize(c->ev_b));
        JPGENC_CUDA(c, cudaEventElapsedTime(&c->stats.ms_h2d, c->ev_a, c->ev_b));
        c->upload_pending = false;
    }
    if (c->forward_pending && (rc = refresh_forward_stats(c))) return rc;
    if (c->stats_pending) {
        c->stats.ms_stats = 0;
        if (c->stats_timed >= 2) {
            JPGENC_CUDA(c, cudaEventSynchronize(c->ev_t1));        // recorded right behind K2, whose flag the host has seen long ago
            JPGENC_CUDA(c, cudaEventElapsedTime(&c->stats.ms_stats, c->ev_t0, c->ev_t1));
        }
        c->stats_pending = false;
    }
    c->last_whole = whole;
    c->last_k1 = c->stats.ms_k1; c->last_fwd = c->stats.ms_forward; c->last_st = c->stats.ms_stats;
    return JPGENC_OK;
}

// ---- K3/K4 of one image with tables built on the host ----
// Host part: the tables in the lookup form K3 reads, and -- from histogram x code length -- the exact geometry of the
// scan (the PassMeta block a batch computes on the device, finalize.cu), both into pinned staging; buffers sized for it.
// *k4_tiles = the exact number of K4 tiles.
static int prepare_entropy(jpgenc_ctx* c, const jpgenc_huff_table* tables, uint32_t* k4_tiles) {
    if (c->nframes != 1) return fail(c, JPGENC_ERR_ARG, "stage calls work on one image; a batch is bound");
    if (c->host_hist.size() != 1024) return fail(c, JPGENC_ERR_ARG, "symbol statistics missing: run jpgenc_symbol_stats first");
    int rc;
    if ((rc = ensure_pinned(c, stage_bytes(1)))) return rc;
    uint8_t* h = static_cast<uint8_t*>(c->h_pinned);
    DeviceTables* ht = reinterpret_cast<DeviceTables*>(h + stage_tables_off(1));
    const PassMeta m = pass_meta_view(h + stage_meta_off(1), 1);
    // exact size of the scan from the statistics the tables were built from: a symbol costs its code length plus
    // (symbol & 15) magnitude bits
    const uint32_t* hist = c->host_hist.data();
    uint64_t bits = 0;
    for (int t = 0; t < 4; ++t) {
        const jpgenc_huff_table& tab = tables[t];
        for (int s = 0; s < 256; ++s) {
            const uint32_t len = tab.length[s];
            const uint32_t code = len ? tab.code_msb[s] >> (32 - len) : 0u, cat = s & 15;
            ht->entry[t][s] = len ? (len << 16) | code : 0u;
            ht->fast[t][s] = (len && len + cat <= 27) ? ((len + cat) << 27) | (code << cat) : 0u;
            if (hist[t * 256 + s]) {
                if (!len) return fail(c, JPGENC_ERR_ARG, "Huffman table lacks a symbol that occurs in the image");
                bits += static_cast<uint64_t>(hist[t * 256 + s]) * (len + cat);
            }
        }
    }
    if (bits == 0) return fail(c, JPGENC_ERR_ARG, "symbol statistics missing: run jpgenc_symbol_stats first");
    const uint64_t nbytes = (bits + 7) / 8, tiles = (nbytes + kK4TileBytes - 1) / kK4TileBytes;
    if (tiles > 0x7FFFFFFFull) return fail(c, JPGENC_ERR_ARG, "scan too large");
    c->frame_bits.assign(1, bits);
    m.raw_off[0] = 0;
    m.raw_bytes[0] = nbytes;
    m.frame_bits[0] = bits;
    m.file_base[0] = 0;                                          // the bare scan
    m.k4_tile0[0] = 0;
    m.k4_tile0[1] = static_cast<uint32_t>(tiles);
    m.hdr_len[0] = 0;
    *m.hdr = PassHeader{};
    m.hdr->raw_total = raw_slot_bytes(nbytes);
    m.hdr->out_total = nbytes;
    m.hdr->raw_sum = nbytes;
    m.hdr->k4_tiles = static_cast<uint32_t>(tiles);
    m.hdr->nframes = 1;
    c->file_mode = false;
    *k4_tiles = static_cast<uint32_t>(tiles);
    // the look-back words are sized for the largest K4 grid the raw buffer allows (graph replays launch that many CTAs)
    if ((rc = ensure_entropy_buffers(c, m.hdr->raw_total, 2 * nbytes, tiles))) return rc;
    return ensure_entropy_buffers(c, m.hdr->raw_total, 2 * nbytes, c->raw_cap / kK4TileBytes + 1);
}
// GPU part, enqueue only: tables + geometry to the device, K3a, K3b, K4, totals into the mailbox
static int enqueue_entropy_phase(jpgenc_ctx* c, uint32_t k4_grid) {
    const uint8_t* h = static_cast<const uint8_t*>(c->h_pinned);
    // (Measured and rejected: passing the 8 KB of tables as kernel parameters instead -- the launches get slower and the
    // per-thread reads of the parameter bank serialise; K3+K4 went from 185 to 212 us.)
    JPGENC_CUDA(c, cudaMemcpyAsync(c->d_tables, h + stage_tables_off(1), sizeof(DeviceTables) + pass_meta_input_bytes(1), cudaMemcpyHostToDevice, c->stream));
    JPGENC_CUDA(c, stage_record(c, c->ev_e0, 2));
    const int rc = launch_entropy(c, k4_grid);
    if (rc) return rc;
    JPGENC_CUDA(c, stage_record(c, c->ev_e1, 2));
    return JPGENC_OK;
}
// the host's half: stage times that are final by now, then the totals from the mailbox
static int wait_entropy(jpgenc_ctx* c) {
    int rc = read_completed_times(c);                            // K3/K4 are running: the host has nothing else to do
    if (rc) return rc;
    c->ent_pending = true;
    c->ent_timed = c->stage_timing;
    unsigned long long bits = 0, ff = 0;
    if ((rc = poll_mailbox(c, kMailTotals, &bits))) return rc;   // the totals are in the mailbox (launch_entropy's last kernel)
    if ((rc = poll_mailbox(c, kMailTotals + 1, &ff))) return rc;
    if (bits != c->frame_bits[0]) {
        c->error = "entropy coder wrote " + std::to_string(bits) + " bits, statistics predicted " + std::to_string(c->frame_bits[0]);
        return JPGENC_ERR_ARG;
    }
    c->stats.scan_bits = bits;
    c->stats.stuffed_ff = ff;
    c->stats.scan_bytes = (bits + 7) / 8 + ff;
    c->have_scan = true;
    return JPGENC_OK;
}

// tables[4], built on the host.  Afterwards the stuffed scan is in d_scan, its size in c->stats.
static int entropy_frames(jpgenc_ctx* c, const jpgenc_huff_table* tables) {
    JPGENC_CUDA(c, cudaSetDevice(c->device));
    uint32_t k4_tiles = 0;
    int rc = prepare_entropy(c, tables, &k4_tiles);
    if (rc) return rc;
    if ((rc = enqueue_entropy_phase(c, k4_tiles))) return rc;
    return wait_entropy(c);
}

int jpgenc_symbol_stats(jpgenc_ctx* c, uint32_t count[4][256], uint64_t first_pos[4][256]) try {
    if (!c || !count || !first_pos) return JPGENC_ERR_ARG;
    if (!c->have_coef) return fail(c, JPGENC_ERR_ARG, "no coefficients: run jpgenc_color_dct_quant first");
    if (c->nframes != 1) return fail(c, JPGENC_ERR_ARG, "stage calls work on one image; a batch is bound");
    const int rc = stats_frames(c);
    if (rc) return rc;
    std::memcpy(count, c->stat_count, 4096);
    std::memcpy(first_pos, c->stat_first, 8192);
    return JPGENC_OK;
} JPGENC_CATCH(c)

// the device build's code (array restatement of the container orders) executed on the host, no GPU involved
int jpgenc_build_huffman_arrays(const uint32_t count[256], const uint64_t first_pos[256], jpgenc_huff_table* out) {
    if (!count || !first_pos || !out) return JPGENC_ERR_ARG;
    return build_table_arrays_host(count, first_pos, out);
}

// generateHuffmanCode on the device (tables_device.cu) for n independent (count, first_pos) pairs; what the batched-frame
// calls use on hosts with few cores per GPU, exposed so that it can be checked against jpgenc_build_huffman directly
int jpgenc_build_huffman_device(jpgenc_ctx* c, uint32_t n, const uint32_t (*count)[256], const uint64_t (*first_pos)[256],
                                jpgenc_huff_table* out) try {
    if (!c || !count || !first_pos || !out || n == 0) return JPGENC_ERR_ARG;
    JPGENC_CUDA(c, cudaSetDevice(c->device));
    const uint32_t frames = (n + 3) / 4;                       // the kernel reads K2's layout: 4 tables per frame
    std::vector<uint8_t> host(static_cast<size_t>(frames) * kStatsBytes, 0);
    for (uint32_t i = 0; i < frames * 4; ++i) {
        uint8_t* f = host.data() + static_cast<size_t>(i >> 2) * kStatsBytes;
        if (i < n) {
            std::memcpy(f + (i & 3) * 1024, count[i], 1024);
            std::memcpy(f + 4096 + (i & 3) * 2048, first_pos[i], 2048);
        } else {
            std::memset(f + 4096 + (i & 3) * 2048, 0xFF, 2048);
        }
    }
    int rc;
    uint8_t* d_in = nullptr;
    size_t cap = 0;
    if ((rc = ensure(c, &d_in, &cap, host.size()))) return rc;
    auto cleanup = [&] { cudaFree(d_in); };
    const uint32_t nt = frames * 4;
    if ((rc = ensure(c, reinterpret_cast<uint8_t**>(&c->d_tab_scratch), &c->tab_scratch_cap, nt * table_scratch_bytes()))) { cleanup(); return rc; }
    if ((rc = ensure(c, &c->d_built_tables, &c->built_tables_cap, nt * (sizeof(jpgenc_huff_table) + sizeof(uint32_t))))) { cleanup(); return rc; }
    std::vector<jpgenc_huff_table> res(nt);
    cudaError_t e = cudaMemcpyAsync(d_in, host.data(), host.size(), cudaMemcpyHostToDevice, c->stream);
    if (e == cudaSuccess) {
        rc = launch_build_tables(c, d_in, kStatsBytes, nt, c->d_tab_scratch, c->d_built_tables, reinterpret_cast<uint32_t*>(c->d_built_tables + nt));
        if (rc) { cleanup(); return rc; }
        e = cudaMemcpyAsync(res.data(), c->d_built_tables, nt * sizeof(jpgenc_huff_table), cudaMemcpyDeviceToHost, c->stream);
    }
    if (e == cudaSuccess) e = cudaStreamSynchronize(c->stream);
    cleanup();
    if (e != cudaSuccess) { c->error = std::string("device table build: ") + cudaGetErrorString(e); return JPGENC_ERR_CUDA; }
    for (uint32_t i = 0; i < n; ++i) {
        if (res[i].nsymbols <= 0) return fail(c, JPGENC_ERR_ARG, "Huffman table build failed: a table has no symbol");
        out[i] = res[i];
    }
    return JPGENC_OK;
} JPGENC_CATCH(c)

int jpgenc_entropy_encode(jpgenc_ctx* c, const jpgenc_huff_table tables[4], uint64_t* scan_bytes) try {
    if (!c || !tables) return JPGENC_ERR_ARG;
    if (!c->have_coef) return fail(c, JPGENC_ERR_ARG, "no coefficients: run jpgenc_color_dct_quant first");
    if (!c->have_items) return fail(c, JPGENC_ERR_ARG, "symbol statistics missing: run jpgenc_symbol_stats first");
    if (c->nframes != 1) return fail(c, JPGENC_ERR_ARG, "stage calls work on one image; a batch is bound");
    const int rc = entropy_frames(c, tables);
    if (rc) return rc;
    if (scan_bytes) *scan_bytes = c->stats.scan_bytes;
    return JPGENC_OK;
} JPGENC_CATCH(c)

int jpgenc_download_scan(jpgenc_ctx* c, uint8_t* dst, uint64_t cap) try {
    if (!c || !dst) return JPGENC_ERR_ARG;
    if (!c->have_scan) return fail(c, JPGENC_ERR_ARG, "no scan yet: run jpgenc_entropy_encode first");
    if (cap < c->stats.scan_bytes) return fail(c, JPGENC_ERR_CAPACITY, "scan buffer too small");
    JPGENC_CUDA(c, jpgenc_record(c, c->ev_t0));
    JPGENC_CUDA(c, cudaMemcpyAsync(dst, c->d_scan, c->stats.scan_bytes, cudaMemcpyDeviceToHost, c->stream));
    JPGENC_CUDA(c, jpgenc_record(c, c->ev_t1));
    JPGENC_CUDA(c, cudaStreamSynchronize(c->stream));
    JPGENC_CUDA(c, cudaEventElapsedTime(&c->stats.ms_d2h, c->ev_t0, c->ev_t1));
    return JPGENC_OK;
} JPGENC_CATCH(c)

// K2 .. K4 on the coefficients K1 left on the device
static int run_entropy_stages(jpgenc_ctx* c, jpgenc_huff_table tables[4], uint64_t* scan) {
    int rc;
    uint32_t count[4][256];
    uint64_t first_pos[4][256];
    // the pool's workers spin from arm() until the statistics arrive: fine for the ~0.2 ms of K2 on resident pixels, not for
    // the milliseconds an upload takes (VERDICT round 1: 3 spinning workers x 8 ranks on a 32-core host)
    if (!c->parallel_tables || c->upload_pending) {
        if ((rc = jpgenc_symbol_stats(c, count, first_pos))) return rc;
        for (int t = 0; t < 4; ++t)
            if ((rc = jpgenc_build_huffman(count[t], first_pos[t], &tables[t]))) return fail(c, rc, "Huffman table build failed");
    } else {
        if (!c->pool) c->pool = new TablePool(kTableWorkers);
        c->pool->arm();                                             // the workers wake up while K2 runs
        if ((rc = jpgenc_symbol_stats(c, count, first_pos))) {
            c->pool->build(nullptr, nullptr, nullptr);              // release them again
            return rc;
        }
        if ((rc = c->pool->build(count, first_pos, tables))) return fail(c, rc, "Huffman table build failed");
    }
    if ((rc = jpgenc_entropy_encode(c, tables, scan))) return rc;
    std::memcpy(c->last_tables, tables, sizeof c->last_tables);
    c->have_tables = true;
    return JPGENC_OK;
}

// ---- whole encode of the pixels bound to the context, its two GPU phases replayed as CUDA graphs ----------------------
// A small frame is launch-bound: phase A is 8 stream operations (counters, K1, refinement, 3 clears, K2, publish) plus
// their events, phase B 5 (tables upload, K3a, K3b, K4, publish); at ~4-5 us of host time per call the GPU waits for its
// next kernel (3840x2160: 35 us of enqueueing in front of 38 us of K3/K4).  Nothing in either phase depends on the
// content of the image: sizes that do (scan length, number of K4 tiles) are read from device memory by the kernels, the
// mailbox sequence number lives in device memory, K4's grid is an upper bound (run_pipeline: k4_grid_hint).  So a phase is
// captured once per configuration (pixels pointer, geometry, buffers: the key) and replayed with one launch.  A
// configuration is captured when it is encoded the second time in a row; JPGENC_GRAPHS=0 disables it.
static bool graphs_enabled() {
    static const bool on = [] { const char* v = std::getenv("JPGENC_GRAPHS"); return !(v && *v == '0'); }();
    return on;
}

// replays (capturing first, if the key is new for the second time) the phase that `enqueue` puts on the stream
static int run_phase(jpgenc_ctx* c, jpgenc_ctx::PhaseGraph& g, const uint64_t (&key)[kGraphKeyWords], const std::function<int()>& enqueue) {
    const bool same_as_graph = g.exec && std::memcmp(g.key, key, sizeof key) == 0;
    if (!same_as_graph) {
        const bool repeat = std::memcmp(g.seen, key, sizeof key) == 0;
        std::memcpy(g.seen, key, sizeof key);
        if (!graphs_enabled() || !repeat) return enqueue();          // first sight of this configuration: plain launches
        if (g.exec) { cudaGraphExecDestroy(g.exec); g.exec = nullptr; }
        const uint64_t launches0 = c->launches;
        const uint32_t seq0 = c->mailbox_seq;
        JPGENC_CUDA(c, cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
        c->capturing = true;
        const int rc = enqueue();
        c->capturing = false;
        cudaGraph_t graph = nullptr;
        const cudaError_t e = cudaStreamEndCapture(c->stream, &graph);
        g.launches = static_cast<uint32_t>(c->launches - launches0);
        c->launches = launches0;                                     // nothing has run yet
        const uint32_t publishes = c->mailbox_seq - seq0;
        c->mailbox_seq = seq0;
        if (rc || e != cudaSuccess || !graph) {
            if (graph) cudaGraphDestroy(graph);
            (void)cudaGetLastError();
            return rc ? rc : fail(c, JPGENC_ERR_CUDA, "stream capture of an encode phase failed");
        }
        const cudaError_t ei = cudaGraphInstantiate(&g.exec, graph, 0);
        cudaGraphDestroy(graph);
        if (ei != cudaSuccess) { g.exec = nullptr; c->error = std::string("cudaGraphInstantiate: ") + cudaGetErrorString(ei); return JPGENC_ERR_CUDA; }
        std::memcpy(g.key, key, sizeof key);
        g.publishes = publishes;
    }
    JPGENC_CUDA(c, cudaGraphLaunch(g.exec, c->stream));
    c->launches += g.launches;
    c->mailbox_seq += g.publishes;                                   // what the replayed publish kernels will announce
    return JPGENC_OK;
}

static int run_pipeline(jpgenc_ctx* c, jpgenc_huff_table tables[4], uint64_t* scan) {
    if (!c->have_pixels) return fail(c, JPGENC_ERR_ARG, "no pixels bound: call jpgenc_upload_rgb / jpgenc_bind_device_rgb first");
    JPGENC_CUDA(c, cudaSetDevice(c->device));
    if (c->nframes != 1) return fail(c, JPGENC_ERR_ARG, "stage calls work on one image; a batch is bound");
    int rc;
    if ((rc = ensure_coef(c))) return rc;
    if ((rc = ensure_stats_buffers(c))) return rc;
    // ---- phase A: K1, refinement, K2, statistics into the mailbox ----
    c->k2_tiles_done = 0;
    // (the pixel layout picks K1, its thresholds and the refinement: it is part of the key, with every plane and pitch)
    const PixelSource& src = c->src;
    const uint64_t key_a[kGraphKeyWords] = {c->alloc_gen, reinterpret_cast<uint64_t>(src.plane[0]), (static_cast<uint64_t>(c->real_w) << 32) | c->real_h,
                                            c->maxval | static_cast<uint64_t>(src.format) << 8 | static_cast<uint64_t>(src.pitch) << 32,
                                            1u | static_cast<uint64_t>(c->stage_timing) << 8, reinterpret_cast<uint64_t>(src.plane[1]),
                                            reinterpret_cast<uint64_t>(src.plane[2]), src.pitch2};
    const bool pool = c->parallel_tables;
    if (pool) {
        if (!c->pool) c->pool = new TablePool(kTableWorkers);
        c->pool->arm();                                             // the table builders wake up while K1 / K2 run
    }
    rc = run_phase(c, c->graph_a, key_a, [&]() -> int {
        const int r = enqueue_forward(c);
        return r ? r : enqueue_stats(c, 0);
    });
    c->forward_pending = true;
    c->fwd_timed = c->stage_timing;
    c->have_coef = true;
    c->have_scan = false;
    if (!rc) rc = wait_stats(c);
    if (rc) {
        if (pool) c->pool->build(nullptr, nullptr, nullptr);        // release the workers again
        return rc;
    }
    // ---- host: the four tables ----
    const uint32_t(*count)[256] = c->stat_count;
    const uint64_t(*first_pos)[256] = c->stat_first;
    if (pool) {
        if ((rc = c->pool->build(count, first_pos, tables))) return fail(c, rc, "Huffman table build failed");
    } else {
        for (int t = 0; t < 4; ++t)
            if ((rc = jpgenc_build_huffman(count[t], first_pos[t], &tables[t]))) return fail(c, rc, "Huffman table build failed");
    }
    // ---- phase B: tables to the device, K3a, K3b, K4, totals into the mailbox ----
    uint32_t k4_tiles = 0;
    if ((rc = prepare_entropy(c, tables, &k4_tiles))) return rc;
    // K4's grid is part of the captured graph, the number of tiles is not (K4 reads it from device memory; surplus CTAs leave at
    // once): an upper bound that follows the images seen -- half as much again as the last one that did not fit, given up
    // when an image needs less than a quarter of it (a context that once encoded 16384^2 would otherwise launch 2 x 2700
    // CTAs for the 83 tiles of every 3840x2160 frame: 10 us), never more than the raw buffer holds
    if (k4_tiles > c->k4_grid_hint || k4_tiles < c->k4_grid_hint / 4) c->k4_grid_hint = k4_tiles + k4_tiles / 2 + 8;
    const uint32_t k4_grid = std::min(c->k4_grid_hint, static_cast<uint32_t>(c->raw_cap / kK4TileBytes + 1));   // raw_cap holds the scan: >= k4_tiles
    const uint64_t key_b[kGraphKeyWords] = {c->alloc_gen, k4_grid, (static_cast<uint64_t>(c->real_w) << 32) | c->real_h, 0,
                                            1u | static_cast<uint64_t>(c->stage_timing) << 8, 0, 0, 0};
    if ((rc = run_phase(c, c->graph_b, key_b, [&]() -> int { return enqueue_entropy_phase(c, k4_grid); }))) return rc;
    if ((rc = wait_entropy(c))) return rc;
    if (scan) *scan = c->stats.scan_bytes;
    std::memcpy(c->last_tables, tables, sizeof c->last_tables);
    c->have_tables = true;
    return JPGENC_OK;
}

// pinned staging for streamed inputs (jpgenc_encode_ppm_file), grown on demand
static int ensure_file_staging(jpgenc_ctx* c, size_t bytes) {
    if (c->file_pinned_bytes >= bytes) return JPGENC_OK;
    if (c->h_file_pinned) JPGENC_CUDA(c, cudaFreeHost(c->h_file_pinned));
    c->h_file_pinned = nullptr; c->file_pinned_bytes = 0;
    JPGENC_CUDA(c, cudaMallocHost(&c->h_file_pinned, bytes));
    c->file_pinned_bytes = bytes;
    return JPGENC_OK;
}

// Host pixels -> coefficients with the upload hidden behind K1: the image is cut into bands of MCU rows, every band
// is copied on the copy stream and transformed on the compute stream as soon as its copy has landed, so after the last
// byte has crossed PCIe only one band of K1 work (plus the refinement) is left.
// `fill` (optional): instead of reading the pixels from `host_rgb`, every band is first produced by fill(dst, byte offset in
// the image, bytes) into one of two pinned staging buffers (a file read, for instance) and uploaded from there: bounded
// pinned memory, full PCIe rate, and the production of band b+1 overlaps the upload of band b.
// Pixels in another layout travel as they are, in their own format, plane by plane (staged_planes), the pitch gaps dropped by
// the copy: on the device they are tight rows of that format, read by the pixel-layout kernels; a band carries every plane's
// rows of its MCU rows.  `host` is checked (check_source); with `fill` its plane is not read.
static int upload_and_forward(jpgenc_ctx* c, const PixelSource& host, uint32_t w, uint32_t h, uint32_t maxval,
                              const std::function<int(uint8_t*, size_t, size_t)>* fill = nullptr) {
    JPGENC_CUDA(c, cudaSetDevice(c->device));
    int rc = set_geometry(c, w, h, maxval);
    if (rc) return rc;
    StagedPlane pl[3];
    const uint32_t np = staged_planes(host, w, h, pl);
    const size_t row_bytes = pl[0].row;
    if ((rc = ensure(c, &c->d_rgb_owned, &c->rgb_cap, staged_bytes(pl, np) + 16))) return rc;
    c->src = host;
    for (uint32_t k = 0; k < 3; ++k) c->src.plane[k] = k < np ? c->d_rgb_owned + pl[k].dev_off : nullptr;
    c->src.pitch = static_cast<uint32_t>(row_bytes);
    if (np > 1) c->src.pitch2 = static_cast<uint32_t>(pl[1].row);
    c->have_pixels = true;
    if ((rc = ensure_coef(c))) return rc;
    const size_t gap = planes_gap(pl, np);                       // planes equally spaced with tight rows: one strided copy per band
    constexpr uint32_t kMaxBands = sizeof(c->ev_band) / sizeof(c->ev_band[0]);
    // bands of at least ~8 MB (a copy that size already runs at full PCIe rate), at most kMaxBands of them
    size_t mcu_row_bytes = 0;
    for (uint32_t k = 0; k < np; ++k) mcu_row_bytes += pl[k].row * (16 >> pl[k].vsub);
    uint32_t rows_per_band = static_cast<uint32_t>(std::max<size_t>(1, (8u << 20) / mcu_row_bytes));
    rows_per_band = std::max(rows_per_band, (c->mcu_h + kMaxBands - 1) / kMaxBands);
    if ((rc = ensure_stats_buffers(c))) return rc;
    const uint32_t tiles = (c->mcu_w * c->mcu_h * kBlocksPerMcu + 383) / 384;
    JPGENC_CUDA(c, cudaEventRecord(c->ev_a, c->copy_stream));
    uint32_t band = 0, k2_done = 0;
    for (uint32_t y0 = 0; y0 < c->mcu_h; y0 += rows_per_band, ++band) {
        const uint32_t rows = std::min(rows_per_band, c->mcu_h - y0);
        const size_t px0 = static_cast<size_t>(y0) * 16, px1 = std::min<size_t>(h, static_cast<size_t>(y0 + rows) * 16);
        if (px1 > px0) {
            const uint8_t* src = fill ? nullptr : pl[0].host + px0 * pl[0].pitch;
            size_t src_pitch = pl[0].pitch;
            if (fill) {
                const size_t band_bytes = static_cast<size_t>(rows_per_band) * 16 * row_bytes;
                if (band == 0) {
                    if ((rc = ensure_file_staging(c, 2 * band_bytes))) return rc;
                } else if (band >= 2) {
                    JPGENC_CUDA(c, cudaEventSynchronize(c->ev_band[band - 2]));     // this slot's previous upload has left it
                }
                uint8_t* slot = static_cast<uint8_t*>(c->h_file_pinned) + (band & 1) * band_bytes;
                if ((rc = (*fill)(slot, px0 * row_bytes, (px1 - px0) * row_bytes))) return fail(c, rc, "truncated PPM payload, or a sample above maxval");
                src = slot;
                src_pitch = row_bytes;
            }
            if (gap)
                JPGENC_CUDA(c, cudaMemcpy2DAsync(c->d_rgb_owned + px0 * row_bytes, pl[1].dev_off, src, gap, (px1 - px0) * row_bytes, np,
                                                 cudaMemcpyHostToDevice, c->copy_stream));
            else
                for (uint32_t k = 0; k < np; ++k) {
                    // the rows of plane k under MCU rows [y0, y0 + rows): [px0, px1) at full height, [px0 / 2, ceil(px1 / 2)) subsampled
                    const size_t r0 = px0 >> pl[k].vsub, r1 = (px1 + pl[k].vsub) >> pl[k].vsub;
                    const uint8_t* from = k ? pl[k].host + r0 * pl[k].pitch : src;
                    const size_t from_pitch = k ? pl[k].pitch : src_pitch;
                    uint8_t* dst = c->d_rgb_owned + pl[k].dev_off + r0 * pl[k].row;
                    if (from_pitch == pl[k].row)
                        JPGENC_CUDA(c, cudaMemcpyAsync(dst, from, (r1 - r0) * pl[k].row, cudaMemcpyHostToDevice, c->copy_stream));
                    else
                        JPGENC_CUDA(c, cudaMemcpy2DAsync(dst, pl[k].row, from, from_pitch, pl[k].row, r1 - r0, cudaMemcpyHostToDevice, c->copy_stream));
                }
        }
        JPGENC_CUDA(c, cudaEventRecord(c->ev_band[band], c->copy_stream));
        JPGENC_CUDA(c, cudaStreamWaitEvent(c->stream, c->ev_band[band], 0));
        if ((rc = launch_forward_rows(c, y0, rows, y0 == 0, false))) return rc;
        // while the next band is on its way: exact refinement of what this band flagged, then K2 for every tile (64 MCUs)
        // that lies completely inside the rows transformed so far -- after the last byte has crossed PCIe only the last
        // band's share of K1, refinement and K2 is left before the tables can be built
        if ((rc = launch_refine_pending(c))) return rc;
        const bool last = y0 + rows >= c->mcu_h;
        const uint32_t upto = last ? tiles : static_cast<uint32_t>((static_cast<uint64_t>(y0 + rows) * c->mcu_w) / 64);
        if (!last && upto > k2_done) {
            if ((rc = launch_symbol_stats(c, k2_done, upto - k2_done, k2_done == 0))) return rc;
            k2_done = upto;
        }
    }
    JPGENC_CUDA(c, cudaEventRecord(c->ev_b, c->copy_stream));
    c->upload_pending = true;
    c->have_coef = true;
    c->have_scan = c->have_items = false;
    c->k2_tiles_done = k2_done;                                  // stats_frames finishes the rest
    return JPGENC_OK;
}

static int assemble(jpgenc_ctx* c, const jpgenc_huff_table tables[4], uint64_t scan, uint8_t* dst, uint64_t cap) {
    const size_t hdr = jpgenc_write_headers(c->real_w, c->real_h, c->qy, c->qc, tables, nullptr);
    if (cap < hdr + scan + 2) return fail(c, JPGENC_ERR_CAPACITY, "JPEG buffer too small");
    jpgenc_write_headers(c->real_w, c->real_h, c->qy, c->qc, tables, dst);
    const int rc = jpgenc_download_scan(c, dst + hdr, cap - hdr);
    if (rc) return rc;
    dst[hdr + scan] = 0xFF;                                      // EOI (JpegSegments.hpp:361-377)
    dst[hdr + scan + 1] = 0xD9;
    return JPGENC_OK;
}

int jpgenc_encode_bound(jpgenc_ctx* c, uint8_t* dst, uint64_t cap, uint64_t* jpeg_bytes) try {
    if (!c) return JPGENC_ERR_ARG;
    jpgenc_huff_table tables[4];
    uint64_t scan = 0;
    int rc = run_pipeline(c, tables, &scan);
    if (rc) return rc;
    const size_t hdr = jpgenc_write_headers(c->real_w, c->real_h, c->qy, c->qc, tables, nullptr);
    if (jpeg_bytes) *jpeg_bytes = hdr + scan + 2;
    if (!dst) return JPGENC_OK;                                  // device-resident run: the scan stays in HBM
    return assemble(c, tables, scan, dst, cap);
} JPGENC_CATCH(c)

int jpgenc_assemble_last(jpgenc_ctx* c, uint8_t* dst, uint64_t cap, uint64_t* jpeg_bytes) try {
    if (!c || !dst) return JPGENC_ERR_ARG;
    if (!c->have_tables || !c->have_scan) return fail(c, JPGENC_ERR_ARG, "no finished encode on this context");
    const size_t hdr = jpgenc_write_headers(c->real_w, c->real_h, c->qy, c->qc, c->last_tables, nullptr);
    if (jpeg_bytes) *jpeg_bytes = hdr + c->stats.scan_bytes + 2;
    return assemble(c, c->last_tables, c->stats.scan_bytes, dst, cap);
} JPGENC_CATCH(c)

// the rest of an encode whose coefficients are on their way: K2 .. K4, then the file into dst (NULL: the size only) or, with
// `out`, into *out, resized to the file
static int finish_encode(jpgenc_ctx* c, uint8_t* dst, uint64_t cap, uint64_t* jpeg_bytes, std::vector<uint8_t>* out = nullptr) {
    jpgenc_huff_table tables[4];
    uint64_t scan = 0;
    const int rc = run_entropy_stages(c, tables, &scan);             // its first synchronisation also covers the copies
    if (rc) return rc;
    const size_t hdr = jpgenc_write_headers(c->real_w, c->real_h, c->qy, c->qc, tables, nullptr);
    if (jpeg_bytes) *jpeg_bytes = hdr + scan + 2;
    if (out) {
        out->resize(hdr + scan + 2);
        dst = out->data();
        cap = out->size();
    }
    if (!dst) return JPGENC_OK;
    return assemble(c, tables, scan, dst, cap);
}

// host pixels: checked, uploaded band by band behind K1, encoded
static int encode_host_source(jpgenc_ctx* c, PixelSource src, uint32_t w, uint32_t h, uint32_t maxval, uint8_t* dst, uint64_t cap,
                              uint64_t* jpeg_bytes) {
    int rc = check_source(c, &src, w, h);
    if (rc) return rc;
    if (!source_within_maxval(src, w, h, maxval)) return fail(c, JPGENC_ERR_FORMAT, "a sample exceeds maxval");
    if ((rc = upload_and_forward(c, src, w, h, maxval))) return rc;
    return finish_encode(c, dst, cap, jpeg_bytes);
}

int jpgenc_encode_rgb(jpgenc_ctx* c, const uint8_t* host_rgb, uint32_t w, uint32_t h, uint32_t maxval, uint8_t* dst,
                      uint64_t cap, uint64_t* jpeg_bytes) try {
    if (!c || !host_rgb) return JPGENC_ERR_ARG;
    return encode_host_source(c, image_source(host_rgb, 0, JPGENC_PIXEL_RGB), w, h, maxval, dst, cap, jpeg_bytes);
} JPGENC_CATCH(c)

int jpgenc_encode_image(jpgenc_ctx* c, const void* host, uint32_t w, uint32_t h, uint32_t row_pitch, int format, uint32_t maxval,
                        uint8_t* dst, uint64_t cap, uint64_t* jpeg_bytes) try {
    if (!c) return JPGENC_ERR_ARG;
    return encode_host_source(c, image_source(host, row_pitch, format), w, h, maxval, dst, cap, jpeg_bytes);
} JPGENC_CATCH(c)

int jpgenc_encode_planar(jpgenc_ctx* c, const void* r, const void* g, const void* b, uint32_t w, uint32_t h, uint32_t row_pitch, uint32_t maxval,
                         uint8_t* dst, uint64_t cap, uint64_t* jpeg_bytes) try {
    if (!c) return JPGENC_ERR_ARG;
    return encode_host_source(c, planar_source(r, g, b, row_pitch), w, h, maxval, dst, cap, jpeg_bytes);
} JPGENC_CATCH(c)

int jpgenc_encode_yuv(jpgenc_ctx* c, const void* y, const void* u, const void* v, uint32_t w, uint32_t h, uint32_t y_pitch,
                      uint32_t c_pitch, int layout, uint8_t* dst, uint64_t cap, uint64_t* jpeg_bytes) try {
    if (!c) return JPGENC_ERR_ARG;
    return encode_host_source(c, yuv_source(y, u, v, y_pitch, c_pitch, layout), w, h, 255, dst, cap, jpeg_bytes);
} JPGENC_CATCH(c)

int jpgenc_encode_yuv420(jpgenc_ctx* c, const void* y, const void* u, const void* v, uint32_t w, uint32_t h, uint32_t y_pitch,
                         uint32_t c_pitch, int layout, uint8_t* dst, uint64_t cap, uint64_t* jpeg_bytes) try {
    if (!c) return JPGENC_ERR_ARG;
    if (!is_yuv420_layout(layout)) return fail(c, JPGENC_ERR_ARG, "unknown YUV 4:2:0 layout");
    return jpgenc_encode_yuv(c, y, u, v, w, h, y_pitch, c_pitch, layout, dst, cap, jpeg_bytes);
} JPGENC_CATCH(c)

// Image::writeJPEG for an image that is not (or no longer) a set of 8-bit samples: planes a caller edited after loadPPM,
// non-integral values, or an image that already is YCbCr (src/Image.cpp:831-846 encodes whatever the three planes hold and
// converts only an RGB image, :112-115).  The planes are uploaded as doubles and every block takes the exact FP64 path.
int jpgenc_encode_planes(jpgenc_ctx* c, const double* p0, const double* p1, const double* p2, uint32_t width, uint32_t height,
                         uint32_t real_w, uint32_t real_h, int ycbcr, uint8_t* dst, uint64_t cap, uint64_t* jpeg_bytes) try {
    if (!c || !p0 || !p1 || !p2) return JPGENC_ERR_ARG;
    JPGENC_CUDA(c, cudaSetDevice(c->device));
    // the reference's stages need whole 16x16 MCUs (loadPPM pads; an Image built in memory must have such a size already)
    if (real_w == 0 || real_h == 0 || width != ((real_w + 15u) & ~15u) || height != ((real_h + 15u) & ~15u))
        return fail(c, JPGENC_ERR_ARG, "planes must be the image padded to whole 16x16 MCUs");
    int rc = set_geometry(c, real_w, real_h, 255);
    if (rc) return rc;
    c->have_pixels = false;
    if ((rc = ensure_coef(c))) return rc;
    const size_t plane = static_cast<size_t>(width) * height;
    if ((rc = ensure(c, &c->d_rgb_owned, &c->rgb_cap, 3 * plane * sizeof(double) + 16))) return rc;
    double* d = reinterpret_cast<double*>(c->d_rgb_owned);
    const double* src[3] = {p0, p1, p2};
    for (int k = 0; k < 3; ++k)
        JPGENC_CUDA(c, cudaMemcpyAsync(d + k * plane, src[k], plane * sizeof(double), cudaMemcpyHostToDevice, c->stream));
    if ((rc = flush_entropy_time(c))) return rc;
    if ((rc = launch_planes_exact(c, d, ycbcr != 0))) return rc;
    JPGENC_CUDA(c, cudaStreamSynchronize(c->stream));            // the caller's planes may change as soon as we return
    c->stats.refined_blocks = static_cast<uint64_t>(c->mcu_w) * c->mcu_h * kBlocksPerMcu;
    c->have_coef = true;
    c->have_scan = c->have_items = false; c->k2_tiles_done = 0;
    return finish_encode(c, dst, cap, jpeg_bytes);
} JPGENC_CATCH(c)

// main.cpp:8-32.  A binary (P6) payload is streamed: the header is parsed from the first bytes, then every band of rows is
// read straight into pinned staging and uploaded while the next band is being read and the previous ones go through
// K1/refinement/K2 (loadPPM's pixel path, src/Image.cpp:411-418, without ever holding the image in host memory).  ASCII
// (P3) files are parsed on the host first (src/Image.cpp:393-408) and then take the same banded upload.
int jpgenc_encode_ppm_file(jpgenc_ctx* c, const char* ppm_path, const char* jpg_path) try {
    if (!c || !ppm_path || !jpg_path) return JPGENC_ERR_ARG;
    std::FILE* in = std::fopen(ppm_path, "rb");
    if (!in) return fail(c, JPGENC_ERR_IO, "Failed to open input file");
    struct Closer { std::FILE* f; ~Closer() { if (f) std::fclose(f); } } closer{in};
    std::vector<uint8_t> head(1 << 16);
    head.resize(std::fread(head.data(), 1, head.size(), in));
    PpmHeader h;
    int rc = parse_ppm_header(head.data(), head.size(), &h);
    if (rc) return fail(c, rc, "Only P3 and P6 format is supported!");
    if (h.magic == 6 && h.maxval <= 255) {
        const size_t need = static_cast<size_t>(h.width) * h.height * 3;
        // a band is read by several threads at once (positional reads): one thread copies from the page cache at ~6 GB/s,
        // which would leave the 55 GB/s link waiting
        ensure_host_pool(c);
        const int fd = fileno(in);
        const std::function<int(uint8_t*, size_t, size_t)> fill = [&](uint8_t* dst, size_t off, size_t n) -> int {
            constexpr size_t kPart = 8u << 20;
            const uint32_t parts = static_cast<uint32_t>((n + kPart - 1) / kPart);
            std::atomic<int> bad{0};
            c->host_pool->parallel_for(parts, [&](uint32_t k) {
                size_t at = static_cast<size_t>(k) * kPart;
                const size_t end = std::min(n, at + kPart);
                while (at < end) {
                    const ssize_t got = pread(fd, dst + at, end - at, static_cast<off_t>(h.payload + off + at));
                    if (got <= 0) { bad.store(1); return; }         // a short payload is an error (the reference's reader
                    at += static_cast<size_t>(got);                  // would run past the end of its buffer)
                }
            });
            (void)need;
            if (!bad.load() && !samples_within_maxval(dst, n, h.maxval)) bad.store(1);     // only scans when maxval < 255
            return bad.load() ? JPGENC_ERR_FORMAT : JPGENC_OK;
        };
        if ((rc = upload_and_forward(c, image_source(nullptr, h.width * 3, JPGENC_PIXEL_RGB), h.width, h.height, h.maxval, &fill))) return rc;
    } else {
        std::vector<uint8_t> file, p3;
        std::fclose(in);
        closer.f = nullptr;
        if ((rc = slurp_file(ppm_path, &file))) return fail(c, rc, "Failed to open input file");
        const uint8_t* samples = nullptr;
        if ((rc = ppm_samples(file.data(), file.size(), h, &p3, &samples))) return fail(c, rc, "truncated PPM payload, or a sample above maxval");
        if ((rc = upload_and_forward(c, image_source(samples, h.width * 3, JPGENC_PIXEL_RGB), h.width, h.height, h.maxval))) return rc;
    }
    std::vector<uint8_t> out;
    if ((rc = finish_encode(c, nullptr, 0, nullptr, &out))) return rc;
    std::FILE* f = std::fopen(jpg_path, "wb");
    if (!f) return fail(c, JPGENC_ERR_IO, "Failed to open output file");
    const size_t wrote = std::fwrite(out.data(), 1, out.size(), f);
    std::fclose(f);
    return wrote == out.size() ? JPGENC_OK : fail(c, JPGENC_ERR_IO, "short write");
} JPGENC_CATCH(c)

int jpgenc_ppm_info(const uint8_t* file, size_t n, uint32_t* width, uint32_t* height, uint32_t* maxval, int* magic,
                    size_t* payload_offset) {
    if (!file) return JPGENC_ERR_ARG;
    PpmHeader h;
    const int rc = parse_ppm_header(file, n, &h);
    if (rc) return rc;
    if (width) *width = h.width;
    if (height) *height = h.height;
    if (maxval) *maxval = h.maxval;
    if (magic) *magic = h.magic;
    if (payload_offset) *payload_offset = h.payload;
    return JPGENC_OK;
}

int jpgenc_ppm_samples(const uint8_t* file, size_t n, uint8_t* dst) {
    if (!file || !dst) return JPGENC_ERR_ARG;
    PpmHeader h;
    int rc = parse_ppm_header(file, n, &h);
    if (rc) return rc;
    std::vector<uint8_t> p3;
    const uint8_t* view = nullptr;
    if ((rc = ppm_samples(file, n, h, &p3, &view))) return rc;
    std::memcpy(dst, view, static_cast<size_t>(h.width) * h.height * 3);
    return JPGENC_OK;
}

int jpgenc_dct_quant_blocks(jpgenc_ctx* c, const float* dev_in, int16_t* dev_out, uint64_t nblocks, const uint8_t q[64],
                            uint64_t* refined_blocks) try {
    if (!c || !dev_in || !dev_out || !q || nblocks == 0 || nblocks > 0xFFFFFFFFull) return JPGENC_ERR_ARG;
    JPGENC_CUDA(c, cudaSetDevice(c->device));
    size_t cap_bytes = c->refine_cap * sizeof(uint32_t);
    int rc = ensure(c, &c->d_refine_list, &cap_bytes, nblocks * sizeof(uint32_t));
    c->refine_cap = cap_bytes / sizeof(uint32_t);
    if (rc) return rc;
    return launch_dct_quant_blocks(c, dev_in, dev_out, nblocks, q, refined_blocks);
} JPGENC_CATCH(c)

// One process per GPU on a multi-socket host: pixels that cross the socket interconnect on their way to the GPU share it with
// every other rank.  Restricting the calling thread to the CPUs of the GPU's NUMA node makes the pinned buffers it allocates
// afterwards node-local (first touch) and keeps the threads it starts there.
int jpgenc_bind_host_to_device_numa(int device, int* numa_node, int* cpus_bound) {
    if (numa_node) *numa_node = -1;
    if (cpus_bound) *cpus_bound = 0;
    char bus[32] = {0};
    if (cudaDeviceGetPCIBusId(bus, sizeof bus, device) != cudaSuccess) return JPGENC_ERR_CUDA;
    for (char* p = bus; *p; ++p) *p = static_cast<char>(std::tolower(static_cast<unsigned char>(*p)));
    int node = -1;
    {
        const std::string path = std::string("/sys/bus/pci/devices/") + bus + "/numa_node";
        std::FILE* f = std::fopen(path.c_str(), "r");
        if (!f) return JPGENC_OK;                                    // no topology information: nothing to do
        if (std::fscanf(f, "%d", &node) != 1) node = -1;
        std::fclose(f);
    }
    if (node < 0) return JPGENC_OK;
    cpu_set_t allowed, want;
    CPU_ZERO(&want);
    if (sched_getaffinity(0, sizeof allowed, &allowed) != 0) return JPGENC_OK;
    {
        const std::string path = "/sys/devices/system/node/node" + std::to_string(node) + "/cpulist";
        std::FILE* f = std::fopen(path.c_str(), "r");
        if (!f) return JPGENC_OK;
        int a = 0, b = 0, n = 0;
        for (;;) {                                                   // "0-15,32-47"
            if (std::fscanf(f, "%d", &a) != 1) break;
            b = a;
            int ch = std::fgetc(f);
            if (ch == '-') { if (std::fscanf(f, "%d", &b) != 1) break; ch = std::fgetc(f); }
            for (int k = a; k <= b && k < CPU_SETSIZE; ++k)
                if (CPU_ISSET(k, &allowed)) { CPU_SET(k, &want); ++n; }
            if (ch != ',') break;
        }
        std::fclose(f);
        if (n == 0) return JPGENC_OK;                                // the node's CPUs are not ours to use (cpuset): leave it
        if (sched_setaffinity(0, sizeof want, &want) != 0) return JPGENC_OK;
        if (cpus_bound) *cpus_bound = n;
    }
    if (numa_node) *numa_node = node;
    return JPGENC_OK;
}

// diagnostics for tests: word `index` of the context's device counters (common.cuh kCnt*), after a stream synchronisation
int jpgenc_debug_counter(jpgenc_ctx* c, int index, uint32_t* value) try {
    if (!c || !value || index < 0 || index >= kCounterWords) return JPGENC_ERR_ARG;
    JPGENC_CUDA(c, cudaStreamSynchronize(c->stream));
    JPGENC_CUDA(c, cudaMemcpy(value, c->d_counters + index, sizeof *value, cudaMemcpyDeviceToHost));
    return JPGENC_OK;
} JPGENC_CATCH(c)

int jpgenc_dev_alloc(jpgenc_ctx* c, size_t bytes, void** p) try {
    if (!c || !p) return JPGENC_ERR_ARG;
    JPGENC_CUDA(c, cudaSetDevice(c->device));
    JPGENC_CUDA(c, cudaMalloc(p, bytes));
    return JPGENC_OK;
} JPGENC_CATCH(c)
int jpgenc_dev_free(jpgenc_ctx* c, void* p) try {
    if (!c) return JPGENC_ERR_ARG;
    JPGENC_CUDA(c, cudaFree(p));
    return JPGENC_OK;
} JPGENC_CATCH(c)
int jpgenc_host_alloc_pinned(size_t bytes, void** p) { return cudaMallocHost(p, bytes) == cudaSuccess ? JPGENC_OK : JPGENC_ERR_CUDA; }
int jpgenc_host_free_pinned(void* p) { return cudaFreeHost(p) == cudaSuccess ? JPGENC_OK : JPGENC_ERR_CUDA; }
int jpgenc_memcpy_h2d(jpgenc_ctx* c, void* d, const void* h, size_t bytes) try {
    if (!c) return JPGENC_ERR_ARG;
    JPGENC_CUDA(c, cudaMemcpyAsync(d, h, bytes, cudaMemcpyHostToDevice, c->stream));
    JPGENC_CUDA(c, cudaStreamSynchronize(c->stream));
    return JPGENC_OK;
} JPGENC_CATCH(c)
int jpgenc_memcpy_d2h(jpgenc_ctx* c, void* h, const void* d, size_t bytes) try {
    if (!c) return JPGENC_ERR_ARG;
    JPGENC_CUDA(c, cudaMemcpyAsync(h, d, bytes, cudaMemcpyDeviceToHost, c->stream));
    JPGENC_CUDA(c, cudaStreamSynchronize(c->stream));
    return JPGENC_OK;
} JPGENC_CATCH(c)
int jpgenc_synth_rgb(jpgenc_ctx* c, void* dev_rgb, uint32_t w, uint32_t h, uint32_t seed) try {
    if (!c || !dev_rgb) return JPGENC_ERR_ARG;
    return launch_synth_rgb(c, static_cast<uint8_t*>(dev_rgb), w, h, seed);
} JPGENC_CATCH(c)
int jpgenc_synth_blocks(jpgenc_ctx* c, float* dev_blocks, uint64_t nblocks) try {
    if (!c || !dev_blocks) return JPGENC_ERR_ARG;
    return launch_synth_blocks(c, dev_blocks, nblocks);
} JPGENC_CATCH(c)
int jpgenc_flush_l2(jpgenc_ctx* c) try {
    if (!c) return JPGENC_ERR_ARG;
    if (!c->d_flush) {
        c->flush_bytes = 256ull << 20;                           // 2x the 126 MB L2
        JPGENC_CUDA(c, cudaMalloc(&c->d_flush, c->flush_bytes));
    }
    return launch_flush(c);
} JPGENC_CATCH(c)
int jpgenc_timer_begin(jpgenc_ctx* c) try {
    if (!c) return JPGENC_ERR_ARG;
    JPGENC_CUDA(c, cudaEventRecord(c->ev_u0, c->stream));
    return JPGENC_OK;
} JPGENC_CATCH(c)
int jpgenc_timer_end(jpgenc_ctx* c, float* ms) try {
    if (!c || !ms) return JPGENC_ERR_ARG;
    JPGENC_CUDA(c, cudaEventRecord(c->ev_u1, c->stream));
    JPGENC_CUDA(c, cudaEventSynchronize(c->ev_u1));
    JPGENC_CUDA(c, cudaEventElapsedTime(ms, c->ev_u0, c->ev_u1));
    return JPGENC_OK;
} JPGENC_CATCH(c)

}  // extern "C"
