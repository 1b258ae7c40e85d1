// Batches of equally sized frames: every pass (a slice of the batch) goes through ALL kernels as one asynchronous chain
//
//     K1 (+ exact refinement) -> K2 -> build_tables_kernel -> finalize_tables_kernel -> K3a -> K3b -> K4
//
// with no host step in between: the Huffman tables are built on the device (tables_device.cu), the sizes and offsets that
// follow from them are computed on the device (finalize.cu), K4 lays the complete files of the pass -- header, stuffed scan,
// EOI per frame -- back to back into one buffer, and ONE small device-to-host copy at the end of the chain tells the host
// what happened.  The host synchronises once per pass.
//
// What this replaces: a caller looping over Image::writeJPEG (src/Image.cpp:831-976) for a sequence of frames; every frame
// keeps its own DC prediction chains, its own four image-optimal tables and its own file (SURVEY.md 8e), results are
// byte-identical to encoding the frames one by one.
//
// Overlap.  A table build is a long, thin kernel (one working thread per table, ~0.2 ms for a 30-symbol alphabet whatever
// the number of frames); K1/K2/K3 are short and wide.  Passes therefore rotate over several SLOTS -- the context itself
// and lazily created further contexts on the same device, each with its own stream and buffers -- so that the table build
// of one pass runs beside the wide kernels of the others.  All slots are driven by the calling thread alone: per pass it
// enqueues about a dozen asynchronous operations and later waits for one event.  No worker threads, nothing spinning beside
// the caller -- eight such processes on a 32-core host do not compete for cores (the first design -- host-built tables,
// three lanes with a thread each, a pool of table builders -- was host-bound there: SCALE_r01 / VERDICT round 1).
#include <algorithm>
#include <cstring>
#include <vector>

#include "internal.hpp"
#include "../host/ppm_reader.hpp"

using namespace jpgenc;
using namespace jpgenc::detail;

namespace {

constexpr uint32_t kDefaultSlots = 4, kMaxSlots = 6;
constexpr uint32_t kMaxHeaderBytes = 2 + 18 + 2 * 69 + 19 + 4 * (21 + 256) + 14;   // SOI APP0 DQTx2 SOF0 DHTx4 SOS

struct Job {
    uint32_t n = 0;
    uint32_t w = 0, h = 0, maxval = 255;
    // images of individual sizes (jpgenc_encode_images_packed): image i is widths[i] x heights[i] (w x h: the first one's);
    // null: every frame is w x h
    const uint32_t* widths = nullptr;
    const uint32_t* heights = nullptr;
    // image i as the caller holds it (checked: pitches filled in), and the format the kernels take: -1 tight RGB, otherwise that
    // of every image (needs widths)
    std::vector<PixelSource> src;
    int format = -1;
    double raw_per_block = 0;              // ... raw-scan bytes reserved per block: 1.5 x the most this call has seen (0: nothing yet)
    // output: per-frame buffers (legacy), one packed buffer, or none (sizes only)
    uint8_t* const* out_ptrs = nullptr;
    const uint64_t* caps = nullptr;
    bool packed_mode = false;              // files back to back: offsets[] are reported, `packed` (may be null) receives them
    uint8_t* packed = nullptr;
    uint64_t packed_cap = 0, packed_at = 0;
    uint64_t* offsets = nullptr;
    uint64_t* sizes = nullptr;
};

struct Pass {
    uint32_t f0 = 0, F = 0;
    uint32_t k4_grid = 0;
    int attempts = 0;
};

uint32_t job_w(const Job& job, uint32_t i) { return job.widths ? job.widths[i] : job.w; }
uint32_t job_h(const Job& job, uint32_t i) { return job.heights ? job.heights[i] : job.h; }
uint64_t job_blocks(const Job& job, uint32_t i) {
    return static_cast<uint64_t>((job_w(job, i) + 15) / 16) * ((job_h(job, i) + 15) / 16) * kBlocksPerMcu;
}

// passes of `per_pass` frames (the last one may be shorter)
std::vector<Pass> uniform_passes(uint32_t n, uint32_t per_pass) {
    std::vector<Pass> pass((n + per_pass - 1) / per_pass);
    for (size_t p = 0; p < pass.size(); ++p) {
        pass[p].f0 = static_cast<uint32_t>(p) * per_pass;
        pass[p].F = std::min(per_pass, n - pass[p].f0);
    }
    return pass;
}

// the largest pass one slot can hold: item slabs (worst-case reservation, 96 KB per tile) within ~2 GB, block ids in 31 bits
uint32_t frames_per_pass_cap(const jpgenc_ctx* c) {
    const size_t nblocks = static_cast<size_t>(c->mcu_w) * c->mcu_h * kBlocksPerMcu, tiles = (nblocks + 383) / 384;
    size_t per_pass = std::max<size_t>(1, (2ull << 30) / (tiles * 384 * 64 * 4));
    per_pass = std::min<size_t>(per_pass, 0x7FFFFFFFull / nblocks);
    return static_cast<uint32_t>(std::min<size_t>(per_pass, 1024));
}

// Frames per pass.  A pass costs ~0.1 ms of launch gaps and one host wait whatever its size, its wide kernels run the better
// the larger they are, and its table build (~0.2 ms, independent of the number of frames) only hides behind OTHER passes' wide
// kernels: passes should be large, but a batch should still give every slot about two of them.  Measured on 1920x1080
// frames, 4 slots, device tables at 0.21 ms (frames per pass -> frames/s):
// 1024 frames: 64 -> 147 k, 128 -> 159 k, 256 -> 157 k;  128 frames: 32 -> 117 k, 64 -> 120 k, 128 -> 120 k.
uint32_t pass_frames(const jpgenc_ctx* c, uint32_t n, uint32_t slots) {
    const size_t px = static_cast<size_t>(c->mcu_w) * c->mcu_h * 256;
    const uint32_t lo = static_cast<uint32_t>(std::max<size_t>(1, (128u << 20) / px));    // ~128 Mpx: 64 frames of 1920x1080
    const uint32_t hi = static_cast<uint32_t>(std::max<size_t>(1, (256u << 20) / px));    // ~256 Mpx: 128 such frames
    uint32_t per = std::min(hi, std::max(lo, (n + 2 * slots - 1) / (2 * slots)));
    per = env_u32("JPGENC_FRAMES_PER_PASS", per);
    return std::max(1u, std::min({per, frames_per_pass_cap(c), n}));
}

// Images of individual sizes: the list is cut, in input order, into passes of the same pixel budget as pass_frames (MCU-padded
// pixels; ~128..256 Mpx, about two passes per slot) under the limits of frames_per_pass_cap (item slabs within ~2 GB, block
// ids in 31 bits, 1024 frames); JPGENC_FRAMES_PER_PASS bounds the images per pass.  An image that exceeds a limit alone
// gets a pass of its own.
std::vector<Pass> image_passes(const Job& job, uint32_t slots) {
    constexpr uint64_t kMaxSlabTiles = (2ull << 30) / (384 * 64 * 4), kMaxBlocks = 0x7FFFFFFFull;
    uint64_t total_px = 0;
    for (uint32_t i = 0; i < job.n; ++i) total_px += job_blocks(job, i) / kBlocksPerMcu * 256;
    const uint64_t target = std::min<uint64_t>(256ull << 20, std::max<uint64_t>(128ull << 20, (total_px + 2 * slots - 1) / (2 * slots)));
    const uint32_t max_frames = std::max(1u, std::min(1024u, env_u32("JPGENC_FRAMES_PER_PASS", 1024)));
    std::vector<Pass> pass;
    uint64_t px = 0, tiles = 0, blocks = 0;
    for (uint32_t i = 0; i < job.n; ++i) {
        const uint64_t b = job_blocks(job, i), t = (b + 383) / 384, x = b / kBlocksPerMcu * 256;
        if (pass.empty() || pass.back().F == max_frames || px + x > target || tiles + t > kMaxSlabTiles || blocks + b > kMaxBlocks) {
            pass.emplace_back();
            pass.back().f0 = i;
            px = tiles = blocks = 0;
        }
        ++pass.back().F;
        px += x; tiles += t; blocks += b;
    }
    return pass;
}

// The geometry of a pass of images of individual sizes (FrameGeom, F + 1 entries) and its totals.  K3's split follows
// launch_entropy's rule, applied to the pass's tiles.  FrameGeom holds each image's first plane and pitch; formats of several
// planes put the others in extra[f].
MixedPass image_geometry(const Job& job, const Pass& ps, const PixelSource* src, FrameGeom* g, ExtraPlanes* extra) {
    MixedPass m;
    m.on = true;
    m.aligned = true;
    m.format = job.format;
    uint64_t all_tiles = 0;
    for (uint32_t f = 0; f < ps.F; ++f) all_tiles += (job_blocks(job, ps.f0 + f) + 383) / 384;
    m.split = all_tiles < 4096 ? 4u : 1u;
    for (uint32_t f = 0; f <= ps.F; ++f) {
        g[f] = FrameGeom{};
        g[f].block0 = m.blocks; g[f].strip0 = m.strips; g[f].tile0 = m.tiles; g[f].group0 = m.groups; g[f].super0 = m.supers;
        if (f == ps.F) break;
        const uint32_t w = job_w(job, ps.f0 + f), h = job_h(job, ps.f0 + f);
        g[f].rgb = src[f].plane[0];
        if (source_planes(job.format) == 3) extra[f] = ExtraPlanes{{src[f].plane[1], src[f].plane[2]}, src[f].pitch2};
        g[f].real_w = w; g[f].real_h = h; g[f].mcu_w = (w + 15) / 16; g[f].mcu_h = (h + 15) / 16;
        if (job.format >= 0) g[f].pitch = src[f].pitch;
        const uint32_t blocks = g[f].mcu_w * g[f].mcu_h * kBlocksPerMcu, tiles = (blocks + 383) / 384, groups = (tiles * m.split + 7) / 8;
        m.blocks += blocks;
        m.strips += (g[f].mcu_w + 31) / 32 * g[f].mcu_h;
        m.tiles += tiles;
        m.groups += groups;
        m.supers += (groups + 255) / 256;
        m.aligned = m.aligned && w % 16 == 0 && reinterpret_cast<uintptr_t>(g[f].rgb) % 16 == 0;
    }
    return m;
}

int prepare_slot(jpgenc_ctx* root, jpgenc_ctx* l, const Job& job, const uint8_t* prefix, uint32_t prefix_len) {
    if (l != root) {
        std::memcpy(l->qy, root->qy, 64); std::memcpy(l->qc, root->qc, 64);
        std::memcpy(l->dct_a, root->dct_a, sizeof root->dct_a); std::memcpy(l->dct_s, root->dct_s, sizeof root->dct_s);
    }
    int rc = set_geometry(l, job.w, job.h, job.maxval);
    if (rc) return rc;
    if (!l->d_hdr_prefix) JPGENC_CUDA(l, cudaMalloc(reinterpret_cast<void**>(&l->d_hdr_prefix), 256));
    if (l->hdr_prefix_len != prefix_len || std::memcmp(l->hdr_prefix_host, prefix, prefix_len) != 0) {   // new size or quantisers
        JPGENC_CUDA(l, cudaMemcpyAsync(l->d_hdr_prefix, prefix, prefix_len, cudaMemcpyHostToDevice, l->stream));
        JPGENC_CUDA(l, cudaStreamSynchronize(l->stream));      // `prefix` lives on the caller's stack
        std::memcpy(l->hdr_prefix_host, prefix, prefix_len);
        l->hdr_prefix_len = prefix_len;
    }
    if (!l->ev_done) JPGENC_CUDA(l, cudaEventCreateWithFlags(&l->ev_done, cudaEventDisableTiming));
    if (!l->ev_fwd) JPGENC_CUDA(l, cudaEventCreateWithFlags(&l->ev_fwd, cudaEventDisableTiming));
    if (!l->ev_k4) JPGENC_CUDA(l, cudaEventCreateWithFlags(&l->ev_k4, cudaEventDisableTiming));
    if (!l->ev_copied) JPGENC_CUDA(l, cudaEventCreateWithFlags(&l->ev_copied, cudaEventDisableTiming));
    if (!l->out_stream) JPGENC_CUDA(l, cudaStreamCreateWithFlags(&l->out_stream, cudaStreamNonBlocking));
    l->copy_pending = false;
    return JPGENC_OK;
}

// K3/K4 of a pass: buffers for the limits, finalize (tables -> lookup form, sizes, offsets), K3a, K3b, K4, read-back
int enqueue_entropy(jpgenc_ctx* l, Pass& ps, cudaEvent_t prev_k4 = nullptr) {
    const uint32_t F = ps.F;
    int rc;
    const uint64_t k4_grid = l->raw_limit / kK4TileBytes + F;
    if ((rc = ensure_entropy_buffers(l, l->raw_limit, l->out_limit, k4_grid))) return rc;
    ps.k4_grid = static_cast<uint32_t>(k4_grid);
    if (l->copy_pending) {                                     // the previous pass's files are still leaving d_scan
        JPGENC_CUDA(l, cudaStreamWaitEvent(l->stream, l->ev_copied, 0));
        l->copy_pending = false;
    }
    if ((rc = launch_finalize_tables(l))) return rc;
    // K3/K4 of the passes run one pass after the other (each of them fills the GPU anyway): the passes then FINISH one
    // after the other and the files of pass p travel while pass p + 1 is packed, instead of all slots' files queueing up
    // behind the last kernel (trace of 4 slots in step: 4 x 11 MB = 0.8 ms of copies after the last K4)
    if (prev_k4) JPGENC_CUDA(l, cudaStreamWaitEvent(l->stream, prev_k4, 0));
    if ((rc = launch_entropy(l, ps.k4_grid))) return rc;
    JPGENC_CUDA(l, cudaEventRecord(l->ev_k4, l->stream));
    uint8_t* h = static_cast<uint8_t*>(l->h_pinned) + stage_meta_off(F);
    JPGENC_CUDA(l, cudaMemcpyAsync(h, l->d_meta, pass_meta_bytes(F), cudaMemcpyDeviceToHost, l->stream));
    JPGENC_CUDA(l, cudaEventRecord(l->ev_done, l->stream));
    ++ps.attempts;
    return JPGENC_OK;
}

// the whole chain of one pass on slot `l` over the device images src[0 .. F); `ready` (optional): event after which the pixels are
// valid; `after` (optional): the event after the previous pass's K1 (see run_passes)
int enqueue_pass(jpgenc_ctx* root, jpgenc_ctx* l, const Job& job, Pass& ps, const PixelSource* src, cudaEvent_t ready, cudaEvent_t after,
                 cudaEvent_t prev_k4) {
    const uint32_t F = ps.F;
    int rc;
    l->nframes = F;
    l->have_coef = l->have_scan = l->have_items = false; l->k2_tiles_done = 0;
    l->file_mode = true;
    bool aligned = true;
    for (uint32_t f = 0; f < F; ++f) aligned = aligned && (reinterpret_cast<uintptr_t>(src[f].plane[0]) % 16 == 0);
    l->frames_aligned = aligned;
    l->src.plane[0] = src[0].plane[0];
    l->have_pixels = true;
    std::vector<FrameGeom> geom;
    std::vector<ExtraPlanes> extra;
    if (job.widths) {
        geom.resize(F + 1);
        extra.resize(source_planes(job.format) == 3 ? F : 0);
        l->mixed = image_geometry(job, ps, src, geom.data(), extra.data());
    }
    if ((rc = ensure_coef(l))) return rc;
    if ((rc = ensure_stats_buffers(l))) return rc;               // also sizes the pinned staging (stage_bytes(F))
    if (job.widths) {
        // the geometry (with the frame pointers, and the extra planes behind it) travels through pinned memory like the pointer
        // array below
        const size_t gbytes = geom.size() * sizeof(FrameGeom), bytes = gbytes + extra.size() * sizeof(ExtraPlanes);
        if ((rc = ensure(l, &l->d_geom, &l->geom_cap, bytes))) return rc;
        std::memcpy(l->h_pinned, geom.data(), gbytes);
        if (!extra.empty()) std::memcpy(static_cast<uint8_t*>(l->h_pinned) + gbytes, extra.data(), extra.size() * sizeof(ExtraPlanes));
        JPGENC_CUDA(l, cudaMemcpyAsync(l->d_geom, l->h_pinned, bytes, cudaMemcpyHostToDevice, l->stream));
    } else {
        size_t cap = l->frame_ptrs_cap;
        void* p = l->d_frame_ptrs;
        if ((rc = ensure(l, reinterpret_cast<uint8_t**>(&p), &cap, F * sizeof(void*)))) return rc;
        l->d_frame_ptrs = static_cast<const uint8_t**>(p);
        l->frame_ptrs_cap = cap;
        // the pointer array travels through pinned memory (the statistics' staging area is unused in this path), so that the
        // copy is asynchronous and the caller's array need not outlive the call
        const uint8_t** ptrs = static_cast<const uint8_t**>(l->h_pinned);
        for (uint32_t f = 0; f < F; ++f) ptrs[f] = src[f].plane[0];
        JPGENC_CUDA(l, cudaMemcpyAsync(l->d_frame_ptrs, l->h_pinned, F * sizeof(void*), cudaMemcpyHostToDevice, l->stream));
    }
    if (ready) JPGENC_CUDA(l, cudaStreamWaitEvent(l->stream, ready, 0));
    if (after) JPGENC_CUDA(l, cudaStreamWaitEvent(l->stream, after, 0));
    if ((rc = job.widths ? launch_forward_mixed(l) : launch_forward_rows(l, 0, l->mcu_h, true, true))) return rc;   // K1 + exact refinement
    l->have_coef = true;
    JPGENC_CUDA(l, cudaEventRecord(l->ev_fwd, l->stream));
    const size_t nblocks = static_cast<size_t>(l->mcu_w) * l->mcu_h * kBlocksPerMcu, tiles = (nblocks + 383) / 384;
    if ((rc = launch_symbol_stats(l, 0, job.widths ? l->mixed.tiles : static_cast<uint32_t>(tiles * F), true))) return rc;     // K2
    l->have_items = true;
    const uint32_t nt = 4 * F;
    if ((rc = ensure(l, reinterpret_cast<uint8_t**>(&l->d_tab_scratch), &l->tab_scratch_cap, nt * table_scratch_bytes()))) return rc;
    if ((rc = ensure(l, &l->d_built_tables, &l->built_tables_cap, nt * (sizeof(jpgenc_huff_table) + sizeof(uint32_t))))) return rc;
    if ((rc = launch_build_tables(l, l->d_stats, static_cast<uint32_t>(kStatsBytes), nt, l->d_tab_scratch, l->d_built_tables,
                                  reinterpret_cast<uint32_t*>(l->d_built_tables + nt)))) return rc;
    // how much raw scan / output the pass may use: 1.5 x the largest frame the batch has produced so far
    // (root->batch_raw_per_frame), before the first pass has finished a guess of 12 bytes per block; a pass that needs more
    // is refused by finalize_tables_kernel and its entropy stage re-run with what it asked for (finish_pass)
    // (JPGENC_RAW_GUESS_PER_BLOCK: tests set it to 0 so that every first pass is refused and re-run)
    // (images of individual sizes: the same per block -- 12 bytes, then 1.5 x the most bytes per block this call has seen)
    if (job.widths) {
        const double per_block = job.raw_per_block ? job.raw_per_block : env_u32("JPGENC_RAW_GUESS_PER_BLOCK", 12);
        l->raw_limit = 0;
        for (uint32_t f = 0; f < F; ++f) l->raw_limit += raw_slot_bytes(static_cast<uint64_t>((geom[f + 1].block0 - geom[f].block0) * per_block) + 4096);
    } else {
        const uint64_t per_frame = root->batch_raw_per_frame ? root->batch_raw_per_frame : nblocks * env_u32("JPGENC_RAW_GUESS_PER_BLOCK", 12) + 4096;
        l->raw_limit = F * raw_slot_bytes(per_frame);
    }
    l->out_limit = F * (kMaxHeaderBytes + 2ull) + 2 * l->raw_limit;
    ps.attempts = 0;
    return enqueue_entropy(l, ps, prev_k4);
}

// waits for the pass on slot `l`, re-runs its entropy stage with larger buffers if it was refused, reports sizes and sends
// the files on their way to the caller's memory (the copies are enqueued on the slot's stream; the caller of run_passes
// synchronises all slots at the end)
int finish_pass(jpgenc_ctx* root, jpgenc_ctx* l, Pass& ps, Job& job) {
    const uint32_t F = ps.F;
    for (;;) {
        JPGENC_CUDA(l, cudaEventSynchronize(l->ev_done));
        const PassMeta m = pass_meta_view(static_cast<uint8_t*>(l->h_pinned) + stage_meta_off(F), F);
        const PassHeader& hd = *m.hdr;
        if (hd.nframes != F) return fail(l, JPGENC_ERR_CUDA, "batched pass: the device left no result");
        if (hd.error & kPassMissingSymbol) return fail(l, JPGENC_ERR_ARG, "Huffman table lacks a symbol that occurs in the image");
        if (hd.error & kPassNoSymbols) return fail(l, JPGENC_ERR_ARG, "Huffman table build failed: a table has no symbol");
        if (hd.error & (kPassRawOverflow | kPassOutOverflow)) {
            if (ps.attempts >= 3) return fail(l, JPGENC_ERR_CUDA, "batched pass: scan buffers still too small after two retries");
            // finalize computed the full requirement before refusing: reserve that (plus a margin) and run K3/K4 again --
            // coefficients, symbol items and tables are still on the device
            l->raw_limit = hd.raw_total + hd.raw_total / 8 + 4096;
            l->out_limit = F * (kMaxHeaderBytes + 2ull) + 2 * l->raw_limit;
            const int rc = enqueue_entropy(l, ps);
            if (rc) return rc;
            continue;
        }
        uint64_t max_raw = 0;
        double max_per_block = 0;
        for (uint32_t f = 0; f < F; ++f) {
            if (m.total_bits[f] != m.frame_bits[f]) {
                l->error = "entropy coder wrote " + std::to_string(m.total_bits[f]) + " bits, statistics predicted " + std::to_string(m.frame_bits[f]);
                return JPGENC_ERR_ARG;
            }
            max_raw = std::max<uint64_t>(max_raw, m.raw_bytes[f]);
            if (job.widths) max_per_block = std::max(max_per_block, static_cast<double>(m.raw_bytes[f]) / job_blocks(job, ps.f0 + f));
        }
        // later passes reserve 1.5 x the largest frame (images of individual sizes: bytes per block) seen so far
        if (job.widths) job.raw_per_block = std::max(job.raw_per_block, 1.5 * max_per_block);
        else root->batch_raw_per_frame = std::max<uint64_t>(root->batch_raw_per_frame, max_raw + max_raw / 2 + 4096);
        const uint64_t total = hd.out_total + m.ff_incl[F - 1];
        // The files go home on the slot's OUTPUT stream (behind ev_done, i.e. behind K4), so that the slot's next pass can
        // start its K1/K2/table build meanwhile; only its K3/K4, which overwrite d_scan, wait for the copy (enqueue_entropy).
        uint64_t base = 0;
        const bool copies = job.packed || job.out_ptrs;
        if (copies) JPGENC_CUDA(l, cudaStreamWaitEvent(l->out_stream, l->ev_done, 0));
        if (job.packed_mode) {                                       // passes finish in order: the files end up in frame order
            base = job.packed_at;
            job.packed_at += total;
            if (job.packed) {
                if (job.packed_at > job.packed_cap) return fail(l, JPGENC_ERR_CAPACITY, "JPEG buffer too small");
                JPGENC_CUDA(l, cudaMemcpyAsync(job.packed + base, l->d_scan, total, cudaMemcpyDeviceToHost, l->out_stream));
            }
        }
        for (uint32_t f = 0; f < F; ++f) {
            const uint64_t before = f ? m.ff_incl[f - 1] : 0;
            const uint64_t off = m.file_base[f] + before;
            const uint64_t size = m.hdr_len[f] + m.raw_bytes[f] + (m.ff_incl[f] - before) + 2;
            job.sizes[ps.f0 + f] = size;
            if (job.offsets) job.offsets[ps.f0 + f] = base + off;
            if (job.out_ptrs) {
                if (job.caps[ps.f0 + f] < size) return fail(l, JPGENC_ERR_CAPACITY, "JPEG buffer too small");
                JPGENC_CUDA(l, cudaMemcpyAsync(job.out_ptrs[ps.f0 + f], l->d_scan + off, size, cudaMemcpyDeviceToHost, l->out_stream));
            }
        }
        if (copies) {
            JPGENC_CUDA(l, cudaEventRecord(l->ev_copied, l->out_stream));
            l->copy_pending = true;
        }
        return JPGENC_OK;
    }
}

// Runs the passes over the slots.  frames_of(p, slot context) -> device sources of pass p's images and the event after which
// they are valid; done_with(p) is called when pass p's pixels are no longer needed.
template <class FramesOf, class DoneWith>
int run_passes(jpgenc_ctx* c, Job& job, std::vector<Pass>& pass, uint32_t nslots, FramesOf&& frames_of, DoneWith&& done_with) {
    const uint32_t npasses = static_cast<uint32_t>(pass.size());
    // SOI .. SOF0 are the same bytes for every frame of the batch: jpgenc_write_headers with empty tables gives
    // prefix + 4 x (DHT with no symbol: 21 bytes) + SOS (14 bytes).  (Images of individual sizes: the first image's size
    // stands in SOF0; K4 writes every image's own.)
    uint8_t hdr[512];
    jpgenc_huff_table empty[4];
    std::memset(empty, 0, sizeof empty);
    const size_t hdr_all = jpgenc_write_headers(job.w, job.h, c->qy, c->qc, empty, hdr);
    const uint32_t prefix_len = static_cast<uint32_t>(hdr_all - 4 * 21 - 14);
    int rc;
    while (c->lanes.size() + 1 < nslots) {
        jpgenc_ctx* l = nullptr;
        if ((rc = jpgenc_create(c->device, &l))) return fail(c, rc, jpgenc_last_error(nullptr));
        c->lanes.push_back(l);
    }
    std::vector<jpgenc_ctx*> slot(nslots);
    for (uint32_t k = 0; k < nslots; ++k) {
        slot[k] = k ? c->lanes[k - 1] : c;
        if ((rc = prepare_slot(c, slot[k], job, hdr, prefix_len))) return k ? fail(c, rc, jpgenc_last_error(slot[k])) : rc;
    }
    // The streams run side by side, except in a call of exactly two passes: there nothing else will ever run beside the table
    // builds, and letting pass 1's K1 start when pass 0's K1 is through puts pass 0's table build beside pass 1's wide kernels
    // (timeline, 128 frames: 1.057 -> 1.014 ms).  Staggering more passes does not pay: 256 and 1024 frames are 2-4 % slower
    // that way, and making every pass wait for the previous pass's K2 took 128 frames 1.26 -> 1.33 ms, 1024 frames 6.9 -> 7.2 ms
    // -- the cross-stream waits cost more than the earlier table builds gain.
    const bool stagger = npasses == 2 && nslots > 1;
    rc = JPGENC_OK;
    jpgenc_ctx* failed = nullptr;
    for (uint32_t p = 0; p < npasses + nslots && rc == JPGENC_OK; ++p) {
        if (p >= nslots) {                                          // the slot's previous pass: results, files, slot free again
            const uint32_t q = p - nslots;
            jpgenc_ctx* l = slot[q % nslots];
            rc = finish_pass(c, l, pass[q], job);
            if (rc) { failed = l; break; }
            done_with(q);
        }
        if (p < npasses) {
            jpgenc_ctx* l = slot[p % nslots];
            const PixelSource* ptrs = nullptr;
            cudaEvent_t ready = nullptr;
            rc = frames_of(p, l, &ptrs, &ready);
            // Staggering: the wide kernels of pass p start when pass p - 1's K1 is through.  Left alone, the streams run the
            // same stage of all passes side by side, every table build then starts at the same (late) moment and nothing wide
            // is left to run beside it.
            cudaEvent_t after = (stagger && p > 0) ? slot[(p - 1) % nslots]->ev_fwd : nullptr;
            // (only when files travel back: sizes-only calls are 2-5 % faster with the slots' K3/K4 side by side.  Measured,
            // 1024 frames, in order / not: files returned 6.61 / 7.00 ms, sizes only 6.30 / 6.20 ms)
            const bool in_order = job.packed != nullptr || job.out_ptrs != nullptr;
            cudaEvent_t prev_k4 = (in_order && p > 0 && nslots > 1) ? slot[(p - 1) % nslots]->ev_k4 : nullptr;
            if (rc == JPGENC_OK) rc = enqueue_pass(c, l, job, pass[p], ptrs, ready, after, prev_k4);
            if (rc) { failed = l; break; }
        }
    }
    // the files' copies are still in flight; also after a failure: nothing may run once the caller's buffers are gone
    for (uint32_t k = 0; k < nslots; ++k) {
        cudaError_t e = cudaStreamSynchronize(slot[k]->stream);
        if (e == cudaSuccess && slot[k]->out_stream) e = cudaStreamSynchronize(slot[k]->out_stream);
        slot[k]->copy_pending = false;
        if (e != cudaSuccess && rc == JPGENC_OK) { rc = JPGENC_ERR_CUDA; c->error = std::string("batched pass: ") + cudaGetErrorString(e); }
    }
    if (failed && failed != c) c->error = failed->error;
    for (uint32_t k = 1; k < nslots; ++k) {
        c->launches += slot[k]->launches;
        slot[k]->launches = 0;
        leave_batch_state(slot[k]);
    }
    leave_batch_state(c);
    return rc;
}

uint32_t slots_for(size_t npasses) {
    uint32_t s = env_u32("JPGENC_SLOTS", kDefaultSlots);
    return std::max(1u, static_cast<uint32_t>(std::min<size_t>({s, kMaxSlots, npasses})));
}

// the passes of a call: equal frames in passes of pass_frames() frames, images of individual sizes by image_passes()
std::vector<Pass> plan_passes(const jpgenc_ctx* c, const Job& job) {
    const uint32_t nslots0 = std::max(1u, std::min(kMaxSlots, env_u32("JPGENC_SLOTS", kDefaultSlots)));
    return job.widths ? image_passes(job, nslots0) : uniform_passes(job.n, pass_frames(c, job.n, nslots0));
}

int check_job(jpgenc_ctx* c, const Job& job, const void* frames) {
    if (!c || !frames || !job.sizes) return JPGENC_ERR_ARG;
    if (job.out_ptrs && !job.caps) return JPGENC_ERR_ARG;
    if (job.packed_mode && !job.offsets) return JPGENC_ERR_ARG;
    return JPGENC_OK;
}

int encode_device_frames(jpgenc_ctx* c, Job& job) {
    // an empty batch is legal and touches nothing: an image bound to the context keeps its geometry
    if (job.n == 0) return (job.w && job.h && job.maxval && job.maxval <= 255) ? JPGENC_OK : fail(c, JPGENC_ERR_ARG, "width/height/maxval out of range");
    JPGENC_CUDA(c, cudaSetDevice(c->device));
    int rc = set_geometry(c, job.w, job.h, job.maxval);
    if (rc) return rc;
    // what earlier calls learnt about the size of such frames' scans stays valid (a later frame that needs more is refused on the
    // device and re-run, finish_pass); a new frame size starts from the guess again
    if (!job.widths && (c->batch_geom_w != job.w || c->batch_geom_h != job.h)) { c->batch_raw_per_frame = 0; c->batch_geom_w = job.w; c->batch_geom_h = job.h; }
    std::vector<Pass> pass = plan_passes(c, job);
    const uint32_t nslots = slots_for(pass.size());
    return run_passes(c, job, pass, nslots,
                      [&](uint32_t p, jpgenc_ctx*, const PixelSource** src, cudaEvent_t* ready) {
                          *src = job.src.data() + pass[p].f0;
                          *ready = nullptr;
                          return JPGENC_OK;
                      },
                      [](uint32_t) {});
}

// Frames in host memory (pinned for full PCIe speed): they travel on the copy stream into a ring of pass-sized slices
// of device memory, always a few passes ahead of the kernels; when pass p is finished its slice is re-filled with the
// frames of pass p + ring.  A slice holds the bytes of the largest pass (passes of images of individual sizes differ);
// every frame starts on 256 bytes.  Pixels in another layout travel in their own format, the pitch gap dropped by the copy.
int encode_host_frames(jpgenc_ctx* c, Job& job) {
    // an empty batch is legal and touches nothing: an image bound to the context keeps its geometry
    if (job.n == 0) return (job.w && job.h && job.maxval && job.maxval <= 255) ? JPGENC_OK : fail(c, JPGENC_ERR_ARG, "width/height/maxval out of range");
    JPGENC_CUDA(c, cudaSetDevice(c->device));
    int rc = set_geometry(c, job.w, job.h, job.maxval);
    if (rc) return rc;
    // what earlier calls learnt about the size of such frames' scans stays valid (a later frame that needs more is refused on the
    // device and re-run, finish_pass); a new frame size starts from the guess again
    if (!job.widths && (c->batch_geom_w != job.w || c->batch_geom_h != job.h)) { c->batch_raw_per_frame = 0; c->batch_geom_w = job.w; c->batch_geom_h = job.h; }
    std::vector<Pass> pass = plan_passes(c, job);
    const uint32_t nslots = slots_for(pass.size());
    const uint32_t npasses = static_cast<uint32_t>(pass.size());
    constexpr uint32_t kRingMax = sizeof(c->ev_band) / sizeof(c->ev_band[0]);
    const uint32_t ring = std::min({nslots + 2, npasses, kRingMax});
    // image i: its planes as they are uploaded (staged_planes), at slice (p % ring) + at[i] of the ring
    std::vector<StagedPlane> pl(3 * static_cast<size_t>(job.n));
    std::vector<uint32_t> np(job.n);
    std::vector<size_t> at(job.n);
    auto fstride = [&](uint32_t i) { return (staged_bytes(&pl[3 * i], np[i]) + 255) & ~static_cast<size_t>(255); };
    size_t slice = 0;
    for (const Pass& ps : pass) {
        size_t o = 0;
        for (uint32_t i = ps.f0; i < ps.f0 + ps.F; ++i) {
            np[i] = staged_planes(job.src[i], job_w(job, i), job_h(job, i), &pl[3 * i]);
            at[i] = o;
            o += fstride(i);
        }
        slice = std::max(slice, o);
    }
    if ((rc = ensure(c, &c->d_rgb_owned, &c->rgb_cap, static_cast<size_t>(ring) * slice + 16))) return rc;
    auto upload = [&](uint32_t p) -> int {
        const uint32_t f0 = pass[p].f0, F = pass[p].F, s = p % ring;
        for (uint32_t f = 0; f < F;) {
            const uint32_t i = f0 + f;
            const StagedPlane* q = &pl[3 * i];
            uint8_t* dst = c->d_rgb_owned + static_cast<size_t>(s) * slice + at[i];
            // equal frames that follow each other in host memory (a video buffer) travel as one strided copy
            const size_t fbytes = staged_bytes(q, np[i]);
            uint32_t run = 1;
            while (!job.widths && f + run < F && job.src[i + run].plane[0] == job.src[i + run - 1].plane[0] + fbytes) ++run;
            if (run > 1) {
                JPGENC_CUDA(c, cudaMemcpy2DAsync(dst, fstride(i), q[0].host, fbytes, fbytes, run, cudaMemcpyHostToDevice, c->copy_stream));
            } else if (const size_t gap = planes_gap(q, np[i])) {
                JPGENC_CUDA(c, cudaMemcpy2DAsync(dst, q[1].dev_off, q[0].host, gap, q[1].dev_off, np[i], cudaMemcpyHostToDevice, c->copy_stream));
            } else {
                for (uint32_t k = 0; k < np[i]; ++k) {
                    if (q[k].pitch == q[k].row)
                        JPGENC_CUDA(c, cudaMemcpyAsync(dst + q[k].dev_off, q[k].host, q[k].row * q[k].rows, cudaMemcpyHostToDevice, c->copy_stream));
                    else
                        JPGENC_CUDA(c, cudaMemcpy2DAsync(dst + q[k].dev_off, q[k].row, q[k].host, q[k].pitch, q[k].row, q[k].rows, cudaMemcpyHostToDevice,
                                                         c->copy_stream));
                }
            }
            f += run;
        }
        JPGENC_CUDA(c, cudaEventRecord(c->ev_band[s], c->copy_stream));
        return JPGENC_OK;
    };
    for (uint32_t p = 0; p < ring; ++p)
        if ((rc = upload(p))) return rc;
    std::vector<std::vector<PixelSource>> staged(nslots);
    int upload_rc = JPGENC_OK;
    rc = run_passes(c, job, pass, nslots,
                    [&](uint32_t p, jpgenc_ctx*, const PixelSource** out, cudaEvent_t* ready) {
                        const uint32_t f0 = pass[p].f0, F = pass[p].F, s = p % ring;
                        std::vector<PixelSource>& v = staged[p % nslots];
                        v.resize(F);
                        for (uint32_t f = 0; f < F; ++f) {
                            const StagedPlane* q = &pl[3 * (f0 + f)];
                            v[f] = job.src[f0 + f];
                            for (uint32_t k = 0; k < 3; ++k)
                                v[f].plane[k] = k < np[f0 + f] ? c->d_rgb_owned + static_cast<size_t>(s) * slice + at[f0 + f] + q[k].dev_off : nullptr;
                            v[f].pitch = static_cast<uint32_t>(q[0].row);
                            if (np[f0 + f] > 1) v[f].pitch2 = static_cast<uint32_t>(q[1].row);
                        }
                        *out = v.data();
                        *ready = c->ev_band[s];
                        return JPGENC_OK;
                    },
                    [&](uint32_t q) {
                        // every kernel of pass q has finished (its event is behind K4): the slice is free again.  The copy
                        // stream must not overtake the kernels that still read it -- it does not: they are done.
                        if (q + ring < npasses && upload_rc == JPGENC_OK) upload_rc = upload(q + ring);
                    });
    if (rc == JPGENC_OK) rc = upload_rc;
    const cudaError_t e = cudaStreamSynchronize(c->copy_stream);
    if (e != cudaSuccess && rc == JPGENC_OK) rc = fail(c, JPGENC_ERR_CUDA, "host-to-device copy of a frame failed");
    c->src.plane[0] = c->d_rgb_owned;
    return rc;
}

// equal tight RGB frames of one call (the pointers are not checked one by one)
void rgb_frames(Job& job, const void* const* frames) {
    job.src.resize(job.n);
    for (uint32_t i = 0; i < job.n; ++i) job.src[i] = image_source(frames[i], job.w * 3, JPGENC_PIXEL_RGB);
}

// The packed calls: images of individual sizes in any source.  Every source is checked (from host memory: its samples against
// maxval too).  Tight RGB takes the kernels of tight RGB, and when every image has one size, the batched-frame path as it is.
int encode_packed(jpgenc_ctx* c, std::vector<PixelSource>& src, int images_on_device, const uint32_t* widths, const uint32_t* heights,
                  uint32_t maxval, uint8_t* out, uint64_t cap, uint64_t* offsets, uint64_t* sizes, uint64_t* total_bytes) {
    const uint32_t n = static_cast<uint32_t>(src.size());
    bool same = true, tight_rgb = true;
    for (uint32_t i = 0; i < n; ++i) {
        const int rc = check_source(c, &src[i], widths[i], heights[i]);
        if (rc) return rc;
        same = same && widths[i] == widths[0] && heights[i] == heights[0];
        tight_rgb = tight_rgb && src[i].format == JPGENC_PIXEL_RGB && src[i].pitch == widths[i] * 3;
    }
    if (!images_on_device)
        for (uint32_t i = 0; i < n; ++i)
            if (!source_within_maxval(src[i], widths[i], heights[i], maxval)) return fail(c, JPGENC_ERR_FORMAT, "a sample exceeds maxval");
    Job job;
    job.n = n; job.w = widths[0]; job.h = heights[0]; job.maxval = maxval;
    if (!tight_rgb || !same) { job.widths = widths; job.heights = heights; }   // the pass pipeline of images of individual sizes
    job.format = tight_rgb ? -1 : src[0].format;
    job.src = std::move(src);
    job.packed_mode = true; job.packed = out; job.packed_cap = cap; job.offsets = offsets; job.sizes = sizes;
    const int rc = images_on_device ? encode_device_frames(c, job) : encode_host_frames(c, job);
    if (total_bytes) *total_bytes = job.packed_at;
    return rc;
}

}  // namespace

extern "C" {

int jpgenc_encode_frames_device(jpgenc_ctx* c, uint32_t n, const void* const* dev_frames, uint32_t w, uint32_t h, uint32_t maxval,
                                uint8_t* const* out, const uint64_t* caps, uint64_t* sizes) try {
    Job job;
    job.n = n; job.w = w; job.h = h; job.maxval = maxval;
    job.out_ptrs = out; job.caps = caps; job.sizes = sizes;
    const int rc = check_job(c, job, dev_frames);
    if (rc) return rc;
    rgb_frames(job, dev_frames);
    return encode_device_frames(c, job);
} JPGENC_CATCH(c)

int jpgenc_encode_frames(jpgenc_ctx* c, uint32_t n, const uint8_t* const* frames, uint32_t w, uint32_t h, uint32_t maxval,
                         uint8_t* const* out, const uint64_t* caps, uint64_t* sizes) try {
    Job job;
    job.n = n; job.w = w; job.h = h; job.maxval = maxval;
    job.out_ptrs = out; job.caps = caps; job.sizes = sizes;
    const int rc = check_job(c, job, frames);
    if (rc) return rc;
    rgb_frames(job, reinterpret_cast<const void* const*>(frames));
    return encode_host_frames(c, job);
} JPGENC_CATCH(c)

int jpgenc_encode_frames_packed(jpgenc_ctx* c, uint32_t n, const void* const* frames, int frames_on_device, uint32_t w, uint32_t h,
                                uint32_t maxval, uint8_t* out, uint64_t cap, uint64_t* offsets, uint64_t* sizes, uint64_t* total_bytes) try {
    Job job;
    job.n = n; job.w = w; job.h = h; job.maxval = maxval;
    job.packed_mode = true; job.packed = out; job.packed_cap = cap; job.offsets = offsets; job.sizes = sizes;
    int rc = check_job(c, job, frames);
    if (rc) return rc;
    rgb_frames(job, frames);
    rc = frames_on_device ? encode_device_frames(c, job) : encode_host_frames(c, job);
    if (total_bytes) *total_bytes = job.packed_at;
    return rc;
} JPGENC_CATCH(c)

int jpgenc_encode_images_packed(jpgenc_ctx* c, uint32_t n, const void* const* images, int images_on_device, const uint32_t* widths,
                                const uint32_t* heights, uint32_t maxval, uint8_t* out, uint64_t cap, uint64_t* offsets, uint64_t* sizes,
                                uint64_t* total_bytes) try {
    if (!c) return JPGENC_ERR_ARG;
    if (total_bytes) *total_bytes = 0;
    if (maxval == 0 || maxval > 255) return fail(c, JPGENC_ERR_ARG, "maxval out of range");
    if (n == 0) return JPGENC_OK;                                // an empty batch is legal and touches nothing
    if (!images || !widths || !heights || !offsets || !sizes) return fail(c, JPGENC_ERR_ARG, "null argument");
    std::vector<PixelSource> src(n);
    for (uint32_t i = 0; i < n; ++i) src[i] = image_source(images[i], 0, JPGENC_PIXEL_RGB);
    return encode_packed(c, src, images_on_device, widths, heights, maxval, out, cap, offsets, sizes, total_bytes);
} JPGENC_CATCH(c)

int jpgenc_encode_images_packed_layout(jpgenc_ctx* c, uint32_t n, const void* const* images, int images_on_device, const uint32_t* widths,
                                       const uint32_t* heights, const uint32_t* row_pitches, int format, uint32_t maxval, uint8_t* out,
                                       uint64_t cap, uint64_t* offsets, uint64_t* sizes, uint64_t* total_bytes) try {
    if (!c) return JPGENC_ERR_ARG;
    if (total_bytes) *total_bytes = 0;
    if (image_source(nullptr, 0, format).format < 0) return fail(c, JPGENC_ERR_ARG, "unknown pixel format");
    if (maxval == 0 || maxval > 255) return fail(c, JPGENC_ERR_ARG, "maxval out of range");
    if (n == 0) return JPGENC_OK;                                // an empty batch is legal and touches nothing
    if (!images || !widths || !heights || !offsets || !sizes) return fail(c, JPGENC_ERR_ARG, "null argument");
    std::vector<PixelSource> src(n);
    for (uint32_t i = 0; i < n; ++i) src[i] = image_source(images[i], row_pitches ? row_pitches[i] : 0, format);
    return encode_packed(c, src, images_on_device, widths, heights, maxval, out, cap, offsets, sizes, total_bytes);
} JPGENC_CATCH(c)

int jpgenc_encode_images_packed_planar(jpgenc_ctx* c, uint32_t n, const void* const* planes, int images_on_device, const uint32_t* widths,
                                       const uint32_t* heights, const uint32_t* row_pitches, uint32_t maxval, uint8_t* out, uint64_t cap,
                                       uint64_t* offsets, uint64_t* sizes, uint64_t* total_bytes) try {
    if (!c) return JPGENC_ERR_ARG;
    if (total_bytes) *total_bytes = 0;
    if (maxval == 0 || maxval > 255) return fail(c, JPGENC_ERR_ARG, "maxval out of range");
    if (n == 0) return JPGENC_OK;                                // an empty batch is legal and touches nothing
    if (!planes || !widths || !heights || !offsets || !sizes) return fail(c, JPGENC_ERR_ARG, "null argument");
    std::vector<PixelSource> src(n);
    for (uint32_t i = 0; i < n; ++i) src[i] = planar_source(planes[3 * i], planes[3 * i + 1], planes[3 * i + 2], row_pitches ? row_pitches[i] : 0);
    return encode_packed(c, src, images_on_device, widths, heights, maxval, out, cap, offsets, sizes, total_bytes);
} JPGENC_CATCH(c)

int jpgenc_encode_images_packed_yuv(jpgenc_ctx* c, uint32_t n, const void* const* planes, int images_on_device, const uint32_t* widths,
                                    const uint32_t* heights, const uint32_t* y_pitches, const uint32_t* c_pitches, int layout, uint8_t* out,
                                    uint64_t cap, uint64_t* offsets, uint64_t* sizes, uint64_t* total_bytes) try {
    if (!c) return JPGENC_ERR_ARG;
    if (total_bytes) *total_bytes = 0;
    if (yuv_source(nullptr, nullptr, nullptr, 0, 0, layout).format < 0) return fail(c, JPGENC_ERR_ARG, "unknown YUV layout");
    if (n == 0) return JPGENC_OK;                                // an empty batch is legal and touches nothing
    if (!planes || !widths || !heights || !offsets || !sizes) return fail(c, JPGENC_ERR_ARG, "null argument");
    std::vector<PixelSource> src(n);
    for (uint32_t i = 0; i < n; ++i)
        src[i] = yuv_source(planes[3 * i], planes[3 * i + 1], planes[3 * i + 2], y_pitches ? y_pitches[i] : 0, c_pitches ? c_pitches[i] : 0, layout);
    return encode_packed(c, src, images_on_device, widths, heights, 255, out, cap, offsets, sizes, total_bytes);
} JPGENC_CATCH(c)

int jpgenc_encode_images_packed_yuv420(jpgenc_ctx* c, uint32_t n, const void* const* planes, int images_on_device, const uint32_t* widths,
                                       const uint32_t* heights, const uint32_t* y_pitches, const uint32_t* c_pitches, int layout, uint8_t* out,
                                       uint64_t cap, uint64_t* offsets, uint64_t* sizes, uint64_t* total_bytes) try {
    if (!c) return JPGENC_ERR_ARG;
    if (total_bytes) *total_bytes = 0;
    if (!is_yuv420_layout(layout)) return fail(c, JPGENC_ERR_ARG, "unknown YUV 4:2:0 layout");
    return jpgenc_encode_images_packed_yuv(c, n, planes, images_on_device, widths, heights, y_pitches, c_pitches, layout, out, cap, offsets,
                                          sizes, total_bytes);
} JPGENC_CATCH(c)

}  // extern "C"
