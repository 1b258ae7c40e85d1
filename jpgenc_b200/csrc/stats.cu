// K2 — DC differencing + run-length/category symbol generation.  One pass over the coefficients produces
//   * the 4 x 256 symbol histogram and, per symbol, the position of its first occurrence in the reference's symbol
//     text (what the Huffman table build needs), and
//   * the symbol stream itself, as flat 32-bit items in scan order (blockwalk.cuh), which is all K3 reads.
//
// Replaces Image::applyDCdifferenceCoding, Image::doRLEandCategoryCoding and the symbol-text collection
// (reference src/Image.cpp:638-735, 888-906; include/Coding.hpp:148-283).  The first-occurrence key is needed because
// generateHuffmanCode (src/Huffman.cpp:6-14) feeds package_merge in unordered_map iteration order, which depends on the
// order symbols first appear (SURVEY.md H2).  Text order (src/Image.cpp:892-906): Y blocks raster over the block grid,
// chroma = all Cb blocks then all Cr blocks; DC and AC symbols go to separate texts.
//
// Work distribution.  Blocks hold very different numbers of non-zero coefficients, so "one thread walks one block"
// diverges badly.  Instead a tile of 384 blocks is flattened: every thread sizes its block with a popcount of the
// block's 64-bit non-zero mask, a CTA scan gives each block its first item index, the threads expand their masks into
// (block, position, run) descriptors -- a loop of a few instructions per set bit -- and then consecutive lanes process
// consecutive non-zero COEFFICIENTS: no lane ever loops over zeros, the work per lane is equal whatever the blocks look
// like, the loop body is branch-free and the item stores are coalesced.  The DC and EOB symbols
// exist exactly once (at most once) per block and stay with the block's own thread.
#include <algorithm>

#include "blockwalk.cuh"

namespace jpgenc {

constexpr int kDescCap = 2048;                           // descriptors per round (typical tiles need ~1300)

struct StatsParams {
    const int16_t* coef;
    uint32_t nblocks;                 // blocks per frame
    uint32_t tiles_per_frame;         // CTA blockIdx.x handles tile t % tiles_per_frame of frame t / tiles_per_frame, t = tile0 + blockIdx.x
    uint32_t tile0;                   // first tile of this launch (band-wise encodes run K2 behind every band; one frame only)
    uint32_t tiles_total;
    uint32_t mcu_w;
    uint32_t n_mcu;
    uint8_t* g_stats;                 // per frame kStatsBytes: hist u32[4][256], then first-occurrence keys u64[4][256]
    uint32_t* items;                  // item stream: tile t owns the slab [t * kSlabItems, (t + 1) * kSlabItems)
    uint32_t* tile_cnt;               // [tiles] items of the tile
    const uint32_t* refine_count;     // K1's refinement counter ...
    uint32_t* refine_copy;            // ... copied next to the statistics so that one read-back fetches everything
};

// Histogram updates are a plain shared-memory atomic per lane: grouping lanes of the same bin (MATCH.ANY, round 1) costs
// ~25 instructions per step in a kernel bound by instruction issue, while same-address shared-memory atomics are serialised
// by the LSU at no issue cost (DESIGN.md, K2).
//
// Keys inside a tile are 32-bit and TILE-LOCAL (TileKeys): shared memory has a native 32-bit atomic minimum, a 64-bit one is
// a compare-and-swap loop.
//
// Tile-local first-occurrence keys.  The global key of a symbol is (block index in the reference's text order) * 256 +
// position key.  Inside one tile (64 consecutive MCUs) the luma text indices lie within a few block rows of the tile's
// first block, and the chroma ones are the tile's MCU numbers, once for Cb and once -- n_mcu later -- for Cr:
//   luma    local = (text index - text index of the tile's first Y block) * 256 + position key      (< 2^24)
//   chroma  local = (is Cr) << 30 | (MCU - first MCU of the tile) * 256 + position key
// TileKeys converts a tile-local key back to the global form when the tile flushes.
struct TileKeys {
    unsigned long long y_base, cb_base, cr_base;          // global keys of local key 0
    static constexpr uint32_t kCr = 1u << 30, kSpan = 64u * 256u;
    __device__ __forceinline__ unsigned long long to_global(int table, uint32_t k) const {
        if (table < 2) return y_base + k;
        return ((k & kCr) ? cr_base : cb_base) + (k & (kCr - 1));
    }
};

constexpr size_t kStatsBytes = 4096 + 8192;

constexpr int kStatsSmem = kTileSmemBytes                // masks + dc
                           + kTileBlocks * 4             // local text key of the block
                           + kTileBlocks * 4             // first item / first AC descriptor of the block
                           + kDescCap * 4                // descriptors
                           + 4096 + 4096                 // histogram, local first-occurrence keys
                           + 36 * 4;                     // scan scratch

// (the thread index comes from the kernel: there the compiler knows its range from the launch bounds)
__device__ __forceinline__ void symbol_stats_body(const StatsParams& p, unsigned thread) {
    extern __shared__ __align__(128) uint8_t smem[];
    const TileView tv = tile_view(smem);
    uint8_t* at = smem + kTileSmemBytes;
    uint32_t* s_key = reinterpret_cast<uint32_t*>(at);                        at += kTileBlocks * 4;
    uint32_t* s_base = reinterpret_cast<uint32_t*>(at);                       at += kTileBlocks * 4;
    uint32_t* s_desc = reinterpret_cast<uint32_t*>(at);                       at += kDescCap * 4;
    uint32_t* s_hist = reinterpret_cast<uint32_t*>(at);                       at += 4096;
    uint32_t* s_first = reinterpret_cast<uint32_t*>(at);                      at += 4096;
    uint32_t* s_scan = reinterpret_cast<uint32_t*>(at);
    __shared__ uint32_t s_origin[2];                                      // MCU column / row of the tile's first MCU

    const int tid = thread, lane = tid & 31;
    const uint32_t gtile = p.tile0 + blockIdx.x;
    const uint32_t frame = p.tiles_total == p.tiles_per_frame ? 0u : gtile / p.tiles_per_frame;   // one image: no division
    const uint32_t first = (gtile - frame * p.tiles_per_frame) * kTileBlocks;           // first block of the tile, within its frame
    const int nb = static_cast<int>(min(static_cast<uint32_t>(kTileBlocks), p.nblocks - first));
    const int16_t* __restrict__ coef = p.coef + static_cast<size_t>(frame) * p.nblocks * kCoefPerBlock;
    uint32_t* __restrict__ g_hist = reinterpret_cast<uint32_t*>(p.g_stats + frame * kStatsBytes);
    unsigned long long* __restrict__ g_first = reinterpret_cast<unsigned long long*>(p.g_stats + frame * kStatsBytes + 4096);

    // First-occurrence keys start at "none" in every tile: a symbol's first occurrence in the tile costs one shared-memory
    // atomic (a few dozen symbols per tile), later ones none; the tile's minima meet the global ones when it flushes.  (Round 1
    // fetched the 8 KB of global minima into every CTA and converted them to tile-local form -- 1024 conversions and 134 MB of
    // L2 reads per image -- to save those few atomics.)
    if (tid == 0) {
        const uint32_t m0 = first / kBlocksPerMcu, y0 = m0 / p.mcu_w;  // the tile's only division
        s_origin[0] = m0 - y0 * p.mcu_w;
        s_origin[1] = y0;
    }
    for (int i = tid; i < 1024; i += kTileBlocks) { s_hist[i] = 0; s_first[i] = 0xFFFFFFFFu; }
    scan_tile(tv, coef + static_cast<size_t>(first) * kCoefPerBlock, nb, tid, kTileBlocks);
    __syncthreads();
    const uint32_t m_first = first / kBlocksPerMcu;
    const uint32_t y_text0 = (s_origin[1] * 2u) * (2u * p.mcu_w) + s_origin[0] * 2u;     // text index of the tile's first Y block
    TileKeys tk;
    tk.y_base = 256ull * y_text0;
    tk.cb_base = 256ull * m_first;
    tk.cr_base = 256ull * (static_cast<unsigned long long>(p.n_mcu) + m_first);

    // ---- per block: mask, DC difference, text key, item counts ----
    const bool live = tid < nb;
    const int k = tid % kBlocksPerMcu;                                    // tiles start on an MCU boundary
    const int tdc = k < 4 ? 0 : 2;
    uint32_t lo = 0, hi = 0, nac = 0, eob = 0;
    int diff = 0;
    uint32_t key = 0;
    if (live) {
        load_mask(tv, tid, lo, hi);
        diff = tv.dc[tid] - dc_predictor(tv, coef, first, tid);
        nac = __popc(lo) + __popc(hi);
        eob = (hi >> 31) ? 0u : 1u;                                       // no EOB when coefficient 63 is non-zero
        const uint32_t lm = tid / kBlocksPerMcu;
        uint32_t mx = s_origin[0] + lm, my = s_origin[1];
        while (mx >= p.mcu_w) { mx -= p.mcu_w; ++my; }                    // a 64-MCU tile wraps rarely
        key = k < 4 ? 256u * ((my * 2 + (k >> 1)) * (2u * p.mcu_w) + mx * 2 + (k & 1) - y_text0)
                    : (static_cast<uint32_t>(k - 4) << 30) | (256u * lm);
        s_key[tid] = key;
    }
    // one scan for both prefix sums: items (DC + ACs + EOB) in the low half, AC descriptors in the high half
    const uint32_t count = live ? 1u + nac + eob : 0u;
    uint32_t totals;
    const uint32_t base2 = block_exclusive_scan(count | (nac << 16), s_scan, &totals);
    const uint32_t base = base2 & 0xFFFFu, total = totals & 0xFFFFu, total_ac = totals >> 16;
    s_base[tid] = base2;
    if (tid == 0) {
        p.tile_cnt[gtile] = total;
        if (gtile + 1 == p.tiles_total) *p.refine_copy = *p.refine_count;    // the last tile runs in the last launch
    }
    uint32_t* __restrict__ out = p.items + static_cast<size_t>(gtile) * kSlabItems;

    // ---- DC and EOB: exactly one (at most one) per block, so the block's own thread handles them ----
    const int dcat = category_of(diff);
    if (live) {
        out[base] = make_item(tdc, dcat, 0, diff);
        if (eob) out[base + count - 1] = make_item(tdc + 1, 0, 0, 0);
    }
    if (live) {
        atomicAdd(&s_hist[tdc * 256 + dcat], 1u);
        if (key < s_first[tdc * 256 + dcat]) atomicMin(&s_first[tdc * 256 + dcat], key);
    }
    {
        const bool ey = eob && k < 4, ec = eob && k >= 4;
        const unsigned by = __ballot_sync(0xffffffffu, ey), bc = __ballot_sync(0xffffffffu, ec);
        if (lane == 0) {
            if (by) atomicAdd(&s_hist[256], static_cast<uint32_t>(__popc(by)));
            if (bc) atomicAdd(&s_hist[768], static_cast<uint32_t>(__popc(bc)));
        }
        const int ti = (tdc + 1) * 256;
        const bool better = eob && key + 129u < s_first[ti];
        if (__any_sync(0xffffffffu, better)) {
            const uint32_t ky = __reduce_min_sync(0xffffffffu, better && k < 4 ? key + 129u : 0xFFFFFFFFu);
            const uint32_t kc = __reduce_min_sync(0xffffffffu, better && k >= 4 ? key + 129u : 0xFFFFFFFFu);
            if (lane == 0) {
                if (ky != 0xFFFFFFFFu) atomicMin(&s_first[256], ky);
                if (kc != 0xFFFFFFFFu) atomicMin(&s_first[768], kc);
            }
        }
    }

    // ---- AC coefficients, flattened ----
    const uint32_t base_ac = base2 >> 16;
    for (uint32_t win = 0; win < total_ac; win += kDescCap) {
        // expand: one descriptor per non-zero AC coefficient in [win, win + kDescCap):
        //   [5:0] zigzag position, [11:6] zeros since the previous non-zero coefficient (or the DC), [20:12] block, [21] chroma
        if (live && base_ac < win + kDescCap && base_ac + nac > win) {
            uint32_t g = base_ac - win;                                   // wraps to a huge value while g is before the window
            const uint32_t tag = (static_cast<uint32_t>(tid) << 12) | (k < 4 ? 0u : 1u << 21);
            int prev = 0;
#pragma unroll 1
            for (int half = 0; half < 2; ++half) {
                uint32_t m = half ? hi : lo;
#pragma unroll 1
                while (m) {
                    const int pos = half * 32 + __ffs(m) - 1;
                    m &= m - 1;
                    if (g < kDescCap) s_desc[g] = tag | static_cast<uint32_t>((pos - prev - 1) << 6) | static_cast<uint32_t>(pos);
                    prev = pos;
                    ++g;
                }
            }
        }
        __syncthreads();
        // consecutive lanes take consecutive coefficients
        const uint32_t n = min(static_cast<uint32_t>(kDescCap), total_ac - win);
        for (uint32_t j0 = 0; j0 < n; j0 += kTileBlocks) {              // uniform trip count: the __any_sync below is warp-wide
            const uint32_t j = j0 + tid;
            const bool has = j < n;
            int idx = 0, nzrl = 0, table = 0;
            uint32_t ikey = 0;
            if (has) {
                const uint32_t d = s_desc[j], pos = d & 63u, run = (d >> 6) & 63u, b = (d >> 12) & 511u;
                nzrl = static_cast<int>(run >> 4);
                const int value = coef[static_cast<size_t>(first + b) * kCoefPerBlock + pos];     // L1/L2 hit: the tile was just read
                const int symbol = static_cast<int>((run & 15u) << 4) | category_of(value);
                table = static_cast<int>(d >> 21) * 2 + 1;
                idx = table * 256 + symbol;
                ikey = s_key[b] + 2 * pos + 1;
                const uint32_t sb = s_base[b];
                out[(sb & 0xFFFFu) + 1u + (win + j - (sb >> 16))] = make_item(table, symbol, nzrl, value);
            }
            if (has) {                                                   // plain shared-memory atomics: same-address lanes are serialised by the LSU
                atomicAdd(&s_hist[idx], 1u);
                if (ikey < s_first[idx]) atomicMin(&s_first[idx], ikey);
            }
            if (__any_sync(0xffffffffu, nzrl != 0)) {                   // ZRLs (runs of 16 zeros) are rare
                if (nzrl) {
                    const int zi = table * 256 + 0xF0;
                    atomicAdd(&s_hist[zi], static_cast<uint32_t>(nzrl));
                    const uint32_t kz = ikey - 1;                        // 2*pos: just before the symbol of position pos
                    if (kz < s_first[zi]) atomicMin(&s_first[zi], kz);
                }
            }
        }
        __syncthreads();                                                // s_desc is reused by the next window
    }

    __syncthreads();                                                    // all shared-memory histogram updates are in
    for (int i = tid; i < 1024; i += kTileBlocks) {
        const uint32_t n = s_hist[i];
        if (n) {
            atomicAdd(&g_hist[i], n);
            const unsigned long long k = tk.to_global(i >> 8, s_first[i]);
            if (k < __ldcg(&g_first[i])) atomicMin(&g_first[i], k);
        }
    }
}

__global__ void __launch_bounds__(kTileBlocks, 5) symbol_stats_kernel(const __grid_constant__ StatsParams p) {
    symbol_stats_body(p, threadIdx.x);
}

// Images of individual sizes (geom[nframes + 1]): a tile finds its image by the first-tile prefix and runs as a tile of a
// batch of that one image -- the parameters are rebased onto the image's coefficients, statistics, item slabs and tile
// counts, and carry its own block count and MCU geometry.  (K1's refinement counter is then copied by the last tile of
// every image: the same value each time.)
__global__ void __launch_bounds__(kTileBlocks, 5) symbol_stats_mixed_kernel(const __grid_constant__ StatsParams p, const FrameGeom* __restrict__ geom,
                                                                            uint32_t nframes) {
    const uint32_t gtile = p.tile0 + blockIdx.x;
    const uint32_t f = geom_find_warp(geom, nframes, gtile, &FrameGeom::tile0);
    const FrameGeom& g = geom[f];
    StatsParams q = p;
    q.coef = p.coef + static_cast<size_t>(g.block0) * kCoefPerBlock;
    q.nblocks = g.mcu_w * g.mcu_h * kBlocksPerMcu;
    q.tiles_per_frame = q.tiles_total = geom[f + 1].tile0 - g.tile0;
    q.tile0 = p.tile0 - g.tile0;                                        // tile0 + blockIdx.x = the tile within the image
    q.mcu_w = g.mcu_w;
    q.n_mcu = g.mcu_w * g.mcu_h;
    q.g_stats = p.g_stats + static_cast<size_t>(f) * kStatsBytes;
    q.items = p.items + static_cast<size_t>(g.tile0) * kSlabItems;
    q.tile_cnt = p.tile_cnt + g.tile0;
    symbol_stats_body(q, threadIdx.x);
}

// One image: hand the statistics to the host through its mailbox (mapped pinned memory).  A kernel of its own, in stream
// order behind K2: making the last CTA of K2 do this needs a __threadfence per CTA behind its histogram atomics, which cost
// K2 24 us at 16384 tiles.  Only the symbols that occur travel (a few dozen of 1024), each as two self-validating 64-bit
// words (common.cuh: value | tag); the tag comes from a sequence number kept in device memory (*dseq, incremented here) and
// mirrored by the host (jpgenc_ctx::mailbox_seq): it is not a kernel parameter, so a captured CUDA graph of the encode can be
// replayed as is.  No flag word, no __threadfence_system: the first version (12 KB of statistics, a system fence, then a flag)
// took 11 us, most of it the fence waiting for 96 PCIe writes to be acknowledged.
__global__ void __launch_bounds__(1024) publish_stats_kernel(const uint8_t* __restrict__ stats, const uint32_t* __restrict__ refine_count,
                                                             unsigned long long* mailbox, uint32_t* dseq) {
    __shared__ uint32_t s_warp[32];
    __shared__ uint32_t s_seq;
    const uint32_t e = threadIdx.x, lane = e & 31, warp = e >> 5;
    const uint32_t cnt = __ldcg(reinterpret_cast<const uint32_t*>(stats) + e);
    const unsigned long long first = __ldcg(reinterpret_cast<const unsigned long long*>(stats + 4096) + e);
    const unsigned present = __ballot_sync(0xffffffffu, cnt != 0);
    if (lane == 0) s_warp[warp] = __popc(present);
    if (e == 0) { s_seq = *dseq + 1u; *dseq = s_seq; }
    __syncthreads();
    uint32_t before = 0, total = 0;
    for (uint32_t w = 0; w < 32; ++w) { const uint32_t n = s_warp[w]; if (w < warp) before += n; total += n; }
    const uint32_t seq = s_seq;
    volatile unsigned long long* box = mailbox + kMailStatsHead;
    if (cnt != 0) {
        const uint32_t k = before + __popc(present & ((1u << lane) - 1u));
        box[1 + 2 * k] = mail_word(static_cast<unsigned long long>(cnt) | (static_cast<unsigned long long>(e) << 32), seq);
        box[2 + 2 * k] = mail_word(first, seq);
    }
    if (e == 0) box[0] = mail_word(static_cast<unsigned long long>(total) | (static_cast<unsigned long long>(*refine_count) << 11), seq);
}

// Everything an encode accumulates into, cleared by ONE kernel in front of K1 (four memset nodes before: one ahead of K1, three
// between the refinement and K2, each a link of a few microseconds in the chain of a small frame): K1's counters, per frame
// histogram = 0 and first-occurrence keys = all ones, K3a's group / super-group sums = 0.
__global__ void encode_clear_kernel(uint32_t* counters, uint32_t* stats, uint32_t stat_words, unsigned long long* range_base, uint32_t range_words) {
    const uint32_t i0 = blockIdx.x * blockDim.x + threadIdx.x, step = gridDim.x * blockDim.x;
    for (uint32_t i = i0; i < stat_words; i += step) stats[i] = (i % (kStatsBytes / 4)) < 1024u ? 0u : 0xFFFFFFFFu;
    for (uint32_t i = i0; i < range_words; i += step) range_base[i] = 0ull;
    if (i0 < 4) counters[i0] = 0u;                             // refinement list length .. entries refined so far
}

bool launch_encode_clear(jpgenc_ctx* c) {
    // one image only: in batches (four streams side by side) the same kernel in front of every pass's K1 costs 6 % (1024 frames
    // 5.89 -> 6.23 ms, measured twice; the memsets stay there)
    if (c->nframes > 1) return false;
    const size_t stat_bytes = static_cast<size_t>(c->nframes) * kStatsBytes;
    if (!c->d_stats || !c->d_range_base || c->stats_cap < stat_bytes || stat_bytes / 4 > 0xFFFFFFFFull || c->range_base_cap / 8 > 0xFFFFFFFFull) return false;
    const uint32_t stat_words = static_cast<uint32_t>(stat_bytes / 4), range_words = static_cast<uint32_t>(c->range_base_cap / 8);
    const uint32_t work = std::max(stat_words, range_words);
    encode_clear_kernel<<<std::max(1u, std::min(296u, (work + 1023u) / 1024u)), 256, 0, c->stream>>>(c->d_counters, reinterpret_cast<uint32_t*>(c->d_stats), stat_words,
                                                                                                 c->d_range_base, range_words);
    if (cudaGetLastError() != cudaSuccess) return false;
    c->launches += 1;
    c->stats_clear_valid = true;
    c->stats_clear_gen = c->alloc_gen;
    c->stats_clear_frames = c->nframes;
    return true;
}

int launch_symbol_stats(jpgenc_ctx* c, uint32_t tile0, uint32_t ntiles, bool first) {
    const uint64_t n_mcu = static_cast<uint64_t>(c->mcu_w) * c->mcu_h, nblocks = n_mcu * kBlocksPerMcu;
    const unsigned tiles = static_cast<unsigned>((nblocks + kTileBlocks - 1) / kTileBlocks);
    if (first) {
        if (!(c->stats_clear_valid && c->stats_clear_gen == c->alloc_gen && c->stats_clear_frames == c->nframes)) {
            // (no K1 in front of this K2 -- coefficients set by a test hook, planes, a second K2 over the same coefficients)
            // per frame: histogram = 0, first-occurrence keys = all ones
            JPGENC_CUDA(c, cudaMemset2DAsync(c->d_stats, kStatsBytes, 0, 4096, c->nframes, c->stream));
            JPGENC_CUDA(c, cudaMemset2DAsync(c->d_stats + 4096, kStatsBytes, 0xFF, 8192, c->nframes, c->stream));
            // K3a accumulates bit counts per group of 8 tiles and per 256 groups into d_range_base
            JPGENC_CUDA(c, cudaMemsetAsync(c->d_range_base, 0, c->range_base_cap, c->stream));
        }
        c->stats_clear_valid = false;
        c->entropy_runs = 0;
    }
    if (ntiles == 0) return JPGENC_OK;
    StatsParams p{};
    p.coef = c->d_coef;
    p.nblocks = static_cast<uint32_t>(nblocks);
    p.tiles_per_frame = tiles;
    p.tile0 = tile0;
    p.tiles_total = tiles * c->nframes;
    p.mcu_w = c->mcu_w;
    p.n_mcu = static_cast<uint32_t>(n_mcu);
    p.g_stats = c->d_stats;
    p.items = c->d_items;
    p.tile_cnt = c->d_tile_cnt;
    p.refine_count = c->d_counters;
    p.refine_copy = reinterpret_cast<uint32_t*>(c->d_stats + c->nframes * kStatsBytes);
    if (!c->k2_configured) {                                   // (the first encode of a context is never graph-captured)
        JPGENC_CUDA(c, cudaFuncSetAttribute(symbol_stats_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kStatsSmem));
        JPGENC_CUDA(c, cudaFuncSetAttribute(symbol_stats_mixed_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kStatsSmem));
        c->k2_configured = true;
    }
    if (c->mixed.on) {                                         // images of individual sizes: the per-size fields above are replaced per tile
        symbol_stats_mixed_kernel<<<ntiles, kTileBlocks, kStatsSmem, c->stream>>>(p, c->d_geom, c->nframes);
    } else {
        symbol_stats_kernel<<<ntiles, kTileBlocks, kStatsSmem, c->stream>>>(p);
    }
    JPGENC_CUDA(c, cudaGetLastError());
    c->launches += 1;
    return JPGENC_OK;
}

// one image, behind its last K2 launch: the statistics of the symbols that occur + K1's refinement counter into the host mailbox
int launch_publish_stats(jpgenc_ctx* c) {
    publish_stats_kernel<<<1, 1024, 0, c->stream>>>(c->d_stats, c->d_counters + kCntRefine, c->d_mailbox, c->d_counters + kCntSeq);
    JPGENC_CUDA(c, cudaGetLastError());
    c->launches += 1;
    ++c->mailbox_seq;                                          // the sequence number the kernel will tag its words with
    return JPGENC_OK;
}

}  // namespace jpgenc
