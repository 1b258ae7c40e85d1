// K3 — Huffman encode + MCU interleave + 1-padding;  K4 — FF -> FF 00 byte stuffing.
//
// Replaces Image::doHuffmanEncoding, the per-MCU Bitstream concatenation, Bitstream::fill() and the stuffing
// operator<< (reference src/Image.cpp:737-829, 957-971; include/BitstreamGeneric.hpp:126-146, 182-195, 213-224, 242-248).
//
// K3 reads the symbol items K2 left in HBM (blockwalk.cuh), never the coefficients, in two launches:
//   K3a  one warp per item range (= one K2 tile, 384 blocks): coalesced pass, bits the range encodes to;
//        sizes are also accumulated per group of 8 ranges and per 256 groups, from which
//        K3b derives every range's bit offset with a few hundred additions (no serial scan);
//   K3b  one warp per range: codes assembled MSB-first in a per-warp shared-memory bit buffer and written out as whole
//        32-bit words (only the two words a chunk shares with its neighbours use atomicOr).
// With the offsets known up front no warp ever waits for another one: no tickets, no look-back, no block barriers.
// K4a/K4: FF bytes per tile; then every tile: CTA scan, output position = sum of the earlier tiles' counts, compact.
#include <cstdlib>

#include "blockwalk.cuh"

namespace jpgenc {


// MSB-first bit writer into 32-bit words ("word bit 31 is the earliest bit"); words are byte-swapped when they go
// to memory so that memory byte order is stream order (SURVEY.md H5).
template <bool kGlobal>
struct BitWriter {
    uint32_t* words;        // shared bit buffer (word 0 = the tile's first, partially foreign, word) or global raw scan
    uint32_t word;          // current word index
    uint32_t fill;          // bits already used in the current word
    uint32_t acc;

    __device__ __forceinline__ void start(uint32_t* base, unsigned long long bitpos) {
        words = base;
        word = static_cast<uint32_t>(bitpos >> 5);
        fill = static_cast<uint32_t>(bitpos & 31);
        acc = 0;
    }
    __device__ __forceinline__ void flush_word() {
        if (acc) atomicOr(&words[word], kGlobal ? __byte_perm(acc, 0, 0x0123) : acc);
    }
    __device__ __forceinline__ void put(uint32_t code, uint32_t n) {      // n <= 31, code < 2^n
        const unsigned long long v = static_cast<unsigned long long>(code) << (64 - fill - n);
        acc |= static_cast<uint32_t>(v >> 32);
        fill += n;
        if (fill >= 32) {
            flush_word();
            ++word;
            acc = static_cast<uint32_t>(v);
            fill -= 32;
        }
    }
    __device__ __forceinline__ void finish() { if (fill) flush_word(); }
};

// Per-frame geometry of the entropy stage.  One image is the batch of one frame; in a batch every frame has its own
// tables, its own stretch of the raw scan, its own place in the output and its own totals.  Sizes and offsets are read
// from device memory (PassMeta, common.cuh): for a batch they are computed on the device and never visit the host.
struct EntropyParams {
    const uint32_t* items;              // K2's symbol items: range R = the first range_cnt[R] slots of slab R
    const uint32_t* range_cnt;          // [nframes * ranges_per_frame]
    uint32_t nframes;
    uint32_t split;                     // ranges per K2 tile: 1, or 4 for small images (more warps at work; see launch_entropy)
    uint32_t ranges_per_frame;          // K2 tiles per frame * split
    uint32_t groups_per_frame;          // ceil(ranges_per_frame / 8): one CTA of K3a/K3b each
    uint32_t supers_per_frame;          // ceil(groups_per_frame / 256)
    const DeviceTables* tables;         // [nframes]
    uint32_t* range_bits;               // [nframes * ranges_per_frame] bits the range encodes to (K3a)
    unsigned long long* group_bits;     // [nframes * groups_per_frame] bits of the 8 ranges one CTA handles (K3a)
    unsigned long long* super_bits;     // [nframes * supers_per_frame] bits of 256 consecutive groups (K3a, atomics; zeroed before K2)
    uint32_t* raw;                      // all frames' un-stuffed scans; K3a zeroes it, K3b fills it
    const PassHeader* hdr;              // raw_total, k4_tiles, error
    const unsigned long long* raw_off;  // [nframes] byte offset of the frame's raw scan (multiple of 16)
    const unsigned long long* raw_bytes;// [nframes] bytes of the frame's raw scan = ceil(bits / 8), known from the histogram
    const uint32_t* k4_tile0;           // [nframes + 1] first K4 tile of the frame
    const unsigned long long* file_base;// [nframes] where the frame's output starts, not counting the FFs stuffed before it
    const uint32_t* hdr_len;            // [nframes] bytes of JFIF header in front of the frame's scan (0: scan only)
    unsigned long long* total_bits;     // [nframes] out: bits of the scan (before padding)
    unsigned long long* ff_incl;        // [nframes] out: FF bytes K4 stuffed in frames 0..f of the pass
    uint32_t* tile_ff;                  // FF bytes per K4 tile (K4a), all frames of the pass numbered as ONE sequence
    uint32_t* redo_count;               // chunks K3b had to pack the slow way (diagnostics)
    unsigned long long* mailbox;        // one image: the host's mailbox (common.cuh kMail*); K4's last tile reports the totals there
    uint32_t* dseq;                     // ... tagged with the next sequence number
    // output as complete files (batches): every frame = header + scan + EOI, frames back to back
    const jpgenc_huff_table* built;     // [nframes * 4] tables as the device build left them (DHT segments); null = scan only
    const uint8_t* hdr_prefix;          // SOI .. SOF0, identical for every frame of the pass
    uint32_t hdr_prefix_len;
    uint32_t tail;                      // 2 (EOI) behind every scan, or 0
};

// code bits of one item: `nz` ZRL codes first, then the symbol's code with the magnitude bits appended
// (src/Image.cpp:757-766: table[symbol] top `length` bits, then the category's bits)
template <class Put>
__device__ __forceinline__ void item_codes(uint32_t item, const uint32_t* s_tab, Put&& put) {
    const uint32_t* tab = s_tab + ((item >> 8) & 3u) * 256u;
    const uint32_t nz = (item >> 10) & 3u;
    if (nz) {
        const uint32_t z = tab[0xF0];
        for (uint32_t i = 0; i < nz; ++i) put(z & 0xFFFFu, z >> 16);
    }
    const uint32_t e = tab[item & 0xFFu], cat = item & 15u;
    put(((e & 0xFFFFu) << cat) | (item >> 12), (e >> 16) + cat);
}

__device__ __forceinline__ uint32_t item_bits(uint32_t item, const uint32_t* s_tab) {
    const uint32_t* tab = s_tab + ((item >> 8) & 3u) * 256u;
    return (tab[item & 0xFFu] >> 16) + (item & 15u) + ((item >> 10) & 3u) * (tab[0xF0] >> 16);
}

// the common case in one lookup: returns (bit count << 27) | bits, or 0 when the item needs the general path
// (ZRLs in front of it, or a code + magnitude longer than 27 bits)
__device__ __forceinline__ uint32_t item_fast(uint32_t item, const uint32_t* s_fast) {
    const uint32_t e = s_fast[item & 0x3FFu];
    return ((item >> 10) & 3u) || !e ? 0u : e | (item >> 12);
}

// items of range `range` of frame `frame`: with split == 1 a range is a K2 tile's item slab, with split == 4 a quarter of it
__device__ __forceinline__ const uint32_t* range_items(const EntropyParams& p, uint32_t frame, uint32_t range, uint32_t* n) {
    const uint32_t tile = range / p.split, q = range - tile * p.split;
    const size_t slab = static_cast<size_t>(frame) * (p.ranges_per_frame / p.split) + tile;
    const uint32_t nt = p.range_cnt[slab], begin = static_cast<uint32_t>((static_cast<uint64_t>(nt) * q) / p.split),
                   end = static_cast<uint32_t>((static_cast<uint64_t>(nt) * (q + 1)) / p.split);
    *n = end - begin;
    return p.items + slab * kSlabItems + begin;
}

constexpr int kPackThreads = 256;                       // 8 warps, one item range each
constexpr int kPackWarps = kPackThreads / 32;

// ---- K3a: bits per range (coalesced pass over the items) + housekeeping ---------------------------------------
// Besides sizing the ranges this launch zeroes the raw scan, so that no memset sits between the host's table build and the
// first kernel.  Sizes are kept at three
// levels -- range, group (the 8 ranges of a CTA), super-group (256 groups, accumulated with atomics) -- so that K3b can
// derive any range's bit offset from a few hundred values instead of waiting for a serial scan.
__global__ void __launch_bounds__(kPackThreads) range_bits_kernel(const __grid_constant__ EntropyParams p) {
    __shared__ uint32_t s_len[1024];                           // bits of a symbol with its magnitude: code length + category; 0 = absent
    __shared__ uint32_t s_wbits[kPackWarps];
    if (p.hdr->error) return;                                  // the pass was refused (finalize_tables_kernel): the host re-runs it
    const uint32_t frame = blockIdx.x / p.groups_per_frame, group = blockIdx.x - frame * p.groups_per_frame;
    const DeviceTables* tables = p.tables + frame;
    for (int i = threadIdx.x; i < 1024; i += kPackThreads) {
        const uint32_t e = (&tables->entry[0][0])[i];
        s_len[i] = e ? (e >> 16) + (i & 15u) : 0u;
    }
    {   // housekeeping, spread over the grid
        const unsigned long long gtid = static_cast<unsigned long long>(blockIdx.x) * kPackThreads + threadIdx.x;
        const unsigned long long gsize = static_cast<unsigned long long>(gridDim.x) * kPackThreads;
        const unsigned long long raw_words16 = p.hdr->raw_total / 16;
        uint4* raw16 = reinterpret_cast<uint4*>(p.raw);
        for (unsigned long long i = gtid; i < raw_words16; i += gsize) raw16[i] = make_uint4(0, 0, 0, 0);
        if (gtid == 0) *p.redo_count = 0u;
    }
    __syncthreads();
    const uint32_t range = group * kPackWarps + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    uint32_t bits = 0;
    if (range < p.ranges_per_frame) {
        const size_t slab = static_cast<size_t>(frame) * p.ranges_per_frame + range;
        uint32_t n;
        const uint32_t* __restrict__ items = range_items(p, frame, range, &n);
        // one lookup per item; a ZRL in front of it (rare) adds the ZRL code of its table
        auto size_of = [&](uint32_t item) {
            uint32_t b = s_len[item & 0x3FFu];
            const uint32_t nz = (item >> 10) & 3u;
            if (nz) b += nz * (s_len[(item & 0x300u) | 0xF0u]);            // category 0: s_len is the bare code length
            return b;
        };
        uint32_t head = min(n, static_cast<uint32_t>((16u - (reinterpret_cast<uintptr_t>(items) & 15u)) & 15u) >> 2);   // items up to 16-byte alignment
        if (lane < head) bits += size_of(__ldg(items + lane));
        const uint4* __restrict__ q4 = reinterpret_cast<const uint4*>(items + head);
        const uint32_t nq = (n - head) >> 2;
        uint32_t i = lane;
        for (; i + 96 < nq; i += 128) {                                     // four 16-byte loads in flight per lane
            const uint4 a = __ldg(q4 + i), b = __ldg(q4 + i + 32), c = __ldg(q4 + i + 64), d = __ldg(q4 + i + 96);
            bits += size_of(a.x) + size_of(a.y) + size_of(a.z) + size_of(a.w);
            bits += size_of(b.x) + size_of(b.y) + size_of(b.z) + size_of(b.w);
            bits += size_of(c.x) + size_of(c.y) + size_of(c.z) + size_of(c.w);
            bits += size_of(d.x) + size_of(d.y) + size_of(d.z) + size_of(d.w);
        }
        for (; i < nq; i += 32) {
            const uint4 a = __ldg(q4 + i);
            bits += size_of(a.x) + size_of(a.y) + size_of(a.z) + size_of(a.w);
        }
        const uint32_t tail0 = head + 4u * nq;
        if (tail0 + lane < n) bits += size_of(__ldg(items + tail0 + lane));
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) bits += __shfl_xor_sync(0xffffffffu, bits, d);
        if (lane == 0) p.range_bits[slab] = bits;
    }
    if (lane == 0) s_wbits[threadIdx.x >> 5] = bits;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long sum = 0;
        for (int w = 0; w < kPackWarps; ++w) sum += s_wbits[w];
        p.group_bits[blockIdx.x] = sum;
        atomicAdd(&p.super_bits[frame * p.supers_per_frame + (group >> 8)], sum);
    }
}

// Images of individual sizes (geom[nframes + 1], numbered through the pass): a CTA of K3a / K3b finds its image by the
// first-group prefix and works as a group of a batch of that one image -- the parameters are rebased onto the image's
// tables, tiles, ranges, groups, super-groups and PassMeta entries, and carry its own counts (the split is the pass's).
__device__ __forceinline__ EntropyParams entropy_image(const EntropyParams& p, const FrameGeom* __restrict__ geom, uint32_t* group_base) {
    const uint32_t f = geom_find_warp(geom, p.nframes, blockIdx.x, &FrameGeom::group0);
    const FrameGeom& g = geom[f];
    EntropyParams q = p;
    q.ranges_per_frame = (geom[f + 1].tile0 - g.tile0) * p.split;
    q.groups_per_frame = geom[f + 1].group0 - g.group0;
    q.supers_per_frame = geom[f + 1].super0 - g.super0;
    q.tables = p.tables + f;
    q.range_cnt = p.range_cnt + g.tile0;
    q.items = p.items + static_cast<size_t>(g.tile0) * kSlabItems;
    q.range_bits = p.range_bits + static_cast<size_t>(g.tile0) * p.split;
    q.group_bits = p.group_bits + g.group0;
    q.super_bits = p.super_bits + g.super0;
    q.raw_off = p.raw_off + f;
    q.total_bits = p.total_bits + f;
    *group_base = g.group0;
    return q;
}

// K3a over images of individual sizes.  The same code as range_bits_kernel on the parameters entropy_image rebased onto the
// CTA's image; it is a copy rather than a shared function because moving range_bits_kernel's body into a device function
// changes that kernel's machine code (register allocation and schedule), and the single-size path is to stay as it is.
__global__ void __launch_bounds__(kPackThreads) range_bits_mixed_kernel(const __grid_constant__ EntropyParams pass, const FrameGeom* __restrict__ geom) {
    uint32_t group0;
    const EntropyParams p = entropy_image(pass, geom, &group0);
    __shared__ uint32_t s_len[1024];                           // bits of a symbol with its magnitude: code length + category; 0 = absent
    __shared__ uint32_t s_wbits[kPackWarps];
    if (p.hdr->error) return;                                  // the pass was refused (finalize_tables_kernel): the host re-runs it
    const uint32_t group = blockIdx.x - group0;             // within the image; p is rebased onto it
    const DeviceTables* tables = p.tables;
    for (int i = threadIdx.x; i < 1024; i += kPackThreads) {
        const uint32_t e = (&tables->entry[0][0])[i];
        s_len[i] = e ? (e >> 16) + (i & 15u) : 0u;
    }
    {   // housekeeping, spread over the grid
        const unsigned long long gtid = static_cast<unsigned long long>(blockIdx.x) * kPackThreads + threadIdx.x;
        const unsigned long long gsize = static_cast<unsigned long long>(gridDim.x) * kPackThreads;
        const unsigned long long raw_words16 = p.hdr->raw_total / 16;
        uint4* raw16 = reinterpret_cast<uint4*>(p.raw);
        for (unsigned long long i = gtid; i < raw_words16; i += gsize) raw16[i] = make_uint4(0, 0, 0, 0);
        if (gtid == 0) *p.redo_count = 0u;
    }
    __syncthreads();
    const uint32_t range = group * kPackWarps + (threadIdx.x >> 5), lane = threadIdx.x & 31;
    uint32_t bits = 0;
    if (range < p.ranges_per_frame) {
        uint32_t n;
        const uint32_t* __restrict__ items = range_items(p, 0, range, &n);
        auto size_of = [&](uint32_t item) {
            uint32_t b = s_len[item & 0x3FFu];
            const uint32_t nz = (item >> 10) & 3u;
            if (nz) b += nz * (s_len[(item & 0x300u) | 0xF0u]);
            return b;
        };
        uint32_t head = min(n, static_cast<uint32_t>((16u - (reinterpret_cast<uintptr_t>(items) & 15u)) & 15u) >> 2);
        if (lane < head) bits += size_of(__ldg(items + lane));
        const uint4* __restrict__ q4 = reinterpret_cast<const uint4*>(items + head);
        const uint32_t nq = (n - head) >> 2;
        uint32_t i = lane;
        for (; i + 96 < nq; i += 128) {
            const uint4 a = __ldg(q4 + i), b = __ldg(q4 + i + 32), c = __ldg(q4 + i + 64), d = __ldg(q4 + i + 96);
            bits += size_of(a.x) + size_of(a.y) + size_of(a.z) + size_of(a.w);
            bits += size_of(b.x) + size_of(b.y) + size_of(b.z) + size_of(b.w);
            bits += size_of(c.x) + size_of(c.y) + size_of(c.z) + size_of(c.w);
            bits += size_of(d.x) + size_of(d.y) + size_of(d.z) + size_of(d.w);
        }
        for (; i < nq; i += 32) {
            const uint4 a = __ldg(q4 + i);
            bits += size_of(a.x) + size_of(a.y) + size_of(a.z) + size_of(a.w);
        }
        const uint32_t tail0 = head + 4u * nq;
        if (tail0 + lane < n) bits += size_of(__ldg(items + tail0 + lane));
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) bits += __shfl_xor_sync(0xffffffffu, bits, d);
        if (lane == 0) p.range_bits[range] = bits;
    }
    if (lane == 0) s_wbits[threadIdx.x >> 5] = bits;
    __syncthreads();
    if (threadIdx.x == 0) {
        unsigned long long sum = 0;
        for (int w = 0; w < kPackWarps; ++w) sum += s_wbits[w];
        p.group_bits[group] = sum;
        atomicAdd(&p.super_bits[group >> 8], sum);
    }
}

// ---- K3b: pack ---------------------------------------------------------------------------------------------------
// One warp per range, no block-wide synchronisation.  The range is taken in chunks of 512 items: 16 coalesced row
// loads put the chunk into a padded shared-memory array, from which every lane reads ITS 16 consecutive items
// (blocked arrangement, bank-conflict-free thanks to the padding), sizes them, a warp scan places the lanes, each lane
// assembles its bits MSB-first in registers and ORs whole words into the warp's bit buffer.  The buffer is laid out
// with the same word alignment as the global scan, so flushing is a plain coalesced copy (atomicOr only for the two
// words shared with neighbours).
constexpr int kChunkRows = 16;
constexpr int kChunkItems = kChunkRows * 32;
constexpr int kWarpBitWords = 512;                      // 16 Kbit per chunk (32 bits per item on average) before falling back

// The CTA works on group blockIdx.x - group_base in the numbering of p: 0 for frames of one size, the first group of its image
// for images of individual sizes (entropy_image).  (The thread index comes from the kernel: there the compiler knows its range
// from the launch bounds.)
__device__ __forceinline__ void huffman_pack_body(const EntropyParams& p, uint32_t group_base, unsigned thread) {
    const uint32_t block = blockIdx.x - group_base;
    __shared__ uint32_t s_tab[1024], s_fast[1024];                      // DeviceTables::entry / ::fast
    __shared__ uint32_t s_items[kPackWarps][kChunkItems + kChunkRows];  // item j of the chunk at j + (j >> 5)
    __shared__ uint32_t s_bits[kPackWarps][kWarpBitWords + 2];
    __shared__ unsigned long long s_part[kPackWarps];
    const int tid = thread, lane = tid & 31, warp = tid >> 5;
    if (p.hdr->error) return;
    const uint32_t frame = block / p.groups_per_frame, group = block - frame * p.groups_per_frame;
    const DeviceTables* tables = p.tables + frame;
    for (int i = tid; i < 1024; i += kPackThreads) {
        s_tab[i] = (&tables->entry[0][0])[i];
        s_fast[i] = (&tables->fast[0][0])[i];
    }
    for (int i = lane; i < kWarpBitWords + 2; i += 32) s_bits[warp][i] = 0;
    __syncthreads();
    // bit offset of this CTA's first range inside its frame: whole super-groups before it + the groups before it in its
    // own super-group (at most 255 + 255 values for images up to 500 Mpx; summed cooperatively), then the ranges before
    // this warp's
    unsigned long long part = 0;
    {
        const uint32_t sup = group >> 8;
        const unsigned long long* supers = p.super_bits + static_cast<size_t>(frame) * p.supers_per_frame;
        const unsigned long long* groups = p.group_bits + static_cast<size_t>(frame) * p.groups_per_frame;
        for (uint32_t i = tid; i < sup; i += kPackThreads) part += __ldcg(supers + i);
        for (uint32_t i = (sup << 8) + tid; i < group; i += kPackThreads) part += __ldcg(groups + i);
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) part += __shfl_xor_sync(0xffffffffu, part, d);
    if (lane == 0) s_part[warp] = part;
    __syncthreads();
    const uint32_t range = group * kPackWarps + warp;
    const size_t slab0 = static_cast<size_t>(frame) * p.ranges_per_frame + group * kPackWarps;
    const unsigned long long frame_bit0 = p.raw_off[frame] * 8ull;      // where the frame's scan starts in `raw`
    unsigned long long cur = frame_bit0;                                // global bit position of the next chunk
    for (int w = 0; w < kPackWarps; ++w) cur += s_part[w];
    for (int w = 0; w < warp; ++w)
        if (group * kPackWarps + w < p.ranges_per_frame) cur += __ldcg(p.range_bits + slab0 + w);
    if (range >= p.ranges_per_frame) return;
    uint32_t n;
    const uint32_t* __restrict__ items = range_items(p, frame, range, &n);
    uint32_t* it = s_items[warp];
    uint32_t* bitbuf = s_bits[warp];

    // the rows of chunk c + 1 are requested before chunk c is processed (registers), so that a warp waits for global memory
    // once per range, not once per chunk
    uint32_t v[kChunkRows];
#pragma unroll
    for (int r = 0; r < kChunkRows; ++r) {
        const uint32_t j = r * 32 + lane;
        v[r] = j < n ? __ldg(items + j) : 0u;
    }
    for (uint32_t c0 = 0; c0 < n; c0 += kChunkItems) {
        const uint32_t m = min(static_cast<uint32_t>(kChunkItems), n - c0);
        const uint32_t rows = (m + 31) >> 5;
#pragma unroll
        for (int r = 0; r < kChunkRows; ++r) it[r * 33 + lane] = v[r];
        if (c0 + kChunkItems < n) {
#pragma unroll
            for (int r = 0; r < kChunkRows; ++r) {
                const uint32_t j = c0 + kChunkItems + r * 32 + lane;
                v[r] = j < n ? __ldg(items + j) : 0u;
            }
        }
        __syncwarp();
        const uint32_t j0 = min(m, lane * rows), j1 = min(m, j0 + rows);   // this lane's consecutive items
        const uint32_t lead = static_cast<uint32_t>(cur & 31);          // bits of the first word that belong to whoever came before
        // ---- one pass over the lane's items: their codes are assembled MSB-first into a lane-local bit string whose words
        // replace the items already consumed (word k goes to the slot of the lane's k-th item: an item yields at most 27
        // bits on the one-lookup path, so a word is never complete before its slot is free; items that need the general
        // path -- ZRLs in front, more than 27 bits -- may outrun their slots: then the chunk is redone the slow way) ----
        uint32_t my_bits = 0, nw = 0;
        bool outrun = false;
        {
            unsigned long long acc = 0;                                   // bit 63 = the earliest bit not yet stored
            uint32_t fill = 0;
            for (uint32_t j = j0; j < j1; ++j) {
                const uint32_t item = it[j + (j >> 5)];
                auto put = [&](uint32_t code, uint32_t len) {            // len <= 31, fill < 32
                    acc |= static_cast<unsigned long long>(code) << (64u - fill - len);
                    fill += len;
                    my_bits += len;
                    if (fill >= 32u) {
                        if (j0 + nw <= j) { const uint32_t o = j0 + nw; it[o + (o >> 5)] = static_cast<uint32_t>(acc >> 32); }
                        else outrun = true;
                        ++nw;
                        acc <<= 32;
                        fill -= 32u;
                    }
                };
                const uint32_t w = item_fast(item, s_fast);
                if (w) put(w & 0x07FFFFFFu, w >> 27);
                else item_codes(item, s_tab, put);
            }
            if (fill) {                                                   // the open word (its unused low bits are zero)
                if (j1 > j0 && j0 + nw < j1) { const uint32_t o = j0 + nw; it[o + (o >> 5)] = static_cast<uint32_t>(acc >> 32); }
                else outrun = true;
                ++nw;
            }
        }
        uint32_t inc = my_bits;
#pragma unroll
        for (int d = 1; d < 32; d <<= 1) {
            const uint32_t up = __shfl_up_sync(0xffffffffu, inc, d);
            if (lane >= d) inc += up;
        }
        const uint32_t total = __shfl_sync(0xffffffffu, inc, 31);
        const bool redo = __any_sync(0xffffffffu, outrun) || lead + total > kWarpBitWords * 32u;
        if (!redo) {
            // every lane ORs its words into the warp's bit buffer at its place (neighbours share words: shared-memory atomics)
            const uint32_t at = lead + inc - my_bits;
            for (uint32_t k = 0; k < nw; ++k) {
                const uint32_t o = j0 + k, v = it[o + (o >> 5)];
                const uint32_t pos = at + 32u * k, sh = pos & 31u;
                if (v >> sh) atomicOr(&bitbuf[pos >> 5], v >> sh);
                if (sh && (v << (32u - sh))) atomicOr(&bitbuf[(pos >> 5) + 1], v << (32u - sh));
            }
            __syncwarp();
            const uint32_t nwords = (lead + total + 31) >> 5;
            uint32_t* g = p.raw + (cur >> 5);
            for (uint32_t i = lane; i < nwords; i += 32) {
                const uint32_t v = __byte_perm(bitbuf[i], 0, 0x0123);
                bitbuf[i] = 0;
                if (i == 0 || i == nwords - 1) { if (v) atomicOr(&g[i], v); }
                else g[i] = v;
            }
        } else {
            // very dense chunk: items again (the pass above has overwritten them), straight to the (zeroed) global words
            if (lane == 0) atomicAdd(p.redo_count, 1u);
            __syncwarp();
#pragma unroll 4
            for (uint32_t r = 0; r < rows; ++r) {
                const uint32_t j = r * 32 + lane;
                if (j < m) it[j + r] = __ldg(items + c0 + j);
            }
            __syncwarp();
            if (j0 < j1) {
                BitWriter<true> bw;
                bw.start(p.raw, cur + inc - my_bits);
                for (uint32_t j = j0; j < j1; ++j)
                    item_codes(it[j + (j >> 5)], s_tab, [&](uint32_t code, uint32_t len) { bw.put(code, len); });
                bw.finish();
            }
        }
        __syncwarp();
        cur += total;
    }
    if (range + 1 == p.ranges_per_frame && lane == 0) {
        // 1-padding of Bitstream::fill() (BitstreamGeneric.hpp:242-248): the open byte is completed with ones
        const uint32_t pad = static_cast<uint32_t>((8 - (cur & 7)) & 7);
        if (pad) {
            BitWriter<true> bw;
            bw.start(p.raw, cur);
            bw.put((1u << pad) - 1, pad);
            bw.finish();
        }
        p.total_bits[frame] = cur - frame_bit0;                         // bits of the scan; the host checks it against the histogram
    }
}

__global__ void __launch_bounds__(kPackThreads) huffman_pack_kernel(const __grid_constant__ EntropyParams p) {
    huffman_pack_body(p, 0, threadIdx.x);
}
__global__ void __launch_bounds__(kPackThreads) huffman_pack_mixed_kernel(const __grid_constant__ EntropyParams p, const FrameGeom* __restrict__ geom) {
    uint32_t group0;
    const EntropyParams q = entropy_image(p, geom, &group0);
    huffman_pack_body(q, group0, threadIdx.x);
}

// ---- K4 ---------------------------------------------------------------------------------------------------
// FF -> FF 00 (BitstreamGeneric.hpp:213-224).  A tile is 16 KB of the raw scan.  Every thread counts the FF bytes of its
// 16 input bytes (SIMD byte compare), a CTA scan + look-back give the output position, the tile's output is assembled
// in shared memory (word stores; byte stores only at a thread's unaligned ends or where an FF actually occurs) and
// leaves as coalesced 32-bit stores, funnel-shifted to the alignment of the global position.
constexpr int kStuffThreads = kK4Threads;
constexpr int kStuffBytesPerThread = 16;
constexpr int kStuffTile = kStuffThreads * kStuffBytesPerThread;
static_assert(kStuffTile == kK4TileBytes, "capi.cu numbers K4 tiles with kK4TileBytes");

// header of frame `frame`'s file at `dst`: the common prefix (SOI .. SOF0), the four DHT segments from the tables as the
// device build left them, SOS (src/Image.cpp:933-954, JpegSegments.hpp:188-218; host twin: host/jfif_writer.cpp).
// geom (images of individual sizes): the prefix carries some image's size, the frame's own height and width replace it
// (SOF0 is the prefix's last segment, 19 bytes: FF C0, length, precision, height at +5, width at +7)
__device__ __forceinline__ void write_file_header(uint8_t* dst, const EntropyParams& p, uint32_t frame, int tid, int nthreads,
                                                  const FrameGeom* geom = nullptr) {
    if (geom) {
        const uint32_t hw = (geom[frame].real_h << 16) | geom[frame].real_w, at = p.hdr_prefix_len - 14;
        for (uint32_t i = tid; i < p.hdr_prefix_len; i += nthreads)
            dst[i] = i - at < 4 ? static_cast<uint8_t>(hw >> (8 * (3 - (i - at)))) : p.hdr_prefix[i];
    } else {
        for (uint32_t i = tid; i < p.hdr_prefix_len; i += nthreads) dst[i] = p.hdr_prefix[i];
    }
    uint32_t at = p.hdr_prefix_len;
    const jpgenc_huff_table* tabs = p.built + static_cast<size_t>(frame) * 4;
    for (int t = 0; t < 4; ++t) {
        uint32_t nsym = 0;
        for (int i = 0; i < 16; ++i) nsym += tabs[t].counts[i];
        const uint32_t seg = 21 + nsym;                        // marker 2, length 2, table info 1, counts 16, symbols
        for (uint32_t i = tid; i < seg; i += nthreads) {
            uint32_t b;
            if (i == 0) b = 0xFF;
            else if (i == 1) b = 0xC4;
            else if (i == 2) b = (19 + nsym) >> 8;
            else if (i == 3) b = (19 + nsym) & 0xFFu;
            else if (i == 4) b = ((t & 1) << 4) | (t >> 1);    // (class << 4) | destination: Y_DC 00, Y_AC 10, C_DC 01, C_AC 11
            else if (i < 21) b = tabs[t].counts[i - 5];
            else b = tabs[t].symbols[i - 21];
            dst[at + i] = static_cast<uint8_t>(b);
        }
        at += seg;
    }
    // SOS: Y -> tables 0/0, Cb and Cr -> 1/1, Ss = 0, Se = 63, Ah/Al = 0
    if (tid < 14) {
        // FF DA 00 0C | 03 01 00 02 | 11 03 11 00 | 3F 00
        const uint32_t w = tid < 4 ? 0x0C00DAFFu : tid < 8 ? 0x02000103u : tid < 12 ? 0x00110311u : 0x0000003Fu;
        dst[at + tid] = static_cast<uint8_t>(w >> (8 * (tid & 3)));
    }
}

// frame that owns K4 tile `t` (frame f owns tiles [k4_tile0[f], k4_tile0[f + 1]))
__device__ __forceinline__ uint32_t frame_of_tile(const EntropyParams& p, uint32_t t) {
    uint32_t lo = 0, hi = p.nframes;
    while (hi - lo > 1) {
        const uint32_t mid = (lo + hi) >> 1;
        if (p.k4_tile0[mid] <= t) lo = mid; else hi = mid;
    }
    return lo;
}

// FF bytes among a thread's 16 raw bytes at byte offset `at` of a frame's scan of `nbytes` bytes; the words (bytes past the
// end of the scan cleared: they are not FF candidates) are returned in wv, the number of valid bytes in n
__device__ __forceinline__ uint32_t load_and_count_ff(const uint8_t* __restrict__ raw, uint64_t at, uint64_t nbytes, uint32_t (&wv)[4], int& n) {
    uint4 q = make_uint4(0, 0, 0, 0);
    n = 0;
    if (at < nbytes) {
        n = static_cast<int>(umin64(16, nbytes - at));
        q = *reinterpret_cast<const uint4*>(raw + at);             // raw is padded to a multiple of 16 bytes and zero-filled
    }
    wv[0] = q.x; wv[1] = q.y; wv[2] = q.z; wv[3] = q.w;
    if (n < 16) {
#pragma unroll
        for (int j = 0; j < 16; ++j)
            if (j >= n) wv[j >> 2] &= ~(0xFFu << (8 * (j & 3)));
    }
    return (__popc(__vcmpeq4(wv[0], 0xFFFFFFFFu)) + __popc(__vcmpeq4(wv[1], 0xFFFFFFFFu)) + __popc(__vcmpeq4(wv[2], 0xFFFFFFFFu)) +
            __popc(__vcmpeq4(wv[3], 0xFFFFFFFFu))) >> 3;
}

// ---- K4a: FF bytes per tile.  The raw scan has just been written (it sits in L2); counting it first lets every K4 CTA
// compute its output position by ADDING the counts of the tiles before it -- no ticket, no look-back chain in which a
// tile waits for its predecessors (ncu on the look-back version: 47 % of K4's samples at the barrier behind the look-back).
constexpr int kCountThreads = 256;
__global__ void __launch_bounds__(kCountThreads) ff_count_kernel(const __grid_constant__ EntropyParams p) {
    __shared__ uint32_t s_part[kCountThreads / 32];
    if (p.hdr->error) return;
    const uint32_t gtile = blockIdx.x;
    if (gtile >= p.hdr->k4_tiles) return;                      // the grid is an upper bound (the exact count is only known on the device)
    const uint32_t frame = frame_of_tile(p, gtile), tile = gtile - p.k4_tile0[frame];
    const uint64_t nbytes = p.raw_bytes[frame];
    const uint8_t* __restrict__ raw = reinterpret_cast<const uint8_t*>(p.raw) + p.raw_off[frame];
    const uint64_t tile_at = static_cast<uint64_t>(tile) * kK4TileBytes;
    uint32_t ff = 0;
#pragma unroll
    for (int r = 0; r < static_cast<int>(kK4TileBytes) / (kCountThreads * 16); ++r) {
        uint32_t wv[4];
        int n;
        ff += load_and_count_ff(raw, tile_at + (static_cast<uint64_t>(r) * kCountThreads + threadIdx.x) * 16, nbytes, wv, n);
    }
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) ff += __shfl_xor_sync(0xffffffffu, ff, d);
    if ((threadIdx.x & 31) == 0) s_part[threadIdx.x >> 5] = ff;
    __syncthreads();
    if (threadIdx.x == 0) {
        uint32_t sum = 0;
        for (int w = 0; w < kCountThreads / 32; ++w) sum += s_part[w];
        p.tile_ff[gtile] = sum;
    }
}

// geom: null for frames of one size (their SOF0 is the prefix's), else the geometry of images of individual sizes
__device__ __forceinline__ void stuff_body(const EntropyParams& p, uint8_t* __restrict__ scan, const FrameGeom* geom, unsigned thread) {
    __shared__ alignas(16) uint8_t s_out[2 * kStuffTile + 16];
    __shared__ uint32_t s_scan[33];
    __shared__ unsigned long long s_before[kStuffThreads / 32];
    const int tid = thread;
    if (p.hdr->error) return;
    // tiles are numbered frame by frame through the whole pass; the grid is an upper bound: surplus CTAs leave at once
    const uint32_t gtile = blockIdx.x;
    if (gtile >= p.hdr->k4_tiles) return;
    const uint32_t frame = frame_of_tile(p, gtile), tile = gtile - p.k4_tile0[frame];
    const uint64_t nbytes = p.raw_bytes[frame];
    const uint8_t* __restrict__ raw = reinterpret_cast<const uint8_t*>(p.raw) + p.raw_off[frame];
    uint8_t* __restrict__ file = scan + p.file_base[frame];       // + the FFs stuffed before this frame: part of `base`
    uint8_t* __restrict__ out = file + p.hdr_len[frame];
    const uint64_t tile_at = static_cast<uint64_t>(tile) * kStuffTile;
    // FFs of all earlier tiles of the PASS: a sum over K4a's counts (a few hundred to a few thousand values)
    unsigned long long before = 0;
    for (uint32_t i = tid; i < gtile; i += kStuffThreads) before += __ldcg(p.tile_ff + i);
#pragma unroll
    for (int d = 16; d > 0; d >>= 1) before += __shfl_xor_sync(0xffffffffu, before, d);
    if ((tid & 31) == 0) s_before[tid >> 5] = before;
    uint32_t wv[4];
    int n;
    const uint32_t ff = load_and_count_ff(raw, tile_at + static_cast<uint64_t>(tid) * kStuffBytesPerThread, nbytes, wv, n);
    uint32_t tile_ff;
    const uint32_t local = block_exclusive_scan(ff, s_scan, &tile_ff);       // (its barriers also publish s_before)
    unsigned long long base = 0;
#pragma unroll
    for (int w = 0; w < kStuffThreads / 32; ++w) base += s_before[w];
    // ---- assemble the tile's output at tile-relative positions ----
    uint32_t o = tid * kStuffBytesPerThread + local;
    if (ff == 0 && n == 16) {
        const uint32_t lead = (4u - (o & 3u)) & 3u;            // bytes up to the next word boundary
        if (lead == 0) {
            *reinterpret_cast<uint32_t*>(s_out + o) = wv[0];
            *reinterpret_cast<uint32_t*>(s_out + o + 4) = wv[1];
            *reinterpret_cast<uint32_t*>(s_out + o + 8) = wv[2];
            *reinterpret_cast<uint32_t*>(s_out + o + 12) = wv[3];
        } else {
            for (uint32_t j = 0; j < lead; ++j) s_out[o + j] = static_cast<uint8_t>(wv[0] >> (8 * j));
            const uint32_t sh = 8 * lead;
            uint32_t* w = reinterpret_cast<uint32_t*>(s_out + o + lead);
            w[0] = __funnelshift_r(wv[0], wv[1], sh);
            w[1] = __funnelshift_r(wv[1], wv[2], sh);
            w[2] = __funnelshift_r(wv[2], wv[3], sh);
            for (uint32_t j = 0; j < 4u - lead; ++j) s_out[o + lead + 12 + j] = static_cast<uint8_t>(wv[3] >> (sh + 8 * j));
        }
    } else {
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            if (j < n) {
                const uint8_t b = static_cast<uint8_t>((wv[j >> 2] >> (8 * (j & 3))) & 0xFFu);
                s_out[o++] = b;
                if (b == 0xFF) s_out[o++] = 0;
            }
        }
    }
    __syncthreads();
    // ---- copy out: global word w holds tile-relative bytes [4w - sh, 4w - sh + 4) ----
    const uint32_t in_tile = static_cast<uint32_t>(umin64(kStuffTile, nbytes - tile_at));
    const uint32_t len = in_tile + tile_ff;
    uint8_t* g = out + tile_at + base;
    const uint32_t sh = static_cast<uint32_t>(reinterpret_cast<uintptr_t>(g) & 3u);
    const uint32_t head = min(len, (4u - sh) & 3u);            // bytes before the first aligned global word
    const uint32_t nwords = (len - head) >> 2;
    if (tid < head) g[tid] = s_out[tid];
    const uint32_t* sw = reinterpret_cast<const uint32_t*>(s_out);
    uint32_t* gw = reinterpret_cast<uint32_t*>(g + head);
    for (uint32_t w = tid; w < nwords; w += kStuffThreads)
        gw[w] = head ? __funnelshift_r(sw[w], sw[w + 1], 8 * head) : sw[w];
    const uint32_t tail0 = head + 4 * nwords;
    if (tid < len - tail0) g[tail0 + tid] = s_out[tail0 + tid];
    if (tile_at + kStuffTile >= nbytes) {                      // the frame's last tile
        if (tid == 0) {
            p.ff_incl[frame] = base + tile_ff;
            if (p.mailbox) {
                // one image: scan bits (K3b wrote them, a kernel ago) and stuffed FF bytes go straight to the host's mailbox as
                // self-validating words -- no publishing kernel behind K4
                const uint32_t seq = *p.dseq + 1u;
                volatile unsigned long long* box = p.mailbox + kMailTotals;
                box[0] = mail_word(__ldcg(p.total_bits + frame), seq);
                box[1] = mail_word(base + tile_ff, seq);
                *p.dseq = seq;
            }
        }
        if (tid < p.tail) g[len + tid] = tid ? 0xD9 : 0xFF;   // EOI (JpegSegments.hpp:361-377)
    }
    if (tile == 0 && p.hdr_len[frame]) write_file_header(file + base, p, frame, tid, kStuffThreads, geom);
}

__global__ void __launch_bounds__(kStuffThreads, 6) stuff_kernel(const __grid_constant__ EntropyParams p, uint8_t* __restrict__ scan) {
    stuff_body(p, scan, nullptr, threadIdx.x);
}
__global__ void __launch_bounds__(kStuffThreads, 6) stuff_mixed_kernel(const __grid_constant__ EntropyParams p, uint8_t* __restrict__ scan,
                                                                       const FrameGeom* __restrict__ geom) {
    stuff_body(p, scan, geom, threadIdx.x);
}

// Frame geometry (raw offsets, sizes, K4 tile numbering, output positions) is read from the PassMeta block in device
// memory (c->d_meta): written there by the host for one image, by finalize_tables_kernel for a batch.  `k4_grid` is an
// upper bound of the number of K4 tiles (exact when the host computed the geometry).
int launch_entropy(jpgenc_ctx* c, uint32_t k4_grid) {
    const uint64_t n_mcu = static_cast<uint64_t>(c->mcu_w) * c->mcu_h, nblocks = n_mcu * kBlocksPerMcu;
    const uint32_t F = c->nframes;
    EntropyParams p{};
    p.items = c->d_items;
    p.range_cnt = c->d_tile_cnt;
    p.nframes = F;
    const uint32_t tiles = static_cast<uint32_t>((nblocks + kTileBlocks - 1) / kTileBlocks);
    // one warp walks one range; a small image has too few tiles to occupy the GPU (3840x2160: 507 tiles = 64 CTAs, and every
    // warp walks ~1600 items one after the other), so its tiles are cut into four ranges each
    p.split = static_cast<uint64_t>(tiles) * F < 4096 ? 4u : 1u;
    p.ranges_per_frame = tiles * p.split;
    p.groups_per_frame = (p.ranges_per_frame + kPackWarps - 1) / kPackWarps;
    p.supers_per_frame = (p.groups_per_frame + 255) / 256;
    p.tables = c->d_tables;
    p.range_bits = c->d_range_bits;
    p.group_bits = c->d_range_base;                                  // [F * groups] then [F * supers]
    p.super_bits = c->d_range_base + static_cast<size_t>(F) * p.groups_per_frame;
    size_t groups = static_cast<size_t>(F) * p.groups_per_frame, supers = static_cast<size_t>(F) * p.supers_per_frame;
    if (c->mixed.on) {
        // images of individual sizes: the pass's own counts (FrameGeom, host-built with the same split rule over the pass's
        // tiles); the per-frame counts above are replaced per CTA (entropy_image)
        p.split = c->mixed.split;
        groups = c->mixed.groups;
        supers = c->mixed.supers;
        p.super_bits = c->d_range_base + groups;
    }
    if (c->entropy_runs) {
        // K3a ADDS into the super-group sums, which launch_symbol_stats cleared: a second entropy pass over the same
        // symbol items (other tables) must start from zero again
        JPGENC_CUDA(c, cudaMemsetAsync(p.super_bits, 0, supers * sizeof(unsigned long long), c->stream));
    }
    ++c->entropy_runs;
    p.raw = c->d_raw;
    const PassMeta m = pass_meta_view(c->d_meta, F);
    p.hdr = m.hdr;
    p.raw_off = m.raw_off;
    p.raw_bytes = m.raw_bytes;
    p.k4_tile0 = m.k4_tile0;
    p.file_base = m.file_base;
    p.hdr_len = m.hdr_len;
    p.total_bits = m.total_bits;
    p.ff_incl = m.ff_incl;
    p.tile_ff = reinterpret_cast<uint32_t*>(c->d_lookback);
    p.redo_count = c->d_counters + kCntK3Redo;
    if (F == 1 && !c->file_mode && k4_grid) {                    // one image: K4's last tile writes the totals into the host's mailbox
        p.mailbox = c->d_mailbox;
        p.dseq = c->d_counters + kCntSeq;
        ++c->mailbox_seq;                                        // the sequence number those words will be tagged with
    }
    if (c->file_mode) {
        p.built = c->d_built_tables;
        p.hdr_prefix = c->d_hdr_prefix;
        p.hdr_prefix_len = c->hdr_prefix_len;
        p.tail = 2;
    }
    const unsigned grid = static_cast<unsigned>(groups);
    if (c->mixed.on) {
        range_bits_mixed_kernel<<<grid, kPackThreads, 0, c->stream>>>(p, c->d_geom);
        JPGENC_CUDA(c, cudaGetLastError());
        huffman_pack_mixed_kernel<<<grid, kPackThreads, 0, c->stream>>>(p, c->d_geom);
    } else {
        range_bits_kernel<<<grid, kPackThreads, 0, c->stream>>>(p);
        JPGENC_CUDA(c, cudaGetLastError());
        huffman_pack_kernel<<<grid, kPackThreads, 0, c->stream>>>(p);
    }
    JPGENC_CUDA(c, cudaGetLastError());
    if (k4_grid) {
        ff_count_kernel<<<k4_grid, kCountThreads, 0, c->stream>>>(p);
        JPGENC_CUDA(c, cudaGetLastError());
        if (c->mixed.on) stuff_mixed_kernel<<<k4_grid, kStuffThreads, 0, c->stream>>>(p, c->d_scan, c->d_geom);
        else stuff_kernel<<<k4_grid, kStuffThreads, 0, c->stream>>>(p, c->d_scan);
        JPGENC_CUDA(c, cudaGetLastError());
        c->launches += 2;
    }
    c->launches += 2;
    return JPGENC_OK;
}

}  // namespace jpgenc
