// K1 — fused colour conversion + 4:2:0 mean subsampling + Arai DCT + quantisation + zigzag.
//
// Replaces Image::convertToColorSpace / applySubsampling(S420_m) / applyDCT(Arai) / applyQuantization
// (reference src/Image.cpp:112-148, 198-235, 540-595, 597-636; include/Dct.hpp:47-215; include/Coding.hpp:57-97).
//
// Design (DESIGN.md "K1"):
//  * one CTA = a strip of kMcus 16x16 MCUs; the RGB strip (16 rows) is staged in shared memory by bulk
//    (TMA) copies, one per image row, completing on an mbarrier;
//  * one thread = one 8x8 block, held entirely in registers as 32 packed float pairs: no shuffles, 30 packed FP32x2
//    instructions per PAIR of 8-point AAN passes; the AAN output scales and 1/q are folded into one multiplier per
//    coefficient;
//  * the reference computes in double.  The FP32 result is only trusted when every quotient is further than
//    delta from a rounding boundary; otherwise the block id goes to a refine list and refine_kernel redoes
//    the block in FP64 with the reference's exact operation order (no FMA contraction), so the stored
//    coefficients are the reference's, bit for bit;
//  * coefficients leave through a bank-conflict-free swizzled staging buffer as full 512-byte warp stores,
//    already in the MCU-interleaved order the entropy coder consumes.
#include <algorithm>
#include <cmath>
#include <type_traits>

#include "common.cuh"
#include "exact.cuh"
#include "ptx.cuh"

namespace jpgenc {

__constant__ uint8_t c_zigzag[64] = {JPGENC_ZIGZAG_LIST};

// ---------------------------------------------------------------------------------------------------
// FP32 fast path, packed FP32x2 (sm_100 FADD2 / FFMA2: two IEEE fp32 operations per issue slot)
// ---------------------------------------------------------------------------------------------------
// K1 is bound by instruction issue, not by the FP32 pipes or HBM (ncu, profiles/): as scalar code two thirds of its
// instructions were FADD/FFMA.  Blackwell's packed forms halve those.  The 8-point AAN butterfly has the dataflow of
// Dct.hpp:52-131 re-associated for FMA (30 operations) and leaves out the s_k output scales: they are folded, together
// with 1/q, into one multiplier per coefficient (QuantConsts2::mul).  A block is held as 32 float2: in the first (vertical) pass a
// pair is two neighbouring columns, so the eight 1-D column transforms run as four packed ones; 2x2 register
// transposes then turn pairs of columns into pairs of rows for the horizontal pass.  Every lane of a packed operation is
// an ordinary round-to-nearest fp32 operation, so the results (and the error bound behind the refinement threshold)
// are those of the scalar code.
using f2 = float2;
__device__ __forceinline__ f2 add2(f2 a, f2 b) { return __fadd2_rn(a, b); }
__device__ __forceinline__ f2 sub2(f2 a, f2 b) { return __fadd2_rn(a, make_float2(-b.x, -b.y)); }
__device__ __forceinline__ f2 fma2(f2 a, f2 b, f2 c) { return __ffma2_rn(a, b, c); }
__device__ __forceinline__ f2 fma2s(f2 a, float k, f2 c) { return __ffma2_rn(a, make_float2(k, k), c); }
__device__ __forceinline__ f2 neg2(f2 a) { return make_float2(-a.x, -a.y); }

__device__ __forceinline__ void aan8x2(f2& x0, f2& x1, f2& x2, f2& x3, f2& x4, f2& x5, f2& x6, f2& x7) {
    constexpr float A1 = 0.70710678118654752f, A2 = 0.54119610014619698f, A4 = 1.30656296487637653f,
                    A5 = 0.38268343236508977f;
    const f2 z0 = add2(x0, x7), z1 = add2(x1, x6), z2 = add2(x2, x5), z3 = add2(x3, x4);
    const f2 z4 = sub2(x3, x4), z5 = sub2(x2, x5), z6 = sub2(x1, x6), z7 = sub2(x0, x7);
    const f2 r0 = add2(z0, z3), r1 = add2(z1, z2), r2 = sub2(z1, z2), r3 = sub2(z0, z3);
    const f2 n4 = add2(z4, z5);
    const f2 r5 = add2(z5, z6), r6 = add2(z6, z7);
    const f2 t2 = add2(r2, r3);
    const f2 d = sub2(r6, n4);
    const f2 tmp = __fmul2_rn(d, make_float2(A5, A5));
    const f2 u4 = fma2s(n4, A2, neg2(tmp));
    const f2 u6 = fma2s(r6, A4, neg2(tmp));
    const f2 v5 = fma2s(r5, A1, z7);
    const f2 v7 = fma2s(r5, -A1, z7);
    x0 = add2(r0, r1);
    x4 = sub2(r0, r1);
    x2 = fma2s(t2, A1, r3);
    x6 = fma2s(t2, -A1, r3);
    x5 = add2(u4, v7);
    x1 = add2(v5, u6);
    x7 = sub2(v5, u6);
    x3 = sub2(v7, u4);
}

// Same butterfly, but the last stage is done with scalar operations so that the 16 results can land in ANY registers:
// o[k] receives frequency k of the first lane (.x of the inputs), o[8 + k] that of the second lane.  Used for the
// vertical pass, whose results have to be re-paired (two rows instead of two columns) for the horizontal pass; letting
// the final additions write straight into the new pairs costs 8 extra instructions per call and saves the
// register-to-register moves of an explicit 2x2 transpose.
__device__ __forceinline__ void aan8x2_split(const f2& x0, const f2& x1, const f2& x2, const f2& x3, const f2& x4, const f2& x5,
                                             const f2& x6, const f2& x7, float (&o)[16]) {
    constexpr float A1 = 0.70710678118654752f, A2 = 0.54119610014619698f, A4 = 1.30656296487637653f,
                    A5 = 0.38268343236508977f;
    const f2 z0 = add2(x0, x7), z1 = add2(x1, x6), z2 = add2(x2, x5), z3 = add2(x3, x4);
    const f2 z4 = sub2(x3, x4), z5 = sub2(x2, x5), z6 = sub2(x1, x6), z7 = sub2(x0, x7);
    const f2 r0 = add2(z0, z3), r1 = add2(z1, z2), r2 = sub2(z1, z2), r3 = sub2(z0, z3);
    const f2 n4 = add2(z4, z5);
    const f2 r5 = add2(z5, z6), r6 = add2(z6, z7);
    const f2 t2 = add2(r2, r3);
    const f2 d = sub2(r6, n4);
    const f2 tmp = __fmul2_rn(d, make_float2(A5, A5));
    const f2 u4 = fma2s(n4, A2, neg2(tmp));
    const f2 u6 = fma2s(r6, A4, neg2(tmp));
    const f2 v5 = fma2s(r5, A1, z7);
    const f2 v7 = fma2s(r5, -A1, z7);
    o[0] = r0.x + r1.x;            o[8 + 0] = r0.y + r1.y;
    o[4] = r0.x - r1.x;            o[8 + 4] = r0.y - r1.y;
    o[2] = fmaf(t2.x, A1, r3.x);   o[8 + 2] = fmaf(t2.y, A1, r3.y);
    o[6] = fmaf(t2.x, -A1, r3.x);  o[8 + 6] = fmaf(t2.y, -A1, r3.y);
    o[5] = u4.x + v7.x;            o[8 + 5] = u4.y + v7.y;
    o[1] = v5.x + u6.x;            o[8 + 1] = v5.y + u6.y;
    o[7] = v5.x - u6.x;            o[8 + 7] = v5.y - u6.y;
    o[3] = v7.x - u4.x;            o[8 + 3] = v7.y - u4.y;
}

// in : v[r*4+p] = (s[r][2p], s[r][2p+1])   spatial samples, pairs of neighbouring columns
// out: v[u*4+q] = (F[2q][u], F[2q+1][u])   unscaled frequencies F[v][u], pairs of neighbouring vertical frequencies
// kSplit picks how the pairs are re-formed between the passes: scalar last butterfly stage (fewer instructions: K1,
// which is bound by instruction issue) or packed butterflies + explicit 2x2 register transposes (fewer FP32 operations
// in flight: the stand-alone block kernel, which is bound by HBM and was 20 % slower with the scalar stage).
template <bool kSplit>
__device__ __forceinline__ void dct8x8_packed(f2 (&v)[32]) {
    f2 t[32];                                     // t[c*4+q] = (T[2q][c], T[2q+1][c]): column c after the vertical pass
    if constexpr (kSplit) {
#pragma unroll
        for (int p = 0; p < 4; ++p) {
            float o[16];
            aan8x2_split(v[0 * 4 + p], v[1 * 4 + p], v[2 * 4 + p], v[3 * 4 + p], v[4 * 4 + p], v[5 * 4 + p], v[6 * 4 + p], v[7 * 4 + p], o);
#pragma unroll
            for (int q = 0; q < 4; ++q) {
                t[(2 * p) * 4 + q] = make_float2(o[2 * q], o[2 * q + 1]);
                t[(2 * p + 1) * 4 + q] = make_float2(o[8 + 2 * q], o[8 + 2 * q + 1]);
            }
        }
    } else {
#pragma unroll
        for (int p = 0; p < 4; ++p)
            aan8x2(v[0 * 4 + p], v[1 * 4 + p], v[2 * 4 + p], v[3 * 4 + p], v[4 * 4 + p], v[5 * 4 + p], v[6 * 4 + p], v[7 * 4 + p]);
#pragma unroll
        for (int q = 0; q < 4; ++q)
#pragma unroll
            for (int p = 0; p < 4; ++p) {
                const f2 a = v[(2 * q) * 4 + p], b = v[(2 * q + 1) * 4 + p];
                t[(2 * p) * 4 + q] = make_float2(a.x, b.x);
                t[(2 * p + 1) * 4 + q] = make_float2(a.y, b.y);
            }
    }
#pragma unroll
    for (int q = 0; q < 4; ++q)
        aan8x2(t[0 * 4 + q], t[1 * 4 + q], t[2 * 4 + q], t[3 * 4 + q], t[4 * 4 + q], t[5 * 4 + q], t[6 * 4 + q], t[7 * 4 + q]);
#pragma unroll
    for (int i = 0; i < 32; ++i) v[i] = t[i];
}

// QuantConsts2: the same multipliers/thresholds as QuantConsts, stored in the pair order dct8x8_packed leaves:
// entry [u*4+q] = (natural index (2q)*8+u, natural index (2q+1)*8+u)
__device__ __forceinline__ bool quantize_pack_packed(const f2 (&v)[32], const QuantConsts2& q, uint32_t (&out)[32]) {
    constexpr float kMagic = 12582912.f;
    constexpr int zz[64] = {JPGENC_ZIGZAG_LIST};
    uint32_t bits[64];
    bool boundary = false;
#pragma unroll
    for (int u = 0; u < 8; ++u)
#pragma unroll
        for (int qq = 0; qq < 4; ++qq) {
            const int j = u * 4 + qq;
            const f2 a = fma2(v[j], q.mul[j], make_float2(kMagic, kMagic));
            const f2 k = add2(a, make_float2(-kMagic, -kMagic));
            const f2 d = fma2(v[j], q.mul[j], neg2(k));
            boundary |= fabsf(d.x) > q.thr[j].x;
            boundary |= fabsf(d.y) > q.thr[j].y;
            bits[(2 * qq) * 8 + u] = __float_as_uint(a.x);
            bits[(2 * qq + 1) * 8 + u] = __float_as_uint(a.y);
        }
#pragma unroll
    for (int j = 0; j < 32; ++j) out[j] = __byte_perm(bits[zz[2 * j]], bits[zz[2 * j + 1]], 0x5410);
    return boundary;
}

// bytes `lo` and `hi` of the 24-byte row segment w[] as floats: PRMT splices each byte under the exponent of 2^23
// (0x4B0000bb == 8388608 + b exactly), one packed subtraction removes the 2^23.  Runs on the ALU + FMA pipes; the
// plain I2F.U8 conversion is a quarter-rate XU instruction (measured: routing one to three of the channels through
// I2F instead changes K1's time by -0.6 % .. +4 %, so the single PRMT path is kept).
template <int N>
__device__ __forceinline__ f2 bytes_to_f2(const uint32_t (&w)[N], int lo, int hi) {
    const uint32_t a = __byte_perm(w[lo >> 2], 0x4B000000u, 0x7650 | (lo & 3));
    const uint32_t b = __byte_perm(w[hi >> 2], 0x4B000000u, 0x7650 | (hi & 3));
    return add2(make_float2(__uint_as_float(a), __uint_as_float(b)), make_float2(-8388608.f, -8388608.f));
}

// the same with the level shift of YUV samples folded in: 8388608 + b - 8388736 == b - 128, exact
template <int N>
__device__ __forceinline__ f2 bytes_to_f2_centred(const uint32_t (&w)[N], int lo, int hi) {
    const uint32_t a = __byte_perm(w[lo >> 2], 0x4B000000u, 0x7650 | (lo & 3));
    const uint32_t b = __byte_perm(w[hi >> 2], 0x4B000000u, 0x7650 | (hi & 3));
    return add2(make_float2(__uint_as_float(a), __uint_as_float(b)), make_float2(-8388736.f, -8388736.f));
}

// staging slot layout: 128 B per block, 16-byte chunk c of slot s lives at chunk (c ^ (s & 7)) — conflict-free
// both for the per-thread 16-byte writes and for the linear copy-out
__device__ __forceinline__ void stage_block(uint8_t* staging, int slot, const uint32_t (&w)[32]) {
    uint4* base = reinterpret_cast<uint4*>(staging + slot * kBlockBytes);
#pragma unroll
    for (int c = 0; c < 8; ++c) base[c ^ (slot & 7)] = make_uint4(w[4 * c], w[4 * c + 1], w[4 * c + 2], w[4 * c + 3]);
}
__device__ __forceinline__ void copy_out(const uint8_t* staging, int16_t* gdst, int nslots, int tid, int nthreads) {
    uint4* g = reinterpret_cast<uint4*>(gdst);
    const int chunks = nslots * 8;
    for (int j = tid; j < chunks; j += nthreads) {
        const int s = j >> 3, c = j & 7;
        g[j] = *reinterpret_cast<const uint4*>(staging + s * kBlockBytes + ((c ^ (s & 7)) << 4));
    }
}

__device__ __forceinline__ void push_refine(const ForwardParams& p, uint32_t block_id) {
    const uint32_t at = atomicAdd(p.refine_count, 1u);
    if (at < p.refine_cap) p.refine_list[at] = block_id;
}

template <int kMcus>
struct ForwardSmem {
    static constexpr int kPitch = kMcus * 48;                 // bytes of RGB per tile row
    static constexpr int kTileBytes = 16 * kPitch;            // == kMcus*6*128: the staging buffer aliases it
    static constexpr int kChromaW = kMcus * 8;
    alignas(1024) uint8_t tile[kTileBytes];               // 1 KB: the 128-byte swizzle of the tensor store is taken from address bits 7..9
    alignas(16) float chroma[2][8][kChromaW];
    alignas(8) uint64_t bar;
};

// The image of a K1 strip and where the strip lies in it
struct StripImage {
    PixelSource src;                      // planes and pitches (the format is the kernel's template parameter)
    uint32_t real_w, real_h, mcu_w;
    uint32_t block0;                      // the image's first coefficient block
    uint32_t my, mcu0;                    // the strip's MCU row and first MCU column
};

// A strip's position in the grid: the CTA's own (ThisCta; each coordinate is read where it is used, which keeps the scheduling
// of the tight-RGB kernels) or another one (GridPos)
struct ThisCta {
    __device__ uint32_t x() const { return blockIdx.x; }
    __device__ uint32_t y() const { return blockIdx.y; }
    __device__ uint32_t z() const { return blockIdx.z; }
};
struct GridPos {
    uint32_t x_, y_, z_;
    __device__ uint32_t x() const { return x_; }
    __device__ uint32_t y() const { return y_; }
    __device__ uint32_t z() const { return z_; }
};

// The image of strip (x, y, z) of the one-size grid (strip of the row, MCU row of the launch, frame), or of strip x of the grid
// over images of individual sizes: there the image is found by a search over the first-strip prefix, in which every lane of
// the warp takes part.
template <int kMcus, bool kMixed, int kFmt, class Pos>
__device__ __forceinline__ StripImage strip_image(const ForwardParams& p, Pos at) {
    StripImage s;
    if constexpr (kMixed) {
        const uint32_t gi = geom_find_warp(p.geom, p.nframes, at.x(), &FrameGeom::strip0);
        const FrameGeom& g = p.geom[gi];
        if constexpr (source_planes(kFmt) == 3) {
            const ExtraPlanes& e = p.extra[gi];
            s.src.plane[1] = e.plane[0];
            s.src.plane[2] = e.plane[1];
            s.src.pitch2 = static_cast<uint32_t>(e.pitch2);
        }
        s.mcu_w = g.mcu_w;
        const uint32_t per_row = (s.mcu_w + kMcus - 1) / kMcus, k = at.x() - g.strip0;
        s.my = k / per_row;
        s.mcu0 = (k - s.my * per_row) * kMcus;
        s.src.plane[0] = g.rgb;
        s.block0 = g.block0;
        s.real_w = g.real_w;
        s.real_h = g.real_h;
        s.src.pitch = g.pitch;
    } else {
        s.my = p.mcu_y0 + at.y();
        s.mcu0 = at.x() * kMcus;
        s.src = p.src;
        s.src.plane[0] = p.frames ? p.frames[at.z()] : p.rgb;             // batch: grid.z walks over the frames
        s.block0 = at.z() * p.blocks_per_frame;
        s.real_w = p.real_w;
        s.real_h = p.real_h;
        s.mcu_w = p.mcu_w;
    }
    return s;
}

// The image of the strip `prefetch_ahead` CTAs after this one, for the L2 prefetch of the pixel-layout kernels; false past the
// end of the grid (the one-size grid of these kernels holds one image).  Called by a whole warp.
template <int kMcus, bool kMixed, int kFmt>
__device__ __forceinline__ bool ahead_image(const ForwardParams& p, StripImage& s) {
    if constexpr (kMixed) {
        const uint32_t t = blockIdx.x + p.prefetch_ahead;
        if (t >= p.strips) return false;                                    // uniform over the warp
        s = strip_image<kMcus, true, kFmt>(p, GridPos{t, 0, 0});
    } else {
        const uint32_t lin = blockIdx.y * gridDim.x + blockIdx.x + p.prefetch_ahead, y = lin / gridDim.x;
        if (y >= gridDim.y) return false;
        s = strip_image<kMcus, false, kFmt>(p, GridPos{lin - y * gridDim.x, y, blockIdx.z});
    }
    return true;
}

// Staging of the pixel-layout kernels: the same 16-row tile of 3 bytes per pixel, in the byte order of the source (the colour
// read below swaps R and B of BGR / BGRA at compile time).  Each CTA picks its path from its own image:
//  * 3 bytes per pixel, base and pitch 16-byte aligned, real_w % 16 == 0: one bulk copy per row, as forward_kernel;
//  * 4 bytes per pixel: 16-byte vector loads (4 pixels) from a 16-byte aligned base and pitch, each turned into 12 bytes of the
//    tile by three byte permutes (the 4th byte never reaches the tile); a 4-byte strip staged whole would be 32 KB and cost
//    K1 its 5 CTAs per SM.  Chunks past the right edge, and every chunk of an unaligned image, take clamped byte loads;
//  * otherwise a clamped byte loader with the pitch.
template <int kMcus, int kFmt, bool kMixed>
__device__ __forceinline__ void stage_layout(const ForwardParams& p, ForwardSmem<kMcus>& sm, int tid, const StripImage& s, int nm) {
    using Smem = ForwardSmem<kMcus>;
    constexpr int kThreads = kMcus * 4;
    constexpr uint32_t kBpp = pixel_bytes(kFmt);
    const uint8_t* __restrict__ rgb = s.src.plane[0];
    const uint32_t pitch = s.src.pitch, real_w = s.real_w, real_h = s.real_h, my = s.my, mcu0 = s.mcu0;
    const bool aligned = ((reinterpret_cast<uintptr_t>(rgb) | pitch) & 15) == 0;
    const bool bulk = kBpp == 3 && aligned && real_w % 16 == 0;           // the same for every thread of the CTA
    if (bulk) {
        if (tid == 0) {
            ptx::mbar_init(&sm.bar, 1);
            ptx::mbar_init_fence();
        }
        __syncthreads();
        if (tid < 16) {
            const uint32_t row_bytes = nm * 48;
            if (tid == 0) ptx::mbar_expect_tx(&sm.bar, 16 * row_bytes);
            const uint32_t sy = min(my * 16 + tid, real_h - 1);
            ptx::bulk_g2s(sm.tile + tid * Smem::kPitch, rgb + static_cast<size_t>(sy) * pitch + mcu0 * 48, row_bytes, &sm.bar);
        }
    }
    // the strip `prefetch_ahead` CTAs later into L2, when its rows are whole 16-byte multiples inside the image (the range must
    // not pass the end of a row)
    if (p.prefetch_ahead && tid >= 32 && tid < 64) {
        StripImage a;
        if (ahead_image<kMcus, kMixed, kFmt>(p, a) && tid < 48 && ((reinterpret_cast<uintptr_t>(a.src.plane[0]) | a.src.pitch | a.real_w) & 15) == 0) {
            const uint32_t pnm = min(static_cast<uint32_t>(kMcus), a.mcu_w - a.mcu0);
            const uint32_t sy = min(a.my * 16 + (tid - 32), a.real_h - 1);
            ptx::bulk_prefetch_l2(a.src.plane[0] + static_cast<size_t>(sy) * a.src.pitch + a.mcu0 * 16 * kBpp, pnm * 16 * kBpp);
        }
    }
    if (bulk) {
        ptx::mbar_wait(&sm.bar, 0);
        return;
    }
    if constexpr (kBpp == 4) {
        if (tid < nm * 4) {                                                 // thread = 4 pixels of every row of the strip
            const uint32_t x0 = mcu0 * 16 + tid * 4;
            const bool vec = aligned && x0 + 4 <= real_w;
#pragma unroll 4
            for (int r = 0; r < 16; ++r) {
                const uint8_t* row = rgb + static_cast<size_t>(min(my * 16 + r, real_h - 1)) * pitch;
                uint32_t q[4];
                if (vec) {
                    const uint4 v = __ldg(reinterpret_cast<const uint4*>(row + x0 * 4));
                    q[0] = v.x; q[1] = v.y; q[2] = v.z; q[3] = v.w;
                } else {
#pragma unroll
                    for (int k = 0; k < 4; ++k) {
                        const uint8_t* px = row + min(x0 + k, real_w - 1) * 4;
                        q[k] = px[0] | (px[1] << 8) | (px[2] << 16);
                    }
                }
                uint32_t* dst = reinterpret_cast<uint32_t*>(sm.tile + r * Smem::kPitch + tid * 12);
                dst[0] = __byte_perm(q[0], q[1], 0x4210);                  // c0 c1 c2 | c0 of the next pixel ...
                dst[1] = __byte_perm(q[1], q[2], 0x5421);
                dst[2] = __byte_perm(q[2], q[3], 0x6542);
            }
        }
    } else {
        const int row_bytes = nm * 48;
        for (int idx = tid; idx < 16 * row_bytes; idx += kThreads) {
            const int r = idx / row_bytes, b = idx - r * row_bytes;
            const uint32_t sx = min(mcu0 * 16 + b / 3, real_w - 1);
            const uint32_t sy = min(my * 16 + r, real_h - 1);
            sm.tile[r * Smem::kPitch + b] = rgb[static_cast<size_t>(sy) * pitch + sx * 3 + (b % 3)];
        }
    }
    __syncthreads();
}

// Staging of grey (one plane) and planar RGB (three planes) pixels: the tile holds the strip in the source's own layout, kPlanes
// planes of 16 rows of kMcus * 16 bytes (planar: 24 KB, the whole tile), and the colour read in forward_body takes the three
// channels from the planes (grey: one byte for all three).  Interleaving the planes here instead would cost what the 4-byte
// formats' byte permutes cost above.  Each CTA picks its path from its own image:
//  * every plane's base and the pitch 16-byte aligned, real_w % 16 == 0: one bulk copy per plane row (16 / 48 per CTA);
//  * otherwise 16-byte chunks: a vector load where the chunk lies inside an aligned image, clamped byte loads elsewhere.
// The L2 prefetch of the strip `prefetch_ahead` CTAs later covers every plane.
template <int kMcus, int kFmt, bool kMixed>
__device__ __forceinline__ void stage_planes(const ForwardParams& p, ForwardSmem<kMcus>& sm, int tid, const StripImage& s, int nm) {
    using Smem = ForwardSmem<kMcus>;
    constexpr int kThreads = kMcus * 4, kRow = kMcus * 16, kPlanes = source_planes(kFmt);
    static_assert(kPlanes * 16 * kRow <= Smem::kTileBytes, "the planes fit the tile");
    const auto& plane = s.src.plane;
    const uint32_t pitch = s.src.pitch, real_w = s.real_w, real_h = s.real_h, my = s.my, mcu0 = s.mcu0;
    auto pick = [](const auto& pl, int k) { return kPlanes == 1 || k == 0 ? pl[0] : k == 1 ? pl[1] : pl[2]; };
    uintptr_t bits = pitch;
#pragma unroll
    for (int k = 0; k < kPlanes; ++k) bits |= reinterpret_cast<uintptr_t>(plane[k]);
    const bool aligned = (bits & 15) == 0;
    const bool bulk = aligned && real_w % 16 == 0;                         // the same for every thread of the CTA
    if (bulk) {
        if (tid == 0) {
            ptx::mbar_init(&sm.bar, 1);
            ptx::mbar_init_fence();
        }
        __syncthreads();
        if (tid < 16 * kPlanes) {
            const uint32_t row_bytes = nm * 16;
            if (tid == 0) ptx::mbar_expect_tx(&sm.bar, 16 * kPlanes * row_bytes);
            const uint32_t sy = min(my * 16 + (tid & 15), real_h - 1);
            ptx::bulk_g2s(sm.tile + tid * kRow, pick(plane, tid >> 4) + static_cast<size_t>(sy) * pitch + mcu0 * 16, row_bytes, &sm.bar);
        }
    }
    if (p.prefetch_ahead && tid >= 32 && tid < 64) {
        StripImage a;
        if (ahead_image<kMcus, kMixed, kFmt>(p, a)) {
            const uint32_t pnm = min(static_cast<uint32_t>(kMcus), a.mcu_w - a.mcu0);
            for (int i = tid - 32; i < 16 * kPlanes; i += 32) {
                const uint8_t* src = pick(a.src.plane, i >> 4);
                if (((reinterpret_cast<uintptr_t>(src) | a.src.pitch | a.real_w) & 15) == 0) {
                    const uint32_t sy = min(a.my * 16 + (i & 15), a.real_h - 1);
                    ptx::bulk_prefetch_l2(src + static_cast<size_t>(sy) * a.src.pitch + a.mcu0 * 16, pnm * 16);
                }
            }
        }
    }
    if (bulk) {
        ptx::mbar_wait(&sm.bar, 0);
        return;
    }
    const int chunks = kPlanes * 16 * nm;                                   // 16 pixels of one plane row each
    for (int i = tid; i < chunks; i += kThreads) {
        const int k = i / (16 * nm), rm = i - k * 16 * nm, r = rm / nm, m = rm - r * nm;
        const uint8_t* row = pick(plane, k) + static_cast<size_t>(min(my * 16 + r, real_h - 1)) * pitch;
        const uint32_t x0 = (mcu0 + m) * 16;
        uint4 v;
        if (aligned && x0 + 16 <= real_w) {
            v = __ldg(reinterpret_cast<const uint4*>(row + x0));
        } else {                                                            // right edge replication, src/Image.cpp:491-530
            uint32_t q[4];
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const uint32_t x = x0 + 4 * j;
                q[j] = row[min(x, real_w - 1)] | (row[min(x + 1, real_w - 1)] << 8) | (row[min(x + 2, real_w - 1)] << 16) |
                       (static_cast<uint32_t>(row[min(x + 3, real_w - 1)]) << 24);
            }
            v = make_uint4(q[0], q[1], q[2], q[3]);
        }
        *reinterpret_cast<uint4*>(sm.tile + (k * 16 + r) * kRow + m * 16) = v;
    }
    __syncthreads();
}

// Staging of YUV frames: the tile holds the strip's 16 rows of the first plane and behind them its chroma rows, in the source's own
// layout.  kCRows chroma rows per MCU row (8 for 4:2:0, 16 for 4:2:2 and 4:4:4), kMcuC chroma bytes of one MCU in one row:
//  * I420 / NV12: 16 Y rows of kMcus * 16 bytes (8 KB at kMcus 32) and 8 chroma rows, U and V planes of rows of kMcus * 8 bytes
//    (I420) or one plane of rows of kMcus * 16 (U, V) bytes (NV12): 12 KB in all;
//  * I422 / NV16: 16 Y rows and 16 chroma rows of the same sizes: 16 KB;  I444: three planes of 16 rows of kMcus * 16 bytes: 24 KB;
//  * YUYV / UYVY: one plane of 16 rows of kMcus * 32 bytes (two bytes per pixel, the chroma inside): 16 KB.
// Each CTA picks its path from its own image:
//  * every plane's base and pitch 16-byte aligned, real_w % 16 == 0 (so no row needs padding either) and, with 8 chroma bytes
//    per MCU, an even number of MCUs (a bulk copy moves whole 16-byte units): one bulk copy per plane row (16 to 48 per CTA);
//  * otherwise 16-byte chunks, per plane: a vector load where the chunk lies inside the plane's row and the plane is aligned,
//    clamped byte loads elsewhere (edge replication, each plane clamped to its own size; NV12 / NV16 clamp whole U, V pairs, the
//    packed layouts clamp a pixel's Y to the last pixel and its U, V to the last group).
// The L2 prefetch of the strip `prefetch_ahead` CTAs later covers every plane.
template <int kMcus, int kFmt, bool kMixed>
__device__ __forceinline__ void stage_yuv(const ForwardParams& p, ForwardSmem<kMcus>& sm, int tid, const StripImage& s, int nm) {
    constexpr bool kPacked = is_packed_yuv(kFmt), kSemi = kFmt == kPixelNV12 || kFmt == kPixelNV16;
    constexpr int kYB = kPacked ? 32 : 16;                                 // bytes of one MCU in one row of the first plane
    constexpr int kMcuC = kSemi || kFmt == kPixelI444 ? 16 : 8;           // chroma bytes of one MCU in one row
    constexpr int kCRows = chroma_vsub(kFmt) ? 8 : 16, kCPlanes = kPacked ? 0 : kSemi ? 1 : 2;
    constexpr int kThreads = kMcus * 4, kRow = kMcus * kYB, kCRow = kMcus * kMcuC, kRows = 16 + kCRows * kCPlanes;
    static_assert(16 * kRow + kCPlanes * kCRows * kCRow <= ForwardSmem<kMcus>::kTileBytes, "the planes fit the tile");
    const uint8_t *y = s.src.plane[0], *u = s.src.plane[1], *v = s.src.plane[2];
    const uint32_t y_pitch = s.src.pitch, c_pitch = s.src.pitch2, real_w = s.real_w, real_h = s.real_h, my = s.my, mcu0 = s.mcu0;
    const uint32_t cw_bytes = chroma_row_bytes(kFmt, real_w), ch = kCRows == 8 ? (real_h + 1) / 2 : real_h;
    const bool y_aligned = ((reinterpret_cast<uintptr_t>(y) | y_pitch) & 15) == 0;
    const bool c_aligned = kPacked || ((reinterpret_cast<uintptr_t>(u) | (kCPlanes == 1 ? 0 : reinterpret_cast<uintptr_t>(v)) | c_pitch) & 15) == 0;
    const bool bulk = y_aligned && c_aligned && real_w % 16 == 0 && (kMcuC == 16 || nm % 2 == 0);   // the same for every thread of the CTA
    uint8_t* const ctile = sm.tile + 16 * kRow;
    if (bulk) {
        if (tid == 0) {
            ptx::mbar_init(&sm.bar, 1);
            ptx::mbar_init_fence();
        }
        __syncthreads();
        if (tid < kRows) {
            if (tid == 0) ptx::mbar_expect_tx(&sm.bar, 16 * nm * kYB + kCPlanes * kCRows * nm * kMcuC);
            if (tid < 16) {
                const uint32_t sy = min(my * 16 + tid, real_h - 1);
                ptx::bulk_g2s(sm.tile + tid * kRow, y + static_cast<size_t>(sy) * y_pitch + mcu0 * kYB, nm * kYB, &sm.bar);
            } else {
                const int k = (tid - 16) >> (kCRows == 8 ? 3 : 4), r = (tid - 16) & (kCRows - 1);
                const uint32_t sy = min(my * kCRows + r, ch - 1);
                ptx::bulk_g2s(ctile + (k * kCRows + r) * kCRow, (k ? v : u) + static_cast<size_t>(sy) * c_pitch + mcu0 * kMcuC, nm * kMcuC, &sm.bar);
            }
        }
    }
    if (p.prefetch_ahead && tid >= 32 && tid < 64) {
        StripImage a;
        // whole 16-byte units inside the rows only (the range must not pass the end of a row): real_w % 16 == 0 makes every
        // plane's strip end on its row's end
        // (one row per lane of the second warp, two for the 48 rows of I422 / I444)
        if (ahead_image<kMcus, kMixed, kFmt>(p, a) && a.real_w % 16 == 0) {
#pragma unroll
            for (int j = 0; j < (kRows + 31) / 32; ++j) {
                const int i = tid - 32 + 32 * j;
                if (i < kRows) {
                    const uint8_t* src = a.src.plane[i < 16 ? 0 : i < 16 + kCRows ? 1 : 2];
                    const uint32_t pitch = i < 16 ? a.src.pitch : a.src.pitch2;
                    if (((reinterpret_cast<uintptr_t>(src) | pitch) & 15) == 0) {
                        const uint32_t pnm = min(static_cast<uint32_t>(kMcus), a.mcu_w - a.mcu0);
                        const uint32_t sy = i < 16 ? min(a.my * 16 + i, a.real_h - 1)
                                                   : min(a.my * kCRows + ((i - 16) & (kCRows - 1)), (kCRows == 8 ? (a.real_h + 1) / 2 : a.real_h) - 1);
                        const uint32_t x0 = i < 16 ? a.mcu0 * kYB : a.mcu0 * kMcuC, n = (i < 16 ? pnm * kYB : pnm * kMcuC) & ~15u;
                        if (n) ptx::bulk_prefetch_l2(src + static_cast<size_t>(sy) * pitch + x0, n);
                    }
                }
            }
        }
    }
    if (bulk) {
        ptx::mbar_wait(&sm.bar, 0);
        return;
    }
    // one plane: `rows` rows of `chunks` 16-byte chunks from x0 on; es: bytes of one sample (NV12 / NV16 chroma: a U, V pair).  A
    // chunk that ends past `width` takes clamped byte loads.
    auto stage_plane = [&](const uint8_t* src, uint32_t pitch, bool aligned, uint32_t row0, uint32_t last_row, uint32_t width, uint32_t es,
                           uint32_t x0, int rows, int chunks, uint8_t* dst, int dst_row) {
        for (int i = tid; i < rows * chunks; i += kThreads) {
            const int r = i / chunks, m = i - r * chunks;
            const uint8_t* row = src + static_cast<size_t>(min(row0 + r, last_row)) * pitch;
            const uint32_t x = x0 + m * 16;
            uint4 q;
            if (aligned && x + 16 <= width) {
                q = __ldg(reinterpret_cast<const uint4*>(row + x));
            } else {                                                        // right edge replication
                uint32_t b[4];
#pragma unroll
                for (int j = 0; j < 4; ++j) {
                    uint32_t word = 0;
#pragma unroll
                    for (int t = 0; t < 4; ++t) {
                        const uint32_t xx = x + 4 * j + t;
                        uint32_t sx;
                        if constexpr (kPacked) {
                            // byte xx of the packed row: a Y sample of pixel 2g + k (group g = xx / 4) or the U / V of group g
                            constexpr uint32_t kYOff = kFmt == kPixelYUYV ? 0 : 1;
                            const uint32_t g = xx >> 2, pos = xx & 3;
                            if ((pos & 1) == kYOff) {
                                const uint32_t px = min(2 * g + (pos >> 1), real_w - 1);
                                sx = (px >> 1) * 4 + (px & 1) * 2 + kYOff;
                            } else {
                                sx = min(g, (real_w - 1) >> 1) * 4 + pos;
                            }
                        } else {
                            sx = xx < width ? xx : width - es + (xx & (es - 1));
                        }
                        word |= static_cast<uint32_t>(row[sx]) << (8 * t);
                    }
                    b[j] = word;
                }
                q = make_uint4(b[0], b[1], b[2], b[3]);
            }
            *reinterpret_cast<uint4*>(dst + r * dst_row + m * 16) = q;
        }
    };
    // (packed: a chunk lies inside the row when its 8 pixels are inside the image; for odd widths the last group's second Y is not)
    stage_plane(y, y_pitch, y_aligned, my * 16, real_h - 1, kPacked ? 2 * real_w : real_w, 1, mcu0 * kYB, 16, kPacked ? 2 * nm : nm, sm.tile, kRow);
    if constexpr (kCPlanes > 0) {
        const int cchunks = (nm * kMcuC + 15) / 16;                         // 8 bytes per MCU, odd nm: the last chunk's upper half is not read
        stage_plane(u, c_pitch, c_aligned, my * kCRows, ch - 1, cw_bytes, kSemi ? 2 : 1, mcu0 * kMcuC, kCRows, cchunks, ctile, kCRow);
        if constexpr (kCPlanes == 2)
            stage_plane(v, c_pitch, c_aligned, my * kCRows, ch - 1, cw_bytes, 1, mcu0 * kMcuC, kCRows, cchunks, ctile + kCRows * kCRow, kCRow);
    }
    __syncthreads();
}

// kAligned: real_w % 16 == 0 and 16-byte aligned base -> rows are staged with bulk copies; otherwise a clamped
// byte loader fills the tile (odd sizes; right-edge replication, src/Image.cpp:491-530)
// kMixed: images of individual sizes (p.geom): a 1-D grid over the strips of all images; a CTA finds its image by a search
// over the first-strip prefix.  Otherwise one size: grid (strips of a row, rows, frames).
// kFmt >= 0: pixels in that JPGENC_PIXEL_* format with a row pitch (stage_layout; grey and planar RGB: stage_planes; YUV:
// stage_yuv; kAligned is not used); -1: tight RGB
template <int kMcus, bool kAligned, bool kBulkOut, bool kMixed, int kFmt = -1>
// (shared memory and the thread index come from the kernel: there the compiler knows the alignment and, from the launch
// bounds, the range of threadIdx.x)
__device__ __forceinline__ void forward_body(const ForwardParams& p, ForwardSmem<kMcus>& sm, unsigned thread) {
    using Smem = ForwardSmem<kMcus>;
    constexpr int kThreads = kMcus * 4;
    const int tid = thread;
    constexpr bool kPlanar = kFmt == kPixelPlanar, kPlaneTile = kPlanar || kFmt == JPGENC_PIXEL_GRAY;   // stage_planes
    constexpr bool kYuv = is_yuv(kFmt), kNV12 = kFmt == kPixelNV12;                                // stage_yuv
    constexpr bool kYuv420 = kYuv && chroma_vsub(kFmt), kPacked = is_packed_yuv(kFmt);
    const StripImage s = strip_image<kMcus, kMixed, kFmt>(p, ThisCta{});
    const uint8_t* __restrict__ rgb = s.src.plane[0];
    const uint32_t my = s.my, mcu0 = s.mcu0, frame_block0 = s.block0, real_w = s.real_w, real_h = s.real_h, mcu_w = s.mcu_w;
    const int nm = min(kMcus, static_cast<int>(mcu_w - mcu0));

    // ---- stage the 16-row RGB strip ----
    if constexpr (kYuv) {
        stage_yuv<kMcus, kFmt, kMixed>(p, sm, tid, s, nm);
    } else if constexpr (kPlaneTile) {
        stage_planes<kMcus, kFmt, kMixed>(p, sm, tid, s, nm);
    } else if constexpr (kFmt >= 0) {
        stage_layout<kMcus, kFmt, kMixed>(p, sm, tid, s, nm);
    } else if constexpr (kAligned) {
        if (tid == 0) {
            ptx::mbar_init(&sm.bar, 1);
            ptx::mbar_init_fence();
        }
        __syncthreads();
        if (tid < 16) {
            // 16 lanes issue one row each (a single thread issuing all 16 serialises ~0.3 us of TMA issue latency)
            const uint32_t row_bytes = nm * 48;
            if (tid == 0) ptx::mbar_expect_tx(&sm.bar, 16 * row_bytes);
            const uint32_t sy = min(my * 16 + tid, real_h - 1);                // bottom edge replication
            ptx::bulk_g2s(sm.tile + tid * Smem::kPitch, rgb + (static_cast<size_t>(sy) * real_w + mcu0 * 16) * 3, row_bytes, &sm.bar);
        }
        if constexpr (kMixed) {
            // the flat strip order runs across the images: warp 1 finds the image of the strip `prefetch_ahead` CTAs later
            const uint32_t t = blockIdx.x + p.prefetch_ahead;
            if (p.prefetch_ahead && t < p.strips && tid >= 32 && tid < 64) {
                const FrameGeom& g = p.geom[geom_find_warp(p.geom, p.nframes, t, &FrameGeom::strip0)];
                const uint32_t per_row = (g.mcu_w + kMcus - 1) / kMcus, s = t - g.strip0, pby = s / per_row;
                const uint32_t pm0 = (s - pby * per_row) * kMcus, pnm = min(static_cast<uint32_t>(kMcus), g.mcu_w - pm0);
                const uint32_t sy = min(pby * 16 + (tid - 32), g.real_h - 1);
                if (tid < 48) ptx::bulk_prefetch_l2(g.rgb + (static_cast<size_t>(sy) * g.real_w + pm0 * 16) * 3, pnm * 48);
            }
        } else if (p.prefetch_ahead && tid >= 32 && tid < 48) {
            // the CTAs are dispatched in linear order (x, then y, then frame): by the time the CTA `prefetch_ahead`
            // positions later starts, its strip is in L2 and its bulk copies wait for L2 instead of DRAM
            const uint32_t per_frame = gridDim.x * gridDim.y;
            uint32_t lin = blockIdx.y * gridDim.x + blockIdx.x + p.prefetch_ahead, pz = blockIdx.z;
            while (lin >= per_frame && pz + 1 < gridDim.z) { lin -= per_frame; ++pz; }    // at most a few frames ahead
            const uint32_t pby = lin / gridDim.x, pbx = lin - pby * gridDim.x;
            if (pby < gridDim.y) {
                const uint8_t* __restrict__ prgb = p.frames ? p.frames[pz] : p.rgb;
                const uint32_t pm0 = pbx * kMcus, pnm = min(static_cast<uint32_t>(kMcus), p.mcu_w - pm0);
                const uint32_t sy = min((p.mcu_y0 + pby) * 16 + (tid - 32), p.real_h - 1);
                ptx::bulk_prefetch_l2(prgb + (static_cast<size_t>(sy) * p.real_w + pm0 * 16) * 3, pnm * 48);
            }
        }
        ptx::mbar_wait(&sm.bar, 0);
    } else {
        const int row_bytes = nm * 48;
        for (int idx = tid; idx < 16 * row_bytes; idx += kThreads) {
            const int r = idx / row_bytes, b = idx - r * row_bytes;
            const uint32_t sx = min(mcu0 * 16 + b / 3, real_w - 1);
            const uint32_t sy = min(my * 16 + r, real_h - 1);
            sm.tile[r * Smem::kPitch + b] = rgb[(static_cast<size_t>(sy) * real_w + sx) * 3 + (b % 3)];
        }
        __syncthreads();
    }

    // ---- luma thread: block (bx, by) of the strip's 2 x (2*kMcus) block grid ----
    const int bx = tid % (kMcus * 2), by = tid / (kMcus * 2);
    const bool active = (bx >> 1) < nm;
    f2 v[32];                                     // v[r*4+p] = samples (r, 2p) and (r, 2p+1)
    constexpr int kR = (kFmt == JPGENC_PIXEL_BGR || kFmt == JPGENC_PIXEL_BGRA) ? 2 : 0, kB = 2 - kR;   // tile bytes of R and B
    if constexpr (kYuv420) {
        if (active) {
            // The samples themselves, level-shifted: no colour conversion and no 2x2 means.  The chroma sample of an MCU position
            // is the stored one: the reference's S420_m averages four equal values there ((a + a) + (a + a), then / 4, gives
            // exactly a), see exact_sample.  Every value is an integer in [-128, 127], exact in FP32.  The chroma goes first,
            // before the luma block fills its registers.
            constexpr int kRow = kMcus * 16;
            const uint8_t* ctile = sm.tile + 16 * kRow;
#pragma unroll
            for (int rp = 0; rp < 4; ++rp) {          // chroma row by * 4 + rp, columns bx * 4 .. bx * 4 + 3 (this thread's 2x2 cells)
                const int cr = by * 4 + rp;
                f2 cb[2], crr[2];
                if constexpr (kNV12) {
                    const uint2 q = *reinterpret_cast<const uint2*>(ctile + cr * kRow + bx * 8);          // U V U V U V U V
                    const uint32_t w[2] = {q.x, q.y};
                    cb[0] = bytes_to_f2_centred(w, 0, 2); cb[1] = bytes_to_f2_centred(w, 4, 6);
                    crr[0] = bytes_to_f2_centred(w, 1, 3); crr[1] = bytes_to_f2_centred(w, 5, 7);
                } else {
                    constexpr int kCRow = kMcus * 8;
                    const uint32_t wu[1] = {*reinterpret_cast<const uint32_t*>(ctile + cr * kCRow + bx * 4)};
                    const uint32_t wv[1] = {*reinterpret_cast<const uint32_t*>(ctile + (8 + cr) * kCRow + bx * 4)};
                    cb[0] = bytes_to_f2_centred(wu, 0, 1); cb[1] = bytes_to_f2_centred(wu, 2, 3);
                    crr[0] = bytes_to_f2_centred(wv, 0, 1); crr[1] = bytes_to_f2_centred(wv, 2, 3);
                }
                *reinterpret_cast<float4*>(&sm.chroma[0][cr][bx * 4]) = make_float4(cb[0].x, cb[0].y, cb[1].x, cb[1].y);
                *reinterpret_cast<float4*>(&sm.chroma[1][cr][bx * 4]) = make_float4(crr[0].x, crr[0].y, crr[1].x, crr[1].y);
            }
#pragma unroll
            for (int r = 0; r < 8; ++r) {
                const uint2 q = *reinterpret_cast<const uint2*>(sm.tile + (by * 8 + r) * kRow + bx * 8);
                const uint32_t w[2] = {q.x, q.y};
#pragma unroll
                for (int pp = 0; pp < 4; ++pp) v[r * 4 + pp] = bytes_to_f2_centred(w, 2 * pp, 2 * pp + 1);
            }
        }
    } else if constexpr (kYuv) {
        if (active) {
            // 4:2:2 and 4:4:4: level-shifted samples, no colour conversion; the chroma of a 2x2 cell is the mean of its four samples
            // as S420_m takes it (see exact_sample).  4:2:2: the two pixels of a cell share a sample, so the mean is that of the
            // cell's two rows, (a + b) * 0.5; 4:4:4: 2x2 sums * 0.25.  Small integers and halves / quarters of them: exact in FP32.
            constexpr int kRow = kMcus * (kPacked ? 32 : 16);
            constexpr int kCRow = kMcus * (kFmt == kPixelI422 ? 8 : 16);
            const uint8_t* ctile = sm.tile + 16 * kRow;
#pragma unroll
            for (int rp = 0; rp < 4; ++rp) {          // chroma row by * 4 + rp = tile rows r0, r0 + 1; columns bx * 4 .. bx * 4 + 3
                const int r0 = by * 8 + rp * 2;
                f2 cb[2], crr[2];
                if constexpr (kPacked) {
                    // a row's 16 bytes: the thread's 8 pixels as 4 groups, Y0 U Y1 V (YUYV) or U Y0 V Y1 (UYVY)
                    constexpr int kY = kFmt == kPixelYUYV ? 0 : 1, kU = 1 - kY, kV = kU + 2;
                    const uint4 q0 = *reinterpret_cast<const uint4*>(sm.tile + r0 * kRow + bx * 16);
                    const uint4 q1 = *reinterpret_cast<const uint4*>(sm.tile + (r0 + 1) * kRow + bx * 16);
                    const uint32_t w0[4] = {q0.x, q0.y, q0.z, q0.w}, w1[4] = {q1.x, q1.y, q1.z, q1.w};
#pragma unroll
                    for (int pp = 0; pp < 4; ++pp) {
                        v[(rp * 2) * 4 + pp] = bytes_to_f2_centred(w0, 4 * pp + kY, 4 * pp + 2 + kY);
                        v[(rp * 2 + 1) * 4 + pp] = bytes_to_f2_centred(w1, 4 * pp + kY, 4 * pp + 2 + kY);
                    }
#pragma unroll
                    for (int j = 0; j < 2; ++j) {             // groups 2j, 2j + 1
                        cb[j] = __fmul2_rn(add2(bytes_to_f2_centred(w0, 8 * j + kU, 8 * j + 4 + kU), bytes_to_f2_centred(w1, 8 * j + kU, 8 * j + 4 + kU)),
                                           make_float2(0.5f, 0.5f));
                        crr[j] = __fmul2_rn(add2(bytes_to_f2_centred(w0, 8 * j + kV, 8 * j + 4 + kV), bytes_to_f2_centred(w1, 8 * j + kV, 8 * j + 4 + kV)),
                                            make_float2(0.5f, 0.5f));
                    }
                } else if constexpr (kFmt == kPixelI422) {
                    const uint32_t u0[1] = {*reinterpret_cast<const uint32_t*>(ctile + r0 * kCRow + bx * 4)};
                    const uint32_t u1[1] = {*reinterpret_cast<const uint32_t*>(ctile + (r0 + 1) * kCRow + bx * 4)};
                    const uint32_t v0[1] = {*reinterpret_cast<const uint32_t*>(ctile + (16 + r0) * kCRow + bx * 4)};
                    const uint32_t v1[1] = {*reinterpret_cast<const uint32_t*>(ctile + (17 + r0) * kCRow + bx * 4)};
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
                        cb[j] = __fmul2_rn(add2(bytes_to_f2_centred(u0, 2 * j, 2 * j + 1), bytes_to_f2_centred(u1, 2 * j, 2 * j + 1)), make_float2(0.5f, 0.5f));
                        crr[j] = __fmul2_rn(add2(bytes_to_f2_centred(v0, 2 * j, 2 * j + 1), bytes_to_f2_centred(v1, 2 * j, 2 * j + 1)), make_float2(0.5f, 0.5f));
                    }
                } else if constexpr (kFmt == kPixelNV16) {
                    const uint2 q0 = *reinterpret_cast<const uint2*>(ctile + r0 * kCRow + bx * 8);          // U V U V U V U V
                    const uint2 q1 = *reinterpret_cast<const uint2*>(ctile + (r0 + 1) * kCRow + bx * 8);
                    const uint32_t w0[2] = {q0.x, q0.y}, w1[2] = {q1.x, q1.y};
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
                        cb[j] = __fmul2_rn(add2(bytes_to_f2_centred(w0, 4 * j, 4 * j + 2), bytes_to_f2_centred(w1, 4 * j, 4 * j + 2)), make_float2(0.5f, 0.5f));
                        crr[j] = __fmul2_rn(add2(bytes_to_f2_centred(w0, 4 * j + 1, 4 * j + 3), bytes_to_f2_centred(w1, 4 * j + 1, 4 * j + 3)),
                                            make_float2(0.5f, 0.5f));
                    }
                } else {                                      // I444: 8 bytes per row and plane, 2x2 sums
                    static_assert(kFmt == kPixelI444, "a YUV 4:2:2 / 4:4:4 layout");
                    f2 c4[2][2];                              // [plane][j]: the sums of cells 2j, 2j + 1
#pragma unroll
                    for (int k = 0; k < 2; ++k) {
                        const uint2 q0 = *reinterpret_cast<const uint2*>(ctile + (16 * k + r0) * kCRow + bx * 8);
                        const uint2 q1 = *reinterpret_cast<const uint2*>(ctile + (16 * k + r0 + 1) * kCRow + bx * 8);
                        const uint32_t w0[2] = {q0.x, q0.y}, w1[2] = {q1.x, q1.y};
                        float s4[4];
#pragma unroll
                        for (int pp = 0; pp < 4; ++pp) {
                            const f2 sc = add2(bytes_to_f2_centred(w0, 2 * pp, 2 * pp + 1), bytes_to_f2_centred(w1, 2 * pp, 2 * pp + 1));
                            s4[pp] = sc.x + sc.y;
                        }
                        c4[k][0] = make_float2(s4[0], s4[1]);
                        c4[k][1] = make_float2(s4[2], s4[3]);
                    }
#pragma unroll
                    for (int j = 0; j < 2; ++j) {
                        cb[j] = __fmul2_rn(c4[0][j], make_float2(0.25f, 0.25f));
                        crr[j] = __fmul2_rn(c4[1][j], make_float2(0.25f, 0.25f));
                    }
                }
                *reinterpret_cast<float4*>(&sm.chroma[0][by * 4 + rp][bx * 4]) = make_float4(cb[0].x, cb[0].y, cb[1].x, cb[1].y);
                *reinterpret_cast<float4*>(&sm.chroma[1][by * 4 + rp][bx * 4]) = make_float4(crr[0].x, crr[0].y, crr[1].x, crr[1].y);
            }
            if constexpr (!kPacked) {
#pragma unroll
                for (int r = 0; r < 8; ++r) {
                    const uint2 q = *reinterpret_cast<const uint2*>(sm.tile + (by * 8 + r) * kRow + bx * 8);
                    const uint32_t w[2] = {q.x, q.y};
#pragma unroll
                    for (int pp = 0; pp < 4; ++pp) v[r * 4 + pp] = bytes_to_f2_centred(w, 2 * pp, 2 * pp + 1);
                }
            }
        }
    } else if (active) {
        const ColorConsts& cc = p.color;
#pragma unroll
        for (int rp = 0; rp < 4; ++rp) {
            f2 rr[2][4], gg[2][4], bb[2][4];
#pragma unroll
            for (int h = 0; h < 2; ++h) {
                const int r = rp * 2 + h;
                if constexpr (kPlaneTile) {                       // one 8-byte word per plane holds the thread's 8 pixels
                    constexpr int kRow = kMcus * 16, kPlaneBytes = 16 * kRow;
                    const uint8_t* src = sm.tile + (by * 8 + r) * kRow + bx * 8;
                    const uint2 qr = *reinterpret_cast<const uint2*>(src);
                    const uint32_t wr[2] = {qr.x, qr.y};
                    uint32_t wg[2] = {qr.x, qr.y}, wb[2] = {qr.x, qr.y};
                    if constexpr (kPlanar) {
                        const uint2 qg = *reinterpret_cast<const uint2*>(src + kPlaneBytes), qb = *reinterpret_cast<const uint2*>(src + 2 * kPlaneBytes);
                        wg[0] = qg.x; wg[1] = qg.y; wb[0] = qb.x; wb[1] = qb.y;
                    }
#pragma unroll
                    for (int pp = 0; pp < 4; ++pp) {              // pixels 2pp, 2pp+1
                        rr[h][pp] = bytes_to_f2(wr, 2 * pp, 2 * pp + 1);
                        gg[h][pp] = kPlanar ? bytes_to_f2(wg, 2 * pp, 2 * pp + 1) : rr[h][pp];
                        bb[h][pp] = kPlanar ? bytes_to_f2(wb, 2 * pp, 2 * pp + 1) : rr[h][pp];
                        v[r * 4 + pp] = fma2s(rr[h][pp], cc.y[0], fma2s(gg[h][pp], cc.y[1], fma2s(bb[h][pp], cc.y[2], make_float2(-128.f, -128.f))));
                    }
                    continue;
                }
                const uint2* src = reinterpret_cast<const uint2*>(sm.tile + (by * 8 + r) * Smem::kPitch + bx * 24);
                const uint2 q0 = src[0], q1 = src[1], q2 = src[2];
                const uint32_t w[6] = {q0.x, q0.y, q1.x, q1.y, q2.x, q2.y};
#pragma unroll
                for (int pp = 0; pp < 4; ++pp) {                  // pixels 2pp, 2pp+1 = bytes 6pp .. 6pp+5
                    rr[h][pp] = bytes_to_f2(w, 6 * pp + kR, 6 * pp + 3 + kR);
                    gg[h][pp] = bytes_to_f2(w, 6 * pp + 1, 6 * pp + 4);
                    bb[h][pp] = bytes_to_f2(w, 6 * pp + kB, 6 * pp + 3 + kB);
                    v[r * 4 + pp] = fma2s(rr[h][pp], cc.y[0], fma2s(gg[h][pp], cc.y[1], fma2s(bb[h][pp], cc.y[2], make_float2(-128.f, -128.f))));
                }
            }
            // 2x2 sums are sums of small integers: exact in any order (reference order: (a+b)+(c+d), src/Image.cpp:209-224)
            float r4[4], g4[4], b4[4];
#pragma unroll
            for (int pp = 0; pp < 4; ++pp) {
                const f2 sr = add2(rr[0][pp], rr[1][pp]), sg = add2(gg[0][pp], gg[1][pp]), sb = add2(bb[0][pp], bb[1][pp]);
                r4[pp] = sr.x + sr.y;
                g4[pp] = sg.x + sg.y;
                b4[pp] = sb.x + sb.y;
            }
            f2 cb[2], cr[2];
#pragma unroll
            for (int j = 0; j < 2; ++j) {
                const f2 r2 = make_float2(r4[2 * j], r4[2 * j + 1]), g2 = make_float2(g4[2 * j], g4[2 * j + 1]),
                         b2 = make_float2(b4[2 * j], b4[2 * j + 1]);
                cb[j] = fma2s(r2, cc.cb[0], fma2s(g2, cc.cb[1], __fmul2_rn(b2, make_float2(cc.cb[2], cc.cb[2]))));
                cr[j] = fma2s(r2, cc.cr[0], fma2s(g2, cc.cr[1], __fmul2_rn(b2, make_float2(cc.cr[2], cc.cr[2]))));
            }
            *reinterpret_cast<float4*>(&sm.chroma[0][by * 4 + rp][bx * 4]) = make_float4(cb[0].x, cb[0].y, cb[1].x, cb[1].y);
            *reinterpret_cast<float4*>(&sm.chroma[1][by * 4 + rp][bx * 4]) = make_float4(cr[0].x, cr[0].y, cr[1].x, cr[1].y);
        }
    }
    __syncthreads();   // every RGB byte has been consumed (tile may now be reused as staging); chroma planes complete

    const uint32_t mcu_base = my * mcu_w + mcu0;
    const uint32_t block_base = frame_block0 + mcu_base * kBlocksPerMcu;     // first coefficient block of this strip
    uint32_t packed[32];
    if (active) {
        dct8x8_packed<true>(v);
        const bool boundary = quantize_pack_packed(v, p.luma, packed);
        const int m = bx >> 1, k = by * 2 + (bx & 1);
        stage_block(sm.tile, m * kBlocksPerMcu + k, packed);
        if (boundary) push_refine(p, block_base + m * kBlocksPerMcu + k);
    }
    // ---- chroma threads: 2*kMcus blocks (Cb of every MCU, then Cr) ----
    if (tid < 2 * kMcus) {
        const int comp = tid / kMcus, m = tid % kMcus;
        if (m < nm) {
#pragma unroll
            for (int r = 0; r < 8; ++r) {
                const float4 lo = *reinterpret_cast<const float4*>(&sm.chroma[comp][r][m * 8]);
                const float4 hi = *reinterpret_cast<const float4*>(&sm.chroma[comp][r][m * 8 + 4]);
                v[r * 4 + 0] = make_float2(lo.x, lo.y); v[r * 4 + 1] = make_float2(lo.z, lo.w);
                v[r * 4 + 2] = make_float2(hi.x, hi.y); v[r * 4 + 3] = make_float2(hi.z, hi.w);
            }
            dct8x8_packed<true>(v);
            const bool boundary = quantize_pack_packed(v, p.chroma, packed);
            stage_block(sm.tile, m * kBlocksPerMcu + 4 + comp, packed);
            if (boundary) push_refine(p, block_base + m * kBlocksPerMcu + 4 + comp);
        }
    }
    if constexpr (kBulkOut) {
        // full strips leave as ONE tensor store: the staging layout (16-byte chunk c of row s at c ^ (s & 7)) is exactly
        // the 128-byte swizzle of a tensor map whose rows are the 128-byte coefficient blocks
        if (nm == kMcus) {
            ptx::fence_async_smem();              // this thread's staging writes become visible to the copy engine
            __syncthreads();
            if (tid == 0) {
                ptx::tensor_store_2d(&p.coef_map, sm.tile, 0, static_cast<int>(block_base));
                ptx::bulk_commit();
                ptx::bulk_wait_all_read();        // shared memory must stay allocated until the engine has read it
            }
            return;
        }
    }
    __syncthreads();
    copy_out(sm.tile, p.coef + static_cast<size_t>(block_base) * kCoefPerBlock, nm * kBlocksPerMcu, tid, kThreads);
}

template <int kMcus, bool kAligned, bool kBulkOut = false>
__global__ void __launch_bounds__(kMcus * 4, 640 / (kMcus * 4)) forward_kernel(const __grid_constant__ ForwardParams p) {
    __shared__ ForwardSmem<kMcus> sm;
    forward_body<kMcus, kAligned, kBulkOut, false>(p, sm, threadIdx.x);
}

template <int kMcus, bool kAligned, bool kBulkOut>
__global__ void __launch_bounds__(kMcus * 4, 640 / (kMcus * 4)) forward_mixed_kernel(const __grid_constant__ ForwardParams p) {
    __shared__ ForwardSmem<kMcus> sm;
    forward_body<kMcus, kAligned, kBulkOut, true>(p, sm, threadIdx.x);
}

// pixels in another layout (kFmt): one image (p.rgb, p.src) / images of individual sizes
template <int kMcus, int kFmt, bool kBulkOut>
__global__ void __launch_bounds__(kMcus * 4, 640 / (kMcus * 4)) forward_layout_kernel(const __grid_constant__ ForwardParams p) {
    __shared__ ForwardSmem<kMcus> sm;
    forward_body<kMcus, false, kBulkOut, false, kFmt>(p, sm, threadIdx.x);
}

template <int kMcus, int kFmt, bool kBulkOut>
__global__ void __launch_bounds__(kMcus * 4, 640 / (kMcus * 4)) forward_mixed_layout_kernel(const __grid_constant__ ForwardParams p) {
    __shared__ ForwardSmem<kMcus> sm;
    forward_body<kMcus, false, kBulkOut, true, kFmt>(p, sm, threadIdx.x);
}

// ---------------------------------------------------------------------------------------------------
// exact FP64 path (the reference's arithmetic, operation for operation, no contraction)
// ---------------------------------------------------------------------------------------------------
// quantise one coefficient exactly as Coding.hpp:92-94 does: int(std::round(x / q)), division in double
__device__ __forceinline__ int16_t quantize_exact(double x, uint8_t q) {
    return static_cast<int16_t>(static_cast<int>(round(__ddiv_rn(x, static_cast<double>(q)))));
}

// colour conversion of one pixel, src/Image.cpp:131-143: float constants widened to double, double arithmetic
__device__ __forceinline__ double exact_channel(int comp, double r, double g, double b) {
    if (comp == 0) return dsub(dadd(0.0, dadd(dadd(dmul((double).299f, r), dmul((double).587f, g)), dmul((double).114f, b))), 128.0);
    if (comp == 1) return dsub(dadd(128.0, dadd(dadd(dmul((double)-.1687f, r), dmul((double)-.3312f, g)), dmul((double).5f, b))), 128.0);
    return dsub(dadd(128.0, dadd(dadd(dmul((double).5f, r), dmul((double)-.4186f, g)), dmul((double)-.0813f, b))), 128.0);
}

// kFmt: -1 tight RGB, otherwise the JPGENC_PIXEL_* format (or kPixelPlanar) of pixels whose rows are s.pitch bytes apart; `rgb` is
// the first plane, s.plane[1] and s.plane[2] are the G and B planes of planar RGB.  A grey pixel v is the pixel (v, v, v).
template <int kFmt>
__device__ __forceinline__ double exact_pixel(const uint8_t* rgb, const PixelSource& s, uint32_t real_w, uint32_t real_h, uint32_t x, uint32_t y,
                                              int comp, double scale) {
    const uint32_t sx = min(x, real_w - 1), sy = min(y, real_h - 1);            // src/Image.cpp:491-530
    if constexpr (kFmt == JPGENC_PIXEL_GRAY || kFmt == kPixelPlanar) {
        const size_t at = static_cast<size_t>(sy) * s.pitch + sx;
        const double r = dmul(static_cast<double>(rgb[at]), scale);
        if constexpr (kFmt == JPGENC_PIXEL_GRAY) return exact_channel(comp, r, r, r);
        else return exact_channel(comp, r, dmul(static_cast<double>(s.plane[1][at]), scale), dmul(static_cast<double>(s.plane[2][at]), scale));
    }
    const uint8_t* px;
    if constexpr (kFmt < 0) px = rgb + (static_cast<size_t>(sy) * real_w + sx) * 3;
    else px = rgb + static_cast<size_t>(sy) * s.pitch + sx * pixel_bytes(kFmt);
    constexpr int kR = (kFmt == JPGENC_PIXEL_BGR || kFmt == JPGENC_PIXEL_BGRA) ? 2 : 0, kB = 2 - kR;
    return exact_channel(comp, dmul(static_cast<double>(px[kR]), scale), dmul(static_cast<double>(px[1]), scale),
                         dmul(static_cast<double>(px[kB]), scale));
}

// Column c of block `id` (mcu*6+k) of an image: located once per thread (the divisions), then sampled row by row
struct ExactColumn {
    const uint8_t* rgb;
    uint32_t x, y;          // top pixel of the column (luma) / of the column's 2x2 cells (chroma)
    int comp;               // 0 = Y, 1 = Cb, 2 = Cr
};
__device__ __forceinline__ ExactColumn exact_locate(const uint8_t* rgb, uint32_t mcu_w, uint32_t id, int c) {
    const uint32_t mcu = id / kBlocksPerMcu, k = id % kBlocksPerMcu;
    const uint32_t my = mcu / mcu_w, mx = mcu - my * mcu_w;
    if (k < 4) return ExactColumn{rgb, mx * 16 + (k & 1) * 8 + c, my * 16 + (k >> 1) * 8, 0};
    return ExactColumn{rgb, mx * 16 + 2 * c, my * 16, static_cast<int>(k) - 3};
}
// Spatial sample of row r in the reference's arithmetic, of the image whose first plane is b.rgb and whose other planes and
// pitches are those of `s`.
// YUV 4:2:0: what Image::writeJPEG computes for the image whose level-shifted Y, Cb, Cr planes are the clamped bytes minus 128
// (the frame padded to whole MCUs by edge replication, every chroma sample repeated over its 2x2 pixels; jpgenc_encode_planes(...,
// ycbcr = 1)), bit for bit: such an image skips the colour conversion (src/Image.cpp:112-115); a luma sample is (double)byte -
// 128, exact; S420_m (src/Image.cpp:207-226) sums the four pixels of a cell as (0 + a + a) + (0 + a + a) -- a cell's four
// clamped pixels map to one chroma sample a (x, x + 1 with x even, or both clamped to the last column; the same for rows) -- and
// quarters the sum: every step is exact on these small integers and gives a again.  So the chroma sample of cell (x / 2, y / 2)
// is U[min(y / 2, ch - 1)][min(x / 2, cw - 1)] - 128 (V for Cr; NV12: the pair's first / second byte).
// YUV 4:2:2 and 4:4:4: the image whose level-shifted planes are the clamped bytes minus 128 at full resolution (a 4:2:2 chroma
// sample at both pixels of its group); luma as above, chroma by S420_m over the four clamped pixels of the cell in the reference's
// order, ((0 + p00) + p01) + ((0 + p10) + p11), times 0.25.
template <int kFmt>
__device__ __forceinline__ double exact_yuv_byte(const uint8_t* y, const PixelSource& s, uint32_t sx, uint32_t sy, int comp) {
    if constexpr (is_packed_yuv(kFmt)) {                                   // group sx / 2: Y0 U Y1 V (YUYV) or U Y0 V Y1 (UYVY)
        constexpr uint32_t kY = kFmt == kPixelYUYV ? 0 : 1;
        const uint32_t at = (sx >> 1) * 4 + (comp == 0 ? kY + (sx & 1) * 2 : (1 - kY) + (comp - 1) * 2);
        return dsub(static_cast<double>(y[static_cast<size_t>(sy) * s.pitch + at]), 128.0);
    } else {
        if (comp == 0) return dsub(static_cast<double>(y[static_cast<size_t>(sy) * s.pitch + sx]), 128.0);
        const uint32_t cx = sx >> chroma_hsub(kFmt);
        const size_t row = static_cast<size_t>(sy) * s.pitch2;
        const uint8_t v = kFmt == kPixelNV16 ? s.plane[1][row + 2 * cx + (comp - 1)] : (comp == 1 ? s.plane[1] : s.plane[2])[row + cx];
        return dsub(static_cast<double>(v), 128.0);
    }
}

template <int kFmt>
__device__ __forceinline__ double exact_sample(const ExactColumn& b, const PixelSource& s, uint32_t real_w, uint32_t real_h, int r, double scale) {
    if constexpr (is_yuv(kFmt) && !chroma_vsub(kFmt)) {
        if (b.comp == 0) return exact_yuv_byte<kFmt>(b.rgb, s, min(b.x, real_w - 1), min(b.y + r, real_h - 1), 0);
        const uint32_t x0 = min(b.x, real_w - 1), x1 = min(b.x + 1, real_w - 1);
        const uint32_t y = b.y + 2 * r, y0 = min(y, real_h - 1), y1 = min(y + 1, real_h - 1);
        const double top = dadd(dadd(0.0, exact_yuv_byte<kFmt>(b.rgb, s, x0, y0, b.comp)), exact_yuv_byte<kFmt>(b.rgb, s, x1, y0, b.comp));
        const double bot = dadd(dadd(0.0, exact_yuv_byte<kFmt>(b.rgb, s, x0, y1, b.comp)), exact_yuv_byte<kFmt>(b.rgb, s, x1, y1, b.comp));
        return dmul(dadd(top, bot), 0.25);
    } else if constexpr (is_yuv(kFmt)) {
        if (b.comp == 0) {
            const uint32_t sx = min(b.x, real_w - 1), sy = min(b.y + r, real_h - 1);
            return dsub(static_cast<double>(b.rgb[static_cast<size_t>(sy) * s.pitch + sx]), 128.0);
        }
        const uint32_t cx = min(b.x / 2, (real_w + 1) / 2 - 1), cy = min(b.y / 2 + r, (real_h + 1) / 2 - 1);
        const size_t row = static_cast<size_t>(cy) * s.pitch2;
        const uint8_t v = kFmt == kPixelNV12 ? s.plane[1][row + 2 * cx + (b.comp - 1)] : (b.comp == 1 ? s.plane[1] : s.plane[2])[row + cx];
        return dsub(static_cast<double>(v), 128.0);
    } else {
        if (b.comp == 0) return exact_pixel<kFmt>(b.rgb, s, real_w, real_h, b.x, b.y + r, 0, scale);
        const uint32_t x = b.x, y = b.y + 2 * r;                                // S420_m, src/Image.cpp:207-226
        const double top = dadd(dadd(0.0, exact_pixel<kFmt>(b.rgb, s, real_w, real_h, x, y, b.comp, scale)),
                                exact_pixel<kFmt>(b.rgb, s, real_w, real_h, x + 1, y, b.comp, scale));
        const double bot = dadd(dadd(0.0, exact_pixel<kFmt>(b.rgb, s, real_w, real_h, x, y + 1, b.comp, scale)),
                                exact_pixel<kFmt>(b.rgb, s, real_w, real_h, x + 1, y + 1, b.comp, scale));
        return dmul(dadd(top, bot), 0.25);      // the reference divides by 4: the same double, bit for bit, without a division
    }
}

// Exact 8x8 transform, 8 threads per block (4 blocks per warp), everything in registers: thread c fetches column c
// of the block and runs the vertical pass on it (the reference's pass 1 turns column j into row j of its temporary,
// Dct.hpp:52-132), an 8x8 register transpose over the 8 lanes (three butterfly exchanges) hands every thread one column
// of the temporary, the second pass turns that into row j of the result (Dct.hpp:134-214), and the thread quantises
// and stores its 8 coefficients.  No shared memory, no barriers.
constexpr int kRefineThreads = 256;

// x[i] <-> partner's x[i ^ m] for the lanes whose bit `m` differs: one butterfly stage of the 8x8 transpose
template <int kM>
__device__ __forceinline__ void transpose_stage(double (&x)[8], int lane8) {
    const bool upper = (lane8 & kM) != 0;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
        if (i & kM) continue;
        // lower lanes send x[i | kM] and receive into it; upper lanes send x[i] and receive into it
        const double send = upper ? x[i] : x[i | kM];
        const double got = __shfl_xor_sync(0xffffffffu, send, kM);
        if (upper) x[i] = got; else x[i | kM] = got;
    }
}

__constant__ uint8_t c_inv_zigzag[64] = {0,  1,  5,  6,  14, 15, 27, 28, 2,  4,  7,  13, 16, 26, 29, 42, 3,  8,  12, 17, 25, 30,
                                         41, 43, 9,  11, 18, 24, 31, 40, 44, 53, 10, 19, 23, 32, 39, 45, 52, 54, 20, 22, 33, 38,
                                         46, 51, 55, 60, 21, 34, 37, 47, 50, 56, 59, 61, 35, 36, 48, 49, 57, 58, 62, 63};

// processes list entries (or, with `all`, block ids) [n0, n)
// locate(id, column) finds the thread's column once; sample(column, r) returns its row r
template <class Locate, class Sample>
__device__ __forceinline__ void refine_loop(uint32_t n0, uint32_t n, const uint32_t* __restrict__ list, bool all, int16_t* __restrict__ out,
                                            uint32_t blocks_per_frame, const uint8_t* qtab_y, const uint8_t* qtab_c, const ExactConsts& e,
                                            Locate&& locate, Sample&& sample) {
    const int lane8 = threadIdx.x & 7;
    const uint32_t group = (blockIdx.x * kRefineThreads + threadIdx.x) >> 3, ngroups = (gridDim.x * kRefineThreads) >> 3;
    const uint32_t rounds = (n - min(n0, n) + ngroups - 1) / ngroups;   // same trip count for every lane of a warp (shuffles inside)
    for (uint32_t it = 0; it < rounds; ++it) {
        const uint32_t i = n0 + it * ngroups + group;
        const bool valid = i < n;
        const uint32_t id = valid ? (all ? i : list[i]) : 0;
        double x[8], t[8];
        const auto col = locate(id, lane8);
#pragma unroll
        for (int r = 0; r < 8; ++r) x[r] = valid ? sample(col, r) : 0.0;
        aan8_exact_regs(x, t, e);                                     // t[k] = temporary(row lane8, column k)
        transpose_stage<1>(t, lane8);
        transpose_stage<2>(t, lane8);
        transpose_stage<4>(t, lane8);                                 // t[k] = temporary(row k, column lane8)
        aan8_exact_regs(t, x, e);                                     // x[k] = result(row lane8, column k)
        if (valid) {
            const uint8_t* q = ((id % blocks_per_frame) % kBlocksPerMcu) < 4 ? qtab_y : qtab_c;
            int16_t* dst = out + static_cast<size_t>(id) * kCoefPerBlock;
#pragma unroll
            for (int k = 0; k < 8; ++k) {
                const int nat = lane8 * 8 + k;
                dst[c_inv_zigzag[nat]] = quantize_exact(x[k], q[nat]);
            }
        }
    }
}

// The same with 64 threads per block (two blocks per warp).  The 8-thread form is a chain of ~800 dependent FP64
// instructions per thread (8 samples of up to 4 pixel conversions each, two passes, 8 divisions): a small image has too few
// flagged blocks to hide it (3840x2160: ~800 blocks, 15 us = a tenth of the encode).  Here thread (r, c) converts ONE sample and
// quantises ONE coefficient, the two 1-D passes run on 8 of the 64 threads out of shared memory: ~180 dependent instructions,
// and fewer warp instructions in total (the samples and divisions fill all lanes).
template <class Locate, class Sample>
__device__ __forceinline__ void refine_loop64(uint32_t n0, uint32_t n, const uint32_t* __restrict__ list, bool all, int16_t* __restrict__ out,
                                              uint32_t blocks_per_frame, const uint8_t* qtab_y, const uint8_t* qtab_c, const ExactConsts& e,
                                              Locate&& locate, Sample&& sample) {
    __shared__ double s_x[kRefineThreads / 64][64], s_t[kRefineThreads / 64][64];
    const int sub = threadIdx.x >> 6, t64 = threadIdx.x & 63, r = t64 >> 3, c = t64 & 7;
    double* X = s_x[sub];
    double* T = s_t[sub];
    const uint32_t group = blockIdx.x * (kRefineThreads / 64) + sub, ngroups = gridDim.x * (kRefineThreads / 64);
    const uint32_t rounds = (n - min(n0, n) + ngroups - 1) / ngroups;   // same trip count for every thread of the grid (barriers inside)
    for (uint32_t it = 0; it < rounds; ++it) {
        const uint32_t i = n0 + it * ngroups + group;
        const bool valid = i < n;
        const uint32_t id = valid ? (all ? i : list[i]) : 0;
        const auto col = locate(id, c);
        X[r * 8 + c] = valid ? sample(col, r) : 0.0;
        __syncthreads();
        if (t64 < 8) aan8_exact(X + t64, 8, T + t64 * 8, 1, e);          // column t64 of the block -> row t64 of the temporary
        __syncthreads();
        if (t64 < 8) aan8_exact(T + t64, 8, X + t64 * 8, 1, e);          // column t64 of the temporary -> row t64 of the result
        __syncthreads();
        if (valid) {
            const uint8_t* q = ((id % blocks_per_frame) % kBlocksPerMcu) < 4 ? qtab_y : qtab_c;
            out[static_cast<size_t>(id) * kCoefPerBlock + c_inv_zigzag[t64]] = quantize_exact(X[t64], q[t64]);
        }
        __syncthreads();                                                // X is overwritten by the next round's samples
    }
}

// ids are global block indices; with `frames` (a batch) block id belongs to frame id / blocks_per_frame, whose first plane is
// frames[id / blocks_per_frame]; otherwise the image is `src`, whose first plane `rgb` also is (a parameter of its own: as a
// restricted pointer its bytes take the read-only load path).  kFmt: -1 tight RGB, otherwise src.format.
template <bool k64, int kFmt>
__global__ void __launch_bounds__(kRefineThreads) refine_kernel(const uint8_t* __restrict__ rgb, const uint8_t* const* __restrict__ frames,
                                                                    uint32_t blocks_per_frame, int16_t* __restrict__ coef,
                                                                    const uint32_t* __restrict__ list,
                                                                    const uint32_t* __restrict__ count, uint32_t cap, int all,
                                                                    uint32_t nblocks, uint32_t real_w, uint32_t real_h,
                                                                    uint32_t mcu_w, const __grid_constant__ ExactConsts e,
                                                                    const __grid_constant__ PixelSource src) {
    // count[0] = entries in the list, count[3] = entries already refined (band-wise encodes refine after every band)
    const uint32_t n = all ? nblocks : min(count[0], cap), n0 = all ? 0u : count[3];
    auto locate = [&](uint32_t id, int c) {
        const uint32_t f = frames ? id / blocks_per_frame : 0u;
        return exact_locate(frames ? frames[f] : rgb, mcu_w, id - f * blocks_per_frame, c);
    };
    auto sample = [&](const ExactColumn& col, int r) { return exact_sample<kFmt>(col, src, real_w, real_h, r, e.scale); };
    if constexpr (k64) refine_loop64(n0, n, list, all != 0, coef, blocks_per_frame, e.qy, e.qc, e, locate, sample);
    else refine_loop(n0, n, list, all != 0, coef, blocks_per_frame, e.qy, e.qc, e, locate, sample);
}

// images of individual sizes: block id -> image by a search over the first-block prefix (every image starts on an MCU, so
// id % 6 still tells luma from chroma: blocks_per_frame = 2^32 - 1 leaves ids < 2^31 as they are).  Formats of several planes:
// image f's other planes at extra[f].
template <bool k64, int kFmt>
__global__ void __launch_bounds__(kRefineThreads) refine_mixed_kernel(const FrameGeom* __restrict__ geom, uint32_t nframes,
                                                                          int16_t* __restrict__ coef, const uint32_t* __restrict__ list,
                                                                          const uint32_t* __restrict__ count, uint32_t cap,
                                                                          const __grid_constant__ ExactConsts e, const ExtraPlanes* __restrict__ extra) {
    const uint32_t n = min(count[0], cap), n0 = count[3];
    struct Column { ExactColumn col; uint32_t real_w, real_h; PixelSource src; };
    auto locate = [&](uint32_t id, int c) {
        uint32_t lo = 0, hi = nframes;
        while (hi - lo > 1) {
            const uint32_t mid = (lo + hi) >> 1;
            if (geom[mid].block0 <= id) lo = mid; else hi = mid;
        }
        const FrameGeom& g = geom[lo];
        Column col{exact_locate(g.rgb, g.mcu_w, id - g.block0, c), g.real_w, g.real_h, {}};
        if constexpr (kFmt >= 0) col.src.pitch = g.pitch;
        if constexpr (source_planes(kFmt) == 3) {
            col.src.plane[1] = extra[lo].plane[0];
            col.src.plane[2] = extra[lo].plane[1];
            col.src.pitch2 = static_cast<uint32_t>(extra[lo].pitch2);
        }
        return col;
    };
    auto sample = [&](const Column& col, int r) { return exact_sample<kFmt>(col.col, col.src, col.real_w, col.real_h, r, e.scale); };
    if constexpr (k64) refine_loop64(n0, n, list, false, coef, 0xFFFFFFFFu, e.qy, e.qc, e, locate, sample);
    else refine_loop(n0, n, list, false, coef, 0xFFFFFFFFu, e.qy, e.qc, e, locate, sample);
}

// Images that are not 8-bit samples: three planes of doubles as the reference holds them (Image::R/G/B after loadPPM, or
// planes a caller computed; already YCbCr when `ycbcr`: Image::writeJPEG converts only an RGB image, src/Image.cpp:112-115,
// 839).  Every block takes the exact path; width x height are the padded plane dimensions (multiples of 16).
struct PlaneColumn { uint32_t x, y; int comp; };
__global__ void __launch_bounds__(kRefineThreads) planes_exact_kernel(const double* __restrict__ p0, const double* __restrict__ p1,
                                                                          const double* __restrict__ p2, uint32_t width, uint32_t mcu_w,
                                                                          uint32_t nblocks, int16_t* __restrict__ coef, int ycbcr,
                                                                          const __grid_constant__ ExactConsts e) {
    auto pixel = [&](uint32_t x, uint32_t y, int comp) {
        const size_t i = static_cast<size_t>(y) * width + x;
        if (ycbcr) return (comp == 0 ? p0 : comp == 1 ? p1 : p2)[i];
        return exact_channel(comp, p0[i], p1[i], p2[i]);
    };
    refine_loop(0u, nblocks, nullptr, true, coef, nblocks, e.qy, e.qc, e,
                [&](uint32_t id, int c) {
                    const uint32_t mcu = id / kBlocksPerMcu, k = id % kBlocksPerMcu, my = mcu / mcu_w, mx = mcu - my * mcu_w;
                    if (k < 4) return PlaneColumn{mx * 16 + (k & 1) * 8 + c, my * 16 + (k >> 1) * 8, 0};
                    return PlaneColumn{mx * 16 + 2 * c, my * 16, static_cast<int>(k) - 3};
                },
                [&](const PlaneColumn& col, int r) {
                    if (col.comp == 0) return pixel(col.x, col.y + r, 0);
                    const uint32_t x = col.x, y = col.y + 2 * r;                                // S420_m, src/Image.cpp:207-226
                    const double top = dadd(dadd(0.0, pixel(x, y, col.comp)), pixel(x + 1, y, col.comp));
                    const double bot = dadd(dadd(0.0, pixel(x, y + 1, col.comp)), pixel(x + 1, y + 1, col.comp));
                    return dmul(dadd(top, bot), 0.25);
                });
}

// ---------------------------------------------------------------------------------------------------
// config-1 microbenchmark: stand-alone fp32 blocks -> dctArai -> quantize -> zigzag int16
// ---------------------------------------------------------------------------------------------------
constexpr int kMbThreads = 128;
constexpr int kMbPitch = 256 + 16;            // bytes between blocks in shared memory (conflict-free 16-byte reads)

__global__ void __launch_bounds__(kMbThreads) dct_blocks_kernel(const float* __restrict__ in, int16_t* __restrict__ out,
                                                                uint64_t nblocks, uint32_t* refine_list,
                                                                uint32_t* refine_count, uint32_t refine_cap,
                                                                const __grid_constant__ QuantConsts2 q) {
    __shared__ alignas(128) uint8_t tile[kMbThreads * kMbPitch];
    __shared__ alignas(8) uint64_t bar;
    const int tid = threadIdx.x;
    const uint64_t first = static_cast<uint64_t>(blockIdx.x) * kMbThreads;
    const int nb = static_cast<int>(umin64(kMbThreads, nblocks - first));
    if (tid == 0) {
        ptx::mbar_init(&bar, 1);
        ptx::mbar_init_fence();
    }
    __syncthreads();
    if (tid == 0) ptx::mbar_expect_tx(&bar, nb * 256);
    __syncthreads();                            // the expected byte count is armed before any copy can complete
    if (tid < nb) ptx::bulk_g2s(tile + tid * kMbPitch, in + (first + tid) * 64, 256, &bar);
    ptx::mbar_wait(&bar, 0);

    f2 v[32];                                   // v[r*4+p] = samples (r, 2p), (r, 2p+1)
    if (tid < nb) {
        const float4* src = reinterpret_cast<const float4*>(tile + tid * kMbPitch);
#pragma unroll
        for (int j = 0; j < 16; ++j) {
            const float4 f = src[j];
            v[2 * j] = make_float2(f.x, f.y);
            v[2 * j + 1] = make_float2(f.z, f.w);
        }
    }
    __syncthreads();                            // all inputs are in registers: reuse the tile as output staging
    if (tid < nb) {
        uint32_t packed[32];
        dct8x8_packed<false>(v);
        if (quantize_pack_packed(v, q, packed)) {
            const uint32_t at = atomicAdd(refine_count, 1u);
            if (at < refine_cap) refine_list[at] = static_cast<uint32_t>(first + tid);
        }
        stage_block(tile, tid, packed);
    }
    // (a tensor store as in forward_kernel was measured here too: this kernel is bound by HBM, not by instruction issue,
    // and holding the CTA until the copy engine has read the tile costs more than the saved instructions: 1.06 -> 1.11 ms)
    __syncthreads();
    copy_out(tile, out + first * 64, nb, tid, kMbThreads);
}

// stand-alone blocks: every block uses table e.qy; ids index blocks directly
__global__ void __launch_bounds__(kRefineThreads) refine_blocks_kernel(const float* __restrict__ in, int16_t* __restrict__ out,
                                                                           const uint32_t* __restrict__ list,
                                                                           const uint32_t* __restrict__ count, uint32_t cap,
                                                                           uint32_t nblocks, int all,
                                                                           const __grid_constant__ ExactConsts e) {
    const uint32_t n = all ? nblocks : min(*count, cap);
    refine_loop(0u, n, list, all != 0, out, 0xFFFFFFFFu, e.qy, e.qy, e,
                [&](uint32_t id, int c) { return in + static_cast<size_t>(id) * 64 + c; },
                [](const float* col, int r) { return static_cast<double>(col[r * 8]); });
}

// band-wise encodes: everything in the list so far has been refined
__global__ void refine_advance_kernel(uint32_t* counters, uint32_t cap) { counters[3] = min(counters[0], cap); }

// reference planar natural-order int32 planes -> MCU-ordered zigzag int16 (test hook behind jpgenc_set_coefficients)
__global__ void planes_to_mcu_kernel(const int32_t* __restrict__ qy, const int32_t* __restrict__ qcb,
                                     const int32_t* __restrict__ qcr, int16_t* __restrict__ coef, uint32_t mcu_w,
                                     uint32_t nblocks) {
    const uint64_t i = static_cast<uint64_t>(blockIdx.x) * blockDim.x + threadIdx.x;
    if (i >= static_cast<uint64_t>(nblocks) * 64) return;
    const uint32_t id = static_cast<uint32_t>(i >> 6), z = i & 63, n = c_zigzag[z];
    const uint32_t mcu = id / kBlocksPerMcu, k = id % kBlocksPerMcu, mx = mcu % mcu_w, my = mcu / mcu_w;
    int32_t val;
    if (k < 4) {
        const size_t W = static_cast<size_t>(mcu_w) * 16;
        val = qy[(static_cast<size_t>(my) * 16 + (k >> 1) * 8 + (n >> 3)) * W + mx * 16 + (k & 1) * 8 + (n & 7)];
    } else {
        const size_t W = static_cast<size_t>(mcu_w) * 8;
        val = (k == 4 ? qcb : qcr)[(static_cast<size_t>(my) * 8 + (n >> 3)) * W + mx * 8 + (n & 7)];
    }
    coef[i] = static_cast<int16_t>(val);
}

// ---------------------------------------------------------------------------------------------------
// host side
// ---------------------------------------------------------------------------------------------------
void default_dct_constants(double a[5], double s[8]) {
    // the reference's expressions, include/Dct.hpp:21-43 (pi and root_two are Boost's double constants)
    const double pi = 3.141592653589793238462643383279502884;
    const double root_two = 1.414213562373095048801688724209698078;
    double c[8];
    for (int k = 1; k < 8; ++k) c[k] = std::cos(k * pi / 16);
    a[0] = c[4];
    a[1] = c[2] - c[6];
    a[2] = c[4];
    a[3] = c[6] + c[2];
    a[4] = c[6];
    s[0] = 1 / (2 * root_two);
    for (int k = 1; k < 8; ++k) s[k] = 1 / (4 * c[k]);
}

// ---- how far the FP32 fast path can be from the reference: a computed, rigorous bound per coefficient ------------
// Every intermediate of the two packed AAN passes (aan8x2 / aan8x2_split, identical operation sequences) is tracked as
// (mag, err): mag bounds the magnitude of the ideal (real-arithmetic = reference, whose double rounding is ~1e-13)
// value, err bounds |fp32 value - ideal value|.  With u = 2^-24: an addition adds u*(|x|+|y|) to the incoming errors, a
// multiplication by a constant c (itself rounded to fp32) scales them by |c| and adds 2u|c||x|; an FMA does both.
// Magnitudes are propagated as sums, i.e. for the worst 8-bit input pattern.  The result (0.009 for the DC term up to
// 0.030 for the (1,1)/(7,7)-type terms) replaces a single hand-derived constant: low frequencies, where almost all
// rounding-boundary hits occur, get a 2-3 times tighter threshold, which cuts the number of blocks sent to the FP64 path.
namespace {
struct Bound { double mag, err; };
constexpr double kU = 5.9604644775390625e-8;                      // 2^-24
Bound b_add(Bound x, Bound y) { return {x.mag + y.mag, x.err + y.err + kU * (x.mag + y.mag + x.err + y.err)}; }
Bound b_mul(Bound x, double c) {
    c = std::fabs(c);
    return {c * x.mag, c * (1 + kU) * x.err + kU * c * x.mag + kU * c * (1 + kU) * (x.mag + x.err)};
}
Bound b_fma(Bound x, double c, Bound y) {                            // x * c + y
    c = std::fabs(c);
    const double prod = c * (1 + kU) * (x.mag + x.err);
    return {c * x.mag + y.mag, c * (1 + kU) * x.err + kU * c * x.mag + y.err + kU * (prod + y.mag + y.err)};
}
void b_aan8(const Bound (&x)[8], Bound (&o)[8]) {                    // same dataflow as aan8x2
    constexpr double A1 = 0.70710678118654752, A2 = 0.54119610014619698, A4 = 1.30656296487637653, A5 = 0.38268343236508977;
    const Bound z0 = b_add(x[0], x[7]), z1 = b_add(x[1], x[6]), z2 = b_add(x[2], x[5]), z3 = b_add(x[3], x[4]);
    const Bound z4 = b_add(x[3], x[4]), z5 = b_add(x[2], x[5]), z6 = b_add(x[1], x[6]), z7 = b_add(x[0], x[7]);
    const Bound r0 = b_add(z0, z3), r1 = b_add(z1, z2), r2 = b_add(z1, z2), r3 = b_add(z0, z3);
    const Bound n4 = b_add(z4, z5), r5 = b_add(z5, z6), r6 = b_add(z6, z7);
    const Bound t2 = b_add(r2, r3);
    const Bound tmp = b_mul(b_add(r6, n4), A5);
    const Bound u4 = b_fma(n4, A2, tmp), u6 = b_fma(r6, A4, tmp), v5 = b_fma(r5, A1, z7), v7 = b_fma(r5, A1, z7);
    o[0] = b_add(r0, r1); o[4] = b_add(r0, r1); o[2] = b_fma(t2, A1, r3); o[6] = b_fma(t2, A1, r3);
    o[5] = b_add(u4, v7); o[1] = b_add(v5, u6); o[7] = b_add(v5, u6); o[3] = b_add(v7, u4);
}
// bounds of the unscaled 2-D output F[v][u] for samples in [-128, 128] that carry an input error of at most err_in
void aan2d_bounds(double err_in, Bound (&out)[64]) {
    Bound in[8], pass1[8];
    for (Bound& b : in) b = {128.0, err_in};
    b_aan8(in, pass1);
    for (int v = 0; v < 8; ++v) {
        Bound row[8], res[8];
        for (Bound& b : row) b = pass1[v];
        b_aan8(row, res);
        for (int u = 0; u < 8; ++u) out[v * 8 + u] = res[u];
    }
}
// error of the colour conversion feeding the transform (the reference's value is exact to ~1e-13: float constants times
// small integers, summed in double).  maxval 255: the folded constants ARE the reference's float constants (Y) or those
// divided by 4 (Cb, Cr, applied to the exact 2x2 sums), so only the three roundings of the FMA chain remain, each at most
// half an ulp of a value below 128 in magnitude: 3 x 2^-18 = 1.15e-5.  Other maxvals: the constants carry the rounded
// factor 255/maxval (<= 1404 u for Y).  The stand-alone block kernel has exact inputs.
constexpr double kColourErr255 = 2.0e-5, kColourErrScaled = 1.0e-4;
}  // namespace

void fill_quant_consts(const uint8_t q[64], const double s[8], QuantConsts* out, double input_err) {
    Bound bound[64];
    aan2d_bounds(input_err, bound);
    for (int v = 0; v < 8; ++v)
        for (int u = 0; u < 8; ++u) {
            const int i = v * 8 + u;
            const double m = s[v] * s[u] / static_cast<double>(q[i]);
            out->mul[i] = static_cast<float>(m);
            // |fp32 quotient - reference quotient| <= m * (err + u * mag)  [transform error, rounding of m]  + the final FMA
            double delta = 1.0001 * m * (bound[i].err + kU * bound[i].mag) + 1e-7;
            if (delta > 0.25) delta = 0.25;
            out->thr[i] = static_cast<float>(0.5 - delta);
        }
}

static void fill_quant_consts2(const uint8_t q[64], const double s[8], QuantConsts2* out, double input_err) {
    QuantConsts c;
    fill_quant_consts(q, s, &c, input_err);
    for (int u = 0; u < 8; ++u)
        for (int qq = 0; qq < 4; ++qq) {
            const int lo = (2 * qq) * 8 + u, hi = (2 * qq + 1) * 8 + u;
            out->mul[u * 4 + qq] = make_float2(c.mul[lo], c.mul[hi]);
            out->thr[u * 4 + qq] = make_float2(c.thr[lo], c.thr[hi]);
        }
}

static void fill_exact(const jpgenc_ctx* c, const uint8_t* qy, const uint8_t* qc, double scale, ExactConsts* e) {
    e->a1 = c->dct_a[0]; e->a2 = c->dct_a[1]; e->a3 = c->dct_a[2]; e->a4 = c->dct_a[3]; e->a5 = c->dct_a[4];
    for (int i = 0; i < 8; ++i) e->s[i] = c->dct_s[i];
    e->scale = scale;
    for (int i = 0; i < 64; ++i) { e->qy[i] = qy[i]; e->qc[i] = qc[i]; }
}

// tensor map over an array of coefficient blocks as [blocks][64 x int16] with a box of `box_blocks` rows and the 128-byte
// swizzle: what a CTA has staged in shared memory (stage_block) leaves with one tensor store
static bool make_block_map(void* base, uint64_t nblocks, uint32_t box_blocks, CUtensorMap* map) {
    using Encode = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*, const cuuint32_t*,
                                const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
    static Encode encode = [] {                   // libcuda is not linked: the entry point comes from the runtime
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q) != cudaSuccess || q != cudaDriverEntryPointSuccess) fn = nullptr;
        return reinterpret_cast<Encode>(fn);
    }();
    if (!encode || nblocks == 0 || (reinterpret_cast<uintptr_t>(base) & 15)) return false;
    const cuuint64_t gdim[2] = {64, nblocks};
    const cuuint64_t gstride[1] = {kBlockBytes};
    const cuuint32_t box[2] = {64, box_blocks};
    const cuuint32_t estride[2] = {1, 1};
    return encode(map, CU_TENSOR_MAP_DATA_TYPE_UINT16, 2, base, gdim, gstride, box, estride, CU_TENSOR_MAP_INTERLEAVE_NONE,
                  CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}
// Everything K1 needs to know about the image(s) bound to the context
static void fill_forward_params(const jpgenc_ctx* c, ForwardParams* p) {
    p->rgb = c->src.plane[0];
    p->src = c->src;
    p->frames = c->nframes > 1 ? c->d_frame_ptrs : nullptr;
    p->blocks_per_frame = c->mcu_w * c->mcu_h * kBlocksPerMcu;
    p->coef = c->d_coef;
    p->refine_list = c->d_refine_list;
    p->refine_count = c->d_counters;
    p->refine_cap = static_cast<uint32_t>(c->refine_cap);
    p->real_w = c->real_w; p->real_h = c->real_h; p->mcu_w = c->mcu_w; p->mcu_h = c->mcu_h;
    const double scale = 255. / c->maxval;
    const float fy[3] = {.299f, .587f, .114f}, fcb[3] = {-.1687f, -.3312f, .5f}, fcr[3] = {.5f, -.4186f, -.0813f};
    for (int i = 0; i < 3; ++i) {
        p->color.y[i] = static_cast<float>(fy[i] * scale);
        p->color.cb[i] = static_cast<float>(fcb[i] * scale / 4);
        p->color.cr[i] = static_cast<float>(fcr[i] * scale / 4);
    }
    // YUV 4:2:0 samples reach the transform unconverted: byte - 128, exact integers in [-128, 127], inside the [-128, 128] that
    // aan2d_bounds assumes, with no input error -- the stand-alone block kernel's case.  Their thresholds are tighter than the
    // RGB ones, so an RGB encode must never take them (nor a YUV encode the RGB ones, which would only flag more blocks): they
    // follow the layout of the image(s) bound, computed anew for every launch.
    const int format = c->mixed.on ? c->mixed.format : c->src.format;
    const double colour_err = is_yuv(format) ? 0.0 : c->maxval == 255 ? kColourErr255 : kColourErrScaled;
    fill_quant_consts2(c->qy, c->dct_s, &p->luma, colour_err);
    fill_quant_consts2(c->qc, c->dct_s, &p->chroma, colour_err);
}

// calls f(std::integral_constant<int, format>) for an internal format, or -1 for tight RGB: the kernels take the format as a
// template parameter; false (and no call) for a code that is no format (check_source refuses those before anything is bound)
template <class F>
static bool with_format(int format, F&& f) {
    switch (format) {
        case -1: f(std::integral_constant<int, -1>{}); break;
        case JPGENC_PIXEL_RGB: f(std::integral_constant<int, JPGENC_PIXEL_RGB>{}); break;
        case JPGENC_PIXEL_BGR: f(std::integral_constant<int, JPGENC_PIXEL_BGR>{}); break;
        case JPGENC_PIXEL_RGBA: f(std::integral_constant<int, JPGENC_PIXEL_RGBA>{}); break;
        case JPGENC_PIXEL_BGRA: f(std::integral_constant<int, JPGENC_PIXEL_BGRA>{}); break;
        case JPGENC_PIXEL_GRAY: f(std::integral_constant<int, JPGENC_PIXEL_GRAY>{}); break;
        case kPixelPlanar: f(std::integral_constant<int, kPixelPlanar>{}); break;
        case kPixelI420: f(std::integral_constant<int, kPixelI420>{}); break;
        case kPixelNV12: f(std::integral_constant<int, kPixelNV12>{}); break;
        case kPixelI422: f(std::integral_constant<int, kPixelI422>{}); break;
        case kPixelNV16: f(std::integral_constant<int, kPixelNV16>{}); break;
        case kPixelI444: f(std::integral_constant<int, kPixelI444>{}); break;
        case kPixelYUYV: f(std::integral_constant<int, kPixelYUYV>{}); break;
        case kPixelUYVY: f(std::integral_constant<int, kPixelUYVY>{}); break;
        default: return false;
    }
    return true;
}
static int unknown_format(jpgenc_ctx* c) {
    c->error = "internal: pixel format without kernels";
    return JPGENC_ERR_ARG;
}

// the format the kernels of the single image bound take: its own, or -1 when it is tight RGB
static int kernel_format(const jpgenc_ctx* c) {
    return c->src.format != JPGENC_PIXEL_RGB || c->src.pitch != c->real_w * 3 ? c->src.format : -1;
}

// The refinement over `total` blocks: grid-stride over the list; a small image does not need (and should not wait for) 2368
// mostly empty CTAs.  64 threads per block where the flagged blocks are few (latency: 3840x2160 15 -> 6 us), 8 per block where
// they are many (throughput: at 16384^2 the 64-thread form's barriers cost 42 us against 28).  f(std::bool_constant<k64>, grid).
template <class F>
static void with_refine_grid(const jpgenc_ctx* c, uint64_t total, F&& f) {
    const unsigned grid = static_cast<unsigned>(std::max<uint64_t>(c->sm_count, std::min<uint64_t>(c->sm_count * 16, total / 256 + 1)));
    if (total < (3u << 19)) f(std::true_type{}, grid);
    else f(std::false_type{}, grid);
}

// exact FP64 pass over the blocks K1 flagged (all == false) or over every block (all == true)
static int launch_refine(jpgenc_ctx* c, bool all) {
    ExactConsts e;
    fill_exact(c, c->qy, c->qc, 255. / c->maxval, &e);
    const uint32_t bpf = c->mcu_w * c->mcu_h * kBlocksPerMcu;
    const uint32_t cap = all ? 0u : static_cast<uint32_t>(c->refine_cap);
    const uint8_t* const* frames = c->nframes > 1 ? c->d_frame_ptrs : nullptr;
    if (!with_format(kernel_format(c), [&](auto fmt) {
            with_refine_grid(c, static_cast<uint64_t>(bpf) * c->nframes, [&](auto k64, unsigned grid) {
                refine_kernel<decltype(k64)::value, decltype(fmt)::value><<<grid, kRefineThreads, 0, c->stream>>>(
                    c->src.plane[0], frames, bpf, c->d_coef, c->d_refine_list, c->d_counters, cap, all ? 1 : 0, bpf * c->nframes, c->real_w, c->real_h, c->mcu_w,
                    e, c->src);
            });
        }))
        return unknown_format(c);
    JPGENC_CUDA(c, cudaGetLastError());
    c->launches += 1;
    return JPGENC_OK;
}

// K1 over the MCU rows [y0, y0 + rows) of every frame.  The whole image is the common case; jpgenc_encode_rgb launches
// it band by band behind the matching host-to-device copies.  `first` clears the refinement list, `last` appends the
// exact refinement pass over everything the bands flagged.
int launch_forward_rows(jpgenc_ctx* c, uint32_t y0, uint32_t rows, bool first, bool last) {
    ForwardParams p{};
    fill_forward_params(c, &p);
    p.mcu_y0 = y0;
    // measured on 16384^2 (740 resident CTAs): 150..550 strips ahead all take K1 from 0.328 to 0.317 ms; further ahead loses
    p.prefetch_ahead = 256;
    if (first && !launch_encode_clear(c))                                                          // counters + K2's / K3a's accumulators in one kernel
        JPGENC_CUDA(c, cudaMemsetAsync(c->d_counters, 0, 4 * sizeof(uint32_t), c->stream));          // (no statistics buffers yet) list length .. refined so far
    bool aligned = (c->real_w % 16 == 0) && (reinterpret_cast<uintptr_t>(c->src.plane[0]) % 16 == 0);
    if (c->nframes > 1) aligned = (c->real_w % 16 == 0) && c->frames_aligned;
    // (strips of 24 and of 40 MCUs, which divide 1920- and 3840-pixel rows evenly, were measured: no gain on those frames
    // -- the partial fourth strip is not what costs -- and 24 is 7 % slower where 32 divides the row)
    const dim3 grid((c->mcu_w + 31) / 32, rows, c->nframes);
    if (kernel_format(c) >= 0) {
        // each CTA picks its staging path from the image (stage_layout); the tensor store serves every full strip
        const bool bulk = make_block_map(c->d_coef, static_cast<uint64_t>(c->mcu_w) * c->mcu_h * kBlocksPerMcu, 32 * kBlocksPerMcu, &p.coef_map);
        if (!with_format(c->src.format, [&](auto fmt) {
                constexpr int kFmt = decltype(fmt)::value;
                if constexpr (kFmt >= 0) {
                    if (bulk) forward_layout_kernel<32, kFmt, true><<<grid, 128, 0, c->stream>>>(p);
                    else forward_layout_kernel<32, kFmt, false><<<grid, 128, 0, c->stream>>>(p);
                }
            }))
            return unknown_format(c);
        JPGENC_CUDA(c, cudaGetLastError());
        c->launches += 1;
        return last ? launch_refine(c, false) : JPGENC_OK;
    }
    const bool bulk_out = aligned &&
                          make_block_map(c->d_coef, static_cast<uint64_t>(c->mcu_w) * c->mcu_h * kBlocksPerMcu * c->nframes, 32 * kBlocksPerMcu, &p.coef_map);
    if (bulk_out) forward_kernel<32, true, true><<<grid, 128, 0, c->stream>>>(p);
    else if (aligned) forward_kernel<32, true><<<grid, 128, 0, c->stream>>>(p);
    else forward_kernel<32, false><<<grid, 128, 0, c->stream>>>(p);
    JPGENC_CUDA(c, cudaGetLastError());
    c->launches += 1;
    return last ? launch_refine(c, false) : JPGENC_OK;
}

// K1 + exact refinement over a pass of images of individual sizes.  The bulk copies need every image of the pass to qualify
// (c->mixed.aligned); the tensor store serves the full strips of every image, the copy-out the partial ones.  Pixels in another
// layout (c->mixed.format >= 0) take the pixel-layout kernels, where each CTA picks its staging path from its own image.
int launch_forward_mixed(jpgenc_ctx* c) {
    ForwardParams p{};
    fill_forward_params(c, &p);                                   // (its per-size fields are not read by forward_mixed_kernel)
    p.geom = c->d_geom;
    p.nframes = c->nframes;
    p.strips = c->mixed.strips;
    p.prefetch_ahead = 256;
    JPGENC_CUDA(c, cudaMemsetAsync(c->d_counters, 0, 4 * sizeof(uint32_t), c->stream));
    c->stats_clear_valid = false;                                 // K2 clears the statistics and K3a's sums itself
    const bool layout = c->mixed.format >= 0;
    const bool aligned = c->mixed.aligned;
    // formats of several planes: each image's other planes lie behind the geometry (enqueue_pass copies them in the same transfer)
    p.extra = source_planes(c->mixed.format) == 3 ? reinterpret_cast<const ExtraPlanes*>(c->d_geom + c->nframes + 1) : nullptr;
    const bool bulk_out = (aligned || layout) && make_block_map(c->d_coef, c->mixed.blocks, 32 * kBlocksPerMcu, &p.coef_map);
    if (layout) {
        if (!with_format(c->mixed.format, [&](auto fmt) {
                constexpr int kFmt = decltype(fmt)::value;
                if constexpr (kFmt >= 0) {
                    if (bulk_out) forward_mixed_layout_kernel<32, kFmt, true><<<c->mixed.strips, 128, 0, c->stream>>>(p);
                    else forward_mixed_layout_kernel<32, kFmt, false><<<c->mixed.strips, 128, 0, c->stream>>>(p);
                }
            }))
            return unknown_format(c);
    } else if (bulk_out) forward_mixed_kernel<32, true, true><<<c->mixed.strips, 128, 0, c->stream>>>(p);
    else if (aligned) forward_mixed_kernel<32, true, false><<<c->mixed.strips, 128, 0, c->stream>>>(p);
    else forward_mixed_kernel<32, false, false><<<c->mixed.strips, 128, 0, c->stream>>>(p);
    JPGENC_CUDA(c, cudaGetLastError());
    ExactConsts e;
    fill_exact(c, c->qy, c->qc, 255. / c->maxval, &e);
    const uint32_t cap = static_cast<uint32_t>(c->refine_cap);
    if (!with_format(c->mixed.format, [&](auto fmt) {
            with_refine_grid(c, c->mixed.blocks, [&](auto k64, unsigned grid) {
                refine_mixed_kernel<decltype(k64)::value, decltype(fmt)::value><<<grid, kRefineThreads, 0, c->stream>>>(
                    c->d_geom, c->nframes, c->d_coef, c->d_refine_list, c->d_counters, cap, e, p.extra);
            });
        }))
        return unknown_format(c);
    JPGENC_CUDA(c, cudaGetLastError());
    c->launches += 2;
    return JPGENC_OK;
}

// exact pass over the list entries that have not been refined yet (after a band of K1), and remember how far it got
int launch_refine_pending(jpgenc_ctx* c) {
    const int rc = launch_refine(c, false);
    if (rc) return rc;
    refine_advance_kernel<<<1, 1, 0, c->stream>>>(c->d_counters, static_cast<uint32_t>(c->refine_cap));
    JPGENC_CUDA(c, cudaGetLastError());
    return JPGENC_OK;
}

int launch_forward(jpgenc_ctx* c) {
    JPGENC_CUDA(c, stage_record(c, c->ev_k0, 1));
    // the fast kernel alone is timed (ev_k0..ev_k1): it is the roofline kernel; the refinement follows
    const int rc = launch_forward_rows(c, 0, c->mcu_h, true, false);
    if (rc) return rc;
    JPGENC_CUDA(c, stage_record(c, c->ev_k1, 1));
    return launch_refine(c, false);
}

int launch_exact_all(jpgenc_ctx* c) { return launch_refine(c, true); }

// coefficients of the image bound as planes of doubles (d_planes: three planes of (mcu_w*16) x (mcu_h*16) doubles back to back)
int launch_planes_exact(jpgenc_ctx* c, const double* d_planes, bool ycbcr) {
    ExactConsts e;
    fill_exact(c, c->qy, c->qc, 1.0, &e);
    const uint32_t nblocks = c->mcu_w * c->mcu_h * kBlocksPerMcu;
    const size_t plane = static_cast<size_t>(c->mcu_w) * 16 * c->mcu_h * 16;
    const unsigned grid = static_cast<unsigned>(std::max<uint64_t>(1, std::min<uint64_t>(c->sm_count * 16, (static_cast<uint64_t>(nblocks) * 8 + kRefineThreads - 1) / kRefineThreads)));
    planes_exact_kernel<<<grid, kRefineThreads, 0, c->stream>>>(d_planes, d_planes + plane, d_planes + 2 * plane, c->mcu_w * 16, c->mcu_w, nblocks, c->d_coef,
                                                               ycbcr ? 1 : 0, e);
    JPGENC_CUDA(c, cudaGetLastError());
    c->launches += 1;
    return JPGENC_OK;
}

int launch_dct_quant_blocks(jpgenc_ctx* c, const float* in, int16_t* out, uint64_t nblocks, const uint8_t q[64],
                            uint64_t* refined) {
    QuantConsts2 qc;
    fill_quant_consts2(q, c->dct_s, &qc, 0.0);                 // stand-alone blocks: the samples are the inputs themselves
    ExactConsts e;
    fill_exact(c, q, q, 1.0, &e);
    JPGENC_CUDA(c, cudaMemsetAsync(c->d_counters, 0, sizeof(uint32_t), c->stream));
    const uint64_t grid = (nblocks + kMbThreads - 1) / kMbThreads;
    dct_blocks_kernel<<<static_cast<unsigned>(grid), kMbThreads, 0, c->stream>>>(
        in, out, nblocks, c->d_refine_list, c->d_counters, static_cast<uint32_t>(c->refine_cap), qc);
    JPGENC_CUDA(c, cudaGetLastError());
    refine_blocks_kernel<<<c->sm_count * 16, kRefineThreads, 0, c->stream>>>(
        in, out, c->d_refine_list, c->d_counters, static_cast<uint32_t>(c->refine_cap), static_cast<uint32_t>(nblocks), 0, e);
    JPGENC_CUDA(c, cudaGetLastError());
    c->launches += 2;
    if (refined) {
        uint32_t n = 0;
        JPGENC_CUDA(c, cudaMemcpyAsync(&n, c->d_counters, sizeof n, cudaMemcpyDeviceToHost, c->stream));
        JPGENC_CUDA(c, cudaStreamSynchronize(c->stream));
        if (n > c->refine_cap) {   // list overflowed: redo everything exactly (correct, slow, never seen on real data)
            refine_blocks_kernel<<<c->sm_count * 16, kRefineThreads, 0, c->stream>>>(
                in, out, c->d_refine_list, c->d_counters, static_cast<uint32_t>(c->refine_cap), static_cast<uint32_t>(nblocks), 1, e);
            JPGENC_CUDA(c, cudaGetLastError());
            c->launches += 1;
        }
        *refined = n;
    }
    return JPGENC_OK;
}

int launch_planes_to_mcu(jpgenc_ctx* c, const int32_t* d_qy, const int32_t* d_qcb, const int32_t* d_qcr) {
    const uint32_t nblocks = c->mcu_w * c->mcu_h * kBlocksPerMcu;
    const uint64_t n = static_cast<uint64_t>(nblocks) * 64;
    planes_to_mcu_kernel<<<static_cast<unsigned>((n + 255) / 256), 256, 0, c->stream>>>(d_qy, d_qcb, d_qcr, c->d_coef,
                                                                                       c->mcu_w, nblocks);
    JPGENC_CUDA(c, cudaGetLastError());
    c->launches += 1;
    return JPGENC_OK;
}

}  // namespace jpgenc
