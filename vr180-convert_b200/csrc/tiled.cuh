// tiled.cuh -- definitions shared by the TMA-tiled kernels (tiled.cu: batches of frames per tile; stream.cu: tiles
// streamed through persistent CTAs for launches of one or two frames): shared-memory layout, TMA / mbarrier
// primitives, the tile-packed LUT format and the per-interpolation sampling modes.
#pragma once
#include <cuda.h>  // CUtensorMap + enums only; cuTensorMapEncodeTiled is fetched with cudaGetDriverEntryPoint

#include <cmath>
#include <cstdlib>
#include <mutex>
#include <type_traits>
#include <vector>

#include "chain_fast.cuh"
#include "common.cuh"
#include "sampler.cuh"

namespace vr180 {
namespace tiled {

constexpr int kTileW = 32;      // output tile width.  Per step a warp covers 32 pixels: one output row (bilinear: the
                                // taps of a row are ~26 consecutive source pixels = ~20 consecutive words, one
                                // wavefront per load while the row stays in one source row) or an 8 x 4 patch (bicubic)
constexpr int kSamplers = 256;  // 8 sampling warps
constexpr int kThreads = kSamplers + 32;  // + the TMA producer warp
constexpr int kMaxStages = 8;   // ring depth is chosen per tile: kStageArea / (bytes of the tile's source rectangle)
constexpr int kRowsStep = 4, kRowSizes = 9;  // TMA load box heights: Mode::kRowsMin + 4 r, r < 9
// Staged row pitch = TMA box width (bytes), a multiple of 16 picked PER TILE: the smallest kPitchCands widths that
// hold the tile's source rectangle are compared by the bank conflicts of the tile's own tap addresses (counted with
// match.any in the prologue) plus the shared-memory wavefronts of the TMA write of the box itself.
constexpr int kPitchMin = 96, kPitchMax = 256, kPitchStep = 16;
constexpr int kWidths = (kPitchMax - kPitchMin) / kPitchStep + 1;  // 11 box widths
constexpr int kPitchCands = 4;
constexpr int kStageAreaDefault = 40960;  // >= 1 two-frame stage of the largest admissible rectangle (64 rows x 256 B)
constexpr int kOutBufs = 4;        // ofull / oempty barrier slots; out buffers in use: M::kOutTiles / FR (a power of two <= 4)
// Shared-memory layout of a CTA; the staging area is a property of the interpolation mode (M::kStageArea).
template <class M>
struct Lay {
    static constexpr int kStageArea = M::kStageArea;
    static constexpr int kOutArea = M::kOutTiles * M::kTileH * kTileW * 3;
    static constexpr int kOffOut = kStageArea;
    static constexpr int kOffTrig = kOffOut + kOutArea;
    static constexpr int kOffRed = kOffTrig + 7 * 32 * 8;  // double[4][32] sincos of the tile's columns / rows, or chain_fast.cuh's tables [4 + 3][32]
    static constexpr int kOffBar = kOffRed + 8 * 4 * 4;  // full[kMaxStages], empty[kMaxStages], ofull[kOutBufs], oempty[kOutBufs]
    static constexpr int kOffOrg = kOffBar + (2 * kMaxStages + 2 * kOutBufs) * 8;  // int2 origin of the rectangle in each stage
    static constexpr int kOffExt = kOffOrg + kMaxStages * 8;                         // double[8][4] per-warp normalised extremes
    static constexpr int kOffCost = kOffExt + 8 * 4 * 8;                             // int[kPitchCands] candidate pitch costs
    static constexpr int kOffW = (kOffCost + 16 + 15) & ~15;  // M::kWeightSmem bytes of per-pixel weights (Lanczos4)
    static constexpr int kSmemBytes = kOffW + M::kWeightSmem;
};

// stage slot of the tile-streaming kernel (stream.cu): a ring of 3 fixed-size slots in the mode's staging area
template <class M>
constexpr int kStreamSlotBytes = (M::kStageArea / 3) & ~127;

// The standard chain shape, lowered once on the host (see match_std_chain):
//   Normalize, EquirectangularEncoder, [Euclidean3DRotator], [PolynomialScaler], FisheyeDecoder("equidistant"),
//   Denormalize
struct StdChain {
    int valid, lat_is_y, has_rot, n_poly;
    int fast, pad_;   // R orthonormal (identity without a rotation): the folded evaluation of chain_fast.cuh applies
    double norm[3];   // cx, cy, scale
    double R[9];
    double poly[VR180_MAX_OP_PARAMS];
    double den[4];    // sx, sy, cx, cy
};

struct TiledParams {
    int tiles_x;
    int n_tiles;     // tiles of one map (tiles_x * tiles_y): layout of a tile-packed LUT
    int sep_prefix;  // generic chains only: ops[0..1] = Normalize, EquirectangularEncoder
    int debug;       // VR180_TILED_DEBUG: bit 8 = the standard chain through the op-by-op interpreter (chain.cuh)
    int zero_border; // BORDER_CONSTANT with a zero colour: TMA's out-of-bounds zero fill IS the border, so tiles that
                     // straddle the source edge stay staged; any other border only stages tiles that lie inside the source
    const short* tab;  // bicubic: OpenCV's 1024 x 16 int16 weight table (device)
    StdChain std[2];
};

// TMA descriptors of one launch (kernel parameter; the TMA unit reads them from the parameter bank).
struct alignas(64) TmaMaps {
    CUtensorMap src[2][kWidths][kRowSizes];  // [view][box bytes kPitchMin + 16 w][box rows kRowsMin + 8 r]: uint8 (cols * 3, rows, frames)
    CUtensorMap dst;                   // uint8 (dst_pitch, H, frames), box (96, tile height, 1)
};

// ---- tile-packed LUT (include/vr180_b200.h, vr180_pack_lut_tiles) -----------------------------------------------
// buffer = [n_tiles x PackedHdr][pad to 256 bytes][n_tiles x (256 threads x kPx) uint32, thread-major]
// entry  = (ix - mnx) | (iy - mny) << 8 | ax << 16 | ay << 21     (ax = ay = 0 for INTER_NEAREST)
struct PackedHdr {
    short mnx, mxx, mny, mxy;  // integer source coordinates of the tile: min / max of ix and iy
    int flags;                 // kHdr* bits | box width index << 8 | box row index << 12 (see k_pack_tiles)
    int pad;
};
constexpr int kHdrPackable = 1;   // full tile, finite unsaturated coordinates, extents <= 255: the entries are valid
constexpr int kHdrStageable = 2;  // the source rectangle fits a TMA box of this mode (width <= kPitchMax, rows <= the largest box)
constexpr int kHdrFitsSlot = 4;   // ... and one stage slot of the tile-streaming kernel
// bits 8-11: (row pitch - kPitchMin) / kPitchStep chosen for the tile; bits 12-15: box rows = kRowsMin + kRowsStep * r
static_assert(sizeof(PackedHdr) == 16, "PackedHdr is one 128-bit load");
__host__ __device__ inline size_t packed_entries_offset(long long n_tiles) { return ((size_t)n_tiles * 16 + 255) & ~(size_t)255; }
// the header as loaded (the streaming kernel keeps the prefetched next header in this form: three live registers)
__device__ __forceinline__ int4 packed_header_raw(const void* packed, int tile) {
    return __ldg(reinterpret_cast<const int4*>(packed) + tile);
}
struct TileHdr {  // a decoded PackedHdr
    int mnx, mxx, mny, mxy, flags;
};
__device__ __forceinline__ TileHdr decode_header(const int4& v) {
    return {(short)(v.x & 0xffff), v.x >> 16, (short)(v.y & 0xffff), v.y >> 16, v.z};
}
// the tile's kPx entries of thread `tid`: ONE 128-bit (bilinear / nearest), 64-bit (bicubic) or 32-bit (Lanczos4)
// coalesced load
template <class M>
__device__ __forceinline__ void load_packed_entries(const void* packed, int n_tiles, int tile, int tid, uint32_t (&e)[M::kPx]) {
    const uint32_t* ent = reinterpret_cast<const uint32_t*>(static_cast<const uint8_t*>(packed) + packed_entries_offset(n_tiles)) +
                          ((size_t)tile * kSamplers + tid) * M::kPx;
    if constexpr (M::kPx == 4) {
        const uint4 v = __ldg(reinterpret_cast<const uint4*>(ent));
        e[0] = v.x; e[1] = v.y; e[2] = v.z; e[3] = v.w;
    } else if constexpr (M::kPx == 2) {
        const uint2 v = __ldg(reinterpret_cast<const uint2*>(ent));
        e[0] = v.x; e[1] = v.y;
    } else {
        e[0] = __ldg(ent);
    }
}
// entry -> the mode's quantised coordinates (sx, sy), as M::quant would have produced them
template <class M>
__device__ __forceinline__ int2 unpack_entry(int hdr_mnx, int hdr_mny, uint32_t e) {
    return make_int2(((hdr_mnx + (int)(e & 255u)) << M::kShift) | (int)((e >> 16) & 31u),
                     ((hdr_mny + (int)((e >> 8) & 255u)) << M::kShift) | (int)((e >> 21) & 31u));
}

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

// ---- mbarrier / TMA primitives (PTX ISA 8.x, sm_90+) -----------------------------------------------------------
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
// try_wait suspends the warp for up to kSuspendNs before it reports "not yet": fewer polls = fewer shared-memory
// wavefronts and issue slots taken from the sampling warps
constexpr uint32_t kSuspendNs = 4000;
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "WAIT_%=:\n\t"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1, %2;\n\t"
        "@p bra DONE_%=;\n\t"
        "bra WAIT_%=;\n\t"
        "DONE_%=:\n\t}" ::"r"(bar), "r"(parity), "r"(kSuspendNs)
        : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
// global (tensor map, coordinates {x bytes, row, frame}) -> shared, completion counted in bytes on `bar`
__device__ __forceinline__ void tma_load_3d(uint32_t dst, const CUtensorMap* map, int x, int y, int z, uint32_t bar) {
    asm volatile(
        "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%2, %3, %4}], [%5];" ::
            "r"(dst), "l"(map), "r"(x), "r"(y), "r"(z), "r"(bar)
        : "memory");
}
// shared -> global (tensor map, coordinates), tracked by the thread's bulk async-group
__device__ __forceinline__ void tma_store_3d(const CUtensorMap* map, int x, int y, int z, uint32_t src) {
    asm volatile("cp.async.bulk.tensor.3d.global.shared::cta.tile.bulk_group [%0, {%1, %2, %3}], [%4];" ::"l"(map), "r"(x),
                 "r"(y), "r"(z), "r"(src)
                 : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() {  // all but the N newest bulk groups have finished READING smem
    asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory");
}

__device__ __forceinline__ void sts32(uint32_t addr, uint32_t v) {
    asm volatile("st.shared.u32 [%0], %1;" ::"r"(addr), "r"(v) : "memory");
}

// [sat_u8(c0) sat_u8(c1) sat_u8(c2) 0] from three int32: two saturating packs (I2IP) instead of six min / max and
// the shifts / ors that assemble the bytes
__device__ __forceinline__ uint32_t pack_sat_u8x3(int c0, int c1, int c2) {
    uint32_t t, d;
    asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(t) : "r"(0), "r"(c2), "r"(0));
    asm("cvt.pack.sat.u8.s32.b32 %0, %1, %2, %3;" : "=r"(d) : "r"(c1), "r"(c0), "r"(t));
    return d;
}

__device__ __forceinline__ uint32_t dp2a_lo_su(uint32_t w, uint32_t px, uint32_t acc) {  // s16 x u8, bytes 0..1
    uint32_t d;
    asm("dp2a.lo.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(w), "r"(px), "r"(acc));
    return d;
}
__device__ __forceinline__ uint32_t dp2a_hi_su(uint32_t w, uint32_t px, uint32_t acc) {  // s16 x u8, bytes 2..3
    uint32_t d;
    asm("dp2a.hi.s32.u32 %0, %1, %2, %3;" : "=r"(d) : "r"(w), "r"(px), "r"(acc));
    return d;
}

// ---- interpolation modes -------------------------------------------------------------------------------------
// A mode fixes: pixels per thread (the per-pixel constants must stay in registers across the frames of the batch),
// the tile height, the tap footprint (taps start kLo pixels / rows before the integer coordinate and end kHi after
// it), the per-pixel constants and the sampling of one pixel from the staged rectangle.
// INTER_LINEAR: the byte alignment of the taps is done by PRMT with per-pixel selectors rather than by funnel shifts
// (measured on the 64-pair 8K launch: 2.42 G instead of 2.57 G warp instructions, 2.89 instead of 2.95 ms).
// The window of a row is bytes s .. s + 5 (s = offset & 3) of the words [a0 a1 (a2)]:
//   u  = PRMT(a0, a1, selA) = [c0 c0' . .]            c0 at s, c0' at s + 3 <= 6: always inside (a0, a1)
//   t  = PRMT(a0, a1, selT) = [c1 c1' c2 c2']         offsets s + 1, s + 4, s + 2, s + 5 <= 7 for s <= 2; for s == 3
//        the third word is loaded into a0's register first (a0 is dead once u exists) and selT = 0x0574 picks
//        [a1.0 a1.3 a1.1 a0.0]
// i.e. 5 PRMT per pixel instead of 4 SHF + 3 PRMT.  selA shares a register with the window offset (PRMT reads only
// the low 16 bits of its selector; the address is one LEA.HI).
struct LinearP {
    static constexpr int kPx = 4, kTileH = 32, kLo = 0, kHi = 1, kRowsMin = 32, kInterp = VR180_INTER_LINEAR;
    static constexpr int kShift = kInterBits;  // coordinates are 1/32-pixel fixed point: sx = cvRound(x * 32)
    __device__ static __forceinline__ int quant(float m) { return quantise(m); }
    static constexpr int kStageArea = kStageAreaDefault, kWeightSmem = 0, kOutTiles = 4;
    static constexpr bool kRowPatch = true;  // a warp step = 32 pixels of one output row (pixel k of a thread: row 4 band + k)
    struct Pixel {  // constant over the frames of the batch
        uint32_t osel;     // window byte offset (4-aligned) << 16 | selA
        uint32_t selT;
        uint32_t W01, W23; // 16-bit lanes {64 w00, 64 w01}, {64 w10, 64 w11}
    };
    __device__ static __forceinline__ void set_offset(Pixel& p, int off, bool valid) {
        // selA = s | (s + 3) << 4 = 0x30 + 0x11 s;  selT = (s + 1) | (s + 4) << 4 | (s + 2) << 8 | (s + 5) << 12 = 0x5241 +
        // 0x1111 s for s < 3 and 0x0574 = (0x5241 + 0x3333) & 0x7fff for s == 3
        const uint32_t s = (uint32_t)off & 3u;
        p.osel = ((valid ? ((uint32_t)off & ~3u) : 0u) << 16) | (0x30u + 0x11u * s);
        p.selT = (0x5241u + 0x1111u * s) & 0x7fffu;
    }
    // w00 = 1024 (ax = ay = 0, all other weights 0) is encoded as 65535: (65535 p + 32768) >> 16 is still exactly p.
    __device__ static __forceinline__ void weights(Pixel& p, int ax, int ay, const short*) {
        const int w00 = (32 - ax) * (32 - ay), w01 = ax * (32 - ay), w10 = (32 - ax) * ay, w11 = ax * ay;
        p.W01 = (uint32_t)min(64 * w00, 65535) | ((uint32_t)(64 * w01) << 16);
        p.W23 = (uint32_t)(64 * w10) | ((uint32_t)(64 * w11) << 16);
    }
    // One output pixel from the staged rectangle: the three result bytes [c0 c1 c2 0].
    // `sbuf`: shared-window address of the stage, `pitch`: its row pitch in bytes
    __device__ static __forceinline__ uint32_t sample(uint32_t sbuf, const Pixel& p, uint32_t pitch) {
        const uint32_t row0 = sbuf + (p.osel >> 16);
        uint32_t q0, t0, t1;
        asm volatile(
            "{\n\t.reg .pred p;\n\t.reg .b32 a0, a1, b0, b1, u0, u1;\n\t"
            "setp.eq.u32 p, %6, 0x574;\n\t"
            "ld.shared.u32 a0, [%3];\n\t"
            "ld.shared.u32 a1, [%3+4];\n\t"
            "ld.shared.u32 b0, [%4];\n\t"
            "ld.shared.u32 b1, [%4+4];\n\t"
            "prmt.b32 u0, a0, a1, %5;\n\t"
            "prmt.b32 u1, b0, b1, %5;\n\t"
            "@p ld.shared.u32 a0, [%3+8];\n\t"
            "@p ld.shared.u32 b0, [%4+8];\n\t"
            "prmt.b32 %0, u0, u1, 0x5410;\n\t"
            "prmt.b32 %1, a0, a1, %6;\n\t"
            "prmt.b32 %2, b0, b1, %6;\n\t}"
            : "=&r"(q0), "=&r"(t0), "=&r"(t1)
            : "r"(row0), "r"(row0 + pitch), "r"(p.osel), "r"(p.selT));
        // (sum_t w_t p_t + 512) >> 10 == (sum_t 64 w_t p_t + 32768) >> 16: the result is byte 2 of s (s < 2^24)
        const uint32_t s0 = __dp2a_hi(p.W23, q0, __dp2a_lo(p.W01, q0, 32768u));
        const uint32_t s1 = __dp2a_lo(p.W23, t1, __dp2a_lo(p.W01, t0, 32768u));
        const uint32_t s2 = __dp2a_hi(p.W23, t1, __dp2a_hi(p.W01, t0, 32768u));
        return __byte_perm(__byte_perm(s0, s1, 0x0062), s2, 0x7610);
    }
};

// INTER_NEAREST: ix = saturate_int16(cvRound(x)) (no sub-pixel grid), out = src[iy, ix].
struct Nearest {
    static constexpr int kPx = 4, kTileH = 32, kLo = 0, kHi = 0, kRowsMin = 32, kInterp = VR180_INTER_NEAREST;
    static constexpr int kShift = 0;
    __device__ static __forceinline__ int quant(float m) { return cv_round(m); }
    static constexpr int kStageArea = kStageAreaDefault, kWeightSmem = 0, kOutTiles = 4;
    static constexpr bool kRowPatch = true;
    struct Pixel {
        int boff;  // byte offset (4-aligned) of the 8-byte window that holds the pixel
        int sh;    // 8 * (byte offset & 3)
    };
    __device__ static __forceinline__ void set_offset(Pixel& p, int off, bool valid) {
        p.boff = valid ? (off & ~3) : 0;
        p.sh = (off & 3) * 8;
    }
    __device__ static __forceinline__ void weights(Pixel&, int, int, const short*) {}
    __device__ static __forceinline__ uint32_t sample(uint32_t sbuf, const Pixel& p, uint32_t) {
        uint32_t a0, a1;
        asm volatile("ld.shared.u32 %0, [%2];\n\tld.shared.u32 %1, [%2+4];" : "=r"(a0), "=r"(a1) : "r"(sbuf + (uint32_t)p.boff));
        return __funnelshift_r(a0, a1, p.sh);  // [c0 c1 c2 .]: the re-pack never looks at byte 3
    }
};

struct Cubic {
    static constexpr int kPx = 2, kTileH = 16, kLo = 1, kHi = 2, kRowsMin = 16, kInterp = VR180_INTER_CUBIC;
    static constexpr int kShift = kInterBits;  // coordinates are 1/32-pixel fixed point: sx = cvRound(x * 32)
    __device__ static __forceinline__ int quant(float m) { return quantise(m); }
    // a thread owns only 2 pixels (their 16 table weights take 16 registers), so an item is FOUR frames: the
    // per-item bookkeeping is paid once per 8 pixels of a thread, as for the bilinear mode
    static constexpr int kStageArea = kStageAreaDefault, kWeightSmem = 0, kOutTiles = 8;
    static constexpr bool kRowPatch = true;  // a warp step = 32 pixels of one output row (pixel k of a thread: row 2 warp + k)
    struct Pixel {
        int boff;       // byte offset (4-aligned) of the 16-byte window of tap row 0 (iy - 1), first tap ix - 1
        int sh;
        uint32_t w[8];  // itab[ay][ax][ky][kx] as int16 pairs: w[2 ky] = {kx 0, kx 1}, w[2 ky + 1] = {kx 2, kx 3}
    };
    __device__ static __forceinline__ void set_offset(Pixel& p, int off, bool valid) {
        p.boff = valid ? (off & ~3) : 0;
        p.sh = (off & 3) * 8;
    }
    __device__ static __forceinline__ void weights(Pixel& p, int ax, int ay, const short* tab) {
        const uint4* t = reinterpret_cast<const uint4*>(tab + ((ay << 5) | ax) * 16);
        const uint4 lo = __ldg(t), hi = __ldg(t + 1);
        p.w[0] = lo.x; p.w[1] = lo.y; p.w[2] = lo.z; p.w[3] = lo.w;
        p.w[4] = hi.x; p.w[5] = hi.y; p.w[6] = hi.z; p.w[7] = hi.w;
    }
    __device__ static __forceinline__ uint32_t sample(uint32_t sbuf, const Pixel& p, uint32_t pitch) {
        const uint32_t* r = reinterpret_cast<const uint32_t*>(
            static_cast<const uint8_t*>(__cvta_shared_to_generic(sbuf)) + p.boff);
        const int sh = p.sh;
        uint32_t acc0 = 16384u, acc1 = 16384u, acc2 = 16384u;  // + 1 << 14 before the >> 15
#pragma unroll
        for (int ky = 0; ky < 4; ++ky, r += pitch / 4) {
            const uint32_t a0 = r[0], a1 = r[1], a2 = r[2], a3 = r[3];
            // byte-align the 12 tap bytes (taps t0..t3, channels 0..2):
            //   A0 = [t0c0 t0c1 t0c2 t1c0]  A1 = [t1c1 t1c2 t2c0 t2c1]  A2 = [t2c2 t3c0 t3c1 t3c2]
            const uint32_t A0 = __funnelshift_r(a0, a1, sh), A1 = __funnelshift_r(a1, a2, sh),
                           A2 = __funnelshift_r(a2, a3, sh);
            const uint32_t q0 = __byte_perm(__byte_perm(A0, A1, 0x0630), A2, 0x5210);  // [t0c0 t1c0 t2c0 t3c0]
            const uint32_t q1 = __byte_perm(__byte_perm(A0, A1, 0x0741), A2, 0x6210);  // [t0c1 t1c1 t2c1 t3c1]
            const uint32_t q2 = __byte_perm(__byte_perm(A0, A1, 0x0052), A2, 0x7410);  // [t0c2 t1c2 t2c2 t3c2]
            const uint32_t w01 = p.w[2 * ky], w23 = p.w[2 * ky + 1];
            acc0 = dp2a_hi_su(w23, q0, dp2a_lo_su(w01, q0, acc0));
            acc1 = dp2a_hi_su(w23, q1, dp2a_lo_su(w01, q1, acc1));
            acc2 = dp2a_hi_su(w23, q2, dp2a_lo_su(w01, q2, acc2));
        }
        return pack_sat_u8x3((int)acc0 >> 15, (int)acc1 >> 15, (int)acc2 >> 15);  // clip((acc + 16384) >> 15, 0, 255)
    }
};

// INTER_LANCZOS4 (the default interpolation of the reference's apply(), remapper.py:330): 8 x 8 taps.  The 64 int16
// weights of a pixel (OpenCV's 1024 x 64 table) do not fit the register file, so a thread owns ONE pixel (tile
// 32 x 8) and its 128 bytes of weights are copied once per tile into shared memory, laid out [tap row][thread] so
// that a warp reads 512 contiguous bytes per tap row (straight from the table every lane would touch its own cache
// line: 32 tag look-ups per load).  The 8 tap rows are 28-byte windows of the staged rectangle.  ~300 instructions
// and ~120 shared-memory wavefronts per pixel step.
struct Lanczos4 {
    static constexpr int kPx = 1, kTileH = 8, kLo = 3, kHi = 4, kRowsMin = 16, kInterp = VR180_INTER_LANCZOS4;
    static constexpr bool kRowPatch = true;  // a warp = one output row of the tile
    static constexpr int kShift = kInterBits;  // coordinates are 1/32-pixel fixed point: sx = cvRound(x * 32)
    __device__ static __forceinline__ int quant(float m) { return quantise(m); }
    static constexpr int kStageArea = 16384, kWeightSmem = kSamplers * 128;  // 16 KB of stages + 32 KB of weights
    static constexpr int kOutTiles = 4;
    struct Pixel {
        int boff;        // byte offset (4-aligned) of the 28-byte window of tap row 0 (iy - 3), first tap ix - 3
        int sh;
        const short* w;  // itab[ay][ax][ky][kx], 64 int16 in the table (device memory)
        uint32_t ws;     // shared-window address of the thread's staged copy of them ([tap row][thread] x 16 bytes), 0 = none
    };
    __device__ static __forceinline__ void set_offset(Pixel& p, int off, bool valid) {
        p.boff = valid ? (off & ~3) : 0;
        p.sh = (off & 3) * 8;
    }
    __device__ static __forceinline__ void weights(Pixel& p, int ax, int ay, const short* tab) {
        p.w = tab + (((ay << 5) | ax) << 6);
        p.ws = 0;
    }
    // NF frames of an item at once: a tap row's weights are loaded once and applied to every frame
    template <int NF>
    __device__ static __forceinline__ void sample_frames(uint32_t sbuf, uint32_t frame_bytes, const Pixel& p, uint32_t pitch,
                                                         uint32_t (&out)[NF]) {
        const uint8_t* base = static_cast<const uint8_t*>(__cvta_shared_to_generic(sbuf)) + p.boff;
        const int sh = p.sh;
        uint32_t acc[NF][3];
#pragma unroll
        for (int f = 0; f < NF; ++f) acc[f][0] = acc[f][1] = acc[f][2] = 16384u;  // + 1 << 14 before the >> 15
#pragma unroll
        for (int ky = 0; ky < 8; ++ky) {
            uint4 wv;
            if (p.ws) {
                asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];"
                             : "=r"(wv.x), "=r"(wv.y), "=r"(wv.z), "=r"(wv.w)
                             : "r"(p.ws + ky * (kSamplers * 16)));
            } else {
                wv = __ldg(reinterpret_cast<const uint4*>(p.w + ky * 8));
            }
            const uint32_t wp[4] = {wv.x, wv.y, wv.z, wv.w};  // {kx 0, 1} {2, 3} {4, 5} {6, 7}
#pragma unroll
            for (int f = 0; f < NF; ++f) {
                const uint32_t* r = reinterpret_cast<const uint32_t*>(base + f * frame_bytes + ky * pitch);
                uint32_t x[7], A[6];
#pragma unroll
                for (int i = 0; i < 7; ++i) x[i] = r[i];
#pragma unroll
                for (int i = 0; i < 6; ++i) A[i] = __funnelshift_r(x[i], x[i + 1], sh);  // 24 tap bytes, byte-aligned
#pragma unroll
                for (int g = 0; g < 2; ++g) {  // taps 4 g .. 4 g + 3 = the 12 bytes of A[3 g .. 3 g + 2]
                    const uint32_t A0 = A[3 * g], A1 = A[3 * g + 1], A2 = A[3 * g + 2];
                    const uint32_t q0 = __byte_perm(__byte_perm(A0, A1, 0x0630), A2, 0x5210);  // [t0c0 t1c0 t2c0 t3c0]
                    const uint32_t q1 = __byte_perm(__byte_perm(A0, A1, 0x0741), A2, 0x6210);  // [t0c1 t1c1 t2c1 t3c1]
                    const uint32_t q2 = __byte_perm(__byte_perm(A0, A1, 0x0052), A2, 0x7410);  // [t0c2 t1c2 t2c2 t3c2]
                    acc[f][0] = dp2a_hi_su(wp[2 * g + 1], q0, dp2a_lo_su(wp[2 * g], q0, acc[f][0]));
                    acc[f][1] = dp2a_hi_su(wp[2 * g + 1], q1, dp2a_lo_su(wp[2 * g], q1, acc[f][1]));
                    acc[f][2] = dp2a_hi_su(wp[2 * g + 1], q2, dp2a_lo_su(wp[2 * g], q2, acc[f][2]));
                }
            }
        }
#pragma unroll
        for (int f = 0; f < NF; ++f) {
            out[f] = pack_sat_u8x3((int)acc[f][0] >> 15, (int)acc[f][1] >> 15, (int)acc[f][2] >> 15);
        }
    }
    __device__ static __forceinline__ uint32_t sample(uint32_t sbuf, const Pixel& p, uint32_t pitch) {
        uint32_t out[1];
        sample_frames<1>(sbuf, 0u, p, pitch, out);
        return out[0];
    }
};

// Per-frame radius (vr180_mapsrc_t::radius_dev): the chain is evaluated WITHOUT its final DenormalizeTransformer
// once per tile; frame f then only applies  x = nx * radius[f] + cx  (transformer.py:202-203), rounds to float32
// and quantises.  That composition is monotone in nx, so the integer bounding box of a tile in frame f follows
// from the tile's extreme normalised coordinates.
struct DynRadius {
    const double* radius;  // device, one per frame; nullptr = radius baked into the chain
    double cx, cy;         // centre of the final DenormalizeTransformer
    double ext[4];         // tile extremes: nx min, nx max, ny min, ny max
};
template <class M>
__device__ __forceinline__ int denorm_q(double n, double rad, double c) {  // astype(float32), the mode's cvRound
    return M::quant(__double2float_rn(add_rn(mul_rn(n, rad), c)));
}
// integer pixel range [lo, hi] of the taps' base coordinate over the tile for one frame
template <class M>
__device__ __forceinline__ void dyn_range(double nmin, double nmax, double rad, double c, int& lo, int& hi) {
    const int a = sat16(denorm_q<M>(nmin, rad, c) >> M::kShift), b = sat16(denorm_q<M>(nmax, rad, c) >> M::kShift);
    lo = min(a, b);
    hi = max(a, b);
}

// ---- tile geometry: one definition for k_warp_tiled, k_pack_tiles (which stores it in the tile header) and
// k_warp_stream (which reads it back) ---------------------------------------------------------------------------
// Block-wide integer bounding box {min ix, max ix, min iy, max iy} of the sampling warps' pixels, in two halves around
// a barrier of the caller: every warp reduces its own box and lane 0 of a sampling warp stores it as record `warp`;
// after the barrier lane w reads record w -- one 128-bit load + four REDUX (a loop over the 8 records is 64
// instructions per thread, and a one-frame tile has few to amortise them over).
template <class M>
__device__ __forceinline__ void block_box_store(const int (&sx)[M::kPx], const int (&sy)[M::kPx], int4* s_red, int warp,
                                                bool store) {
    int mnx = INT_MAX, mxx = INT_MIN, mny = INT_MAX, mxy = INT_MIN;
#pragma unroll
    for (int k = 0; k < M::kPx; ++k) {
        const int ix = sat16(sx[k] >> M::kShift), iy = sat16(sy[k] >> M::kShift);
        mnx = min(mnx, ix);
        mxx = max(mxx, ix);
        mny = min(mny, iy);
        mxy = max(mxy, iy);
    }
    mnx = __reduce_min_sync(0xffffffffu, mnx);
    mxx = __reduce_max_sync(0xffffffffu, mxx);
    mny = __reduce_min_sync(0xffffffffu, mny);
    mxy = __reduce_max_sync(0xffffffffu, mxy);
    if (store) s_red[warp] = make_int4(mnx, mxx, mny, mxy);
}
__device__ __forceinline__ int4 block_box_load(const int4* s_red, int lane) {
    int4 r = make_int4(INT_MAX, INT_MIN, INT_MAX, INT_MIN);
    if (lane < kSamplers / 32) r = s_red[lane];
    r.x = __reduce_min_sync(0xffffffffu, r.x);
    r.y = __reduce_max_sync(0xffffffffu, r.y);
    r.z = __reduce_min_sync(0xffffffffu, r.z);
    r.w = __reduce_max_sync(0xffffffffu, r.w);
    return r;
}

// TMA box rows for a rectangle of `nrows` source rows: M::kRowsMin + kRowsStep * rsel (rsel < kRowSizes to fit a box)
template <class M>
__device__ __forceinline__ int box_rsel(int nrows) {
    return nrows <= M::kRowsMin ? 0 : (nrows - M::kRowsMin + kRowsStep - 1) / kRowsStep;
}
// Source rectangle of a tile from the extreme integer coordinates of its pixels: the taps cover columns
// ix - kLo .. ix + kHi and rows iy - kLo .. iy + kHi; columns in 16-byte granules (a TMA box starts 16-byte aligned)
struct TileRect {
    int bx0, wbytes;         // first source byte column (may be negative) and width in bytes
    int ry0, nrows;          // first source row and row count
    int rsel, box_rows;      // TMA box rows = M::kRowsMin + kRowsStep * rsel
};
template <class M>
__device__ __forceinline__ TileRect tile_rect(int mnx, int mxx, int mny, int mxy) {
    TileRect r;
    r.bx0 = (3 * (mnx - M::kLo)) & ~15;
    r.wbytes = ((3 * (mxx + M::kHi + 1) + 15) & ~15) - r.bx0;
    r.ry0 = mny - M::kLo;
    r.nrows = mxy + M::kHi + 1 - r.ry0;
    r.rsel = box_rsel<M>(r.nrows);
    r.box_rows = M::kRowsMin + r.rsel * kRowsStep;
    return r;
}

// Row pitch of the staged rectangle (= TMA box width).  Candidates: the kPitchCands widths pitch0 + kPitchStep e.
// Cost of a candidate in shared-memory wavefronts per (frame, eye) item: the tap loads (every sampling warp measures
// the wavefronts = max distinct words per bank, counted with match.any, of the first tap load of its step k = 0; a
// tile has kStepsPerWarp steps of kLoads loads with the same address pattern) + the TMA write of the box (64 bytes per
// wavefront, measured).  pitch_costs: one sampling warp's share, added into s_cost[kPitchCands] (zeroed by the
// caller); pick_pitch, after a barrier: the cheapest candidate that is <= kPitchMax and that `fits` admits.
template <class M>
__device__ __forceinline__ void pitch_costs(int sx0, int sy0, const TileRect& rc, int pitch0, int lane, int* s_cost) {
    const int row = (sy0 >> M::kShift) - M::kLo - rc.ry0, col = 3 * ((sx0 >> M::kShift) - M::kLo) - rc.bx0;
    int cost = 0;
#pragma unroll
    for (int e = 0; e < kPitchCands; ++e) {
        const int w = (row * (pitch0 + kPitchStep * e) + col) >> 2;
        const unsigned same = __match_any_sync(0xffffffffu, w);
        const bool leader = (__ffs(same) - 1) == lane;  // one lane per distinct word
        const unsigned lm = __ballot_sync(0xffffffffu, leader);
        int deg = 0;
        if (leader) deg = __popc(__match_any_sync(lm, w & 31));
        deg = __reduce_max_sync(0xffffffffu, deg);
        if (lane == e) cost = deg;
    }
    constexpr int kStepsPerWarp = M::kTileH * kTileW / kSamplers;  // warp steps (32 pixels) of a tile, per warp
    constexpr int kLoads = M::kInterp == VR180_INTER_NEAREST ? 2 : M::kInterp == VR180_INTER_LINEAR ? 6
                         : M::kInterp == VR180_INTER_CUBIC ? 16 : 56;
    if (lane < kPitchCands) atomicAdd(&s_cost[lane], cost * (kStepsPerWarp * kLoads));
}
template <class Fits>
__device__ __forceinline__ int pick_pitch(const int* s_cost, int pitch0, int box_rows, Fits fits) {
    int best = 0, best_cost = INT_MAX;
#pragma unroll
    for (int e = 0; e < kPitchCands; ++e) {
        const int pe = pitch0 + kPitchStep * e;
        const int c = s_cost[e] + box_rows * pe / 64;
        if (pe <= kPitchMax && fits(pe) && c < best_cost) { best_cost = c; best = e; }
    }
    return pitch0 + kPitchStep * best;
}

// Per-pixel gather from global memory with full border handling (the tiles that are not staged): one output pixel
// (i, j) of frame f for the views v_begin .. v_end - 1, which share the quantised coordinates (qx, qy).
template <class M>
__device__ __forceinline__ void gather_pixel(const RemapArgs& a, int f, int i, int j, int v_begin, int v_end, int qx, int qy,
                                             const short* tab) {
    uint8_t* drow = a.dst + (long long)f * a.dst_frame_stride + (long long)j * a.dst_pitch;
    for (int v = v_begin; v < v_end; ++v) {
        const ViewArgs& vw = a.view[v];
        Src s{vw.src + (long long)f * vw.frame_stride, vw.rows, vw.cols, vw.pitch};
        int px[3];
        if (M::kInterp == VR180_INTER_NEAREST)
            fetch_tap<3>(s, sat16(qx), sat16(qy), a.border_mode, a.bv, px);
        else if (M::kInterp == VR180_INTER_LINEAR)
            sample_linear<3>(s, qx, qy, a.border_mode, a.bv, px);
        else if (M::kInterp == VR180_INTER_CUBIC)
            sample_tab<3, 4>(s, qx, qy, tab, a.border_mode, a.bv, px);
        else
            sample_tab<3, 8>(s, qx, qy, tab, a.border_mode, a.bv, px);
        uint8_t* o = drow + (long long)(vw.dst_x_offset + i) * 3;
        o[0] = (uint8_t)px[0];
        o[1] = (uint8_t)px[1];
        o[2] = (uint8_t)px[2];
    }
}

// the FR frames of an item for one pixel; only modes with per-row state worth sharing implement sample_frames
template <class M, int FR>
__device__ __forceinline__ void sample_item(uint32_t sbuf, uint32_t frame_bytes, const typename M::Pixel& p, uint32_t pitch,
                                            uint32_t (&out)[FR]) {
    if constexpr (M::kInterp == VR180_INTER_LANCZOS4) {
        M::template sample_frames<FR>(sbuf, frame_bytes, p, pitch, out);
    } else {
#pragma unroll
        for (int f = 0; f < FR; ++f) out[f] = M::sample(sbuf + f * frame_bytes, p, pitch);
    }
}

// ---- host ----------------------------------------------------------------------------------------------------
// BORDER_CONSTANT with a zero colour: TMA's out-of-bounds zero fill is the border
inline int zero_border(const RemapArgs& a) {
    return (a.border_mode == VR180_BORDER_CONSTANT && !(a.bv[0] | a.bv[1] | a.bv[2])) ? 1 : 0;
}
// The kernel's dynamic shared-memory limit, raised once per device; `dev` = the current device
template <auto Kernel>
int max_dyn_smem_once(int bytes, int& dev) {
    static std::atomic<int> done[64];
    dev = 0;
    VR180_CUDA(cudaGetDevice(&dev));
    if (dev < 64 && !done[dev].load(std::memory_order_acquire)) {
        VR180_CUDA(cudaFuncSetAttribute(Kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
        done[dev].store(1, std::memory_order_release);
    }
    return VR180_OK;
}

}  // namespace tiled

// tiled.cu
const tiled::TmaMaps* tma_maps_for(const RemapArgs& a0, int interp, int rows_min, int tile_h, int fr);
int tiled_debug_flags();
// stream.cu: tiles streamed through persistent CTAs (tile-packed LUT, a few frames per launch);
// VR180_ERR_UNSUPPORTED = not eligible
int launch_remap_stream(const RemapArgs& a, int interp, const short* weight_tab, cudaStream_t st);
}  // namespace vr180
