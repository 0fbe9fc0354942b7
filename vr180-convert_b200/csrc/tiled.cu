// tiled.cu -- the tiled fast path of the fused warp: uint8 x 3 channels, INTER_LINEAR or INTER_CUBIC,
// BORDER_CONSTANT (0).
//
// Replaces cv.remap per eye + np.concatenate (/root/reference/src/vr180_convert/remapper.py:388-398, :518) and,
// for MAPSRC_ANALYTIC, get_map (remapper.py:23-59) for a batch of frames that share their maps (the reference's
// apply(): ONE map, N images, remapper.py:381-398).
//
// One CTA owns a tile of one eye's output (32 x 32 bilinear, 32 x 16 bicubic; of both eyes when they share a map)
// for every frame of its frame chunk:
//   prologue   coordinates of the tile's pixels, once: analytic chain in float64 (row / column sincos of the
//              Normalize + EquirectangularEncoder prefix are separable and computed 64x per tile instead of
//              2048x; the standard chain shape runs in the folded form of chain_fast.cuh, anything else through
//              the op interpreter of chain.cuh), or float32 maps, or the fixed-point LUT; quantised exactly like
//              cv::remap (sampler.cuh); per pixel only {smem offset of the first tap, byte shift, packed integer
//              weights} stay in registers.
//   bbox       block-wide min / max of the integer source coordinates -> the tile's source rectangle.
//   pitch      the row pitch of the staged rectangle = the TMA box width, a multiple of 16 bytes, is picked per
//              tile from the 4 tightest widths: every sampling warp counts the bank conflicts of its own tap
//              addresses under each candidate (match.any: wavefronts of a load = max distinct words per bank)
//              and the cheapest candidate in shared-memory wavefronts (tap loads + TMA write of the box) wins.
//   pipeline   an item = 2 consecutive frames of one eye (1 with a per-frame radius).  Its source rectangles are
//              fetched by ONE TMA box load (cp.async.bulk.tensor.3d over the (bytes, rows, frames) view of the
//              source batch, box depth 2, completion on an mbarrier) into a ring of stages sized for this tile;
//              a dedicated producer warp runs the loads S - 1 items ahead.  TMA's out-of-bounds zero fill IS
//              BORDER_CONSTANT(0), so tiles that straddle the source edge stay on the fast path.  No LSU
//              instruction touches the source in global memory.  (A TMA box must start at a 16-byte aligned
//              global address -- B200 traps with "illegal instruction" otherwise, for loads and stores.)
//   sampling   bilinear: a warp step = 32 pixels of one output row: their taps are ~26 consecutive source pixels,
//              i.e. ~20 consecutive words, one wavefront per load while the row stays inside one source row.
//              6 LDS.32 per pixel (2 rows x 12 bytes, the third word only for a byte offset of 3), funnel shifts
//              to byte-align, PRMT to pair the taps, 2 x dp2a (16-bit weight x 8-bit pixel) per channel:
//              (sum_t w_t p_t + 512) >> 10  ==  (sum_t 64 w_t p_t + 32768) >> 16, i.e. byte 2 of the dp2a chain.
//              Bicubic: a warp step = an 8 x 4 patch; 4 rows x 16-byte windows, the pixel's 16 int16 table
//              weights (OpenCV's 1024 x 16 table, tables.cuh) live in 8 registers, 2 x dp2a (s16 x u8) per
//              channel and row, clip((acc + 16384) >> 15).
//   store      the 3-byte results of a step are re-packed with ONE shuffle (every lane fetches the pixel of
//              lane + 1; lanes 4 m + i, i < 3, then hold word 3 m + i of the row segment) into a dense output
//              tile in shared memory; the producer writes the item's tiles into the eye's half of the SBS frames
//              with one TMA store (full 32-byte sectors, no STG) and hands the buffer back once it has been read.
// Tiles whose footprint is unbounded (NaN / huge coordinates) or exceeds the staging buffer, and partial edge
// tiles, take the per-pixel global-memory gather of sampler.cuh inside the same kernel.
//
// Measured dead ends (profiles/README.md): re-packing the staged rectangle into 4-byte pixels in shared memory
// (the conversion costs as many wavefronts as the whole-word taps save), 3 CTAs per SM with 72 registers, 8 pitch
// candidates, sampling warps storing straight to global memory (STG) instead of the TMA tile store.
#include "tiled.cuh"

namespace vr180 {
namespace tiled {

struct TileGeom {
    int rsel;           // TMA box rows of the tile's rectangle: M::kRowsMin + kRowsStep * rsel
    int bx0, ry0;       // first source byte column (16-aligned, may be negative) and first source row
    int x0, y0;         // output tile origin
};

// The frame loop of one tile.  Items are (FR consecutive frames, view) in frame-major order.  NV = views sampled
// with this CTA's coordinates (2 when both eyes share the map).
//
// Warp-specialised: warps 0-7 sample, lane 0 of warp 8 drives the TMA unit and nothing else, so no sampling warp
// ever blocks on a copy.  TMA work is kept to TWO operations per item (one load box = the source rectangles of
// the item's frames, one store box = their output tiles): a version with 5 load boxes + 8 per-warp store boxes
// per item measured TMA-issue bound (~50 clk per operation, profiles/r1_v7_*).  With FR = 2 the per-item
// bookkeeping (barrier waits, ring counters, proxy fence, arrive: ~45 instructions per warp) is paid once per 8
// pixels of a thread instead of once per 4.
//
// The staging area is a ring of S stages of exactly the tile's footprint (FR x box rows x pitch bytes), so a
// typical bilinear tile (2 x 36 rows x 128 B = 9.2 KB) gets S = 4 and the loads run up to S - 1 items ahead.
// No CTA-wide barrier; three kinds of mbarrier:
//   full[s]    (1 + tx bytes)  the box of the item in stage s has landed; the sampling warps wait on it
//   ofull[o]   (8)             one arrive per sampling warp when its rows of the item's tiles are in out buffer o
//                              (OB = 4 / FR deep) -- which also says the warp has left the item's stage; the
//                              producer waits, issues the TMA store and re-fills the stage with item n + S
//   oempty[o]  (1)             the producer arrives as soon as the store that used out buffer o has finished
//                              reading it (bulk wait_group.read); the sampling warps wait before rewriting it
//                              (item n - OB), so a warp can run at most OB items ahead of the slowest one
// SPLIT: the descriptors' boxes are ONE frame deep (a launch with per-frame radii needs those for its mixed chunks), so
// an FR-frame item of an equal-radii chunk is fetched and stored as FR boxes on the same barrier / in the same bulk group.
// VPAIR (with SPLIT, FR == 2, NV == 2): the item's two rectangles are the two EYES of one frame instead of two frames of
// one eye -- for launches whose CTAs get a single frame (one stereo pair per call): one barrier round per frame, and
// per-row state (Lanczos4's weights) serves both eyes.
template <class M, int NV, bool DYN, int FR, bool SPLIT = false, bool VPAIR = false>  // FR: frames per item (2: one box load / tile store / barrier round per 2 frames)
__device__ __forceinline__ void frame_loop(const RemapArgs& a, const TmaMaps& tm, int v_begin, int f0, int f1,
                                           const typename M::Pixel (&pc)[M::kPx], const TileGeom& tg, const int pitch,
                                           uint8_t* smem, int band, int cg, const DynRadius& dr,
                                           const double (&nx)[M::kPx], const double (&ny)[M::kPx], const short* tab) {
    static_assert(FR == 1 || !DYN, "a per-frame radius gives every frame its own rectangle");
    static_assert(M::kOutTiles / FR >= 2, "at least two out buffers of one item each");
    constexpr int kOutTileBytes = M::kTileH * kTileW * 3;
    constexpr int kOutItemBytes = FR * kOutTileBytes;
    constexpr int OB = M::kOutTiles / FR < kOutBufs ? M::kOutTiles / FR : kOutBufs;  // out buffers of one item each
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    uint32_t s_stage = smem_u32(smem);
    asm volatile("" : "+r"(s_stage));  // opaque: otherwise the window base is re-derived (S2R SR_CgaCtaId + MOV + LEA) in every item
    const uint32_t s_full = s_stage + Lay<M>::kOffBar;
    const uint32_t s_ofull = s_full + 2 * kMaxStages * 8, s_oempty = s_ofull + kOutBufs * 8, s_out = s_stage + Lay<M>::kOffOut;

    int2* const s_org = reinterpret_cast<int2*>(smem + Lay<M>::kOffOrg);
    // item n = FR consecutive frames of one view; a chunk with an odd frame count ends with a phantom frame: the
    // host keeps chunks even, so it lies past the end of the batch, where TMA loads zeros and drops the store
    static_assert(!VPAIR || (SPLIT && FR == 2 && NV == 2 && !DYN), "an eye pair is two one-frame boxes of two views");
    const int n_items = VPAIR ? (f1 - f0) : ((f1 - f0 + FR - 1) / FR) * NV;
    const int rect_bytes = (M::kRowsMin + tg.rsel * kRowsStep) * pitch;  // one frame's box; multiple of 64
    const int stage_bytes = FR * rect_bytes;                          // bytes the box load(s) of an item deliver
    // distance of an item's frames inside a stage: packed by a box FR frames deep; one-frame boxes land 128-byte aligned
    const int frame_pitch = SPLIT ? (rect_bytes + 127) & ~127 : rect_bytes;
    const int stage_stride = (FR * frame_pitch + 127) & ~127;         // TMA destinations are 128-byte aligned
    // stages that fit the staging area: both are multiples of 128 bytes, and the +0.5 keeps the approximate float quotient
    // of the two small integers on the right side of every integer (an integer division is ~20 instructions)
    static_assert(Lay<M>::kStageArea % 128 == 0 && Lay<M>::kStageArea / 128 <= 1024, "float quotient below");
    const int S = min(kMaxStages, (int)__fdividef((float)(Lay<M>::kStageArea / 128) + 0.5f, (float)(stage_stride >> 7)));

    if (warp == kSamplers / 32) {  // ---- producer ----
        if (lane != 0) return;
        const CUtensorMap* const map0 = &tm.src[v_begin][(pitch - kPitchMin) / kPitchStep][tg.rsel];
        const int dst_x0 = (a.view[v_begin].dst_x_offset + tg.x0) * 3;
        const int dst_x1 = (a.view[v_begin + NV - 1].dst_x_offset + tg.x0) * 3;
        int p_item = 0, p_stage = 0;  // next item to fetch and its stage
        auto load = [&]() {
            const uint32_t bar = s_full + p_stage * 8;
            const int v = (NV == 2 && !VPAIR) ? (p_item & 1) : 0;
            const int f = VPAIR ? f0 + p_item : f0 + FR * ((NV == 2) ? (p_item >> 1) : p_item);
            int bx0 = tg.bx0, ry0 = tg.ry0;
            if (DYN) {  // this frame's rectangle; its origin travels to the samplers next to the stage
                const double rad = __ldg(dr.radius + f);
                if (rad == rad) {
                    int xlo, xhi, ylo, yhi;
                    dyn_range<M>(dr.ext[0], dr.ext[1], rad, dr.cx, xlo, xhi);
                    dyn_range<M>(dr.ext[2], dr.ext[3], rad, dr.cy, ylo, yhi);
                    const TileRect rc = tile_rect<M>(xlo, xhi, ylo, yhi);
                    bx0 = rc.bx0;
                    ry0 = rc.ry0;
                } else {  // get_radius found no transition: every coordinate is NaN -> border colour
                    bx0 = ry0 = -(1 << 20);
                }
                s_org[p_stage] = make_int2(bx0, ry0);  // released to the samplers by the arrive below
            }
            mbar_expect_tx(bar, (uint32_t)stage_bytes);
            if (SPLIT) {
#pragma unroll
                for (int fr = 0; fr < FR; ++fr)  // a frame past the batch is all zero fill, and still rect_bytes on the barrier
                    tma_load_3d(s_stage + p_stage * stage_stride + fr * frame_pitch,
                                map0 + (VPAIR ? fr : v) * (kWidths * kRowSizes), bx0, ry0, VPAIR ? f : f + fr, bar);
            } else {
                tma_load_3d(s_stage + p_stage * stage_stride, map0 + v * (kWidths * kRowSizes), bx0, ry0, f, bar);
            }
            ++p_item;
            if (++p_stage == S) p_stage = 0;
        };
        for (int n = 0; n < S && n < n_items; ++n) load();  // fill the ring
        for (int n = 0; n < n_items; ++n) {
            const int o = n & (OB - 1);
            const int v = (NV == 2 && !VPAIR) ? (n & 1) : 0;
            const int f = VPAIR ? f0 + n : f0 + FR * ((NV == 2) ? (n >> 1) : n);
            mbar_wait(s_ofull + o * 8, (uint32_t)(n / OB) & 1u);  // every sampling warp has written item n
            if (n + S < n_items) load();  // ofull(n) also means: every warp has left the stage of item n -> re-fill it
            if (SPLIT) {
#pragma unroll
                for (int fr = 0; fr < FR; ++fr)
                    tma_store_3d(&tm.dst, (VPAIR ? fr : v) ? dst_x1 : dst_x0, tg.y0, VPAIR ? f : f + fr,
                                 s_out + o * kOutItemBytes + fr * kOutTileBytes);
            } else {
                tma_store_3d(&tm.dst, v ? dst_x1 : dst_x0, tg.y0, f, s_out + o * kOutItemBytes);
            }
            bulk_commit();
            // hand the out buffer back as soon as the store has read it (the next ofull is an item time away, so
            // the producer has nothing else to do): a sampling warp may then run OB items ahead of the slowest one
            bulk_wait_read<0>();
            mbar_arrive(s_oempty + o * 8);
        }
        bulk_wait_read<0>();  // shared memory must stay valid until the last store has read it
        return;
    }

    // ---- sampling warps ----
    // The 3-byte results [c0 c1 c2 .] of a warp step are re-packed into words of the dense out tile with ONE
    // shuffle: every lane fetches the pixel of lane + 1; lanes 4 m + i, i < 3, then hold word 3 m + i of the row
    // segment (12 bytes of 4 pixels = 3 words): [c0 c1 c2 c0'], [c1 c2 c0' c1'], [c2 c0' c1' c2'].
    const int sub = lane & 3;
    const uint32_t out_sel = sub == 0 ? 0x4210u : (sub == 1 ? 0x5421u : 0x6542u);
    const bool writer = sub != 3;
    // this lane's word of step k inside the dense out tile
    //   row patch: row 4 band + k, word 3 (lane >> 2) + sub
    //   8 x 4 patch: row 4 band + (lane >> 3), byte 24 (kPx cg + k), word 3 ((lane & 7) >> 2) + sub
    constexpr int kOutStep = M::kRowPatch ? kTileW * 3 : 24;
    const int sw = band * (4 / M::kPx) + cg;  // sampling warp index; with row patches it owns rows kPx sw .. kPx sw + kPx - 1
    uint32_t outp = s_out + (M::kRowPatch ? (M::kPx * sw) * (kTileW * 3) + (3 * (lane >> 2) + sub) * 4
                                          : (4 * band + (lane >> 3)) * (kTileW * 3) + M::kPx * cg * 24 +
                                                (3 * ((lane & 7) >> 2) + sub) * 4);
    uint32_t flags = (writer ? 1u : 0u) | (lane == 0 ? 2u : 0u);
    // opaque to the compiler: otherwise it re-derives them from S2R SR_TID.X inside the frame loop
    asm volatile("" : "+r"(outp), "+r"(flags));

    int st = 0;
    uint32_t ph = 0;
    typename M::Pixel cur[M::kPx];  // DYN: constants of the current radius
    double cur_rad = CUDART_NAN;
    bool cur_have = false;
#pragma unroll
    for (int k = 0; k < M::kPx; ++k) cur[k] = pc[k];
    for (int n = 0; n < n_items; ++n) {
        mbar_wait(s_full + st * 8, ph);
        const uint32_t buf = s_stage + st * stage_stride;
        uint32_t res[FR][M::kPx];
        if (DYN) {
            // The per-pixel constants depend on the frame only through its radius: they are rebuilt when the radius
            // changes (a static rig gives runs of equal radii; both eyes of a frame always share it).
            const int f = f0 + ((NV == 2) ? (n >> 1) : n);  // FR == 1
            const double rad = __ldg(dr.radius + f);
            if (!(rad == cur_rad)) {
                const int2 org = s_org[st];
                cur_have = rad == rad;
#pragma unroll
                for (int k = 0; k < M::kPx; ++k) {
                    const int qx = denorm_q<M>(nx[k], rad, dr.cx), qy = denorm_q<M>(ny[k], rad, dr.cy);
                    const int off = ((qy >> M::kShift) - M::kLo - org.y) * pitch + 3 * ((qx >> M::kShift) - M::kLo) - org.x;
                    M::set_offset(cur[k], off, cur_have);
                    M::weights(cur[k], qx & 31, qy & 31, tab);
                }
                cur_rad = rad;
            }
#pragma unroll
            for (int k = 0; k < M::kPx; ++k) {
                const uint32_t r = M::sample(buf, cur[k], (uint32_t)pitch);
                res[0][k] = cur_have ? r : 0u;  // NaN radius (no transition found): border colour
            }
        }
        uint32_t word[FR][M::kPx];
        if (!DYN && M::kInterp == VR180_INTER_LANCZOS4) {  // a tap row's weights serve every frame of the item
#pragma unroll
            for (int k = 0; k < M::kPx; ++k) {
                uint32_t r[FR];
                sample_item<M, FR>(buf, (uint32_t)frame_pitch, pc[k], (uint32_t)pitch, r);
#pragma unroll
                for (int fr = 0; fr < FR; ++fr) res[fr][k] = r[fr];
            }
        }
#pragma unroll
        for (int fr = 0; fr < FR; ++fr) {
            if (!DYN && M::kInterp != VR180_INTER_LANCZOS4) {
#pragma unroll
                for (int k = 0; k < M::kPx; ++k) res[fr][k] = M::sample(buf + fr * frame_pitch, pc[k], (uint32_t)pitch);
            }
            // re-pack frame fr right away: its shuffles are in flight while the next frame is sampled
#pragma unroll
            for (int k = 0; k < M::kPx; ++k)
                word[fr][k] = __byte_perm(res[fr][k], __shfl_down_sync(0xffffffffu, res[fr][k], 1), out_sel);
        }
        const int o = n & (OB - 1);
        if (n >= OB) mbar_wait(s_oempty + o * 8, (uint32_t)(n / OB + 1) & 1u);  // store n - OB has read out[o]
        if (flags & 1u) {
            const uint32_t ob = outp + o * kOutItemBytes;
#pragma unroll
            for (int fr = 0; fr < FR; ++fr)
#pragma unroll
                for (int k = 0; k < M::kPx; ++k) sts32(ob + fr * kOutTileBytes + k * kOutStep, word[fr][k]);
        }
        fence_proxy_async();
        __syncwarp();
        if (flags & 2u) mbar_arrive(s_ofull + o * 8);  // this warp's rows of item n are in out[o]; it has left stage st
        if (++st == S) { st = 0; ph ^= 1u; }
    }
}

// DYN: per-frame radius from device memory (vr180_mapsrc_t::radius_dev); FR: frames per pipeline item.  4 CTAs per SM
// (56 registers).
template <class M, bool DYN, int FR>
__global__ void __launch_bounds__(kThreads, 4)
k_warp_tiled(const __grid_constant__ RemapArgs a, const __grid_constant__ vr180_chain_t chain0,
             const __grid_constant__ vr180_chain_t chain1, const __grid_constant__ TiledParams tp,
             const __grid_constant__ TmaMaps tm) {
    constexpr int kPx = M::kPx;
    constexpr int kChainUnroll = (FR == 1 && !DYN) ? kPx : 1;  // pixels of a thread whose chains are interleaved
    constexpr int kWarpsPerBand = 4 / kPx;  // a band = 4 output rows x 32 columns = 4 / kPx warps of 8 kPx columns
    extern __shared__ __align__(1024) uint8_t smem[];
    double* s_trig = reinterpret_cast<double*>(smem + Lay<M>::kOffTrig);  // [4][32]
    int4* s_red = reinterpret_cast<int4*>(smem + Lay<M>::kOffRed);        // [8]: box of each sampling warp

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    if (tid < 2 * kMaxStages + 2 * kOutBufs) {  // one barrier per thread: a single-frame launch is latency bound, and one
        const uint32_t bars = smem_u32(smem + Lay<M>::kOffBar);  // thread initialising all 24 kept the whole CTA waiting
        // layout: full[kMaxStages] (1: the producer + tx bytes), empty[kMaxStages] (one arrive per sampling warp),
        //         ofull[kOutBufs] (one arrive per sampling warp), oempty[kOutBufs] (1: the producer)
        const bool by_warps = (tid >= kMaxStages && tid < 2 * kMaxStages + kOutBufs);
        mbar_init(bars + tid * 8, by_warps ? kSamplers / 32 : 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");  // visible to the async proxy (TMA)
    }
    int* const s_cost = reinterpret_cast<int*>(smem + Lay<M>::kOffCost);  // wavefront cost of each candidate pitch
    if (tid < kPitchCands) s_cost[tid] = 0;
    // grid = (tiles_x, tiles_y, map groups x frame chunks): no division by a runtime tile count in a CTA that may live for
    // one frame only
    const int tx = blockIdx.x, ty = blockIdx.y, tile = ty * tp.tiles_x + tx;  // tile: index into a tile-packed LUT
    const int x0 = tx * kTileW, y0 = ty * M::kTileH;
    const bool two_groups = !a.share_map && a.n_views == 2;
    const int g = two_groups ? (int)(blockIdx.z & 1u) : 0;  // map group: the view whose coordinates drive this CTA
    const int chunk = two_groups ? (int)(blockIdx.z >> 1) : (int)blockIdx.z;
    const ViewArgs& mv = a.view[g];
    const int v_begin = g, v_end = a.share_map ? a.n_views : g + 1, nv = v_end - v_begin;
    const int f0 = chunk * a.frames_per_cta, f1 = min(a.n_frames, f0 + a.frames_per_cta);
    const bool sampler = warp < kSamplers / 32;  // the last warp = TMA producer: no pixels of its own
    const int sw = warp & (kSamplers / 32 - 1), band = sw / kWarpsPerBand, cg = sw % kWarpsPerBand;
    // pixel k of this thread (tile-local): 8 x 4 patches: column lx + 8 k, row ly; row patches: column lane, row 4 band + k
    const int lx = M::kRowPatch ? lane : 8 * kPx * cg + (lane & 7), ly = M::kRowPatch ? kPx * sw : 4 * band + (lane >> 3);
    auto pcol = [&](int k) { return M::kRowPatch ? lx : lx + 8 * k; };
    auto prow = [&](int k) { return M::kRowPatch ? ly + k : ly; };
    const bool full_tile = (x0 + kTileW <= a.W) && (y0 + M::kTileH <= a.H);

    // tile-packed LUT: the tile's header (every thread: the producer warp needs the rectangle too)
    TileHdr hdr = {0, 0, 0, 0, 0};
    if (mv.map_kind != VR180_MAPSRC_ANALYTIC && mv.packed) hdr = decode_header(packed_header_raw(mv.packed, tile));
    const bool packed_tile = (hdr.flags & 1) != 0;  // CTA-uniform: coordinates and bounding box come from the packed LUT

    // ---- coordinates of this thread's pixels --------------------------------------------------------------
    int sx[kPx], sy[kPx];
    double nx[kPx], ny[kPx];  // dyn: coordinates before the final Denormalize
#pragma unroll
    for (int k = 0; k < kPx; ++k) {
        sx[k] = sy[k] = 0;
        nx[k] = ny[k] = 0.0;
    }
    constexpr bool dyn = DYN;  // host guarantees: DYN <=> every map group is ANALYTIC with a radius_dev
    if (mv.map_kind == VR180_MAPSRC_ANALYTIC) {
        const vr180_chain_t& ch = mv.chain_idx ? chain1 : chain0;
        const StdChain& sc = tp.std[mv.chain_idx ? 1 : 0];
        const bool fastc = sc.valid && sc.fast && !(tp.debug & 256);  // VR180_TILED_DEBUG bit 8: op-by-op evaluation (run_ops)
        if (sc.valid || tp.sep_prefix) {
            // Normalize + EquirectangularEncoder prefix (transformer.py:153-164, :545-566): the angle of a column
            // (row) depends on the column (row) only, so its sincos is evaluated once per tile column (row).
            if (tid < 64) {
                const bool is_row = tid >= 32;
                const int idx = tid & 31;
                const double* nm = ch.ops[0].p;
                const double c = (double)((is_row ? y0 : x0) + idx);
                const double n = mul_rn(__ddiv_rn(add_rn(c, -(is_row ? nm[1] : nm[0])), nm[2]), 2.0);
                double sv, cv;
                sincos(mul_rn(n, kHalfPi), &sv, &cv);
                if (fastc) {  // the rotation folded into per-column / per-row terms (chain_fast.cuh)
                    std_tables(sc.R, sc.lat_is_y != 0, is_row, sv, cv, s_trig, s_trig + 128, idx);
                } else {
                    s_trig[(is_row ? 64 : 0) + idx] = sv;
                    s_trig[(is_row ? 96 : 32) + idx] = cv;
                }
            }
            __syncthreads();
            const bool lat_is_y = ch.ops[1].iparam != 0;
            auto seed = [&](int k, ChainState& s) {
                const double s_row = s_trig[64 + prow(k)], c_row = s_trig[96 + prow(k)];
                const double s_col = s_trig[pcol(k)], c_col = s_trig[32 + pcol(k)];
                s.mode = MODE_VEC3;
                s.x = s.y = s.r = s.ux = s.uy = 0.0;
                if (lat_is_y) {  // lat from the row, lon from the column
                    s.vx = mul_rn(c_row, s_col);
                    s.vy = s_row;
                    s.vz = mul_rn(c_row, c_col);
                } else {  // lat from the column, lon from the row
                    s.vx = s_col;
                    s.vy = mul_rn(c_col, s_row);
                    s.vz = mul_rn(c_col, c_row);
                }
            };
            if (!sampler) {
            } else if (fastc) {  // the standard chain, folded (chain_fast.cuh)
                // instantiated once per chain so that the polynomial and the denormalisation are read with static
                // constant-bank operands (no indexed LDC, no register copies); one pixel at a time, not unrolled: a CTA
                // that serves one frame runs this exactly once, and instruction fetch is what such a launch waits for
                auto std_eval = [&](const StdChain& c) {
                    // v = scale A + B (chain_fast.cuh).  A thread's pixels share their column (row patches) or their row
                    // (8 x 4 patches): that side of the table is read once, the other per pixel -- these are 8-byte
                    // loads on the pipe that bounds the kernel
                    const bool x_fixed = M::kRowPatch ? !c.lat_is_y : (c.lat_is_y != 0);  // side X = rows iff lat_is_y
                    const int fi = M::kRowPatch ? lx : ly;
                    const double* const ft = s_trig + (x_fixed ? 0 : 128) + fi;
                    const double f0 = ft[0], f1 = ft[32], f2 = ft[64], f3 = x_fixed ? ft[96] : 0.0;
#pragma unroll(kChainUnroll)
                    for (int k = 0; k < kPx; ++k) {
                        const int vi = M::kRowPatch ? prow(k) : pcol(k);
                        double vx, vy, vz;
                        if (x_fixed) {  // (uniform)
                            vx = fma(f0, s_trig[128 + vi], f1); vy = fma(f0, s_trig[160 + vi], f2); vz = fma(f0, s_trig[192 + vi], f3);
                        } else {
                            const double sc_ = s_trig[vi];
                            vx = fma(sc_, f0, s_trig[32 + vi]); vy = fma(sc_, f1, s_trig[64 + vi]); vz = fma(sc_, f2, s_trig[96 + vi]);
                        }
                        double ox, oy;
                        int qx = 0, qy = 0;
                        if (dyn) {
                            std_pixel<true>(vx, vy, vz, c.poly, c.n_poly, c.den, ox, oy);
                        } else {
                            std_pixel<false>(vx, vy, vz, c.poly, c.n_poly, c.den, ox, oy);
                            qx = M::quant(__double2float_rn(ox));  // astype(float32) then cvRound(x * 32)
                            qy = M::quant(__double2float_rn(oy));
                        }
#pragma unroll
                        for (int kk = 0; kk < kPx; ++kk)  // (no indexed register arrays)
                            if (kk == k) { sx[kk] = qx; sy[kk] = qy; nx[kk] = ox; ny[kk] = oy; }
                    }
                };
                if (mv.chain_idx) std_eval(tp.std[1]);
                else std_eval(tp.std[0]);
            } else {
#pragma unroll 1
                for (int k = 0; k < kPx; ++k) {
                    ChainState s;
                    seed(k, s);
                    run_ops(ch, 2, ch.n_ops - (dyn ? 1 : 0), s);
                    to_xy(s);
                    const int qx = M::quant(__double2float_rn(s.x)), qy = M::quant(__double2float_rn(s.y));
#pragma unroll
                    for (int kk = 0; kk < kPx; ++kk)
                        if (kk == k) { sx[kk] = qx; sy[kk] = qy; nx[kk] = s.x; ny[kk] = s.y; }
                }
            }
        } else if (sampler) {
#pragma unroll 1
            for (int k = 0; k < kPx; ++k) {
                double xs, ys;
                if (dyn) eval_chain_normalised(ch, x0 + pcol(k), y0 + prow(k), xs, ys);
                else eval_chain(ch, x0 + pcol(k), y0 + prow(k), xs, ys);
                const int qx = M::quant(__double2float_rn(xs)), qy = M::quant(__double2float_rn(ys));
#pragma unroll
                for (int kk = 0; kk < kPx; ++kk)
                    if (kk == k) { sx[kk] = qx; sy[kk] = qy; nx[kk] = xs; ny[kk] = ys; }
            }
        }
    } else if (sampler) {
        // Tile-packed LUT (vr180_pack_lut_tiles): 16-byte tile header + one uint32 per pixel in thread order
        bool unpacked = false;
        {
            if (packed_tile) {
                uint32_t e[kPx];
                load_packed_entries<M>(mv.packed, tp.n_tiles, tile, tid, e);
#pragma unroll
                for (int k = 0; k < kPx; ++k) {
                    const int2 q = unpack_entry<M>(hdr.mnx, hdr.mny, e[k]);
                    sx[k] = q.x;
                    sy[k] = q.y;
                }
                unpacked = true;
            }
        }
#pragma unroll
        for (int k = 0; k < kPx; ++k) {
            if (unpacked) break;
            const int i = x0 + pcol(k), j = y0 + prow(k);
            sx[k] = sy[k] = (int)0x80000000;
            if (i < a.W && j < a.H) {
                if (mv.map_kind == VR180_MAPSRC_FLOAT2) {
                    sx[k] = M::quant(__ldg(mv.xmap + (long long)j * mv.map_pitch + i));
                    sy[k] = M::quant(__ldg(mv.ymap + (long long)j * mv.map_pitch + i));
                } else {
                    const int2 q = __ldg(mv.fixed + (long long)j * mv.map_pitch + i);
                    sx[k] = q.x;
                    sy[k] = q.y;
                }
            }
        }
    }

    // ---- per-frame radius: a chunk whose frames all share one (finite) radius is a fixed-radius chunk ----------
    // (a static rig: get_radius returns the same value frame after frame).  Its coordinates get their Denormalize
    // here and the tile takes the fixed-radius pipeline -- per-tile pitch choice, constants built once, no
    // per-item radius loads; only chunks with varying radii run the per-frame-rectangle loop.
    bool dynr = dyn;  // CTA-uniform
    if (dyn) {
        const vr180_chain_t& ch = mv.chain_idx ? chain1 : chain0;
        const double r0 = __ldg(mv.radius_dev + f0);
        int same = r0 == r0;
        for (int f = f0 + 1 + lane; f < f1; f += 32) same &= __ldg(mv.radius_dev + f) == r0;
        if (__all_sync(0xffffffffu, same)) {
            dynr = false;
            const double cx = ch.ops[ch.n_ops - 1].p[2], cy = ch.ops[ch.n_ops - 1].p[3];
#pragma unroll
            for (int k = 0; k < kPx; ++k) {
                sx[k] = denorm_q<M>(nx[k], r0, cx);
                sy[k] = denorm_q<M>(ny[k], r0, cy);
            }
        }
    }

    // ---- source rectangle of the tile ---------------------------------------------------------------------
    // a packed tile carries its bounding box in the header: no reduction
    if (!packed_tile) block_box_store<M>(sx, sy, s_red, warp, lane == 0 && sampler);
    DynRadius dr;
    dr.radius = nullptr;
    dr.cx = dr.cy = 0.0;
    dr.ext[0] = dr.ext[1] = dr.ext[2] = dr.ext[3] = 0.0;
    int nan_px = 0;
    if (dynr) {  // tile extremes of the normalised coordinates (frame independent)
        double* s_ext = reinterpret_cast<double*>(smem + Lay<M>::kOffExt);
        double e0 = CUDART_INF, e1 = -CUDART_INF, e2 = CUDART_INF, e3 = -CUDART_INF;
        if (sampler) {
#pragma unroll
            for (int k = 0; k < kPx; ++k) {
                nan_px |= (nx[k] != nx[k]) | (ny[k] != ny[k]);
                e0 = fmin(e0, nx[k]);
                e1 = fmax(e1, nx[k]);
                e2 = fmin(e2, ny[k]);
                e3 = fmax(e3, ny[k]);
            }
        }
#pragma unroll
        for (int d = 16; d > 0; d >>= 1) {
            e0 = fmin(e0, __shfl_xor_sync(0xffffffffu, e0, d));
            e1 = fmax(e1, __shfl_xor_sync(0xffffffffu, e1, d));
            e2 = fmin(e2, __shfl_xor_sync(0xffffffffu, e2, d));
            e3 = fmax(e3, __shfl_xor_sync(0xffffffffu, e3, d));
        }
        if (lane == 0 && sampler) {
            s_ext[warp * 4 + 0] = e0;
            s_ext[warp * 4 + 1] = e1;
            s_ext[warp * 4 + 2] = e2;
            s_ext[warp * 4 + 3] = e3;
        }
    }
    nan_px = __syncthreads_or(nan_px);
    static_assert(Lay<M>::kOffRed % 16 == 0, "s_red is read as int4");
    const int4 box = packed_tile ? make_int4(hdr.mnx, hdr.mxx, hdr.mny, hdr.mxy) : block_box_load(s_red, lane);
    const int mnx = box.x, mxx = box.y, mny = box.z, mxy = box.w;
    const TileRect rc = tile_rect<M>(mnx, mxx, mny, mxy);
    // Taps outside the source read TMA's zero fill = BORDER_CONSTANT(0); only unbounded footprints (NaN / huge
    // coordinates saturate to +-32768) and partial edge tiles leave the fast path.
    // ... and tiles whose item (FR frames x box rows x pitch) does not fit the staging area
    // (a chunk with varying radii runs one-frame items; FR-frame items of a DYN launch are FR one-frame boxes, each 128-byte aligned)
    // (a launch that gives its CTAs single frames pairs the two eyes of a shared map in one item: see VPAIR)
    const bool vpair = !DYN && FR == 1 && nv == 2;
    const int fr_item = dynr ? 1 : (vpair ? 2 : FR);
    auto stage_fits = [&](int box_rows, int pitch_bytes) {
        const int rect = box_rows * pitch_bytes;
        return ((fr_item * ((DYN || vpair) ? (rect + 127) & ~127 : rect) + 127) & ~127) <= Lay<M>::kStageArea;
    };
    // Any other border (a colour, REPLICATE, REFLECT, WRAP, REFLECT_101) needs real taps or the border colour where the
    // footprint leaves the source: those tiles take the per-pixel path below; tiles inside the source never see a border.
    const int src_cols = a.view[v_begin].cols, src_rows = a.view[v_begin].rows;
    auto inside_src = [&](int x_lo, int x_hi, int y_lo, int y_hi) {  // extreme integer coordinates of the tile
        return x_lo - M::kLo >= 0 && x_hi + M::kHi <= src_cols - 1 && y_lo - M::kLo >= 0 && y_hi + M::kHi <= src_rows - 1;
    };
    bool fast = full_tile && rc.wbytes <= kPitchMax && rc.rsel < kRowSizes && mnx > -32768 && mny > -32768 &&
                mxx < 32767 && mxy < 32767 && stage_fits(rc.box_rows, max(rc.wbytes, kPitchMin)) &&
                (tp.zero_border || inside_src(mnx, mxx, mny, mxy));
    int dyn_wbytes = 0, dyn_nrows = 0;  // the largest rectangle over the frames of the chunk
    if (dynr) {
        const double* s_ext = reinterpret_cast<const double*>(smem + Lay<M>::kOffExt);
        dr.ext[0] = dr.ext[2] = CUDART_INF;
        dr.ext[1] = dr.ext[3] = -CUDART_INF;
#pragma unroll
        for (int w = 0; w < kSamplers / 32; ++w) {
            dr.ext[0] = fmin(dr.ext[0], s_ext[w * 4 + 0]);
            dr.ext[1] = fmax(dr.ext[1], s_ext[w * 4 + 1]);
            dr.ext[2] = fmin(dr.ext[2], s_ext[w * 4 + 2]);
            dr.ext[3] = fmax(dr.ext[3], s_ext[w * 4 + 3]);
        }
        const vr180_chain_t& ch = mv.chain_idx ? chain1 : chain0;
        dr.radius = mv.radius_dev;
        dr.cx = ch.ops[ch.n_ops - 1].p[2];
        dr.cy = ch.ops[ch.n_ops - 1].p[3];
        // largest rectangle over the frames of this chunk (lanes stride over the frames; every warp redundantly)
        int ok = 1;
        for (int f = f0 + lane; f < f1; f += 32) {
            const double rad = __ldg(dr.radius + f);
            if (rad == rad) {
                int lo, hi, ylo, yhi;
                dyn_range<M>(dr.ext[0], dr.ext[1], rad, dr.cx, lo, hi);
                ok &= (lo > -32768) & (hi < 32767);
                dyn_range<M>(dr.ext[2], dr.ext[3], rad, dr.cy, ylo, yhi);
                ok &= (ylo > -32768) & (yhi < 32767);
                const TileRect rf = tile_rect<M>(lo, hi, ylo, yhi);
                dyn_wbytes = max(dyn_wbytes, rf.wbytes);
                dyn_nrows = max(dyn_nrows, rf.nrows);
                if (!tp.zero_border) ok &= inside_src(lo, hi, ylo, yhi) ? 1 : 0;
            } else if (!tp.zero_border) {
                ok = 0;  // NaN coordinates: the border colour / the replicated edge pixel -- per-pixel path
            }
        }
        dyn_wbytes = __reduce_max_sync(0xffffffffu, dyn_wbytes);
        dyn_nrows = __reduce_max_sync(0xffffffffu, dyn_nrows);
        ok = __all_sync(0xffffffffu, ok);
        fast = full_tile && ok && !nan_px && dyn_wbytes <= kPitchMax && box_rsel<M>(dyn_nrows) < kRowSizes &&
               stage_fits(M::kRowsMin + box_rsel<M>(dyn_nrows) * kRowsStep, max(dyn_wbytes, kPitchMin));
    }

    if (!fast) {  // per-pixel gather from global memory with full border handling (rare tiles)
        if (sampler) {
#pragma unroll
            for (int k = 0; k < kPx; ++k) {
                const int i = x0 + pcol(k), j = y0 + prow(k);
                if (i < a.W && j < a.H) {
                    for (int f = f0; f < f1; ++f) {
                        int qx = sx[k], qy = sy[k];
                        if (dynr) {
                            const double rad = __ldg(dr.radius + f);
                            qx = denorm_q<M>(nx[k], rad, dr.cx);
                            qy = denorm_q<M>(ny[k], rad, dr.cy);
                        }
                        gather_pixel<M>(a, f, i, j, v_begin, v_end, qx, qy, tp.tab);
                    }
                }
            }
        }
        return;
    }

    // ---- row pitch of the stages = TMA box width: the kPitchCands smallest multiples of 16 bytes that hold the
    // rectangle compete (pitch_costs) ----------------------------------------------------------------------------
    int pitch = max(dynr ? dyn_wbytes : rc.wbytes, kPitchMin);
    // (not worth ~100 instructions per thread when the tile serves only a few frames: tightest box then)
    if (!dynr && (f1 - f0) * nv >= 8) {
        if (sampler) pitch_costs<M>(sx[0], sy[0], rc, pitch, lane, s_cost);
        __syncthreads();
        pitch = pick_pitch(s_cost, pitch, rc.box_rows, [&](int pe) { return stage_fits(rc.box_rows, pe); });
    }

    // ---- per-pixel constants of the frame loop ------------------------------------------------------------
    typename M::Pixel pc[kPx];
#pragma unroll
    for (int k = 0; k < kPx; ++k) {
        const int ix = sx[k] >> M::kShift, iy = sy[k] >> M::kShift;
        const int off = (iy - M::kLo - rc.ry0) * pitch + 3 * (ix - M::kLo) - rc.bx0;
        M::set_offset(pc[k], off, true);
        if (sampler && !dynr) M::weights(pc[k], sx[k] & 31, sy[k] & 31, tp.tab);
    }
    if constexpr (M::kWeightSmem != 0) {
        // fixed radius: the pixel's weights do not change from frame to frame -> private copy in shared memory
        // (written and read by this thread only: no barrier)
        if (!dynr && sampler) {
            uint8_t* slot = smem + Lay<M>::kOffW + tid * 16;
#pragma unroll
            for (int ky = 0; ky < 8; ++ky)
                *reinterpret_cast<uint4*>(slot + ky * (kSamplers * 16)) = __ldg(reinterpret_cast<const uint4*>(pc[0].w) + ky);
            pc[0].ws = smem_u32(slot);
        }
    }
    TileGeom tg;
    tg.rsel = dynr ? box_rsel<M>(dyn_nrows) : rc.rsel;
    tg.bx0 = rc.bx0;
    tg.ry0 = rc.ry0;
    tg.x0 = x0;
    tg.y0 = y0;
    if (DYN && dynr) {
        if (nv == 2) frame_loop<M, 2, DYN, 1>(a, tm, v_begin, f0, f1, pc, tg, pitch, smem, band, cg, dr, nx, ny, tp.tab);
        else         frame_loop<M, 1, DYN, 1>(a, tm, v_begin, f0, f1, pc, tg, pitch, smem, band, cg, dr, nx, ny, tp.tab);
    } else {
        // (a DYN launch has one-frame boxes: its equal-radii chunks run FR-frame items as FR boxes each)
        if constexpr (!DYN && FR == 1) {
            if (nv == 2) frame_loop<M, 2, false, 2, true, true>(a, tm, v_begin, f0, f1, pc, tg, pitch, smem, band, cg, dr, nx, ny, tp.tab);
            else         frame_loop<M, 1, false, 1, false>(a, tm, v_begin, f0, f1, pc, tg, pitch, smem, band, cg, dr, nx, ny, tp.tab);
        } else {
            if (nv == 2) frame_loop<M, 2, false, FR, DYN>(a, tm, v_begin, f0, f1, pc, tg, pitch, smem, band, cg, dr, nx, ny, tp.tab);
            else         frame_loop<M, 1, false, FR, DYN>(a, tm, v_begin, f0, f1, pc, tg, pitch, smem, band, cg, dr, nx, ny, tp.tab);
        }
    }
}

// float32 maps -> tile-packed LUT of mode M (one CTA per tile, the thread <-> pixel assignment of k_warp_tiled)
template <class M>
__global__ void __launch_bounds__(kSamplers) k_pack_tiles(const float* __restrict__ xmap, const float* __restrict__ ymap,
                                                         long long map_pitch, int W, int H, int tiles_x, int n_tiles,
                                                         void* __restrict__ packed) {
    constexpr int kPx = M::kPx;
    __shared__ int4 s_red[kSamplers / 32];
    __shared__ int s_cost[kPitchCands];
    const int tid = threadIdx.x, lane = tid & 31, sw = tid >> 5;
    const int tx = blockIdx.x % tiles_x, ty = blockIdx.x / tiles_x;
    const int x0 = tx * kTileW, y0 = ty * M::kTileH;
    const bool full_tile = (x0 + kTileW <= W) && (y0 + M::kTileH <= H);
    if (tid < kPitchCands) s_cost[tid] = 0;
    int sx[kPx], sy[kPx];
#pragma unroll
    for (int k = 0; k < kPx; ++k) {
        const int i = x0 + lane, j = y0 + kPx * sw + k;  // row patches: a warp owns rows kPx sw .. kPx sw + kPx - 1
        sx[k] = sy[k] = (int)0x80000000;
        if (i < W && j < H) {
            sx[k] = M::quant(__ldg(xmap + (long long)j * map_pitch + i));
            sy[k] = M::quant(__ldg(ymap + (long long)j * map_pitch + i));
        }
    }
    block_box_store<M>(sx, sy, s_red, sw, lane == 0);
    __syncthreads();
    const int4 box = block_box_load(s_red, lane);
    const int mnx = box.x, mxx = box.y, mny = box.z, mxy = box.w;
    const bool ok = full_tile && mnx > -32768 && mny > -32768 && mxx < 32767 && mxy < 32767 && mxx - mnx <= 255 &&
                    mxy - mny <= 255;
    // Geometry of the tile's source rectangle for the tile-streaming kernel (stream.cu), which has no time to derive it
    // per launch: box rows, and the row pitch (= TMA box width) that k_warp_tiled's choice gives a stage slot.
    const TileRect rc = tile_rect<M>(mnx, mxx, mny, mxy);
    const bool stageable = ok && rc.wbytes <= kPitchMax && rc.rsel < kRowSizes;
    const int pitch0 = max(rc.wbytes, kPitchMin);
    if (stageable) pitch_costs<M>(sx[0], sy[0], rc, pitch0, lane, s_cost);  // (CTA-uniform)
    __syncthreads();
    const int pitch = !stageable ? kPitchMin : pick_pitch(s_cost, pitch0, rc.box_rows, [&](int pe) {
        return pe == pitch0 || rc.box_rows * pe <= kStreamSlotBytes<M>;
    });
    const int widx = (pitch - kPitchMin) / kPitchStep;
    if (tid == 0) {
        int4 h;
        h.x = (mnx & 0xffff) | (mxx << 16);
        h.y = (mny & 0xffff) | (mxy << 16);
        h.z = (ok ? kHdrPackable : 0) | (stageable ? kHdrStageable : 0) |
              (stageable && rc.box_rows * pitch <= kStreamSlotBytes<M> ? kHdrFitsSlot : 0) | (widx << 8) | (rc.rsel << 12);
        h.w = 0;
        reinterpret_cast<int4*>(packed)[blockIdx.x] = h;
    }
    uint32_t* ent = reinterpret_cast<uint32_t*>(static_cast<uint8_t*>(packed) + packed_entries_offset(n_tiles)) +
                    ((size_t)blockIdx.x * kSamplers + tid) * kPx;
#pragma unroll
    for (int k = 0; k < kPx; ++k) {
        const int ix = sat16(sx[k] >> M::kShift), iy = sat16(sy[k] >> M::kShift);
        const uint32_t fx = M::kShift ? (uint32_t)(sx[k] & 31) : 0u, fy = M::kShift ? (uint32_t)(sy[k] & 31) : 0u;
        ent[k] = ok ? ((uint32_t)(ix - mnx) | ((uint32_t)(iy - mny) << 8) | (fx << 16) | (fy << 21)) : 0u;
    }
}

}  // namespace tiled

static int tile_height_of(int interp) {
    return interp == VR180_INTER_LINEAR || interp == VR180_INTER_NEAREST ? tiled::LinearP::kTileH
           : interp == VR180_INTER_CUBIC                                  ? tiled::Cubic::kTileH
           : interp == VR180_INTER_LANCZOS4                               ? tiled::Lanczos4::kTileH
                                                                          : 0;
}

size_t packed_lut_bytes(int out_w, int out_h, int interp) {
    const int th = tile_height_of(interp);
    if (!th) return 0;
    const long long n_tiles = (long long)((out_w + tiled::kTileW - 1) / tiled::kTileW) * ((out_h + th - 1) / th);
    return tiled::packed_entries_offset(n_tiles) + (size_t)n_tiles * tiled::kTileW * th * 4;
}

int launch_pack_lut_tiles(const float* xmap, const float* ymap, int64_t map_pitch, int W, int H, int interp, void* packed,
                          cudaStream_t st) {
    using namespace tiled;
    const int th = tile_height_of(interp);
    if (!th) return VR180_ERR_UNSUPPORTED;
    const int tiles_x = (W + kTileW - 1) / kTileW, tiles_y = (H + th - 1) / th;
    const long long n_tiles = (long long)tiles_x * tiles_y;
    if (n_tiles > 0x7fffffffLL) return VR180_ERR_UNSUPPORTED;
    const dim3 grid((unsigned)n_tiles);
    if (interp == VR180_INTER_NEAREST)
        k_pack_tiles<Nearest><<<grid, kSamplers, 0, st>>>(xmap, ymap, (long long)map_pitch, W, H, tiles_x, (int)n_tiles, packed);
    else if (interp == VR180_INTER_LINEAR)
        k_pack_tiles<LinearP><<<grid, kSamplers, 0, st>>>(xmap, ymap, (long long)map_pitch, W, H, tiles_x, (int)n_tiles, packed);
    else if (interp == VR180_INTER_CUBIC)
        k_pack_tiles<Cubic><<<grid, kSamplers, 0, st>>>(xmap, ymap, (long long)map_pitch, W, H, tiles_x, (int)n_tiles, packed);
    else
        k_pack_tiles<Lanczos4><<<grid, kSamplers, 0, st>>>(xmap, ymap, (long long)map_pitch, W, H, tiles_x, (int)n_tiles, packed);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    VR180_CUDA(cudaGetLastError());
    return VR180_OK;
}

// Host: recognise the standard chain shape (see StdChain).
static void match_std_chain(const vr180_chain_t& c, tiled::StdChain& out) {
    memset(&out, 0, sizeof(out));
    out.n_poly = -1;
    if (c.n_ops < 4 || c.ops[0].code != VR180_OP_NORMALIZE || c.ops[1].code != VR180_OP_EQUIRECT_ENC) return;
    memcpy(out.norm, c.ops[0].p, sizeof(out.norm));
    out.lat_is_y = c.ops[1].iparam != 0;
    int k = 2;
    if (c.ops[k].code == VR180_OP_ROT3) {
        out.has_rot = 1;
        memcpy(out.R, c.ops[k].p, sizeof(out.R));
        ++k;
    }
    if (k < c.n_ops && c.ops[k].code == VR180_OP_POLY) {
        out.n_poly = c.ops[k].iparam;
        memcpy(out.poly, c.ops[k].p, sizeof(out.poly));
        ++k;
    }
    if (k + 2 != c.n_ops || c.ops[k].code != VR180_OP_FISHEYE_DEC || c.ops[k].iparam != VR180_MAP_EQUIDISTANT ||
        c.ops[k + 1].code != VR180_OP_DENORMALIZE)
        return;
    memcpy(out.den, c.ops[k + 1].p, sizeof(out.den));
    out.valid = 1;
    // chain_fast.cuh takes theta from (hypot(vx, vy), vz) as a point of the unit circle: R has to be orthonormal
    if (!out.has_rot) {
        out.R[0] = out.R[4] = out.R[8] = 1.0;
        out.fast = 1;
    } else {
        double err = 0.0;
        for (int i = 0; i < 3; ++i)
            for (int j = 0; j < 3; ++j) {
                double d = i == j ? -1.0 : 0.0;
                for (int m = 0; m < 3; ++m) d += out.R[3 * m + i] * out.R[3 * m + j];
                err = std::fmax(err, std::fabs(d));
            }
        out.fast = err < 1e-12 ? 1 : 0;  // (NaN -> 0)
    }
}

// ---- TMA descriptors (host) ---------------------------------------------------------------------------------
using EncodeTiledFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                   const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                   CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeTiledFn encode_tiled_fn() {
    static EncodeTiledFn fn = [] {
        void* p = nullptr;
        cudaDriverEntryPointQueryResult q = cudaDriverEntryPointSymbolNotFound;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
            q != cudaDriverEntryPointSuccess)
            p = nullptr;
        cudaGetLastError();
        return reinterpret_cast<EncodeTiledFn>(p);
    }();
    return fn;
}

// uint8 tensor (row_bytes, rows, frames) with byte strides (pitch, frame_stride); box (box_w, box_h, 1).
// Out-of-bounds box elements are filled with zeros on loads and dropped on stores.
static bool encode_u8_3d(CUtensorMap* out, const void* base, long long row_bytes, long long rows, long long frames,
                         long long pitch, long long frame_stride, int box_w, int box_h, int box_d) {
    EncodeTiledFn fn = encode_tiled_fn();
    if (!fn) return false;
    if (frames <= 1 || frame_stride < pitch * rows) frame_stride = ((pitch * rows + 15) / 16) * 16;  // unused when frames == 1
    const cuuint64_t dims[3] = {(cuuint64_t)row_bytes, (cuuint64_t)rows, (cuuint64_t)(frames < 1 ? 1 : frames)};
    const cuuint64_t strides[2] = {(cuuint64_t)pitch, (cuuint64_t)frame_stride};
    const cuuint32_t box[3] = {(cuuint32_t)box_w, (cuuint32_t)box_h, (cuuint32_t)box_d};
    const cuuint32_t estr[3] = {1u, 1u, 1u};
    return fn(out, CU_TENSOR_MAP_DATA_TYPE_UINT8, 3, const_cast<void*>(base), dims, strides, box, estr,
              CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
              CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

int tiled_debug_flags() {  // vr180_debug_set(1, flags), else $VR180_TILED_DEBUG
    static const int env_debug = [] { const char* e = getenv("VR180_TILED_DEBUG"); return e ? atoi(e) : 0; }();
    const int set_debug = g_debug_tiled_flags.load(std::memory_order_relaxed);
    return set_debug >= 0 ? set_debug : env_debug;
}

constexpr int kMaxFramesPerCta = 64;
// frames per CTA: the coordinates are evaluated once per CTA, so keep the chunk as large as the grid allows
static int frames_per_cta(long long tiles, int n_frames, int views_per_cta = 1) {
    const int forced = g_debug_frames_per_cta.load(std::memory_order_relaxed);  // vr180_debug_set(0, n): tests
    if (forced > 0) return forced < n_frames ? forced : n_frames;
    // A CTA streams through its frames one after the other and the CTAs of neighbouring tiles -- which share the halo
    // of their source rectangles through L2 -- drift apart the longer they run: beyond ~64 (frame, eye) rectangles per
    // CTA a launch loses more to that than the per-tile prologue amortises.  Measured, B200: 512 5.7K pairs (both eyes
    // per CTA) in ONE chunk 37 us per pair, chunks of 128 / 64 / 32 frames 31 / 27 / 25 us; 128 8K pairs (one eye per
    // CTA) in chunks of 128 / 64 / 32 frames 53.8 / 48.6 / 50.5 us per pair.
    const int cap_set = g_debug_max_frames_per_cta.load(std::memory_order_relaxed);
    const int cap = cap_set > 0 ? cap_set : kMaxFramesPerCta / views_per_cta;
    int fpc = n_frames;
    if (fpc > cap) fpc = (n_frames + (n_frames + cap - 1) / cap - 1) / ((n_frames + cap - 1) / cap);  // equal chunks
    while (fpc > 1 && tiles * ((n_frames + fpc - 1) / fpc) < 148LL * 4 * 2) fpc = (fpc + 1) / 2;
    return fpc;
}

// TMA descriptors of a launch.  They depend only on the buffers' geometry: video loops call with the same buffers again
// and again, so the last few sets are kept per host thread (a ring of batches cycles through a handful of buffers, and
// 199 cuTensorMapEncodeTiled calls cost about as much host time as a single-pair launch takes on the GPU).
// `fr`: frames per box (depth of the load and store boxes).  nullptr = a descriptor could not be encoded.
const tiled::TmaMaps* tma_maps_for(const RemapArgs& a0, int interp, int rows_min, int tile_h, int fr) {
    using namespace tiled;
    struct Key {
        const void* src[2];
        long long pitch[2], fs[2];
        int rows, cols, n_views, n_frames, H, mode, fr, pad;
        const void* dst;
        long long dst_pitch, dst_fs;
    };
    Key key;
    memset(&key, 0, sizeof(key));
    for (int v = 0; v < a0.n_views; ++v) {
        key.src[v] = a0.view[v].src;
        key.pitch[v] = a0.view[v].pitch;
        key.fs[v] = a0.view[v].frame_stride;
    }
    key.rows = a0.view[0].rows;
    key.cols = a0.view[0].cols;
    key.n_views = a0.n_views;
    key.n_frames = a0.n_frames;
    key.H = a0.H;
    key.mode = interp;
    key.fr = fr;
    key.dst = a0.dst;
    key.dst_pitch = a0.dst_pitch;
    key.dst_fs = a0.dst_frame_stride;
    struct Entry {
        Key key;
        TmaMaps tm;
        uint64_t stamp;
    };
    constexpr size_t kCacheEntries = 8;
    static thread_local std::vector<Entry> cache;
    static thread_local uint64_t clock_ = 0;
    Entry* hit = nullptr;
    for (Entry& e : cache)
        if (memcmp(&key, &e.key, sizeof(key)) == 0) hit = &e;
    if (!hit) {
        if (cache.size() < kCacheEntries) {
            cache.emplace_back();
            hit = &cache.back();
        } else {
            hit = &cache[0];
            for (Entry& e : cache)
                if (e.stamp < hit->stamp) hit = &e;
        }
        memset(&hit->key, 0xff, sizeof(hit->key));  // invalid until every descriptor is encoded
        TmaMaps& t = hit->tm;
        memset(&t, 0, sizeof(t));
        for (int v = 0; v < a0.n_views; ++v) {
            const ViewArgs& vw = a0.view[v];
            for (int w = 0; w < kWidths; ++w)
                for (int r = 0; r < kRowSizes; ++r)
                    if (!encode_u8_3d(&t.src[v][w][r], vw.src, (long long)vw.cols * 3, vw.rows, a0.n_frames, vw.pitch,
                                      vw.frame_stride, kPitchMin + w * kPitchStep, rows_min + r * kRowsStep, fr))
                        return nullptr;
        }
        if (a0.n_views == 1) memcpy(&t.src[1], &t.src[0], sizeof(t.src[0]));
        if (!encode_u8_3d(&t.dst, a0.dst, a0.dst_pitch, a0.H, a0.n_frames, a0.dst_pitch, a0.dst_frame_stride, kTileW * 3,
                          tile_h, fr))
            return nullptr;
        hit->key = key;
    }
    hit->stamp = ++clock_;
    return &hit->tm;
}

template <class M, bool DYN, int FR>
static int launch_mode(const RemapArgs& a0, const vr180_chain_t& c0, const vr180_chain_t& c1, const short* tab,
                       cudaStream_t st) {
    using namespace tiled;
    const int n_groups = a0.share_map ? 1 : a0.n_views;
    const TmaMaps* tmp = tma_maps_for(a0, M::kInterp, M::kRowsMin, M::kTileH, DYN ? 1 : FR);
    if (!tmp) return VR180_ERR_UNSUPPORTED;
    const TmaMaps& tm = *tmp;

    int dev = 0;
    const int rc = max_dyn_smem_once<k_warp_tiled<M, DYN, FR>>(Lay<M>::kSmemBytes, dev);
    if (rc != VR180_OK) return rc;

    RemapArgs a = a0;
    TiledParams tp;
    memset(&tp, 0, sizeof(tp));
    const int tiles_x = (a.W + kTileW - 1) / kTileW, tiles_y = (a.H + M::kTileH - 1) / M::kTileH;
    tp.tiles_x = tiles_x;
    tp.n_tiles = tiles_x * tiles_y;
    tp.tab = tab;
    tp.zero_border = zero_border(a);
    tp.debug = tiled_debug_flags();
    const long long tiles = (long long)tiles_x * tiles_y * n_groups;
    int fpc = frames_per_cta(tiles, a.n_frames, a.share_map ? a.n_views : 1);
    fpc = (fpc + FR - 1) / FR * FR;  // chunks start at multiples of FR: phantom frames can only lie past the batch
    a.frames_per_cta = fpc;
    const int chunks = (a.n_frames + fpc - 1) / fpc;
    if (n_groups > 2 || chunks * n_groups > 65535 || tiles_y > 65535 || tiles_x * (long long)tiles_y > 0x7fffffffLL)
        return VR180_ERR_UNSUPPORTED;
    auto is_sep = [](const vr180_chain_t& c) {
        return c.n_ops >= 2 && c.ops[0].code == VR180_OP_NORMALIZE && c.ops[1].code == VR180_OP_EQUIRECT_ENC;
    };
    tp.sep_prefix = 1;
    for (int g = 0; g < n_groups; ++g) {
        if (a.view[g].map_kind != VR180_MAPSRC_ANALYTIC) continue;
        const vr180_chain_t& c = a.view[g].chain_idx ? c1 : c0;
        if (!is_sep(c)) tp.sep_prefix = 0;
        match_std_chain(c, tp.std[a.view[g].chain_idx ? 1 : 0]);
    }
    dim3 grid((unsigned)tiles_x, (unsigned)tiles_y, (unsigned)(n_groups * chunks));  // z = chunk * n_groups + map group
    k_warp_tiled<M, DYN, FR><<<grid, kThreads, Lay<M>::kSmemBytes, st>>>(a, c0, c1, tp, tm);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    VR180_CUDA(cudaGetLastError());
    return VR180_OK;
}

// FR = frames per pipeline item for `fpc` frames per CTA: 2 from two frames on, bicubic 4 from eight on
template <class M>
static int launch_tiled(const RemapArgs& a0, const vr180_chain_t& c0, const vr180_chain_t& c1, const short* tab, bool dyn,
                        int fpc, cudaStream_t st) {
    if constexpr (M::kInterp == VR180_INTER_CUBIC) {
        if (fpc >= 8) return dyn ? launch_mode<M, true, 4>(a0, c0, c1, tab, st) : launch_mode<M, false, 4>(a0, c0, c1, tab, st);
    }
    if (fpc >= 2) return dyn ? launch_mode<M, true, 2>(a0, c0, c1, tab, st) : launch_mode<M, false, 2>(a0, c0, c1, tab, st);
    return dyn ? launch_mode<M, true, 1>(a0, c0, c1, tab, st) : launch_mode<M, false, 1>(a0, c0, c1, tab, st);
}

// Host-side eligibility + launch.  Returns VR180_ERR_UNSUPPORTED when the request is outside the fast path (the
// caller then launches the generic k_remap); any other value is final.  `weight_tab`: device copy of the weight table of
// the requested interpolation (1024 x 16 bicubic, 1024 x 64 Lanczos4; unused otherwise).
int launch_remap_tiled(const RemapArgs& a0, int channels, int interp, const vr180_chain_t& c0, const vr180_chain_t& c1,
                       const short* weight_tab, cudaStream_t st) {
    if (channels != 3 || a0.depth != VR180_DEPTH_8U) return VR180_ERR_UNSUPPORTED;
    if (interp != VR180_INTER_NEAREST && interp != VR180_INTER_LINEAR && interp != VR180_INTER_CUBIC &&
        interp != VR180_INTER_LANCZOS4)
        return VR180_ERR_UNSUPPORTED;
    if (interp == VR180_INTER_NEAREST)  // the fixed-point LUT is a 1/32-pixel grid; NEAREST rounds the float coordinate itself
        for (int v = 0; v < a0.n_views; ++v)
            if (a0.view[v].map_kind == VR180_MAPSRC_FIXED) return VR180_ERR_UNSUPPORTED;
    const int n_groups = a0.share_map ? 1 : a0.n_views;
    for (int v = 0; v < a0.n_views; ++v) {
        const ViewArgs& vw = a0.view[v];
        // TMA: 16-byte aligned base and strides
        if (((uintptr_t)vw.src & 15) || (vw.pitch & 15) || (vw.frame_stride & 15) || vw.pitch < (long long)vw.cols * 3)
            return VR180_ERR_UNSUPPORTED;
        if (a0.n_frames > 1 && vw.frame_stride < vw.pitch * vw.rows) return VR180_ERR_UNSUPPORTED;
        if (vw.rows != a0.view[0].rows || vw.cols != a0.view[0].cols) return VR180_ERR_UNSUPPORTED;
        // a TMA box must start at a 16-byte aligned global address: tile columns are multiples of 32 pixels (96
        // bytes), so the eye's column offset inside the SBS frame has to be one too (an unaligned start traps
        // with "illegal instruction" on B200, for loads and stores alike)
        if ((vw.dst_x_offset * 3) & 15) return VR180_ERR_UNSUPPORTED;
    }
    if (((uintptr_t)a0.dst & 15) || (a0.dst_pitch & 15) || (a0.dst_frame_stride & 15)) return VR180_ERR_UNSUPPORTED;
    if (a0.n_frames > 1 && a0.dst_frame_stride < a0.dst_pitch * a0.H) return VR180_ERR_UNSUPPORTED;
    // per-frame radius: all map groups or none (a mixed request takes the generic kernel)
    int n_dyn = 0;
    for (int g = 0; g < n_groups; ++g)
        n_dyn += (a0.view[g].map_kind == VR180_MAPSRC_ANALYTIC && a0.view[g].radius_dev) ? 1 : 0;
    if (n_dyn != 0 && n_dyn != n_groups) return VR180_ERR_UNSUPPORTED;
    const bool dyn = n_dyn != 0;
    // A few frames per launch with tile-packed LUTs: little to amortise a tile's prologue over -> persistent CTAs that
    // stream the tiles (stream.cu), two of a tile's (frame, eye) rectangles per pipeline item.  Measured, B200, streamed vs
    // batched: 4K pairs sharing a map 1 / 2 / 4 / 8 / 12 / 16 pairs 24.0 / 36.9 / 60.2 / 109 / 158 / 208 us vs 36.3 / 45.7 /
    // 78.5 / 116 / 155 / 196 us; 8K pairs with per-eye maps 1 / 2 / 4 / 8 / 12 / 16 / 24 pairs 110 / 151 / 240 / 431 / 618 / 806 /
    // 1206 us vs 217 / 245 / 310 / 548 / 690 / 827 / 1125 us.  VR180_TILED_DEBUG bit 1: whenever eligible; bit 2: never.
    const int kStreamMaxItems = a0.share_map ? 20 : 16;  // (frame, eye) rectangles per tile
    {
        bool all_packed = !dyn;
        for (int g = 0; g < n_groups; ++g) all_packed = all_packed && a0.view[g].packed != nullptr;
        const int dbg = tiled_debug_flags();
        const int items = a0.n_frames * (a0.share_map ? a0.n_views : 1);
        const bool tab_ok = (interp != VR180_INTER_CUBIC && interp != VR180_INTER_LANCZOS4) || weight_tab != nullptr;
        if (all_packed && tab_ok && !(dbg & 4) && ((dbg & 2) || items <= kStreamMaxItems) &&
            g_debug_frames_per_cta.load(std::memory_order_relaxed) <= 0) {
            const int rc = launch_remap_stream(a0, interp, weight_tab, st);
            if (rc != VR180_ERR_UNSUPPORTED) return rc;
        }
    }
    // two frames per pipeline item when the frames share their rectangles (per-frame radii: the chunks whose frames all
    // share one radius, a static rig) and every CTA gets at least two of them
    const int tile_h = tile_height_of(interp);
    const long long tiles = (long long)((a0.W + tiled::kTileW - 1) / tiled::kTileW) * ((a0.H + tile_h - 1) / tile_h) * n_groups;
    const int fpc = frames_per_cta(tiles, a0.n_frames, a0.share_map ? a0.n_views : 1);
    if (interp == VR180_INTER_NEAREST) return launch_tiled<tiled::Nearest>(a0, c0, c1, nullptr, dyn, fpc, st);
    if (interp == VR180_INTER_LINEAR) return launch_tiled<tiled::LinearP>(a0, c0, c1, nullptr, dyn, fpc, st);
    if (!weight_tab) return VR180_ERR_UNSUPPORTED;
    if (interp == VR180_INTER_LANCZOS4) return launch_tiled<tiled::Lanczos4>(a0, c0, c1, weight_tab, dyn, fpc, st);
    return launch_tiled<tiled::Cubic>(a0, c0, c1, weight_tab, dyn, fpc, st);
}

}  // namespace vr180
