// stream.cu -- the tiled warp for launches of ONE or a few frames: tiles streamed through persistent CTAs.
//
// Replaces cv.remap per eye + np.concatenate (/root/reference/src/vr180_convert/remapper.py:388-398, :518) for the
// frame-at-a-time form of the path (a video loop calling apply_lr / lr_frame once per stereo pair with cached maps:
// BASELINE configs[1], north_star (2) "cached-LUT path for repeated video frames").
//
// k_warp_tiled (tiled.cu) gives every CTA ONE tile and amortises the tile's prologue over the frames of a batch.  With
// one frame per launch nothing is amortised and the CTA is a chain of latencies (header -> coordinates -> bounding box
// -> TMA load -> sample -> TMA store), 100 instructions per 32 pixels and 41 us for a 4K pair (HBM time: 7 us).
// Here a CTA is persistent and walks the tiles  blockIdx.x, blockIdx.x + gridDim.x, ...  of the launch:
//   * the coordinates come from the tile-packed LUT (vr180_pack_lut_tiles), whose 16-byte tile header carries the
//     tile's bounding box, its TMA box sizes and the row pitch chosen at pack time: the producer warp needs nothing
//     from the sampling warps to fetch a tile's source rectangle, so it runs up to kSlots items (tile, frame, eye)
//     AHEAD of them -- the TMA loads of the next tiles are in flight while the current one is sampled;
//   * the sampling warps prefetch the next tile's header and LUT entries (one 128-bit load per thread) before they
//     sample the current one;
//   * per tile a thread only unpacks its 4 entries into the sampling constants (offset and selectors by multiply-add,
//     the bilinear weight pair by one LDS.64 from a table built once per CTA); no block-wide reduction, no pitch
//     search, no per-launch-mode branches.
// Pipeline, barriers and the sampling / re-packing of a tile are those of k_warp_tiled (tiled.cuh); an item is one
// frame of one eye -- or of both eyes when they share the coordinates and both rectangles fit a slot; the stage ring
// has fixed-size slots because consecutive items belong to different tiles.
// Tiles that cannot be packed (partial edge tiles, NaN / huge coordinates), whose rectangle exceeds a slot, or that
// touch the source edge under a non-zero border are noted while the CTA streams and gathered per pixel afterwards.
// Measured (B200): one 4K pair 24 us (k_warp_tiled 36-41 us), one 8K pair with per-eye maps 108 us (217 us); faster
// than k_warp_tiled up to ~24 (shared map) / ~14 (per-eye maps) rectangles per tile (DESIGN.md 5.6).
#include "tiled.cuh"

namespace vr180 {
namespace tiled {

constexpr int kSlots = 3;       // stage ring: slots of Lay<M>::kStageArea / 3 bytes (13.5 KB; a bilinear 8K tile needs <= 10.5 KB)
constexpr int kSlowCap = 128;   // non-staged tiles a CTA notes before it stops streaming to gather them
constexpr int kStreamCtas = 3;  // CTAs per SM: 72 registers (4 CTAs / 56 registers spill and measure 1-2 % slower)

template <class M>
struct SLay {
    static constexpr int kSlotBytes = kStreamSlotBytes<M>;
    static_assert(kSlots == 3, "kStreamSlotBytes (tiled.cuh) is a third of the staging area");
    static constexpr int kOutTileBytes = M::kTileH * kTileW * 3;
    static constexpr int kOB = kOutBufs;  // out buffers of one item each: the tile of one eye or of both
    static constexpr int kOutItemBytes = 2 * kOutTileBytes;
    static constexpr int kOffOut = kSlots * kSlotBytes;
    static constexpr int kOffBar = kOffOut + kOB * kOutItemBytes;  // full[kSlots], ofull[kOB], oempty[kOB]
    static constexpr int kOffQ = (kOffBar + (kSlots + 2 * kOB) * 8 + 15) & ~15;  // int4 per slot: store coordinates of the item in it
    static constexpr int kOffW = (kOffQ + kSlots * 16 + 15) & ~15;
    // bilinear: the packed weight pairs {W01, W23} of all 32 x 32 sub-pixel positions, built once per CTA -- a tile's
    // pixels then fetch their weights with one LDS.64 instead of computing four products and two packs each
    static constexpr int kWeightTab = M::kInterp == VR180_INTER_LINEAR ? 1024 * 8 : 0;
    static constexpr int kOffTab = kOffW + M::kWeightSmem;
    static constexpr int kOffSlow = kOffTab + kWeightTab;  // int2 (map group, tile) of the tiles left to the per-pixel gather
    static constexpr int kSmemBytes = kOffSlow + kSlowCap * 8;
};

struct StreamParams {
    int tiles_x, n_tiles, n_units;  // units = map groups x tiles
    int zero_border;
    const short* tab;
};

// Source rectangle of a packed tile from its header alone (both the producer and the sampling warps evaluate it): the
// box sizes were chosen by k_pack_tiles, only the origin and the border test are left.
struct UnitGeom {
    int fast, bx0, ry0, pitch, rsel, rect_bytes, org;
    int eye_pitch;  // distance of the two eyes' rectangles inside a slot (TMA destinations are 128-byte aligned)
};
template <class M>
__device__ __forceinline__ UnitGeom unit_geom(const int4& raw, int zero_border, int src_cols, int src_rows) {
    UnitGeom g;
    const TileHdr h = decode_header(raw);
    const TileRect rc = tile_rect<M>(h.mnx, h.mxx, h.mny, h.mxy);
    g.bx0 = rc.bx0;
    g.org = 3 * (h.mnx - M::kLo) - rc.bx0;  // byte offset of the tile's first tap column in the box
    g.ry0 = rc.ry0;
    g.pitch = kPitchMin + kPitchStep * ((h.flags >> 8) & 15);
    g.rsel = (h.flags >> 12) & 15;
    g.rect_bytes = (M::kRowsMin + g.rsel * kRowsStep) * g.pitch;
    g.eye_pitch = (g.rect_bytes + 127) & ~127;
    constexpr int kAll = kHdrPackable | kHdrStageable | kHdrFitsSlot;
    g.fast = (h.flags & kAll) == kAll;
    if (!zero_border)  // any other border needs real taps where the footprint leaves the source: per-pixel path
        g.fast = g.fast && (int)h.mnx - M::kLo >= 0 && (int)h.mxx + M::kHi <= src_cols - 1 && (int)h.mny - M::kLo >= 0 &&
                 (int)h.mxy + M::kHi <= src_rows - 1;
    return g;
}

// Tiles that are not staged: per-pixel gather from global memory with full border handling (rare: partial edge tiles,
// NaN / huge coordinates, footprints beyond a stage slot, the source edge under a non-zero border).  The pixel loop is
// unrolled: an indexed access to the entries would put them in local memory for the streaming loop too.
template <int N>
struct Entries {
    uint32_t e[N];
};
template <class M>
__device__ __forceinline__ void gather_tile(const RemapArgs& a, const StreamParams& sp, int grp, int tile, int nv, bool packed,
                                         int mnx, int mny, Entries<M::kPx> ev) {
    constexpr int kPx = M::kPx;
    const int tid = threadIdx.x, lane = tid & 31, sw = tid >> 5;
    const ViewArgs& mv = a.view[grp];
    const int ty = tile / sp.tiles_x, tx = tile - ty * sp.tiles_x;
    const int x0 = tx * kTileW, y0 = ty * M::kTileH;
#pragma unroll
    for (int k = 0; k < kPx; ++k) {
        const int i = x0 + lane, j = y0 + kPx * sw + k;
        if (i >= a.W || j >= a.H) continue;
        int2 q;
        if (packed) {
            q = unpack_entry<M>(mnx, mny, ev.e[k]);
        } else {
            q.x = M::quant(__ldg(mv.xmap + (long long)j * mv.map_pitch + i));
            q.y = M::quant(__ldg(mv.ymap + (long long)j * mv.map_pitch + i));
        }
        for (int f = 0; f < a.n_frames; ++f) gather_pixel<M>(a, f, i, j, grp, grp + nv, q.x, q.y, sp.tab);
    }
}

template <class M>
__global__ void __launch_bounds__(kThreads, kStreamCtas)
k_warp_stream(const __grid_constant__ RemapArgs a, const __grid_constant__ StreamParams sp,
              const __grid_constant__ TmaMaps tm) {
    constexpr int kPx = M::kPx;
    constexpr int kOB = SLay<M>::kOB, kOutTileBytes = SLay<M>::kOutTileBytes, kSlotBytes = SLay<M>::kSlotBytes;
    constexpr int kOutItemBytes = SLay<M>::kOutItemBytes;
    extern __shared__ __align__(1024) uint8_t smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const uint32_t s_stage = smem_u32(smem), s_full = s_stage + SLay<M>::kOffBar;
    const uint32_t s_ofull = s_full + kSlots * 8, s_oempty = s_ofull + kOB * 8, s_out = s_stage + SLay<M>::kOffOut;
    int4* const s_q = reinterpret_cast<int4*>(smem + SLay<M>::kOffQ);
    if (tid < kSlots + 2 * kOB) {
        const bool by_warps = tid >= kSlots && tid < kSlots + kOB;  // ofull: one arrive per sampling warp
        mbar_init(s_full + tid * 8, by_warps ? kSamplers / 32 : 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if constexpr (SLay<M>::kWeightTab != 0) {
        uint2* const wt = reinterpret_cast<uint2*>(smem + SLay<M>::kOffTab);
        for (int i = tid; i < 1024; i += kThreads) {
            typename M::Pixel p;
            M::weights(p, i & 31, i >> 5, nullptr);
            wt[i] = make_uint2(p.W01, p.W23);
        }
    }
    __syncthreads();
    const int nv = a.share_map ? a.n_views : 1;
    const int src_cols = a.view[0].cols, src_rows = a.view[0].rows;
    const int stride = gridDim.x;

    if (warp == kSamplers / 32) {  // ---- producer: one thread drives the TMA unit ----
        if (lane != 0) return;
        int n_load = 0, n_store = 0, l_slot = 0, s_slot = 0;
        auto store_next = [&]() {  // the oldest item in flight: its tile is complete -> TMA store, slot and out buffer are free
            const int o = n_store & (kOB - 1);
            mbar_wait(s_ofull + o * 8, (uint32_t)(n_store / kOB) & 1u);
            const int4 q = s_q[s_slot];
            tma_store_3d(&tm.dst, q.x, q.y, q.z & 0xffff, s_out + o * kOutItemBytes);
            if (q.w >= 0) tma_store_3d(&tm.dst, q.w, q.y, q.z >> 16, s_out + o * kOutItemBytes + kOutTileBytes);  // the item's second rectangle
            bulk_commit();
            bulk_wait_read<0>();
            mbar_arrive(s_oempty + o * 8);
            ++n_store;
            if (++s_slot == kSlots) s_slot = 0;
        };
        int grp_n = 0, tile_n = blockIdx.x;  // unit = (map group, tile); blockIdx.x < n_units
        while (tile_n >= sp.n_tiles) { tile_n -= sp.n_tiles; ++grp_n; }
        int4 hn = packed_header_raw(a.view[grp_n].packed, tile_n);  // kept as loaded: three registers
        for (int u = blockIdx.x; u < sp.n_units; u += stride) {
            const int4 hdr = hn;
            const int grp = grp_n, tile = tile_n;
            tile_n += stride;
            while (tile_n >= sp.n_tiles) { tile_n -= sp.n_tiles; ++grp_n; }
            if (u + stride < sp.n_units) hn = packed_header_raw(a.view[grp_n].packed, tile_n);
            const UnitGeom g = unit_geom<M>(hdr, sp.zero_border, src_cols, src_rows);
            if (!g.fast) continue;
            const int ty = tile / sp.tiles_x, tx = tile - ty * sp.tiles_x;
            const CUtensorMap* const map0 = &tm.src[grp][(g.pitch - kPitchMin) / kPitchStep][g.rsel];
            // The tile's rectangles (frame-major, eye-minor: they all share the tile's coordinates) travel two per item when
            // two fit one slot: two box loads on one barrier, one hand-shake with the sampling warps, two tile stores.
            const int n_rects = a.n_frames * nv, per_item = 2 * g.eye_pitch <= kSlotBytes ? 2 : 1;
            const int x_l = (a.view[grp].dst_x_offset + tx * kTileW) * 3;
            const int x_r = nv == 2 ? (a.view[grp + 1].dst_x_offset + tx * kTileW) * 3 : x_l;
            for (int r = 0; r < n_rects; r += per_item) {
                if (n_load - n_store == kSlots) store_next();
                const uint32_t bar = s_full + l_slot * 8;
                const uint32_t dst = s_stage + l_slot * kSlotBytes;
                const bool two = per_item == 2 && r + 1 < n_rects;
                const int v0 = nv == 2 ? (r & 1) : 0, f0 = nv == 2 ? (r >> 1) : r;
                const int v1 = nv == 2 ? ((r + 1) & 1) : 0, f1 = nv == 2 ? ((r + 1) >> 1) : r + 1;
                s_q[l_slot] = make_int4(v0 ? x_r : x_l, ty * M::kTileH, f0 | (f1 << 16), two ? (v1 ? x_r : x_l) : -1);
                mbar_expect_tx(bar, (two ? 2u : 1u) * (uint32_t)g.rect_bytes);
                tma_load_3d(dst, map0 + v0 * (kWidths * kRowSizes), g.bx0, g.ry0, f0, bar);
                if (two) tma_load_3d(dst + g.eye_pitch, map0 + v1 * (kWidths * kRowSizes), g.bx0, g.ry0, f1, bar);
                ++n_load;
                if (++l_slot == kSlots) l_slot = 0;
            }
        }
        while (n_store < n_load) store_next();
        bulk_wait_read<0>();  // shared memory must stay valid until the last store has read it
        return;
    }

    // ---- sampling warps ----
    const int sw = warp;  // owns rows kPx sw .. kPx sw + kPx - 1 of a tile, column = lane
    const int sub = lane & 3;
    const uint32_t out_sel = sub == 0 ? 0x4210u : (sub == 1 ? 0x5421u : 0x6542u);
    uint32_t outp = s_out + (kPx * sw) * (kTileW * 3) + (3 * (lane >> 2) + sub) * 4;
    uint32_t flags = (sub != 3 ? 1u : 0u) | (lane == 0 ? 2u : 0u);
    asm volatile("" : "+r"(outp), "+r"(flags));

    // Tiles that are not staged are only noted (s_slow) while the CTA streams; they are gathered per pixel afterwards,
    // outside the streaming loop, whose registers the gather code would otherwise claim (the prefetched header and entries
    // ended up in local memory).  A full list ends the streaming phase early; the outer loop resumes it after the drain.
    int2* const s_slow = reinterpret_cast<int2*>(smem + SLay<M>::kOffSlow);
    int n = 0, st = 0;
    uint32_t ph = 0;
    int grp_n = 0, tile_n = blockIdx.x;  // unit = (map group, tile); blockIdx.x < n_units
    while (tile_n >= sp.n_tiles) { tile_n -= sp.n_tiles; ++grp_n; }
    int u = blockIdx.x;
  for (;;) {
    int n_slow = 0;
    int4 hn = packed_header_raw(a.view[grp_n].packed, tile_n);  // kept as loaded: three registers
    uint32_t en[kPx];
    load_packed_entries<M>(a.view[grp_n].packed, sp.n_tiles, tile_n, tid, en);
    for (; u < sp.n_units && n_slow < kSlowCap; u += stride) {
        const int4 hdr = hn;
        uint32_t e[kPx];
#pragma unroll
        for (int k = 0; k < kPx; ++k) e[k] = en[k];
        const int grp = grp_n, tile = tile_n;
        tile_n += stride;
        while (tile_n >= sp.n_tiles) { tile_n -= sp.n_tiles; ++grp_n; }
        if (u + stride < sp.n_units) {  // the next tile's header and entries travel while this one is sampled
            hn = packed_header_raw(a.view[grp_n].packed, tile_n);
            load_packed_entries<M>(a.view[grp_n].packed, sp.n_tiles, tile_n, tid, en);
        }
        const UnitGeom g = unit_geom<M>(hdr, sp.zero_border, src_cols, src_rows);

        if (!g.fast) {
            if (tid == 0) s_slow[n_slow] = make_int2(grp, tile);
            ++n_slow;
            continue;
        }

        // ---- sampling constants of this thread's pixels ----
        typename M::Pixel pc[kPx];
#pragma unroll
        for (int k = 0; k < kPx; ++k) {
            const int dx = (int)(e[k] & 255u), dy = (int)((e[k] >> 8) & 255u);  // iy - kLo - ry0 == dy
            M::set_offset(pc[k], dy * g.pitch + 3 * dx + g.org, true);
            if constexpr (SLay<M>::kWeightTab != 0) {
                asm("ld.shared.v2.u32 {%0, %1}, [%2];"
                    : "=r"(pc[k].W01), "=r"(pc[k].W23)
                    : "r"(s_stage + SLay<M>::kOffTab + ((e[k] >> 13) & (1023u << 3))));
            } else {
                M::weights(pc[k], (int)((e[k] >> 16) & 31u), (int)((e[k] >> 21) & 31u), sp.tab);
            }
        }
        if constexpr (M::kWeightSmem != 0) {  // Lanczos4: the pixel's 64 weights, private copy in shared memory
            uint8_t* slot = smem + SLay<M>::kOffW + tid * 16;
#pragma unroll
            for (int ky = 0; ky < 8; ++ky)
                *reinterpret_cast<uint4*>(slot + ky * (kSamplers * 16)) = __ldg(reinterpret_cast<const uint4*>(pc[0].w) + ky);
            pc[0].ws = smem_u32(slot);
        }

        const int n_rects = a.n_frames * nv, per_item = 2 * g.eye_pitch <= kSlotBytes ? 2 : 1;  // as the producer decides
        auto item_loop = [&](auto rects_tag, int n_items) {
            constexpr int EYES = decltype(rects_tag)::value;  // rectangles of an item
#pragma unroll 1
            for (int it = 0; it < n_items; ++it) {
                mbar_wait(s_full + st * 8, ph);
                const uint32_t buf = s_stage + st * kSlotBytes;
                const int o = n & (kOB - 1);
                const uint32_t ob = outp + o * kOutItemBytes;
#pragma unroll
                for (int v = 0; v < EYES; ++v) {
                    uint32_t word[kPx];
#pragma unroll
                    for (int k = 0; k < kPx; ++k) {
                        const uint32_t r = M::sample(buf + v * g.eye_pitch, pc[k], (uint32_t)g.pitch);
                        word[k] = __byte_perm(r, __shfl_down_sync(0xffffffffu, r, 1), out_sel);
                    }
                    // (after the first rectangle's sampling, which does not need the out buffer yet)
                    if (v == 0 && n >= kOB) mbar_wait(s_oempty + o * 8, (uint32_t)(n / kOB + 1) & 1u);  // store n - kOB has read out[o]
                    if (flags & 1u) {
#pragma unroll
                        for (int k = 0; k < kPx; ++k) sts32(ob + v * kOutTileBytes + k * (kTileW * 3), word[k]);
                    }
                }
                fence_proxy_async();
                __syncwarp();
                if (flags & 2u) mbar_arrive(s_ofull + o * 8);  // this warp's rows of the item are in out[o]; it has left the slot
                ++n;
                if (++st == kSlots) { st = 0; ph ^= 1u; }
            }
        };
        if (per_item == 2 && n_rects > 1) {
            item_loop(std::integral_constant<int, 2>{}, n_rects >> 1);
            if (n_rects & 1) item_loop(std::integral_constant<int, 1>{}, 1);
        } else {
            item_loop(std::integral_constant<int, 1>{}, n_rects);
        }
    }
    // ---- drain: per-pixel gather of the noted tiles (sampling warps only: named barrier 1) ----
    if (n_slow == 0 && u >= sp.n_units) break;  // the common case: nothing noted
    asm volatile("bar.sync 1, %0;" ::"n"(kSamplers) : "memory");
    for (int i = 0; i < n_slow; ++i) {
        const int2 gt = s_slow[i];
        const int4 hdr = packed_header_raw(a.view[gt.x].packed, gt.y);
        Entries<kPx> ev;
        load_packed_entries<M>(a.view[gt.x].packed, sp.n_tiles, gt.y, tid, ev.e);
        const TileHdr h = decode_header(hdr);
        gather_tile<M>(a, sp, gt.x, gt.y, nv, (h.flags & kHdrPackable) != 0, h.mnx, h.mny, ev);
    }
    if (u >= sp.n_units) break;
    asm volatile("bar.sync 1, %0;" ::"n"(kSamplers) : "memory");  // the list is rewritten by the next streaming phase
  }
}

template <class M>
static int launch_stream_mode(const RemapArgs& a, const short* tab, cudaStream_t st) {
    const int n_groups = a.share_map ? 1 : a.n_views;
    if (a.n_frames > 0x7fff) return VR180_ERR_UNSUPPORTED;  // an item's two frame indices travel in one int
    const TmaMaps* tm = tma_maps_for(a, M::kInterp, M::kRowsMin, M::kTileH, 1);
    if (!tm) return VR180_ERR_UNSUPPORTED;
    int dev = 0;
    const int rc = max_dyn_smem_once<k_warp_stream<M>>(SLay<M>::kSmemBytes, dev);
    if (rc != VR180_OK) return rc;
    static std::atomic<int> sm_count[64];
    int sms = dev < 64 ? sm_count[dev].load(std::memory_order_acquire) : 0;
    if (!sms) {
        VR180_CUDA(cudaDeviceGetAttribute(&sms, cudaDevAttrMultiProcessorCount, dev));
        if (dev < 64) sm_count[dev].store(sms, std::memory_order_release);
    }
    StreamParams sp;
    memset(&sp, 0, sizeof(sp));
    sp.tiles_x = (a.W + kTileW - 1) / kTileW;
    const long long tiles = (long long)sp.tiles_x * ((a.H + M::kTileH - 1) / M::kTileH);
    if (tiles * n_groups > 0x7fffffffLL) return VR180_ERR_UNSUPPORTED;
    sp.n_tiles = (int)tiles;
    sp.n_units = (int)(tiles * n_groups);
    sp.zero_border = zero_border(a);
    sp.tab = tab;
    const int forced = g_debug_stream_grid.load(std::memory_order_relaxed);  // vr180_debug_set(3, n): tests
    int grid = forced > 0 ? forced : sms * kStreamCtas;
    if (grid > sp.n_units) grid = sp.n_units;
    k_warp_stream<M><<<grid, kThreads, SLay<M>::kSmemBytes, st>>>(a, sp, *tm);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    VR180_CUDA(cudaGetLastError());
    return VR180_OK;
}

}  // namespace tiled

// Eligibility is decided by the caller (launch_remap_tiled: 3 channels, aligned buffers, every map group with a packed LUT
// of this interpolation, no per-frame radius).
int launch_remap_stream(const RemapArgs& a, int interp, const short* weight_tab, cudaStream_t st) {
    using namespace tiled;
    if (interp == VR180_INTER_NEAREST) return launch_stream_mode<Nearest>(a, nullptr, st);
    if (interp == VR180_INTER_LINEAR) return launch_stream_mode<LinearP>(a, nullptr, st);
    if (interp == VR180_INTER_CUBIC) return launch_stream_mode<Cubic>(a, weight_tab, st);
    if (interp == VR180_INTER_LANCZOS4) return launch_stream_mode<Lanczos4>(a, weight_tab, st);
    return VR180_ERR_UNSUPPORTED;
}

}  // namespace vr180
