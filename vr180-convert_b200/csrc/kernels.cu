// kernels.cu -- sm_100a kernels of the reprojection hot path and their launchers.
//
//   k_build_map   analytic float64 chain -> float32 maps        (get_map, remapper.py:23-59)
//   k_pack_lut    float32 maps -> cv2-exact fixed-point LUT     (cv::remap's internal convertMaps step)
//   k_remap       [analytic | float2 | fixed LUT] coordinates -> OpenCV-exact gather, both eyes written
//                 straight into the SBS frame, a batch of frames per launch
//                                                                (cv.remap remapper.py:388-398 + concatenate :518)
//   k_get_radius  black-pixel transition scan                    (get_radius, transformer.py:108-140)
#include <cmath>
#include <cstdlib>
#include <mutex>
#include <vector>

#include "chain.cuh"
#include "common.cuh"
#include "sampler.cuh"
#include "tables.cuh"

namespace vr180 {

// ---------------------------------------------------------------------------------------------------------
// weight tables (device copies, one per device, filled on first use)
// ---------------------------------------------------------------------------------------------------------
__device__ __align__(16) short g_tab_cubic[1024 * 16];
__device__ __align__(16) short g_tab_lanczos[1024 * 64];

static std::once_flag g_tab_host_once;
static std::vector<int16_t> g_tab_cubic_host, g_tab_lanczos_host;
static std::mutex g_tab_mutex;
static bool g_tab_on_device[64] = {};

const std::vector<int16_t>& host_table(int K) {
    std::call_once(g_tab_host_once, [] {
        g_tab_cubic_host = build_weight_table(4);
        g_tab_lanczos_host = build_weight_table(8);
    });
    return K == 4 ? g_tab_cubic_host : g_tab_lanczos_host;
}

static int ensure_tables(cudaStream_t st) {
    int dev = 0;
    VR180_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> lock(g_tab_mutex);
    if (dev < 64 && g_tab_on_device[dev]) return VR180_OK;
    const auto& c = host_table(4);
    const auto& l = host_table(8);
    // synchronous copies on purpose: happens once per device, and later launches on any stream must see them
    (void)st;
    VR180_CUDA(cudaMemcpyToSymbol(g_tab_cubic, c.data(), c.size() * sizeof(int16_t)));
    VR180_CUDA(cudaMemcpyToSymbol(g_tab_lanczos, l.data(), l.size() * sizeof(int16_t)));
    if (dev < 64) g_tab_on_device[dev] = true;
    return VR180_OK;
}

// The float tables of 16-bit CUBIC (1024 x 16) and LANCZOS4 (1024 x 64) in device global memory, built on the host once
// and uploaded once per device; they live as long as the process.
static const float* g_ftab_dev[64][2] = {};

static int ensure_float_table(int K, const float** out) {
    int dev = 0;
    VR180_CUDA(cudaGetDevice(&dev));
    if (dev >= 64) return VR180_ERR_UNSUPPORTED;
    std::lock_guard<std::mutex> lock(g_tab_mutex);
    const float*& slot = g_ftab_dev[dev][K == 4 ? 0 : 1];
    if (!slot) {
        const std::vector<float> t = build_float_table(K);
        void* p = nullptr;
        VR180_CUDA(cudaMalloc(&p, t.size() * sizeof(float)));
        const cudaError_t e = cudaMemcpy(p, t.data(), t.size() * sizeof(float), cudaMemcpyHostToDevice);  // once
        if (e != cudaSuccess) {
            cudaFree(p);
            set_cuda_error(e, "cudaMemcpy(float weight table)");
            return VR180_ERR_CUDA;
        }
        slot = static_cast<const float*>(p);
    }
    *out = slot;
    return VR180_OK;
}

// ---------------------------------------------------------------------------------------------------------
// k_build_map
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_build_map(const __grid_constant__ vr180_chain_t chain, int W, int H,
                                                   float* __restrict__ xmap, float* __restrict__ ymap, long long pitch) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int j = blockIdx.y * blockDim.y + threadIdx.y;
    if (i >= W || j >= H) return;
    double xs, ys;
    eval_chain(chain, i, j, xs, ys);
    xmap[(long long)j * pitch + i] = __double2float_rn(xs);  // astype(np.float32), remapper.py:58
    ymap[(long long)j * pitch + i] = __double2float_rn(ys);
}

int launch_build_map(const vr180_chain_t* chain, int W, int H, float* xmap, float* ymap, int64_t pitch, cudaStream_t st) {
    dim3 block(32, 8), grid((W + 31) / 32, (H + 7) / 8);
    k_build_map<<<grid, block, 0, st>>>(*chain, W, H, xmap, ymap, (long long)pitch);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    VR180_CUDA(cudaGetLastError());
    return VR180_OK;
}

// ---------------------------------------------------------------------------------------------------------
// k_pack_lut
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_pack_lut(const float* __restrict__ xmap, const float* __restrict__ ymap,
                                                  long long map_pitch, int W, int H, int2* __restrict__ fixed,
                                                  long long fixed_pitch) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int j = blockIdx.y * blockDim.y + threadIdx.y;
    if (i >= W || j >= H) return;
    const float mx = __ldg(xmap + (long long)j * map_pitch + i), my = __ldg(ymap + (long long)j * map_pitch + i);
    fixed[(long long)j * fixed_pitch + i] = make_int2(quantise(mx), quantise(my));
}

int launch_pack_lut(const float* xmap, const float* ymap, int64_t map_pitch, int W, int H, int32_t* fixed,
                    int64_t fixed_pitch, cudaStream_t st) {
    dim3 block(32, 8), grid((W + 31) / 32, (H + 7) / 8);
    k_pack_lut<<<grid, block, 0, st>>>(xmap, ymap, (long long)map_pitch, W, H, reinterpret_cast<int2*>(fixed),
                                       (long long)fixed_pitch);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    VR180_CUDA(cudaGetLastError());
    return VR180_OK;
}

// ---------------------------------------------------------------------------------------------------------
// k_remap
// ---------------------------------------------------------------------------------------------------------
template <int C, int INTERP>
__device__ __forceinline__ void sample_and_store(const Src& s, int sx, int sy, float mx, float my, int border_mode,
                                                 const uint8_t* bv, uint8_t* __restrict__ out) {
    int px[C];
    if (INTERP == VR180_INTER_NEAREST) sample_nearest<C>(s, mx, my, border_mode, bv, px);
    else if (INTERP == VR180_INTER_LINEAR) sample_linear<C>(s, sx, sy, border_mode, bv, px);
    else if (INTERP == VR180_INTER_CUBIC) sample_tab<C, 4>(s, sx, sy, g_tab_cubic, border_mode, bv, px);
    else sample_tab<C, 8>(s, sx, sy, g_tab_lanczos, border_mode, bv, px);
#pragma unroll
    for (int c = 0; c < C; ++c) out[c] = (uint8_t)px[c];
}

template <int C, int INTERP>
__device__ __forceinline__ void sample_and_store16(const Src& s, int sx, int sy, float mx, float my, int border_mode,
                                                   const float* cval, const float* ftab, uint16_t* __restrict__ out) {
    int px[C];
    if (INTERP == VR180_INTER_NEAREST) sample16_nearest<C>(s, mx, my, border_mode, cval, px);
    else if (INTERP == VR180_INTER_LINEAR) sample16_linear<C>(s, sx, sy, border_mode, cval, px);
    else if (INTERP == VR180_INTER_CUBIC) sample16_tab<C, 4>(s, sx, sy, ftab, border_mode, cval, px);
    else sample16_tab<C, 8>(s, sx, sy, ftab, border_mode, cval, px);
#pragma unroll
    for (int c = 0; c < C; ++c) out[c] = (uint16_t)px[c];
}

// One thread = one output pixel of the tile; coordinates are evaluated once and reused for every frame of the
// CTA's frame chunk (and for both eyes when they share a map).  grid = (tiles_x, tiles_y, frame_chunks).
// T = uint8_t (OpenCV's fixed-point 8-bit arithmetic) or uint16_t (its float arithmetic for other depths).
template <typename T, int C, int INTERP>
__global__ void __launch_bounds__(256) k_remap(const __grid_constant__ RemapArgs a,
                                               const __grid_constant__ vr180_chain_t chain0,
                                               const __grid_constant__ vr180_chain_t chain1,
                                               const __grid_constant__ Remap16 x16) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int j = blockIdx.y * blockDim.y + threadIdx.y;
    if (i >= a.W || j >= a.H) return;
    const int f0 = blockIdx.z * a.frames_per_cta;
    const int f1 = min(a.n_frames, f0 + a.frames_per_cta);
    const int n_groups = a.share_map ? 1 : a.n_views;

    for (int g = 0; g < n_groups; ++g) {
        const ViewArgs& mv = a.view[g];  // the view whose map drives this group
        const int v_begin = g, v_end = a.share_map ? a.n_views : g + 1;
        float mx = 0.f, my = 0.f;
        int sx = 0, sy = 0;
        double nx = 0.0, ny = 0.0, cx = 0.0, cy = 0.0;
        const bool per_frame_radius = (mv.map_kind == VR180_MAPSRC_ANALYTIC) && (mv.radius_dev != nullptr);
        if (mv.map_kind == VR180_MAPSRC_ANALYTIC) {
            const vr180_chain_t& ch = mv.chain_idx ? chain1 : chain0;
            if (per_frame_radius) {
                eval_chain_normalised(ch, i, j, nx, ny);
                cx = ch.ops[ch.n_ops - 1].p[2];
                cy = ch.ops[ch.n_ops - 1].p[3];
            } else {
                double xs, ys;
                eval_chain(ch, i, j, xs, ys);
                mx = __double2float_rn(xs);
                my = __double2float_rn(ys);
            }
        } else if (mv.map_kind == VR180_MAPSRC_FLOAT2) {
            mx = __ldg(mv.xmap + (long long)j * mv.map_pitch + i);
            my = __ldg(mv.ymap + (long long)j * mv.map_pitch + i);
        } else {
            const int2 q = __ldg(mv.fixed + (long long)j * mv.map_pitch + i);
            sx = q.x;
            sy = q.y;
        }
        if (mv.map_kind != VR180_MAPSRC_FIXED && !per_frame_radius && INTERP != VR180_INTER_NEAREST) {
            sx = quantise(mx);
            sy = quantise(my);
        }
        for (int f = f0; f < f1; ++f) {
            if (per_frame_radius) {
                const double rad = __ldg(mv.radius_dev + f);
                mx = __double2float_rn(add_rn(mul_rn(nx, rad), cx));  // DenormalizeTransformer, transformer.py:202-203
                my = __double2float_rn(add_rn(mul_rn(ny, rad), cy));
                if (INTERP != VR180_INTER_NEAREST) {
                    sx = quantise(mx);
                    sy = quantise(my);
                }
            }
            uint8_t* drow = a.dst + (long long)f * a.dst_frame_stride + (long long)j * a.dst_pitch;
            for (int v = v_begin; v < v_end; ++v) {
                const ViewArgs& vw = a.view[v];
                Src s{vw.src + (long long)f * vw.frame_stride, vw.rows, vw.cols, vw.pitch};
                if constexpr (sizeof(T) == 1) {
                    sample_and_store<C, INTERP>(s, sx, sy, mx, my, a.border_mode, a.bv,
                                                drow + (long long)(vw.dst_x_offset + i) * C);
                } else {
                    sample_and_store16<C, INTERP>(s, sx, sy, mx, my, a.border_mode, x16.cval, x16.ftab,
                                                  reinterpret_cast<uint16_t*>(drow) + (long long)(vw.dst_x_offset + i) * C);
                }
            }
        }
    }
}

template <typename T, int C>
static void dispatch_interp(int interp, dim3 grid, dim3 block, cudaStream_t st, const RemapArgs& a,
                            const vr180_chain_t& c0, const vr180_chain_t& c1, const Remap16& x) {
    switch (interp) {
        case VR180_INTER_NEAREST: k_remap<T, C, VR180_INTER_NEAREST><<<grid, block, 0, st>>>(a, c0, c1, x); break;
        case VR180_INTER_LINEAR: k_remap<T, C, VR180_INTER_LINEAR><<<grid, block, 0, st>>>(a, c0, c1, x); break;
        case VR180_INTER_CUBIC: k_remap<T, C, VR180_INTER_CUBIC><<<grid, block, 0, st>>>(a, c0, c1, x); break;
        default: k_remap<T, C, VR180_INTER_LANCZOS4><<<grid, block, 0, st>>>(a, c0, c1, x); break;
    }
}

template <typename T>
static void dispatch_channels(int C, int interp, dim3 grid, dim3 block, cudaStream_t st, const RemapArgs& a,
                              const vr180_chain_t& c0, const vr180_chain_t& c1, const Remap16& x) {
    if (C == 3) dispatch_interp<T, 3>(interp, grid, block, st, a, c0, c1, x);
    else if (C == 1) dispatch_interp<T, 1>(interp, grid, block, st, a, c0, c1, x);
    else dispatch_interp<T, 4>(interp, grid, block, st, a, c0, c1, x);
}

// saturate_cast<uchar / ushort>(double): round half to even, clamp (NaN -> 0, as cvRound gives INT_MIN)
static int saturate_scalar(double v, int maxval) {
    if (!(v == v)) return 0;
    const double r = std::nearbyint(v);
    return r <= 0.0 ? 0 : (r >= (double)maxval ? maxval : (int)r);
}

int validate_chain(const vr180_chain_t* c) {
    if (!c || c->n_ops < 1 || c->n_ops > VR180_MAX_OPS) return VR180_ERR_CHAIN;
    for (int k = 0; k < c->n_ops; ++k) {
        const vr180_op_t& op = c->ops[k];
        if (op.code < VR180_OP_NORMALIZE || op.code > VR180_OP_ROT3) return VR180_ERR_CHAIN;
        if (op.code == VR180_OP_POLY && (op.iparam < 0 || op.iparam > VR180_MAX_OP_PARAMS)) return VR180_ERR_CHAIN;
        if ((op.code == VR180_OP_FISHEYE_ENC || op.code == VR180_OP_FISHEYE_DEC) &&
            (op.iparam < VR180_MAP_RECTILINEAR || op.iparam > VR180_MAP_ORTHOGRAPHIC))
            return VR180_ERR_CHAIN;
    }
    return VR180_OK;
}

int launch_remap(const vr180_remap_params_t* p, const double* border_scalar, cudaStream_t st) {
    if (p->n_views < 1 || p->n_views > 2 || p->n_frames < 0 || p->out_w <= 0 || p->out_h <= 0 || !p->dst)
        return VR180_ERR_INVALID_ARG;
    if (p->n_frames == 0) return VR180_OK;
    const int interp = p->interpolation;
    if (interp != VR180_INTER_NEAREST && interp != VR180_INTER_LINEAR && interp != VR180_INTER_CUBIC &&
        interp != VR180_INTER_LANCZOS4)
        return VR180_ERR_UNSUPPORTED;
    if (p->border_mode < VR180_BORDER_CONSTANT || p->border_mode > VR180_BORDER_REFLECT_101) return VR180_ERR_UNSUPPORTED;
    const int C = p->view[0].src.channels;
    if (C != 1 && C != 3 && C != 4) return VR180_ERR_UNSUPPORTED;
    const int depth = p->view[0].src.depth;
    if (depth != VR180_DEPTH_8U && depth != VR180_DEPTH_16U) return VR180_ERR_UNSUPPORTED;
    if (depth == VR180_DEPTH_16U && (((uintptr_t)p->dst | (uintptr_t)p->dst_pitch | (uintptr_t)p->dst_frame_stride) & 1))
        return VR180_ERR_INVALID_ARG;  // uint16 elements must be 2-byte aligned

    RemapArgs a;
    memset(&a, 0, sizeof(a));
    static const vr180_chain_t kEmpty = {};
    const vr180_chain_t* chains[2] = {&kEmpty, &kEmpty};
    for (int v = 0; v < p->n_views; ++v) {
        const vr180_view_t& vw = p->view[v];
        if (!vw.src.data || vw.src.rows <= 0 || vw.src.cols <= 0 || vw.src.channels != C) return VR180_ERR_INVALID_ARG;
        if (vw.src.depth != depth) return VR180_ERR_UNSUPPORTED;
        if (depth == VR180_DEPTH_16U &&
            (((uintptr_t)vw.src.data | (uintptr_t)vw.src.pitch | (uintptr_t)vw.src.frame_stride) & 1))
            return VR180_ERR_INVALID_ARG;
        ViewArgs& o = a.view[v];
        o.src = vw.src.data;
        o.rows = vw.src.rows;
        o.cols = vw.src.cols;
        o.pitch = vw.src.pitch;
        o.frame_stride = vw.src.frame_stride;
        o.map_kind = vw.map.kind;
        o.chain_idx = v;
        o.dst_x_offset = vw.dst_x_offset;
        if (v == 1 && p->share_map) continue;  // coordinates come from view 0
        switch (vw.map.kind) {
            case VR180_MAPSRC_ANALYTIC: {
                const int rc = validate_chain(vw.map.chain);
                if (rc != VR180_OK) return rc;
                if (vw.map.radius_dev && vw.map.chain->ops[vw.map.chain->n_ops - 1].code != VR180_OP_DENORMALIZE)
                    return VR180_ERR_CHAIN;
                chains[v] = vw.map.chain;
                o.radius_dev = vw.map.radius_dev;
                break;
            }
            case VR180_MAPSRC_PACKED:  // the float32 maps + (tiled kernel, same interpolation only) their packed tiles
                if (!vw.map.packed) return VR180_ERR_INVALID_ARG;
                if (vw.map.packed_interpolation == interp) o.packed = vw.map.packed;
                o.map_kind = VR180_MAPSRC_FLOAT2;
                [[fallthrough]];
            case VR180_MAPSRC_FLOAT2:
                if (!vw.map.xmap || !vw.map.ymap || vw.map.map_pitch < p->out_w) return VR180_ERR_INVALID_ARG;
                o.xmap = vw.map.xmap;
                o.ymap = vw.map.ymap;
                o.map_pitch = vw.map.map_pitch;
                break;
            case VR180_MAPSRC_FIXED:
                if (!vw.map.fixed || vw.map.map_pitch < p->out_w) return VR180_ERR_INVALID_ARG;
                if (interp == VR180_INTER_NEAREST) return VR180_ERR_UNSUPPORTED;  // LUT holds x*32, NEAREST rounds x
                o.fixed = reinterpret_cast<const int2*>(vw.map.fixed);
                o.map_pitch = vw.map.map_pitch;
                break;
            default: return VR180_ERR_INVALID_ARG;
        }
    }
    a.n_views = p->n_views;
    a.n_frames = p->n_frames;
    a.share_map = (p->n_views == 2 && p->share_map) ? 1 : 0;
    a.W = p->out_w;
    a.H = p->out_h;
    a.border_mode = p->border_mode;
    a.depth = depth;
    Remap16 x16;
    memset(&x16, 0, sizeof(x16));
    for (int c = 0; c < 4; ++c) {
        a.bv[c] = border_scalar ? (uint8_t)saturate_scalar(border_scalar[c], 255) : p->border_value[c];
        x16.cval[c] = border_scalar ? (float)saturate_scalar(border_scalar[c], 65535) : (float)p->border_value[c];
    }
    a.dst = p->dst;
    a.dst_pitch = p->dst_pitch;
    a.dst_frame_stride = p->dst_frame_stride;

    if (interp == VR180_INTER_CUBIC || interp == VR180_INTER_LANCZOS4) {
        const int rc = depth == VR180_DEPTH_16U ? ensure_float_table(interp == VR180_INTER_CUBIC ? 4 : 8, &x16.ftab)
                                                : ensure_tables(st);
        if (rc != VR180_OK) return rc;
    }

    // fast path: tiled, smem-staged kernel (tiled.cu); VR180_DISABLE_TILED=1 forces the generic gather (A/B tests)
    static const bool tiled_off = [] { const char* e = getenv("VR180_DISABLE_TILED"); return e && *e == '1'; }();
    if (!tiled_off) {
        const short* weight_tab = nullptr;
        if (interp == VR180_INTER_CUBIC) VR180_CUDA(cudaGetSymbolAddress((void**)&weight_tab, g_tab_cubic));
        if (interp == VR180_INTER_LANCZOS4) VR180_CUDA(cudaGetSymbolAddress((void**)&weight_tab, g_tab_lanczos));
        const int rc = launch_remap_tiled(a, C, interp, *chains[0], *chains[1], weight_tab, x16, st);
        if (rc != VR180_ERR_UNSUPPORTED) return rc;
    }

    // frames per CTA: amortise the coordinate evaluation over up to 16 frames, but keep >= ~4 waves of CTAs
    dim3 block(32, 8);
    const int tiles = ((a.W + 31) / 32) * ((a.H + 7) / 8);
    int fpc = 16;
    while (fpc > 1 && (long long)tiles * ((a.n_frames + fpc - 1) / fpc) < 148LL * 8 * 4) fpc >>= 1;
    a.frames_per_cta = fpc;
    dim3 grid((a.W + 31) / 32, (a.H + 7) / 8, (a.n_frames + fpc - 1) / fpc);
    if (grid.z > 65535) return VR180_ERR_UNSUPPORTED;

    if (depth == VR180_DEPTH_16U) dispatch_channels<uint16_t>(C, interp, grid, block, st, a, *chains[0], *chains[1], x16);
    else dispatch_channels<uint8_t>(C, interp, grid, block, st, a, *chains[0], *chains[1], x16);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    VR180_CUDA(cudaGetLastError());
    return VR180_OK;
}

// ---------------------------------------------------------------------------------------------------------
// k_get_radius: one CTA per frame; warp-shuffle min / max reduction of the transition indices
// ---------------------------------------------------------------------------------------------------------
struct RadiusArgs {
    vr180_image_t view[2];
    int n_views;
    double threshold;
};

template <typename T>
__device__ __forceinline__ bool is_black(const uint8_t* __restrict__ p, int C, double threshold) {
    const T* px = reinterpret_cast<const T*>(p);
    int sum = 0;
    for (int c = 0; c < C; ++c) sum += __ldg(px + c);
    return __ddiv_rn((double)sum, (double)C) < threshold;  // np.mean(center_row, axis=-1) < threshold, transformer.py:133
}

// T: the element type of every view (uint8_t / uint16_t); pixel offsets below are in bytes
template <typename T>
__global__ void __launch_bounds__(256) k_get_radius(const __grid_constant__ RadiusArgs a, int* __restrict__ transitions,
                                                    double* __restrict__ radius) {
    __shared__ int s_pos[8], s_neg[8];
    const int f = blockIdx.x;
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    double best = -CUDART_INF;
    bool missing = false;
    for (int v = 0; v < a.n_views; ++v) {
        const vr180_image_t& im = a.view[v];
        const int C = im.channels;
        const uint8_t* base = im.data + (long long)f * im.frame_stride;
        long long step;
        int n;
        if (im.cols > im.rows) {  // centre row, transformer.py:126-127
            base += (long long)(im.rows / 2) * im.pitch;
            step = C * (long long)sizeof(T);
            n = im.cols;
        } else {  // centre column (also for square images), :128-129
            base += (long long)(im.cols / 2) * C * (long long)sizeof(T);
            step = im.pitch;
            n = im.rows;
        }
        int pos = INT_MAX, neg = -1;
        for (int k = threadIdx.x; k < n - 1; k += blockDim.x) {
            const bool b0 = is_black<T>(base + (long long)k * step, C, a.threshold);
            const bool b1 = is_black<T>(base + (long long)(k + 1) * step, C, a.threshold);
            if (!b0 && b1) pos = min(pos, k);  // np.diff(...) == +1, first index (:137)
            if (b0 && !b1) neg = max(neg, k);  // np.diff(...) == -1, last index  (:138)
        }
#pragma unroll
        for (int o = 16; o > 0; o >>= 1) {
            pos = min(pos, __shfl_xor_sync(0xffffffffu, pos, o));
            neg = max(neg, __shfl_xor_sync(0xffffffffu, neg, o));
        }
        if (lane == 0) { s_pos[warp] = pos; s_neg[warp] = neg; }
        __syncthreads();
        if (warp == 0) {
            pos = lane < (blockDim.x >> 5) ? s_pos[lane] : INT_MAX;
            neg = lane < (blockDim.x >> 5) ? s_neg[lane] : -1;
#pragma unroll
            for (int o = 4; o > 0; o >>= 1) {
                pos = min(pos, __shfl_xor_sync(0xffffffffu, pos, o));
                neg = max(neg, __shfl_xor_sync(0xffffffffu, neg, o));
            }
            if (lane == 0) {
                if (pos == INT_MAX) pos = -1;
                if (transitions) {
                    transitions[(f * a.n_views + v) * 2 + 0] = pos;
                    transitions[(f * a.n_views + v) * 2 + 1] = neg;
                }
                if (pos < 0 || neg < 0) missing = true;
                else best = fmax(best, (double)(neg - pos) / 2.0);  // (end - start) / 2, :139; max over images, remapper.py:84
            }
        }
        __syncthreads();
    }
    if (threadIdx.x == 0 && radius) radius[f] = missing ? CUDART_NAN : best;
}

int launch_get_radius(const vr180_image_t* views, int n_views, int n_frames, double threshold, int32_t* transitions,
                      double* radius, cudaStream_t st) {
    if (!views || n_views < 1 || n_views > 2 || n_frames < 0) return VR180_ERR_INVALID_ARG;
    if (n_frames == 0) return VR180_OK;
    RadiusArgs a;
    memset(&a, 0, sizeof(a));
    for (int v = 0; v < n_views; ++v) {
        if (!views[v].data || views[v].rows <= 0 || views[v].cols <= 0 || views[v].channels < 1 || views[v].channels > 4)
            return VR180_ERR_INVALID_ARG;
        if (views[v].depth != views[0].depth || (views[v].depth != VR180_DEPTH_8U && views[v].depth != VR180_DEPTH_16U))
            return VR180_ERR_UNSUPPORTED;
        if (views[v].depth == VR180_DEPTH_16U &&
            (((uintptr_t)views[v].data | (uintptr_t)views[v].pitch | (uintptr_t)views[v].frame_stride) & 1))
            return VR180_ERR_INVALID_ARG;
        a.view[v] = views[v];
    }
    a.n_views = n_views;
    a.threshold = threshold;
    if (views[0].depth == VR180_DEPTH_16U) k_get_radius<uint16_t><<<n_frames, 256, 0, st>>>(a, transitions, radius);
    else k_get_radius<uint8_t><<<n_frames, 256, 0, st>>>(a, transitions, radius);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    VR180_CUDA(cudaGetLastError());
    return VR180_OK;
}

// ---------------------------------------------------------------------------------------------------------
// k_anaglyph: the merge=True branch of apply_lr (remapper.py:485-498) on the device-resident SBS frame
// ---------------------------------------------------------------------------------------------------------
// combine = mean_c(L)[..., None] * (0, 128, 255) + mean_c(R)[..., None] * (255, 128, 0);  combine /= 255   (float64,
// one rounding per NumPy ufunc), then cv.imwrite's float64 -> uint8 conversion (round half to even, saturate).
__global__ void __launch_bounds__(256) k_anaglyph(const uint8_t* __restrict__ sbs, long long pitch, long long frame_stride,
                                                  int W, int right_col, int H, uint8_t* __restrict__ out,
                                                  long long out_pitch, long long out_frame_stride) {
    const int i = blockIdx.x * blockDim.x + threadIdx.x;
    const int j = blockIdx.y;
    if (i >= W) return;
    const uint8_t* row = sbs + (long long)blockIdx.z * frame_stride + (long long)j * pitch;
    const uint8_t* l = row + (long long)i * 3;
    const uint8_t* r = row + (long long)(right_col + i) * 3;
    const double ml = __ddiv_rn((double)(__ldg(l) + __ldg(l + 1) + __ldg(l + 2)), 3.0);  // np.mean(axis=-1)
    const double mr = __ddiv_rn((double)(__ldg(r) + __ldg(r + 1) + __ldg(r + 2)), 3.0);
    const double cl[3] = {0.0, 128.0, 255.0}, cr[3] = {255.0, 128.0, 0.0};
    uint8_t* o = out + (long long)blockIdx.z * out_frame_stride + (long long)j * out_pitch + (long long)i * 3;
#pragma unroll
    for (int c = 0; c < 3; ++c) {
        const double v = __ddiv_rn(__dadd_rn(__dmul_rn(ml, cl[c]), __dmul_rn(mr, cr[c])), 255.0);
        o[c] = (uint8_t)min(255, max(0, __double2int_rn(v)));
    }
}

int launch_anaglyph(const uint8_t* sbs, int64_t pitch, int64_t frame_stride, int W, int right_col, int H, int n_frames,
                    uint8_t* out, int64_t out_pitch, int64_t out_frame_stride, cudaStream_t st) {
    if (n_frames == 0) return VR180_OK;
    if (H > 65535 || n_frames > 65535) return VR180_ERR_UNSUPPORTED;
    dim3 grid((W + 255) / 256, H, n_frames);
    k_anaglyph<<<grid, 256, 0, st>>>(sbs, pitch, frame_stride, W, right_col, H, out, out_pitch, out_frame_stride);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    VR180_CUDA(cudaGetLastError());
    return VR180_OK;
}

// ---------------------------------------------------------------------------------------------------------
// k_transform_points: a lowered chain on arbitrary points (match_lr's pixel -> 3-D step, remapper.py:291-320)
// ---------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) k_transform_points(const __grid_constant__ vr180_chain_t chain, long long n,
                                                          const double* __restrict__ x, const double* __restrict__ y,
                                                          double* __restrict__ ox, double* __restrict__ oy,
                                                          double* __restrict__ v3) {
    const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
    if (i >= n) return;
    ChainState s;
    s.mode = MODE_XY;
    s.x = __ldg(x + i);
    s.y = __ldg(y + i);
    s.r = s.ux = s.uy = s.vx = s.vy = s.vz = 0.0;
    run_ops(chain, 0, chain.n_ops, s);
    if (v3) {  // equidistant_to_3d (transformer.py:483-508)
        to_vec3(s);
        v3[3 * i + 0] = s.vx;
        v3[3 * i + 1] = s.vy;
        v3[3 * i + 2] = s.vz;
    }
    if (ox && oy) {
        to_xy(s);
        ox[i] = s.x;
        oy[i] = s.y;
    }
}

int launch_transform_points(const vr180_chain_t* chain, long long n, const double* x, const double* y, double* ox,
                            double* oy, double* v3, cudaStream_t st) {
    if (n == 0) return VR180_OK;
    k_transform_points<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(*chain, n, x, y, ox, oy, v3);
    g_launches.fetch_add(1, std::memory_order_relaxed);
    VR180_CUDA(cudaGetLastError());
    return VR180_OK;
}

}  // namespace vr180
