// common.cuh -- host-side helpers shared by the translation units of libvr180_b200.so
#pragma once
#include <cuda_runtime.h>

#include <atomic>
#include <cstdint>
#include <cstdio>
#include <cstring>

#include "../../include/vr180_b200.h"

namespace vr180 {

extern std::atomic<uint64_t> g_launches;
// test / profiling hooks (vr180_debug_set): 0 = automatic
extern std::atomic<int> g_debug_frames_per_cta;  // frames per CTA of the tiled kernel (tests force long frame loops on small outputs)
extern std::atomic<int> g_debug_tiled_flags;     // -1 = take VR180_TILED_DEBUG from the environment
extern std::atomic<int> g_debug_max_frames_per_cta;  // cap of the automatic choice (0 = default)
extern std::atomic<int> g_debug_stream_grid;  // CTAs of the streaming kernel (0 = 3 per SM): tests force many tiles per CTA
void set_cuda_error(cudaError_t e, const char* where);

#define VR180_CUDA(call)                                  \
    do {                                                  \
        cudaError_t e__ = (call);                         \
        if (e__ != cudaSuccess) {                         \
            ::vr180::set_cuda_error(e__, #call);          \
            return VR180_ERR_CUDA;                        \
        }                                                 \
    } while (0)

// Select the device that owns `ptr` for the duration of a call (this library links its own static cudart, whose
// current-device state is independent of the caller's).
struct DeviceGuard {
    int prev = -1;
    int dev = -1;
    bool ok = false;
    explicit DeviceGuard(const void* ptr) {
        cudaPointerAttributes a;
        if (cudaPointerGetAttributes(&a, ptr) != cudaSuccess || a.type != cudaMemoryTypeDevice) {
            cudaGetLastError();
            return;
        }
        dev = a.device;
        if (cudaGetDevice(&prev) != cudaSuccess) return;
        if (prev != dev && cudaSetDevice(dev) != cudaSuccess) return;
        ok = true;
    }
    explicit DeviceGuard(int device) {
        dev = device;
        if (cudaGetDevice(&prev) != cudaSuccess) return;
        if (prev != dev && cudaSetDevice(dev) != cudaSuccess) return;
        ok = true;
    }
    ~DeviceGuard() {
        if (ok && prev != dev && prev >= 0) cudaSetDevice(prev);
    }
};

// kernel-side description of one vr180_remap call (kernels.cu fills it, kernels.cu / tiled.cu consume it)
struct ViewArgs {
    const uint8_t* src;
    int rows, cols;
    long long pitch, frame_stride;
    int map_kind;
    int chain_idx;  // which of the two kernel-parameter chains
    const float* xmap;
    const float* ymap;
    const int2* fixed;
    long long map_pitch;
    const double* radius_dev;
    int dst_x_offset;
    const void* packed;  // tile-packed LUT built for THIS interpolation (tiled kernel only), or nullptr
};

struct RemapArgs {
    ViewArgs view[2];
    int n_views, n_frames, share_map;
    int W, H;
    int border_mode;
    uint8_t bv[4];
    int depth;  // VR180_DEPTH_8U / VR180_DEPTH_16U, sources and destination alike (fills the padding before dst)
    uint8_t* dst;
    long long dst_pitch, dst_frame_stride;
    int frames_per_cta;
};

// What 16-bit requests add: a trailing kernel parameter, so that RemapArgs keeps its size and the parameters after it
// their offsets in the 8-bit kernels.
struct Remap16 {
    float cval[4];      // border colour saturated to 16 bits (exact in float)
    const float* ftab;  // float weight table of CUBIC / LANCZOS4 (generic kernel)
};

inline int depth_bytes(int depth) { return depth == VR180_DEPTH_16U ? 2 : 1; }

// internal launchers (kernels.cu); the device is already selected by the caller
int launch_build_map(const vr180_chain_t* chain, int out_w, int out_h, float* xmap, float* ymap, int64_t pitch,
                     cudaStream_t st);
int launch_pack_lut(const float* xmap, const float* ymap, int64_t map_pitch, int out_w, int out_h, int32_t* fixed,
                    int64_t fixed_pitch, cudaStream_t st);
// border_scalar: the cv::Scalar border colour, saturated to the depth here; nullptr = p->border_value
int launch_remap(const vr180_remap_params_t* p, const double* border_scalar, cudaStream_t st);
size_t packed_lut_bytes(int out_w, int out_h, int interp);  // tiled.cu; 0 = interpolation without a tiled mode
int launch_pack_lut_tiles(const float* xmap, const float* ymap, int64_t map_pitch, int out_w, int out_h, int interp,
                          void* packed, cudaStream_t st);
int launch_remap_tiled(const RemapArgs& a, int channels, int interp, const vr180_chain_t& c0, const vr180_chain_t& c1,
                       const short* weight_tab, cudaStream_t st);  // tiled.cu; VR180_ERR_UNSUPPORTED = not eligible, use the generic kernel
int launch_get_radius(const vr180_image_t* views, int n_views, int n_frames, double threshold, int32_t* transitions,
                      double* radius, cudaStream_t st);
int validate_chain(const vr180_chain_t* c);
int launch_anaglyph(const uint8_t* sbs, int64_t pitch, int64_t frame_stride, int W, int right_col, int H, int n_frames,
                    uint8_t* out, int64_t out_pitch, int64_t out_frame_stride, cudaStream_t st);  // right eye at column right_col
int launch_transform_points(const vr180_chain_t* chain, long long n, const double* x, const double* y, double* ox,
                            double* oy, double* v3, cudaStream_t st);

}  // namespace vr180
