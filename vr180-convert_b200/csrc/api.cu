// api.cu -- extern "C" entry points declared in include/vr180_b200.h (device-pointer API + host-buffer pipeline).
#include <algorithm>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "common.cuh"

namespace vr180 {

std::atomic<uint64_t> g_launches{0};
std::atomic<int> g_debug_frames_per_cta{0};
std::atomic<int> g_debug_tiled_flags{-1};
std::atomic<int> g_debug_max_frames_per_cta{0};
std::atomic<int> g_debug_stream_grid{0};
static thread_local std::string t_cuda_error;

void set_cuda_error(cudaError_t e, const char* where) {
    t_cuda_error = std::string(cudaGetErrorName(e)) + ": " + cudaGetErrorString(e) + " at " + where;
    cudaGetLastError();  // clear the sticky-less error state
}

const std::vector<int16_t>& host_table(int K);  // kernels.cu

}  // namespace vr180

using namespace vr180;

extern "C" {

int vr180_abi_version(void) { return VR180_ABI_VERSION; }

const char* vr180_status_string(int status) {
    switch (status) {
        case VR180_OK: return "ok";
        case VR180_ERR_INVALID_ARG: return "invalid argument";
        case VR180_ERR_UNSUPPORTED: return "unsupported configuration";
        case VR180_ERR_CUDA: return "CUDA error";
        case VR180_ERR_NO_DEVICE: return "no CUDA device";
        case VR180_ERR_CHAIN: return "malformed chain descriptor";
        case VR180_ERR_NOMEM: return "out of memory";
        default: return "unknown status";
    }
}

const char* vr180_last_cuda_error(void) { return t_cuda_error.c_str(); }

int vr180_device_info(int device, char* name, size_t name_len, int* sm_count, int* cc_major, int* cc_minor) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) {
        cudaGetLastError();
        return 0;
    }
    if (device >= 0 && device < n) {
        cudaDeviceProp prop;
        if (cudaGetDeviceProperties(&prop, device) == cudaSuccess) {
            if (name && name_len) {
                strncpy(name, prop.name, name_len - 1);
                name[name_len - 1] = 0;
            }
            if (sm_count) *sm_count = prop.multiProcessorCount;
            if (cc_major) *cc_major = prop.major;
            if (cc_minor) *cc_minor = prop.minor;
        }
    }
    return n;
}

uint64_t vr180_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

/* test hook: the host-built OpenCV weight tables (K = 4 cubic, K = 8 lanczos4), 1024*K*K int16 */
int vr180_debug_weight_table(int K, int16_t* out) {
    if ((K != 4 && K != 8) || !out) return VR180_ERR_INVALID_ARG;
    const auto& t = host_table(K);
    memcpy(out, t.data(), t.size() * sizeof(int16_t));
    return VR180_OK;
}

/* test / profiling hook: what 0 = frames per CTA of the tiled kernel (0 = automatic), 1 = VR180_TILED_DEBUG flags
   (-1 = from the environment), 2 = cap of the automatic frames-per-CTA choice (0 = default).  Returns the previous value. */
int vr180_debug_set(int what, int value) {
    if (what == 0) return g_debug_frames_per_cta.exchange(value < 0 ? 0 : value);
    if (what == 1) return g_debug_tiled_flags.exchange(value);
    if (what == 2) return g_debug_max_frames_per_cta.exchange(value < 0 ? 0 : value);
    if (what == 3) return g_debug_stream_grid.exchange(value < 0 ? 0 : value);
    return VR180_ERR_INVALID_ARG;
}

int vr180_build_map(const vr180_chain_t* chain, int out_w, int out_h, float* xmap_dev, float* ymap_dev,
                    int64_t map_pitch, void* stream) {
    if (!chain || !xmap_dev || !ymap_dev || out_w <= 0 || out_h <= 0 || map_pitch < out_w) return VR180_ERR_INVALID_ARG;
    const int rc = validate_chain(chain);
    if (rc != VR180_OK) return rc;
    DeviceGuard g(xmap_dev);
    if (!g.ok) return VR180_ERR_INVALID_ARG;
    return launch_build_map(chain, out_w, out_h, xmap_dev, ymap_dev, map_pitch, (cudaStream_t)stream);
}

int vr180_pack_lut(const float* xmap_dev, const float* ymap_dev, int64_t map_pitch, int out_w, int out_h,
                   int32_t* fixed_dev, int64_t fixed_pitch, void* stream) {
    if (!xmap_dev || !ymap_dev || !fixed_dev || out_w <= 0 || out_h <= 0 || map_pitch < out_w || fixed_pitch < out_w)
        return VR180_ERR_INVALID_ARG;
    DeviceGuard g(fixed_dev);
    if (!g.ok) return VR180_ERR_INVALID_ARG;
    return launch_pack_lut(xmap_dev, ymap_dev, map_pitch, out_w, out_h, fixed_dev, fixed_pitch, (cudaStream_t)stream);
}

size_t vr180_packed_lut_bytes(int out_w, int out_h, int interpolation) {
    if (out_w <= 0 || out_h <= 0) return 0;
    return packed_lut_bytes(out_w, out_h, interpolation);
}

int vr180_pack_lut_tiles(const float* xmap_dev, const float* ymap_dev, int64_t map_pitch, int out_w, int out_h,
                         int interpolation, void* packed_dev, void* stream) {
    if (!xmap_dev || !ymap_dev || !packed_dev || out_w <= 0 || out_h <= 0 || map_pitch < out_w) return VR180_ERR_INVALID_ARG;
    if (packed_lut_bytes(out_w, out_h, interpolation) == 0) return VR180_ERR_UNSUPPORTED;
    DeviceGuard g(packed_dev);
    if (!g.ok) return VR180_ERR_INVALID_ARG;
    return launch_pack_lut_tiles(xmap_dev, ymap_dev, map_pitch, out_w, out_h, interpolation, packed_dev, (cudaStream_t)stream);
}

int vr180_remap(const vr180_remap_params_t* params, void* stream) {
    if (!params || !params->dst) return VR180_ERR_INVALID_ARG;
    DeviceGuard g(params->dst);
    if (!g.ok) return VR180_ERR_INVALID_ARG;
    return launch_remap(params, nullptr, (cudaStream_t)stream);
}

int vr180_remap_ex(const vr180_remap_params_t* params, const double border_scalar[4], void* stream) {
    if (!params || !params->dst) return VR180_ERR_INVALID_ARG;
    DeviceGuard g(params->dst);
    if (!g.ok) return VR180_ERR_INVALID_ARG;
    return launch_remap(params, border_scalar, (cudaStream_t)stream);
}

int vr180_anaglyph(const uint8_t* sbs_dev, int64_t sbs_pitch, int64_t sbs_frame_stride, int eye_w, int h, int n_frames,
                   uint8_t* out_dev, int64_t out_pitch, int64_t out_frame_stride, void* stream) {
    if (!sbs_dev || !out_dev || eye_w <= 0 || h <= 0 || n_frames < 0 || sbs_pitch < (int64_t)eye_w * 6 ||
        out_pitch < (int64_t)eye_w * 3)
        return VR180_ERR_INVALID_ARG;
    DeviceGuard g(out_dev);
    if (!g.ok) return VR180_ERR_INVALID_ARG;
    return launch_anaglyph(sbs_dev, sbs_pitch, sbs_frame_stride, eye_w, eye_w, h, n_frames, out_dev, out_pitch,
                           out_frame_stride, (cudaStream_t)stream);
}

int vr180_transform_points(const vr180_chain_t* chain, int64_t n, const double* x_dev, const double* y_dev,
                           double* out_x_dev, double* out_y_dev, double* out_v3_dev, void* stream) {
    if (!chain || n < 0 || !x_dev || !y_dev || (!out_v3_dev && !(out_x_dev && out_y_dev))) return VR180_ERR_INVALID_ARG;
    const int rc = validate_chain(chain);
    if (rc != VR180_OK) return rc;
    DeviceGuard g(x_dev);
    if (!g.ok) return VR180_ERR_INVALID_ARG;
    return launch_transform_points(chain, n, x_dev, y_dev, out_x_dev, out_y_dev, out_v3_dev, (cudaStream_t)stream);
}

int vr180_get_radius(const vr180_image_t* views, int n_views, int n_frames, double threshold, int32_t* transitions_dev,
                     double* radius_dev, void* stream) {
    if (!views || (!transitions_dev && !radius_dev)) return VR180_ERR_INVALID_ARG;
    DeviceGuard g(transitions_dev ? (const void*)transitions_dev : (const void*)radius_dev);
    if (!g.ok) return VR180_ERR_INVALID_ARG;
    return launch_get_radius(views, n_views, n_frames, threshold, transitions_dev, radius_dev, (cudaStream_t)stream);
}

/* ---------------------------------------------------------------------------------------------------------
 * pinned host memory helpers
 * ------------------------------------------------------------------------------------------------------- */
int vr180_host_alloc(size_t bytes, void** out) {
    if (!out) return VR180_ERR_INVALID_ARG;
    VR180_CUDA(cudaHostAlloc(out, bytes ? bytes : 1, cudaHostAllocPortable));
    return VR180_OK;
}
int vr180_host_free(void* p) {
    if (p) VR180_CUDA(cudaFreeHost(p));
    return VR180_OK;
}
int vr180_host_register(void* p, size_t bytes) {
    if (!p) return VR180_ERR_INVALID_ARG;
    VR180_CUDA(cudaHostRegister(p, bytes, cudaHostRegisterPortable));
    return VR180_OK;
}
int vr180_host_unregister(void* p) {
    if (!p) return VR180_ERR_INVALID_ARG;
    VR180_CUDA(cudaHostUnregister(p));
    return VR180_OK;
}

}  // extern "C"
