/*
 * vr180_b200.h -- C ABI of the B200-native reprojection hot path of vr180-convert.
 *
 * Drop-in boundary (SURVEY.md §8b).  The reference (34j/vr180-convert v0.6.2, pure Python) has no FFI of
 * its own; the boundary is the two native calls its hot path makes:
 *
 *   (1) the NumPy float64 ufunc chain that builds the float32 maps
 *         reference: src/vr180_convert/remapper.py:23-59 (get_map),
 *                    src/vr180_convert/transformer.py:93-98 (MultiTransformer.transform) and the
 *                    transformer classes at :143-213, :268-286, :350-480, :533-604, :607-679
 *   (2) cv2.remap per eye + np.concatenate
 *         reference: src/vr180_convert/remapper.py:388-398 (cv.remap), :518 (SBS concatenate)
 *   (3) the get_radius line scan
 *         reference: src/vr180_convert/transformer.py:108-140, remapper.py:62-90
 *
 * Every entry point below replaces one of those and says which.  Conventions:
 *   - plain C structs / pointers / sizes; no C++ or torch types cross the boundary;
 *   - all `*_dev` / device-buffer pointers are CUDA device memory owned by the caller; the device-pointer
 *     entry points never allocate and are asynchronous on `stream` (a cudaStream_t passed as void*;
 *     NULL = the legacy default stream);
 *   - the launch device is derived from the destination pointer, so one process may drive several GPUs;
 *   - return value: VR180_OK (0) or a negative vr180_status; nothing throws across the ABI;
 *   - thread-safe as long as concurrently running calls use different streams and output buffers.
 */
#ifndef VR180_B200_H
#define VR180_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define VR180_ABI_VERSION 2

typedef enum vr180_status {
    VR180_OK = 0,
    VR180_ERR_INVALID_ARG = -1,  /* NULL pointer, non-positive size, bad enum value            */
    VR180_ERR_UNSUPPORTED = -2,  /* valid request the kernels do not implement                 */
    VR180_ERR_CUDA = -3,         /* a CUDA runtime call failed; see vr180_last_cuda_error()    */
    VR180_ERR_NO_DEVICE = -4,    /* no usable sm_100 device                                    */
    VR180_ERR_CHAIN = -5,        /* malformed chain descriptor                                 */
    VR180_ERR_NOMEM = -6
} vr180_status;

/* Numeric values are OpenCV's, because they are the reference's API (remapper.py:330-331, cli.py:57-79). */
enum { VR180_INTER_NEAREST = 0, VR180_INTER_LINEAR = 1, VR180_INTER_CUBIC = 2, VR180_INTER_LANCZOS4 = 4 };
enum {
    VR180_BORDER_CONSTANT = 0,
    VR180_BORDER_REPLICATE = 1,
    VR180_BORDER_REFLECT = 2,
    VR180_BORDER_WRAP = 3,
    VR180_BORDER_REFLECT_101 = 4,
    VR180_BORDER_TRANSPARENT = 5
};

/* ------------------------------------------------------------------------------------------------------
 * Chain descriptor: the transformer chain of transformer.py lowered to plain data.
 * One op per reference transformer; parameters in p[].
 * ---------------------------------------------------------------------------------------------------- */
typedef enum vr180_op_code {
    VR180_OP_NORMALIZE = 1,       /* transformer.py:153-164   p = {cx, cy, scale}: (x-cx)/scale*2          */
    VR180_OP_DENORMALIZE = 2,     /* transformer.py:197-204   p = {sx, sy, cx, cy}: x*sx+cx                */
    VR180_OP_DENORMALIZE_INV = 3, /* transformer.py:206-213   p = {sx, sy, cx, cy}: (x-cx)/sx              */
    VR180_OP_ZOOM = 4,            /* transformer.py:468-473   p = {scale}: x/scale                         */
    VR180_OP_ZOOM_INV = 5,        /* transformer.py:475-480   p = {scale}: x*scale                         */
    VR180_OP_EQUIRECT_ENC = 6,    /* transformer.py:540-568   iparam = is_latitude_y                       */
    VR180_OP_EQUIRECT_DEC = 7,    /* transformer.py:570-584   iparam = is_latitude_y                       */
    VR180_OP_FISHEYE_ENC = 8,     /* transformer.py:359-377   iparam = vr180_mapping (r -> theta)          */
    VR180_OP_FISHEYE_DEC = 9,     /* transformer.py:379-397   iparam = vr180_mapping (theta -> r)          */
    VR180_OP_RECTILINEAR_DEC = 10,     /* transformer.py:338-341  p = {factor}: tan(theta)*factor          */
    VR180_OP_RECTILINEAR_DEC_INV = 11, /* transformer.py:343-347  p = {factor}: atan(theta/factor)         */
    VR180_OP_POLY = 12,           /* transformer.py:448-451   iparam = n coefs, p = coefs_reverse c0..c(n-1) */
    VR180_OP_ROT3 = 13            /* transformer.py:651-657,675-676  p = row-major 3x3 rotation matrix      */
} vr180_op_code;

typedef enum vr180_mapping {
    VR180_MAP_RECTILINEAR = 0,
    VR180_MAP_STEREOGRAPHIC = 1,
    VR180_MAP_EQUIDISTANT = 2,
    VR180_MAP_EQUISOLID = 3,
    VR180_MAP_ORTHOGRAPHIC = 4
} vr180_mapping;

#define VR180_MAX_OPS 12
#define VR180_MAX_OP_PARAMS 12

typedef struct vr180_op {
    int32_t code;   /* vr180_op_code */
    int32_t iparam;
    double p[VR180_MAX_OP_PARAMS];
} vr180_op_t;

typedef struct vr180_chain {
    int32_t n_ops;
    int32_t reserved;
    vr180_op_t ops[VR180_MAX_OPS];
} vr180_chain_t;

/* ------------------------------------------------------------------------------------------------------
 * Images.  uint8 or uint16 elements, interleaved channels (HWC), rows may be strided (remapper.py:455-456 passes
 * views).  A batch is `n_frames` images `frame_stride` bytes apart.  `depth` uses OpenCV's depth codes; a zeroed field
 * is 8-bit.  Pitches and strides stay in bytes for every depth.
 * ---------------------------------------------------------------------------------------------------- */
enum { VR180_DEPTH_8U = 0, VR180_DEPTH_16U = 2 };

typedef struct vr180_image {
    const uint8_t* data; /* device pointer to frame 0, row 0 */
    int32_t rows, cols, channels;
    int32_t depth;        /* VR180_DEPTH_8U or VR180_DEPTH_16U */
    int64_t pitch;        /* bytes between rows   */
    int64_t frame_stride; /* bytes between frames */
} vr180_image_t;

/* Where the source coordinates of an output pixel come from. */
typedef enum vr180_map_kind {
    VR180_MAPSRC_ANALYTIC = 0, /* evaluate `chain` per output pixel in registers; no LUT is read or written */
    VR180_MAPSRC_FLOAT2 = 1,   /* planar float32 xmap / ymap, exactly what cv2.remap takes                 */
    VR180_MAPSRC_FIXED = 2,    /* int32 pairs (sx, sy) = cvRound(map*32) produced by vr180_pack_lut         */
    VR180_MAPSRC_PACKED = 3    /* tile-packed 4-byte LUT from vr180_pack_lut_tiles + the float32 maps it was built
                                  from (xmap / ymap, read only by tiles that cannot be packed)                 */
} vr180_map_kind;

typedef struct vr180_mapsrc {
    int32_t kind; /* vr180_map_kind */
    int32_t packed_interpolation; /* PACKED: the VR180_INTER_* the packed LUT was built for (tile shape and rounding
                                     are per mode); a mismatch with the request falls back to xmap / ymap */
    const vr180_chain_t* chain; /* host pointer; ANALYTIC: full chain Normalize..Denormalize (copied at call) */
    const float* xmap;          /* FLOAT2: device, H rows of W floats, `map_pitch` elements apart            */
    const float* ymap;
    const int32_t* fixed;       /* FIXED: device, H*W interleaved (sx, sy), `map_pitch` pairs per row        */
    int64_t map_pitch;          /* elements (FLOAT2) or pairs (FIXED) between map rows                       */
    /* Optional per-frame radius on the device (float64, one per frame): replaces BOTH scales of the chain's
       final DENORMALIZE op, so a radius produced by vr180_get_radius is consumed without a host sync
       (remapper.py:379 -> :54-56).  ANALYTIC only; NULL = use the scale stored in the chain.  A NaN radius
       (get_radius found no transition) makes every coordinate NaN -> border colour. */
    const double* radius_dev;
    const void* packed;         /* PACKED: device buffer filled by vr180_pack_lut_tiles                       */
} vr180_mapsrc_t;

/* One eye / one image stream: source frames, their coordinate source, and where the result lands. */
typedef struct vr180_view {
    vr180_image_t src;
    vr180_mapsrc_t map;
    int32_t dst_x_offset; /* first output column of this view inside the destination frame (SBS: eye*W) */
    int32_t reserved;
} vr180_view_t;

typedef struct vr180_remap_params {
    int32_t n_views;  /* 1 (apply, remapper.py:388-398) or 2 (apply_lr SBS, :474-484 + :518) */
    int32_t n_frames; /* batch: frames (apply's N images / video frames) sharing the views' maps */
    vr180_view_t view[2];
    /* When view[1].map describes the same coordinates as view[0].map (single transformer, remapper.py:475-484:
       ONE map for both eyes) set share_map=1: coordinates are evaluated once and sampled from both sources. */
    int32_t share_map;
    int32_t out_w, out_h; /* per-view output size: size_output=(W,H), remapper.py:50 */
    int32_t interpolation; /* VR180_INTER_*  */
    int32_t border_mode;   /* VR180_BORDER_* */
    uint8_t border_value[4]; /* per channel; a Python scalar v becomes {v,0,0,0} exactly like cv2 (8-bit colours; see
                                vr180_remap_ex for a full-range colour) */
    uint8_t* dst;            /* device, HWC, same channel count and depth (view[0].src.depth) as the sources */
    int64_t dst_pitch;        /* bytes between destination rows (SBS: >= 2*W*C) */
    int64_t dst_frame_stride; /* bytes between destination frames */
} vr180_remap_params_t;

/* ------------------------------------------------------------------------------------------------------
 * Library / device
 * ---------------------------------------------------------------------------------------------------- */
int vr180_abi_version(void);
const char* vr180_status_string(int status);
/* Text of the last CUDA error seen by the calling thread ("" if none). */
const char* vr180_last_cuda_error(void);
/* Number of CUDA devices; fills name/sm_count/cc for `device` when the pointers are non-NULL. */
int vr180_device_info(int device, char* name, size_t name_len, int* sm_count, int* cc_major, int* cc_minor);
/* Kernels launched by this library in the calling process since load (all threads). */
uint64_t vr180_launch_count(void);

/* ------------------------------------------------------------------------------------------------------
 * (1) analytic map build -- replaces get_map (remapper.py:23-59): evaluates the chain in float64 for every
 *     output pixel (col i, row j) and rounds once to float32 (remapper.py:58).
 *     xmap_dev/ymap_dev: device float32, `map_pitch` elements between rows (>= out_w).
 * ---------------------------------------------------------------------------------------------------- */
int vr180_build_map(const vr180_chain_t* chain, int out_w, int out_h, float* xmap_dev, float* ymap_dev,
                    int64_t map_pitch, void* stream);

/* ------------------------------------------------------------------------------------------------------
 * (2a) LUT pack -- quantises float32 maps exactly as cv::remap does internally for LINEAR/CUBIC/LANCZOS4
 *      (sx = cvRound(x*32), NaN/inf/overflow -> INT_MIN) into interleaved int32 (sx, sy); lossless w.r.t.
 *      the remap output.  The cached-LUT path for repeated video frames (apply's one-map-many-images loop,
 *      remapper.py:381-398).
 * ---------------------------------------------------------------------------------------------------- */
int vr180_pack_lut(const float* xmap_dev, const float* ymap_dev, int64_t map_pitch, int out_w, int out_h,
                   int32_t* fixed_dev, int64_t fixed_pitch, void* stream);

/* ------------------------------------------------------------------------------------------------------
 * (2a') tile-packed LUT -- the cached-LUT form the tiled kernel reads with one 128-bit load per thread.
 *      For every output tile of the requested interpolation (32 x 32 px NEAREST / LINEAR, 32 x 16 CUBIC, 32 x 8
 *      LANCZOS4) it stores a 16-byte header {min ix, max ix, min iy, max iy (int16), flags} and one uint32
 *      per pixel {ix - min ix : 8, iy - min iy : 8, ax : 5, ay : 5} in the order the kernel's threads consume them
 *      (thread-major), with (ix, iy, ax, ay) exactly the integers cv::remap derives from the float32 maps
 *      (sx = cvRound(x * 32), ix = sx >> 5, ax = sx & 31; NEAREST: ix = cvRound(x)) -- lossless w.r.t. the remap
 *      output.  4 bytes per pixel instead of 8, and the tile's source rectangle comes from the header instead of a
 *      block-wide reduction.  Tiles that cannot be packed (NaN / saturated coordinates, footprints wider than 255 px,
 *      partial edge tiles) are flagged and read the float32 maps instead.  The header's flags also carry the geometry of
 *      the tile's source rectangle (TMA box rows, and the box width = staged row pitch with the fewest shared-memory bank
 *      conflicts for the tile's own tap addresses), chosen once here instead of in every launch: with it, launches of
 *      one or a few frames stream the tiles through persistent CTAs whose producer warp fetches the next tiles'
 *      rectangles from the headers alone (csrc/stream.cu).  The buffer's layout is private to one build of the library:
 *      build it at run time with the library that consumes it, do not persist it.  Replaces the convertMaps step inside
 *      cv.remap at remapper.py:389 for apply()'s one-map-many-images loop (remapper.py:381-398).
 *      vr180_packed_lut_bytes: size of the device buffer for an out_w x out_h map.
 * ---------------------------------------------------------------------------------------------------- */
size_t vr180_packed_lut_bytes(int out_w, int out_h, int interpolation);
int vr180_pack_lut_tiles(const float* xmap_dev, const float* ymap_dev, int64_t map_pitch, int out_w, int out_h,
                         int interpolation, void* packed_dev, void* stream);

/* ------------------------------------------------------------------------------------------------------
 * (2b) remap / fused warp + SBS packing -- replaces cv.remap per image (remapper.py:388-398) and
 *      np.concatenate(axis=1) (remapper.py:518): each view is written straight into its column range of the
 *      destination frame.  uint8 (16-bit: vr180_remap_ex), 1/3/4 channels.  Bit-exact to cv2.remap for the same
 *      float32 maps.
 *      Performance note (results are identical either way): the TMA-tiled kernel serves 3 channels, NEAREST /
 *      LINEAR / CUBIC / LANCZOS4 (NEAREST not with a MAPSRC_FIXED LUT, which stores x * 32) when every base pointer, row
 *      pitch and frame stride is a multiple of 16 bytes and every view's dst_x_offset * 3 is too (a TMA box must start at
 *      a 16-byte aligned global address).  With BORDER_CONSTANT and a zero colour, tiles that straddle the source edge
 *      are staged too (TMA's zero fill is the border); with any other border mode / colour only tiles whose footprint
 *      lies inside the source are staged and the (few) edge tiles are gathered per pixel inside the same kernel.  Any
 *      other request runs in the generic per-pixel kernel.
 * ---------------------------------------------------------------------------------------------------- */
int vr180_remap(const vr180_remap_params_t* params, void* stream);
/* vr180_remap with the border colour given as the cv::Scalar the reference passes (borderValue): the library saturates
 * each entry to the depth of the images (round half to even, clamp), as cv2 does.  NULL = use params->border_value.
 * 16-bit images (src.depth = VR180_DEPTH_16U for every view; the destination has the same depth) follow cv::remap's
 * float-weight arithmetic for non-8-bit depths and are bit-exact to cv2.remap on uint16 images; they run in the generic
 * per-pixel kernel (base pointers, pitches and strides 2-byte aligned).  Any other depth, or views of different depths,
 * is VR180_ERR_UNSUPPORTED. */
int vr180_remap_ex(const vr180_remap_params_t* params, const double border_scalar[4], void* stream);

/* ------------------------------------------------------------------------------------------------------
 * (3) get_radius -- replaces transformer.py:108-140 for a batch.  For frame f and view v it scans the centre
 *     row (cols > rows) or centre column (otherwise) and writes
 *        transitions_dev[(f*n_views+v)*2 + 0] = first k with !black[k] && black[k+1]   (or -1)
 *        transitions_dev[(f*n_views+v)*2 + 1] = last  k with  black[k] && !black[k+1]  (or -1)
 *     with black[k] <=> mean_c px[k][c] < threshold (float64, as np.mean does; 8- or 16-bit elements per views[v].depth,
 *     every view of one call with the same depth).  If radius_dev is non-NULL it also writes
 *        radius_dev[f] = max_v (last - first) / 2          (remapper.py:82-84, "auto")
 *     as float64, NaN when any view of the frame lacks a transition (the reference raises IndexError; the
 *     Python layer re-raises it from the -1 sentinels).
 * ---------------------------------------------------------------------------------------------------- */
int vr180_get_radius(const vr180_image_t* views, int n_views, int n_frames, double threshold,
                     int32_t* transitions_dev, double* radius_dev, void* stream);

/* ------------------------------------------------------------------------------------------------------
 * (4) anaglyph merge -- replaces the merge=True branch of apply_lr (remapper.py:485-498) on the device-resident SBS
 *     frame (H, 2 * eye_w, 3): out[y, x, c] = (mean_c L[y, x] * (0, 128, 255)[c] + mean_c R[y, x] * (255, 128, 0)[c]) / 255
 *     in float64 with one rounding per NumPy ufunc, then the float64 -> uint8 conversion cv.imwrite applies to the
 *     reference's float64 image (round half to even, saturate).  The "L" / "R" labels (cv.putText, :499-516) stay on
 *     the host: on a float64 image OpenCV draws them without anti-aliasing, i.e. as pure colours over these bytes.
 * ---------------------------------------------------------------------------------------------------- */
int vr180_anaglyph(const uint8_t* sbs_dev, int64_t sbs_pitch, int64_t sbs_frame_stride, int eye_w, int h, int n_frames,
                   uint8_t* out_dev, int64_t out_pitch, int64_t out_frame_stride, void* stream);

/* ------------------------------------------------------------------------------------------------------
 * (5) chain on points -- the pixel -> 3-D step of match_lr (remapper.py:291-320: (decoder * Denormalize)
 *     .inverse_transform on the matched points, then equidistant_to_3d, transformer.py:483-508) for a batch of points.
 *     `chain` is applied to (x[i], y[i]) in float64; out_x / out_y receive the transformed coordinates and/or out_v3
 *     the n x 3 unit vectors of equidistant_to_3d of the result (either may be NULL, not both).
 * ---------------------------------------------------------------------------------------------------- */
int vr180_transform_points(const vr180_chain_t* chain, int64_t n, const double* x_dev, const double* y_dev,
                           double* out_x_dev, double* out_y_dev, double* out_v3_dev, void* stream);

/* ------------------------------------------------------------------------------------------------------
 * (6) optional codec offload (nvJPEG, loaded with dlopen at first use) -- stands in for cv.imread / cv.imwrite around
 *     the hot path (remapper.py:373, :453, :519) so that a JPEG -> warp -> JPEG conversion moves only compressed bytes
 *     over PCIe.  OPT-IN: nvJPEG's decoder is not bit-compatible with the libjpeg-turbo decoder inside cv.imread (a few
 *     grey levels on some pixels), so the default file path keeps cv2 and its bit-exact contract.
 *     vr180_jpeg_available: 1 when libnvjpeg could be loaded.  vr180_jpeg_decode: host JPEG bytes -> interleaved BGR
 *     uint8 on the device (the layout cv.imread returns; width / height from vr180_jpeg_info).  vr180_jpeg_encode:
 *     interleaved BGR on the device -> host JPEG bytes with cv.imwrite's defaults (4:2:0, standard Huffman tables);
 *     *out_len is the capacity on entry and the stream length on return (VR180_ERR_NOMEM + needed size if too small).
 *     All entry points return VR180_ERR_UNSUPPORTED when libnvjpeg is absent.
 * ---------------------------------------------------------------------------------------------------- */
int vr180_jpeg_available(void);
int vr180_jpeg_info(const uint8_t* jpeg_host, size_t n, int* width, int* height, int* channels);
int vr180_jpeg_decode(const uint8_t* jpeg_host, size_t n, uint8_t* bgr_dev, int64_t pitch, int width, int height,
                      void* stream);
int vr180_jpeg_encode(const uint8_t* bgr_dev, int64_t pitch, int width, int height, int quality, uint8_t* out_host,
                      size_t* out_len, void* stream);

/* ------------------------------------------------------------------------------------------------------
 * Host-buffer pipeline (what the Python `apply` / `apply_lr` call with NumPy arrays): a context owns device
 * staging buffers and three streams (H2D, compute, D2H) and runs upload -> [get_radius] -> warp -> download
 * for a batch of frames with the copies of neighbouring frames overlapped.
 * ---------------------------------------------------------------------------------------------------- */
typedef struct vr180_ctx vr180_ctx_t;

int vr180_ctx_create(int device, vr180_ctx_t** out);
int vr180_ctx_destroy(vr180_ctx_t* ctx);
int vr180_ctx_device(const vr180_ctx_t* ctx);

/* Pinned host memory helpers (cudaHostAlloc / cudaHostRegister), so callers need no CUDA binding. */
int vr180_host_alloc(size_t bytes, void** out);
int vr180_host_free(void* p);
int vr180_host_register(void* p, size_t bytes);
int vr180_host_unregister(void* p);

typedef struct vr180_host_job {
    int32_t n_views, n_frames;
    /* host source frames: view v, frame f at src[v] + f*src_frame_stride[v]; same geometry rules as vr180_image_t */
    const uint8_t* src[2];
    int32_t src_rows, src_cols, channels;
    int32_t depth; /* VR180_DEPTH_8U (0) or VR180_DEPTH_16U, for the sources and the destination alike */
    int64_t src_pitch[2];
    int64_t src_frame_stride[2];
    /* coordinate source per view.  ANALYTIC: chain (host).  FLOAT2: HOST float32 maps, uploaded once per call and
       cached in the context keyed by pointer+size while `maps_cache_key` is unchanged and non-zero. */
    int32_t map_kind;
    int32_t share_map;
    const vr180_chain_t* chain[2];
    const float* xmap[2];
    const float* ymap[2];
    uint64_t maps_cache_key;
    /* radius: radius_mode 0 = as stored in the chain / maps; 1 = "auto": vr180_get_radius per frame (max over the
       frame's views), consumed on the device (ANALYTIC only) */
    int32_t radius_mode;
    int32_t reserved1;
    double threshold;
    int32_t out_w, out_h;
    int32_t interpolation, border_mode;
    uint8_t border_value[4];
    /* host destination: frame f at dst + f*dst_frame_stride, view v at column v*out_w */
    uint8_t* dst;
    int64_t dst_pitch;
    int64_t dst_frame_stride;
    /* optional outputs (may be NULL): per (frame, view) transitions [n_frames*n_views*2] and per-frame radius */
    int32_t* transitions_out;
    double* radius_out;
    /* Scattered frames -- apply()'s list of separate arrays (remapper.py:371-378, :388-398 loops over them with ONE
       map): when src_frames[0] is non-NULL, frame f of view v starts at src_frames[v][f] (src[v] and
       src_frame_stride[v] are ignored; src_pitch[v] still applies to every frame); when dst_frames is non-NULL,
       destination frame f starts at dst_frames[f] (dst and dst_frame_stride are ignored). */
    const uint8_t* const* src_frames[2];
    uint8_t* const* dst_frames;
    /* Host buffers that are not page-locked (plain NumPy arrays) cannot be DMA'd asynchronously: they are packed
       into / unpacked from a pinned ring owned by the context by `copy_threads` host threads (0 = default:
       min(12, cores / 2), or $VR180_COPY_THREADS), overlapped with the GPU work of the neighbouring chunks.
       staging: VR180_STAGE_AUTO = per buffer, decided with cudaPointerGetAttributes; ALWAYS / NEVER force it. */
    int32_t staging;
    int32_t copy_threads;
    /* merge != 0 (n_views == 2, 3 channels, 8-bit): vr180_anaglyph runs on the device SBS frame and the destination frames
       are the merged (out_h, out_w, 3) images -- half the download, no host pass (apply_lr(merge=True)). */
    int32_t merge;
    int32_t reserved2;
} vr180_host_job_t;

enum { VR180_STAGE_AUTO = 0, VR180_STAGE_ALWAYS = 1, VR180_STAGE_NEVER = 2 };

/* Synchronous: returns when every destination frame is complete in host memory. */
int vr180_ctx_run(vr180_ctx_t* ctx, const vr180_host_job_t* job);
/* vr180_ctx_run with the border colour as a cv::Scalar saturated to job->depth (see vr180_remap_ex); NULL = use
 * job->border_value. */
int vr180_ctx_run_ex(vr180_ctx_t* ctx, const vr180_host_job_t* job, const double border_scalar[4]);

/* ------------------------------------------------------------------------------------------------------
 * Test / profiling hooks (not part of the drop-in surface; no reference counterpart).
 * ---------------------------------------------------------------------------------------------------- */
/* The host-built OpenCV weight tables the kernels use (K = 4 bicubic, K = 8 Lanczos4): 1024*K*K int16. */
int vr180_debug_weight_table(int K, int16_t* out);
/* what 0: frames per CTA of the tiled kernel (0 = automatic) -- lets tests drive long frame loops (stage-ring
   refills, mbarrier phase flips) with small outputs; what 1: tiled-kernel experiment flags (-1 = environment
   variable VR180_TILED_DEBUG; bit 1: take the tile-streaming kernel whenever the request is eligible, bit 2: never,
   bit 8: the standard chain through the op-by-op interpreter of chain.cuh instead of its folded form, chain_fast.cuh);
   what 2: cap of the automatic frames-per-CTA choice (0 = default 64); what 3: CTAs of the tile-streaming kernel
   (0 = 3 per SM) -- lets tests push hundreds of tiles through one CTA.  Returns the previous value. */
int vr180_debug_set(int what, int value);
/* The byte mover of the pipeline's copy threads (packs pageable frames into the page-locked ring: streaming stores for
   copies of 8 KB and more on CPUs with AVX2, memcpy otherwise; VR180_NT_COPY=0 forces memcpy) applied to caller buffers. */
int vr180_debug_host_copy(void* dst, const void* src, size_t bytes);
/* Copy-only ceiling of the host-buffer pipeline (bench.py e2e.copy_ceiling): page-locked host <-> device copies of
   `bytes` each way, `reps` times, no kernel: out_gbs[4] = {H2D alone, D2H alone, H2D and D2H while both run}. */
int vr180_debug_copy_ceiling(int device, size_t bytes, int reps, double* out_gbs);

#ifdef __cplusplus
}
#endif
#endif /* VR180_B200_H */
