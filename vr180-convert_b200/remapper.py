"""`get_map`, `get_radius_smart`, `apply`, `apply_lr` with the reference's signatures
(/root/reference/src/vr180_convert/remapper.py:23-90, 324-520), executed by libvr180_b200.so.

NumPy arrays in, NumPy arrays out; the arithmetic (chain evaluation, OpenCV-exact sampling, radius scan, SBS
packing) happens in CUDA kernels through the C ABI.  There is no CPU fallback: without the shared object or a
CUDA device these functions raise.
"""
from __future__ import annotations

import ctypes as C
import os
import threading
import weakref
from collections import OrderedDict
from logging import getLogger
from pathlib import Path
from typing import Any, Literal, Sequence

import numpy as np
from numpy.typing import NDArray

from . import _native as N
from .transformer import DenormalizeTransformer, NormalizeTransformer, TransformerBase

LOG = getLogger(__name__)

# OpenCV's integer constants are the reference's API (remapper.py:330-331; cli.py:57-79 resolves names via getattr(cv, ...))
INTER_NEAREST, INTER_LINEAR, INTER_CUBIC, INTER_AREA, INTER_LANCZOS4 = 0, 1, 2, 3, 4
BORDER_CONSTANT, BORDER_REPLICATE, BORDER_REFLECT, BORDER_WRAP, BORDER_REFLECT_101, BORDER_TRANSPARENT = 0, 1, 2, 3, 4, 5

_codec = os.environ.get("VR180_CODEC", "cv2")


def set_codec(name: str) -> None:
    """"cv2" (default: files are read / written by OpenCV on the host, bit-identical to the reference) or "nvjpeg"
    (opt-in: the JPEG -> warp -> JPEG form of apply_lr decodes, warps and encodes on the GPU, see codec.py)."""
    global _codec
    if name not in ("cv2", "nvjpeg"):
        raise ValueError("codec must be 'cv2' or 'nvjpeg'")
    _codec = name


_ctx_lock = threading.Lock()
_ctxs: dict[int, C.c_void_p] = {}
_default_device = 0


def set_device(device: int) -> None:
    """CUDA device used by the NumPy-level API of this process (one process per GPU)."""
    global _default_device
    _default_device = int(device)


def _ctx(device: int | None = None) -> C.c_void_p:
    dev = _default_device if device is None else int(device)
    with _ctx_lock:
        if dev not in _ctxs:
            handle = C.c_void_p()
            N.check(N.lib().vr180_ctx_create(dev, C.byref(handle)), "vr180_ctx_create")
            _ctxs[dev] = handle
        return _ctxs[dev]


# ---------------------------------------------------------------------------------------------------------
# page-locked result arrays
# ---------------------------------------------------------------------------------------------------------
class _PinnedPool:
    """Result frames are allocated in page-locked host memory (vr180_host_alloc), so the download of every frame is
    a plain DMA into the array the caller receives -- no pageable bounce copy.  A buffer goes back to the pool when
    the last NumPy view of it is garbage-collected; a video loop therefore recycles the same few buffers."""

    def __init__(self, keep_bytes: int = 4 << 30) -> None:
        self._free: dict[int, list[int]] = {}
        self._free_bytes = 0
        self._keep = keep_bytes
        self._lock = threading.Lock()

    def empty(self, shape: tuple[int, ...], dtype: Any = np.uint8) -> NDArray:
        dtype = np.dtype(dtype)
        count = int(np.prod(shape))
        nbytes = max(1, count * dtype.itemsize)  # the pool recycles byte buffers; the array is a view of any dtype
        with self._lock:
            lst = self._free.get(nbytes)
            ptr = lst.pop() if lst else None
            if ptr is not None:
                self._free_bytes -= nbytes
        if ptr is None:
            handle = C.c_void_p()
            N.check(N.lib().vr180_host_alloc(nbytes, C.byref(handle)), "vr180_host_alloc")
            ptr = int(handle.value)
        owner = (C.c_uint8 * nbytes).from_address(ptr)
        weakref.finalize(owner, self._release, ptr, nbytes)
        return np.frombuffer(owner, dtype=dtype, count=count).reshape(shape)

    def _release(self, ptr: int, nbytes: int) -> None:
        with self._lock:
            if self._free_bytes + nbytes <= self._keep:
                self._free.setdefault(nbytes, []).append(ptr)
                self._free_bytes += nbytes
                return
        try:
            N.lib().vr180_host_free(C.c_void_p(ptr))
        except Exception:  # noqa: BLE001 -- interpreter shutdown
            pass


_pinned = _PinnedPool()


def pinned_empty(shape: tuple[int, ...], dtype: Any = np.uint8) -> NDArray:
    """A uint8 (or `dtype`) array in page-locked host memory (vr180_host_alloc), recycled when garbage-collected.
    Frames a capture or decode loop writes straight into such arrays are uploaded by DMA without the packing copy plain NumPy arrays
    need (the host pipeline decides per buffer, include/vr180_b200.h `staging`)."""
    return _pinned.empty(tuple(int(v) for v in shape), dtype)


def _result_empty(shape: tuple[int, ...], dtype: Any = np.uint8) -> NDArray:
    if os.environ.get("VR180_PINNED_OUTPUTS", "1") == "0":
        return np.empty(shape, dtype=dtype)
    return _pinned.empty(shape, dtype)


# ---------------------------------------------------------------------------------------------------------
# lowering helpers
# ---------------------------------------------------------------------------------------------------------
def full_chain(transformer: TransformerBase, *, radius: float, size_input: tuple[int, int]) -> TransformerBase:
    """Normalize * t * Denormalize(scale=(r, r), center=(cols//2, rows//2)) -- remapper.py:51-57."""
    return (NormalizeTransformer() * transformer
            * DenormalizeTransformer(scale=(radius, radius), center=(size_input[1] // 2, size_input[0] // 2)))


def lower_full(transformer: TransformerBase, *, radius: float, size_input: tuple[int, int],
               size_output: tuple[int, int]) -> "list[tuple] | None":
    ops = full_chain(transformer, radius=radius, size_input=size_input).lower(
        shape=(size_output[1], size_output[0]), inverse=False)
    if ops is None or len(ops) > N.MAX_OPS:
        return None
    return ops


_chain_cache: "OrderedDict[tuple, Any]" = OrderedDict()
_chain_lock = threading.Lock()


def lowered_chain(transformer: TransformerBase, *, radius: float, size_input: tuple[int, int],
                  size_output: tuple[int, int]) -> "N.Chain | None":
    """vr180_chain_t of Normalize * t * Denormalize, cached on repr(transformer) (the reference's transformers are
    attrs classes with a stable repr) + radius + sizes: a video loop lowers its chain once, not once per frame."""
    try:
        key = (repr(transformer), float(radius), tuple(size_input), tuple(size_output))
        hash(key)
    except Exception:  # noqa: BLE001 -- exotic radius / repr: do not cache
        key = None
    if key is not None:
        with _chain_lock:
            if key in _chain_cache:
                _chain_cache.move_to_end(key)
                return _chain_cache[key]
    ops = lower_full(transformer, radius=radius, size_input=size_input, size_output=size_output)
    chain = N.make_chain(ops) if ops is not None else None
    if key is not None:
        with _chain_lock:
            _chain_cache[key] = chain
            while len(_chain_cache) > 64:
                _chain_cache.popitem(last=False)
    return chain


def host_maps(transformer: TransformerBase, *, radius: float, size_input: tuple[int, int],
              size_output: tuple[int, int]) -> tuple[NDArray[np.float32], NDArray[np.float32]]:
    """Opaque (user-defined) transformers: run THEIR NumPy code once on the pixel grid (remapper.py:50-58)."""
    xmap, ymap = np.meshgrid(np.arange(size_output[0]), np.arange(size_output[1]))
    with np.errstate(invalid="ignore", divide="ignore"):
        xmap, ymap = full_chain(transformer, radius=radius, size_input=size_input).transform(xmap, ymap)
    return np.ascontiguousarray(xmap, dtype=np.float32), np.ascontiguousarray(ymap, dtype=np.float32)


def get_map(
    transformer: TransformerBase,
    *,
    radius: float,
    size_input: tuple[int, int],
    size_output: tuple[int, int] = (2048, 2048),
) -> tuple[NDArray[np.float32], NDArray[np.float32]]:
    """float32 (H, W) source-coordinate maps for cv2.remap-style sampling (remapper.py:23-59).

    Recognised transformer chains are evaluated per pixel in float64 by csrc/kernels.cu:k_build_map and rounded
    once to float32; chains containing user-defined Python transformers are evaluated by that Python code."""
    ops = lower_full(transformer, radius=radius, size_input=size_input, size_output=size_output)
    if ops is None:
        return host_maps(transformer, radius=radius, size_input=size_input, size_output=size_output)
    import torch

    w, h = int(size_output[0]), int(size_output[1])
    dev = torch.device("cuda", _default_device)
    maps = torch.empty((2, h, w), dtype=torch.float32, device=dev)
    chain = N.make_chain(ops)
    stream = torch.cuda.current_stream(dev).cuda_stream
    N.check(N.lib().vr180_build_map(C.byref(chain), w, h, maps[0].data_ptr(), maps[1].data_ptr(), w, stream),
            "vr180_build_map")
    out = maps.cpu().numpy()
    return out[0], out[1]


# ---------------------------------------------------------------------------------------------------------
# radius
# ---------------------------------------------------------------------------------------------------------
def _centre_line(img: NDArray) -> NDArray:
    """The one row / column get_radius reads (transformer.py:125-129), as a (1, n, C) or (n, 1, C) image
    whose centre line is that row / column again -- so only ~n*C bytes are uploaded."""
    if img.ndim != 3:
        raise IndexError("too many indices for array: get_radius needs an (H, W, C) image")
    height, width = img.shape[:2]
    if width > height:
        return np.ascontiguousarray(img[height // 2: height // 2 + 1, :, :])
    return np.ascontiguousarray(img[:, width // 2: width // 2 + 1, :])


def _device_radius(images: Sequence[NDArray], threshold: float = 10) -> list[float]:
    """get_radius (transformer.py:108-140) of every image: the centre lines of all images of one geometry go up in
    ONE upload, are scanned by ONE k_get_radius launch and come back with ONE blocking read."""
    import torch

    lines = []
    for img in images:
        line = _centre_line(np.asarray(img))
        if line.dtype not in _DEPTHS:
            raise TypeError(f"get_radius kernel takes uint8 or uint16 images, got {line.dtype}")
        rows, cols, ch = line.shape
        if ch > 4:
            raise ValueError("get_radius kernel supports up to 4 channels")
        # keep the reference's row-vs-column decision: a 1 x n line has cols > rows unless n == 1
        if cols <= rows and rows == 1:
            raise IndexError("index 0 is out of bounds for axis 0 with size 0")
        lines.append(line)
    dev = torch.device("cuda", _default_device)
    stream = torch.cuda.current_stream(dev).cuda_stream
    out: list[float] = [0.0] * len(lines)
    groups: dict[tuple, list[int]] = {}
    for i, line in enumerate(lines):
        groups.setdefault((line.shape, line.dtype), []).append(i)
    for ((rows, cols, ch), dtype), idx in groups.items():
        stack = np.stack([lines[i] for i in idx])  # (n, rows, cols, ch), one of rows / cols is 1
        d_lines = torch.from_numpy(stack).to(dev)
        trans = torch.empty((len(idx), 2), dtype=torch.int32, device=dev)
        esz = dtype.itemsize
        im = N.Image(d_lines.data_ptr(), rows, cols, ch, _DEPTHS[dtype], cols * ch * esz, rows * cols * ch * esz)
        N.check(N.lib().vr180_get_radius(C.byref(im), 1, len(idx), float(threshold), trans.data_ptr(), None, stream),
                "vr180_get_radius")
        for i, (first, last) in zip(idx, trans.cpu().tolist()):
            if first < 0 or last < 0:
                raise IndexError("index 0 is out of bounds for axis 0 with size 0")  # np.where(...)[0][0] on empty
            out[i] = (last - first) / 2
    return out


def get_radius_smart(radius: float | Literal["auto", "max"], images: Sequence[NDArray]) -> float:
    """remapper.py:62-90."""
    if isinstance(radius, str) and radius == "auto":
        radius_ = max(_device_radius(images))
    elif isinstance(radius, str) and radius == "max":
        radius_ = min(images[0].shape[0] / 2, images[0].shape[1] / 2)
    else:
        radius_ = radius
    LOG.info(f"Radius: {radius_}, strategy: {radius}, image shape: {images[0].shape}")
    return radius_


# ---------------------------------------------------------------------------------------------------------
# apply / apply_lr
# ---------------------------------------------------------------------------------------------------------
def _border_scalar(value: Any) -> "C.Array[C.c_double]":
    """The cv::Scalar cv2 builds from a border value: a Python scalar v becomes (v, 0, 0, 0), a sequence its first four
    entries.  The library saturates it to the image depth (vr180_remap_ex / vr180_ctx_run_ex)."""
    vals = [float(value), 0.0, 0.0, 0.0] if np.isscalar(value) else [*map(float, value), 0.0, 0.0, 0.0, 0.0][:4]
    return (C.c_double * 4)(*vals)


def _border_bytes(value: Any, channels: int) -> tuple[int, int, int, int]:
    """cv2 converts a Python scalar to Scalar(v, 0, 0, 0) and saturates each entry to uint8."""
    vals = [float(value), 0.0, 0.0, 0.0] if np.isscalar(value) else [*map(float, value), 0.0, 0.0, 0.0, 0.0][:4]
    return tuple(int(min(255, max(0, np.rint(v)))) for v in vals)  # type: ignore[return-value]


def _check_modes(interpolation: int, border_mode: int) -> tuple[int, int]:
    interpolation = int(interpolation)
    if interpolation == INTER_AREA:  # cv::remap treats INTER_AREA as INTER_LINEAR
        interpolation = INTER_LINEAR
    if interpolation not in (INTER_NEAREST, INTER_LINEAR, INTER_CUBIC, INTER_LANCZOS4):
        raise ValueError(f"Unknown interpolation method {interpolation}")
    border_mode = int(border_mode)
    if border_mode == BORDER_TRANSPARENT:
        raise NotImplementedError("BORDER_TRANSPARENT leaves uninitialised memory in the reference; not supported")
    if border_mode not in (BORDER_CONSTANT, BORDER_REPLICATE, BORDER_REFLECT, BORDER_WRAP, BORDER_REFLECT_101):
        raise ValueError(f"Unknown/unsupported border type {border_mode}")
    return interpolation, border_mode


# element types of the remap path -> vr180 depth codes
_DEPTHS = {np.dtype(np.uint8): N.DEPTH_8U, np.dtype(np.uint16): N.DEPTH_16U}


def _as_image(a: Any) -> NDArray:
    img = np.asarray(a)
    if img.dtype not in _DEPTHS:
        raise TypeError(f"the B200 remap path takes uint8 or uint16 images (what cv.imread returns), got {img.dtype}")
    if img.ndim == 2:
        img = img[:, :, None]
    if img.ndim != 3 or img.shape[2] not in (1, 3, 4):
        raise ValueError(f"unsupported image shape {img.shape}")
    e = img.itemsize
    if img.strides[2] != e or img.strides[1] != img.shape[2] * e or img.strides[0] < img.shape[1] * img.shape[2] * e:
        img = np.ascontiguousarray(img)  # only pixel-contiguous rows can be described by a pitch
    return img


def _run_job(job: "N.HostJob", dtype: np.dtype, border_value: Any) -> None:
    """vr180_ctx_run with the job's depth and border colour: 8-bit colours as saturated bytes, 16-bit ones as the
    cv::Scalar the library saturates (a colour above 255 does not fit the job's byte field)."""
    job.depth = _DEPTHS[np.dtype(dtype)]
    if job.depth == N.DEPTH_8U:
        for i, b in enumerate(_border_bytes(border_value, job.channels)):
            job.border_value[i] = b
        N.check(N.lib().vr180_ctx_run(_ctx(), C.byref(job)), "vr180_ctx_run")
    else:
        N.check(N.lib().vr180_ctx_run_ex(_ctx(), C.byref(job), _border_scalar(border_value)), "vr180_ctx_run_ex")


def warp_host(
    transformers: Sequence[TransformerBase],
    images: Sequence[Any],
    *,
    radii: Sequence[float],
    share_map: bool,
    size_output: tuple[int, int],
    interpolation: int,
    border_mode: int,
    border_value: Any,
    auto_radius: bool = False,
    threshold: float = 10,
    merge: bool = False,
) -> "NDArray[np.uint8] | list[NDArray[np.uint8]]":
    """ONE host job (vr180_ctx_run) for a whole batch.

    `images` holds one entry per view (1 = apply(), 2 = the eyes of apply_lr()); an entry is either one image or a
    LIST of images of equal geometry (the frames of the batch: apply()'s image list, remapper.py:388-398; a clip of
    stereo pairs).  Every frame is written as (H, n_views * W, C) with the views side by side.  Returns one array for
    single images and a list of arrays (one per frame) for lists.

    `auto_radius`: per-frame radius = max over the frame's views of get_radius (remapper.py:82-84 for one pair),
    scanned and consumed on the device; a frame without a transition raises IndexError like the reference.

    `merge` (two views, 3 channels): the frames that come back are the anaglyph of the two eyes (H, W, 3), computed by
    vr180_anaglyph on the device SBS frame (remapper.py:485-498) -- the SBS frame itself never leaves the GPU."""
    lib = N.lib()
    batched = isinstance(images[0], (list, tuple))
    frames = [[_as_image(im) for im in (v if batched else [v])] for v in images]
    n_views, n_frames = len(frames), len(frames[0])
    if any(len(v) != n_frames for v in frames):
        raise ValueError("every view needs the same number of frames")
    if n_frames == 0:
        return []
    rows, cols, ch = frames[0][0].shape
    dtype = frames[0][0].dtype
    for v in frames:
        for im in v:
            if im.shape != (rows, cols, ch):
                raise ValueError("all frames / eyes of one job must have the same shape")
            if im.dtype != dtype:
                raise ValueError("all frames / eyes of one job must have the same dtype")
    w, h = int(size_output[0]), int(size_output[1])
    first = np.asarray(images[0][0] if batched else images[0])
    squeeze = first.ndim == 2
    if merge and (n_views != 2 or ch != 3):
        raise ValueError("merge needs two 3-channel views")
    if merge and dtype != np.uint8:
        raise ValueError("merge (the anaglyph) takes uint8 images")
    outs = [_result_empty((h, w * (1 if merge else n_views), ch), dtype) for _ in range(n_frames)]

    job = N.HostJob()
    job.n_views, job.n_frames = n_views, n_frames
    job.src_rows, job.src_cols, job.channels = rows, cols, ch
    keep: list[Any] = [frames]
    n_maps = 1 if (share_map or n_views == 1) else n_views
    chains = [lowered_chain(transformers[m], radius=(1.0 if auto_radius else radii[m]), size_input=(rows, cols),
                            size_output=(w, h)) for m in range(n_maps)]
    analytic = all(c is not None for c in chains)
    if auto_radius and not analytic:
        raise ValueError("a per-frame radius is consumed on the device by lowerable transformer chains only")
    job.map_kind = N.MAPSRC_ANALYTIC if analytic else N.MAPSRC_FLOAT2
    job.share_map = 1 if (share_map and n_views == 2) else 0
    for m in range(n_maps):
        if analytic:
            job.chain[m] = C.pointer(chains[m])
            keep.append(chains[m])
        else:
            xm, ym = (get_map if chains[m] is not None else host_maps)(
                transformers[m], radius=radii[m], size_input=(rows, cols), size_output=(w, h))
            xm, ym = np.ascontiguousarray(xm), np.ascontiguousarray(ym)
            keep += [xm, ym]
            job.xmap[m], job.ymap[m] = xm.ctypes.data, ym.ctypes.data
    for v in range(n_views):
        # the job carries one row pitch per view: a view whose frames disagree is made contiguous
        pitch = frames[v][0].strides[0]
        if any(im.strides[0] != pitch for im in frames[v]):
            frames[v] = [np.ascontiguousarray(im) for im in frames[v]]
            pitch = frames[v][0].strides[0]
        ptrs = (C.c_void_p * n_frames)(*[im.ctypes.data for im in frames[v]])
        keep.append(ptrs)
        job.src[v] = ptrs[0]
        job.src_frames[v] = ptrs
        job.src_pitch[v] = pitch
        job.src_frame_stride[v] = pitch * rows
    job.out_w, job.out_h = w, h
    job.interpolation, job.border_mode = interpolation, border_mode
    dptrs = (C.c_void_p * n_frames)(*[o.ctypes.data for o in outs])
    keep.append(dptrs)
    job.dst = dptrs[0]
    job.dst_frames = dptrs
    job.dst_pitch = outs[0].strides[0]
    job.dst_frame_stride = outs[0].strides[0] * h
    job.merge = 1 if merge else 0
    trans = None
    if auto_radius:
        job.radius_mode = 1
        job.threshold = float(threshold)
        trans = np.empty((n_frames, n_views, 2), dtype=np.int32)
        job.transitions_out = trans.ctypes.data
    _run_job(job, dtype, border_value)
    del keep
    if trans is not None and (trans < 0).any():
        raise IndexError("index 0 is out of bounds for axis 0 with size 0")  # get_radius found no transition
    if trans is not None and LOG.isEnabledFor(20):
        for f in range(n_frames):
            r = max((int(trans[f, v, 1]) - int(trans[f, v, 0])) / 2 for v in range(n_views))
            LOG.info(f"Radius: {r}, strategy: auto, image shape: {(rows, cols, ch)}")
    if squeeze:
        outs = [o[:, :, 0] for o in outs]
    return outs if batched else outs[0]


def _imread(path: Any) -> NDArray:
    import cv2 as cv  # file decode only (out of the hot path, SURVEY.md §2 row 15)

    return cv.imread(Path(path).as_posix())


def _imwrite(path: Any, image: NDArray) -> None:
    import cv2 as cv

    cv.imwrite(Path(path).as_posix(), image)


def apply(
    transformer: TransformerBase,
    *,
    in_paths: Sequence[Path | str | NDArray] | Path | str | NDArray,
    out_paths: Sequence[Path | str] | None | Path | str = None,
    size_output: tuple[int, int] = (2048, 2048),
    interpolation: int = INTER_LANCZOS4,
    boarder_mode: int = BORDER_CONSTANT,
    boarder_value: int | tuple[int, int, int] = 0,
    radius: float | Literal["auto", "max"] = "auto",
) -> Sequence[NDArray[np.uint8]]:
    """Remap every input image with ONE map built from images[0]'s shape (remapper.py:324-403).
    Argument names (including the `boarder_*` spelling) are the reference's.

    All images of the call go through ONE host job (one radius scan launch, one chain lowering, uploads / warps /
    downloads of neighbouring images overlapped) instead of the reference's per-image cv.remap loop."""
    in_list = [in_paths] if isinstance(in_paths, (str, Path, np.ndarray)) else list(in_paths)
    out_list = [out_paths] if isinstance(out_paths, (str, Path)) else out_paths
    interpolation, border_mode = _check_modes(interpolation, boarder_mode)

    images = [_imread(p) if isinstance(p, (str, Path)) else p for p in in_list]
    radius_ = get_radius_smart(radius, images)
    size_in = (images[0].shape[0], images[0].shape[1])
    # one job for the images of images[0]'s shape and dtype; cv.remap takes every image on its own, in its own dtype
    first = np.asarray(images[0])
    same = [i for i, img in enumerate(images)
            if np.asarray(img).shape == first.shape and np.asarray(img).dtype == first.dtype]
    results: list[Any] = [None] * len(images)
    warped = warp_host([transformer], [[images[i] for i in same]], radii=[radius_], share_map=True,
                       size_output=size_output, interpolation=interpolation, border_mode=border_mode,
                       border_value=boarder_value)
    for i, r in zip(same, warped):
        results[i] = r
    for i, img in enumerate(images):
        if results[i] is None:
            # the reference samples a differently-sized image with images[0]'s map; keep that behaviour
            if np.asarray(img).shape != first.shape:
                LOG.warning("image shape %s differs from the first image %s; using the first image's map",
                            np.asarray(img).shape, size_in)
            results[i] = _warp_with_first_geometry(transformer, img, size_in, radius_, size_output, interpolation,
                                                   border_mode, boarder_value)
    if out_list is not None:
        for to_path, image in zip(out_list, results):
            _imwrite(to_path, image)
    return results


def _warp_with_first_geometry(transformer, img, size_in, radius_, size_output, interpolation, border_mode, border_value):
    img = np.asarray(img)
    if img.shape[:2] == size_in:
        return warp_host([transformer], [img], radii=[radius_], share_map=True, size_output=size_output,
                         interpolation=interpolation, border_mode=border_mode, border_value=border_value)
    # map geometry (centre, radius) comes from the first image, sampling bounds from this one: FLOAT2 route
    xm, ym = get_map(transformer, radius=radius_, size_input=size_in, size_output=size_output)
    return remap_maps(img, xm, ym, interpolation=interpolation, border_mode=border_mode, border_value=border_value)


def remap_maps(img: NDArray, xmap: NDArray, ymap: NDArray, *, interpolation: int = INTER_LINEAR,
               border_mode: int = BORDER_CONSTANT, border_value: Any = 0) -> NDArray[np.uint8]:
    """cv2.remap(img, xmap, ymap, interpolation, borderMode, borderValue) for uint8 / uint16 images and float32 maps."""
    interpolation, border_mode = _check_modes(interpolation, border_mode)
    xm = np.ascontiguousarray(xmap, dtype=np.float32)
    ym = np.ascontiguousarray(ymap, dtype=np.float32)
    if xm.shape != ym.shape or xm.ndim != 2:
        raise ValueError("xmap / ymap must be 2-D float32 arrays of equal shape")
    view = _as_image(img)
    rows, cols, ch = view.shape
    h, w = xm.shape
    dst = _result_empty((h, w, ch), view.dtype)
    job = N.HostJob()
    job.n_views = job.n_frames = 1
    job.src[0] = view.ctypes.data
    job.src_rows, job.src_cols, job.channels = rows, cols, ch
    job.src_pitch[0] = view.strides[0]
    job.src_frame_stride[0] = view.strides[0] * rows
    job.map_kind = N.MAPSRC_FLOAT2
    job.xmap[0], job.ymap[0] = xm.ctypes.data, ym.ctypes.data
    job.out_w, job.out_h = w, h
    job.interpolation, job.border_mode = interpolation, border_mode
    job.dst, job.dst_pitch, job.dst_frame_stride = dst.ctypes.data, dst.strides[0], dst.strides[0] * h
    _run_job(job, view.dtype, border_value)
    return dst[:, :, 0] if np.asarray(img).ndim == 2 else dst


def _anaglyph_labels(combine: NDArray[np.uint8]) -> NDArray[np.uint8]:
    """The "L" / "R" labels of apply_lr(merge=True) (remapper.py:499-516).  The reference draws them with cv.putText on
    its FLOAT64 image, where OpenCV has no anti-aliasing: pure (0, 128, 255) / (255, 128, 0) pixels with the LINE_8
    raster, which cv.imwrite then stores unchanged -- so drawing with LINE_8 on the uint8 result of vr180_anaglyph is
    the same picture.  (Font scale len(combine) // 1000: nothing is drawn below 1000 rows.)  cv2 only draws text here."""
    import cv2 as cv

    colors = [(0, 128, 255), (255, 128, 0)]
    combine = np.ascontiguousarray(combine)
    cv.putText(combine, "L", (0, len(combine[1]) // 10), cv.FONT_HERSHEY_SIMPLEX, len(combine) // 1000, colors[0], 2,
               cv.LINE_8)
    cv.putText(combine, "R", (len(combine[1]) // 2, len(combine[0]) // 10), cv.FONT_HERSHEY_SIMPLEX,
               len(combine) // 1000, colors[1], 2, cv.LINE_8)
    return combine


def apply_lr(
    transformer: TransformerBase | tuple[TransformerBase, TransformerBase],
    *,
    left_path: Path | str | NDArray,
    right_path: Path | str | NDArray,
    out_path: Path | str,
    size_output: tuple[int, int] = (2048, 2048),
    interpolation: int = INTER_LANCZOS4,
    boarder_mode: int = BORDER_CONSTANT,
    boarder_value: int | tuple[int, int, int] = 0,
    radius: float | Literal["auto", "max"] = "auto",
    merge: bool = False,
) -> None:
    """Stereo pair -> side-by-side frame written to `out_path` (remapper.py:406-520).  Both eyes are warped by
    one kernel launch that writes each eye into its half of the SBS frame (no separate concatenate)."""
    if _codec == "nvjpeg" and _lr_files_on_device(transformer, left_path, right_path, out_path, size_output, interpolation,
                                                  boarder_mode, boarder_value, radius, merge):
        LOG.info(f"Saved to {Path(out_path).absolute()}")
        return
    sbs = lr_frame(transformer, left_path, right_path, size_output=size_output, interpolation=interpolation,
                   boarder_mode=boarder_mode, boarder_value=boarder_value, radius=radius, merge=merge)
    if merge:
        sbs = _anaglyph_labels(sbs)
    _imwrite(out_path, sbs)
    LOG.info(f"Saved to {Path(out_path).absolute()}")


def _lr_files_on_device(transformer, left_path, right_path, out_path, size_output, interpolation, boarder_mode,
                        boarder_value, radius, merge) -> bool:
    """set_codec("nvjpeg"): JPEG inputs are decoded by nvJPEG into device memory, warped there (SbsWarper: the same
    kernels as the host path) and -- for a .jpg output without merge -- encoded there, so only compressed bytes cross
    PCIe (remapper.py:448-456 split, :460-484 radius / map rules, :518-519).  Returns False when the request is not of
    that form (the caller then takes the cv2 path)."""
    from . import codec
    from .video import SbsWarper

    if not (codec.is_jpeg_path(left_path) and codec.is_jpeg_path(right_path) and codec.available()):
        return False
    import torch

    dev = torch.device("cuda", _default_device)
    interpolation, border_mode = _check_modes(interpolation, boarder_mode)
    with torch.cuda.device(dev):
        if Path(left_path) == Path(right_path):  # one SBS source file: halves as views (remapper.py:448-456)
            full = codec.decode_jpeg_device(left_path, dev)
            half = full.shape[1] // 2
            eyes = [full[:, :half], full[:, half:]]
        else:
            eyes = [codec.decode_jpeg_device(p, dev) for p in (left_path, right_path)]
        if eyes[0].shape != eyes[1].shape:
            return False
        rows, cols = int(eyes[0].shape[0]), int(eyes[0].shape[1])
        left, right = (e.unsqueeze(0) for e in eyes)
        per_eye = isinstance(transformer, tuple)
        plan_radius: Any = radius
        if isinstance(radius, str) and radius == "auto":
            probe = SbsWarper(transformer, size_input=(rows, cols), size_output=size_output, interpolation=interpolation,
                              boarder_mode=border_mode, boarder_value=boarder_value, radius="auto", device=dev)
            _, trans = probe.radius_per_frame(left, right)
            trans = trans[0].cpu().numpy()  # (view, {first, last})
            if (trans < 0).any():
                raise IndexError("index 0 is out of bounds for axis 0 with size 0")
            per_view = [(int(t[1]) - int(t[0])) / 2 for t in trans]
            plan_radius = per_view if per_eye else max(per_view)  # remapper.py:460-473 / :82-84
            LOG.info(f"Radius: {plan_radius}, strategy: auto, image shape: {tuple(eyes[0].shape)}")
        wp = SbsWarper(transformer, size_input=(rows, cols), size_output=size_output, interpolation=interpolation,
                       boarder_mode=border_mode, boarder_value=boarder_value, radius=plan_radius, device=dev)
        sbs = wp(left, right)[0]
        w = int(size_output[0])
        if merge:
            out = torch.empty((sbs.shape[0], w, 3), dtype=torch.uint8, device=dev)
            N.check(N.lib().vr180_anaglyph(sbs.data_ptr(), sbs.stride(0), 0, w, int(sbs.shape[0]), 1, out.data_ptr(),
                                           out.stride(0), 0, torch.cuda.current_stream(dev).cuda_stream), "vr180_anaglyph")
            _imwrite(out_path, _anaglyph_labels(out.cpu().numpy()))
        elif codec.is_jpeg_path(out_path):
            Path(out_path).write_bytes(codec.encode_jpeg_device(sbs))
        else:
            _imwrite(out_path, sbs.cpu().numpy())
    return True


def _split_if_same_path(left, right):
    if isinstance(left, (str, Path)) and isinstance(right, (str, Path)) and left == right:
        image = _imread(left)  # one SBS source file: split into halves (views, not copies) -- remapper.py:448-456
        return image[:, : image.shape[1] // 2], image[:, image.shape[1] // 2:]
    return left, right


def lr_frame(transformer, left, right, *, size_output=(2048, 2048), interpolation=INTER_LANCZOS4,
             boarder_mode=BORDER_CONSTANT, boarder_value=0, radius="auto", merge=False) -> NDArray[np.uint8]:
    """The in-memory part of apply_lr: returns the (H, 2W, C) SBS frame, or with merge=True the (H, W, 3) anaglyph of
    the two eyes without its text labels (remapper.py:485-498)."""
    interpolation, border_mode = _check_modes(interpolation, boarder_mode)
    left, right = _split_if_same_path(left, right)
    eyes = [_imread(p) if isinstance(p, (str, Path)) else p for p in (left, right)]
    if merge and any(np.asarray(e).dtype != np.uint8 for e in eyes):
        raise ValueError("merge (the anaglyph) takes uint8 images")
    kw = dict(size_output=size_output, interpolation=interpolation, border_mode=border_mode, border_value=boarder_value)
    # eyes of different dtypes are warped one by one, and np.concatenate promotes the halves as in the reference
    same_shape = (np.asarray(eyes[0]).shape == np.asarray(eyes[1]).shape
                  and np.asarray(eyes[0]).dtype == np.asarray(eyes[1]).dtype)
    fused_merge = merge and same_shape and np.asarray(eyes[0]).ndim == 3 and np.asarray(eyes[0]).shape[2] == 3

    def finish(halves):  # eyes that had to be warped separately
        if merge:
            return _merge_device(halves[0], halves[1])
        return np.concatenate(halves, axis=1)

    if isinstance(transformer, tuple):  # per-eye transformer: own radius and own map per eye (remapper.py:460-473)
        if isinstance(radius, str) and radius == "auto":  # both eyes' scan lines in ONE upload / launch / read
            radii = _device_radius(eyes)
            for eye, r in zip(eyes, radii):
                LOG.info(f"Radius: {r}, strategy: {radius}, image shape: {np.asarray(eye).shape}")
        else:
            radii = [get_radius_smart(radius, [eye]) for eye in eyes]
        if same_shape and (fused_merge or not merge):
            return warp_host(list(transformer), eyes, radii=radii, share_map=False, merge=fused_merge, **kw)
        # eyes of different geometry (unequal crops): the reference runs apply() per eye with that eye's size_input
        return finish([warp_host([t], [eye], radii=[r], share_map=True, **kw) for t, eye, r in zip(transformer, eyes, radii)])
    if (isinstance(radius, str) and radius == "auto" and same_shape and (fused_merge or not merge)
            and np.asarray(eyes[0]).ndim == 3
            and transformer.lower(shape=(int(size_output[1]), int(size_output[0]))) is not None):
        # one radius = max over both eyes (remapper.py:82-84, :475-484), scanned and consumed on the device inside the
        # job: no separate upload / launch / blocking read for the two scan lines
        return warp_host([transformer], eyes, radii=[1.0], share_map=True, auto_radius=True, merge=fused_merge, **kw)
    radius_ = get_radius_smart(radius, eyes)  # one radius = max over both eyes, ONE map (remapper.py:475-484)
    if same_shape and (fused_merge or not merge):
        return warp_host([transformer], eyes, radii=[radius_], share_map=True, merge=fused_merge, **kw)
    # the reference builds the map from the LEFT image's shape and samples the right image with it (remapper.py:385)
    size_in = (np.asarray(eyes[0]).shape[0], np.asarray(eyes[0]).shape[1])
    return finish([_warp_with_first_geometry(transformer, eye, size_in, radius_, size_output, interpolation, border_mode,
                                             boarder_value) for eye in eyes])


def _merge_device(left: NDArray, right: NDArray) -> NDArray[np.uint8]:
    """vr180_anaglyph on two already-warped eyes (the rare paths where they could not share one job)."""
    import torch

    if left.shape != right.shape or left.ndim != 3 or left.shape[2] != 3:
        raise ValueError("anaglyph merge needs two 3-channel images of equal shape")
    dev = torch.device("cuda", _default_device)
    h, w = left.shape[:2]
    sbs = torch.from_numpy(np.concatenate([left, right], axis=1)).to(dev)
    out = torch.empty((h, w, 3), dtype=torch.uint8, device=dev)
    N.check(N.lib().vr180_anaglyph(sbs.data_ptr(), sbs.stride(0), 0, w, h, 1, out.data_ptr(), out.stride(0), 0,
                                   torch.cuda.current_stream(dev).cuda_stream), "vr180_anaglyph")
    return out.cpu().numpy()


def lr_frames(transformer, lefts: Sequence[Any], rights: Sequence[Any], *, size_output=(2048, 2048),
              interpolation=INTER_LANCZOS4, boarder_mode=BORDER_CONSTANT, boarder_value=0,
              radius="auto") -> "list[NDArray[np.uint8]]":
    """apply_lr's in-memory part for a CLIP: `lefts[i]`, `rights[i]` -> SBS frame i, every pair exactly as
    `lr_frame` would produce it (per-pair radius for radius="auto": the max over the pair's eyes,
    remapper.py:82-84, :475-484), but as ONE host job -- uploads, warps and downloads of neighbouring pairs overlap.
    Pairs must share one geometry.  A per-eye transformer tuple with radius="auto" needs a radius per EYE
    (remapper.py:460-473) and is processed pair by pair."""
    interpolation, border_mode = _check_modes(interpolation, boarder_mode)
    if len(lefts) != len(rights):
        raise ValueError("lefts / rights differ in length")
    lefts = [_imread(p) if isinstance(p, (str, Path)) else p for p in lefts]
    rights = [_imread(p) if isinstance(p, (str, Path)) else p for p in rights]
    if not lefts:
        return []
    kw = dict(size_output=size_output, interpolation=interpolation, border_mode=border_mode, border_value=boarder_value)
    auto = isinstance(radius, str) and radius == "auto"
    shapes = {(np.asarray(im).shape, np.asarray(im).dtype) for im in (*lefts, *rights)}
    per_eye = isinstance(transformer, tuple)
    lowerable = all(t.lower(shape=(int(size_output[1]), int(size_output[0]))) is not None
                    for t in (transformer if per_eye else (transformer,)))
    if len(shapes) != 1 or (auto and (per_eye or not lowerable)):
        return [lr_frame(transformer, le, ri, size_output=size_output, interpolation=interpolation,
                         boarder_mode=boarder_mode, boarder_value=boarder_value, radius=radius)
                for le, ri in zip(lefts, rights)]
    ts = list(transformer) if per_eye else [transformer]
    if auto:
        return warp_host(ts, [lefts, rights], radii=[1.0] * len(ts), share_map=not per_eye, auto_radius=True, **kw)
    radius_ = get_radius_smart(radius, [lefts[0], rights[0]])  # "max" / a number: the same for every pair
    return warp_host(ts, [lefts, rights], radii=[radius_] * len(ts), share_map=not per_eye, **kw)


def match_lr(
    decoder: TransformerBase | tuple[TransformerBase, TransformerBase],
    points_l: Sequence[tuple[float, float]],
    points_r: Sequence[tuple[float, float]],
    in_paths: Sequence[Path | str | NDArray],
    *,
    radius: float | Literal["auto", "max"] = "auto",
) -> tuple[NDArray, NDArray]:
    """Matched pixel positions of the two eyes -> unit vectors, the arguments of rotation_match() (remapper.py:251-321):
    (decoder * Denormalize(scale=(r, r), center)).inverse_transform on the points, then equidistant_to_3d.  All points
    of the call go through ONE vr180_transform_points launch per decoder (float64 on the device; the reference runs
    the same chain in float32 NumPy, so results agree to float32 rounding).  `in_paths` may hold arrays as well."""
    import torch

    if len(points_l) != len(points_r):
        raise ValueError("The number of points must be the same.")
    images = [_imread(p) if isinstance(p, (str, Path)) else p for p in in_paths]
    center = (images[0].shape[1] // 2, images[0].shape[0] // 2)
    radius_ = get_radius_smart(radius, images)
    dev = torch.device("cuda", _default_device)
    stream = torch.cuda.current_stream(dev).cuda_stream

    def to_3d(dec: TransformerBase, pts) -> NDArray:
        pts = np.asarray(pts, dtype=np.float64).reshape(-1, 2).astype(np.float32).astype(np.float64)  # :295, :309
        chain_t = dec * DenormalizeTransformer(scale=(radius_, radius_), center=center)
        ops = chain_t.lower(inverse=True)
        if ops is None or len(ops) > N.MAX_OPS:  # user-defined decoder: its own NumPy code
            from .transformer import equidistant_to_3d

            x, y = chain_t.inverse_transform(pts[:, 0], pts[:, 1])
            return equidistant_to_3d(x, y)
        chain = N.make_chain(ops)
        xy = torch.from_numpy(np.ascontiguousarray(pts.T)).to(dev)
        v3 = torch.empty((pts.shape[0], 3), dtype=torch.float64, device=dev)
        N.check(N.lib().vr180_transform_points(C.byref(chain), pts.shape[0], xy[0].data_ptr(), xy[1].data_ptr(), None,
                                               None, v3.data_ptr(), stream), "vr180_transform_points")
        return v3.cpu().numpy()

    if isinstance(decoder, tuple):
        return to_3d(decoder[0], points_l), to_3d(decoder[1], points_r)
    v = to_3d(decoder, np.concatenate([np.asarray(points_l).reshape(-1, 2), np.asarray(points_r).reshape(-1, 2)], axis=0))
    return v[: len(points_l)], v[len(points_l):]
