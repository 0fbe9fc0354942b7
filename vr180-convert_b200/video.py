"""Batched, device-resident stereo warping for video: N fisheye pairs -> N side-by-side equirect frames.

The reference handles "many frames, one map" with `apply`'s image loop (remapper.py:381-398: ONE get_map, then
cv.remap per image) followed by np.concatenate per pair (:518).  Here a batch of frames already resident in
HBM (torch CUDA tensors are only the buffer type) is warped by one kernel launch per batch:

  * map_source="analytic": the fused kernel evaluates the chain per output pixel in registers -- no LUT exists;
  * map_source="lut":      float32 maps built once (k_build_map, or the host for opaque transformers), cached;
  * map_source="lut_fixed": the maps quantised once to cv2's fixed-point (k_pack_lut), cached;
  * map_source="lut_packed": the tile-packed 4-byte LUT (k_pack_tiles): one 128-bit load per thread, cached;
  * map_source="auto" (default): "analytic" for batches; a plan with a fixed radius that is called again and again
    with one or a few pairs (a frame-at-a-time video loop) builds the tile-packed LUT on its second such call and
    serves them from it -- vr180_remap then streams the tiles through persistent CTAs (csrc/stream.cu): a 4K pair
    takes 25 us instead of 60 us, an 8K pair 110 us instead of ~300 us.  Costs 12 bytes of HBM per output pixel and map.
    (Capturing calls in a CUDA graph: pass the source explicitly, or let the plan build its LUT -- `packed_lut()` --
    before the capture, so that no LUT construction lands inside the graph);
  * radius="auto": k_get_radius per frame (max over the two eyes) feeds the warp kernel through device memory.

Frames of a clip are independent, so multi-GPU runs shard them statically with `shard_range` (no collective).
"""
from __future__ import annotations

import ctypes as C
from typing import Any, Literal, Sequence

import numpy as np

from . import _native as N
from .remapper import (BORDER_CONSTANT, INTER_LINEAR, INTER_NEAREST, _border_bytes, _border_scalar, _check_modes,
                       host_maps, lower_full)
from .shard import shard_range  # noqa: F401  (re-exported)
from .transformer import TransformerBase


class SbsWarper:
    """Plan for warping stereo pairs of one geometry with one transformer (or a per-eye tuple)."""

    def __init__(
        self,
        transformer: TransformerBase | tuple[TransformerBase, TransformerBase],
        *,
        size_input: tuple[int, int],
        size_output: tuple[int, int] = (2048, 2048),
        interpolation: int = INTER_LINEAR,
        boarder_mode: int = BORDER_CONSTANT,
        boarder_value: Any = 0,
        radius: float | Sequence[float] | Literal["auto", "max"] = "max",
        map_source: Literal["auto", "analytic", "lut", "lut_fixed", "lut_packed"] = "auto",
        channels: int = 3,
        threshold: float = 10,
        device: Any = None,
    ) -> None:
        import torch

        self.torch = torch
        self.device = torch.device("cuda", torch.cuda.current_device()) if device is None else torch.device(device)
        self.transformers = list(transformer) if isinstance(transformer, tuple) else [transformer]
        self.share_map = len(self.transformers) == 1
        self.rows, self.cols = int(size_input[0]), int(size_input[1])
        self.w, self.h = int(size_output[0]), int(size_output[1])
        self.interpolation, self.border_mode = _check_modes(interpolation, boarder_mode)
        self.border_value = _border_bytes(boarder_value, channels)
        self.border_scalar = _border_scalar(boarder_value)  # 16-bit frames: saturated by the library
        self.channels = channels
        self.threshold = float(threshold)
        if map_source not in ("auto", "analytic", "lut", "lut_fixed", "lut_packed"):
            raise ValueError(f"unknown map_source {map_source!r}")
        self.map_source = map_source
        self._small_calls = 0  # "auto": calls with <= _STREAM_ITEMS (frame, eye) items per tile so far
        self.auto_radius = isinstance(radius, str) and radius == "auto"
        if self.auto_radius and map_source not in ("analytic", "auto"):
            raise ValueError('radius="auto" per frame is consumed on the device by the analytic kernel only')
        if isinstance(radius, str) and radius == "max":
            radius = min(self.rows / 2, self.cols / 2)
        if self.auto_radius:
            radii = [1.0] * len(self.transformers)  # placeholder scale; replaced per frame from device memory
        elif np.isscalar(radius):
            radii = [float(radius)] * len(self.transformers)
        else:
            radii = [float(r) for r in radius]
        self.radii = radii
        self._lowered = [lower_full(t, radius=r, size_input=(self.rows, self.cols), size_output=(self.w, self.h))
                         for t, r in zip(self.transformers, radii)]
        self._lowerable = all(o is not None for o in self._lowered)
        if map_source == "analytic" and not self._lowerable:
            raise ValueError("transformer has no lowering (user-defined Python class): use map_source='lut'")
        if self.auto_radius and not self._lowerable:
            raise ValueError('radius="auto" per frame needs a lowerable transformer (the analytic kernel consumes it)')
        if map_source == "lut_fixed" and self.interpolation == INTER_NEAREST:
            raise ValueError("the fixed-point LUT stores x*32; INTER_NEAREST needs map_source='lut' or 'analytic'")
        self._chains = [N.make_chain(o) if o is not None else None for o in self._lowered]
        self._maps = None   # (n_maps, 2, H, W) float32 on device
        self._fixed = None  # (n_maps, H, W, 2) int32 on device
        self._packed = None  # n_maps tile-packed LUTs (uint8 buffers) on device, built for self.interpolation
        self._radius_buf = None
        self._trans_buf = None

    # --- LUT construction (once per plan) --------------------------------------------------------------
    def maps(self):
        """float32 maps on the device, shape (n_maps, 2, H, W): built by k_build_map for lowerable chains."""
        torch = self.torch
        if self._maps is None:
            lib = N.lib()
            stream = torch.cuda.current_stream(self.device).cuda_stream
            maps = torch.empty((len(self.transformers), 2, self.h, self.w), dtype=torch.float32, device=self.device)
            for m, (t, r) in enumerate(zip(self.transformers, self.radii)):
                if self._chains[m] is not None:
                    N.check(lib.vr180_build_map(C.byref(self._chains[m]), self.w, self.h, maps[m, 0].data_ptr(),
                                                maps[m, 1].data_ptr(), self.w, stream), "vr180_build_map")
                else:
                    xm, ym = host_maps(t, radius=r, size_input=(self.rows, self.cols), size_output=(self.w, self.h))
                    maps[m, 0].copy_(torch.from_numpy(xm))
                    maps[m, 1].copy_(torch.from_numpy(ym))
            self._maps = maps
        return self._maps

    def fixed_lut(self):
        """cv2-exact fixed-point LUT (n_maps, H, W, 2) int32 = cvRound(map*32), from k_pack_lut."""
        torch = self.torch
        if self._fixed is None:
            maps = self.maps()
            fixed = torch.empty((maps.shape[0], self.h, self.w, 2), dtype=torch.int32, device=self.device)
            stream = torch.cuda.current_stream(self.device).cuda_stream
            for m in range(maps.shape[0]):
                N.check(N.lib().vr180_pack_lut(maps[m, 0].data_ptr(), maps[m, 1].data_ptr(), self.w, self.w, self.h,
                                               fixed[m].data_ptr(), self.w, stream), "vr180_pack_lut")
            self._fixed = fixed
        return self._fixed

    def packed_lut(self):
        """Tile-packed LUT (vr180_pack_lut_tiles) per map for this plan's interpolation: 16-byte tile headers + 4 bytes
        per pixel in the tiled kernel's thread order; the float32 maps stay alongside for tiles that cannot be packed."""
        torch = self.torch
        if self._packed is None:
            maps = self.maps()
            lib = N.lib()
            nbytes = int(lib.vr180_packed_lut_bytes(self.w, self.h, self.interpolation))
            if nbytes == 0:
                raise ValueError("no tiled mode for this interpolation")
            stream = torch.cuda.current_stream(self.device).cuda_stream
            packed = torch.empty((maps.shape[0], nbytes), dtype=torch.uint8, device=self.device)
            for m in range(maps.shape[0]):
                N.check(lib.vr180_pack_lut_tiles(maps[m, 0].data_ptr(), maps[m, 1].data_ptr(), self.w, self.w, self.h,
                                                 self.interpolation, packed[m].data_ptr(), stream), "vr180_pack_lut_tiles")
            self._packed = packed
        return self._packed

    # --- per batch ---------------------------------------------------------------------------------------
    # (frame, eye) rectangles per tile up to which vr180_remap streams the tiles (csrc/tiled.cu: 20 with a shared map)
    _STREAM_ITEMS = {True: 20, False: 16}

    def _source_for(self, n_frames: int, wide: bool = False) -> str:
        """The coordinate source of one call: the plan's, or for "auto" the faster one for this batch size (`wide`:
        16-bit frames, which the tile-streaming kernel does not take)."""
        if self.map_source != "auto":
            return self.map_source
        has_tiled_lut = self.channels == 3 and not wide
        if not self._lowerable:  # user-defined Python transformer: host maps, once
            return "lut_packed" if has_tiled_lut else "lut"
        if self.auto_radius or not has_tiled_lut:
            return "analytic"
        if n_frames * (2 if self.share_map else 1) > self._STREAM_ITEMS[self.share_map]:
            return "analytic"
        self._small_calls += 1  # the first small call is not worth a LUT yet (a plan used once)
        return "lut_packed" if self._small_calls > 1 or self._packed is not None else "analytic"

    def _image(self, t) -> N.Image:
        torch = self.torch
        depths = {torch.uint8: N.DEPTH_8U, torch.uint16: N.DEPTH_16U}
        if t.dtype not in depths:
            raise TypeError(f"frames must be torch.uint8 or torch.uint16, got {t.dtype}")
        if t.dim() != 4 or t.shape[1] != self.rows or t.shape[2] != self.cols \
                or t.shape[3] != self.channels or t.stride(3) != 1 or t.stride(2) != self.channels:
            raise ValueError(f"frames must be (F, {self.rows}, {self.cols}, {self.channels}) with contiguous pixels")
        e = t.element_size()  # torch strides count elements; the ABI's pitches are bytes
        return N.Image(t.data_ptr(), self.rows, self.cols, self.channels, depths[t.dtype], t.stride(1) * e,
                       t.stride(0) * e)

    def radius_per_frame(self, left, right):
        """k_get_radius over the batch: float64 radius per frame (max over both eyes) and the raw transitions."""
        torch = self.torch
        n = left.shape[0]
        if self._radius_buf is None or self._radius_buf.shape[0] < n:
            self._radius_buf = torch.empty(n, dtype=torch.float64, device=self.device)
            self._trans_buf = torch.empty((n, 2, 2), dtype=torch.int32, device=self.device)
        ims = (N.Image * 2)(self._image(left), self._image(right))
        stream = torch.cuda.current_stream(self.device).cuda_stream
        N.check(N.lib().vr180_get_radius(ims, 2, n, self.threshold, self._trans_buf.data_ptr(),
                                         self._radius_buf.data_ptr(), stream), "vr180_get_radius")
        return self._radius_buf[:n], self._trans_buf[:n]

    def __call__(self, left, right, out=None, radius=None):
        """left / right: uint8 or uint16 CUDA tensors (F, rows, cols, C) -> out (F, H, 2W, C) of the same dtype, eyes
        side by side.

        `radius` (plans built with radius="auto" only): float64 CUDA tensor (F,) of per-frame radii to use instead
        of running get_radius, e.g. radii estimated once and smoothed over a clip; NaN = "no transition found"."""
        torch = self.torch
        n = left.shape[0]
        if right.shape != left.shape or right.dtype != left.dtype:
            raise ValueError("left / right batches differ in shape or dtype")
        wide = left.dtype == torch.uint16
        if out is None:
            out = torch.empty((n, self.h, 2 * self.w, self.channels), dtype=left.dtype, device=self.device)
        if out.dtype != left.dtype:
            raise ValueError("out must have the dtype of the frames")
        p = N.RemapParams()
        p.n_views, p.n_frames = 2, n
        p.share_map = 1 if self.share_map else 0
        p.out_w, p.out_h = self.w, self.h
        p.interpolation, p.border_mode = self.interpolation, self.border_mode
        for i, b in enumerate(self.border_value):
            p.border_value[i] = b
        e = out.element_size()
        p.dst, p.dst_pitch, p.dst_frame_stride = out.data_ptr(), out.stride(1) * e, out.stride(0) * e
        radius_dev = None
        if radius is not None:
            if not self.auto_radius:
                raise ValueError('per-frame radii need a plan built with radius="auto"')
            if radius.dtype != torch.float64 or radius.dim() != 1 or radius.shape[0] != n or not radius.is_contiguous():
                raise ValueError(f"radius must be a contiguous float64 CUDA tensor of shape ({n},)")
            radius_dev = radius
        elif self.auto_radius:
            radius_dev, _ = self.radius_per_frame(left, right)
        source = self._source_for(n, wide)
        for v, frames in enumerate((left, right)):
            vw = p.view[v]
            vw.src = self._image(frames)
            vw.dst_x_offset = v * self.w
            m = 0 if self.share_map else v
            if source == "analytic":
                vw.map.kind = N.MAPSRC_ANALYTIC
                vw.map.chain = C.pointer(self._chains[m])
                vw.map.radius_dev = radius_dev.data_ptr() if radius_dev is not None else None
            elif source == "lut":
                maps = self.maps()
                vw.map.kind = N.MAPSRC_FLOAT2
                vw.map.xmap, vw.map.ymap, vw.map.map_pitch = maps[m, 0].data_ptr(), maps[m, 1].data_ptr(), self.w
            elif source == "lut_packed":
                maps, packed = self.maps(), self.packed_lut()
                vw.map.kind = N.MAPSRC_PACKED
                vw.map.xmap, vw.map.ymap, vw.map.map_pitch = maps[m, 0].data_ptr(), maps[m, 1].data_ptr(), self.w
                vw.map.packed, vw.map.packed_interpolation = packed[m].data_ptr(), self.interpolation
            else:
                fixed = self.fixed_lut()
                vw.map.kind = N.MAPSRC_FIXED
                vw.map.fixed, vw.map.map_pitch = fixed[m].data_ptr(), self.w
        stream = torch.cuda.current_stream(self.device).cuda_stream
        if wide:
            N.check(N.lib().vr180_remap_ex(C.byref(p), self.border_scalar, stream), "vr180_remap_ex")
        else:
            N.check(N.lib().vr180_remap(C.byref(p), stream), "vr180_remap")
        return out
