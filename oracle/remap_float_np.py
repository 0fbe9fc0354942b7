"""ORACLE (test infrastructure, NOT product code) -- float32 restatement of `cv2.remap` for uint16 images.

For depths other than 8 bits cv::remap (modules/imgproc/src/imgwarp.cpp: remapBilinear / remapBicubic / remapLanczos4)
uses float weights instead of the int16 tables of the 8-bit path (remap_np.py):

  * coordinates are quantised exactly as for uint8 (sx = cvRound(x * 32), ix = sx >> 5, ax = sx & 31; NEAREST rounds x);
  * 1-D tables t = float(i) * float(1/32): bilinear {1 - t, t}, cubic / Lanczos4 the float coefficients of
    remap_np._coef_cubic / _coef_lanczos4; 2-D weight w[ky][kx] = float32(tab[ay][ky] * tab[ax][kx]), no sum fix-up;
  * every product and sum is one float32 operation (no fused multiply-add), in OpenCV's order;
  * result = saturate(cvRound(s)), round half to even.

Pinned live against the installed `cv2.remap` by tests/test_u16_host.py.  Only tests/, scripts/ and bench legs may
import this module.
"""
from __future__ import annotations

import numpy as np

from .remap_np import (BORDER_CONSTANT, INTER_CUBIC, INTER_LANCZOS4, INTER_LINEAR, INTER_NEAREST, _coef_cubic,
                       _coef_lanczos4, _fetch, _sat16, cv_round_f32, quantise)

_FTAB_CACHE: dict[int, np.ndarray] = {}


def float_table(interpolation: int) -> np.ndarray:
    """float32 table [ay*32+ax][ky][kx]: w = float32(tab[ay][ky] * tab[ax][kx]) rounded once (initInterTab2D with
    fixpt = false: no fix-up of the sum)."""
    if interpolation in _FTAB_CACHE:
        return _FTAB_CACHE[interpolation]
    f = np.float32
    if interpolation == INTER_LINEAR:
        one = [np.array([f(1) - f(i) * f(1 / 32), f(i) * f(1 / 32)], np.float32) for i in range(32)]
    elif interpolation == INTER_CUBIC:
        one = [_coef_cubic(f(i) * f(1 / 32)) for i in range(32)]
    elif interpolation == INTER_LANCZOS4:
        one = [_coef_lanczos4(f(i) * f(1 / 32)) for i in range(32)]
    else:
        raise ValueError(interpolation)
    k = len(one[0])
    tab = np.zeros((1024, k, k), np.float32)
    for ay in range(32):
        for ax in range(32):
            tab[ay * 32 + ax] = one[ay][:, None] * one[ax][None, :]
    _FTAB_CACHE[interpolation] = tab
    return tab


def border_scalar_u16(value, channels: int) -> np.ndarray:
    """cv::Scalar -> per-channel border colour of a uint16 image: saturate_cast<ushort> (round half to even, clamp);
    a Python scalar fills channel 0 only."""
    v = [value, 0, 0, 0] if np.isscalar(value) else (list(value) + [0] * 4)[:4]
    return np.clip(np.rint(np.asarray(v[:channels], np.float64)), 0, 65535).astype(np.int64)


def remap(src: np.ndarray, xmap: np.ndarray, ymap: np.ndarray, interpolation: int = INTER_LINEAR,
          border_mode: int = BORDER_CONSTANT, border_value=0) -> np.ndarray:
    """Bit-exact restatement of cv2.remap(src uint16 HxW[xC], float32 maps, ...)."""
    if src.dtype != np.uint16:
        raise TypeError("remap_float_np restates the uint16 path; uint8 is remap_np.remap")
    squeeze = src.ndim == 2
    if squeeze:
        src = src[..., None]
    h, w, c = src.shape
    cval = border_scalar_u16(border_value, c)
    fc = cval.astype(np.float32)
    xmap = np.asarray(xmap, np.float32)
    ymap = np.asarray(ymap, np.float32)

    if interpolation == INTER_NEAREST:
        out = _fetch(src, _sat16(cv_round_f32(ymap)), _sat16(cv_round_f32(xmap)), border_mode, cval)
        out = out.astype(np.uint16)
        return out[..., 0] if squeeze else out

    ix, iy, ax, ay = quantise(xmap, ymap)
    wt = float_table(interpolation)[ay * 32 + ax]  # (..., k, k) float32
    k = wt.shape[-1]
    off = k // 2 - 1
    x0, y0 = ix - off, iy - off

    def tap(ky, kx):
        return _fetch(src, y0 + ky, x0 + kx, border_mode, cval).astype(np.float32)

    def wk(ky, kx):
        return wt[..., ky, kx][..., None]

    if interpolation == INTER_LINEAR:
        # ((v00 w00 + v01 w01) + v10 w10) + v11 w11, inside and at the edges; a footprint entirely outside the source
        # under BORDER_CONSTANT is the border colour itself
        s = tap(0, 0) * wk(0, 0) + tap(0, 1) * wk(0, 1)
        s = s + tap(1, 0) * wk(1, 0)
        s = s + tap(1, 1) * wk(1, 1)
        if border_mode == BORDER_CONSTANT:
            out_all = (ix >= w) | (ix + 1 < 0) | (iy >= h) | (iy + 1 < 0)
            s = np.where(out_all[..., None], fc, s)
    else:
        # interior: each row summed left to right, then the rows left to right
        s_in = None
        for ky in range(k):
            r = tap(ky, 0) * wk(ky, 0)
            for kx in range(1, k):
                r = r + tap(ky, kx) * wk(ky, kx)
            s_in = r if s_in is None else s_in + r
        # elsewhere, in EVERY border mode: s = cval, then s += (S - cval) * w for each valid tap in row-major order
        # (under BORDER_CONSTANT a tap outside the source is not valid; other modes remap its index)
        s_edge = np.broadcast_to(fc, s_in.shape).copy()
        for ky in range(k):
            for kx in range(k):
                d = (tap(ky, kx) - fc) * wk(ky, kx)
                if border_mode == BORDER_CONSTANT:
                    valid = ((x0 + kx >= 0) & (x0 + kx < w) & (y0 + ky >= 0) & (y0 + ky < h))[..., None]
                    s_edge = np.where(valid, s_edge + d, s_edge)
                else:
                    s_edge = s_edge + d
        inside = ((x0 >= 0) & (x0 < w - (k - 1)) & (y0 >= 0) & (y0 < h - (k - 1)))[..., None]
        s = np.where(inside, s_in, s_edge)
    out = np.clip(np.rint(s.astype(np.float64)), 0, 65535).astype(np.uint16)
    return out[..., 0] if squeeze else out


def apply_lr_sbs(src_l, src_r, maps_l, maps_r, interpolation=INTER_LINEAR, border_mode=BORDER_CONSTANT,
                 border_value=0):
    """remapper.py:388-398 per eye + np.concatenate(axis=1) (:518), uint16."""
    left = remap(src_l, maps_l[0], maps_l[1], interpolation, border_mode, border_value)
    right = remap(src_r, maps_r[0], maps_r[1], interpolation, border_mode, border_value)
    return np.concatenate([left, right], axis=1)


__all__ = ["float_table", "border_scalar_u16", "remap", "apply_lr_sbs", "INTER_NEAREST", "INTER_LINEAR",
           "INTER_CUBIC", "INTER_LANCZOS4"]
