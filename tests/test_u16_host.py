"""16-bit (uint16) images without a GPU: the float restatement of cv::remap (oracle/remap_float_np.py) against the
installed cv2.remap, the C ABI's depth fields and new entry points, and the Python layer's dtype checks."""
from __future__ import annotations

import ctypes as C
import itertools
import subprocess
from pathlib import Path

import cv2
import numpy as np
import pytest

import vr180_convert_b200 as V
from oracle import remap_float_np as RF
from vr180_convert_b200 import _native as N

ROOT = Path(__file__).resolve().parent.parent
COLOURS = [0, 70000.4, (60000, 1000, 7, 300), (256.5, 65535.5, 300.5, 1e9)]


def _maps(rng, h, w, hout, wout, reach=9):
    xm = rng.uniform(-reach, w + reach, (hout, wout)).astype(np.float32)
    ym = rng.uniform(-reach, h + reach, (hout, wout)).astype(np.float32)
    return xm, ym


@pytest.mark.parametrize("interp", [0, 1, 2, 4])
def test_float_oracle_matches_cv2_every_border_and_channel_count(interp):
    rng = np.random.default_rng(interp)
    for ch, border in itertools.product((1, 3, 4), range(5)):
        src = rng.integers(0, 65536, (97, 131, ch), dtype=np.uint16)
        src = src[..., 0] if ch == 1 else src
        xm, ym = _maps(rng, 97, 131, 23, 37)
        for bv in COLOURS:
            want = cv2.remap(src, xm, ym, interp, borderMode=border, borderValue=bv)
            got = RF.remap(src, xm, ym, interp, border, bv)
            assert got.dtype == np.uint16 and np.array_equal(got, want), (interp, ch, border, bv)


@pytest.mark.parametrize("interp", [2, 4])
def test_border_colour_reaches_non_constant_modes(interp):
    """cv::remap's CUBIC / LANCZOS4 start the edge sum at the border colour in EVERY mode (s = cval + sum (S - cval) w),
    so the colour changes some results under REPLICATE / REFLECT / WRAP / REFLECT_101 too."""
    rng = np.random.default_rng(5)
    src = rng.integers(0, 65536, (64, 80, 3), dtype=np.uint16)
    xm, ym = _maps(rng, 64, 80, 64, 80, reach=6)
    for border in (1, 2, 3, 4):
        a = cv2.remap(src, xm, ym, interp, borderMode=border, borderValue=0)
        b = cv2.remap(src, xm, ym, interp, borderMode=border, borderValue=(60000, 1000, 7))
        assert (a != b).any(), border
        assert np.array_equal(RF.remap(src, xm, ym, interp, border, 0), a)
        assert np.array_equal(RF.remap(src, xm, ym, interp, border, (60000, 1000, 7)), b)


def _adversarial_maps(h, w):
    vals = [np.nan, np.inf, -np.inf, 1e9, -1e9, 7e7, -7e7]
    # ties of cvRound(x * 32) and of cvRound(x) (NEAREST), both parities
    vals += [k + d / 32 for k in (3, 4, 10) for d in (0.5, 1.5, 15.5, 16.5, 31.5)] + [2.5, 3.5, -0.5, -1.5]
    # every interpolation's interior / edge boundary: x = -4 .. 3 and w - 5 .. w + 3 (plus a hair either side)
    for b in [*range(-4, 4), *range(w - 5, w + 4)]:
        vals += [b, b - 1 / 64, b + 1 / 64]
    xs = np.array(vals, np.float32)
    ys = np.array([v * h / w if np.isfinite(v) and abs(v) < 1e6 else v for v in vals], np.float32)
    xm, ym = np.meshgrid(xs, ys)
    return xm.astype(np.float32), ym.astype(np.float32)


@pytest.mark.parametrize("interp", [0, 1, 2, 4])
def test_float_oracle_adversarial_maps(interp):
    rng = np.random.default_rng(9)
    h, w = 21, 29
    xm, ym = _adversarial_maps(h, w)
    for ch, border in itertools.product((1, 3, 4), range(5)):
        src = rng.integers(0, 65536, (h, w, ch), dtype=np.uint16)
        src = src[..., 0] if ch == 1 else src
        for bv in (0, (65535, 40000, 300, 12345)):
            want = cv2.remap(src, xm, ym, interp, borderMode=border, borderValue=bv)
            assert np.array_equal(RF.remap(src, xm, ym, interp, border, bv), want), (interp, ch, border, bv)


def test_float_tables_are_the_unfixed_products():
    """The float tables are the products the int16 tables round (no sum fix-up), so they round back to them except
    at the fix-up entries."""
    from oracle import remap_np

    for interp in (2, 4):
        f = RF.float_table(interp)
        i16 = remap_np.weight_table(interp).astype(np.int64)
        r = np.clip(np.rint((f * np.float32(32768)).astype(np.float32)), -32768, 32767).astype(np.int64)
        assert (r != i16).sum(axis=(1, 2)).max() <= 1


def test_depth_fields_and_new_entry_points():
    header = (ROOT / "include" / "vr180_b200.h").read_text()
    assert "VR180_DEPTH_8U = 0" in header and "VR180_DEPTH_16U = 2" in header
    assert N.DEPTH_8U == 0 and N.DEPTH_16U == 2
    handle = N.lib()
    for name in ("vr180_remap_ex", "vr180_ctx_run_ex"):
        assert hasattr(handle, name) and name in N.SYMBOLS
    assert N.Image.depth.offset == 20 and N.HostJob.depth.offset == 36


def test_depth_fields_gcc_layout(tmp_path):
    src = tmp_path / "depth.c"
    src.write_text("\n".join([
        '#include <stdio.h>', '#include <stddef.h>', '#include "vr180_b200.h"', "int main(void) {",
        'printf("%zu %zu %zu %zu\\n", offsetof(vr180_image_t, depth), sizeof(vr180_image_t),',
        '       offsetof(vr180_host_job_t, depth), sizeof(vr180_host_job_t));',
        "return 0; }"]))
    exe = tmp_path / "depth"
    subprocess.run(["gcc", "-I", str(ROOT / "include"), str(src), "-o", str(exe)], check=True)
    got = [int(v) for v in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split()]
    assert got == [N.Image.depth.offset, C.sizeof(N.Image), N.HostJob.depth.offset, C.sizeof(N.HostJob)]


@pytest.mark.parametrize("dtype", [np.int16, np.float32, np.int8, np.uint32, np.float64])
def test_other_dtypes_raise_type_error_naming_both(dtype):
    img = np.zeros((8, 8, 3), dtype)
    m = np.zeros((4, 4), np.float32)
    with pytest.raises(TypeError, match="uint8 or uint16"):
        V.remap_maps(img, m, m)
    with pytest.raises(TypeError, match="uint8 or uint16"):
        V.apply(V.FisheyeDecoder("equidistant"), in_paths=img, radius="auto")


def test_merge_on_uint16_raises_value_error():
    img = np.zeros((16, 16, 3), np.uint16)
    with pytest.raises(ValueError, match="uint8"):
        V.lr_frame(V.FisheyeDecoder("equidistant"), img, img, size_output=(8, 8), radius=4.0, merge=True)
