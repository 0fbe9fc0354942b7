"""16-bit (uint16) images on the GPU: every frame bit for bit against cv2.remap on uint16 (float-weight arithmetic of
cv::remap for non-8-bit depths), through the host pipeline (remap_maps / apply / lr_frame / lr_frames) and the
device-resident SbsWarper, for every interpolation, border mode, coordinate source and radius form."""
from __future__ import annotations

import itertools

import cv2
import numpy as np
import pytest

import vr180_convert_b200 as V
from oracle import chain_np
from vr180_convert_b200 import _native as N

pytestmark = pytest.mark.gpu

COLOURS = [0, 70000.4, (60000, 1000, 7, 300)]


def _chain(q=(0.03, -0.02, 0.05)):
    rot = V.from_rotation_vector(list(q))
    t = V.EquirectangularEncoder() * V.Euclidean3DRotator(rot) * V.PolynomialScaler([0, 1, 0.05]) * V.FisheyeDecoder(
        "equidistant")
    ops = [("equirect_enc", True), ("rot3", chain_np.quat_to_matrix(*rot.components).ravel().tolist()),
           ("poly", [0, 1, 0.05]), ("fisheye_dec", "equidistant")]
    return t, ops


def _disc16(n, h, w, seed, margin=8):
    rng = np.random.default_rng(seed)
    img = rng.integers(0, 65536, (n, h, w, 3), dtype=np.uint16)
    yy, xx = np.ogrid[:h, :w]
    r = min(h, w) // 2 - margin - seed % 5
    img[:, (xx - w // 2) ** 2 + (yy - h // 2) ** 2 > r * r] = 0
    return img


def _cv2_sbs(lf, rf, ml, mr, interp, border, bv):
    return np.concatenate([cv2.remap(lf, ml[0], ml[1], interp, borderMode=border, borderValue=bv),
                           cv2.remap(rf, mr[0], mr[1], interp, borderMode=border, borderValue=bv)], axis=1)


@pytest.mark.parametrize("interp", [0, 1, 2, 4])
def test_remap_maps_uint16_every_border_channel_and_colour(interp):
    rng = np.random.default_rng(interp)
    for ch, border in itertools.product((1, 3, 4), range(5)):
        src = rng.integers(0, 65536, (97, 131, ch), dtype=np.uint16)
        src = src[..., 0] if ch == 1 else src
        xm = rng.uniform(-9, 140, (45, 70)).astype(np.float32)
        ym = rng.uniform(-9, 106, (45, 70)).astype(np.float32)
        xm[0, :5] = [np.nan, np.inf, -np.inf, 1e9, -1e9]
        for bv in COLOURS:
            got = V.remap_maps(src, xm, ym, interpolation=interp, border_mode=border, border_value=bv)
            want = cv2.remap(src, xm, ym, interp, borderMode=border, borderValue=bv)
            assert got.dtype == np.uint16 and np.array_equal(got, want), (interp, ch, border, bv)


@pytest.mark.parametrize("interp", [0, 1, 2, 4])
@pytest.mark.parametrize("per_eye", [False, True])
def test_sbs_warper_uint16_sources_borders_and_colours(interp, per_eye):
    import torch

    n, hin, win, wout, hout = 5, 192, 224, 208, 104  # the footprint leaves the source on every side (radius 150)
    tl, ol = _chain((0.03, -0.02, 0.05))
    tr, orr = _chain((-0.03, 0.02, -0.05))
    t = (tl, tr) if per_eye else tl
    rng = np.random.default_rng(3)
    ln = rng.integers(0, 65536, (n, hin, win, 3), dtype=np.uint16)
    rn = rng.integers(0, 65536, (n, hin, win, 3), dtype=np.uint16)
    left, right = torch.from_numpy(ln).cuda(), torch.from_numpy(rn).cuda()
    radius = 150.0
    ml = chain_np.get_map(ol, radius=radius, size_input=(hin, win), size_output=(wout, hout))
    mr = chain_np.get_map(orr, radius=radius, size_input=(hin, win), size_output=(wout, hout)) if per_eye else ml
    for border, bv in itertools.product(range(5), COLOURS):
        for src in ("analytic", "lut", "lut_fixed", "lut_packed"):
            if src == "lut_fixed" and interp == 0:
                continue
            wp = V.SbsWarper(t, size_input=(hin, win), size_output=(wout, hout), interpolation=interp,
                             boarder_mode=border, boarder_value=bv, radius=radius, map_source=src)
            got = wp(left, right).cpu().numpy()
            assert got.dtype == np.uint16
            for f in range(n):
                want = _cv2_sbs(ln[f], rn[f], ml, mr, interp, border, bv)
                assert np.array_equal(got[f], want), (interp, per_eye, border, bv, src, f)


@pytest.mark.parametrize("interp", [0, 1, 2, 4])
def test_sbs_warper_uint16_per_frame_and_nan_radius(interp):
    import torch

    hin, win, wout, hout = 192, 224, 160, 96
    radii = [90.0, 150.0, float("nan"), -100.5, 60.25, 149.5, 33.0]
    n = len(radii)
    t, ops = _chain()
    rng = np.random.default_rng(11)
    ln = rng.integers(0, 65536, (n, hin, win, 3), dtype=np.uint16)
    rn = rng.integers(0, 65536, (n, hin, win, 3), dtype=np.uint16)
    left, right = torch.from_numpy(ln).cuda(), torch.from_numpy(rn).cuda()
    bv = (60000, 1000, 7)
    wp = V.SbsWarper(t, size_input=(hin, win), size_output=(wout, hout), interpolation=interp, radius="auto",
                     boarder_value=bv)
    got = wp(left, right, radius=torch.tensor(radii, dtype=torch.float64, device="cuda")).cpu().numpy()
    for f, r in enumerate(radii):
        if r != r:
            assert (got[f] == np.array(bv, np.uint16)).all(), f  # NaN coordinates: the border colour everywhere
            continue
        m = chain_np.get_map(ops, radius=r, size_input=(hin, win), size_output=(wout, hout))
        assert np.array_equal(got[f], _cv2_sbs(ln[f], rn[f], m, m, interp, 0, bv)), (interp, f, r)


def test_sbs_warper_uint16_auto_radius_on_discs():
    import torch

    n, hin, win, wout, hout = 4, 200, 200, 96, 96
    t, ops = _chain()
    ln, rn = _disc16(n, hin, win, 0), _disc16(n, hin, win, 3)
    left, right = torch.from_numpy(ln).cuda(), torch.from_numpy(rn).cuda()
    wp = V.SbsWarper(t, size_input=(hin, win), size_output=(wout, hout), interpolation=2, radius="auto")
    got = wp(left, right).cpu().numpy()
    rad = wp.radius_per_frame(left, right)[0].cpu().numpy()
    for f in range(n):
        r = max(chain_np.get_radius(ln[f]), chain_np.get_radius(rn[f]))
        assert rad[f] == r
        m = chain_np.get_map(ops, radius=r, size_input=(hin, win), size_output=(wout, hout))
        assert np.array_equal(got[f], _cv2_sbs(ln[f], rn[f], m, m, 2, 0, 0)), f


@pytest.mark.parametrize("interp", [1, 2, 4])
def test_sbs_warper_uint16_unaligned_buffers(interp):
    """Sources and destination that start 2 bytes off any 16-byte boundary, with odd row pitches."""
    import torch

    n, hin, win, wout, hout = 3, 97, 131, 61, 47
    t, ops = _chain()
    rng = np.random.default_rng(13)
    big_l = torch.from_numpy(rng.integers(0, 65536, (n, hin, win + 1, 3), dtype=np.uint16).reshape(-1)).cuda()
    big_r = torch.from_numpy(rng.integers(0, 65536, (n, hin, win + 1, 3), dtype=np.uint16).reshape(-1)).cuda()
    left = big_l[1:1 + n * hin * (win + 1) * 3 - 3].as_strided((n, hin, win, 3), (hin * (win + 1) * 3, (win + 1) * 3, 3, 1))
    right = big_r[1:1 + n * hin * (win + 1) * 3 - 3].as_strided((n, hin, win, 3), (hin * (win + 1) * 3, (win + 1) * 3, 3, 1))
    out_buf = torch.empty(1 + n * hout * (2 * wout + 1) * 3, dtype=torch.uint16, device="cuda")
    out = out_buf[1:].as_strided((n, hout, 2 * wout, 3), (hout * (2 * wout + 1) * 3, (2 * wout + 1) * 3, 3, 1))
    wp = V.SbsWarper(t, size_input=(hin, win), size_output=(wout, hout), interpolation=interp, radius=70.0,
                     boarder_mode=1, boarder_value=(300, 40000, 65535))
    wp(left, right, out=out)
    got = out.cpu().numpy()
    ln, rn = left.cpu().numpy(), right.cpu().numpy()
    m = chain_np.get_map(ops, radius=70.0, size_input=(hin, win), size_output=(wout, hout))
    for f in range(n):
        assert np.array_equal(got[f], _cv2_sbs(ln[f], rn[f], m, m, interp, 1, (300, 40000, 65535))), (interp, f)


@pytest.mark.parametrize("size", [(16, 8), (17, 9), (33, 19), (208, 104)])
def test_lr_frames_uint16_odd_sizes(size):
    wout, hout = size
    n, hin, win = 3, 120, 136
    t, ops = _chain()
    ln, rn = _disc16(n, hin, win, 1), _disc16(n, hin, win, 2)
    got = V.lr_frames(t, list(ln), list(rn), size_output=(wout, hout), interpolation=1, radius=60.0,
                      boarder_value=(1000, 2000, 3000))
    m = chain_np.get_map(ops, radius=60.0, size_input=(hin, win), size_output=(wout, hout))
    for f in range(n):
        assert got[f].dtype == np.uint16
        assert np.array_equal(got[f], _cv2_sbs(ln[f], rn[f], m, m, 1, 0, (1000, 2000, 3000))), (size, f)


def test_apply_lr_frame_lr_frames_uint16_auto_radius(tmp_path):
    n, hin, win, wout, hout = 3, 160, 176, 128, 96
    t, ops = _chain()
    ln, rn = _disc16(n, hin, win, 4), _disc16(n, hin, win, 7)
    # apply: one map from images[0]'s radius ("auto"), every image; 16-bit PNG written through cv2
    outs = [tmp_path / f"o{i}.png" for i in range(n)]
    res = V.apply(t, in_paths=list(ln), out_paths=outs, size_output=(wout, hout), interpolation=4, radius="auto")
    r = max(chain_np.get_radius(im) for im in ln)
    m = chain_np.get_map(ops, radius=r, size_input=(hin, win), size_output=(wout, hout))
    for f in range(n):
        want = cv2.remap(ln[f], m[0], m[1], 4)
        assert res[f].dtype == np.uint16 and np.array_equal(res[f], want), f
        assert np.array_equal(cv2.imread(str(outs[f]), cv2.IMREAD_UNCHANGED), want), f
    # lr_frame / lr_frames: per-pair radius = max over the pair's eyes
    frames = V.lr_frames(t, list(ln), list(rn), size_output=(wout, hout), interpolation=1, radius="auto")
    for f in range(n):
        r = max(chain_np.get_radius(ln[f]), chain_np.get_radius(rn[f]))
        m = chain_np.get_map(ops, radius=r, size_input=(hin, win), size_output=(wout, hout))
        want = _cv2_sbs(ln[f], rn[f], m, m, 1, 0, 0)
        assert np.array_equal(frames[f], want), f
        one = V.lr_frame(t, ln[f], rn[f], size_output=(wout, hout), interpolation=1, radius="auto")
        assert np.array_equal(one, want), f


def test_remap_ex_border_scalar_saturates_and_null_keeps_bytes():
    """vr180_remap_ex saturates the cv::Scalar to the depth; NULL uses border_value -- for 8-bit the same bytes as
    vr180_remap."""
    import ctypes as C

    import torch

    for dtype, scalar in ((torch.uint16, (70000.0, -5.0, 300.5, 0.0)), (torch.uint8, (300.0, 7.5, 8.5, 0.0))):
        src = torch.from_numpy(np.zeros((1, 8, 8, 3), np.uint16 if dtype == torch.uint16 else np.uint8)).cuda()
        out = torch.empty((1, 4, 4, 3), dtype=dtype, device="cuda")
        e = src.element_size()
        p = N.RemapParams()
        p.n_views, p.n_frames, p.out_w, p.out_h, p.interpolation, p.border_mode = 1, 1, 4, 4, 1, 0
        p.dst, p.dst_pitch, p.dst_frame_stride = out.data_ptr(), out.stride(1) * e, out.stride(0) * e
        depth = N.DEPTH_16U if dtype == torch.uint16 else N.DEPTH_8U
        p.view[0].src = N.Image(src.data_ptr(), 8, 8, 3, depth, 8 * 3 * e, 64 * 3 * e)
        xm = torch.full((4, 4), -100.0, dtype=torch.float32, device="cuda")  # entirely outside: the border colour
        p.view[0].map.kind, p.view[0].map.xmap, p.view[0].map.ymap, p.view[0].map.map_pitch = N.MAPSRC_FLOAT2, \
            xm.data_ptr(), xm.data_ptr(), 4
        N.check(N.lib().vr180_remap_ex(C.byref(p), (C.c_double * 4)(*scalar), None))
        torch.cuda.synchronize()
        want = [65535, 0, 300] if dtype == torch.uint16 else [255, 8, 8]
        assert (out.cpu().numpy().reshape(-1, 3) == want).all(), dtype
        for i, b in enumerate((9, 10, 11, 0)):
            p.border_value[i] = b
        N.check(N.lib().vr180_remap_ex(C.byref(p), None, None))
        torch.cuda.synchronize()
        assert (out.cpu().numpy().reshape(-1, 3) == [9, 10, 11]).all(), dtype
    # views of different depths are refused
    p.view[0].src.depth = 1
    assert N.lib().vr180_remap_ex(C.byref(p), None, None) == -2


def test_apply_and_lr_frame_mixed_uint8_uint16():
    """cv.remap takes every image on its own: a call mixing uint8 and uint16 arrays of one shape returns each image in
    its own dtype (apply), and the two eyes of a pair are concatenated with NumPy's promotion (lr_frame)."""
    hin, win, wout, hout = 160, 176, 96, 64
    t, ops = _chain()
    a16 = _disc16(2, hin, win, 5)
    a8 = (a16[0] >> 8).astype(np.uint8)
    res = V.apply(t, in_paths=[a16[0], a8, a16[1]], size_output=(wout, hout), interpolation=1, radius=70.0)
    m = chain_np.get_map(ops, radius=70.0, size_input=(hin, win), size_output=(wout, hout))
    for got, src in zip(res, (a16[0], a8, a16[1])):
        want = cv2.remap(src, m[0], m[1], 1)
        assert got.dtype == src.dtype and np.array_equal(got, want)
    sbs = V.lr_frame(t, a16[0], a8, size_output=(wout, hout), interpolation=2, radius=70.0)
    want = np.concatenate([cv2.remap(a16[0], m[0], m[1], 2), cv2.remap(a8, m[0], m[1], 2)], axis=1)
    assert sbs.dtype == want.dtype == np.uint16 and np.array_equal(sbs, want)
    pairs = V.lr_frames(t, [a16[0], a16[1]], [a8, a16[0]], size_output=(wout, hout), interpolation=1, radius=70.0)
    for got, (le, ri) in zip(pairs, ((a16[0], a8), (a16[1], a16[0]))):
        want = np.concatenate([cv2.remap(le, m[0], m[1], 1), cv2.remap(ri, m[0], m[1], 1)], axis=1)
        assert np.array_equal(got, want)
