"""16-bit (uint16) frames on the TMA-tiled kernel (csrc/tiled.cu, modes Linear16 / Nearest16 of csrc/tiled.cuh).

3-channel uint16 requests with INTER_NEAREST / INTER_LINEAR and 16-byte aligned buffers run k_warp_tiled; everything
else at 16 bits (CUBIC, LANCZOS4, 1 / 4 channels, an SBS right eye whose column is not a multiple of 8 pixels) keeps the
generic k_remap.  Which kernel ran is read from torch.profiler; every frame is compared with cv2.remap on the oracle's
maps (oracle/chain_np.py) bit for bit.
"""
from __future__ import annotations

import cv2
import numpy as np
import pytest

import vr180_convert_b200 as V
from oracle import chain_np

pytestmark = pytest.mark.gpu

HIN, WIN, WOUT, HOUT = 96, 128, 128, 64  # 4 x 2 tiles of 32 x 32, all full
N_FRAMES = 47
QL = (0.9995, 0.012, -0.02, 0.015)
QR = (0.9995, -0.012, 0.02, -0.015)
POLY = [0, 1, 0.04]
COLOURS = [0, 70000.4, (60000, 1000, 7, 300)]
MODE = {0: "Nearest16", 1: "Linear16"}


@pytest.fixture()
def frames_per_cta():
    lib = V._native.lib()

    def set_(n):
        lib.vr180_debug_set(0, int(n))

    yield set_
    lib.vr180_debug_set(0, 0)


def _chain(q):
    return (V.EquirectangularEncoder() * V.Euclidean3DRotator(V.quaternion(*q)) * V.PolynomialScaler(POLY)
            * V.FisheyeDecoder("equidistant"))


def _ops(q):
    return [("equirect_enc", True), ("rot3", chain_np.quat_to_matrix(*q).ravel().tolist()), ("poly", POLY),
            ("fisheye_dec", "equidistant")]


_MAPS: dict = {}


def _omap(q, radius, size_input=(HIN, WIN), size_output=(WOUT, HOUT)):
    key = (q, radius, size_input, size_output)
    if key not in _MAPS:
        _MAPS[key] = chain_np.get_map(_ops(q), radius=radius, size_input=size_input, size_output=size_output)
    return _MAPS[key]


def _frames16(n, seed, h=HIN, w=WIN):
    return np.random.default_rng(seed).integers(0, 65536, (n, h, w, 3), dtype=np.uint16)


def _sbs(lf, rf, ml, mr, interp, border=0, bv=0):
    return np.concatenate([cv2.remap(lf, ml[0], ml[1], interp, borderMode=border, borderValue=bv),
                           cv2.remap(rf, mr[0], mr[1], interp, borderMode=border, borderValue=bv)], axis=1)


def _kernels(fn):
    """(result of fn(), names of the CUDA kernels it ran)"""
    import torch
    from torch.profiler import ProfilerActivity, profile

    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    return res, {e.key for e in prof.key_averages()}


def _ran_tiled16(names, interp):
    return any("k_warp_tiled" in k and MODE[interp] in k for k in names) and not any("k_remap<" in k for k in names)


def _ran_generic(names):
    return any("k_remap<" in k for k in names) and not any("k_warp_tiled" in k for k in names)


def _check(got, ln, rn, interp, per_eye, radii):
    for f in range(len(radii)):
        r = radii[f]
        if r != r:  # NaN radius: every coordinate NaN -> border colour 0
            assert not got[f].any(), ("nan frame", f)
            continue
        ml = _omap(QL, r)
        mr = _omap(QR, r) if per_eye else ml
        want = _sbs(ln[f], rn[f], ml, mr, interp)
        assert np.array_equal(got[f], want), (interp, per_eye, f, r, int((got[f] != want).sum()))


# ---- 1. routing ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("src", ["analytic", "lut", "lut_fixed", "lut_packed"])
@pytest.mark.parametrize("interp", [0, 1])
@pytest.mark.parametrize("per_eye", [False, True])
def test_uint16_nearest_linear_run_the_tiled_kernel(interp, src, per_eye):
    import torch

    if src == "lut_fixed" and interp == 0:
        pytest.skip("the fixed-point LUT stores x * 32; INTER_NEAREST rounds x itself")
    n, radius = 5, 70.0  # > HIN / 2: tiles straddle the top / bottom source edge (TMA zero fill)
    t = (_chain(QL), _chain(QR)) if per_eye else _chain(QL)
    ln, rn = _frames16(n, 1), _frames16(n, 2)
    left, right = torch.from_numpy(ln).cuda(), torch.from_numpy(rn).cuda()
    wp = V.SbsWarper(t, size_input=(HIN, WIN), size_output=(WOUT, HOUT), interpolation=interp, radius=radius,
                     map_source=src)
    wp(left, right)  # builds the maps / LUTs outside the profiled call
    got, names = _kernels(lambda: wp(left, right).cpu().numpy())
    assert _ran_tiled16(names, interp), names
    _check(got, ln, rn, interp, per_eye, [radius] * n)


@pytest.mark.parametrize("case", ["cubic", "lanczos4", "c1", "c4", "w_not_multiple_of_8"])
def test_uint16_requests_outside_the_tiled_modes_run_the_generic_kernel(case):
    import torch

    rng = np.random.default_rng(5)
    if case in ("c1", "c4"):
        ch = 1 if case == "c1" else 4
        src = rng.integers(0, 65536, (HIN, WIN, ch), dtype=np.uint16)
        m = _omap(QL, 70.0)
        got, names = _kernels(lambda: V.remap_maps(src[..., 0] if ch == 1 else src, m[0], m[1], interpolation=1))
        want = cv2.remap(src[..., 0] if ch == 1 else src, m[0], m[1], 1)
    else:
        interp = {"cubic": 2, "lanczos4": 4}.get(case, 1)
        wout = 100 if case == "w_not_multiple_of_8" else WOUT
        ln, rn = _frames16(2, 3), _frames16(2, 4)
        wp = V.SbsWarper(_chain(QL), size_input=(HIN, WIN), size_output=(wout, HOUT), interpolation=interp, radius=70.0)
        left, right = torch.from_numpy(ln).cuda(), torch.from_numpy(rn).cuda()
        got, names = _kernels(lambda: wp(left, right).cpu().numpy())
        m = _omap(QL, 70.0, size_output=(wout, HOUT))
        want = np.stack([_sbs(ln[f], rn[f], m, m, interp) for f in range(2)])
    assert _ran_generic(names), (case, names)
    assert np.array_equal(got, want), case


# ---- 2. long frame loops ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("fpc", [24, 47])
@pytest.mark.parametrize("interp", [0, 1])
@pytest.mark.parametrize("per_eye", [False, True])
def test_uint16_long_frame_loop_fixed_radius(frames_per_cta, interp, per_eye, fpc):
    """Ring refills and phase flips over 24 / 47 one-frame items per view; a guard frame behind the batch stays
    untouched."""
    import torch

    frames_per_cta(fpc)
    radius = 70.0
    t = (_chain(QL), _chain(QR)) if per_eye else _chain(QL)
    ln, rn = _frames16(N_FRAMES, 11), _frames16(N_FRAMES, 12)
    out = torch.full((N_FRAMES + 1, HOUT, 2 * WOUT, 3), 999, dtype=torch.uint16, device="cuda")
    wp = V.SbsWarper(t, size_input=(HIN, WIN), size_output=(WOUT, HOUT), interpolation=interp, radius=radius)
    _, names = _kernels(lambda: wp(torch.from_numpy(ln).cuda(), torch.from_numpy(rn).cuda(), out=out[:N_FRAMES]))
    assert _ran_tiled16(names, interp), names
    got = out.cpu().numpy()
    assert (got[N_FRAMES] == 999).all(), "a frame was stored behind the batch"
    _check(got, ln, rn, interp, per_eye, [radius] * N_FRAMES)


def _radii(kind):
    if kind == "all_different":
        base = [40.0, 70.25, -55.5, 63.0, 48.5, 90.0, -62.0, 57.75]
        return [base[i % len(base)] + 0.5 * (i // len(base)) for i in range(N_FRAMES)]
    if kind == "runs":  # runs of equal radii with NaN (no transition found) in between
        pat = [60.5] * 5 + [float("nan")] * 3 + [60.5] * 2 + [44.0] * 7 + [float("nan")] + [71.5] * 6
        return [pat[i % len(pat)] for i in range(N_FRAMES)]
    if kind == "equal_chunk_then_mixed":  # chunk 0 takes the fixed-radius pipeline inside the DYN kernel
        return [58.5] * 24 + [58.5, 47.0] * 11 + [float("nan")]
    raise AssertionError(kind)


@pytest.mark.parametrize("kind", ["all_different", "runs", "equal_chunk_then_mixed"])
@pytest.mark.parametrize("interp", [0, 1])
@pytest.mark.parametrize("per_eye", [False, True])
def test_uint16_long_frame_loop_per_frame_radius(frames_per_cta, interp, per_eye, kind):
    import torch

    frames_per_cta(24)
    radii = _radii(kind)
    t = (_chain(QL), _chain(QR)) if per_eye else _chain(QL)
    ln, rn = _frames16(N_FRAMES, 13), _frames16(N_FRAMES, 14)
    wp = V.SbsWarper(t, size_input=(HIN, WIN), size_output=(WOUT, HOUT), interpolation=interp, radius="auto")
    rad = torch.tensor(radii, dtype=torch.float64, device="cuda")
    got, names = _kernels(lambda: wp(torch.from_numpy(ln).cuda(), torch.from_numpy(rn).cuda(), radius=rad).cpu().numpy())
    assert _ran_tiled16(names, interp), names
    _check(got, ln, rn, interp, per_eye, radii)


# ---- 3. one and two pairs per launch ------------------------------------------------------------------------------
@pytest.mark.parametrize("n", [1, 2])
@pytest.mark.parametrize("interp", [0, 1])
@pytest.mark.parametrize("per_eye", [False, True])
@pytest.mark.parametrize("src", ["analytic", "lut_packed"])
def test_uint16_one_and_two_pairs(interp, per_eye, n, src):
    import torch

    radius = 61.5
    t = (_chain(QL), _chain(QR)) if per_eye else _chain(QL)
    ln, rn = _frames16(n, 15), _frames16(n, 16)
    left, right = torch.from_numpy(ln).cuda(), torch.from_numpy(rn).cuda()
    wp = V.SbsWarper(t, size_input=(HIN, WIN), size_output=(WOUT, HOUT), interpolation=interp, radius=radius,
                     map_source=src)
    wp(left, right)
    got, names = _kernels(lambda: wp(left, right).cpu().numpy())
    assert _ran_tiled16(names, interp), names
    _check(got, ln, rn, interp, per_eye, [radius] * n)


# ---- 4. edge tiles under every border mode --------------------------------------------------------------------------
@pytest.mark.parametrize("interp", [0, 1])
@pytest.mark.parametrize("border", range(5))
def test_uint16_edge_tiles_every_border_and_colour(frames_per_cta, interp, border):
    """A radius larger than the source: many tiles straddle its edge (staged under BORDER_CONSTANT(0), gathered per
    pixel otherwise); a 120 x 72 output adds partial edge tiles; fixed and per-frame radius."""
    import torch

    frames_per_cta(6)
    n, wout, hout = 6, 120, 72
    ln, rn = _frames16(n, 17), _frames16(n, 18)
    left, right = torch.from_numpy(ln).cuda(), torch.from_numpy(rn).cuda()
    t = _chain(QL)
    radii = [75.0, 40.0, float("nan"), 75.0, 52.5, -66.0]
    for bv in COLOURS:
        def want(f, r):
            if r != r:
                xm = np.full((hout, wout), np.nan, np.float32)
                m = (xm, xm)
            else:
                m = _omap(QL, r, size_output=(wout, hout))
            return _sbs(ln[f], rn[f], m, m, interp, border, bv)

        wp = V.SbsWarper(t, size_input=(HIN, WIN), size_output=(wout, hout), interpolation=interp, radius=75.0,
                         boarder_mode=border, boarder_value=bv)
        got, names = _kernels(lambda: wp(left, right).cpu().numpy())
        assert _ran_tiled16(names, interp), names
        for f in range(n):
            assert np.array_equal(got[f], want(f, 75.0)), (interp, border, bv, f)
        wp = V.SbsWarper(t, size_input=(HIN, WIN), size_output=(wout, hout), interpolation=interp, radius="auto",
                         boarder_mode=border, boarder_value=bv)
        got = wp(left, right, radius=torch.tensor(radii, dtype=torch.float64, device="cuda")).cpu().numpy()
        for f in range(n):
            assert np.array_equal(got[f], want(f, radii[f])), (interp, border, bv, "dyn", f, radii[f])


# ---- 5. values and weights ------------------------------------------------------------------------------------------
def _fraction_maps(w=256, h=128):
    """x = 6 + i + (i % 32) / 32, y = 5 + 0.75 j + (j % 32) / 32: inside every 32 x 32 tile, pixel (i, j) has the
    fractions (ax, ay) = (i % 32, j % 32) up to the 0.75 j grid, i.e. every (ax, ay) pair occurs in staged tiles."""
    i = np.arange(w, dtype=np.float64)
    j = np.arange(h, dtype=np.float64)
    xm = np.broadcast_to((6 + i + (i % 32) / 32)[None, :], (h, w)).astype(np.float32)
    ym = np.broadcast_to((5 + np.floor(0.75 * j) + (j % 32) / 32)[:, None], (h, w)).astype(np.float32)
    return np.ascontiguousarray(xm), np.ascontiguousarray(ym)


@pytest.mark.parametrize("values", ["full_range", "all_65535", "ties"])
@pytest.mark.parametrize("interp", [0, 1])
def test_uint16_values_and_every_weight_pair(interp, values):
    rng = np.random.default_rng(19)
    xm, ym = _fraction_maps()
    ax, ay = np.rint(xm * 32).astype(np.int64) & 31, np.rint(ym * 32).astype(np.int64) & 31
    assert len(set(zip(ax.ravel(), ay.ravel()))) == 1024
    shape = (2, 140, 300, 3)
    if values == "full_range":
        ln = rng.integers(0, 65536, shape, dtype=np.uint16)
    elif values == "all_65535":
        ln = np.full(shape, 65535, np.uint16)
    else:  # neighbouring values 1 apart with half-pixel weights: sums that end in .5 (round half to even)
        ln = (rng.integers(0, 4, shape) + rng.choice([0, 32767, 65531], shape)).astype(np.uint16)
    # SbsWarper does not take arbitrary maps: run vr180_remap through remap_maps (host pipeline) frame by frame
    for f in range(shape[0]):
        got, names = _kernels(lambda: V.remap_maps(ln[f], xm, ym, interpolation=interp))
        assert any("k_warp_tiled" in k and MODE[interp] in k for k in names), names
        assert np.array_equal(got, cv2.remap(ln[f], xm, ym, interp)), (values, f)


@pytest.mark.parametrize("interp", [0, 1])
@pytest.mark.parametrize("border", [0, 1])
def test_uint16_nan_inf_and_huge_coordinates(interp, border):
    rng = np.random.default_rng(23)
    src = rng.integers(0, 65536, (140, 300, 3), dtype=np.uint16)
    xm, ym = _fraction_maps()
    xm, ym = xm.copy(), ym.copy()
    bad = [np.nan, np.inf, -np.inf, 1e9, -1e9]
    for k, v in enumerate(bad):  # one bad coordinate in some tiles, a whole tile of them in another
        xm[3 + k, 40 + 7 * k] = v
        ym[40 + k, 100 + 5 * k] = v
    xm[96:128, 224:256] = np.nan
    for bv in COLOURS:
        got = V.remap_maps(src, xm, ym, interpolation=interp, border_mode=border, border_value=bv)
        assert np.array_equal(got, cv2.remap(src, xm, ym, interp, borderMode=border, borderValue=bv)), (border, bv)


# ---- 6. descriptor cache: one allocation as uint8 and as uint16 ------------------------------------------------------
@pytest.mark.parametrize("interp", [0, 1])
def test_uint8_and_uint16_views_of_one_allocation(interp):
    """Same pointers, rows, cols and byte pitches at both depths: the TMA descriptors of one must not serve the other.
    One pair per launch, analytic coordinates: both depths run k_warp_tiled with one-frame boxes, so without the depth
    in the descriptor cache's key the second request would find the first one's descriptors."""
    import torch

    n, radius = 1, 61.5
    pitch = WIN * 6  # bytes per source row, both views
    buf_l = torch.from_numpy(_frames16(n, 21)).cuda()
    buf_r = torch.from_numpy(_frames16(n, 22)).cuda()
    out16 = torch.empty((n, HOUT, 2 * WOUT, 3), dtype=torch.uint16, device="cuda")

    def u8(t16, rows, cols, row_bytes):  # uint8 (n, rows, cols, 3) view of the same bytes, rows `row_bytes` apart
        return t16.view(torch.uint8).as_strided((n, rows, cols, 3), (rows * row_bytes, row_bytes, 3, 1))

    l8, r8 = u8(buf_l, HIN, WIN, pitch), u8(buf_r, HIN, WIN, pitch)
    out8 = u8(out16, HOUT, 2 * WOUT, 2 * WOUT * 6)
    wp = V.SbsWarper(_chain(QL), size_input=(HIN, WIN), size_output=(WOUT, HOUT), interpolation=interp, radius=radius,
                     map_source="analytic")
    m = _omap(QL, radius)
    for dtype in ("u8", "u16", "u8", "u16"):
        if dtype == "u8":
            _, names = _kernels(lambda: wp(l8, r8, out=out8))
            got, ln, rn = out8.cpu().numpy(), l8.cpu().numpy(), r8.cpu().numpy()
            assert any("k_warp_tiled" in k and "Linear16" not in k and "Nearest16" not in k for k in names), names
        else:
            _, names = _kernels(lambda: wp(buf_l, buf_r, out=out16))
            got, ln, rn = out16.cpu().numpy(), buf_l.cpu().numpy(), buf_r.cpu().numpy()
            assert _ran_tiled16(names, interp), names
        for f in range(n):
            assert np.array_equal(got[f], _sbs(ln[f], rn[f], m, m, interp)), (dtype, f)


# ---- 7. production size ---------------------------------------------------------------------------------------------
def test_uint16_8k_pair_per_eye_maps():
    import torch

    n = 4096
    ql, qr = (0.9999, 0.004, -0.008, 0.006), (0.9999, -0.004, 0.008, -0.006)
    t = (_chain(ql), _chain(qr))
    ln, rn = _frames16(1, 31, n, n), _frames16(1, 32, n, n)
    wp = V.SbsWarper(t, size_input=(n, n), size_output=(n, n), interpolation=1, radius=n / 2)
    left, right = torch.from_numpy(ln).cuda(), torch.from_numpy(rn).cuda()
    got, names = _kernels(lambda: wp(left, right).cpu().numpy())
    assert _ran_tiled16(names, 1), names
    ml = chain_np.get_map(_ops(ql), radius=n / 2, size_input=(n, n), size_output=(n, n))
    mr = chain_np.get_map(_ops(qr), radius=n / 2, size_input=(n, n), size_output=(n, n))
    want = _sbs(ln[0], rn[0], ml, mr, 1)
    assert int((got[0] != want).sum()) == 0


# ---- 8. host pipeline ---------------------------------------------------------------------------------------------
@pytest.mark.parametrize("interp", [0, 1])
def test_uint16_lr_frames_right_eye_at_an_aligned_column(interp):
    """W % 8 != 0: the host pipeline stages the right eye at a 16-byte aligned column, so the pair still takes the
    tiled kernel."""
    n, wout, hout, radius = 3, 100, 70, 60.0
    ln, rn = _frames16(n, 25), _frames16(n, 26)
    got, names = _kernels(lambda: V.lr_frames(_chain(QL), list(ln), list(rn), size_output=(wout, hout),
                                              interpolation=interp, radius=radius))
    assert _ran_tiled16(names, interp), names
    m = _omap(QL, radius, size_output=(wout, hout))
    for f in range(n):
        assert got[f].dtype == np.uint16 and np.array_equal(got[f], _sbs(ln[f], rn[f], m, m, interp)), f
