"""CPU tests (-m "not gpu") of the host side: transformer algebra, lowering to the chain descriptor, the C-ABI
library (loads, exports every declared symbol, host-only entry points), frame sharding."""
from __future__ import annotations

import ctypes as C
import re
from pathlib import Path

import numpy as np
import pytest

import vr180_convert_b200 as V
from oracle import chain_np, remap_np
from vr180_convert_b200 import _native as N
from vr180_convert_b200.remapper import lower_full

ROOT = Path(__file__).resolve().parent.parent
NS = {k: getattr(V, k) for k in V.__all__}
NS["np"] = np


def test_library_exports_every_declared_symbol():
    header = (ROOT / "include" / "vr180_b200.h").read_text()
    declared = set(re.findall(r"^\s*(?:int|uint64_t|const char\*)\s+(vr180_\w+)\s*\(", header, flags=re.M))
    assert declared, "no declarations parsed"
    handle = N.lib()
    for name in declared:
        assert hasattr(handle, name), f"{name} declared in include/vr180_b200.h but not exported"
        assert name in N.SYMBOLS, f"{name} has no ctypes prototype"
    assert handle.vr180_abi_version() == N.ABI_VERSION == 2
    assert handle.vr180_status_string(-5) == b"malformed chain descriptor"
    assert isinstance(handle.vr180_launch_count(), int)


def test_struct_sizes_match_header_layout():
    # natural-alignment layouts of include/vr180_b200.h
    assert C.sizeof(N.Op) == 8 + 8 * 12
    assert C.sizeof(N.Chain) == 8 + 12 * C.sizeof(N.Op)
    assert C.sizeof(N.Image) == 40
    assert C.sizeof(N.MapSrc) == 64
    assert C.sizeof(N.View) == 40 + 64 + 8
    assert C.sizeof(N.RemapParams) == 8 + 2 * 112 + 24 + 24


def test_ctypes_structs_match_the_c_header(tmp_path):
    """sizeof / offsetof of every ABI struct as gcc lays it out from include/vr180_b200.h == the ctypes mirror."""
    import subprocess

    fields = {"vr180_host_job_t": ("HostJob", ["n_frames", "src_pitch", "map_kind", "chain", "maps_cache_key", "threshold",
                                               "border_value", "dst", "radius_out", "src_frames", "dst_frames", "staging",
                                               "copy_threads"]),
              "vr180_remap_params_t": ("RemapParams", ["view", "share_map", "border_value", "dst", "dst_frame_stride"]),
              "vr180_view_t": ("View", ["map", "dst_x_offset"]),
              "vr180_mapsrc_t": ("MapSrc", ["packed_interpolation", "chain", "fixed", "map_pitch", "radius_dev", "packed"]),
              "vr180_image_t": ("Image", ["pitch", "frame_stride"]),
              "vr180_chain_t": ("Chain", ["ops"]),
              "vr180_op_t": ("Op", ["p"])}
    lines = ['#include <stdio.h>', '#include <stddef.h>', '#include "vr180_b200.h"', "int main(void) {"]
    for cname, (_, fl) in fields.items():
        lines.append(f'printf("{cname} %zu\\n", sizeof({cname}));')
        for f in fl:
            lines.append(f'printf("{cname}.{f} %zu\\n", offsetof({cname}, {f}));')
    lines += ["return 0; }"]
    src = tmp_path / "layout.c"
    src.write_text("\n".join(lines))
    exe = tmp_path / "layout"
    subprocess.run(["gcc", "-I", str(ROOT / "include"), str(src), "-o", str(exe)], check=True)
    got = dict(line.split() for line in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.splitlines())
    for cname, (pyname, fl) in fields.items():
        cls = getattr(N, pyname)
        assert int(got[cname]) == C.sizeof(cls), cname
        for f in fl:
            assert int(got[f"{cname}.{f}"]) == getattr(cls, f).offset, (cname, f)


def test_weight_tables_match_oracle():
    """The host-built cubic / lanczos4 tables the kernels use == the oracle's (== OpenCV's, pinned against cv2)."""
    for k, interp in ((4, 2), (8, 4)):
        buf = np.empty(1024 * k * k, np.int16)
        assert N.lib().vr180_debug_weight_table(k, buf.ctypes.data) == 0
        assert np.array_equal(buf.reshape(1024, k, k), remap_np.weight_table(interp))


def test_lowering_matches_golden_ops(golden_maps):
    """eval(expr) against the PRODUCT classes lowers to exactly the op list the oracle was pinned with."""
    _, meta = golden_maps
    for name, case in meta["cases"].items():
        t = eval(case["expr"], NS)  # noqa: S307 - fixture strings
        for size_out, size_in, radius in meta["shapes"]:
            ops = lower_full(t, radius=radius, size_input=tuple(size_in), size_output=tuple(size_out))
            w, h = size_out
            want = [("normalize", (w / 2, h / 2), float(min(w, h))), *[tuple(o) for o in case["ops"]],
                    ("denormalize", (radius, radius), (size_in[1] // 2, size_in[0] // 2))]
            assert len(ops) == len(want), name
            for got, exp in zip(ops, want):
                assert got[0] == exp[0], (name, got, exp)
                flat = lambda o: np.concatenate([np.atleast_1d(np.asarray(p, dtype=np.float64)).ravel()  # noqa: E731
                                                 if not isinstance(p, str) else np.array([hash(p) % 997.0]) for p in o[1:]])
                assert np.allclose(flat(got), flat(exp), rtol=0, atol=1e-15), (name, got, exp)
            N.make_chain(ops)  # encodable


def test_array_api_matches_oracle_on_points(golden_maps):
    """TransformerBase.transform on arbitrary arrays (points API) agrees with the reference restatement."""
    _, meta = golden_maps
    rng = np.random.default_rng(0)
    x, y = rng.uniform(-0.9, 0.9, (2, 50, 40))
    for name, case in meta["cases"].items():
        t = eval(case["expr"], NS)  # noqa: S307
        with np.errstate(all="ignore"):
            gx, gy = t.transform(x, y)
            wx, wy = chain_np.run_chain([tuple(o) for o in case["ops"]], x, y)
        np.testing.assert_allclose(gx, wx, rtol=1e-9, atol=1e-12, equal_nan=True, err_msg=name)
        np.testing.assert_allclose(gy, wy, rtol=1e-9, atol=1e-12, equal_nan=True, err_msg=name)


def test_equidistant_3d_round_trip():
    """Reference tests/test_remapper.py:112-115."""
    x = np.random.rand(101, 100)
    y = np.random.rand(101, 100)
    np.testing.assert_allclose(V.equidistant_from_3d(V.equidistant_to_3d(x, y)), (x, y))


def test_composition_and_errors():
    a, b, c = V.ZoomTransformer(2.0), V.EquirectangularEncoder(), V.FisheyeDecoder("equidistant")
    ab = a * b
    assert isinstance(ab, V.MultiTransformer) and ab.transformers == [a, b]
    assert (ab * c).transformers == [a, b, c] and (a * (b * c)).transformers == [a, b, c]
    assert ((a * b) * (b * c)).transformers == [a, b, b, c]
    x, y = np.array([[0.1, 0.2]]), np.array([[0.3, -0.1]])
    with pytest.raises(ValueError, match="Unknown mapping type"):
        V.FisheyeEncoder("fish").transform(x, y)
    with pytest.raises(NotImplementedError):
        V.PolynomialScaler([0, 1]).inverse_transform(x, y)
    # inverse of the inverse is the forward transform
    fx, fy = V.FisheyeEncoder("stereographic").transform(x, y)
    ix, iy = V.FisheyeDecoder("stereographic").inverse_transform(x, y)
    assert np.array_equal(fx, ix) and np.array_equal(fy, iy)
    assert repr(V.PolynomialScaler()) == "PolynomialScaler(coefs_reverse=[0, 1])"


def test_user_defined_transformer_is_opaque():
    class Mine(V.PolarRollTransformer):  # README.md:204-219
        def transform_polar(self, theta, roll, **kwargs):
            return theta**0.98 + theta**1.01, roll

    t = V.EquirectangularEncoder() * Mine() * V.FisheyeDecoder("equidistant")
    assert lower_full(t, radius=10.0, size_input=(32, 32), size_output=(16, 16)) is None

    class Tweaked(V.FisheyeEncoder):  # subclass that overrides the math must not be lowered as the parent
        def transform_polar(self, theta, roll, **kwargs):
            return theta * 2, roll

    assert Tweaked("equidistant").lower() is None
    assert V.FisheyeEncoder("equidistant").lower() == [("fisheye_enc", "equidistant")]

    class MyMulti(V.MultiTransformer):  # containers that override the math are opaque too
        def transform(self, x, y, **kwargs):
            return x * 2, y

    class MyInverse(V.InverseTransformer):
        def transform(self, x, y, **kwargs):
            return x, y * 2

    assert MyMulti(transformers=[V.ZoomTransformer(2.0)]).lower() is None
    assert MyInverse(V.FisheyeEncoder("equidistant")).lower() is None
    assert (V.EquirectangularEncoder() * MyInverse(V.FisheyeEncoder("equidistant"))).lower() is None


def test_transformers_are_sklearn_estimators_like_the_reference():
    """transformer.py:11, :14-18: BaseEstimator + TransformerMixin."""
    from sklearn.base import BaseEstimator, TransformerMixin, clone

    t = V.PolynomialScaler([0, 1, -0.1])
    assert isinstance(t, BaseEstimator) and isinstance(t, TransformerMixin)
    assert t.get_params()["coefs_reverse"] == [0, 1, -0.1]
    assert clone(V.ZoomTransformer(3.0)).scale == 3.0
    z = V.ZoomTransformer(2.0)
    z.set_params(scale=4.0)
    assert z.lower() == [("zoom", 4.0)]
    assert "transformers" in (V.ZoomTransformer(2.0) * V.EquirectangularEncoder()).get_params()


def test_quaternion_helpers_match_scipy():
    from scipy.spatial.transform import Rotation

    from vr180_convert_b200.quat import rotation_matrix

    q = V.from_rotation_vector([0.1, 0.2, 0.3])
    assert np.abs(rotation_matrix(q) - Rotation.from_rotvec([0.1, 0.2, 0.3]).as_matrix()).max() < 1e-15
    q = V.from_euler_angles(0.3, 0.5, -0.2)
    assert np.abs(rotation_matrix(q) - Rotation.from_euler("ZYZ", [0.3, 0.5, -0.2]).as_matrix()).max() < 1e-15
    assert np.abs(rotation_matrix((2.0, 0.2, 0.4, 0.6)) - rotation_matrix((1.0, 0.1, 0.2, 0.3))).max() < 1e-15
    v = np.random.default_rng(1).normal(size=(7, 3))
    assert np.allclose(V.rotate_vectors(q, v), v @ rotation_matrix(q).T)


def test_shard_range_partitions_frames():
    for n in (0, 1, 7, 1024, 1025):
        for ws in (1, 2, 4, 8):
            parts = [V.shard_range(n, ws, r) for r in range(ws)]
            flat = [i for p in parts for i in p]
            assert flat == list(range(n))
            assert max(len(p) for p in parts) - min(len(p) for p in parts) <= -(-n // ws)
    with pytest.raises(ValueError):
        V.shard_range(4, 2, 2)


def test_bind_host_near_gpu_is_a_no_op_without_topology():
    """No GPU / no sysfs entry: the NUMA binding helper reports None and leaves the affinity alone."""
    import os

    from vr180_convert_b200.shard import bind_host_near_gpu

    before = os.sched_getaffinity(0)
    bound = bind_host_near_gpu(0)
    assert bound is None or set(bound) <= before
    if bound is None:
        assert os.sched_getaffinity(0) == before


def test_argument_validation_without_gpu():
    with pytest.raises(ValueError):
        V.remap_maps(np.zeros((4, 4, 3), np.uint8), np.zeros((2, 2), np.float32), np.zeros((2, 2), np.float32),
                     interpolation=7)
    with pytest.raises(NotImplementedError):
        V.remap_maps(np.zeros((4, 4, 3), np.uint8), np.zeros((2, 2), np.float32), np.zeros((2, 2), np.float32),
                     border_mode=5)
    with pytest.raises(ValueError):
        N.make_chain([("poly", list(range(13)))])
    with pytest.raises(ValueError):
        N.make_chain([])
    # C-side validation: NULL / bad sizes are rejected before any CUDA call
    handle = N.lib()
    assert handle.vr180_build_map(None, 4, 4, None, None, 4, None) == -1
    assert handle.vr180_remap(None, None) == -1
    assert handle.vr180_ctx_run(None, None) == -1


def test_sbs_warper_auto_source_policy():
    """SbsWarper(map_source="auto") picks the coordinate source per call from the batch size alone (no GPU needed to
    check the policy): batches analytic, a plan's second and later small calls its tile-packed LUT, per-frame auto radius
    always analytic, user-defined transformers always a LUT."""
    from vr180_convert_b200.video import SbsWarper

    def plan(**kw):
        p = object.__new__(SbsWarper)
        p.map_source, p.channels, p._lowerable, p.auto_radius, p.share_map = "auto", 3, True, False, True
        p._small_calls, p._packed = 0, None
        for k, v in kw.items():
            setattr(p, k, v)
        return p

    p = plan()
    assert p._source_for(64) == "analytic" and p._small_calls == 0      # 128 rectangles per tile: a batch
    assert p._source_for(1) == "analytic"                               # first small call: not worth a LUT yet
    assert p._source_for(10) == "lut_packed"                            # 20 rectangles per tile with a shared map: small
    assert p._source_for(11) == "analytic"
    q = plan(share_map=False)
    assert q._source_for(16) == "analytic" and q._source_for(16) == "lut_packed" and q._source_for(17) == "analytic"
    assert plan(auto_radius=True)._source_for(1) == "analytic"
    r = plan(auto_radius=True)
    assert [r._source_for(1) for _ in range(3)] == ["analytic"] * 3
    assert plan(_lowerable=False)._source_for(64) == "lut_packed"
    assert plan(_lowerable=False, channels=1)._source_for(1) == "lut"
    assert plan(channels=4)._source_for(1) == "analytic"
    assert plan(map_source="lut_fixed")._source_for(1) == "lut_fixed"


def test_host_copy_moves_every_byte_at_every_alignment():
    """The copy threads' byte mover (csrc/hostcopy.cpp: streaming stores behind an aligned head, memcpy tail) against
    NumPy slices: every source / destination misalignment 0..33, sizes around the 8 KB switch and the 128-byte blocks;
    the bytes next to the destination range stay untouched."""
    import ctypes as C

    lib = N.lib()
    rng = np.random.default_rng(3)
    src = rng.integers(0, 256, 1 << 18, dtype=np.uint8)
    for n in (0, 1, 31, 127, 128, 8191, 8192, 8193, 8192 + 127, 65536 + 5, 200_003):
        for so, do in ((0, 0), (1, 0), (0, 1), (3, 29), (31, 32), (33, 17), (7, 64)):
            dst = np.full(n + 256, 0xA5, np.uint8)
            rc = lib.vr180_debug_host_copy(C.c_void_p(dst.ctypes.data + do), C.c_void_p(src.ctypes.data + so), n)
            assert rc == 0
            assert np.array_equal(dst[do:do + n], src[so:so + n]), (n, so, do)
            assert (dst[:do] == 0xA5).all() and (dst[do + n:] == 0xA5).all(), (n, so, do)


def test_bench_dump_outputs_is_a_seeded_row_sample(tmp_path, monkeypatch):
    """bench.py --dump-outputs: whole rows of one step's SBS frames as float32 with their (frame, row), within the byte
    budget, and the same rows on every run."""
    import torch

    import bench

    sbs = torch.from_numpy(np.random.default_rng(4).integers(0, 256, (5, 40, 64, 3), dtype=np.uint8))
    monkeypatch.setattr(bench, "DUMP_BYTES", 50 * 64 * 3 * 4)
    for d in ("a", "b"):
        bench.dump_outputs(torch, sbs, tmp_path / d)
    rows, index = np.load(tmp_path / "a" / "sbs_rows.npy"), np.load(tmp_path / "a" / "sbs_rows_index.npy")
    assert rows.dtype == np.float32 and index.dtype == np.float64 and rows.shape == (50, 64, 3)
    assert len({tuple(i) for i in index}) == 50
    assert np.array_equal(rows, sbs.numpy()[index[:, 0].astype(int), index[:, 1].astype(int)])
    for name in ("sbs_rows.npy", "sbs_rows_index.npy"):
        assert np.array_equal(np.load(tmp_path / "a" / name), np.load(tmp_path / "b" / name))
