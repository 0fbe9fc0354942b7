"""Generate tests/golden/*.npz by running the UNMODIFIED reference (a checkout of the original vr180-convert
project).  Run from the repo root:   VR180_CONVERT_REF=/path/to/vr180-convert python tests/golden/make_golden.py

The reference is pure Python; its `quaternion` (numpy-quaternion) and `strenum` dependencies are served by the
test-only stand-ins in tests/refshim/, which are put on sys.path first (SURVEY.md Appendix D).  The tests never need
the reference itself, which is why the vectors are committed.

Every case stores (a) the Python expression that builds the transformer (evaluated both against the
reference and, in the tests, against the product package), (b) the op-tuple lowering fed to the oracle, and
(c) the reference's float32 maps / uint8 pixels.
"""
from __future__ import annotations

import json
import os
import sys
import tempfile
from pathlib import Path

import numpy as np

HERE = Path(__file__).resolve().parent
REF = Path(os.environ["VR180_CONVERT_REF"])  # checkout of the original vr180-convert project
sys.path.insert(0, str(HERE.parent / "refshim"))
sys.path.insert(0, str(REF / "src"))

import cv2  # noqa: E402
import quaternion as Q  # noqa: E402  (the shim)
import vr180_convert as ref  # noqa: E402
from vr180_convert import remapper as ref_remapper  # noqa: E402
from vr180_convert import transformer as ref_t  # noqa: E402
from vr180_convert.testing import generate_test_image  # noqa: E402

# ---- rotations used by the cases (w, x, y, z) ---------------------------------------------------------
Q_SMALL = (0.9999093510664558, 0.00500054686470522, 0.01000109372941044, -0.00750082029705783)
Q_EULER = tuple(Q.from_euler_angles(0.0, np.pi / 4, 0.0).components)  # reference tests/test_remapper.py:80
Q_NONUNIT = (1.3, 0.02, -0.05, 0.04)  # cli.py:308-311 builds non-unit half rotations


def rmat(q):
    return Q.as_rotation_matrix(Q.quaternion(*q)).reshape(-1).tolist()


# name -> (python expression, op tuples)
CASES = {
    "base": ('EquirectangularEncoder() * FisheyeDecoder("equidistant")',
             [("equirect_enc", True), ("fisheye_dec", "equidistant")]),
    "poly_default": ('EquirectangularEncoder() * PolynomialScaler() * FisheyeDecoder("equidistant")',
                     [("equirect_enc", True), ("poly", [0, 1]), ("fisheye_dec", "equidistant")]),
    "rot_poly": (f'EquirectangularEncoder() * Euclidean3DRotator(quaternion{Q_SMALL}) * '
                 'PolynomialScaler([0, 1, -0.02, 0.003]) * FisheyeDecoder("equidistant")',
                 [("equirect_enc", True), ("rot3", rmat(Q_SMALL)), ("poly", [0, 1, -0.02, 0.003]),
                  ("fisheye_dec", "equidistant")]),
    "rot_euler_lr": (f'EquirectangularEncoder() * Euclidean3DRotator(quaternion{Q_EULER}) * '
                     'FisheyeDecoder("equidistant")',
                     [("equirect_enc", True), ("rot3", rmat(Q_EULER)), ("fisheye_dec", "equidistant")]),
    "rot_nonunit": (f'EquirectangularEncoder() * Euclidean3DRotator(quaternion{Q_NONUNIT}) * '
                    'FisheyeDecoder("equidistant")',
                    [("equirect_enc", True), ("rot3", rmat(Q_NONUNIT)), ("fisheye_dec", "equidistant")]),
    "fe_rot": (f'FisheyeEncoder("equidistant") * Euclidean3DRotator(quaternion{Q_EULER}) * '
               'FisheyeDecoder("equidistant")',
               [("fisheye_enc", "equidistant"), ("rot3", rmat(Q_EULER)), ("fisheye_dec", "equidistant")]),
    "fe_poly": ('FisheyeEncoder("equidistant") * PolynomialScaler([0, 1, -0.1]) * FisheyeDecoder("equidistant")',
                [("fisheye_enc", "equidistant"), ("poly", [0, 1, -0.1]), ("fisheye_dec", "equidistant")]),
    "lat_x": ('EquirectangularEncoder(is_latitude_y=False) * FisheyeDecoder("equisolid")',
              [("equirect_enc", False), ("fisheye_dec", "equisolid")]),
    "zoom": ('EquirectangularEncoder() * ZoomTransformer(1.25) * FisheyeDecoder("stereographic")',
             [("equirect_enc", True), ("zoom", 1.25), ("fisheye_dec", "stereographic")]),
    "rectilinear": ('EquirectangularEncoder() * ZoomTransformer(3.0) * RectilinearDecoder(18.0, 36.0)',
                    [("equirect_enc", True), ("zoom", 3.0), ("rectilinear_dec", 2 * 18.0 / 36.0)]),
    "equirect_dec": ('FisheyeEncoder("equidistant") * EquirectangularDecoder()',
                     [("fisheye_enc", "equidistant"), ("equirect_dec", True)]),
    "neg_poly": ('EquirectangularEncoder() * PolynomialScaler([0.2, -1.0, 0.3]) * ZoomTransformer(-0.8) * '
                 'FisheyeDecoder("equidistant")',
                 [("equirect_enc", True), ("poly", [0.2, -1.0, 0.3]), ("zoom", -0.8), ("fisheye_dec", "equidistant")]),
}
for m in ("rectilinear", "stereographic", "equidistant", "equisolid", "orthographic"):  # test_remapper.py:42-74
    CASES[f"fe_{m}"] = (f'FisheyeEncoder("{m}") * FisheyeDecoder("equidistant")',
                        [("fisheye_enc", m), ("fisheye_dec", "equidistant")])

NS = {k: getattr(ref_t, k) for k in dir(ref_t) if not k.startswith("_")}
NS.update(quaternion=Q.quaternion, np=np)

MAP_SHAPES = [  # (size_output (W,H), size_input (rows, cols), radius)
    ((48, 40), (37, 53), 17.5),
    ((64, 64), (64, 64), 32.0),
    ((33, 57), (80, 60), -29.5),
]


def make_maps():
    out = {}
    meta = {}
    for name, (expr, ops) in CASES.items():
        t = eval(expr, NS)  # noqa: S307 - fixed strings above
        for si, (size_out, size_in, radius) in enumerate(MAP_SHAPES):
            with np.errstate(all="ignore"):
                xm, ym = ref.get_map(t, radius=radius, size_input=size_in, size_output=size_out)
            out[f"{name}/{si}/x"] = xm
            out[f"{name}/{si}/y"] = ym
        meta[name] = {"expr": expr, "ops": ops}
    out["meta"] = np.array(json.dumps({"cases": meta, "shapes": MAP_SHAPES}))
    np.savez_compressed(HERE / "maps.npz", **out)
    print("maps.npz", len(CASES), "cases")


def make_big_map_hashes():
    """Sparse samples of full-size reference maps (cfg2 / cfg3 shapes) -- the whole map is too big to commit."""
    out = {}
    rng = np.random.default_rng(1234)
    for name, n in (("base", 2048), ("rot_poly", 4096)):
        t = eval(CASES[name][0], NS)  # noqa: S307
        xm, ym = ref.get_map(t, radius=n / 2, size_input=(n, n), size_output=(n, n))
        idx = rng.integers(0, n, size=(4096, 2))
        idx[:8] = [[0, 0], [0, n - 1], [n - 1, 0], [n - 1, n - 1], [n // 2, n // 2], [n // 2, 0], [0, n // 2], [1, 1]]
        out[f"{name}/{n}/idx"] = idx.astype(np.int32)
        out[f"{name}/{n}/x"] = xm[idx[:, 0], idx[:, 1]]
        out[f"{name}/{n}/y"] = ym[idx[:, 0], idx[:, 1]]
        # one full row and one full column
        out[f"{name}/{n}/row"] = np.stack([xm[n // 3], ym[n // 3]])
        out[f"{name}/{n}/col"] = np.stack([xm[:, n // 5], ym[:, n // 5]])
    np.savez_compressed(HERE / "maps_fullsize_samples.npz", **out)
    print("maps_fullsize_samples.npz")


def make_remap():
    rng = np.random.default_rng(7)
    src = rng.integers(0, 256, (37, 53, 3), dtype=np.uint8)
    h, w = 40, 56
    xm = (rng.random((h, w)) * 70 - 8).astype(np.float32)
    ym = (rng.random((h, w)) * 50 - 6).astype(np.float32)
    special = np.array([np.nan, np.inf, -np.inf, 1e9, -1e9, 7e7, -7e7, 6e7], np.float32)
    xm[0, :8] = special
    ym[1, :8] = special
    xm[2] = np.round(xm[2])
    ym[3] = np.round(ym[3])
    xm[4] = np.floor(xm[4]) + 0.5 + 1 / 64  # exact ties of x*32
    ym[5] = np.floor(ym[5]) + 1 / 64
    xm[6] = np.floor(xm[6]) + 3 / 64
    out = {"src": src, "xmap": xm, "ymap": ym}
    for interp in (0, 1, 2, 4):
        for bm in (0, 1, 2, 3, 4):
            for bi, bv in enumerate((0, 7, (3, 200, 90))):
                out[f"out/{interp}/{bm}/{bi}"] = cv2.remap(src, xm, ym, interpolation=interp, borderMode=bm,
                                                          borderValue=bv)
    np.savez_compressed(HERE / "remap.npz", **out)
    print("remap.npz")


def make_radius():
    cases = {}
    for h, w, r in ((1000, 1000, 400), (1000, 1500, 450), (1500, 1000, 450), (64, 64, 20), (31, 64, 9)):
        yy, xx = np.mgrid[:h, :w]
        img = np.where(((xx - w // 2) ** 2 + (yy - h // 2) ** 2 <= r * r)[..., None], 200, 0).astype(np.uint8)
        img = np.repeat(img, 3, axis=2) if img.shape[2] == 1 else img
        cases[f"{h}x{w}x{r}"] = float(ref_t.get_radius(img))
    card = generate_test_image(256)
    halves = [card[:, :128], card[:, 128:]]
    cases["card256_left"] = float(ref_t.get_radius(np.ascontiguousarray(halves[0])))
    cases["card256_right"] = float(ref_t.get_radius(np.ascontiguousarray(halves[1])))
    try:
        ref_t.get_radius(card)
        cases["card256_full"] = "no error"
    except IndexError:
        cases["card256_full"] = "IndexError"
    for nm, img in (("black64", np.zeros((64, 64, 3), np.uint8)), ("white64", np.full((64, 64, 3), 255, np.uint8))):
        try:
            cases[nm] = float(ref_t.get_radius(img))
        except IndexError:
            cases[nm] = "IndexError"
    (HERE / "radius.json").write_text(json.dumps(cases, indent=1))
    print("radius.json", cases)


def make_apply():
    """End-to-end apply / apply_lr through the reference on the 256 px test card (ndarray inputs, PNG out)."""
    card = generate_test_image(256)
    left, right = card[:, :128], card[:, 128:]
    out = {"card": card}
    with tempfile.TemporaryDirectory() as d:
        for name, interp, radius in (("base", cv2.INTER_LINEAR, "max"), ("rot_poly", cv2.INTER_CUBIC, 100.0),
                                     ("poly_default", cv2.INTER_LANCZOS4, "auto"), ("base", cv2.INTER_NEAREST, 90.5)):
            t = eval(CASES[name][0], NS)  # noqa: S307
            p = Path(d) / "o.png"
            ref.apply_lr(t, left_path=left, right_path=right, out_path=p, size_output=(96, 80),
                         interpolation=interp, radius=radius)
            out[f"lr/{name}/{interp}/{radius}"] = cv2.imread(str(p))
        # per-eye tuple (cli.py:312-319 shape): own radius + own map per eye
        tl = eval(CASES["rot_poly"][0], NS)  # noqa: S307
        tr = eval(CASES["rot_nonunit"][0], NS)  # noqa: S307
        p = Path(d) / "o2.png"
        ref.apply_lr((tl, tr), left_path=left, right_path=right, out_path=p, size_output=(96, 80),
                     interpolation=cv2.INTER_LINEAR, radius="auto")
        out["lr_tuple/rot_poly+rot_nonunit/1/auto"] = cv2.imread(str(p))
        imgs = ref.apply(eval(CASES["fe_poly"][0], NS), in_paths=[card, card[::-1].copy()],  # noqa: S307
                         size_output=(72, 72), interpolation=cv2.INTER_LINEAR, radius="max", boarder_value=9)
        out["apply/fe_poly/0"], out["apply/fe_poly/1"] = imgs
    np.savez_compressed(HERE / "apply.npz", **out)
    print("apply.npz")


def make_merge_and_match():
    """apply_lr(merge=True) (remapper.py:485-516: float64 anaglyph + putText labels + imwrite's uint8 conversion) and
    match_lr (remapper.py:251-321) through the unmodified reference."""
    card = generate_test_image(256)
    left, right = card[:, :128], card[:, 128:]
    out = {}
    with tempfile.TemporaryDirectory() as d:
        for name, size in (("small", (96, 80)), ("labels", (512, 1024))):  # 1024 rows: font scale 1, labels drawn
            p = Path(d) / "m.png"
            ref.apply_lr(eval(CASES["rot_poly"][0], NS), left_path=left, right_path=right, out_path=p,  # noqa: S307
                         size_output=size, interpolation=cv2.INTER_LINEAR, radius="max", merge=True)
            out[f"merge/{name}"] = cv2.imread(str(p))
        tl = eval(CASES["rot_poly"][0], NS)  # noqa: S307
        tr = eval(CASES["rot_nonunit"][0], NS)  # noqa: S307
        p = Path(d) / "m2.png"
        ref.apply_lr((tl, tr), left_path=left, right_path=right, out_path=p, size_output=(96, 80),
                     interpolation=cv2.INTER_CUBIC, radius="auto", merge=True)
        out["merge/tuple_auto"] = cv2.imread(str(p))
        # match_lr reads files
        pl, pr = Path(d) / "l.png", Path(d) / "r.png"
        cv2.imwrite(str(pl), np.ascontiguousarray(left))
        cv2.imwrite(str(pr), np.ascontiguousarray(right))
        rng = np.random.default_rng(5)
        pts_l = rng.uniform(20, 108, (24, 2))
        pts_r = pts_l + rng.normal(0, 1.5, (24, 2))
        out["match/pts_l"], out["match/pts_r"] = pts_l, pts_r
        dec = ref_t.FisheyeDecoder("equidistant")
        for rname, radius in (("max", "max"), ("auto", "auto"), ("60.5", 60.5)):
            vl, vr = ref_remapper.match_lr(dec, pts_l, pts_r, [pl, pr], radius=radius)
            out[f"match/single/{rname}/vl"], out[f"match/single/{rname}/vr"] = vl, vr
        dec2 = (ref_t.FisheyeDecoder("stereographic"), ref_t.ZoomTransformer(1.1) * ref_t.FisheyeDecoder("equisolid"))
        vl, vr = ref_remapper.match_lr(dec2, pts_l, pts_r, [pl, pr], radius=70.0)
        out["match/tuple/70.0/vl"], out["match/tuple/70.0/vr"] = vl, vr
    np.savez_compressed(HERE / "merge_match.npz", **out)
    print("merge_match.npz", {k: v.shape for k, v in out.items()})


def make_cfg1():
    """BASELINE.json configs[0] (SURVEY.md §8d cfg1): `v1c lr test.jpg test.jpg --transformer 'EquirectangularEncoder()
    * PolynomialScaler() * FisheyeDecoder("equidistant")' --interpolation INTER_LINEAR` with the CLI's default size
    4096x4096 per eye (cli.py:117-380 -> remapper.py:406-520), run through the unmodified reference's apply_lr.
    The 2048 x 2048 README image is split into two PORTRAIT halves (2048 x 1024: get_radius scans the centre COLUMN)
    and upsampled to 4096^2 per eye.  Stored: the input JPEG (reference docs/_static/test.jpg, a data file), the
    sha256 of its decoded pixels, the radius the reference logs, the sha256 of the (4096, 8192, 3) output and 200 000
    sparse output samples + 8 full rows (the whole frame is 100 MB)."""
    import hashlib
    import shutil

    src = REF / "docs" / "_static" / "test.jpg"
    shutil.copyfile(src, HERE / "cfg1_test.jpg")
    (HERE / "cfg1_test.jpg").chmod(0o644)
    img = cv2.imread(str(src))
    t = eval(CASES["poly_default"][0], NS)  # noqa: S307
    halves = [img[:, : img.shape[1] // 2], img[:, img.shape[1] // 2:]]
    radius = ref_remapper.get_radius_smart("auto", halves)
    with tempfile.TemporaryDirectory() as d:
        p = Path(d) / "o.png"
        ref.apply_lr(t, left_path=src, right_path=src, out_path=p, size_output=(4096, 4096),
                     interpolation=cv2.INTER_LINEAR, radius="auto")
        out = cv2.imread(str(p))
    assert out.shape == (4096, 8192, 3)
    rng = np.random.default_rng(2024)
    idx = np.stack([rng.integers(0, 4096, 200_000), rng.integers(0, 8192, 200_000)], axis=1).astype(np.int16)  # keeps the file < 1 MB
    rows = np.array([0, 1, 1023, 2047, 2048, 3000, 4094, 4095], np.int32)
    np.savez_compressed(HERE / "cfg1.npz", idx=idx, px=out[idx[:, 0], idx[:, 1]], rows=rows, row_px=out[rows],
                        meta=np.array(json.dumps({
                            "radius": float(radius), "expr": CASES["poly_default"][0], "size_output": [4096, 4096],
                            "interpolation": int(cv2.INTER_LINEAR),
                            "input_sha256": hashlib.sha256(np.ascontiguousarray(img).tobytes()).hexdigest(),
                            "output_sha256": hashlib.sha256(np.ascontiguousarray(out).tobytes()).hexdigest(),
                            "cv2": cv2.__version__, "numpy": np.__version__})))
    print("cfg1.npz radius", radius, "sha", hashlib.sha256(np.ascontiguousarray(out).tobytes()).hexdigest())


if __name__ == "__main__":
    if len(sys.argv) > 1 and sys.argv[1] == "cfg1":
        make_cfg1()
        raise SystemExit(0)
    if len(sys.argv) > 1 and sys.argv[1] == "merge":
        make_merge_and_match()
        raise SystemExit(0)
    make_maps()
    make_big_map_hashes()
    make_remap()
    make_radius()
    make_apply()
    make_merge_and_match()
    make_cfg1()
