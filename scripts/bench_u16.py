"""16-bit (uint16) batched 8K warp benchmark: one JSON line.

Workload: B pairs of 2 x 4096^2 uint16 BGR fisheye frames -> B x (8192 x 4096) uint16 SBS frames, per-eye
Euclidean3DRotator + PolynomialScaler chain (bench.py's 8k_rot_poly_linear, at 16 bits), INTER_LINEAR (or
--interpolation 0: INTER_NEAREST), BORDER_CONSTANT 0.  64 pairs per launch move about 12.9 GB in and 12.9 GB out.
Aligned requests run the TMA-tiled kernel (k_warp_tiled<Linear16 / Nearest16>), or the generic per-pixel kernel
(k_remap<uint16_t, 3, INTERP>) under VR180_DISABLE_TILED=1.  Legs (same frames):
  * analytic: coordinates evaluated from the chain per output pixel;
  * lut: coordinates read from the plan's cached float32 maps;
  * lut_packed: coordinates read from the plan's tile-packed LUT;
  * unaligned: the analytic request with a source row pitch that is not a multiple of 16 bytes (generic kernel).
Each leg: warm-up launches, then `--steps` launches timed with CUDA events.  Algorithmic bytes per output pixel:
6 written + 6 x (fraction of source pixels the bilinear footprints touch).  The HBM fraction uses the same peak as
bench.py's roofline (bench.measured_peak()), and is also given against the nominal 8 TB/s.  The first and last frame of
the analytic leg are compared with cv2.remap on the NumPy restatement's maps (oracle/chain_np.py).

    [VR180_DISABLE_TILED=1] python scripts/bench_u16.py [--pairs 64] [--steps 20] [--warmup 3] [--interpolation {0,1}]
                                                        [--out FILE]
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))


def card_info() -> dict:
    try:
        r = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm",
                            "--format=csv,noheader"], capture_output=True, text=True, timeout=30)
        name, power, sm = [v.strip() for v in r.stdout.strip().split(",")]
        return {"gpu": name, "power_limit": power, "sm_max_clock": sm}
    except Exception as e:  # noqa: BLE001
        return {"gpu": None, "error": str(e)}


def synth_frames_u16(torch, n_frames: int, n: int, seed: int, pitch_px: int):
    """uint16 disc frames (random values in [4096, 65536) inside the disc, zeros outside), rows `pitch_px` pixels apart."""
    g = torch.Generator(device="cuda")
    g.manual_seed(seed)
    buf = torch.empty((n_frames, n, pitch_px, 3), dtype=torch.uint16, device="cuda")
    yy = torch.arange(n, device="cuda").view(n, 1)
    xx = torch.arange(n, device="cuda").view(1, n)
    inside = (((xx - n // 2) ** 2 + (yy - n // 2) ** 2) <= (n // 2 - 8) ** 2).to(torch.int32).view(1, n, n, 1)
    for i0 in range(0, n_frames, 4):
        part = buf[i0:i0 + 4, :, :n]
        vals = torch.randint(4096, 65536, tuple(part.shape), dtype=torch.int32, device="cuda", generator=g)
        part.copy_((vals * inside).to(torch.uint16))
    return buf[:, :, :n]


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=64)
    ap.add_argument("--n", type=int, default=4096)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--interpolation", type=int, choices=(0, 1), default=1)
    ap.add_argument("--out", type=Path, default=None)
    args = ap.parse_args()

    import cv2
    import torch

    import bench
    import vr180_convert_b200 as V
    from oracle import chain_np

    if not torch.cuda.is_available():
        raise SystemExit("bench_u16 needs a CUDA device")
    n, pairs = args.n, args.pairs
    t = bench.build_transformers(V, "rot_poly", True)
    interp = args.interpolation
    iname = "LINEAR" if interp == 1 else "NEAREST"
    kw = dict(size_input=(n, n), size_output=(n, n), interpolation=interp, radius=n / 2)
    left = synth_frames_u16(torch, pairs, n, 1, n)
    right = synth_frames_u16(torch, pairs, n, 2, n)
    out = torch.empty((pairs, n, 2 * n, 3), dtype=torch.uint16, device="cuda")

    plans = {"analytic": V.SbsWarper(t, map_source="analytic", **kw), "lut": V.SbsWarper(t, map_source="lut", **kw),
             "lut_packed": V.SbsWarper(t, map_source="lut_packed", **kw)}
    maps = plans["lut"].maps()
    peak_gbs, peak_src = bench.measured_peak()
    touched = np.mean([bench.touched_fraction(torch, maps[m], n, 2) for m in range(2)])
    out_px = pairs * n * 2 * n
    alg_bytes = out_px * 6 * (1.0 + touched)

    def timed(fn):
        for _ in range(args.warmup):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(args.steps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / args.steps
        return {"ms_per_launch": round(ms, 3), "gpix_per_s": round(out_px / ms / 1e6, 2),
                "alg_gb_per_s": round(alg_bytes / ms / 1e6, 1),
                "roofline_frac": round(alg_bytes / ms / 1e6 / peak_gbs, 3),
                "frac_of_nominal_8TBs": round(alg_bytes / ms / 1e6 / 8000.0, 3)}

    res = {"workload": "8k_rot_poly_linear_u16", "pairs_per_launch": pairs, "dtype": "uint16", "channels": 3,
           "interpolation": iname, "in_gb": round(2 * pairs * n * n * 6 / 1e9, 2), "out_gb": round(out_px * 6 / 1e9, 2),
           "touched_fraction": round(float(touched), 4), "alg_bytes_per_out_px": round(6 * (1 + touched), 3),
           "kernel": (f"k_remap<uint16_t, 3, {iname}> (generic, VR180_DISABLE_TILED=1)"
                      if os.environ.get("VR180_DISABLE_TILED") == "1"
                      else f"k_warp_tiled<{'Linear16' if interp == 1 else 'Nearest16'}> (TMA-tiled)"), "roofline_peak_gbs": peak_gbs,
           "roofline_peak_source": peak_src, "steps": args.steps, "warmup": args.warmup, **card_info(), "legs": {}}
    for name, wp in plans.items():
        res["legs"][name] = timed(lambda wp=wp: wp(left, right, out=out))
        if name == "analytic":
            first, last = out[0].cpu().numpy(), out[-1].cpu().numpy()
        else:
            res["legs"][name]["same_as_analytic"] = bool(np.array_equal(out[0].cpu().numpy(), first))
    # a source row pitch of n + 1 pixels (6 * 4097 bytes, not a multiple of 16)
    del left, right
    torch.cuda.empty_cache()
    left_u = synth_frames_u16(torch, pairs, n, 1, n + 1)
    right_u = synth_frames_u16(torch, pairs, n, 2, n + 1)
    res["legs"]["unaligned"] = timed(lambda: plans["analytic"](left_u, right_u, out=out))
    res["legs"]["unaligned"]["same_as_analytic"] = bool(np.array_equal(out[0].cpu().numpy(), first))

    # oracle: first and last frame against cv2.remap on the NumPy restatement's maps
    ok = []
    ml = chain_np.get_map(bench.oracle_ops("rot_poly", conj=True), radius=n / 2, size_input=(n, n), size_output=(n, n))
    mr = chain_np.get_map(bench.oracle_ops("rot_poly", conj=False), radius=n / 2, size_input=(n, n), size_output=(n, n))
    for f, got in ((0, first), (pairs - 1, last)):
        lf, rf = left_u[f].cpu().numpy(), right_u[f].cpu().numpy()
        want = np.concatenate([cv2.remap(np.ascontiguousarray(lf), ml[0], ml[1], interp),
                               cv2.remap(np.ascontiguousarray(rf), mr[0], mr[1], interp)], axis=1)
        ok.append(int((got != want).sum()))
    res["oracle_differing_samples_first_last"] = ok
    line = json.dumps(res)
    print(line)
    if args.out:
        args.out.parent.mkdir(parents=True, exist_ok=True)
        args.out.write_text(line + "\n")


if __name__ == "__main__":
    main()
