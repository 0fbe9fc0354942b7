#!/usr/bin/env python
"""bench.py -- SBS equirect output Mpix/s of the reprojection hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--workload NAME] [--impl reference] [--dump-outputs DIR]

A "step" is one pass of the hot path over one batch of synthetic stereo pairs.  Default workload (the
configuration BASELINE.json's target is quoted on -- "bit-exact INTER_LINEAR SBS equirectangular output ... on
batched 8K stereo frames"): B pairs of 2 x 4096^2 fisheye frames -> B x (8192 x 4096) SBS frames, per-eye
Euclidean3DRotator + PolynomialScaler chain (configs[2]), fused analytic warp, INTER_LINEAR.

  value      whole-job Mpix/s with the frames resident in HBM (CUDA events on the launch stream, max over ranks)
  e2e        the same metric through the C-ABI host call the NumPy API uses (vr180_ctx_run) with pinned HOST
             buffers: H2D of every source frame and D2H of every SBS frame inside the timed region
  roofline   algorithmic bytes of one launch / its measured duration vs the measured HBM copy bandwidth
  cpu_baseline / --impl reference
             the reference's CPU path (NumPy chain restated in oracle/chain_np.py + the real cv2.remap +
             np.concatenate) on this box's host cores, on a bounded sample of the same workload

N > 1: one process per GPU (torchrun or self-spawned), frames sharded statically, no data-path collective
(weak scaling: every rank warps its own B pairs); torch.distributed is used only for the barrier and the
max-over-ranks of the device time.

--dump-outputs DIR: after the timed steps, rank 0 writes the SBS frames its last timed step produced, as a seeded
sample of whole output rows (DIR/sbs_rows.npy, float32 (rows, 2n, 3)) and the (frame, row) of each sampled row
(DIR/sbs_rows_index.npy, float64).  The input frames are generated from fixed seeds, so two builds run with the same
arguments can be compared array for array.
"""
from __future__ import annotations

import argparse
import json
import os
import socket
import statistics
import subprocess
import sys
import time
from pathlib import Path

import numpy as np

ROOT = Path(__file__).resolve().parent
if str(ROOT) not in sys.path:
    sys.path.insert(0, str(ROOT))

Q_HALF = (0.9999093510664558, 0.00500054686470522, 0.01000109372941044, -0.00750082029705783)
POLY = [0, 1, -0.02, 0.003]

WORKLOADS = {
    # name: (per-eye input n, output n, interpolation, per_eye_tuple, map_source, radius, default pairs per step)
    "8k_rot_poly_linear": dict(n=4096, interp=1, tuple_=True, chain="rot_poly", src="analytic", radius="fixed", pairs=64,
                               desc="batched 8K stereo pairs (2x4096^2 -> 8192x4096), per-eye Euclidean3DRotator+"
                                    "PolynomialScaler, fused analytic warp, INTER_LINEAR [BASELINE configs[2], batched]"),
    "8k_rot_poly_lut": dict(n=4096, interp=1, tuple_=True, chain="rot_poly", src="lut_packed", radius="fixed", pairs=64,
                            desc="the headline workload with the coordinates cached in two tile-packed LUTs (built once, "
                                 "outside the timed region) instead of being re-evaluated by every launch: the video-loop path"),
    "4k_pair_linear": dict(n=2048, interp=1, tuple_=False, chain="base", src="analytic", radius="fixed", pairs=1,
                           desc="single 4K pair (2x2048^2 -> 4096x2048), base chain, fused analytic, INTER_LINEAR "
                                "[BASELINE configs[1]]; a ring of pairs larger than L2 is cycled"),
    "5k7_lut_linear": dict(n=2880, interp=1, tuple_=False, chain="base", src="lut_packed", radius="fixed", pairs=64,
                           desc="batched 5.7K pairs (2x2880^2 -> 5760x2880), cached tile-packed LUT (4 B/px), INTER_LINEAR "
                                "[BASELINE configs[3]]"),
    "5k7_lut_linear_512": dict(n=2880, interp=1, tuple_=False, chain="base", src="lut_packed", radius="fixed", pairs=512,
                               desc="512 resident 5.7K pairs per GPU (25.5 GB in + 25.5 GB out), cached tile-packed LUT, "
                                    "INTER_LINEAR, one launch [BASELINE configs[3]: 1024 pairs over >= 2 GPUs]"),
    "5k7_lutfixed_linear": dict(n=2880, interp=1, tuple_=False, chain="base", src="lut_fixed", radius="fixed", pairs=64,
                                desc="as 5k7_lut_linear with the 8 B/px fixed-point LUT (int32 sx, sy)"),
    "4k_pair_lut_linear": dict(n=2048, interp=1, tuple_=False, chain="base", src="lut_packed", radius="fixed", pairs=1,
                               desc="single 4K pair, cached tile-packed LUT instead of the FP64 chain: the per-frame path of a "
                                    "video loop, what SbsWarper's default map_source='auto' serves from a plan's second "
                                    "one-pair call on (tile-streaming kernel) [BASELINE configs[1]]"),
    "8k_pair_lut_linear": dict(n=4096, interp=1, tuple_=True, chain="rot_poly", src="lut_packed", radius="fixed", pairs=1,
                               desc="ONE 8K pair per launch (2x4096^2 -> 8192x4096), per-eye rotation + PolynomialScaler, cached "
                                    "tile-packed LUTs: the tile-streaming kernel [BASELINE configs[2], unbatched video loop]"),
    "8k_pair_linear": dict(n=4096, interp=1, tuple_=True, chain="rot_poly", src="analytic", radius="fixed", pairs=1,
                           desc="ONE 8K pair per launch, per-eye rotation + PolynomialScaler, fused analytic (no LUT): one "
                                "apply_lr call of the reference [BASELINE configs[2], unbatched]"),
    "8k_nearest_fixed": dict(n=4096, interp=0, tuple_=False, chain="base", src="analytic", radius="fixed", pairs=16,
                             desc="batched 8K pairs, base chain, fused analytic, INTER_NEAREST, fixed radius (the pipeline "
                                  "without the interpolation arithmetic)"),
    "8k_cubic_fixed": dict(n=4096, interp=2, tuple_=False, chain="base", src="analytic", radius="fixed", pairs=16,
                           desc="batched 8K pairs, base chain, fused analytic, INTER_CUBIC, fixed radius"),
    "8k_lanczos4_fixed": dict(n=4096, interp=4, tuple_=False, chain="base", src="analytic", radius="fixed", pairs=16,
                              desc="batched 8K pairs, base chain, fused analytic, INTER_LANCZOS4 (the default interpolation "
                                   "of the reference's apply(), remapper.py:330), fixed radius"),
    "8k_cubic_auto": dict(n=4096, interp=2, tuple_=False, chain="base", src="analytic", radius="auto", pairs=16,
                          desc="batched 8K pairs, base chain, fused analytic + get_radius per frame consumed on device, "
                               "INTER_CUBIC [BASELINE configs[4]]"),
    "8k_cubic_auto_varying": dict(n=4096, interp=2, tuple_=False, chain="base", src="analytic", radius="auto", pairs=16,
                                  vary=True,
                                  desc="as 8k_cubic_auto, but consecutive frames have different disc radii, so the "
                                       "per-pixel constants are rebuilt for every frame"),
}


# ---------------------------------------------------------------------------------------------------------
# helpers
# ---------------------------------------------------------------------------------------------------------
def measured_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        try:
            return float(json.loads(p.read_text())["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:  # noqa: BLE001
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")

    def __init__(self, device_index: int):
        self.idx = device_index
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.idx}", f"--query-gpu={self.QUERY}",
                                          "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE,
                                         stderr=subprocess.DEVNULL, text=True)
        except OSError:
            self.proc = None

    def stop(self) -> dict:
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
            out, _ = self.proc.communicate()
        sm, smax, reasons, power = [], [], set(), []
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                smax.append(float(f[2]))
                power.append(float(f[3]))
            except ValueError:
                continue
            for name, val in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if val.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(smax) if smax else None,
                "reasons": sorted(reasons), "samples": len(sm), "power_w_max": max(power) if power else None}


def build_transformers(V, kind: str, tuple_: bool):
    enc, dec = V.EquirectangularEncoder(), V.FisheyeDecoder("equidistant")
    if kind == "base":
        return enc * dec
    ql = V.quaternion(*Q_HALF)
    qr = ql.conj()  # cli.py:312-319: left eye gets conj(half_q), right eye half_q
    tl = enc * V.Euclidean3DRotator(qr) * V.PolynomialScaler(POLY) * dec
    tr = enc * V.Euclidean3DRotator(ql) * V.PolynomialScaler(POLY) * dec
    return (tl, tr) if tuple_ else tl


def oracle_ops(kind: str, conj: bool):
    from oracle import chain_np

    if kind == "base":
        return [("equirect_enc", True), ("fisheye_dec", "equidistant")]
    w, x, y, z = Q_HALF
    if conj:
        x, y, z = -x, -y, -z
    return [("equirect_enc", True), ("rot3", chain_np.quat_to_matrix(w, x, y, z).ravel().tolist()), ("poly", POLY),
            ("fisheye_dec", "equidistant")]


def synth_frames_torch(torch, n_frames: int, n: int, seed: int, device, vary_margin: bool = False):
    """Synthetic fisheye frames (SURVEY.md §8d): uniform random bytes inside the disc, zeros outside.  The bytes
    are drawn from [16, 256) so that no pixel INSIDE the disc is "black" for get_radius (b + g + r < 30,
    transformer.py:133): with [0, 256) about one pixel per scan line is, and radius="auto" then returns the
    distance between two noise pixels (0.5 ...) instead of the disc radius -(R + 0.5)."""
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    frames = torch.empty((n_frames, n, n, 3), dtype=torch.uint8, device=device)
    yy = torch.arange(n, device=device).view(n, 1)
    xx = torch.arange(n, device=device).view(1, n)
    r2 = (xx - n // 2) ** 2 + (yy - n // 2) ** 2
    for i0 in range(0, n_frames, 32):  # chunks: a 512-pair batch must not need a second copy of itself
        part = frames[i0:i0 + 32]
        part.copy_(torch.randint(16, 256, tuple(part.shape), dtype=torch.uint8, device=device, generator=g))
        if vary_margin:  # every frame gets a different disc radius (margin 8, 12, 16, 20, 8, ...)
            for i in range(part.shape[0]):
                part[i, r2 > (n // 2 - 8 - 4 * ((i0 + i) % 4)) ** 2] = 0
        else:
            part[:, r2 > (n // 2 - 8) ** 2] = 0
    return frames


def touched_fraction(torch, maps, n_in: int, taps: int) -> float:
    """Unique source pixels touched by the interpolation footprint / source pixels (algorithmic input bytes)."""
    xm, ym = maps[0].reshape(-1), maps[1].reshape(-1)
    ok = torch.isfinite(xm) & torch.isfinite(ym)
    if taps == 1:  # INTER_NEAREST: the pixel at cvRound(x), no sub-pixel grid
        sx, sy = torch.round(xm[ok].double()).long(), torch.round(ym[ok].double()).long()
        lo = hi = 0
    else:
        sx = torch.round(xm[ok].double() * 32).long() >> 5
        sy = torch.round(ym[ok].double() * 32).long() >> 5
        lo, hi = -(taps // 2 - 1), taps // 2
    touched = torch.zeros(n_in * n_in, dtype=torch.bool, device=maps.device)
    for dy in range(lo, hi + 1):
        for dx in range(lo, hi + 1):
            x, y = sx + dx, sy + dy
            m = (x >= 0) & (x < n_in) & (y >= 0) & (y < n_in)
            touched[(y[m] * n_in + x[m])] = True
    return float(touched.float().mean().item())


DUMP_BYTES = 48 << 20  # float32 row sample written by --dump-outputs: all rows of a small step, a sample of a batch


def dump_outputs(torch, sbs, out_dir: Path) -> None:
    """Seeded sample of whole rows of `sbs` (frames, rows, cols, channels uint8, one step's output) -> out_dir."""
    f, h, w, c = sbs.shape
    n_rows = max(1, min(f * h, DUMP_BYTES // (w * c * 4)))
    pick = np.sort(np.random.default_rng(0).choice(f * h, n_rows, replace=False))
    rows = sbs.reshape(f * h, w, c).index_select(0, torch.from_numpy(pick).to(sbs.device))
    out_dir.mkdir(parents=True, exist_ok=True)
    np.save(out_dir / "sbs_rows.npy", rows.cpu().numpy().astype(np.float32))
    np.save(out_dir / "sbs_rows_index.npy", np.stack([pick // h, pick % h], axis=1).astype(np.float64))


# ---------------------------------------------------------------------------------------------------------
# CPU reference path (oracle port: NumPy chain restatement + the real cv2.remap + concatenate)
# ---------------------------------------------------------------------------------------------------------
_ORACLE_MAPS: dict = {}


def oracle_maps(wl: dict):
    """The reference's maps for this workload from the NumPy restatement (oracle/chain_np.py), built once per process:
    [(xmap, ymap)] per eye-map, and the seconds the (single-threaded) build took."""
    from oracle import chain_np

    key = (wl["chain"], wl["tuple_"], wl["n"], wl["radius"])
    if key not in _ORACLE_MAPS:
        n = wl["n"]
        t0 = time.perf_counter()
        n_maps = 2 if wl["tuple_"] else 1
        # radius: the fixed-radius workloads use n / 2; the "auto" ones get_radius of the synthetic disc = -(n/2 - 8) - 0.5
        radius = n / 2 if wl["radius"] == "fixed" else -(n // 2 - 8) - 0.5
        maps = [chain_np.get_map(oracle_ops(wl["chain"], conj=(m == 0 and wl["tuple_"])), radius=radius,
                                 size_input=(n, n), size_output=(n, n)) for m in range(n_maps)]
        _ORACLE_MAPS[key] = (maps, time.perf_counter() - t0)
    return _ORACLE_MAPS[key]


CV_INTERP = {0: 0, 1: 1, 2: 2, 4: 4}  # cv2.INTER_NEAREST / LINEAR / CUBIC / LANCZOS4 are the API's integers


def oracle_sbs(wl: dict, left: np.ndarray, right: np.ndarray) -> np.ndarray:
    """What the reference produces for one pair: cv2.remap per eye on the oracle's maps + np.concatenate."""
    import cv2

    maps, _ = oracle_maps(wl)
    eyes = []
    for e, img in enumerate((left, right)):
        xm, ym = maps[e if len(maps) == 2 else 0]
        eyes.append(cv2.remap(img, xm, ym, interpolation=CV_INTERP[wl["interp"]], borderMode=cv2.BORDER_CONSTANT, borderValue=0))
    return np.concatenate(eyes, axis=1)


def cpu_reference_setup(wl: dict, sample_pairs: int):
    import cv2

    from oracle import chain_np

    n = wl["n"]
    rng_frames = []
    yy, xx = np.ogrid[:n, :n]
    outside = (xx - n // 2) ** 2 + (yy - n // 2) ** 2 > (n // 2 - 8) ** 2
    for i in range(2 * sample_pairs):
        img = np.random.default_rng(i).integers(16, 256, (n, n, 3), dtype=np.uint8)
        img[outside] = 0
        rng_frames.append(img)
    maps, t_maps = oracle_maps(wl)
    n_maps = len(maps)
    interp = CV_INTERP[wl["interp"]]

    def step():
        for p in range(sample_pairs):
            eyes = []
            for e in range(2):
                img = rng_frames[2 * p + e]
                if wl["radius"] == "auto":
                    chain_np.get_radius(img)
                xm, ym = maps[e if n_maps == 2 else 0]
                eyes.append(cv2.remap(img, xm, ym, interpolation=interp, borderMode=cv2.BORDER_CONSTANT, borderValue=0))
            np.concatenate(eyes, axis=1)

    return step, t_maps, cv2.getNumThreads()


def run_reference(args, wl_name: str, wl: dict) -> dict:
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return {}
    n = wl["n"]
    sample_pairs = 2 if n >= 4096 else 4
    step, t_maps, threads = cpu_reference_setup(wl, sample_pairs)
    for _ in range(max(1, min(args.warmup, 2))):
        step()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step()
    dt = (time.perf_counter() - t0) / args.steps
    mpix = sample_pairs * n * 2 * n / 1e6
    value = mpix / dt
    pairs = wl["pairs"]
    incl = pairs * n * 2 * n / 1e6 / (t_maps + pairs * dt / sample_pairs)
    return {
        "impl": "reference", "metric": "SBS equirect output Mpix/s", "value": value, "unit": "Mpix/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt * 1e3, "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "f64 maps / u8 fixed-point sampling", "data": "synthetic",
        "config": {"workload": wl_name, "description": wl["desc"], "sample_pairs_per_step": sample_pairs},
        "cpu_baseline": {"value": value, "unit": "Mpix/s", "cores": os.cpu_count(), "kind": "port",
                         "cv2_threads": threads,
                         "sample": f"{sample_pairs} pairs per step: cv2.remap x2 + np.concatenate with the maps cached "
                                   f"(reference apply(): one get_map for N images); get_map itself took {t_maps:.2f} s "
                                   f"for {2 if wl['tuple_'] else 1} map(s), single-threaded NumPy",
                         "map_build_s": t_maps, "value_incl_map_build_for_step_batch": incl},
        "e2e": {"value": value, "unit": "Mpix/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }


# ---------------------------------------------------------------------------------------------------------
# GPU arm
# ---------------------------------------------------------------------------------------------------------
def time_device(torch, fn, steps: int, warmup: int, dist):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record()
    for _ in range(steps):
        fn()
    ev1.record()
    torch.cuda.synchronize()
    ms = ev0.elapsed_time(ev1)
    if dist is not None:
        from vr180_convert_b200.shard import max_over_ranks

        ms = max_over_ranks(ms, dist, device="cuda")
        dist.barrier()
    return ms / steps


def run_workload(torch, V, wl_name: str, wl: dict, steps: int, warmup: int, dist, pairs: int | None = None,
                 want_e2e: bool = True, device=None, check_frames=(), dump_dir: Path | None = None):
    n = wl["n"]
    pairs = pairs or wl["pairs"]
    ring = 1
    if pairs * n * n * 3 * 4 < 300e6:  # keep the working set of consecutive steps above the 126 MB L2
        ring = int(np.ceil(300e6 / (pairs * n * n * 3 * 4)))
    t = build_transformers(V, wl["chain"], wl["tuple_"])
    radius = "auto" if wl["radius"] == "auto" else n / 2
    wp = V.SbsWarper(t, size_input=(n, n), size_output=(n, n), interpolation=wl["interp"], radius=radius,
                     map_source=wl["src"], device=device)
    left = synth_frames_torch(torch, pairs * ring, n, 1, device, vary_margin=wl.get("vary", False))
    right = synth_frames_torch(torch, pairs * ring, n, 2, device, vary_margin=wl.get("vary", False))
    out = torch.empty((pairs * ring, n, 2 * n, 3), dtype=torch.uint8, device=device)
    if wl["src"] != "analytic":
        {"lut_fixed": wp.fixed_lut, "lut_packed": wp.packed_lut, "lut": wp.maps}[wl["src"]]()
    state = {"i": 0}

    def step():
        k = state["i"] % ring
        state["i"] += 1
        s = slice(k * pairs, (k + 1) * pairs)
        wp(left[s], right[s], out=out[s])

    lib = V._native.lib()
    l0 = lib.vr180_launch_count()
    step()
    launches_per_step = lib.vr180_launch_count() - l0
    graphs = None
    if pairs * n * n <= 72e6:
        # a single pair (or a few small ones) per step is launch-bound from Python (ctypes call + 25 KB of kernel parameters ~ the kernel's
        # own duration): the step is captured once per ring slot in a CUDA graph and replayed, as a video loop would
        torch.cuda.synchronize()
        cap = torch.cuda.Stream(device)
        graphs = []
        with torch.cuda.stream(cap):
            for k in range(ring):
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g, stream=cap):
                    wp(left[k * pairs:(k + 1) * pairs], right[k * pairs:(k + 1) * pairs], out=out[k * pairs:(k + 1) * pairs])
                graphs.append(g)
        torch.cuda.synchronize()

        def step():  # noqa: F811
            k = state["i"] % ring
            state["i"] += 1
            graphs[k].replay()

    ms = time_device(torch, step, steps, warmup, dist)
    if dump_dir is not None:
        k = (state["i"] - 1) % ring  # the ring slot the last timed step wrote
        dump_outputs(torch, out[k * pairs:(k + 1) * pairs], dump_dir)
    mpix_step = pairs * n * 2 * n / 1e6

    # algorithmic bytes (DESIGN.md "roofline"): output written once + unique source pixels touched, per eye
    taps = {0: 1, 1: 2, 2: 4, 4: 8}[wl["interp"]]
    plan_for_maps = wp if not wp.auto_radius else V.SbsWarper(t, size_input=(n, n), size_output=(n, n),
                                                              interpolation=wl["interp"], radius=-(n // 2 - 8) - 0.5,
                                                              map_source="lut", device=device)
    maps = plan_for_maps.maps()
    fracs = [touched_fraction(torch, maps[m], n, taps) for m in range(maps.shape[0])]
    frac_in = sum(fracs) / len(fracs)
    if plan_for_maps is not wp or wl["src"] == "analytic":
        plan_for_maps._maps = None
    del maps
    lut_bytes = {"analytic": 0, "lut": 8, "lut_fixed": 8, "lut_packed": 4}[wl["src"]] * n * n * (1 if not wl["tuple_"] else 2)
    bytes_step = pairs * (2 * n * n * 3 + 2 * frac_in * n * n * 3) + lut_bytes  # LUT is read once per launch
    res = {"ms_per_step": ms, "mpix_per_step": mpix_step, "value": mpix_step / (ms / 1e3), "pairs": pairs,
           "launches_per_step": launches_per_step, "bytes_per_step": bytes_step, "touched_fraction": frac_in,
           "ring": ring, "launch": "CUDA graph replay" if graphs else "vr180_remap call per step"}

    if check_frames:
        # parity of the TIMED regime: frames of the batch launch itself (not of a separate small launch) go to the
        # host, where run_gpu compares them with cv2.remap on the oracle's maps
        out[:pairs].zero_()
        if graphs:
            graphs[0].replay()
        else:
            wp(left[:pairs], right[:pairs], out=out[:pairs])
        torch.cuda.synchronize()
        res["samples"] = [(f, left[f].cpu().numpy(), right[f].cpu().numpy(), out[f].cpu().numpy())
                          for f in sorted({min(max(f, 0), pairs - 1) for f in check_frames})]

    if want_e2e:
        import ctypes as C

        N = V._native
        pe = min(pairs, 32)
        nbytes_in, nbytes_out = pe * n * n * 3, pe * n * 2 * n * 3
        ptrs = []
        for nb in (nbytes_in, nbytes_in, nbytes_out):
            p = C.c_void_p()
            N.check(lib.vr180_host_alloc(nb, C.byref(p)), "vr180_host_alloc")
            ptrs.append(p)
        h_l = np.ctypeslib.as_array(C.cast(ptrs[0], C.POINTER(C.c_uint8)), shape=(pe, n, n, 3))
        h_r = np.ctypeslib.as_array(C.cast(ptrs[1], C.POINTER(C.c_uint8)), shape=(pe, n, n, 3))
        h_o = np.ctypeslib.as_array(C.cast(ptrs[2], C.POINTER(C.c_uint8)), shape=(pe, n, 2 * n, 3))
        h_l[:] = left[:pe].cpu().numpy()
        h_r[:] = right[:pe].cpu().numpy()
        job = N.HostJob()
        job.n_views, job.n_frames = 2, pe
        job.src[0], job.src[1] = ptrs[0].value, ptrs[1].value
        job.src_rows, job.src_cols, job.channels = n, n, 3
        for v in range(2):
            job.src_pitch[v], job.src_frame_stride[v] = n * 3, n * n * 3
        keep = []
        if wl["src"] == "analytic":
            job.map_kind = N.MAPSRC_ANALYTIC
            for m, ch in enumerate(wp._chains):
                job.chain[m] = C.pointer(ch)
        else:
            job.map_kind = N.MAPSRC_FLOAT2
            hm = wp.maps().cpu().numpy()
            keep.append(hm)
            for m in range(hm.shape[0]):
                job.xmap[m], job.ymap[m] = hm[m, 0].ctypes.data, hm[m, 1].ctypes.data
            job.maps_cache_key = 1
        job.share_map = 1 if wp.share_map else 0
        job.radius_mode = 1 if wp.auto_radius else 0
        job.threshold = 10.0
        job.out_w = job.out_h = n
        job.interpolation, job.border_mode = wl["interp"], 0
        job.dst, job.dst_pitch, job.dst_frame_stride = ptrs[2].value, 2 * n * 3, n * 2 * n * 3
        handle = C.c_void_p()
        N.check(lib.vr180_ctx_create(torch.cuda.current_device(), C.byref(handle)), "ctx_create")

        def e2e_step():
            N.check(lib.vr180_ctx_run(handle, C.byref(job)), "vr180_ctx_run")

        def timed_host(fn, reps):
            for _ in range(2):
                fn()
            if dist is not None:
                dist.barrier()
            t0 = time.perf_counter()
            for _ in range(reps):
                fn()  # synchronous: returns when every SBS frame is in host memory
            dt = (time.perf_counter() - t0) / reps
            if dist is not None:
                tt = torch.tensor([dt], dtype=torch.float64, device="cuda")
                dist.all_reduce(tt, op=dist.ReduceOp.MAX)
                dt = float(tt.item())
            return dt

        e_steps = max(3, min(steps, 10))
        dt = timed_host(e2e_step, e_steps)
        res["e2e"] = {"value": pe * n * 2 * n / 1e6 / dt, "unit": "Mpix/s", "h2d_bytes_per_step": 2 * nbytes_in,
                      "d2h_bytes_per_step": nbytes_out, "pairs_per_step": pe, "ms_per_step": dt * 1e3,
                      "api": "vr180_ctx_run (the C-ABI host call behind apply / apply_lr / lr_frames), page-locked host buffers"}
        res["e2e_frame0"] = h_o[0].copy()  # compared with the oracle by run_gpu

        # copy-only ceiling of the same traffic: page-locked H2D + D2H, no kernel, both directions at once; under
        # torchrun every rank measures at the same time, so the sum is the box's ceiling for N GPUs
        rates = (C.c_double * 4)()
        if dist is not None:
            dist.barrier()
        N.check(lib.vr180_debug_copy_ceiling(torch.cuda.current_device(), 256 << 20, 12, rates), "copy_ceiling")
        t_pair = max(2 * n * n * 3 / (rates[2] * 1e9), n * 2 * n * 3 / (rates[3] * 1e9))
        res["e2e"].update({"copy_ceiling": n * 2 * n / 1e6 / t_pair, "frac_of_ceiling": res["e2e"]["value"] / (n * 2 * n / 1e6 / t_pair),
                           "copy_gbs": {"h2d_alone": rates[0], "d2h_alone": rates[1], "h2d_concurrent": rates[2],
                                        "d2h_concurrent": rates[3]},
                           "copy_ceiling_note": "Mpix/s if the pair's 2 source frames (H2D) and its SBS frame (D2H) moved at "
                                                "the measured concurrent page-locked copy rates with no kernel and no "
                                                "pipeline fill / drain"})
        lib.vr180_ctx_destroy(handle)
        for p in ptrs:
            lib.vr180_host_free(p)
        del keep, h_l, h_r, h_o

        # the same metric through the PYTHON API on plain (pageable) NumPy arrays: V.lr_frames = apply_lr's in-memory
        # part for a clip, one host job; the sources are packed into the context's pinned ring by copy threads, the
        # SBS frames are returned as page-locked arrays
        lefts = [left[i].cpu().numpy() for i in range(pe)]
        rights = [right[i].cpu().numpy() for i in range(pe)]
        py_radius = "auto" if wl["radius"] == "auto" else n / 2
        state_py = {}

        def py_step():
            state_py["out"] = V.lr_frames(t, lefts, rights, size_output=(n, n), interpolation=wl["interp"], radius=py_radius)

        dtp = timed_host(py_step, max(3, min(steps, 5)))
        res["e2e_python_api"] = {"value": pe * n * 2 * n / 1e6 / dtp, "unit": "Mpix/s", "pairs_per_step": pe,
                                 "ms_per_step": dtp * 1e3, "h2d_bytes_per_step": 2 * nbytes_in,
                                 "d2h_bytes_per_step": nbytes_out,
                                 "api": "vr180_convert_b200.lr_frames(transformer, [ndarray...], [ndarray...]) on pageable "
                                        "NumPy arrays (apply_lr's in-memory part for a clip)",
                                 "vs_c_abi": (pe * n * 2 * n / 1e6 / dtp) / res["e2e"]["value"]}
        # ... and with the frames in page-locked arrays from V.pinned_empty (what a capture / decode loop that owns its
        # buffers would hand over): no packing copy, the Python layer's own overhead is what is left
        lefts_p, rights_p = [], []
        for i in range(pe):
            for dst_list, src_arr in ((lefts_p, lefts[i]), (rights_p, rights[i])):
                a_ = V.pinned_empty(src_arr.shape)
                a_[...] = src_arr
                dst_list.append(a_)

        def py_step_pinned():
            state_py["out"] = V.lr_frames(t, lefts_p, rights_p, size_output=(n, n), interpolation=wl["interp"], radius=py_radius)

        dtq = timed_host(py_step_pinned, max(3, min(steps, 5)))
        res["e2e_python_api"].update({"pinned_inputs_per_gpu_value": pe * n * 2 * n / 1e6 / dtq, "pinned_inputs_ms_per_step": dtq * 1e3,
                                      "pinned_inputs_vs_c_abi": (pe * n * 2 * n / 1e6 / dtq) / res["e2e"]["value"]})
        del lefts_p, rights_p
        res["e2e_python_frame0"] = np.array(state_py["out"][0])
        del lefts, rights, state_py
    del left, right, out, wp
    torch.cuda.empty_cache()
    return res


def run_gpu(args) -> dict:
    import torch

    import vr180_convert_b200 as V

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU path")
    torch.cuda.set_device(local)
    V.set_device(local)
    device = torch.device("cuda", local)
    if world > 1:  # one process per GPU: keep the rank and its pinned staging buffers on the GPU's NUMA node
        from vr180_convert_b200.shard import bind_host_near_gpu

        bound = bind_host_near_gpu(local)
        print(f"[rank {rank}] host CPUs near GPU {local}: {len(bound) if bound else 'unchanged'}", file=sys.stderr)
    dist = None
    if world > 1:
        import torch.distributed as dist_mod

        dist_mod.init_process_group("nccl", device_id=device)
        dist = dist_mod
    wl = WORKLOADS[args.workload]
    for kv in filter(None, args.debug_set.split(",")):
        what, val = kv.split("=")
        V._native.lib().vr180_debug_set(int(what), int(val))
    peak, peak_src = measured_peak()
    sampler = ClockSampler(local)
    lib = V._native.lib()
    if rank == 0:
        sampler.start()
    launches0 = lib.vr180_launch_count()
    want_parity = rank == 0 and world == 1 and not args.no_cpu_baseline
    n_pairs = args.pairs or wl["pairs"]
    main = run_workload(torch, V, args.workload, wl, args.steps, args.warmup, dist, pairs=args.pairs, device=device,
                        want_e2e=not args.no_e2e,
                        check_frames=(0, n_pairs // 2 - 1, n_pairs - 1) if want_parity else (),
                        dump_dir=args.dump_outputs if rank == 0 else None)
    clocks = sampler.stop() if rank == 0 else {}
    # total shards = world * pairs (weak scaling)
    value = main["value"] * world
    achieved = main["bytes_per_step"] / (main["ms_per_step"] / 1e3) / 1e9
    traffic = None  # DRAM bytes (read + written) of one launch from the committed ncu capture of this workload
    tp = ROOT / "profiles" / "traffic.json"
    if tp.exists():
        try:
            t = json.loads(tp.read_text()).get(args.workload)
            if t and int(t.get("pairs_per_launch", -1)) == int(main["pairs"]):
                traffic = t["dram_bytes_per_launch"]
        except Exception:  # noqa: BLE001
            traffic = None
    line = {
        "metric": "SBS equirect output Mpix/s", "value": value, "unit": "Mpix/s", "n_gpus": world, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": main["ms_per_step"], "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "f64 coordinates / u8 fixed-point (INTER_BITS=5) sampling", "data": "synthetic",
        "config": {"workload": args.workload, "description": wl["desc"], "pairs_per_gpu_per_step": main["pairs"],
                   **({"debug_set": args.debug_set} if args.debug_set else {}),
                   "frame_ring": main["ring"], "launch": main["launch"], "l2": "inputs+outputs of one step exceed the 126 MB L2 (no flush needed)",
                   "parallelism": f"frames sharded over {world} GPU(s), no collective"},
        "gpu_launches": main["launches_per_step"] * args.steps,
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                     "traffic": traffic, "traffic_unit": "DRAM bytes per launch (ncu dram__bytes_read.sum + dram__bytes_write.sum)",
                     "peak_source": peak_src, "frac_of_nominal_8TBs": achieved / 8000.0,
                     "algorithmic_bytes_per_launch": main["bytes_per_step"],
                     "source_touched_fraction": main["touched_fraction"],
                     "kernel": "vr180::tiled::k_warp_tiled (1 launch per step; k_warp_stream for <= 20 / 16 (frame, eye) "
                               "rectangles per tile with tile-packed LUTs)"},
        "e2e": None,
        "clocks": clocks,
    }
    if main.get("e2e"):
        e = dict(main["e2e"])
        ceiling, py = e["copy_ceiling"], main["e2e_python_api"]["value"]
        slowest = ceiling
        if dist is not None:  # whole-job numbers: every rank ran its own pipeline / copy test at the same time
            tt = torch.tensor([ceiling, py], dtype=torch.float64, device="cuda")
            dist.all_reduce(tt, op=dist.ReduceOp.SUM)
            tm = torch.tensor([ceiling], dtype=torch.float64, device="cuda")
            dist.all_reduce(tm, op=dist.ReduceOp.MIN)
            ceiling, py, slowest = float(tt[0].item()), float(tt[1].item()), float(tm[0].item())
        # `value` is timed as the max over ranks, so the fair bound is world x the SLOWEST rank's copy rate (GPUs far from
        # the host's memory get less of it); `copy_ceiling` (the sum of the ranks' rates) is the box's total
        e.update({"per_gpu_value": e["value"], "value": e["value"] * world, "copy_ceiling": ceiling,
                  "frac_of_ceiling": e["value"] * world / ceiling,
                  "copy_ceiling_at_slowest_rank": slowest * world,
                  "frac_of_ceiling_at_slowest_rank": e["value"] / slowest,
                  "h2d_bytes_per_step": e["h2d_bytes_per_step"] * world, "d2h_bytes_per_step": e["d2h_bytes_per_step"] * world})
        line["e2e"] = e
        line["e2e_python_api"] = {**main["e2e_python_api"], "per_gpu_value": main["e2e_python_api"]["value"], "value": py,
                                  "h2d_bytes_per_step": e["h2d_bytes_per_step"], "d2h_bytes_per_step": e["d2h_bytes_per_step"]}

    def parity_of(w, res):
        """Frames of the timed launch (and frame 0 of the two host-buffer legs) against cv2.remap on the oracle's maps."""
        out = {"vs": "cv2.remap + np.concatenate on the maps of oracle/chain_np.py (the reference's get_map restated)",
               "frames_of_the_timed_launch": [], "mismatched_bytes": 0}
        want0 = None
        for f, l, r, o in res.get("samples", []):
            want = oracle_sbs(w, l, r)
            if f == 0:
                want0 = want
            out["frames_of_the_timed_launch"].append(f)
            out["mismatched_bytes"] += int((want != o).sum())
        for key in ("e2e_frame0", "e2e_python_frame0"):
            if key in res and want0 is not None:
                out[key + "_mismatched_bytes"] = int((want0 != res[key]).sum())
        out["bit_exact"] = all(v == 0 for k, v in out.items() if k.endswith("mismatched_bytes"))
        return out

    if want_parity:
        line["parity"] = parity_of(wl, main)
        if not line["parity"]["bit_exact"]:
            print("PARITY FAILURE: the timed launch differs from the oracle", line["parity"], file=sys.stderr)
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        step, t_maps, threads = cpu_reference_setup(wl, 2 if wl["n"] >= 4096 else 4)
        sp = 2 if wl["n"] >= 4096 else 4
        step()
        reps = 3
        t0 = time.perf_counter()
        for _ in range(reps):
            step()
        dt = (time.perf_counter() - t0) / reps
        n = wl["n"]
        line["cpu_baseline"] = {
            "value": sp * n * 2 * n / 1e6 / dt, "unit": "Mpix/s", "cores": os.cpu_count(), "kind": "port",
            "cv2_threads": threads,
            "sample": f"{sp} pairs x {reps} reps of cv2.remap x2 + np.concatenate with cached maps (oracle port of "
                      f"remapper.py:388-398,518); the NumPy get_map restatement took {t_maps:.2f} s for "
                      f"{2 if wl['tuple_'] else 1} map(s) (single thread) and is reported separately",
            "map_build_s": t_maps,
            "value_incl_map_build_for_step_batch":
                main["pairs"] * n * 2 * n / 1e6 / (t_maps + main["pairs"] * dt / sp)}
    for k in ("samples", "e2e_frame0", "e2e_python_frame0"):
        main.pop(k, None)
    if not args.no_other_workloads and world == 1 and args.pairs is None:
        # every other BASELINE config, 5 timed steps each, frames 0 and last of each timed launch checked like above
        others = {}
        for name, w in WORKLOADS.items():
            if name == args.workload:
                continue
            vary = w.get("vary", False)
            # the reference's default interpolation also through the host-buffer call: apply() with default arguments
            e2e_too = name == "8k_lanczos4_fixed" and not args.no_e2e
            r = run_workload(torch, V, name, w, 5, 3, None, want_e2e=e2e_too, device=device,
                             check_frames=((0,) if vary else (0, w["pairs"] - 1)) if want_parity else ())
            a = r["bytes_per_step"] / (r["ms_per_step"] / 1e3) / 1e9
            others[name] = {"value": r["value"], "unit": "Mpix/s", "ms_per_step": r["ms_per_step"], "steps": 5,
                            "pairs_per_step": r["pairs"], "roofline_frac": a / peak, "achieved_gbs": a,
                            "launch": r["launch"], "description": w["desc"]}
            if r.get("e2e"):
                others[name]["e2e"] = {k: r["e2e"][k] for k in ("value", "unit", "pairs_per_step", "ms_per_step", "api", "frac_of_ceiling")}
                others[name]["e2e_python_api"] = {k: r["e2e_python_api"][k] for k in ("value", "unit", "ms_per_step", "api")}
            if want_parity:
                par = parity_of(w, r)
                others[name]["parity_bit_exact"] = par["bit_exact"]
                others[name]["parity_frames"] = par["frames_of_the_timed_launch"]
                if not par["bit_exact"]:
                    print(f"PARITY FAILURE in {name}", par, file=sys.stderr)
            del r
        line["other_workloads"] = others
    line["gpu_launches_total_in_process"] = lib.vr180_launch_count() - launches0
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()
    return line if rank == 0 else {}


def main() -> None:
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="8k_rot_poly_linear", choices=sorted(WORKLOADS))
    ap.add_argument("--pairs", type=int, default=None, help="stereo pairs per GPU per step")
    ap.add_argument("--all-workloads", action="store_true", help="(default at N=1; kept for old command lines)")
    ap.add_argument("--no-other-workloads", action="store_true", help="only the headline workload")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true", help="skip the host-buffer leg (profiling runs)")
    ap.add_argument("--debug-set", default="", help="experiments: comma list of what=value for vr180_debug_set "
                                                    "(0 frames per CTA, 1 tiled flags, 2 frames-per-CTA cap)")
    ap.add_argument("--dump-outputs", type=Path, default=None, metavar="DIR",
                    help="write a seeded sample of the last timed step's SBS frames to DIR/*.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs is not None and args.impl != "b200":
        ap.error("--dump-outputs writes the outputs of the GPU path (--impl b200)")
    args.warmup = max(args.warmup, 3) if args.impl == "b200" else args.warmup

    # stdout carries exactly ONE line, the JSON result: whatever libraries print there while the bench runs (NCCL's
    # version banner, for instance) goes to stderr instead
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        if line:
            print(json.dumps(line), flush=True)

    if args.impl == "reference":
        emit(run_reference(args, args.workload, WORKLOADS[args.workload]))
        return

    if args.gpus > 1 and "WORLD_SIZE" not in os.environ:  # not under torchrun: spawn one rank per GPU ourselves
        with socket.socket() as s:
            s.bind(("127.0.0.1", 0))
            port = s.getsockname()[1]
        cmd = [sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={args.gpus}",
               "--master-addr", "127.0.0.1", "--master-port", str(port), str(Path(__file__).resolve()), *sys.argv[1:]]
        os.dup2(real_stdout, 1)  # the ranks do their own redirection
        raise SystemExit(subprocess.call(cmd))

    emit(run_gpu(args))


if __name__ == "__main__":
    main()
