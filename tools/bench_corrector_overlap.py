"""Whole-volume correction with and without overlapping tiles, on the C2 case: a synthetic 512x512x256 int16 volume,
128^3 tiles, batches of 16, bf16 generator, through CCTAContrastCorrector.__call__ (host int16 in, host HU out).

Rows: the default (disjoint tiles, avg), step 64 with avg, step 64 with gaussian, and each of them with eval_mode.
Per row:
  e2e_ms           median wall time of a call, which ends in a device synchronise
  generator_ms     CUDA events around each batch's generator pass, summed over the volume
  stitch_ms        CUDA events around cgan3d_tile_stitch, mean over repeated launches on the call's own inputs
  stitch_gbps      (every tile read once + the output volume written once) / stitch_ms, against HBM_PEAK_TBPS
  lib_calls        libcgan3d entry-point calls per volume (each enqueues at least one kernel)
The default row is also timed against the previous per-tile stitching (cgan3d_tile_extract / _accumulate / _finalize per
tile, reproduced below), alternating old and new in the same process to show the run-to-run spread.

    python tools/bench_corrector_overlap.py [--iters 7] [--alternate 8] [--out file.json]
"""
from __future__ import annotations

import argparse
import importlib
import json
import subprocess
import sys
import time
from functools import partial
from pathlib import Path

import numpy as np
import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

HBM_PEAK_TBPS = 7.7  # NVIDIA HGX B200 data sheet, per GPU (at up to 1,000 W)
SHAPE, PATCH, BATCH = (512, 512, 256), (128, 128, 128), 16
ROWS = [dict(tile_step=None, blend="avg"), dict(tile_step=64, blend="avg"), dict(tile_step=64, blend="gaussian")]


def card():
    name = torch.cuda.get_device_name(0)
    try:
        r = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i", "0"],
                           capture_output=True, text=True, timeout=30)
        power = r.stdout.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        power = "unknown"
    return name, power


def make(**kw):
    from contrast_gan_3d_b200.data import FactorZeroCenterScaler
    from contrast_gan_3d_b200.eval import CCTAContrastCorrector
    from contrast_gan_3d_b200.model import ResnetGenerator

    torch.manual_seed(0)
    return CCTAContrastCorrector(partial(ResnetGenerator, 4, 2, 16, compute_dtype=torch.bfloat16),
                                 FactorZeroCenterScaler(-1024, 1500, 600), torch.device("cuda:0"),
                                 inference_patch_size=PATCH, **kw)


def old_call(corr, vol):
    """The previous corrector's __call__: per tile one cgan3d_tile_extract and one cgan3d_tile_accumulate, then
    cgan3d_tile_finalize (the entry points are still exported)."""
    from contrast_gan_3d_b200 import ops
    from contrast_gan_3d_b200._lib import call
    from contrast_gan_3d_b200.eval import grid_tiles

    with torch.no_grad():
        v = corr._upload(vol)
        X, Y, Z = v.shape
        tiles = grid_tiles((X, Y, Z), PATCH)
        acc = torch.zeros((X, Y, Z), dtype=torch.float32, device=v.device)
        cnt = torch.zeros_like(acc)
        sh, f, st = float(corr.scaler.shift), float(corr.scaler.factor), ops._st
        for i in range(0, len(tiles), BATCH):
            chunk = tiles[i:i + BATCH]
            xb = torch.empty((len(chunk), 1, *PATCH), dtype=torch.float32, device=v.device)
            for j, (x0, y0, z0) in enumerate(chunk):
                call("cgan3d_tile_extract", v.data_ptr(), X, Y, Z, x0, y0, z0, *PATCH, sh, f, xb[j].data_ptr(), st())
            c = corr._corrected(xb)
            for j, (x0, y0, z0) in enumerate(chunk):
                call("cgan3d_tile_accumulate", c[j].data_ptr(), acc.data_ptr(), cnt.data_ptr(), X, Y, Z, x0, y0, z0,
                     *PATCH, st())
        out = torch.empty_like(acc)
        call("cgan3d_tile_finalize", acc.data_ptr(), cnt.data_ptr(), out.data_ptr(), acc.numel(), sh, f, st())
        host = torch.empty(out.shape, dtype=out.dtype, pin_memory=True)
        host.copy_(out, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return host


def timed(fn, n):
    ts = []
    for _ in range(n):
        t0 = time.perf_counter()
        fn()
        ts.append((time.perf_counter() - t0) * 1e3)
    return ts


def breakdown(corr, vol, repeats=20):
    """One call with CUDA events around the generator passes and around the stitch launch (relaunched `repeats` times
    while its inputs are alive); returns (generator_ms, stitch_ms, lib_calls, n_tiles)."""
    from contrast_gan_3d_b200 import _lib

    mod = importlib.import_module("contrast_gan_3d_b200.eval.CCTAContrastCorrector")  # the module, not the class
    gen, stitch, info = [], [], {}
    inner_corrected, inner_call = corr._corrected, mod.call

    def corrected(xb):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        c = inner_corrected(xb)
        e1.record()
        gen.append((e0, e1))
        return c

    def call(name, *args):
        if name != "cgan3d_tile_stitch":
            return inner_call(name, *args)
        rc = inner_call(name, *args)
        info["n"] = args[1]
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(repeats):
            getattr(_lib.lib(), name)(*args)
        e1.record()
        stitch.append((e0, e1))
        return rc

    corr._corrected, mod.call = corrected, call
    try:
        n0 = _lib.launch_count
        corr(vol, batch_size=BATCH)
        calls = _lib.launch_count - n0
    finally:
        del corr._corrected
        mod.call = inner_call
    torch.cuda.synchronize()
    g = sum(a.elapsed_time(b) for a, b in gen)
    s = stitch[0][0].elapsed_time(stitch[0][1]) / repeats
    return g, s, calls, info["n"]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=7)
    ap.add_argument("--alternate", type=int, default=8, help="old/new pairs for the default row")
    ap.add_argument("--out", default=None)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("needs a CUDA device")
    name, power = card()
    vol = np.clip(np.random.default_rng(0).normal(100, 300, size=SHAPE), -1024, 1500).astype(np.int16)
    res = {"case": "C2 volume 512x512x256 int16, 128^3 tiles, batch 16, bf16 generator", "gpu": name,
           "power_limit": power, "hbm_peak_tbps": HBM_PEAK_TBPS, "rows": []}
    for row in ROWS:
        for eval_mode in (False, True):
            corr = make(eval_mode=eval_mode, **row)
            for _ in range(2):
                corr(vol, batch_size=BATCH)
            torch.cuda.synchronize()
            ts = timed(lambda: corr(vol, batch_size=BATCH), args.iters)
            g, s, calls, n = breakdown(corr, vol)
            nbytes = n * int(np.prod(PATCH)) * 4 + int(np.prod(SHAPE)) * 4
            r = {"tile_step": row["tile_step"], "blend": row["blend"], "eval_mode": eval_mode, "tiles": n,
                 "e2e_ms": float(np.median(ts)), "e2e_ms_min": min(ts), "e2e_ms_max": max(ts), "generator_ms": g,
                 "stitch_ms": s, "stitch_bytes": nbytes, "stitch_gbps": nbytes / s / 1e6,
                 "stitch_share_of_hbm_peak": nbytes / (s * 1e-3) / (HBM_PEAK_TBPS * 1e12), "lib_calls": calls,
                 "tile_stack_bytes": n * int(np.prod(PATCH)) * 4}
            res["rows"].append(r)
            print(json.dumps(r), flush=True)
            del corr
            torch.cuda.empty_cache()
    corr = make()
    for _ in range(2):
        corr(vol, batch_size=BATCH)
        old_call(corr, vol)
    old, new = [], []
    for _ in range(args.alternate):
        old += timed(lambda: old_call(corr, vol), 1)
        new += timed(lambda: corr(vol, batch_size=BATCH), 1)
    from contrast_gan_3d_b200 import _lib
    n0 = _lib.launch_count
    old_call(corr, vol)
    res["default_old_vs_new"] = {"old_ms": old, "new_ms": new, "old_median": float(np.median(old)),
                                 "new_median": float(np.median(new)), "old_lib_calls": _lib.launch_count - n0}
    print(json.dumps(res["default_old_vs_new"]), flush=True)
    if args.out:
        Path(args.out).parent.mkdir(parents=True, exist_ok=True)
        Path(args.out).write_text(json.dumps(res, indent=1) + "\n")


if __name__ == "__main__":
    main()
