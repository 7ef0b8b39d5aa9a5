"""Time SpatialTransform2 (the reference's SpatialTransform_2 on the device) on a seeded C3 batch of 16 patches of
128^3, with CUDA events after warm-up:

  ref     the transform at the reference's probabilities (experiments/b200_conf.py: elastic 0.1, rotation 0.2, scale 0.2)
  forced  every branch on for every sample (elastic, rotation and scaling)
  step    DevicePatchSampler + bf16 Trainer.train_step on C3 (16 opt + 8 low + 8 high), without and with the transform

Prints one JSON line with the card name and power limit read in the same run; --out also writes it to a file."""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
import time
from functools import partial
from pathlib import Path

import numpy as np
import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))

from contrast_gan_3d_b200.data import DevicePatchSampler, SpatialTransform2  # noqa: E402
from contrast_gan_3d_b200.experiments import b200_conf  # noqa: E402

P = (128, 128, 128)


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        q = f"{torch.cuda.get_device_name(0)}, power limit unavailable ({e})"
    return q


def algorithmic_bytes(draws, S=P, pad=12):
    """Bytes each stage must move at least: elastic fields (noise generated in the first pass; 3 passes read and write
    3 fp32 fields, one reduction read, one normalising read + write), the prefilter (read the crop, write the padded
    coefficients, two in-place passes) and the resample (coefficients once, offsets, crop seg, fp32 + u8 outputs)."""
    v, vs = int(np.prod(P)), int(np.prod(S))
    vp = int(np.prod([s + 2 * pad for s in S]))
    total = 0
    for r in draws:
        if r["elastic"]:
            total += 3 * (4 * v + 8 * v + 8 * v) + 3 * 4 * v + 3 * 8 * v
        if "ctr" in r:
            total += 4 * vs + 4 * vp + 2 * 8 * vp
            total += 4 * vp + vs + 5 * v + (12 * v if r["elastic"] else 0)
        else:
            total += 5 * vs + 5 * v
    return total


def time_transform(t, batch, iters):
    for _ in range(3):
        t(batch)
    torch.cuda.synchronize()
    np.random.seed(0)
    nbytes = 0
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    h0 = time.perf_counter()
    e0.record()
    for _ in range(iters):
        state = np.random.get_state()
        nbytes += algorithmic_bytes(t.draw(batch["data"].shape[0], np.random))
        np.random.set_state(state)  # the call below draws the same parameters
        t(batch)
    e1.record()
    torch.cuda.synchronize()
    wall = (time.perf_counter() - h0) / iters * 1e3
    ms = e0.elapsed_time(e1) / iters
    return {"ms_per_batch": round(ms, 4), "host_wall_ms_per_batch": round(wall, 4),
            "algorithmic_MB_per_batch": round(nbytes / iters / 1e6, 2), "GB_per_s": round(nbytes / iters / ms / 1e6, 1)}


def kernel_breakdown(t, batch, iters=5):
    """Device time per batch of each augmentation kernel (torch.profiler, a run of its own)."""
    from torch.profiler import ProfilerActivity, profile

    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        for _ in range(iters):
            t(batch)
        torch.cuda.synchronize()
    names = ("smooth_pass_kernel<true>", "smooth_pass_kernel<false>", "field_partials_kernel", "field_finalize_kernel",
             "field_scale_kernel", "prefilter_z_kernel", "prefilter_xy_kernel", "spatial_resample_kernel", "Memcpy HtoD")
    out = {}
    for ev in prof.key_averages():
        us = getattr(ev, "device_time_total", None) or getattr(ev, "cuda_time_total", 0)
        for n in names:
            if us and n in ev.key:
                out[n] = round(out.get(n, 0.0) + us / iters / 1e3, 4)
    return dict(sorted(out.items(), key=lambda kv: -kv[1]))


def time_steps(transform, vols, steps, warmup):
    from contrast_gan_3d_b200.model import HULoss, PatchGANDiscriminator, ResnetGenerator
    from contrast_gan_3d_b200.optim import FusedAdam
    from contrast_gan_3d_b200.trainer.Trainer import NullLogger, Trainer

    np.random.seed(0)
    torch.manual_seed(0)
    dt = torch.bfloat16
    tr = Trainer(10 ** 9, 2, None, 1, 1, 0, 0, partial(ResnetGenerator, 4, 2, 16, compute_dtype=dt),
                 partial(PatchGANDiscriminator, 1, 8, 3, negative_slope=0.2, compute_dtype=dt),
                 partial(FusedAdam, lr=2e-4, betas=(0.5, 0.999)), partial(FusedAdam, lr=2e-4, betas=(0.5, 0.999)),
                 HULoss(0.18666666666666668, 0.35333333333333333), NullLogger(), torch.device("cuda:0"),
                 weight_clip=0.01, checkpoint_every=None)
    samplers = [DevicePatchSampler(vols, P, b, transform=transform) for b in (16, 8, 8)]

    def step():
        b = [s.generate_train_batch() for s in samplers]
        b[0] = dict(b[0], seg=None)
        return tr.train_step(b, 0)

    for _ in range(warmup):
        step()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        logs = step()
    e1.record()
    torch.cuda.synchronize()
    assert all(np.isfinite(float(v.detach())) for v in logs.values())
    return round(e0.elapsed_time(e1) / steps, 3)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=20)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--out", type=str, default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "bench_augment needs a GPU"
    rng = np.random.default_rng(0)
    vols = []
    for _ in range(4):
        v = np.clip(rng.normal(100, 400, size=(160, 160, 160, 2)), -1024, 1500).astype(np.int16)
        v[..., 1] = rng.random((160, 160, 160)) < 0.01
        vols.append(torch.from_numpy(v).cuda())
    np.random.seed(0)
    batch = DevicePatchSampler(vols, P, 16).generate_train_batch()
    ref = b200_conf.train_transform
    ref.noise_rng = np.random.default_rng(0)
    forced = SpatialTransform2(P, p_el_per_sample=1, p_rot_per_sample=1, p_scale_per_sample=1,
                               angle_x=(-np.pi / 6, np.pi / 6), angle_y=(-np.pi / 6, np.pi / 6),
                               angle_z=(-np.pi / 6, np.pi / 6), scale=(0.7, 1.4), noise_rng=np.random.default_rng(0))
    res = {"card": card(), "batch": "16 x 1 x 128^3 fp32 crops (C3 opt batch)",
           "ref_probabilities": time_transform(ref, batch, a.iters),
           "all_branches": time_transform(forced, batch, a.iters)}
    res["kernel_ms_per_batch_all_branches"] = kernel_breakdown(forced, batch)
    plain, aug = [], []
    for _ in range(3):  # alternated: other work shares the host
        plain.append(time_steps(None, vols, a.steps, a.warmup))
        aug.append(time_steps(ref, vols, a.steps, a.warmup))
    res["sampler_train_step_ms"] = {"no_transform": plain, "ref_transform_on_all_three_samplers": aug}
    line = json.dumps(res)
    print(line)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
