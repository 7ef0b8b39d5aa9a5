"""Cost of the ResNet-block dropout (resnet_dropout_prob > 0), measured with CUDA events after warm-up:

  kernels  bn_apply vs bn_apply_dropout, bn_backward_reduce and bn_backward_apply without and with dropout, at the C3
           ResNet activation (16 x 32^3 x 64 bf16 = 67 MB; keep bitmask 4.2 MB).  Four buffer sets are used in rotation
           (about 0.55 GB), so successive launches do not find their inputs in the 126 MB L2.  GB/s counts the algorithmic
           bytes (each input read once, each output written once, the bitmask included).
  steps    the C3 train step (16 opt + 8 low + 8 high 128^3 patches, bf16, both networks trained, replayed from a CUDA
           graph) with resnet_dropout_prob 0 and 0.5, alternated in the same process for several rounds.

Prints one JSON line with the card name and power limit read in the same run; --out also writes it to a file."""
from __future__ import annotations

import argparse
import json
import subprocess
import sys
from functools import partial
from pathlib import Path

import torch

ROOT = Path(__file__).resolve().parent.parent
sys.path.insert(0, str(ROOT))

from contrast_gan_3d_b200 import _lib  # noqa: E402
from contrast_gan_3d_b200.ops import _p, _st, call  # noqa: E402


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True,
                           text=True, timeout=30).stdout.strip().splitlines()[0]
    except Exception as e:  # noqa: BLE001
        q = f"{torch.cuda.get_device_name(0)}, power limit unavailable ({e})"
    return q


def hbm_peak():
    p = ROOT / "MEASURED_PEAKS.json"
    return (json.loads(p.read_text())["hbm_gbs"], "MEASURED_PEAKS.json") if p.exists() else (6650.0, "fallback")


def time_rotating(fns, iters):
    """ms per launch of fns[i % len(fns)] over `iters` launches (after one warm-up pass over every buffer set)."""
    for f in fns:
        f()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(iters):
        fns[i % len(fns)]()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def kernel_rows(iters, nbuf=4, rows=16 * 32 ** 3, C=64, p=0.5):
    dev, dt = "cuda", _lib.BF16
    act = _lib.ACT_NONE  # block0 of a ResNet block has no activation (reference model/blocks.py:68-88)
    sets = []
    for _ in range(nbuf):
        y = torch.randn(rows, C, device=dev).bfloat16()
        sets.append(dict(y=y, dz=torch.randn_like(y), z=torch.empty_like(y), keep=torch.empty(rows * C // 8, dtype=torch.uint8, device=dev),
                         sums=torch.empty(2 * C, dtype=torch.float64, device=dev)))
    mi = torch.cat([torch.zeros(C, device=dev), torch.ones(C, device=dev)])
    gamma, beta = torch.ones(C, device=dev), torch.zeros(C, device=dev)
    dg, db = torch.empty(C, device=dev), torch.empty(C, device=dev)
    seed = torch.tensor([1234], dtype=torch.int64, device=dev)
    k = (_p(mi), _p(gamma), _p(beta), act, 0.0)
    for s in sets:  # real masks for the backward passes
        call("cgan3d_bn_apply_dropout", _p(s["y"]), _p(s["z"]), _p(s["keep"]), dt, rows, C, *k, p, _p(seed), _st())
    ops = {
        "bn_apply": (lambda s: call("cgan3d_bn_apply", _p(s["y"]), _p(s["z"]), dt, rows, C, *k, None, _st()), 2, False),
        "bn_apply_dropout": (lambda s: call("cgan3d_bn_apply_dropout", _p(s["y"]), _p(s["z"]), _p(s["keep"]), dt, rows, C, *k, p,
                                            _p(seed), _st()), 2, True),
        "bn_backward_reduce": (lambda s: call("cgan3d_bn_backward_reduce", _p(s["dz"]), _p(s["y"]), dt, rows, C, *k, _p(s["sums"]),
                                              _st()), 2, False),
        "bn_backward_reduce_dropout": (lambda s: call("cgan3d_bn_backward_reduce_dropout", _p(s["dz"]), _p(s["y"]), _p(s["keep"]), dt,
                                                      rows, C, *k, p, _p(s["sums"]), _st()), 2, True),
        "bn_backward_apply": (lambda s: call("cgan3d_bn_backward_apply", _p(s["dz"]), _p(s["y"]), _p(s["z"]), dt, rows, C, *k,
                                             _p(s["sums"]), _p(dg), _p(db), 0.0, _st()), 3, False),
        "bn_backward_apply_dropout": (lambda s: call("cgan3d_bn_backward_apply_dropout", _p(s["dz"]), _p(s["y"]), _p(s["keep"]),
                                                     _p(s["z"]), dt, rows, C, *k, p, _p(s["sums"]), _p(dg), _p(db), 0.0, _st()), 3, True),
    }
    peak, src = hbm_peak()
    act_bytes = rows * C * 2
    out = []
    for rnd in range(2):  # two rounds: the spread between them is the run-to-run noise
        for name, (fn, passes, mask) in ops.items():
            ms = time_rotating([partial(fn, s) for s in sets], iters)
            nbytes = passes * act_bytes + (rows * C // 8 if mask else 0)
            gbs = nbytes / (ms * 1e-3) / 1e9
            out.append({"round": rnd, "kernel": name, "shape": f"{rows} x {C} bf16", "p": p if mask else 0.0, "us": round(ms * 1e3, 2),
                        "algorithmic_MB": round(nbytes / 1e6, 1), "GB_per_s": round(gbs, 1), "frac_hbm_peak": round(gbs / peak, 3)})
    return out, src


def time_c3_step(p, steps, warmup):
    from contrast_gan_3d_b200.model import HULoss, PatchGANDiscriminator, ResnetGenerator
    from contrast_gan_3d_b200.optim import FusedAdam
    from contrast_gan_3d_b200.trainer.Trainer import NullLogger, Trainer

    torch.manual_seed(0)
    dt = torch.bfloat16
    tr = Trainer(10 ** 9, 2, None, 1, 1, 0, 0, partial(ResnetGenerator, 4, 2, 16, resnet_dropout_prob=p, compute_dtype=dt),
                 partial(PatchGANDiscriminator, 1, 8, 3, negative_slope=0.2, compute_dtype=dt),
                 partial(FusedAdam, lr=2e-4, betas=(0.5, 0.999)), partial(FusedAdam, lr=2e-4, betas=(0.5, 0.999)),
                 HULoss(0.18666666666666668, 0.35333333333333333), NullLogger(), torch.device("cuda:0"),
                 weight_clip=0.01, checkpoint_every=None)
    tr.enable_cuda_graph()
    g = torch.Generator(device="cuda").manual_seed(1)
    P = (128, 128, 128)
    mk = lambda n: (torch.randn((n, 1, *P), device="cuda", generator=g) * 0.5)
    batch = [dict(data=mk(16), seg=None), dict(data=mk(8), seg=torch.rand((8, 1, *P), device="cuda", generator=g) < 1e-3),
             dict(data=mk(8), seg=torch.rand((8, 1, *P), device="cuda", generator=g) < 1e-3)]
    for i in range(warmup):  # eager warm-up steps, the capture, and a first replay
        tr.train_step(batch, i)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for i in range(steps):
        logs = tr.train_step(batch, warmup + i)
    e1.record()
    torch.cuda.synchronize()
    assert all(bool(torch.isfinite(v)) for v in logs.values())
    launches = tr.graph_launches_per_step()
    tr.release_cuda_graphs()
    return round(e0.elapsed_time(e1) / steps, 3), launches


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--iters", type=int, default=200)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--rounds", type=int, default=3)
    ap.add_argument("--out", type=str, default=None)
    a = ap.parse_args()
    assert torch.cuda.is_available(), "bench_dropout needs a GPU"
    res = {"card": card()}
    res["kernels"], res["hbm_peak_source"] = kernel_rows(a.iters)
    torch.cuda.empty_cache()
    steps = {"p0": [], "p0.5": []}
    launches = {}
    for _ in range(a.rounds):  # alternated: other work shares the host
        for key, p in (("p0", 0.0), ("p0.5", 0.5)):
            ms, launches[key] = time_c3_step(p, a.steps, a.warmup)
            steps[key].append(ms)
            torch.cuda.empty_cache()
    res["c3_step_ms"] = steps
    res["c3_step_spread_ms"] = {k: round(max(v) - min(v), 3) for k, v in steps.items()}
    res["graph_launches_per_step"] = launches
    line = json.dumps(res)
    print(line)
    if a.out:
        Path(a.out).parent.mkdir(parents=True, exist_ok=True)
        Path(a.out).write_text(line + "\n")


if __name__ == "__main__":
    main()
