"""Device time of the reflection-pad kernels at the generator's C3 shapes (CUDA events, L2 flushed between iterations).

    python tools/bench_pad.py
"""
import json
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parent.parent))
from contrast_gan_3d_b200 import ops  # noqa: E402


def timeit(fn, iters=10):
    flush = torch.empty(256 << 20, dtype=torch.uint8, device="cuda")
    fn(); torch.cuda.synchronize()
    tot = 0.0
    for _ in range(iters):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record(); torch.cuda.synchronize()
        tot += e0.elapsed_time(e1)
    return tot / iters


def main():
    dev = torch.device("cuda", 0)
    x1 = torch.randn(16, 128, 128, 128, 1, device=dev).to(torch.bfloat16)
    ref = torch.nn.functional.pad(x1.float().permute(0, 4, 1, 2, 3), (3,) * 6, mode="reflect").permute(0, 2, 3, 4, 1).to(torch.bfloat16)
    assert torch.equal(ops.reflect_pad(x1, 3), ref)
    ms = timeit(lambda: ops.reflect_pad(x1, 3))
    print(json.dumps({"kernel": "reflect_pad 16x128^3x1 bf16", "ms": round(ms, 4), "GBps": round((x1.numel() + ref.numel()) * 2 / ms / 1e6, 1)}))
    g = torch.randn(16, 134, 134, 134, 16, device=dev).to(torch.bfloat16)
    ms = timeit(lambda: ops.reflect_pad_backward(g, 3))
    print(json.dumps({"kernel": "reflect_pad_backward 16x134^3x16 bf16", "ms": round(ms, 4), "GBps": round((g.numel() + 16 * 128 ** 3 * 16) * 2 / ms / 1e6, 1)}))


if __name__ == "__main__":
    main()
