import sys, json
sys.path.insert(0, ".")
import torch
from tests import dropout_oracle as DO
from contrast_gan_3d_b200.model.blocks import ResNetBlock
DEV = "cuda:0"
def cl(x): return x.permute(0, 2, 3, 4, 1).contiguous()
def ncl(x): return x.permute(0, 4, 1, 2, 3).contiguous()
for C in (64, 4):
    for dtype in (torch.float32, torch.bfloat16):
        for p, shift in ((0.0, False), (0.3, False), (0.0, True), (0.3, True)):
            if shift and dtype == torch.float32:
                continue
            torch.manual_seed(2)
            blk = ResNetBlock(False, C, C, dropout_prob=p, compute_dtype=dtype)
            with torch.no_grad():
                for b in (blk.block0, blk.block1):
                    b.normalization.weight.uniform_(0.5, 1.5); b.normalization.bias.uniform_(-0.5, 0.5)
                if shift:
                    blk.block1.normalization.bias.uniform_(6.0, 7.0)
            ref = {k: v.clone() for k, v in blk.state_dict().items()}
            x = torch.randn(2, C, 6, 7, 5); gy = torch.randn(2, C, 6, 7, 5)
            blk = blk.to(DEV)
            xd = cl(x).to(DEV).requires_grad_(True)
            out = blk.forward_cl(xd)
            out.backward(cl(gy).to(DEV).to(out.dtype))
            drop = None
            if p > 0:
                drop = {"block0": (DO.unpack_mask(blk.dropout_mask, (2, 6, 7, 5, C)), p)}
            params = {k: v.clone().requires_grad_(True) for k, v in ref.items() if "running" not in k and "num_batches" not in k}
            bufs = {k: v.clone() for k, v in ref.items() if k not in params}
            layers = [dict(name="block0", kind="res0", cin=C, cout=C, k=3, stride=1, pad=1, pad_mode="zeros", out_pad=0, norm=True, act="none", bias=False),
                      dict(name="block1", kind="res1", cin=C, cout=C, k=3, stride=1, pad=1, pad_mode="zeros", out_pad=0, norm=True, act="relu", bias=False)]
            xr = x.clone().requires_grad_(True)
            yr = DO.generator_forward(params, bufs, xr, layers, train=True, dropout=drop)
            names = list(params)
            grads = torch.autograd.grad(yr, [xr] + [params[k] for k in names], gy)
            rows = [("out", ncl(out), yr), ("dx", ncl(xd.grad), grads[0])]
            rows += [(k, dict(blk.named_parameters())[k].grad, g) for k, g in zip(names, grads[1:])]
            rows += [(k, blk.state_dict()[k], v) for k, v in bufs.items() if "running" in k]
            res = {}
            for nm, a, b in rows:
                a, b = a.detach().float().cpu(), b.detach().float().cpu()
                e = (a - b).abs()
                if dtype == torch.float32:
                    r = float((e / (1e-4 * b.abs() + 1e-5)).max())
                else:
                    r = float((e / (2e-2 * b.abs() + 2e-2 * b.abs().max())).max())
                cos = float(torch.nn.functional.cosine_similarity(a.flatten().double(), b.flatten().double(), dim=0))
                frac_bad = float((e > (1e-4 * b.abs() + 1e-5) if dtype == torch.float32 else e > (2e-2 * b.abs() + 2e-2 * b.abs().max())).float().mean())
                res[nm] = (round(r, 3), f"err/max {float(e.max() / b.abs().max()):.1e}", f"bad {frac_bad:.1e}", f"cos {1 - cos:.1e}")
            print(json.dumps({"C": C, "dtype": str(dtype), "p": p, "shift": shift, "ratio_err_to_tol": res}), flush=True)
