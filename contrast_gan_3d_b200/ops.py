"""Tensor-level wrappers over the libcgan3d C ABI and the autograd.Functions built on them.

PyTorch is used for device memory, streams and the autograd tape only; every numerical
kernel on the hot path is one of ours (include/cgan3d.h).  CUDA tensors are mandatory: a
CPU tensor raises, there is no fallback.

Activation tensors inside the networks are channels-last ``[B, X, Y, Z, C]`` contiguous,
fp32 or bf16 (X, Y, Z are the reference's W, H, D).
"""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass
from typing import Optional, Tuple

import torch

from . import _lib
from ._lib import ConvGeom, call

_CONV_IMPL = _lib.IMPL_AUTO


def set_conv_impl(impl: int) -> int:
    """Select the convolution implementation: IMPL_AUTO / IMPL_GENERIC / IMPL_TC (tests, benches)."""
    global _CONV_IMPL
    old, _CONV_IMPL = _CONV_IMPL, impl
    return old


def _need_cuda(*ts):
    for t in ts:
        if t is not None and not t.is_cuda:
            raise RuntimeError("contrast_gan_3d_b200 runs on CUDA tensors only (no CPU path); got a CPU tensor")


def _p(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


def _st():
    return torch.cuda.current_stream().cuda_stream


def _dt(dtype: torch.dtype) -> int:
    if dtype == torch.float32:
        return _lib.F32
    if dtype == torch.bfloat16:
        return _lib.BF16
    raise TypeError(f"unsupported activation dtype {dtype}")


# ------------------------------------------------------------------------------------------
# plain wrappers
# ------------------------------------------------------------------------------------------
def cast(x: torch.Tensor, dtype: torch.dtype) -> torch.Tensor:
    if x.dtype == dtype:
        return x
    _need_cuda(x)
    x = x.contiguous()
    out = torch.empty_like(x, dtype=dtype)
    call("cgan3d_cast", _p(x), _dt(x.dtype), _p(out), _dt(dtype), x.numel(), _st())
    return out


def pack_weights(w: torch.Tensor, dtype: torch.dtype) -> torch.Tensor:
    """fp32 [Cs, Cb, k, k, k] -> `dtype` [k^3, Cb, Cs]."""
    _need_cuda(w)
    Cs, Cb, k = w.shape[0], w.shape[1], w.shape[2]
    w = w.detach().contiguous()
    out = torch.empty((k ** 3, Cb, Cs), dtype=dtype, device=w.device)
    call("cgan3d_pack_weights", _p(w), _p(out), _dt(dtype), Cs, Cb, k, _st())
    return out


def _workspace(g: ConvGeom, dt: int, op: int, device) -> Tuple[Optional[torch.Tensor], int]:
    n = _lib.lib().cgan3d_conv_workspace_bytes(C.byref(g), dt, op)
    if n == 0:
        return None, 0
    ws = torch.empty(n, dtype=torch.uint8, device=device)
    return ws, n


# Optional per-launch device timing of the convolution kernels (bench.py roofline): CUDA events recorded on the
# launching stream around each conv entry point.  Off by default.
_CONV_TIMING = None


def enable_conv_timing(on: bool = True) -> None:
    global _CONV_TIMING
    _CONV_TIMING = [] if on else None


def conv_timing_summary() -> dict:
    """{(op, dtype, geometry key): (n_launches, total_ms, flops_per_launch, impl)} — call after a synchronize."""
    out = {}
    for key, flops, impl, e0, e1 in _CONV_TIMING or []:
        n, ms, _, _ = out.get(key, (0, 0.0, flops, impl))
        out[key] = (n + 1, ms + e0.elapsed_time(e1), flops, impl)
    return out


class _timed:
    def __init__(self, op: str, g: ConvGeom, dt: int):
        self.rec = None
        if _CONV_TIMING is not None:
            flops = 2.0 * g.B * g.Xs * g.Ys * g.Zs * g.Cs * g.Cb * g.k ** 3  # 2*MAC of the base conv (any of the 3 ops)
            impl = _lib.lib().cgan3d_conv_select(C.byref(g), dt, {"gather": 0, "scatter": 1, "wgrad": 2}[op])
            if _CONV_IMPL == _lib.IMPL_GENERIC:
                impl = 1
            self.rec = ((op, dt) + g.key(), flops, impl, torch.cuda.Event(enable_timing=True),
                        torch.cuda.Event(enable_timing=True))

    def __enter__(self):
        if self.rec is not None:
            self.rec[3].record()

    def __exit__(self, *a):
        if self.rec is not None:
            self.rec[4].record()
            _CONV_TIMING.append(self.rec)


def conv_gather(g: ConvGeom, big, wp, out_dtype=None, impl=None):
    dt = _dt(big.dtype)
    small = torch.empty((g.B, g.Xs, g.Ys, g.Zs, g.Cs), dtype=big.dtype, device=big.device)
    ws, n = _workspace(g, dt, _lib.OP_GATHER, big.device)
    with _timed("gather", g, dt):
        call("cgan3d_conv_gather", C.byref(g), dt, _p(big), _p(wp), None, _p(small), _p(ws), n,
             _CONV_IMPL if impl is None else impl, _st())
    return small


def conv_scatter(g: ConvGeom, small, wp, impl=None):
    dt = _dt(small.dtype)
    big = torch.empty((g.B, g.Xb, g.Yb, g.Zb, g.Cb), dtype=small.dtype, device=small.device)
    ws, n = _workspace(g, dt, _lib.OP_SCATTER, small.device)
    with _timed("scatter", g, dt):
        call("cgan3d_conv_scatter", C.byref(g), dt, _p(small), _p(wp), None, _p(big), _p(ws), n,
             _CONV_IMPL if impl is None else impl, _st())
    return big


def conv_fuses_bnstats(g: ConvGeom, dtype: torch.dtype, transposed: bool) -> bool:
    """True when the tcgen05 kernel of this layer can emit the BatchNorm batch statistics from its epilogue."""
    if _CONV_IMPL == _lib.IMPL_GENERIC or dtype != torch.bfloat16:
        return False
    return bool(_lib.lib().cgan3d_conv_fuses_bnstats(C.byref(g), _dt(dtype), _lib.OP_SCATTER if transposed else _lib.OP_GATHER))


def conv_bnstats(g: ConvGeom, x, wp, transposed: bool):
    """conv (gather, or scatter for a transposed module) + per-channel [sum, sum of squares] (fp64 [2*Cout]) in one launch."""
    dt = _dt(x.dtype)
    op = _lib.OP_SCATTER if transposed else _lib.OP_GATHER
    if transposed:
        out = torch.empty((g.B, g.Xb, g.Yb, g.Zb, g.Cb), dtype=x.dtype, device=x.device)
    else:
        out = torch.empty((g.B, g.Xs, g.Ys, g.Zs, g.Cs), dtype=x.dtype, device=x.device)
    sums = torch.empty(2 * out.shape[-1], dtype=torch.float64, device=x.device)
    ws, n = _workspace(g, dt, op, x.device)
    with _timed("scatter" if transposed else "gather", g, dt):
        call("cgan3d_conv_bnstats", C.byref(g), dt, op, _p(x), _p(wp), _p(out), _p(sums), _p(ws), n, _st())
    return out, sums


def conv_wgrad(g: ConvGeom, big, small, impl=None, out=None, ws=None):
    """dW (fp32, torch layout [Cs, Cb, k, k, k]); with `out` the kernel ACCUMULATES into it (beta = 1).  `ws`: a workspace
    the caller allocated (on the stream that owns the memory pool), else one is allocated on the current stream."""
    dt = _dt(big.dtype)
    dw = out if out is not None else torch.empty((g.Cs, g.Cb, g.k, g.k, g.k), dtype=torch.float32, device=big.device)
    if out is not None and (out.dtype != torch.float32 or not out.is_contiguous() or out.numel() != g.Cs * g.Cb * g.k ** 3):
        raise ValueError("conv_wgrad: `out` must be a contiguous fp32 tensor of the weight's size")
    if ws is None:
        ws, n = _workspace(g, dt, _lib.OP_WGRAD, big.device)
    else:
        n = ws.numel()
    with _timed("wgrad", g, dt):
        call("cgan3d_conv_wgrad", C.byref(g), dt, _p(big), _p(small), _p(dw), 0.0 if out is None else 1.0, _p(ws), n,
             _CONV_IMPL if impl is None else impl, _st())
    return dw


# Weight-gradient sink (parallel.GradBucketReducer between prepare() and finish()): the wgrad kernel accumulates straight
# into the parameter's gradient-bucket slice on a side stream instead of returning a fresh tensor to autograd, so that it
# overlaps the HBM-bound BatchNorm-backward passes that follow on the compute stream.
_GRAD_SINK = None
_FWD_USES = {}  # id(weight) -> forward applications whose weight gradient has not been produced yet


def set_grad_sink(sink) -> None:
    global _GRAD_SINK
    _GRAD_SINK = sink


def _note_forward_use(weight) -> None:
    _FWD_USES[id(weight)] = _FWD_USES.get(id(weight), 0) + 1


def forget_forward_uses(params) -> None:
    for p in params:
        _FWD_USES.pop(id(p), None)


def _direct_target(param):
    """`param.grad` when the active sink wants this parameter's gradient accumulated in place by our kernel, else None."""
    sink = _GRAD_SINK
    if sink is not None and param is not None and sink.accepts(param):
        return param.grad
    return None


def _grad_handled(param, direct: bool) -> None:
    """One pending application of `param` has produced its gradient (in place when `direct`)."""
    if param is None:
        return
    left = _FWD_USES.get(id(param), 1) - 1
    _FWD_USES[id(param)] = max(left, 0)
    if direct and left <= 0:
        _GRAD_SINK.direct_done(param)


def _weight_grad(weight, g: ConvGeom, big, small):
    """The weight gradient of one conv application: returned to autograd, or (sink active) accumulated in place on the
    sink's side stream, in which case None is returned and the sink is told when the parameter's last pending
    application has been handled."""
    sink = _GRAD_SINK
    if sink is None or weight is None or not sink.accepts(weight):
        if weight is not None:
            n = _FWD_USES.get(id(weight), 0)
            if n > 0:
                _FWD_USES[id(weight)] = n - 1
        return conv_wgrad(g, big, small)
    main = torch.cuda.current_stream(big.device)
    # per-kernel timing (bench.py's instrumented pass) needs exclusive durations: keep the kernel on the compute stream then
    side = main if _CONV_TIMING is not None else sink.side_stream(big.device)
    # the workspace comes from the COMPUTE stream's pool: under CUDA-graph capture only that stream's allocations belong to
    # the graph's private pool, and memory handed out to the side stream could be given to someone else between replays
    ws, _ = _workspace(g, _dt(big.dtype), _lib.OP_WGRAD, big.device)
    if side is not main:
        side.wait_stream(main)  # `big` / `small` were produced on the compute stream
    with torch.cuda.stream(side):
        conv_wgrad(g, big, small, out=weight.grad, ws=ws)
    if side is not main:
        for t in (big, small, ws):
            if t is not None:
                t.record_stream(side)
    left = _FWD_USES.get(id(weight), 1) - 1
    _FWD_USES[id(weight)] = max(left, 0)
    if left <= 0:
        sink.direct_done(weight)
    return None


def reflect_pad(x, pad):
    B, X, Y, Z, Cc = x.shape
    out = torch.empty((B, X + 2 * pad, Y + 2 * pad, Z + 2 * pad, Cc), dtype=x.dtype, device=x.device)
    call("cgan3d_reflect_pad", _p(x), _p(out), _dt(x.dtype), B, X, Y, Z, Cc, pad, _st())
    return out


def reflect_pad_backward(gp, pad):
    B, Xp, Yp, Zp, Cc = gp.shape
    X, Y, Z = Xp - 2 * pad, Yp - 2 * pad, Zp - 2 * pad
    out = torch.empty((B, X, Y, Z, Cc), dtype=gp.dtype, device=gp.device)
    call("cgan3d_reflect_pad_backward", _p(gp), _p(out), _dt(gp.dtype), B, X, Y, Z, Cc, pad, _st())
    return out


# ------------------------------------------------------------------------------------------
# conv block: conv -> (BatchNorm | bias) -> activation (+ residual)
# ------------------------------------------------------------------------------------------
@dataclass
class ConvSpec:
    """Static description of one conv layer (reference model/blocks.py:5-38)."""
    transposed: bool
    cin: int
    cout: int
    k: int
    stride: int
    pad: int
    reflect: bool = False
    out_pad: int = 0

    def geometry(self, B: int, spatial: Tuple[int, int, int]) -> Tuple[ConvGeom, Tuple[int, int, int]]:
        """(geometry of the base conv as the kernels see it, output spatial shape)."""
        k, s, p = self.k, self.stride, self.pad
        if not self.transposed:
            big = tuple(d + 2 * p for d in spatial) if self.reflect else tuple(spatial)
            pe = 0 if self.reflect else p
            small = tuple((d + 2 * pe - k) // s + 1 for d in big)
            if min(small) < 1:
                raise ValueError(f"input {spatial} too small for k={k}, stride={s}, pad={p}")
            g = ConvGeom(B, *big, self.cin, *small, self.cout, k, s, pe)
            return g, small
        small = tuple(spatial)
        big = tuple((d - 1) * s - 2 * p + k + self.out_pad for d in small)
        g = ConvGeom(B, *big, self.cout, *small, self.cin, k, s, p)
        return g, big


@dataclass
class BlockCfg:
    spec: ConvSpec
    act: int = _lib.ACT_NONE
    slope: float = 0.0
    dtype: torch.dtype = torch.float32  # storage dtype of this layer's activations
    out_f32: bool = False
    training: bool = True
    momentum: float = 0.1
    eps: float = 1e-5
    pad_out: int = 0          # > 0: return reflect_pad(output, pad_out) -- the padding of the consumer, fused into the normalise pass
    pre_padded: bool = False  # the input already carries this layer's reflection padding (produced with pad_out)
    dropout: float = 0.0      # > 0: element-wise dropout after the activation (BatchNorm blocks, no residual / pad_out)


class ConvBlockFn(torch.autograd.Function):
    """act(norm(conv(x))) [+ residual]  — reference ConvBlock.forward (model/blocks.py:52-53) and the
    skip connection of ResNetBlock.forward (:87-88), as one autograd node.

    With cfg.dropout = p > 0 the node also applies nn.Dropout(p) to its output (the dropout of ResNetBlock, :68-88), fused
    into the normalise pass, and returns (output, keep bitmask): uint8 [ceil(numel / 8)], bit e & 7 of byte e >> 3 set
    when the channels-last element e was kept.  The mask's seed is drawn from torch's CUDA generator on the device, one
    per call, so torch.manual_seed reproduces the masks and every replay of a captured CUDA graph draws new ones."""

    @staticmethod
    def forward(ctx, x, weight, bias, gamma, beta, residual, running_mean, running_var, nbt, cfg: BlockCfg):
        _need_cuda(x, weight)
        spec = cfg.spec
        B, X, Y, Z, Cin = x.shape
        assert Cin == spec.cin, f"expected {spec.cin} input channels, got {Cin}"
        xin = cast(x.detach().contiguous(), cfg.dtype)
        if spec.reflect:
            xin = reflect_pad(xin, spec.pad)
        g, out_sp = spec.geometry(B, (X, Y, Z))
        wp = pack_weights(weight, cfg.dtype)
        n_rows, Co = B * out_sp[0] * out_sp[1] * out_sp[2], spec.cout
        dt = _dt(cfg.dtype)
        sums = None
        if gamma is not None and cfg.training and conv_fuses_bnstats(g, cfg.dtype, spec.transposed):
            y, sums = conv_bnstats(g, xin, wp, spec.transposed)  # batch statistics from the conv epilogue
        else:
            y = conv_scatter(g, xin, wp) if spec.transposed else conv_gather(g, xin, wp)
        mi = keep = None
        padded = False
        if gamma is not None:
            mi = torch.empty(2 * Co, dtype=torch.float32, device=x.device)
            if cfg.training:
                if sums is None:
                    sums = torch.empty(2 * Co, dtype=torch.float64, device=x.device)
                    call("cgan3d_bn_stats", _p(y), dt, n_rows, Co, _p(sums), _st())
                call("cgan3d_bn_finalize", _p(sums), n_rows, Co, cfg.eps, cfg.momentum, _p(mi), _p(running_mean),
                     _p(running_var), _p(nbt), _st())
            else:
                call("cgan3d_bn_eval_params", _p(running_mean), _p(running_var), Co, cfg.eps, _p(mi), _st())
            res = None
            if residual is not None:
                res = cast(residual.detach().contiguous(), cfg.dtype)
            po = cfg.pad_out
            if cfg.dropout > 0:
                if res is not None or po:
                    raise NotImplementedError("dropout is fused only into a block without residual or padded output")
                seed = torch.randint(-2 ** 63, 2 ** 63 - 1, (1,), dtype=torch.int64, device=x.device)
                keep = torch.empty((y.numel() + 7) // 8, dtype=torch.uint8, device=y.device)
                z = torch.empty_like(y)
                call("cgan3d_bn_apply_dropout", _p(y), _p(z), _p(keep), dt, n_rows, Co, _p(mi), _p(gamma.detach()),
                     _p(beta.detach()), cfg.act, cfg.slope, cfg.dropout, _p(seed), _st())
            elif po and res is None and not cfg.out_f32 and Co % 8 == 0:
                # normalise + activate straight into the consumer's reflection-padded input
                z = torch.empty((B, out_sp[0] + 2 * po, out_sp[1] + 2 * po, out_sp[2] + 2 * po, Co), dtype=y.dtype, device=y.device)
                call("cgan3d_bn_apply_pad", _p(y), _p(z), dt, B, out_sp[0], out_sp[1], out_sp[2], Co, _p(mi), _p(gamma.detach()),
                     _p(beta.detach()), cfg.act, cfg.slope, po, _st())
                padded = True
            else:
                z = torch.empty_like(y)
                call("cgan3d_bn_apply", _p(y), _p(z), dt, n_rows, Co, _p(mi), _p(gamma.detach()), _p(beta.detach()),
                     cfg.act, cfg.slope, _p(res), _st())
        else:
            assert residual is None
            if cfg.dropout > 0:
                raise NotImplementedError("dropout is fused only into BatchNorm blocks")
            if bias is None and cfg.act == _lib.ACT_NONE:
                z = y
            else:
                z = torch.empty_like(y)
                call("cgan3d_bias_act", _p(y), _p(z), dt, n_rows, Co, _p(None if bias is None else bias.detach()),
                     cfg.act, cfg.slope, _st())
        if cfg.pad_out and not padded:
            z = reflect_pad(z, cfg.pad_out)
        if cfg.out_f32:
            z = cast(z, torch.float32)
        ctx.cfg, ctx.g = cfg, g
        ctx.wparam = weight if ctx.needs_input_grad[1] else None  # the parameter itself: its .grad may be the wgrad sink
        ctx.small_params = tuple(p if (p is not None and ctx.needs_input_grad[i]) else None
                                 for i, p in ((2, bias), (3, gamma), (4, beta)))
        for p in (ctx.wparam,) + ctx.small_params:
            if p is not None:
                _note_forward_use(p)
        ctx.x_dtype = x.dtype
        ctx.has_res = residual is not None
        ctx.res_dtype = None if residual is None else residual.dtype
        ctx.in_spatial = (X, Y, Z)
        ctx.save_for_backward(xin, wp, y, mi, gamma, beta, bias, keep)
        if keep is not None:
            ctx.mark_non_differentiable(keep)
            return z, keep
        return z

    @staticmethod
    def backward(ctx, dz, *_):
        cfg, g = ctx.cfg, ctx.g
        spec = cfg.spec
        xin, wp, y, mi, gamma, beta, bias, keep = ctx.saved_tensors
        dt = _dt(cfg.dtype)
        dz = cast(dz.contiguous(), cfg.dtype)
        if cfg.pad_out:
            dz = reflect_pad_backward(dz, cfg.pad_out)  # adjoint of the consumer's padding
        Co = spec.cout
        n_rows = y.numel() // Co
        dgamma = dbeta = dbias = None
        if gamma is not None:
            if not cfg.training:
                raise NotImplementedError("backward through eval-mode BatchNorm is not part of the hot path")
            sums = torch.empty(2 * Co, dtype=torch.float64, device=y.device)
            if keep is not None:
                call("cgan3d_bn_backward_reduce_dropout", _p(dz), _p(y), _p(keep), dt, n_rows, Co, _p(mi), _p(gamma), _p(beta),
                     cfg.act, cfg.slope, cfg.dropout, _p(sums), _st())
            else:
                call("cgan3d_bn_backward_reduce", _p(dz), _p(y), dt, n_rows, Co, _p(mi), _p(gamma), _p(beta), cfg.act,
                     cfg.slope, _p(sums), _st())
            dy = torch.empty_like(y)
            pbias, pgamma, pbeta = ctx.small_params
            # parameter gradients: accumulated into the gradient bucket by the same launch when a sink is active
            tg, tb = _direct_target(pgamma), _direct_target(pbeta)
            direct = tg is not None and tb is not None
            if not direct:
                tg = torch.empty(Co, dtype=torch.float32, device=y.device)
                tb = torch.empty(Co, dtype=torch.float32, device=y.device)
            if keep is not None:
                call("cgan3d_bn_backward_apply_dropout", _p(dz), _p(y), _p(keep), _p(dy), dt, n_rows, Co, _p(mi), _p(gamma),
                     _p(beta), cfg.act, cfg.slope, cfg.dropout, _p(sums), _p(tg), _p(tb), 1.0 if direct else 0.0, _st())
            else:
                call("cgan3d_bn_backward_apply", _p(dz), _p(y), _p(dy), dt, n_rows, Co, _p(mi), _p(gamma), _p(beta),
                     cfg.act, cfg.slope, _p(sums), _p(tg), _p(tb), 1.0 if direct else 0.0, _st())
            _grad_handled(pgamma, direct)
            _grad_handled(pbeta, direct)
            dgamma, dbeta = (None, None) if direct else (tg, tb)
        elif bias is not None or cfg.act != _lib.ACT_NONE:
            sums = torch.empty(Co, dtype=torch.float64, device=y.device)
            dy = torch.empty_like(y)
            call("cgan3d_bias_act_backward", _p(dz), _p(y), _p(dy), dt, n_rows, Co, _p(bias), cfg.act, cfg.slope,
                 _p(sums), _st())
            if bias is not None:
                pbias = ctx.small_params[0]
                tb = _direct_target(pbias)
                direct = tb is not None
                dbias = tb if direct else torch.empty(Co, dtype=torch.float32, device=y.device)
                call("cgan3d_sums_to_f32", _p(sums), _p(dbias), Co, 1.0, 1.0 if direct else 0.0, _st())
                _grad_handled(pbias, direct)
                if direct:
                    dbias = None
        else:
            dy = dz
        dres = cast(dz, ctx.res_dtype) if ctx.has_res else None
        dx = None
        if ctx.needs_input_grad[0]:
            if spec.transposed:
                dx = conv_gather(g, dy, wp)
            else:
                dx = conv_scatter(g, dy, wp)
                if spec.reflect:
                    dx = reflect_pad_backward(dx, spec.pad)
            dx = cast(dx, ctx.x_dtype)
        dw = None
        if ctx.needs_input_grad[1]:
            dw = _weight_grad(ctx.wparam, g, dy, xin) if spec.transposed else _weight_grad(ctx.wparam, g, xin, dy)
        return dx, dw, dbias, dgamma, dbeta, dres, None, None, None, None


class GenTailFn(torch.autograd.Function):
    """last_conv (7^3 reflect, bias) -> tanh, optionally fused with opt_hat = subopt - attenuation
    (reference generator.py:77-85 and trainer/Trainer.py:170-171)."""

    @staticmethod
    def forward(ctx, x, weight, bias, subopt, cfg: BlockCfg):
        _need_cuda(x, weight)
        spec = cfg.spec
        B, X, Y, Z, Cin = x.shape
        xin = cast(x.detach().contiguous(), cfg.dtype)
        if cfg.pre_padded:  # the producer wrote its output already reflection-padded (BlockCfg.pad_out)
            assert spec.reflect
            X, Y, Z = X - 2 * spec.pad, Y - 2 * spec.pad, Z - 2 * spec.pad
        elif spec.reflect:
            xin = reflect_pad(xin, spec.pad)
        g, _ = spec.geometry(B, (X, Y, Z))
        wp = pack_weights(weight, cfg.dtype)
        y = conv_gather(g, xin, wp)
        n = y.numel()
        att = torch.empty((B, 1, X, Y, Z), dtype=torch.float32, device=x.device)
        opt_hat = None
        sub = None
        if subopt is not None:
            sub = subopt.detach().contiguous()
            assert sub.dtype == torch.float32 and sub.numel() == n
            opt_hat = torch.empty_like(att)
        call("cgan3d_tanh_residual", _p(y), _p(bias.detach()), _p(sub), _p(att), _p(opt_hat), _dt(cfg.dtype), n, _st())
        ctx.cfg, ctx.g, ctx.x_dtype = cfg, g, x.dtype
        ctx.wparam = weight if ctx.needs_input_grad[1] else None
        ctx.bparam = bias if ctx.needs_input_grad[2] else None
        for p in (ctx.wparam, ctx.bparam):
            if p is not None:
                _note_forward_use(p)
        ctx.save_for_backward(xin, wp, att)
        if opt_hat is None:
            return att, att.new_empty(0)
        return att, opt_hat

    @staticmethod
    def backward(ctx, d_att, d_opt_hat):
        cfg, g = ctx.cfg, ctx.g
        spec = cfg.spec
        xin, wp, att = ctx.saved_tensors
        n = att.numel()
        if d_opt_hat is not None and d_opt_hat.numel() != n:
            d_opt_hat = None
        if d_att is None and d_opt_hat is None:
            return None, None, None, None, None
        da = None if d_att is None else d_att.contiguous()
        do = None if d_opt_hat is None else d_opt_hat.contiguous()
        dy = torch.empty((g.B, g.Xs, g.Ys, g.Zs, 1), dtype=cfg.dtype, device=att.device)
        sums = torch.empty(1, dtype=torch.float64, device=att.device)
        call("cgan3d_tanh_residual_backward", _p(do), _p(da), _p(att), _p(dy), _dt(cfg.dtype), n, _p(sums), _st())
        tb = _direct_target(ctx.bparam)
        direct = tb is not None
        dbias = tb if direct else torch.empty(1, dtype=torch.float32, device=att.device)
        call("cgan3d_sums_to_f32", _p(sums), _p(dbias), 1, 1.0, 1.0 if direct else 0.0, _st())
        _grad_handled(ctx.bparam, direct)
        if direct:
            dbias = None
        dx = None
        if ctx.needs_input_grad[0]:
            dx = conv_scatter(g, dy, wp)
            if spec.reflect and not cfg.pre_padded:
                dx = reflect_pad_backward(dx, spec.pad)
            dx = cast(dx, ctx.x_dtype)
        dw = _weight_grad(ctx.wparam, g, xin, dy) if ctx.needs_input_grad[1] else None
        return dx, dw, dbias, None, None


# ------------------------------------------------------------------------------------------
# losses
# ------------------------------------------------------------------------------------------
class MeanFn(torch.autograd.Function):
    """scale * mean(x) as a 0-dim fp32 tensor (Wasserstein terms, reference model/loss.py:77-79)."""

    @staticmethod
    def forward(ctx, x, scale: float):
        _need_cuda(x)
        xc = x.detach().contiguous()
        out = torch.empty((), dtype=torch.float32, device=x.device)
        scratch = torch.empty(1, dtype=torch.float64, device=x.device)
        call("cgan3d_mean", _p(xc), _dt(xc.dtype), xc.numel(), float(scale), _p(scratch), _p(out), _st())
        ctx.shape, ctx.dtype, ctx.scale = x.shape, x.dtype, float(scale)
        return out

    @staticmethod
    def backward(ctx, gout):
        n = 1
        for s in ctx.shape:
            n *= s
        gx = torch.empty(ctx.shape, dtype=ctx.dtype, device=gout.device)
        g32 = gout.detach().to(torch.float32).contiguous()
        call("cgan3d_fill", _p(gx), _dt(ctx.dtype), n, _p(g32), ctx.scale / n, _st())
        return gx, None


class GenLossFn(torch.autograd.Function):
    """One pass over (opt_hat, subopt, mask) producing w_sim*ZNCC and w_hu*HU
    (reference model/loss.py:11-71).  Returns a 2-vector [sim, hu]."""

    @staticmethod
    def forward(ctx, s, t, mask, lo: float, hi: float, w_sim: float, w_hu: float):
        _need_cuda(s, t)
        sc = s.detach().contiguous()
        tc = t.detach().contiguous()
        if sc.dtype != torch.float32 or tc.dtype != torch.float32:
            raise TypeError("generator losses take fp32 tensors")
        mk = None
        if mask is not None:
            mk = mask.detach().contiguous()
            if mk.dtype == torch.bool:
                mk = mk.view(torch.uint8)
            elif mk.dtype != torch.uint8:
                raise TypeError("mask must be bool or uint8")
            assert mk.numel() == sc.numel()
        n = sc.numel()
        dev = s.device
        sums = torch.empty(7, dtype=torch.float64, device=dev)
        out = torch.empty(2, dtype=torch.float32, device=dev)
        coef = torch.empty(8, dtype=torch.float32, device=dev)
        call("cgan3d_gen_loss_sums", _p(sc), _p(tc), _p(mk), n, float(lo), float(hi), _p(sums), _st())
        call("cgan3d_gen_loss_finalize", _p(sums), n, float(w_sim), float(w_hu), _p(out), _p(coef), _st())
        ctx.lo, ctx.hi = float(lo), float(hi)
        ctx.save_for_backward(sc, tc, mk, coef)
        return out

    @staticmethod
    def backward(ctx, gout):
        sc, tc, mk, coef = ctx.saved_tensors
        ds = torch.empty_like(sc)
        up = gout.detach().to(torch.float32).contiguous()
        call("cgan3d_gen_loss_backward", _p(sc), _p(tc), _p(mk), sc.numel(), ctx.lo, ctx.hi, _p(coef), _p(up), None,
             _p(ds), _st())
        return ds, None, None, None, None, None, None


def adam_step(p, g, m, v, lr, b1, b2, eps, step, clip=0.0):
    call("cgan3d_adam_step", _p(p), _p(g), _p(m), _p(v), p.numel(), float(lr), float(b1), float(b2), float(eps),
         int(step), float(clip), _st())


# ------------------------------------------------------------------------------------------
# Convolution primitives closed under differentiation (WGAN-GP: reference model/utils.py:12-41 differentiates the
# critic's input gradient once more; Trainer.py:122-133).  A convolution is bilinear in (input, filter); its three
# operators are each other's derivatives:
#     gather (x, w) -> y       d/dx = scatter(gy, w)    d/dw = wgrad(x, gy)
#     scatter(y, w) -> x       d/dy = gather (gx, w)    d/dw = wgrad(gx, y)
#     wgrad  (x, y) -> w       d/dx = scatter(y, gw)    d/dy = gather (x, gw)
# so every backward below is expressed through `.apply` of the other two and can itself be differentiated.
# x / y are channels-last activations in the compute dtype, w the fp32 master filter [Cs, Cb, k, k, k].
# ------------------------------------------------------------------------------------------
class ConvGatherFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, big, w, g: ConvGeom):
        _need_cuda(big, w)
        ctx.g, ctx.dtype = g, big.dtype
        ctx.save_for_backward(big, w)
        return conv_gather(g, big.contiguous(), pack_weights(w.float(), big.dtype))

    @staticmethod
    def backward(ctx, gsmall):
        big, w = ctx.saved_tensors
        gsmall = gsmall.to(ctx.dtype)
        dbig = ConvScatterFn.apply(gsmall, w, ctx.g) if ctx.needs_input_grad[0] else None
        dw = ConvWgradFn.apply(big, gsmall, ctx.g) if ctx.needs_input_grad[1] else None
        return dbig, dw, None


class ConvScatterFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, small, w, g: ConvGeom):
        _need_cuda(small, w)
        ctx.g, ctx.dtype = g, small.dtype
        ctx.save_for_backward(small, w)
        return conv_scatter(g, small.contiguous(), pack_weights(w.float(), small.dtype))

    @staticmethod
    def backward(ctx, gbig):
        small, w = ctx.saved_tensors
        gbig = gbig.to(ctx.dtype)
        dsmall = ConvGatherFn.apply(gbig, w, ctx.g) if ctx.needs_input_grad[0] else None
        dw = ConvWgradFn.apply(gbig, small, ctx.g) if ctx.needs_input_grad[1] else None
        return dsmall, dw, None


class ConvWgradFn(torch.autograd.Function):
    @staticmethod
    def forward(ctx, big, small, g: ConvGeom):
        _need_cuda(big, small)
        ctx.g = g
        ctx.save_for_backward(big, small)
        return conv_wgrad(g, big.contiguous(), small.contiguous())

    @staticmethod
    def backward(ctx, gw):
        big, small = ctx.saved_tensors
        dbig = ConvScatterFn.apply(small, gw, ctx.g) if ctx.needs_input_grad[0] else None
        dsmall = ConvGatherFn.apply(big, gw, ctx.g) if ctx.needs_input_grad[1] else None
        return dbig, dsmall, None


def conv_differentiable(x: torch.Tensor, weight: torch.Tensor, spec: ConvSpec, dtype: torch.dtype) -> torch.Tensor:
    """conv(x, weight) for a (non-transposed, zero-padded) layer through the twice-differentiable Functions."""
    if spec.transposed or spec.reflect:
        raise NotImplementedError("the twice-differentiable path covers the critic's zero-padded convolutions")
    B, X, Y, Z, Cin = x.shape
    assert Cin == spec.cin
    g, _ = spec.geometry(B, (X, Y, Z))
    return ConvGatherFn.apply(x.to(dtype), weight, g)
