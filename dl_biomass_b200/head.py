"""Regression head: ``MLP([1024, 128, 128, 4], act=None, dropout=p)`` of the reference
(/root/reference/pointnet2_regressor.py:50,58) through libb2pn's two fused kernels (csrc/head.cu) instead of ~60 ATen
launches.  ``head_apply(mlp, x)`` takes the same parameter container (``pointnet2_regressor.MLP``) the rest of the
model uses, so state_dict keys and optimiser state are untouched."""
from __future__ import annotations

import ctypes

import torch

from . import _lib
from .optim import fresh_alias, grad_dst

MAX_ROWS, MAX_HIDDEN, MAX_OUT = 32, 256, 8


def supported(mlp, x: torch.Tensor) -> bool:
    """Shapes the fused kernels cover: the reference head (3 Linear layers, BatchNorm, no activation) on <= 32 rows."""
    if not x.is_cuda or x.dim() != 2 or x.dtype != torch.float32:
        return False
    if len(mlp.lins) != 3 or len(mlp.norms) != 2 or mlp.act_name is not None:
        return False
    c = mlp.channel_list
    # evaluation mode normalises with the running statistics, i.e. row by row: any number of clouds goes through in
    # chunks of MAX_ROWS (the reference evaluates its whole test set as one batch, testing_model.py:56); training mode
    # needs the batch statistics of all rows in one CTA
    rows_ok = 0 < x.size(0) <= MAX_ROWS or (x.size(0) > 0 and not mlp.training)
    return rows_ok and c[1] <= MAX_HIDDEN and c[2] <= MAX_HIDDEN and c[3] <= MAX_OUT


def _fill(a, x, mlp, training, p, out, saved, seed, counter):
    c = mlp.channel_list
    a.B = x.size(0)
    for i in range(4):
        a.c[i] = c[i]
    n0 = mlp.norms[0]
    a.training, a.p, a.eps = int(training), float(p if training else 0.0), float(n0.eps)
    a.momentum = float(n0.momentum if n0.momentum is not None else 0.1)
    a.x = x.data_ptr()
    for i, lin in enumerate(mlp.lins):
        a.w[i], a.b[i] = lin.weight.data_ptr(), lin.bias.data_ptr()
    for i, n in enumerate(mlp.norms):
        a.gamma[i], a.beta[i] = n.weight.data_ptr(), n.bias.data_ptr()
        a.running_mean[i], a.running_var[i] = n.running_mean.data_ptr(), n.running_var.data_ptr()
        a.num_batches_tracked[i] = n.num_batches_tracked.data_ptr()
    a.seed = int(seed)
    a.rng_counter = None if counter is None else counter.data_ptr()
    a.out = None if out is None else out.data_ptr()
    xh1, xh2, m1, m2, r1, r2 = saved
    a.xhat[0], a.xhat[1] = xh1.data_ptr(), xh2.data_ptr()
    a.mask[0], a.mask[1] = m1.data_ptr(), m2.data_ptr()
    a.rstd[0], a.rstd[1] = r1.data_ptr(), r2.data_ptr()


class _HeadFunction(torch.autograd.Function):
    @staticmethod
    def forward(ctx, mlp, training, p, seed, counter, x, *params):
        lib = _lib.lib()
        ctx.grad_dsts = tuple(grad_dst(t) for t in params)
        for t in params:
            if not (t.is_contiguous() and t.dtype == torch.float32):
                raise ValueError("head parameters must be contiguous float32 tensors")
        x = x.contiguous()
        dev, B, c = x.device, x.size(0), mlp.channel_list
        out = torch.empty(B, c[3], dtype=torch.float32, device=dev)
        saved = (torch.empty(B, c[1], device=dev), torch.empty(B, c[2], device=dev),
                 torch.empty(B, c[1], dtype=torch.uint8, device=dev), torch.empty(B, c[2], dtype=torch.uint8, device=dev),
                 torch.empty(c[1], device=dev), torch.empty(c[2], device=dev))
        a = _lib.HeadArgs()
        _fill(a, x, mlp, training, p, out, saved, seed, counter)
        with torch.cuda.device(dev):
            rc = lib.b2pn_head_forward(ctypes.byref(a), torch.cuda.current_stream(dev).cuda_stream)
        _lib.check(rc, "b2pn_head_forward")
        ctx.mlp, ctx.training, ctx.p, ctx.seed = mlp, training, p, seed
        ctx.save_for_backward(x, *saved)
        return out

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_out):
        lib = _lib.lib()
        x, *saved = ctx.saved_tensors
        mlp = ctx.mlp
        dev = x.device
        grad_out = grad_out.contiguous().to(torch.float32)
        a = _lib.HeadArgs()
        _fill(a, x, mlp, ctx.training, ctx.p, None, saved, ctx.seed, None)
        g = _lib.HeadGrads()
        g.grad_out = grad_out.data_ptr()
        gx = torch.empty_like(x) if ctx.needs_input_grad[5] else None
        g.grad_x = None if gx is None else gx.data_ptr()
        # parameter order of forward: w0 b0 g0 be0 w1 b1 g1 be1 w2 b2; gradients land in the parameter arena when
        # there is one (optim.ParamArena), else in fresh tensors
        d = ctx.grad_dsts
        fresh = lambda dst, like: fresh_alias(dst) if dst is not None else torch.empty_like(like)  # noqa: E731
        gw = [fresh(d[0], mlp.lins[0].weight), fresh(d[4], mlp.lins[1].weight), fresh(d[8], mlp.lins[2].weight)]
        gb = [fresh(d[1], mlp.lins[0].bias), fresh(d[5], mlp.lins[1].bias), fresh(d[9], mlp.lins[2].bias)]
        gg = [fresh(d[2], mlp.norms[0].weight), fresh(d[6], mlp.norms[1].weight)]
        gbe = [fresh(d[3], mlp.norms[0].bias), fresh(d[7], mlp.norms[1].bias)]
        for i in range(3):
            g.grad_w[i], g.grad_b[i] = gw[i].data_ptr(), gb[i].data_ptr()
        for i in range(2):
            g.grad_gamma[i], g.grad_beta[i] = gg[i].data_ptr(), gbe[i].data_ptr()
        with torch.cuda.device(dev):
            rc = lib.b2pn_head_backward(ctypes.byref(a), ctypes.byref(g), torch.cuda.current_stream(dev).cuda_stream)
        _lib.check(rc, "b2pn_head_backward")
        # parameter order of forward: w0 b0 g0 be0 w1 b1 g1 be1 w2 b2
        return (None, None, None, None, None, gx, gw[0], gb[0], gg[0], gbe[0], gw[1], gb[1], gg[1], gbe[1], gw[2], gb[2])


def head_apply(mlp, x: torch.Tensor, counter: torch.Tensor, seed: int) -> torch.Tensor:
    """``mlp(x)`` through the fused kernels.  ``counter``: int64 device scalar owned by the caller (dropout noise index,
    bumped by every training forward); ``seed``: per-model constant."""
    l0, l1, l2 = mlp.lins
    n0, n1 = mlp.norms
    params = (l0.weight, l0.bias, n0.weight, n0.bias, l1.weight, l1.bias, n1.weight, n1.bias, l2.weight, l2.bias)
    if mlp.training and x.size(0) < 2:   # as torch's BatchNorm1d: one row has no batch variance to normalise with
        raise ValueError(f"Expected more than 1 value per channel when training, got input size {tuple(x.shape)}")
    if x.size(0) > MAX_ROWS:
        if mlp.training:
            raise ValueError(f"the fused head trains on at most {MAX_ROWS} clouds per batch")
        outs = [_HeadFunction.apply(mlp, False, 0.0, int(seed), counter, x[i:i + MAX_ROWS], *params)
                for i in range(0, x.size(0), MAX_ROWS)]
        return torch.cat(outs, 0)
    return _HeadFunction.apply(mlp, bool(mlp.training), float(mlp.dropout), int(seed), counter, x, *params)
