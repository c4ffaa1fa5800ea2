"""Set-abstraction level op: ctypes mirror of ``b2pn_sa_args`` + the autograd bridge.

``sa_apply`` is what PyG's ``PointNetConv.propagate`` (message -> local_nn -> max aggregate) and
``global_max_pool(nn(cat[x,pos]))`` are in the reference (/root/reference/pointnet2_regressor.py:18,
:29-30): one call into libb2pn for the forward, one for the backward.
"""
from __future__ import annotations

import ctypes
import threading
from contextlib import contextmanager
from typing import List, Optional, Sequence

import torch

from . import _lib
from .optim import fresh_alias, grad_dst

PREC_F32, PREC_BF16 = 0, 1

# storage format of the FORWARD-domain 16-bit tensors of the tensor-core mode (weights, normalised activations, level
# outputs handed to the next level): fp16 -- 8x finer than bf16 on O(1) values, which the 2e-2 output tolerance needs at
# the reference's batch shape (tools/bf16_attribution.py); gradients stay bf16 inside libb2pn
H16 = torch.float16
SEG_SLOTS, SEG_CLOUDS = 0, 1
ACT_NONE, ACT_RELU = 0, 1

_vp = ctypes.c_void_p


Mlp3, SaArgs, SaGrads = _lib.Mlp3, _lib.SaArgs, _lib.SaGrads


def _dp(t: Optional[torch.Tensor]):
    return None if t is None else t.data_ptr()


# Per-call launch options of the set-abstraction kernels (b2pn_sa_args::sm_limit / ::deterministic).  They are fields of
# every call's argument struct -- libb2pn has no process-wide state.  On the Python side they live in a small holder
# object; every host thread has its own current holder, so the reference's thread-per-GPU callers
# (/root/reference/main.py:140) cannot disturb each other.  A forward call remembers the holder it ran under and its
# backward -- which autograd runs on ITS OWN thread -- reads the same holder at backward time, so a training loop can
# change an option between forward and backward, or in the middle of the backward pass (train.PipelinedTrainStep lifts
# the SM cap before the level-1 backward).
class LaunchOptions:
    __slots__ = ("sm_limit", "deterministic")

    def __init__(self, sm_limit: int = 0, deterministic: int = 0):
        self.sm_limit, self.deterministic = int(sm_limit), int(deterministic)


_tls = threading.local()


def current_options() -> LaunchOptions:
    """The holder the calling thread's next set-abstraction calls are issued with (created on first use)."""
    h = getattr(_tls, "holder", None)
    if h is None:
        h = _tls.holder = LaunchOptions()
    return h


def launch_options():
    """(sm_limit, deterministic) of the calling thread's current holder."""
    h = current_options()
    return h.sm_limit, h.deterministic


def set_sm_limit(n: int) -> None:
    """Cap the persistent tensor-core kernels launched by THIS thread's calls at ``n`` CTAs (0 = one per SM)."""
    if n < 0:
        raise ValueError("sm_limit must be >= 0")
    current_options().sm_limit = int(n)


def set_deterministic(on: bool) -> bool:
    """Fixed-order gradient reductions for the calls of THIS thread (forward AND their backward); returns the
    previous setting."""
    h = current_options()
    prev = bool(h.deterministic)
    h.deterministic = 1 if on else 0
    return prev


@contextmanager
def options(sm_limit: Optional[int] = None, deterministic: Optional[bool] = None):
    h = current_options()
    prev = (h.sm_limit, h.deterministic)
    try:
        if sm_limit is not None:
            set_sm_limit(sm_limit)
        if deterministic is not None:
            set_deterministic(deterministic)
        yield h
    finally:
        h.sm_limit, h.deterministic = prev


def act_code(act) -> int:
    if act is None:
        return ACT_NONE
    name = act if isinstance(act, str) else type(act).__name__
    if name.lower() == "relu":
        return ACT_RELU
    raise NotImplementedError(
        f"activation {act!r}: the B200 kernels implement ReLU (the only activation the reference trains with, "
        f"/root/reference/main.py:45) and None")


def _fill_args(a: SaArgs, *, precision, training, seg_mode, K, n_src, n_dst, c_in, x, pos_src, pos_dst, nbr, cnt,
               batch, chans, act, eps, momentum, ws, bs, gammas, betas, rmeans, rvars, nbts, out, arg, h1, h2, bn,
               rowmap=None, acts=None, out_bf16=None, holder=None):
    a.precision, a.training, a.seg_mode, a.K = precision, int(training), seg_mode, K
    h = holder if holder is not None else current_options()
    a.sm_limit, a.deterministic = h.sm_limit, h.deterministic
    a.out_bf16 = _dp(out_bf16)
    a.n_src, a.n_dst, a.c_in = n_src, n_dst, c_in
    a.x_dtype = 1 if (x is not None and x.dtype == H16) else 0
    a.x, a.pos_src, a.pos_dst = _dp(x), _dp(pos_src), _dp(pos_dst)
    a.nbr, a.cnt, a.batch = _dp(nbr), _dp(cnt), _dp(batch)
    m = a.mlp
    for i in range(4):
        m.c[i] = chans[i]
    m.act, m.eps, m.momentum = act, eps, momentum
    for i in range(3):
        m.w[i], m.b[i] = _dp(ws[i]), _dp(bs[i])
    for i in range(2):
        m.gamma[i], m.beta[i] = _dp(gammas[i]), _dp(betas[i])
        m.running_mean[i], m.running_var[i] = _dp(rmeans[i]), _dp(rvars[i])
        m.num_batches_tracked[i] = _dp(nbts[i])
    a.out, a.arg, a.h1, a.h2, a.bn = _dp(out), _dp(arg), _dp(h1), _dp(h2), _dp(bn)
    if rowmap is not None and rowmap[0] is None:      # CLOUDS levels: only the row-valid vector
        a.row_valid = _dp(rowmap[4])
    elif rowmap is not None:
        rgrp, row_src, num_rows, cap, row_valid = rowmap
        a.rgrp, a.row_src, a.num_rows, a.row_capacity = _dp(rgrp), _dp(row_src), _dp(num_rows), cap
        a.row_valid = _dp(row_valid)
    if acts is not None:
        a.a1, a.a2 = _dp(acts[0]), _dp(acts[1])
        a.g1 = _dp(acts[2]) if len(acts) > 2 else None


def pack_rows(nbr: torch.Tensor, cnt: torch.Tensor, K: int):
    """Compact the filled neighbour slots into rows for the tensor-core kernels (include/b2pn.h,
    b2pn_pack_rows): what ``radius`` returning a compact edge list is in the reference
    (/root/reference/pointnet2_regressor.py:14-16), minus the host round trip -- the row count stays on the
    device.  Returns (rgrp, row_src, num_rows, capacity, row_valid)."""
    lib = _lib.lib()
    dev = nbr.device
    n_dst = cnt.numel()
    cap = int(lib.b2pn_pack_rows_capacity(n_dst, K))
    if cap < 0:
        _lib.check(cap, "b2pn_pack_rows_capacity")
    rgrp = torch.empty(cap // 8, dtype=torch.int32, device=dev)
    row_src = torch.empty(cap, dtype=torch.int32, device=dev)
    num_rows = torch.empty(2, dtype=torch.int64, device=dev)
    row_valid = torch.empty(cap, dtype=torch.float16, device=dev)
    wsb = torch.empty(int(lib.b2pn_pack_rows_workspace_bytes(n_dst)), dtype=torch.uint8, device=dev)
    with torch.cuda.device(dev):
        rc = lib.b2pn_pack_rows(cnt.data_ptr(), nbr.data_ptr(), n_dst, K, rgrp.data_ptr(), row_src.data_ptr(),
                                row_valid.data_ptr(), num_rows.data_ptr(), wsb.data_ptr(), wsb.numel(),
                                torch.cuda.current_stream(dev).cuda_stream)
    _lib.check(rc, "b2pn_pack_rows")
    return rgrp, row_src, num_rows, cap, row_valid


def _l1_input(x: Optional[torch.Tensor], x_bf16: Optional[torch.Tensor] = None):
    """How the kernels take the level's input features: (tensor or None, c_in, image columns).  Raw low-dimensional
    inputs (e.g. lidar intensity) stay fp32 -- the kernels feed them to the tensor cores as bf16 hi+lo column pairs --
    wide feature maps from the previous level go in as fp16, the forward-domain operand format (``x_bf16``: the 16-bit
    copy the previous level's epilogue wrote, if there is one)."""
    c_in = 0 if x is None else x.shape[1]
    split = x is not None and x.dtype == torch.float32 and c_in <= 16
    if x is None:
        xs = None
    elif not split and x_bf16 is not None and x_bf16.shape == x.shape and x_bf16.dtype == H16:
        xs = x_bf16.contiguous()
    else:
        xs = x.detach().to(torch.float32 if split else H16).contiguous()
    return xs, c_in, (2 * c_in if split else c_in) + 6


_RV_CACHE: dict = {}


def _row_valid_clouds(ld: int, n_src: int, dev) -> torch.Tensor:
    """bf16 [ld]: 1 on the n_src real rows of a CLOUDS level (the "ones" operand line of its dW GEMMs).  Read-only and
    a function of two integers: built once per shape."""
    key = (int(ld), int(n_src), str(dev))
    rv = _RV_CACHE.get(key)
    if rv is None:
        if len(_RV_CACHE) >= 64:
            _RV_CACHE.pop(next(iter(_RV_CACHE)))
        rv = torch.zeros(ld, dtype=H16, device=dev)
        rv[:n_src] = 1
        _RV_CACHE[key] = rv
    return rv


def gather_rows(x: Optional[torch.Tensor], pos_src: torch.Tensor, pos_dst: torch.Tensor, K: int, rowmap):
    """The gathered + concatenated layer-1 operand of a SLOTS level (include/b2pn.h, b2pn_sa_gather_rows) for the
    compacted rows ``rowmap``; None when the level is too wide to take one.  Needs no weights, so it can be built
    ahead of the forward pass; hand it to ``sa_apply(..., l1op=...)``."""
    lib = _lib.lib()
    xs, c_in, k_img = _l1_input(x)
    if k_img + 16 > 256:
        return None
    rgrp, row_src, num_rows, cap, row_valid = rowmap
    ld = (cap + 127) // 128 * 128
    dev = pos_src.device
    g = torch.empty(k_img + 1, ld, dtype=H16, device=dev)
    a = SaArgs()
    a.precision, a.seg_mode, a.K = PREC_BF16, SEG_SLOTS, K
    a.n_src, a.n_dst, a.c_in = pos_src.shape[0], pos_dst.shape[0], c_in
    a.x_dtype = 1 if (xs is not None and xs.dtype == H16) else 0
    a.x, a.pos_src, a.pos_dst = _dp(xs), _dp(pos_src.contiguous()), _dp(pos_dst)
    a.mlp.c[0] = c_in + 3
    a.rgrp, a.row_src, a.num_rows, a.row_capacity = _dp(rgrp), _dp(row_src), _dp(num_rows), cap
    a.g1 = g.data_ptr()
    with torch.cuda.device(dev):
        rc = lib.b2pn_sa_gather_rows(ctypes.byref(a), torch.cuda.current_stream(dev).cuda_stream)
    _lib.check(rc, "b2pn_sa_gather_rows")
    return g


class _SAFunction(torch.autograd.Function):
    """forward/backward of one set-abstraction level through libb2pn."""

    @staticmethod
    def forward(ctx, cfg, rowmap_in, l1op_in, extra, x, pos_src, pos_dst, nbr, cnt, batch, w1, b1, g1, be1, w2, b2, g2, be2,
                w3, b3, rm1, rv1, nbt1, rm2, rv2, nbt2):
        lib = _lib.lib()
        ctx.set_materialize_grads(False)  # no zero-filled gradient tensors for the index / bf16 side outputs
        grad_dsts, x_bf16, want_bf16_out, needs_bwd = extra
        dev = pos_src.device
        if not pos_src.is_cuda:
            raise RuntimeError("b2pn set abstraction runs on a B200 only: there is no CPU fallback")
        prec, training, seg_mode, K, n_dst, act, eps, momentum = cfg
        f32 = torch.float32
        ws = [w.detach().to(f32).contiguous() for w in (w1, w2, w3)]
        bs = [b.detach().to(f32).contiguous() for b in (b1, b2, b3)]
        gs = [g.detach().contiguous() for g in (g1, g2)]
        bes = [b.detach().contiguous() for b in (be1, be2)]
        chans = [ws[0].shape[1], ws[0].shape[0], ws[1].shape[0], ws[2].shape[0]]
        c_in = 0 if x is None else x.shape[1]
        if chans[0] != c_in + 3:
            raise ValueError(f"MLP expects {chans[0]} input channels, got {c_in} features + 3")
        pos_src = pos_src.contiguous()
        n_src = pos_src.shape[0]
        rows = n_src if seg_mode == SEG_CLOUDS else n_dst * K
        rowmap = None
        if prec == PREC_BF16 and seg_mode == SEG_SLOTS:
            rowmap = rowmap_in if rowmap_in is not None else pack_rows(nbr, cnt, K)
            rows = rowmap[3]
        out = torch.empty(n_dst, chans[3], dtype=f32, device=dev)
        arg = torch.empty(n_dst, chans[3], dtype=torch.int32, device=dev)
        out_bf16 = (torch.empty(n_dst, chans[3], dtype=H16, device=dev)
                    if (want_bf16_out and prec == PREC_BF16) else None)
        acts = None
        # evaluation without a backward pass to follow: one launch per level, no hidden activation stored (sa_chain.cuh)
        fused_eval = False
        if prec == PREC_BF16 and seg_mode == SEG_SLOTS and not training and not needs_bwd:
            probe = SaArgs()
            probe.precision, probe.training, probe.seg_mode, probe.K, probe.c_in = prec, 0, seg_mode, K, c_in
            probe.x_dtype = 0 if (x is not None and x.dtype == f32 and c_in <= 16) else 1
            for i in range(4):
                probe.mlp.c[i] = chans[i]
            fused_eval = lib.b2pn_sa_eval_fused(ctypes.byref(probe)) == 1
        if fused_eval:
            xs, _, _ = _l1_input(x, x_bf16)
            h1 = h2 = None
            arg = torch.empty(0, dtype=torch.int32, device=dev)   # no backward will follow: arg-max slots not recorded
        elif prec == PREC_F32:   # row-major fp32 activations [rows, c]
            xs = None if x is None else x.detach().to(f32).contiguous()
            h1 = torch.empty(rows, chans[1], dtype=f32, device=dev)
            h2 = torch.empty(rows, chans[2], dtype=f32, device=dev)
        else:                  # feature-major bf16 activations [c, ld], ld = rows rounded up to whole 128-row tiles
            xs, _, k_img = _l1_input(x, x_bf16)
            ld = (rows + 127) // 128 * 128
            h1 = torch.empty(chans[1], ld, dtype=H16, device=dev)
            h2 = torch.empty(chans[2], ld, dtype=H16, device=dev)
            acts = [torch.empty_like(h1), torch.empty_like(h2)]   # post-activation copies (TMA operands)
            if seg_mode == SEG_CLOUDS:   # the "ones" operand line of the dW GEMMs: 1 on every real row
                rowmap = (None, None, None, 0, _row_valid_clouds(ld, n_src, dev))
            if seg_mode == SEG_SLOTS and k_img + 16 <= 256:   # gathered layer-1 operand incl. its ones line
                if l1op_in is not None and tuple(l1op_in.shape) != (k_img + 1, ld):
                    raise ValueError("l1op does not belong to these rows / features")
                acts.append(l1op_in if l1op_in is not None else
                            torch.empty(k_img + 1, ld, dtype=H16, device=dev))
            else:
                l1op_in = None
            acts = tuple(acts)
        cmax = max(chans[1], chans[2])
        bn = None if fused_eval else torch.empty(2, 4, cmax, dtype=f32, device=dev)
        a = SaArgs()
        _fill_args(a, precision=prec, training=training, seg_mode=seg_mode, K=K, n_src=n_src, n_dst=n_dst, c_in=c_in,
                   x=xs, pos_src=pos_src, pos_dst=pos_dst, nbr=nbr, cnt=cnt, batch=batch, chans=chans, act=act,
                   eps=eps, momentum=momentum, ws=ws, bs=bs, gammas=gs, betas=bes, rmeans=(rm1, rm2),
                   rvars=(rv1, rv2), nbts=(nbt1, nbt2), out=out, arg=None if fused_eval else arg, h1=h1, h2=h2, bn=bn,
                   rowmap=rowmap, acts=acts, out_bf16=out_bf16)
        a.g1_ready = 1 if (prec == PREC_BF16 and l1op_in is not None) else 0
        nbytes = lib.b2pn_sa_workspace_bytes(ctypes.byref(a), 0)
        if nbytes < 0:
            _lib.check(int(nbytes), "b2pn_sa_workspace_bytes")
        wsb = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=dev)
        a.workspace, a.workspace_bytes = wsb.data_ptr(), wsb.numel()
        with torch.cuda.device(dev):
            rc = lib.b2pn_sa_forward(ctypes.byref(a), torch.cuda.current_stream(dev).cuda_stream)
        _lib.check(rc, "b2pn_sa_forward")
        ctx.cfg = cfg
        ctx.chans = chans
        ctx.c_in = c_in
        ctx.has_x = x is not None
        ctx.x_needs_grad = x is not None and x.requires_grad
        ctx.row_capacity = None if rowmap is None else rowmap[3]
        ctx.grad_dsts = grad_dsts
        ctx.holder = current_options()   # backward runs on autograd's thread: it reads THIS holder, at backward time
        rmt = (None, None, None, None) if rowmap is None else (rowmap[0], rowmap[1], rowmap[2], rowmap[4])
        at = (None, None, None) if acts is None else (acts + (None,))[:3]
        ctx.save_for_backward(xs, pos_src, pos_dst, nbr, cnt, batch, *ws, *bs, *gs, *bes, rm1, rv1, rm2, rv2,
                              arg, h1, h2, bn, *rmt, *at)
        if out_bf16 is None:
            ctx.mark_non_differentiable(arg)
            return out, arg, None
        ctx.mark_non_differentiable(arg, out_bf16)
        return out, arg, out_bf16

    @staticmethod
    @torch.autograd.function.once_differentiable
    def backward(ctx, grad_out, _grad_arg=None, _grad_bf16=None):
        lib = _lib.lib()
        (xs, pos_src, pos_dst, nbr, cnt, batch, w1, w2, w3, b1, b2, b3, g1, g2, be1, be2, rm1, rv1, rm2, rv2,
         arg, h1, h2, bn, rgrp, row_src, num_rows, row_valid, a1, a2, l1op) = ctx.saved_tensors
        rowmap = None if (rgrp is None and row_valid is None) else (rgrp, row_src, num_rows, ctx.row_capacity, row_valid)
        acts = None if (a1 is None and l1op is None) else ((a1, a2) if l1op is None else (a1, a2, l1op))
        prec, training, seg_mode, K, n_dst, act, eps, momentum = ctx.cfg
        dev = pos_src.device
        chans = ctx.chans
        f32 = torch.float32
        grad_out = grad_out.to(f32).contiguous()
        # gradients land where the parameter arena wants them (optim.ParamArena) or in fresh tensors
        d = ctx.grad_dsts if ctx.grad_dsts is not None else (None,) * 10
        fresh = lambda dst, like: fresh_alias(dst) if dst is not None else torch.empty_like(like)  # noqa: E731
        gw = [fresh(d[0], w1), fresh(d[4], w2), fresh(d[8], w3)]
        gb = [fresh(d[1], b1), fresh(d[5], b2), fresh(d[9], b3)]
        gg = [fresh(d[2], g1), fresh(d[6], g2)]
        gbe = [fresh(d[3], be1), fresh(d[7], be2)]
        # (the tensor-core path clears its scatter-add target itself: a memset node, not an ATen kernel)
        gx = ((torch.empty if prec == PREC_BF16 else torch.zeros)(xs.shape, dtype=f32, device=dev)
              if ctx.x_needs_grad else None)
        a = SaArgs()
        _fill_args(a, precision=prec, training=training, seg_mode=seg_mode, K=K, n_src=pos_src.shape[0], n_dst=n_dst,
                   c_in=ctx.c_in, x=xs, pos_src=pos_src, pos_dst=pos_dst, nbr=nbr, cnt=cnt, batch=batch, chans=chans,
                   act=act, eps=eps, momentum=momentum, ws=(w1, w2, w3), bs=(b1, b2, b3), gammas=(g1, g2),
                   betas=(be1, be2), rmeans=(rm1, rm2), rvars=(rv1, rv2), nbts=(None, None), out=grad_out, arg=arg,
                   h1=h1, h2=h2, bn=bn, rowmap=rowmap, acts=acts, holder=ctx.holder)
        nbytes = lib.b2pn_sa_workspace_bytes(ctypes.byref(a), 1)
        if nbytes < 0:
            _lib.check(int(nbytes), "b2pn_sa_workspace_bytes")
        wsb = torch.empty(max(int(nbytes), 256), dtype=torch.uint8, device=dev)
        a.workspace, a.workspace_bytes = wsb.data_ptr(), wsb.numel()
        g = SaGrads()
        g.grad_out = grad_out.data_ptr()
        for i in range(3):
            g.grad_w[i], g.grad_b[i] = gw[i].data_ptr(), gb[i].data_ptr()
        for i in range(2):
            g.grad_gamma[i], g.grad_beta[i] = gg[i].data_ptr(), gbe[i].data_ptr()
        g.grad_x = _dp(gx)
        with torch.cuda.device(dev):
            rc = lib.b2pn_sa_backward(ctypes.byref(a), ctypes.byref(g), torch.cuda.current_stream(dev).cuda_stream)
        _lib.check(rc, "b2pn_sa_backward")
        return (None, None, None, None, gx, None, None, None, None, None, gw[0], gb[0], gg[0], gbe[0], gw[1], gb[1], gg[1],
                gbe[1], gw[2], gb[2], None, None, None, None, None, None)


def sa_apply(mlp, x, pos_src, pos_dst, nbr, cnt, batch, *, seg_mode: int, K: int, n_dst: int, precision: int,
             rowmap=None, l1op=None, x_bf16=None, want_bf16_out: bool = False):
    """Run one set-abstraction level with the parameters of ``mlp`` (a b2pn ``MLP`` of three Linear layers).
    ``rowmap`` / ``l1op``: the results of ``pack_rows(nbr, cnt, K)`` and ``gather_rows(x, ...)`` if the caller already
    has them (bf16 path; ``l1op`` must have been built from this very ``x``).  ``x_bf16``: a bf16 copy of ``x`` the
    previous level's epilogue already wrote (saves the cast); ``want_bf16_out``: have this level write one too.
    Returns (out, arg), or (out, arg, out_bf16 or None) with ``want_bf16_out``."""
    if len(mlp.lins) != 3 or len(mlp.norms) != 2:
        raise NotImplementedError("set-abstraction kernels are built for the reference's 3-layer MLPs with BatchNorm")
    if mlp.dropout != 0.0 and mlp.training:
        raise NotImplementedError("dropout inside set-abstraction MLPs is not used by the reference")
    n0, n1 = mlp.norms
    cfg = (precision, bool(mlp.training), seg_mode, K, n_dst, act_code(mlp.act_name), float(n0.eps),
           float(n0.momentum if n0.momentum is not None else 0.1))
    l0, l1, l2 = mlp.lins
    params = (l0.weight, l0.bias, n0.weight, n0.bias, l1.weight, l1.bias, n1.weight, n1.bias, l2.weight, l2.bias)
    dsts = tuple(grad_dst(p) for p in params) if torch.is_grad_enabled() else None
    if dsts is not None and all(t is None for t in dsts):
        dsts = None
    # (inside Function.forward grad mode is always off and needs_input_grad ignores it: decide here)
    needs_bwd = torch.is_grad_enabled() and (any(p.requires_grad for p in params) or (x is not None and x.requires_grad))
    extra = (dsts, x_bf16, bool(want_bf16_out), needs_bwd)
    res = _SAFunction.apply(cfg, rowmap, l1op if rowmap is not None else None, extra, x, pos_src, pos_dst, nbr, cnt, batch,
                            *params, n0.running_mean, n0.running_var, n0.num_batches_tracked,
                            n1.running_mean, n1.running_var, n1.num_batches_tracked)
    return res if want_bf16_out else res[:2]


def bf16_available() -> bool:
    """True once libb2pn implements forward AND backward of the set-abstraction levels on tcgen05."""
    a = SaArgs()
    a.precision = PREC_BF16
    a.seg_mode = SEG_SLOTS
    a.K = 64
    a.n_src = a.n_dst = 1
    a.c_in = 1
    a.row_capacity = 128
    for i, c in enumerate((4, 64, 64, 128)):
        a.mlp.c[i] = c
    return _lib.lib().b2pn_sa_workspace_bytes(ctypes.byref(a), 1) > 0
