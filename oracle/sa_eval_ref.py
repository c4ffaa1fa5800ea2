"""Float64 reference of the EVALUATION forward of one set-abstraction level and of the regression head -- TEST
INFRASTRUCTURE, NOT PRODUCT CODE.

Evaluation makes no decision worth pinning: ReLU and max are continuous, so a rounding that flips either moves an
output by at most about one fp16 ulp of an intermediate times a weight.  The level is therefore recomputed from its
INPUTS (x, positions, nbr / cnt or batch, parameters, running statistics), with each rounding point of the 16-bit
kernels on its own switch (``EvalRounding``) and the two ways the kernels apply an evaluation-mode BatchNorm:

* ``bn="fused"``: the single-launch evaluation kernel (csrc/sa_chain.cuh, chain_affine) folds it into one multiply-add,
  ``a = fp16(act(acc * scale + shift))`` with ``scale = gamma * rstd`` and ``shift = (b - mean) * scale + beta``;
  zhat is never formed.
* ``bn="multipass"``: the multi-pass kernels (csrc/sa_tc.cu, NormStoreEpTC) store ``zhat = fp16((acc + b - mean) *
  rstd)`` first and form ``a = fp16(act(gamma * zhat + beta))`` from the STORED zhat.

Layer 3 adds its bias, the max runs over the valid rows of each target (a target without rows gives 0, as PyG's max
aggregation of no messages), and ``out16 = fp16(out)`` is the copy the next level reads.  The SLOTS row order is that
of b2pn_pack_rows (``sa_pinned.pack_rows_cpu``).

``FAULTS`` E1-E7 are one-line mistakes a kernel could plausibly make; ``fault=`` injects one.

Pure CPU torch; nothing here imports the package it checks.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict, Optional

import torch

from oracle import sa_pinned as sp

F64 = torch.float64
f16, bf16, ulp16 = sp.f16, sp.bf16, sp.ulp16

FAULTS = {
    "E1": "the last valid row of each target left out of the max",
    "E2": "the layer-3 bias missing",
    "E3": "the hi + lo split lost (fp16 hi only)",
    "E4": "weight images in bf16 instead of fp16",
    "E5": "the BatchNorm fold without the linear bias (shift = beta - mean * scale)",
    "E6": "the first row of the next target leaking into the max",
    "E7": "out16 rounded to bf16",
}

# bounds of tests/test_sa_eval_gpu.py (kernel vs this reference, every rounding emulated): a level's out in fp16 ulps of
# the reference (ulp_err), as max-abs error over max |want| (rel_err) and as rms error over rms |want| (rms_err); the head
# against float64 as max-abs over max |want|.  ~4x the worst value measured on a B200 (DESIGN.md section 2)
GPU_TOL = {"out_ulp": 48.0, "out_rel": 2e-3, "out_rms": 2e-4, "head_rel": 4e-6}
# the bounds the evaluation path had before: 2e-2 against the fp32 oracle, 5e-3 single-launch vs multi-pass kernels
OLD_TOL = {"vs_fp32": 2e-2, "fused_vs_multipass": 5e-3}


@dataclass(frozen=True)
class EvalRounding:
    """The rounding points of the 16-bit evaluation forward; each can be switched off."""
    w16: bool = True     # fp16 weight images of the three GEMMs
    split: bool = True   # fp32 x (c_in <= 16) and the relative positions as fp16 hi + lo column pairs
    x16: bool = True     # any other fp32 x enters as fp16 (sa._l1_input); fp16 x (the x_bf16 hand-over) is exact
    act16: bool = True   # the fp16 activation operand between layers (multi-pass: zhat too)


ROUND_ALL = EvalRounding()
ROUND_NONE = EvalRounding(False, False, False, False)


def params_of(mlp) -> Dict[str, torch.Tensor]:
    """The parameters and running statistics of a three-layer MLP (``lins`` / ``norms``) as float64 CPU tensors."""
    p = {}
    for i, lin in enumerate(mlp.lins):
        p[f"w{i + 1}"] = lin.weight.detach().cpu().to(F64)
        p[f"b{i + 1}"] = lin.bias.detach().cpu().to(F64)
    for i, n in enumerate(mlp.norms):
        p[f"gamma{i + 1}"] = n.weight.detach().cpu().to(F64)
        p[f"beta{i + 1}"] = n.bias.detach().cpu().to(F64)
        p[f"rm{i + 1}"] = n.running_mean.detach().cpu().to(F64)
        p[f"rv{i + 1}"] = n.running_var.detach().cpu().to(F64)
        p["eps"] = float(n.eps)
    return p


class Rows:
    """The valid rows of a level in kernel row order: target, slot (SLOTS) and source point of each."""

    def __init__(self, n_dst: int, nbr=None, cnt=None, batch=None):
        self.slots = batch is None
        if self.slots:
            K = nbr.shape[1]
            rgrp, row_src, num_rows, _ = sp.pack_rows_cpu(cnt.cpu(), nbr.cpu())
            lay = sp.Layout({"rgrp": rgrp, "row_src": row_src, "num_rows": num_rows}, n_dst, K)
            self.cent, self.src, self.slot = lay.cent, lay.src, lay.slot
        else:
            self.cent = batch.cpu().to(torch.int64)
            self.src = torch.arange(self.cent.numel())
            self.slot = self.src
        self.n_dst = n_dst


def _split(v: torch.Tensor, rnd: EvalRounding, fault) -> torch.Tensor:
    """hi + lo as the GEMM sees a split column (the difference taken in v's own precision)."""
    if fault == "E3":
        return v.to(torch.float16).to(F64)
    hi, lo = sp._split_parts(v, "f16", rnd.split)
    return hi + lo


def layer1_input(x, pos_src, pos_dst, rows: Rows, rnd: EvalRounding = ROUND_ALL, fault=None) -> torch.Tensor:
    """[valid rows, c_in + 3]: [x_j | pos_j - pos_i] as the first GEMM sees it.  x as the kernel receives it: fp32 with
    c_in <= 16 is split, fp16 (the previous level's hand-over) is exact, any other fp32 is rounded to fp16."""
    d = pos_src.cpu()[rows.src] - (pos_dst.cpu()[rows.cent] if rows.slots else 0)
    dpos = _split(d, rnd, fault)
    if x is None or x.shape[1] == 0:
        return dpos
    xv = x.cpu()[rows.src]
    if xv.dtype == torch.float16:
        xv = xv.to(F64)
    elif x.shape[1] <= 16:
        xv = _split(xv, rnd, fault)
    else:
        xv = f16(xv) if rnd.x16 else xv.to(F64)
    return torch.cat([xv, dpos], 1)


def _segment_max(v: torch.Tensor, members: torch.Tensor, targets: torch.Tensor, n_dst: int) -> torch.Tensor:
    """max over the (row, target) pairs; a target without rows gives 0."""
    C = v.shape[1]
    out = torch.zeros(n_dst, C, dtype=F64)
    if members.numel():
        idx = targets[:, None].expand(-1, C)
        mx = torch.full((n_dst, C), float("-inf"), dtype=F64).scatter_reduce(0, idx, v[members], "amax")
        has = torch.zeros(n_dst, dtype=torch.bool)
        has[targets] = True
        out = torch.where(has[:, None], mx, out)
    return out


def eval_level(x, pos_src, params: Dict[str, torch.Tensor], rows: Rows, *, pos_dst=None, bn: str = "fused",
               relu: bool = True, rnd: EvalRounding = ROUND_ALL, fault: Optional[str] = None) -> Dict[str, torch.Tensor]:
    """Evaluation forward of one level.  Returns float64 ``out`` [n_dst, c3], ``out16`` (its 16-bit copy), the per-row
    layer-3 values ``v3`` and the activations ``a1`` / ``a2`` of the valid rows."""
    assert bn in ("fused", "multipass")
    assert fault is None or fault in FAULTS, fault
    w = (bf16 if fault == "E4" else f16) if (rnd.w16 or fault == "E4") else (lambda t: t.to(F64))
    q = f16 if rnd.act16 else (lambda t: t)
    act = (lambda t: t.clamp_min(0)) if relu else (lambda t: t)
    eps = params.get("eps", 1e-5)
    X = layer1_input(x, pos_src, pos_dst, rows, rnd, fault)
    res = {}
    for l in (1, 2):
        acc = X @ w(params[f"w{l}"]).t()
        mean, rstd = params[f"rm{l}"], 1.0 / torch.sqrt(params[f"rv{l}"] + eps)
        g, be = params[f"gamma{l}"], params[f"beta{l}"]
        b = torch.zeros_like(mean) if fault == "E5" else params[f"b{l}"]
        if bn == "fused":
            scale = g * rstd
            X = q(act(acc * scale + ((b - mean) * scale + be)))
        else:
            z = q((acc + b - mean) * rstd)
            X = q(act(g * z + be))
        res[f"a{l}"] = X
    v3 = X @ w(params["w3"]).t()
    if fault != "E2":
        v3 = v3 + params["b3"]
    res["v3"] = v3
    # (row, target) pairs of the max
    n = rows.cent.numel()
    members, targets = torch.arange(n), rows.cent
    if n and fault in ("E1", "E6"):
        first = torch.full((rows.n_dst,), -1, dtype=torch.int64)
        last = torch.full((rows.n_dst,), -1, dtype=torch.int64)
        first.scatter_reduce_(0, rows.cent, torch.arange(n), "amin", include_self=False)
        last.scatter_reduce_(0, rows.cent, torch.arange(n), "amax", include_self=False)
        if fault == "E1":
            keep = torch.ones(n, dtype=torch.bool)
            keep[last[last >= 0]] = False
            members, targets = members[keep], targets[keep]
        else:
            nxt = torch.cat([first[1:], torch.full((1,), -1, dtype=torch.int64)])
            m = torch.nonzero((first >= 0) & (nxt >= 0)).flatten()
            members, targets = torch.cat([members, nxt[m]]), torch.cat([targets, m])
    out = _segment_max(v3, members, targets, rows.n_dst)
    res["out"] = out
    res["out16"] = bf16(out) if fault == "E7" else f16(out)
    return res


def eval_head(x, params: Dict[str, torch.Tensor]) -> torch.Tensor:
    """The regression head in evaluation: Linear -> BatchNorm (running statistics) -> Linear -> BatchNorm -> Linear,
    no activation (the reference head's act=None), float64."""
    eps = params.get("eps", 1e-5)
    h = x.cpu().to(F64)
    for l in (1, 2):
        h = h @ params[f"w{l}"].t() + params[f"b{l}"]
        h = (h - params[f"rm{l}"]) / torch.sqrt(params[f"rv{l}"] + eps) * params[f"gamma{l}"] + params[f"beta{l}"]
    return h @ params["w3"].t() + params["b3"]


def ulp_err(got: torch.Tensor, want: torch.Tensor) -> float:
    """max |got - want| in fp16 ulps of want.  The ulp is floored at that of 1/16 of max |want|: a one-ulp flip of a
    16-bit activation moves every output of its target by the same absolute amount, so outputs near 0 carry the
    absolute noise of the level's scale."""
    got, want = got.detach().cpu().to(F64), want.detach().cpu().to(F64)
    if not want.numel():
        return 0.0
    floor = max(float(want.abs().max()) / 16, 2.0 ** -24)
    return float(((got - want).abs() / ulp16(want.abs().clamp_min(floor))).max())


def rel_err(got: torch.Tensor, want: torch.Tensor) -> float:
    """max |got - want| over max |want|."""
    got, want = got.detach().cpu().to(F64), want.detach().cpu().to(F64)
    if not want.numel():
        return 0.0
    return float((got - want).abs().max()) / max(float(want.abs().max()), 1e-300)


def rms_err(got: torch.Tensor, want: torch.Tensor) -> float:
    """rms |got - want| over rms |want|: small for the rare rounding flips of a correct kernel, not for a fault that
    moves every output a little (E3)."""
    got, want = got.detach().cpu().to(F64), want.detach().cpu().to(F64)
    if not want.numel():
        return 0.0
    return float((got - want).pow(2).mean().sqrt()) / max(float(want.pow(2).mean().sqrt()), 1e-300)
