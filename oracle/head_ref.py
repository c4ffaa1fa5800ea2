"""Float64 reference of the regression head in training mode -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

``MLP([c0, c1, c2, c3], act=None, dropout=p)``: Lin -> BatchNorm1d (batch statistics) -> dropout -> Lin ->
BatchNorm1d -> dropout -> Lin, and its backward written out by hand, so that single terms can be left out (faults
H1-H4).  Dropout replays the keep-masks the kernel saved; a kept value is scaled by 1 / (1 - p).  The BatchNorm
normalises with the biased variance and updates the running variance with the unbiased one, as torch does.

Pure CPU torch; nothing here imports the package it checks.
"""
from __future__ import annotations

from typing import Dict, Optional, Sequence

import torch

F64 = torch.float64

# H1 BatchNorm backward without the xhat * mean(g * xhat) term; H2 unbiased variance used to normalise; H3 the dropout
# keep-scale missing in the backward; H4 the last column slice of dW0 / dx (csrc/head.cu, head_backward_kernel) skipped
FAULTS = ("H1", "H2", "H3", "H4")
GRAD_NAMES = ("w0", "b0", "gamma0", "beta0", "w1", "b1", "gamma1", "beta1", "w2", "b2", "x")

# bounds of tests/test_head_pinned_gpu.py, ~4x the worst value measured on a B200 (DESIGN.md section 2,
# profiles/r05_f32_parity.log): max-abs error over the tensor's maximum; the biases in front of a train-mode BatchNorm
# (b0, b1) and beta0, which reaches BatchNorm 1 through the activation-free lins.1, over their layer's dW / dgamma
# maximum.  GPU_TOL holds for B >= 5.  B = 2 has its own table: with two rows xhat = +-1 and the gradient below each
# BatchNorm is a cancellation residue of size ~eps / (var + eps), so fp32 rounding shows up to ~200x larger there.
GPU_TOL = {"out": 1.2e-6, "run": 4.5e-7, "w0": 4.5e-6, "b0": 4.5e-7, "gamma0": 5e-6, "beta0": 3.2e-6, "w1": 6e-6,
           "b1": 5e-7, "gamma1": 2e-6, "beta1": 1.5e-6, "w2": 3e-6, "b2": 1.1e-6, "x": 5.5e-6}
GPU_TOL_B2 = {"out": 7e-5, "run": 1.8e-6, "w0": 1e-3, "b0": 1.3e-5, "gamma0": 9e-4, "beta0": 4.5e-4, "w1": 9e-4,
              "b1": 3e-5, "gamma1": 4.5e-5, "beta1": 4e-7, "w2": 1.8e-4, "b2": 1.4e-7, "x": 1e-3}


def gpu_tol(B: int):
    """The bounds that hold for a batch of B rows."""
    return GPU_TOL_B2 if B == 2 else GPU_TOL


def column_slices(c0: int):
    """(CTAs, columns per CTA) of head_backward_kernel: 64 input columns per CTA, at most 32 CTAs."""
    grid = min((c0 + 63) // 64, 32)
    return grid, (c0 + grid - 1) // grid


def forward(P: Dict[str, torch.Tensor], x: torch.Tensor, masks: Optional[Sequence[torch.Tensor]], p: float,
            eps: float = 1e-5, momentum: float = 0.1, fault: Optional[str] = None):
    """P: w0..w2, b0..b2, gamma0/1, beta0/1, rm0/1, rv0/1 (running statistics before the call).  Returns the output and
    what the backward needs (xhat, rstd, keep) plus the updated running statistics."""
    B = x.shape[0]
    h = x.to(F64) @ P["w0"].to(F64).t() + P["b0"].to(F64)
    res = {}
    for l in (0, 1):
        mean = h.mean(0)
        var = ((h - mean) ** 2).sum(0) / B
        unb = var * B / (B - 1) if B > 1 else var
        res[f"run_mean{l}"] = (1 - momentum) * P[f"rm{l}"].to(F64) + momentum * mean
        res[f"run_var{l}"] = (1 - momentum) * P[f"rv{l}"].to(F64) + momentum * unb
        rstd = 1.0 / torch.sqrt((unb if fault == "H2" else var) + eps)
        xh = (h - mean) * rstd
        y = xh * P[f"gamma{l}"].to(F64) + P[f"beta{l}"].to(F64)
        keep = torch.ones_like(y) if (masks is None or p == 0) else masks[l].to(F64)
        y = y * keep / (1.0 - p)
        res[f"xhat{l}"], res[f"rstd{l}"], res[f"keep{l}"], res[f"a{l}"] = xh, rstd, keep, y
        h = y @ P[f"w{l + 1}"].to(F64).t() + P[f"b{l + 1}"].to(F64)
    res["out"] = h
    return res


def backward(P: Dict[str, torch.Tensor], x: torch.Tensor, fw, gout: torch.Tensor, p: float,
             fault: Optional[str] = None) -> Dict[str, torch.Tensor]:
    """Every gradient of the head in training mode from the forward record ``fw``."""
    B = x.shape[0]
    g = {}
    d = gout.to(F64)
    ks = 1.0 if fault == "H3" else 1.0 / (1.0 - p)
    for l in (1, 0):
        g[f"w{l + 1}"], g[f"b{l + 1}"] = d.t() @ fw[f"a{l}"], d.sum(0)
        da = d @ P[f"w{l + 1}"].to(F64)
        gy = da * fw[f"keep{l}"] * ks                    # gradient w.r.t. gamma * xhat + beta
        xh = fw[f"xhat{l}"]
        g[f"gamma{l}"], g[f"beta{l}"] = (gy * xh).sum(0), gy.sum(0)
        s2 = torch.zeros_like(g[f"gamma{l}"]) if fault == "H1" else g[f"gamma{l}"] / B
        d = P[f"gamma{l}"].to(F64) * fw[f"rstd{l}"] * (gy - g[f"beta{l}"] / B - xh * s2)
    xs = x.to(F64)
    g["w0"], g["b0"] = d.t() @ xs, d.sum(0)
    g["x"] = d @ P["w0"].to(F64)
    if fault == "H4":
        grid, per = column_slices(x.shape[1])
        k0 = (grid - 1) * per
        g["w0"][:, k0:] = 0
        g["x"][:, k0:] = 0
    return g


def grad_errors(got: Dict[str, torch.Tensor], want: Dict[str, torch.Tensor]) -> Dict[str, float]:
    """max-abs error over the tensor's maximum; b0 / b1 over their layer's dW maximum, beta0 over dgamma0's."""
    scale_of = {"b0": "w0", "b1": "w1", "beta0": "gamma0"}
    errs = {}
    for k in GRAD_NAMES:
        gk, wk = got[k].detach().to(F64).cpu(), want[k].detach().to(F64).cpu()
        s = float(want[scale_of.get(k, k)].abs().max())
        errs[k] = float((gk - wk).abs().max()) / max(s, 1e-300)
    return errs
