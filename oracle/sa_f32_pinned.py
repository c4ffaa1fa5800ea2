"""Decision-pinned float64 reference of one fp32 set-abstraction level -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

The fp32 kernels (csrc/sa_simt.cu) are fp32 FMA with double-precision BatchNorm sums.  ``ref.MLPRef`` recomputes a level
from its inputs and takes its own arg-max and ReLU decisions, so it differentiates a slightly different function than
the kernels wherever fp32 rounding flips a decision.  The functions here start every layer from what the kernels STORED
for it (``_SAFunction``'s saved tensors) and take every decision from the stored state, so the only difference left is
fp32 summation order:

* forward: h1 from the inputs ([x_j | pos_j - pos_i], the difference in the inputs' own precision, as ``__fsub_rn``
  forms it); batch statistics of the STORED h1 over the valid rows; h2 from the stored h1 through the stored ``bn``
  scale / shift; the same for layer 2; per-row layer-3 values from the stored h2; max and first arg-max per (target,
  channel), 0 / -1 for a target without rows.
* backward: dh3 routed by the kernel's ``arg``; ReLU masks from ``h * scale + shift > 0`` with the stored h and bn
  (evaluated in float64: the product of two fp32 values is exact there and the sum keeps the sign ``fmaf`` gives, the
  library being built without flush-to-zero); BatchNorm backward with the stored ``bn``; dW / db per layer, dgamma /
  dbeta, the two dz, and ``grad_x`` (scatter-add in SLOTS, one row per source point in CLOUDS).

Row layout of the fp32 levels (restated from include/b2pn.h and csrc/sa_simt.cu): SLOTS row ``m * K + k`` is neighbour
slot k of target m, valid iff ``k < cnt[m]``, and ``arg`` holds the slot; CLOUDS row r is source point r of cloud
``batch[r]`` and ``arg`` holds the row.  ``h1`` / ``h2`` are the pre-BatchNorm values INCLUDING the bias, row-major
``[rows, c]``, zero on invalid rows; ``bn`` is ``[2, 4, cmax]``: mean, rstd, scale = gamma * rstd, shift = beta -
mean * scale per layer.  The batch statistics divide by the number of valid rows (sum of cnt, or n_src).

Pure CPU torch; nothing here imports the package it checks.
"""
from __future__ import annotations

from typing import Dict, Optional

import torch

F64 = torch.float64

# the slots of _SAFunction.save_for_backward, in order (dl_biomass_b200/sa.py); the fp32 path leaves the row-map and
# 16-bit activation slots (rgrp .. g1) None
SAVED_NAMES = ("xs", "pos_src", "pos_dst", "nbr", "cnt", "batch", "w1", "w2", "w3", "b1", "b2", "b3",
               "gamma1", "gamma2", "beta1", "beta2", "rm1", "rv1", "rm2", "rv2", "arg", "h1", "h2", "bn",
               "rgrp", "row_src", "num_rows", "row_valid", "a1", "a2", "g1")
GRAD_NAMES = ("w1", "b1", "gamma1", "beta1", "w2", "b2", "gamma2", "beta2", "w3", "b3", "x")

# injected faults: F1 BatchNorm backward without the zhat * mean(dz * zhat) term; F2 batch statistics (and the BN
# backward means) over all n_dst * K slots instead of the valid rows; F3 ReLU mask from zhat > 0; F4 one (target,
# channel) arg-max gradient in F4_EVERY routed to the neighbouring slot / row; F5 the rows of the last dW split dropped;
# F6 exact CLOUDS ties resolved towards the last row; F7 grad_x without the last slot of every saturated neighbourhood
FAULTS = ("F1", "F2", "F3", "F4", "F5", "F6", "F7")
F4_EVERY = 10000

# bounds of tests/test_sa_f32_gpu.py (kernels vs this reference), each ~4x the worst value measured on a B200 over every
# case of that file (DESIGN.md section 2, profiles/r05_f32_parity.log): h1 / h2 / out as max-abs error over the
# tensor's maximum, the bn rows and running statistics the same, gradients as max-abs error over the tensor's maximum
# (train-mode b1 / b2: over their layer's dW maximum)
GPU_TOL = {"h": 2.5e-6, "bn": 2.5e-7, "run": 3e-7, "out": 3e-6, "arg": 3e-6,
           "w1": 8e-6, "b1": 4e-6, "gamma1": 3.5e-6, "beta1": 4e-6, "w2": 7e-6, "b2": 4.5e-6, "gamma2": 2e-6,
           "beta2": 1.5e-6, "w3": 1.5e-6, "b3": 2.5e-6, "x": 4.5e-6}


def dw_splits(rows: int):
    """(splits, rows per split) of the fp32 dW GEMMs (csrc/sa_simt.cu, shapes_of / launch_dw)."""
    splits = min(max(rows // 2048, 1), 296)
    rps = ((rows + splits - 1) // splits + 15) // 16 * 16
    return splits, rps


class Layout:
    """Valid rows of an fp32 level: their full row index, target, arg id and source point."""

    def __init__(self, st: Dict[str, Optional[torch.Tensor]], n_dst: int, K: int):
        self.slots = st.get("nbr") is not None
        self.n_dst, self.K = n_dst, K
        if self.slots:
            cnt = st["cnt"].to(torch.int64)
            self.rows = n_dst * K
            k = torch.arange(K)
            valid = (k[None, :] < cnt[:, None]).flatten()
            self.R = torch.nonzero(valid).flatten()            # full row index of each valid row
            self.cent = self.R // K
            self.id = self.R % K                              # what arg[] stores: the slot
            self.src = st["nbr"].to(torch.int64).flatten()[self.R]
            self.edges = int(cnt.sum())
            self.saturated = cnt[self.cent] == K
        else:
            n = st["pos_src"].shape[0]
            self.rows = self.edges = n
            self.R = torch.arange(n)
            self.cent = st["batch"].to(torch.int64)
            self.id = self.R                                  # arg[] stores the row
            self.src = self.R
            self.saturated = torch.zeros(n, dtype=torch.bool)
        self.index = torch.full((max(self.rows, 1),), -1, dtype=torch.int64)   # full row -> valid-row index
        self.index[self.R] = torch.arange(self.R.numel())

    def arg_rows(self, arg: torch.Tensor) -> torch.Tensor:
        """Valid-row index of each (target, channel) arg-max (-1: none)."""
        arg = arg.to(torch.int64)
        full = arg + (torch.arange(self.n_dst)[:, None] * self.K if self.slots else 0)
        return torch.where(arg >= 0, self.index[full.clamp(0, max(self.rows - 1, 0))], torch.full_like(arg, -1))

    def stored(self, t: Optional[torch.Tensor]) -> Optional[torch.Tensor]:
        """The valid rows of a stored [rows, c] tensor, float64."""
        return None if t is None else t[self.R].to(F64)


def layer1_input(st, lay: Layout) -> torch.Tensor:
    """[valid rows, c_in + 3]: [x_j | pos_j - pos_i], the difference in the inputs' precision, then float64."""
    ps = st["pos_src"][lay.src]
    d = ps - st["pos_dst"][lay.cent] if lay.slots else ps
    xs = st.get("xs")
    if xs is None or xs.shape[1] == 0:
        return d.to(F64)
    return torch.cat([xs[lay.src].to(F64), d.to(F64)], 1)


def _act(v, relu):
    return v.clamp_min(0) if relu else v


def _bn_split(bn: torch.Tensor, c: int):
    b = bn.to(F64)
    return b[0, :c], b[1, :c], b[2, :c], b[3, :c]


def first_max(v3: torch.Tensor, lay: Layout, last: bool = False):
    """Per (target, channel): max over the rows and the lowest arg id holding it (``last``: the highest);
    0 / -1 for a target without rows."""
    n_dst, C = lay.n_dst, v3.shape[1]
    out = torch.zeros(n_dst, C, dtype=F64)
    arg = torch.full((n_dst, C), -1, dtype=torch.int64)
    if v3.shape[0] == 0:
        return out, arg
    idx = lay.cent[:, None].expand_as(v3)
    mx = torch.full((n_dst, C), float("-inf"), dtype=F64).scatter_reduce(0, idx, v3, "amax")
    order = lay.id[:, None].expand_as(v3)
    fill = -1 if last else torch.iinfo(torch.int64).max
    cand = torch.where(v3 == mx[lay.cent], order, torch.full_like(order, fill))
    a = torch.full((n_dst, C), fill, dtype=torch.int64).scatter_reduce(0, idx, cand, "amax" if last else "amin")
    has = a != fill
    return torch.where(has, mx, out), torch.where(has, a, arg)


def pinned_forward(st: Dict[str, Optional[torch.Tensor]], *, training: bool, relu: bool, eps: float, momentum: float,
                   n_dst: int, K: int, fault: Optional[str] = None):
    """What the kernels should have stored, layer by layer from the kernels' own stored values.

    ``st['rm*'] / st['rv*']`` must hold the running statistics from BEFORE the call.  Where ``st`` has no h1 / h2 / bn
    (a reference-only run) the reference's own values stand in.  Returns float64 ``h1`` / ``h2`` [valid rows, c],
    ``bn1`` / ``bn2`` [4, c], ``run_mean*`` / ``run_var*`` (train mode), ``v3`` (layer-3 values incl. bias) and
    ``out`` / ``arg``."""
    lay = Layout(st, n_dst, K)
    res = {"layout": lay}
    X = layer1_input(st, lay)
    E = float(lay.rows if fault == "F2" else lay.edges)
    for l in (1, 2):
        h = X @ st[f"w{l}"].to(F64).t() + st[f"b{l}"].to(F64)
        res[f"h{l}"] = h
        hs = lay.stored(st.get(f"h{l}"))
        hs = h if hs is None else hs                     # the STORED h feeds the statistics and the next layer
        c = h.shape[1]
        if training:
            mean = hs.sum(0) / E
            var = (((hs - mean) ** 2).sum(0) + (E - hs.shape[0]) * mean ** 2) / E
            unb = var * E / (E - 1.0) if E > 1 else var
            res[f"run_mean{l}"] = (1 - momentum) * st[f"rm{l}"].to(F64) + momentum * mean
            res[f"run_var{l}"] = (1 - momentum) * st[f"rv{l}"].to(F64) + momentum * unb
        else:
            mean, var = st[f"rm{l}"].to(F64), st[f"rv{l}"].to(F64)
        rstd = 1.0 / torch.sqrt(var + eps)
        scale = st[f"gamma{l}"].to(F64) * rstd
        res[f"bn{l}"] = torch.stack([mean, rstd, scale, st[f"beta{l}"].to(F64) - mean * scale])
        bn = st.get("bn")
        _, _, sc, sh = _bn_split(bn[l - 1], c) if bn is not None else tuple(res[f"bn{l}"])
        X = _act(hs * sc + sh, relu)                     # the STORED scale / shift, as the next loader applies them
    v3 = X @ st["w3"].to(F64).t() + st["b3"].to(F64)
    res["v3"] = v3
    res["out"], res["arg"] = first_max(v3, lay, last=(fault == "F6"))
    return res


def pinned_backward(st: Dict[str, Optional[torch.Tensor]], dout: torch.Tensor, *, training: bool, relu: bool,
                    n_dst: int, K: int, fault: Optional[str] = None,
                    want_dx: bool = True) -> Dict[str, Optional[torch.Tensor]]:
    """Every gradient of the level from the kernels' stored decisions (arg, h, bn).  Keys: GRAD_NAMES (+ dz1, dz2:
    the BN-backward results on the valid rows)."""
    lay = Layout(st, n_dst, K)
    nV = lay.R.numel()
    C3 = st["w3"].shape[0]
    g = dout.to(F64)
    ar = lay.arg_rows(st["arg"])
    if fault == "F4":   # every F4_EVERY-th (target, channel) arg-max gradient lands on the neighbouring row
        flat = ar.flatten().clone()
        nxt = torch.where(flat + 1 < nV, flat + 1, flat - 1)
        same = (flat >= 0) & (nxt >= 0) & (lay.cent[nxt.clamp(0, max(nV - 1, 0))] == lay.cent[flat.clamp(0, max(nV - 1, 0))])
        pick = torch.zeros_like(same)
        pick[::F4_EVERY] = True
        flat = torch.where(pick & same, nxt, flat)
        ar = flat.view_as(ar)
    dh3 = torch.zeros(nV, C3, dtype=F64)
    ok = ar >= 0
    chan = torch.arange(C3)[None, :].expand_as(ar)
    dh3.index_put_((ar[ok], chan[ok]), g[ok], accumulate=True)
    dw_rows = torch.ones(nV, dtype=torch.bool)
    splits, rps = dw_splits(lay.rows)
    if fault == "F5" and splits > 1:
        dw_rows = lay.R < (splits - 1) * rps
    out = {}

    def dw(dy, X):
        dy = dy[dw_rows]
        return dy.t() @ X[dw_rows], dy.sum(0)

    E = float(lay.rows if fault == "F2" else lay.edges)
    dh = dh3
    for l in (2, 1):      # layer l+1's dX / dW, then BatchNorm backward of layer l
        hs = lay.stored(st[f"h{l}"])
        c = hs.shape[1]
        mean, rstd, scale, shift = _bn_split(st["bn"][l - 1], c)
        pre = hs * scale + shift
        out[f"w{l + 1}"], out[f"b{l + 1}"] = dw(dh, _act(pre, relu))
        da = dh @ st[f"w{l + 1}"].to(F64)
        zhat = (hs - mean) * rstd
        dy = da * ((zhat > 0) if fault == "F3" else (pre > 0)) if relu else da
        S1, S2 = dy.sum(0), (dy * zhat).sum(0)
        out[f"beta{l}"], out[f"gamma{l}"] = S1, S2
        if training:
            s1, s2 = S1 / E, S2 / E
            if fault == "F1":
                s2 = torch.zeros_like(s2)
        else:
            s1 = s2 = torch.zeros_like(S1)
        dh = scale * (dy - s1 - zhat * s2)
        out[f"dz{l}"] = dh
    out["w1"], out["b1"] = dw(dh, layer1_input(st, lay))
    xs = st.get("xs")
    if want_dx and xs is not None and xs.shape[1] > 0:
        c_in = xs.shape[1]
        e = dh @ st["w1"][:, :c_in].to(F64)
        keep = ~(lay.saturated & (lay.id == K - 1)) if fault == "F7" else torch.ones(nV, dtype=torch.bool)
        gx = torch.zeros(xs.shape[0], c_in, dtype=F64)
        gx.index_add_(0, lay.src[keep], e[keep])
        out["x"] = gx
    else:
        out["x"] = None
    return out


def max_rel(got: torch.Tensor, want: torch.Tensor, scale: Optional[float] = None) -> float:
    """max |got - want| over max |want| (or over `scale`)."""
    got, want = got.detach().to(F64).cpu(), want.detach().to(F64).cpu()
    s = float(want.abs().max()) if (scale is None and want.numel()) else float(scale or 0.0)
    return float((got - want).abs().max()) / max(s, 1e-300) if want.numel() else 0.0


def grad_errors(got: Dict[str, torch.Tensor], want: Dict[str, torch.Tensor], training: bool,
                zero_b3: bool = False) -> Dict[str, float]:
    """Per-gradient max-abs error relative to the tensor's maximum.  Biases feeding a train-mode BatchNorm are zero in
    theory: they are measured against the maximum of their layer's weight gradient instead.  So is b3 with
    ``zero_b3``: the level's incoming gradient is the feature gradient of a train-mode BatchNorm level (or head)
    downstream, whose column sums vanish."""
    errs = {}
    for k in GRAD_NAMES:
        if got.get(k) is None or want.get(k) is None:
            continue
        if (training and k in ("b1", "b2")) or (zero_b3 and k == "b3"):
            errs[k] = max_rel(got[k], want[k], scale=float(want["w" + k[1]].abs().max()))
        else:
            errs[k] = max_rel(got[k], want[k])
    return errs


def state_from_forward(st, fw, chans):
    """The state the kernels would store had they computed exactly ``fw``: h1 / h2 [rows, c] (zero on invalid rows),
    bn and arg.  For reference-only runs."""
    lay = fw["layout"]
    st = dict(st)
    for l in (1, 2):
        T = torch.zeros(lay.rows, chans[l], dtype=F64)
        T[lay.R] = fw[f"h{l}"]
        st[f"h{l}"] = T
    cmax = max(chans[1], chans[2])
    bn = torch.zeros(2, 4, cmax, dtype=F64)
    for l in (1, 2):
        bn[l - 1, :, : chans[l]] = fw[f"bn{l}"]
    st["bn"], st["arg"] = bn, fw["arg"]
    return st


def with_fault(st, dout, fault: str, *, training: bool, relu: bool, eps: float, momentum: float, n_dst: int, K: int):
    """(forward, backward) of the level with one fault injected, on the same stored state.  F6 acts through the arg
    it picks: the backward then routes by that arg."""
    kw = dict(training=training, relu=relu, n_dst=n_dst, K=K)
    fw = pinned_forward(st, eps=eps, momentum=momentum, fault=fault if fault in ("F2", "F6") else None, **kw)
    stb = dict(st, arg=fw["arg"]) if fault == "F6" else st
    bw = pinned_backward(stb, dout, fault=None if fault == "F6" else fault, **kw)
    return fw, bw


BN_ROWS = ("mean", "rstd", "scale", "shift")


def tol_key(what: str) -> str:
    """The GPU_TOL entry of an error name of forward_errors / grad_errors."""
    if what.startswith("h"):
        return "h"
    if what.startswith("bn"):
        return "bn"
    if what.startswith("run_"):
        return "run"
    return what


def forward_errors(got, want, training: bool) -> Dict[str, float]:
    """h1 / h2 [valid rows, c], bn1 / bn2 [4, c] per row, running statistics (train mode) and out, each as max-abs
    error over the maximum of `want`."""
    e = {}
    for l in (1, 2):
        e[f"h{l}"] = max_rel(got[f"h{l}"], want[f"h{l}"])
        for i, nm in enumerate(BN_ROWS):
            e[f"bn{l} {nm}"] = max_rel(got[f"bn{l}"][i], want[f"bn{l}"][i])
        if training:
            for k in (f"run_mean{l}", f"run_var{l}"):
                e[k] = max_rel(got[k], want[k])
    e["out"] = max_rel(got["out"], want["out"])
    return e


def tie_errors(arg: torch.Tensor, fw) -> int:
    """(target, channel) pairs whose reference maximum is held by several rows exactly and whose `arg` is not the
    first of them."""
    lay, v3 = fw["layout"], fw["v3"]
    if v3.shape[0] == 0:
        return 0
    nmax = torch.zeros(fw["out"].shape, dtype=torch.int64).scatter_add_(
        0, lay.cent[:, None].expand_as(v3), (v3 == fw["out"][lay.cent]).long())
    return int(((nmax > 1) & (arg.to(torch.int64) != fw["arg"])).sum())
