"""Decision-pinned float64 reference of one 16-bit set-abstraction level -- TEST INFRASTRUCTURE, NOT PRODUCT CODE.

``ref.MLPRef(emulate_bf16=True)`` recomputes a level from its inputs and takes its own arg-max and ReLU decisions;
16-bit rounding flips some of them, so it differentiates a slightly different function than the kernels and its
gradients can only be compared loosely.  The functions here instead start every layer from what the kernels STORED for
it (``_SAFunction``'s saved tensors) and take every decision from the stored state, so the only differences left are
the roundings listed in ``Rounding`` (each can be switched off) and fp32 summation order:

* forward: h1 from the stored layer-1 operand ``g1`` (or the gather, where there is none) and the fp16 image of W1;
  batch statistics over the valid rows; the expected zhat1 / a1; h2 from the STORED a1 (or the a1 rebuilt from the
  stored zhat1 when only zhat is kept); the same for layer 2; per-row layer-3 values from the stored a2; max and first
  arg-max per (target, channel).
* backward: dh3 routed by the kernel's ``arg``; ReLU masks from the stored zhat with gamma / beta; the BatchNorm
  backward with the stored ``bn`` buffer; dW / db per layer, dgamma / dbeta, the two dz, and the ``grad_x`` scatter
  through ``row_src`` (SLOTS) or the rows themselves (CLOUDS).

Compacted row layout of the 16-bit SLOTS levels (restated from include/b2pn.h, b2pn_pack_rows): one u32 descriptor per
8-row group -- bits 0..23 centroid (0xFFFFFF none), 24..26 first slot / 8, 27..30 valid rows, 31 last group of the
centroid; ``row_src[row]`` the gathered source point (-1 padding); ``num_rows = [rows in use, edges]``.  Invalid rows
carry zero activations.  CLOUDS levels: row r is source point r of cloud ``batch[r]``, every row valid.

Pure CPU torch; nothing here imports the package it checks.
"""
from __future__ import annotations

from dataclasses import dataclass, replace
from typing import Dict, Optional

import torch

F64 = torch.float64

# the slots of _SAFunction.save_for_backward, in order (dl_biomass_b200/sa.py)
SAVED_NAMES = ("xs", "pos_src", "pos_dst", "nbr", "cnt", "batch", "w1", "w2", "w3", "b1", "b2", "b3",
               "gamma1", "gamma2", "beta1", "beta2", "rm1", "rv1", "rm2", "rv2", "arg", "h1", "h2", "bn",
               "rgrp", "row_src", "num_rows", "row_valid", "a1", "a2", "g1")

GRAD_NAMES = ("w1", "b1", "gamma1", "beta1", "w2", "b2", "gamma2", "beta2", "w3", "b3", "x")

MUTATIONS = ("M1", "M2", "M3", "M4", "M5", "M6")
# M4: fraction of the (target, channel) arg-max gradients moved to the neighbouring slot, tuned so that the fault moves
# some gradient by more than 3x its pinned tolerance while EVERY gradient stays inside the bounds of the emulating
# oracle's tests (tests/test_sa_pinned_ref.py)
M4_FRACTION = 0.001

# bounds of tests/test_sa_pinned_gpu.py (kernel vs this reference, every rounding emulated): stored zhat / a in fp16
# ulps, gradients as max-abs error over the tensor's maximum (train-mode b1 / b2: over their layer's dW maximum)
# ~4x the worst value measured on a B200 over every case of that file (DESIGN.md section 2), never above 5e-3; zhat:
# 0.5 ulp of rounding plus the fp32 batch statistics (measured 1.33 ulp at 12 x 500 rows)
GPU_TOL = {"z_ulp": 2.0, "a_ulp": 1.0,
           "w1": 2.5e-3, "b1": 1.2e-3, "gamma1": 7e-4, "beta1": 8e-4, "w2": 2e-3, "b2": 1e-3, "gamma2": 1e-6,
           "beta2": 1.2e-6, "w3": 2e-6, "b3": 2e-5, "x": 5e-3}


@dataclass(frozen=True)
class Rounding:
    """The rounding points of the 16-bit kernels (csrc/sa_tc.cu, csrc/sa_chain.cuh); each can be switched off."""
    f16_fwd: bool = True     # fp16 weight images of the forward GEMMs, fp16 zhat / a (forward-domain operands)
    split: bool = True       # fp32 inputs (c_in <= 16, relative positions) as fp16 hi + lo column pairs
    bf16_wT: bool = True     # bf16 W^T of the dX GEMMs (backward packs)
    bf16_gout: bool = True   # grad_out -> bf16 in the routed tiles
    bf16_dz: bool = True     # the masked da stored as bf16 (dz) and the BN-backward result dh stored as bf16
    bf16_xdw: bool = True    # fp16 -> bf16 conversion of the X side of the dW GEMMs (each image column on its own)
    fixed_dx: bool = False   # deterministic grad_x: every addend rounded to the 2^-40 fixed-point unit


ROUND_ALL = Rounding()
ROUND_NONE = Rounding(False, False, False, False, False, False, False)


def f16(t):
    return t.to(torch.float16).to(F64)


def bf16(t):
    return t.to(torch.bfloat16).to(F64)


def ulp16(v: torch.Tensor) -> torch.Tensor:
    """fp16 unit in the last place of |v| (subnormal spacing below 2^-14)."""
    e = torch.floor(torch.log2(v.abs().clamp_min(2.0 ** -14)))
    return torch.pow(2.0, e - 10)


# ------------------------------------------------------------------------------------------------------------------
#  row layout
# ------------------------------------------------------------------------------------------------------------------
def pack_rows_cpu(cnt: torch.Tensor, nbr: torch.Tensor):
    """A compacted row layout with the rules of b2pn_pack_rows (centroid m owns max(8, round_up(cnt[m], 8)) consecutive
    rows inside one 64-row block, slots in order).  Returns (rgrp int32, row_src int32, num_rows int64[2], ld)."""
    n_dst, K = nbr.shape
    starts, r = [], 0
    for m in range(n_dst):
        c8 = max(8, (int(cnt[m]) + 7) // 8 * 8)
        if r // 64 != (r + c8 - 1) // 64:
            r = (r // 64 + 1) * 64
        starts.append(r)
        r += c8
    rows = max(64, (r + 63) // 64 * 64)
    ld = (rows + 127) // 128 * 128
    rgrp = torch.full((ld // 8,), 0xFFFFFF, dtype=torch.int64)
    row_src = torch.full((ld,), -1, dtype=torch.int32)
    for m in range(n_dst):
        c = int(cnt[m])
        c8 = max(8, (c + 7) // 8 * 8)
        s = starts[m]
        row_src[s:s + c] = nbr[m, :c]
        for j in range(c8 // 8):
            nv = min(8, max(0, c - 8 * j))
            rgrp[s // 8 + j] = m | (j << 24) | (nv << 27) | ((1 if j == c8 // 8 - 1 else 0) << 31)
    rgrp = torch.where(rgrp >= 2 ** 31, rgrp - 2 ** 32, rgrp).to(torch.int32)
    return rgrp, row_src, torch.tensor([rows, int(cnt.sum())], dtype=torch.int64), ld


class Layout:
    """Valid rows of a level: index V (rows of the stored [c, ld] tensors), target / slot / source per valid row."""

    def __init__(self, st: Dict[str, Optional[torch.Tensor]], n_dst: int, K: int):
        self.slots = st.get("rgrp") is not None
        self.n_dst = n_dst
        if self.slots:
            nr = st["num_rows"].to(torch.int64)
            self.rows_used, self.edges = int(nr[0]), int(nr[1])
            rs = st["row_src"].to(torch.int64)[: self.rows_used]
            self.V = torch.nonzero(rs >= 0).flatten()
            g = st["rgrp"].to(torch.int64) & 0xFFFFFFFF
            gv = g[self.V >> 3]
            self.cent = gv & 0xFFFFFF
            self.slot = ((gv >> 24) & 7) * 8 + (self.V & 7)
            self.src = rs[self.V]
            self.row_of = torch.full((n_dst, max(K, 1)), -1, dtype=torch.int64)   # (target, slot) -> valid-row index
            self.row_of[self.cent, self.slot] = torch.arange(self.V.numel())
        else:
            n = st["pos_src"].shape[0]
            self.rows_used = self.edges = n
            self.V = torch.arange(n)
            self.cent = st["batch"].to(torch.int64)
            self.src = self.V
        self.ld = st["h1"].shape[1] if st.get("h1") is not None else (self.rows_used + 127) // 128 * 128

    def arg_rows(self, arg: torch.Tensor) -> torch.Tensor:
        """Valid-row index of each (target, channel) arg-max (-1: none)."""
        arg = arg.to(torch.int64)
        if not self.slots:
            return arg
        return torch.where(arg >= 0, self.row_of.gather(1, arg.clamp_min(0)), torch.full_like(arg, -1))


def _x_split(xs) -> bool:
    return xs is not None and xs.dtype != torch.float16


def _split_parts(v: torch.Tensor, fmt, on: bool):
    """(hi, lo) as the kernels form them: hi = fmt(v), lo = fmt(v - hi) with the difference in v's own precision."""
    if not on:
        return v.to(F64), torch.zeros_like(v, dtype=F64)
    rnd = torch.float16 if fmt == "f16" else torch.bfloat16
    hi = v.to(rnd).to(v.dtype)
    return hi.to(F64), (v - hi).to(rnd).to(F64)


def _layer1_input(st, lay: Layout, rnd: Rounding, for_dw: bool) -> torch.Tensor:
    """[valid rows, c_in + 3] float64: the layer-1 operand as the GEMM sees it (hi + lo parts summed per weight column).
    for_dw: the X side of dW1, whose fp16 image columns are converted to bf16 one by one."""
    xs, g1 = st.get("xs"), st.get("g1")
    c_in = 0 if xs is None else xs.shape[1]
    split = _x_split(xs)
    conv = (lambda t: bf16(t)) if (for_dw and rnd.bf16_xdw) else (lambda t: t.to(F64))
    if g1 is not None:   # the stored operand: [x | x_lo | dpos_hi | dpos_lo | ones] x ld
        G = g1[:, lay.V].t()
        nx = c_in * (2 if split else 1)
        cols = []
        for k in range(c_in):
            v = conv(G[:, k])
            if split:
                v = v + conv(G[:, c_in + k])
            cols.append(v)
        for j in range(3):
            cols.append(conv(G[:, nx + j]) + conv(G[:, nx + 3 + j]))
        return torch.stack(cols, 1)
    # gathered in the loader warps: fp16 image (forward) or bf16 image (X side of dW1)
    fmt = "bf16" if (for_dw and rnd.bf16_xdw) else "f16"
    on = rnd.split if fmt == "f16" else rnd.bf16_xdw
    pos_src = st["pos_src"]
    d = pos_src[lay.src] - (st["pos_dst"][lay.cent] if lay.slots else 0)
    hi, lo = _split_parts(d, fmt, on)
    dpos = hi + lo
    if xs is None:
        return dpos
    x = xs[lay.src]
    if split:
        hi, lo = _split_parts(x, fmt, on if xs.dtype == torch.float32 else False)
        xv = hi + lo
    else:
        xv = conv(x)
    return torch.cat([xv, dpos], 1)


def _act(v, relu: bool):
    return v.clamp_min(0) if relu else v


def _bn_stats(h: torch.Tensor, denom: float):
    """Batch mean / biased variance of h [rows, c] over `denom` rows (the rows not in h count as zeros)."""
    S = h.sum(0)
    ma = S / denom
    var = ((h - ma) ** 2).sum(0) + (denom - h.shape[0]) * ma ** 2
    return ma, (var / denom).clamp_min(0)


def pinned_forward(st: Dict[str, Optional[torch.Tensor]], *, training: bool, relu: bool, eps: float, momentum: float,
                   n_dst: int, K: int, rnd: Rounding = ROUND_ALL, mutate: Optional[str] = None):
    """What the kernels should have stored, layer by layer from the kernels' own stored inputs.

    Returns float64 [valid rows, c] tensors z1 / a1 / z2 / a2 (a from the STORED z of the same layer, as the kernels
    define it), v3 (layer-3 values incl. bias), per-layer mean / rstd / running mean / running var (train mode: the
    update of ``st['rm*'] / st['rv*']``, which must hold the values from BEFORE the call), and out / arg."""
    lay = Layout(st, n_dst, K)
    w16 = f16 if rnd.f16_fwd else (lambda t: t.to(F64))
    res = {"layout": lay}
    Ws = [st["w1"], st["w2"], st["w3"]]
    bs = [st["b1"].to(F64), st["b2"].to(F64), st["b3"].to(F64)]
    X = _layer1_input(st, lay, rnd, for_dw=False)
    for l in range(2):
        h = X @ w16(Ws[l]).t()                      # bias-free accumulator
        g, be = st[f"gamma{l + 1}"].to(F64), st[f"beta{l + 1}"].to(F64)
        if training:
            denom = float(lay.rows_used if mutate == "M6" else lay.edges)
            ma, var = _bn_stats(h, denom)
            mean = ma + bs[l]
            E = float(lay.edges)
            unb = var * E / (E - 1.0) if E > 1 else var
            res[f"run_mean{l + 1}"] = (1 - momentum) * st[f"rm{l + 1}"].to(F64) + momentum * mean
            res[f"run_var{l + 1}"] = (1 - momentum) * st[f"rv{l + 1}"].to(F64) + momentum * unb
        else:
            mean, var = st[f"rm{l + 1}"].to(F64), st[f"rv{l + 1}"].to(F64)
        rstd = 1.0 / torch.sqrt(var + eps)
        z = (h + bs[l] - mean) * rstd
        res[f"mean{l + 1}"], res[f"rstd{l + 1}"], res[f"z{l + 1}"] = mean, rstd, z
        zs = st.get(f"h{l + 1}")
        zs = z if zs is None else zs[:, lay.V].t().to(F64)     # the STORED zhat decides the activation
        a = _act(zs * g + be, relu)
        a = f16(a) if rnd.f16_fwd else a
        res[f"a{l + 1}"] = a
        a_st = st.get(f"a{l + 1}")
        X = a if a_st is None else a_st[:, lay.V].t().to(F64)  # the next layer starts from the STORED activation
    v3 = X @ w16(Ws[2]).t() + bs[2]
    res["v3"] = v3
    C = v3.shape[1]
    out = torch.zeros(n_dst, C, dtype=F64)
    arg = torch.full((n_dst, C), -1, dtype=torch.int64)
    if v3.shape[0]:
        idx = lay.cent[:, None].expand_as(v3)
        mx = torch.full((n_dst, C), float("-inf"), dtype=F64).scatter_reduce(0, idx, v3, "amax")
        order = (lay.slot if lay.slots else lay.V)[:, None].expand_as(v3)
        big = torch.iinfo(torch.int64).max
        cand = torch.where(v3 == mx[lay.cent], order, torch.full_like(order, big))
        arg = torch.full((n_dst, C), big, dtype=torch.int64).scatter_reduce(0, idx, cand, "amin")
        has = arg != big
        out = torch.where(has, mx, out)
        arg = torch.where(has, arg, torch.full_like(arg, -1))
    res["out"], res["arg"] = out, arg
    return res


def pinned_backward(st: Dict[str, Optional[torch.Tensor]], dout: torch.Tensor, *, training: bool, relu: bool,
                    n_dst: int, K: int, rnd: Rounding = ROUND_ALL, mutate: Optional[str] = None,
                    want_dx: bool = True) -> Dict[str, Optional[torch.Tensor]]:
    """Every gradient of the level from the kernels' stored decisions (arg, zhat, bn).  Keys: GRAD_NAMES (+ dz1, dz2:
    the stored BN-backward results on the valid rows)."""
    lay = Layout(st, n_dst, K)
    nV = lay.V.numel()
    wT = bf16 if rnd.bf16_wT else (lambda t: t.to(F64))
    qd = bf16 if rnd.bf16_dz else (lambda t: t)
    xw = bf16 if rnd.bf16_xdw else (lambda t: t.to(F64))
    C3 = st["w3"].shape[0]
    g = bf16(dout) if rnd.bf16_gout else dout.to(F64)
    # ---- routed gradient of the max
    ar = lay.arg_rows(st["arg"])
    if mutate == "M4":   # a fraction of the (target, channel) arg-max gradients lands on the neighbouring slot
        n_all = ar.numel()
        nm = max(1, int(round(M4_FRACTION * n_all)))
        pick = torch.zeros(n_all, dtype=torch.bool)
        pick[torch.linspace(0, n_all - 1, nm).long()] = True
        pick = pick.view_as(ar)
        if lay.slots:
            cnt = st["cnt"].to(torch.int64)
            a = st["arg"].to(torch.int64)
            nb = torch.where(a + 1 < cnt[:, None], a + 1, (a - 1).clamp_min(0))
            moved = torch.where(nb >= 0, lay.row_of.gather(1, nb.clamp_min(0)), ar)
        else:
            moved = torch.where(ar + 1 < lay.V.numel(), ar + 1, ar - 1)
            moved = torch.where(lay.cent[moved.clamp(0, nV - 1)] == torch.arange(n_dst)[:, None], moved, ar)
        ar = torch.where(pick & (ar >= 0), moved, ar)
    dh3 = torch.zeros(nV, C3, dtype=F64)
    ok = ar >= 0
    chan = torch.arange(C3)[None, :].expand_as(ar)
    dh3.index_put_((ar[ok], chan[ok]), g[ok], accumulate=True)
    # rows that take part in the dW GEMMs (M5: the last 64-row tile in use is dropped)
    dw_rows = torch.ones(nV, dtype=torch.bool)
    if mutate == "M5":
        dw_rows = lay.V < (lay.rows_used - 1) // 64 * 64
    out = {}

    def dw(dy, X):
        dy = dy[dw_rows]
        return dy.t() @ X[dw_rows], dy.sum(0)

    E = float(lay.rows_used if mutate == "M2" else lay.edges)
    dh = dh3
    X_next = None
    for l in (2, 1):      # layer l+1's dX / dW, then BatchNorm backward of layer l
        a_st = st.get(f"a{l}")
        zs = st[f"h{l}"][:, lay.V].t().to(F64)
        ga, be = st[f"gamma{l}"].to(F64), st[f"beta{l}"].to(F64)
        c = zs.shape[1]
        # the X side of dW is the stored activation, fetched by TMA, where the layer width allows 64-channel boxes and
        # a row-valid line exists (csrc/sa_tc.cu, tma_x1 / tma_x2); otherwise -- and when only zhat is stored -- the
        # loaders rebuild a = act(gamma zhat + beta) from zhat straight into bf16
        tma_x = st.get("row_valid") is not None and c % 64 == 0
        if a_st is None or not tma_x:
            A = _act(zs * ga + be, relu)
            X = bf16(A) if rnd.bf16_xdw else (f16(A) if rnd.f16_fwd else A)
        else:
            X = xw(a_st[:, lay.V].t())
        out[f"w{l + 1}"], out[f"b{l + 1}"] = dw(dh, X)
        da = dh @ wT(st[f"w{l + 1}"])
        if relu:
            mask = (zs > 0) if mutate == "M3" else (zs * ga + be > 0)
            dy = da * mask
        else:
            dy = da
        S1, S2 = dy.sum(0), (dy * zs).sum(0)
        out[f"beta{l}"], out[f"gamma{l}"] = S1, S2
        if training:
            s1, s2 = S1 / E, S2 / E
            if mutate == "M1":
                s2 = torch.zeros_like(s2)
        else:
            s1 = s2 = torch.zeros_like(S1)
        scale = st["bn"][l - 1, 2, : S1.numel()].to(F64)
        dh = qd(scale * (qd(dy) - s1 - zs * s2))
        out[f"dz{l}"] = dh
    X1 = _layer1_input(st, lay, rnd, for_dw=True)
    out["w1"], out["b1"] = dw(dh, X1)
    xs = st.get("xs")
    if want_dx and xs is not None and xs.shape[1] > 0:
        c_in = xs.shape[1]
        e = dh @ wT(st["w1"][:, :c_in])
        if rnd.fixed_dx:
            e = torch.round(e * 2.0 ** 40) / 2.0 ** 40
        gx = torch.zeros(xs.shape[0], c_in, dtype=F64)
        gx.index_add_(0, lay.src, e)
        out["x"] = gx
    else:
        out["x"] = None
    return out


def max_rel(got: torch.Tensor, want: torch.Tensor, scale: Optional[float] = None) -> float:
    """max |got - want| over max |want| (or over `scale`)."""
    got, want = got.detach().to(F64).cpu(), want.detach().to(F64).cpu()
    s = float(want.abs().max()) if scale is None else float(scale)
    return float((got - want).abs().max()) / max(s, 1e-300)


def grad_errors(got: Dict[str, torch.Tensor], want: Dict[str, torch.Tensor], training: bool) -> Dict[str, float]:
    """Per-gradient max-abs error relative to the tensor's maximum.  Biases feeding a train-mode BatchNorm are zero in
    theory: they are measured against the maximum of their layer's weight gradient instead."""
    errs = {}
    for k in GRAD_NAMES:
        if got.get(k) is None or want.get(k) is None:
            continue
        if training and k in ("b1", "b2"):
            errs[k] = max_rel(got[k], want[k], scale=float(want["w" + k[1]].abs().max()))
        else:
            errs[k] = max_rel(got[k], want[k])
    return errs


def with_rounding(**kw) -> Rounding:
    return replace(ROUND_ALL, **kw)
