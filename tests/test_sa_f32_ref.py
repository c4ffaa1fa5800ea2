"""The decision-pinned float64 reference of the fp32 set-abstraction kernels (oracle/sa_f32_pinned.py) and the float64
training-mode head reference (oracle/head_ref.py) are right: with the state taken from their own float64 forward they
reproduce torch.autograd through ref.point_conv_ref / GlobalSAModuleRef / BatchNorm1d to 1e-10, and each injected
fault moves some checked tensor by more than 3x its GPU bound.  Which faults the older bounds (1e-4 on outputs, 2e-4 on
gradients, against the fp32 oracle) would let through is printed, not asserted."""
import pytest
import torch
import torch.nn.functional as F

from oracle import head_ref as hr
from oracle import ref
from oracle import sa_f32_pinned as fp

F64 = torch.float64
OLD_OUT, OLD_GRAD = 1e-4, 2e-4


def _params(mlp, st):
    st = dict(st)
    for i in range(3):
        st[f"w{i + 1}"] = mlp.lins[i].weight.detach().clone()
        st[f"b{i + 1}"] = mlp.lins[i].bias.detach().clone()
    for i in range(2):
        st[f"gamma{i + 1}"] = mlp.norms[i].weight.detach().clone()
        st[f"beta{i + 1}"] = mlp.norms[i].bias.detach().clone()
        st[f"rm{i + 1}"] = mlp.norms[i].running_mean.detach().clone()
        st[f"rv{i + 1}"] = mlp.norms[i].running_var.detach().clone()
    return st


def _autograd_grads(mlp, x):
    g = {}
    for i in range(3):
        g[f"w{i + 1}"], g[f"b{i + 1}"] = mlp.lins[i].weight.grad, mlp.lins[i].bias.grad
    for i in range(2):
        g[f"gamma{i + 1}"], g[f"beta{i + 1}"] = mlp.norms[i].weight.grad, mlp.norms[i].bias.grad
    g["x"] = None if x is None else x.grad
    return g


def _slots(c_in, chans, cnts, K, seed, dtype=F64):
    g = torch.Generator().manual_seed(seed)
    n_dst = len(cnts)
    n_src = 2 * K + 3 * n_dst
    pos = torch.randn(n_src, 3, generator=g, dtype=dtype) * 2
    x = None if c_in == 0 else torch.randn(n_src, c_in, generator=g, dtype=dtype)
    pos_dst = torch.randn(n_dst, 3, generator=g, dtype=dtype)
    nbr = torch.full((n_dst, K), -1, dtype=torch.int32)
    for m, c in enumerate(cnts):
        nbr[m, :c] = torch.randperm(n_src, generator=g)[:c].sort().values.to(torch.int32)
    cnt = torch.tensor(cnts, dtype=torch.int32)
    return x, pos, pos_dst, nbr, cnt


def _mlp(chans, seed, train):
    mlp = ref.seeded_init_(ref.MLPRef(chans, act="ReLU"), seed).double()
    mlp.train(train)
    if not train:
        with torch.no_grad():
            for n in mlp.norms:
                n.running_mean.uniform_(-0.5, 0.5)
                n.running_var.uniform_(0.5, 2.0)
    return mlp


@pytest.mark.parametrize("train", [True, False])
@pytest.mark.parametrize("c_in,chans", [(1, [4, 16, 24, 40]), (0, [3, 16, 16, 24]), (20, [23, 32, 16, 24])])
def test_f32_slots_match_autograd_f64(c_in, chans, train):
    K = 16
    cnts = [1, 8, 9, 16, 0, 16, 5, 3]      # one row, one 8-row group, a group and one row, saturated, empty
    x, pos, pos_dst, nbr, cnt = _slots(c_in, chans, cnts, K, 3)
    mlp = _mlp(chans, 4, train)
    st = _params(mlp, {"xs": x, "pos_src": pos, "pos_dst": pos_dst, "nbr": nbr, "cnt": cnt, "batch": None})
    xr = None if x is None else x.clone().requires_grad_(True)
    row, col = ref.slots_to_edges(nbr, cnt)
    want = ref.point_conv_ref(mlp, xr, pos, pos_dst, row, col)
    gout = torch.randn(want.shape, generator=torch.Generator().manual_seed(5), dtype=F64)
    want.backward(gout)
    kw = dict(training=train, relu=True, n_dst=len(cnts), K=K)
    fw = fp.pinned_forward(st, eps=1e-5, momentum=0.1, **kw)
    assert fp.max_rel(fw["out"], want) <= 1e-10
    assert bool((fw["arg"][4] == -1).all()) and bool((fw["out"][4] == 0).all())
    if train:
        for l in (1, 2):
            assert fp.max_rel(fw[f"run_mean{l}"], mlp.norms[l - 1].running_mean) <= 1e-10
            assert fp.max_rel(fw[f"run_var{l}"], mlp.norms[l - 1].running_var) <= 1e-10
    st = fp.state_from_forward(st, fw, chans)
    # the forward from its own stored state reproduces itself
    fw2 = fp.pinned_forward(st, eps=1e-5, momentum=0.1, **kw)
    assert max(fp.forward_errors(fw2, fw, train).values()) <= 1e-12
    got = fp.pinned_backward(st, gout, **kw)
    errs = fp.grad_errors(got, _autograd_grads(mlp, xr), train)
    assert max(errs.values()) <= 1e-10, errs
    assert (xr is None) == (got["x"] is None)


@pytest.mark.parametrize("train", [True, False])
def test_f32_clouds_match_autograd_f64(train):
    g = torch.Generator().manual_seed(5)
    sizes = [130, 1, 0, 257, 64]          # ragged, a cloud of one row, an empty cloud
    n = sum(sizes)
    x = torch.randn(n, 12, generator=g, dtype=F64)
    pos = torch.randn(n, 3, generator=g, dtype=F64) * 3
    batch = torch.repeat_interleave(torch.arange(len(sizes)), torch.tensor(sizes))
    chans = [15, 32, 48, 40]
    mlp = _mlp(chans, 9, train)
    st = _params(mlp, {"xs": x, "pos_src": pos, "pos_dst": None, "nbr": None, "cnt": None, "batch": batch})
    xr = x.clone().requires_grad_(True)
    want, _, _ = ref.GlobalSAModuleRef(mlp)(xr, pos, batch, len(sizes))
    gout = torch.randn(want.shape, generator=g, dtype=F64)
    want.backward(gout)
    kw = dict(training=train, relu=True, n_dst=len(sizes), K=0)
    fw = fp.pinned_forward(st, eps=1e-5, momentum=0.1, **kw)
    assert fp.max_rel(fw["out"], want) <= 1e-10
    assert bool((fw["arg"][2] == -1).all())
    st = fp.state_from_forward(st, fw, chans)
    got = fp.pinned_backward(st, gout, **kw)
    errs = fp.grad_errors(got, _autograd_grads(mlp, xr), train)
    assert max(errs.values()) <= 1e-10, errs


def fault_state(kind):
    """An fp32 level state (reference forward of fp32 inputs, stored as fp32 as the kernels store it) on which every
    fault of its kind shows: SLOTS with saturated and empty neighbourhoods over two dW splits, or CLOUDS with
    duplicated rows (exact ties)."""
    g = torch.Generator().manual_seed(11)
    if kind == "slots":
        K, n_dst = 32, 200                                # 6 400 rows: 3 dW splits
        cnts = torch.randint(0, K + 1, (n_dst,), generator=g)
        cnts[::7] = K
        x, pos, pos_dst, nbr, cnt = _slots(1, None, cnts.tolist(), K, 21, dtype=torch.float32)
        chans = [4, 64, 64, 128]
        st = {"xs": x, "pos_src": pos, "pos_dst": pos_dst, "nbr": nbr, "cnt": cnt, "batch": None}
    else:
        K, sizes = 0, [700, 1, 0, 900, 2500]
        n = sum(sizes)
        x = torch.randn(n, 13, generator=g)
        pos = torch.randn(n, 3, generator=g) * 3
        x[1::5], pos[1::5] = x[0::5][: x[1::5].shape[0]], pos[0::5][: pos[1::5].shape[0]]   # duplicated rows
        batch = torch.repeat_interleave(torch.arange(len(sizes)), torch.tensor(sizes))
        chans, n_dst = [16, 64, 96, 200], len(sizes)
        st = {"xs": x, "pos_src": pos, "pos_dst": None, "nbr": None, "cnt": None, "batch": batch}
    mlp = ref.seeded_init_(ref.MLPRef(chans, act="ReLU"), 12)
    st = {k: (v.float() if (v is not None and v.is_floating_point()) else v) for k, v in _params(mlp, st).items()}
    kw = dict(training=True, relu=True, n_dst=n_dst, K=K)
    fw = fp.pinned_forward(st, eps=1e-5, momentum=0.1, **kw)
    st = fp.state_from_forward(st, fw, chans)
    st = {k: (v.float() if (v is not None and v.is_floating_point()) else v) for k, v in st.items()}
    gout = torch.randn(n_dst, chans[3], generator=g)
    return st, gout, kw


FAULT_KIND = {"F1": "slots", "F2": "slots", "F3": "slots", "F4": "slots", "F5": "slots", "F6": "clouds",
              "F7": "slots"}


def fault_distances(st, gout, kw, fault):
    """Every checked tensor's move under the fault, relative to its maximum (forward_errors / grad_errors), the arg
    tie count, and the largest move in GPU tolerances."""
    fw = fp.pinned_forward(st, eps=1e-5, momentum=0.1, **kw)
    bw = fp.pinned_backward(st, gout, **kw)
    bfw, bbw = fp.with_fault(st, gout, fault, eps=1e-5, momentum=0.1, **kw)
    e = fp.forward_errors(bfw, fw, kw["training"])
    e.update(fp.grad_errors(bbw, bw, kw["training"]))
    ties = fp.tie_errors(bfw["arg"], fw)
    sep = max(v / fp.GPU_TOL[fp.tol_key(k)] for k, v in e.items())
    return e, ties, sep


@pytest.mark.parametrize("fault", fp.FAULTS)
def test_f32_faults_exceed_pinned_bounds(fault):
    st, gout, kw = fault_state(FAULT_KIND[fault])
    e, ties, sep = fault_distances(st, gout, kw, fault)
    old_ok = all(v <= (OLD_OUT if k in ("out", "h1", "h2") or k.startswith("bn") else OLD_GRAD) for k, v in e.items())
    worst = max(e, key=lambda k: e[k] / fp.GPU_TOL[fp.tol_key(k)])
    print(f"{fault}: worst {worst} moved {e[worst]:.3e} = {sep:.1f}x its bound; ties broken wrongly {ties}; "
          f"{'ACCEPTED' if old_ok else 'rejected'} by the old 1e-4 / 2e-4 bounds")
    assert sep > 3.0, (fault, e)
    if fault == "F6":
        assert ties > 0


def test_f32_dw_splits():
    assert fp.dw_splits(2047) == (1, 2048)
    assert fp.dw_splits(4096) == (2, 2048)
    assert fp.dw_splits(640000)[0] == 296 and fp.dw_splits(606208)[0] == 296 and fp.dw_splits(606207)[0] == 295


# ---- head ---------------------------------------------------------------------------------------------------------
def _head_problem(B, chans, p, seed=3):
    g = torch.Generator().manual_seed(seed)
    P = {}
    for l in range(3):
        P[f"w{l}"] = torch.randn(chans[l + 1], chans[l], generator=g, dtype=F64) / chans[l] ** 0.5
        P[f"b{l}"] = torch.randn(chans[l + 1], generator=g, dtype=F64) * 0.1
    for l in range(2):
        P[f"gamma{l}"] = torch.rand(chans[l + 1], generator=g, dtype=F64) + 0.5
        P[f"beta{l}"] = torch.rand(chans[l + 1], generator=g, dtype=F64) - 0.5
        P[f"rm{l}"] = torch.rand(chans[l + 1], generator=g, dtype=F64) * 0.4 - 0.2
        P[f"rv{l}"] = torch.rand(chans[l + 1], generator=g, dtype=F64) * 1.5 + 0.5
    x = torch.randn(B, chans[0], generator=g, dtype=F64)
    masks = [(torch.rand(B, c, generator=g) >= p).to(torch.uint8) for c in chans[1:3]]
    gout = torch.randn(B, chans[3], generator=g, dtype=F64)
    return P, x, masks, gout


@pytest.mark.parametrize("B,p", [(2, 0.0), (5, 0.5), (17, 0.5), (32, 0.0)])
def test_head_ref_matches_autograd_f64(B, p):
    chans = [300, 64, 48, 4]
    P, x, masks, gout = _head_problem(B, chans, p)
    fw = hr.forward(P, x, masks, p)
    Pa = {k: v.clone().requires_grad_(k[0] in "wbg") for k, v in P.items()}
    xa = x.clone().requires_grad_(True)
    rm = [P["rm0"].clone(), P["rm1"].clone()]
    rv = [P["rv0"].clone(), P["rv1"].clone()]
    h = F.linear(xa, Pa["w0"], Pa["b0"])
    for l in (0, 1):
        h = F.batch_norm(h, rm[l], rv[l], Pa[f"gamma{l}"], Pa[f"beta{l}"], True, 0.1, 1e-5)
        h = h * masks[l].to(F64) / (1 - p)
        h = F.linear(h, Pa[f"w{l + 1}"], Pa[f"b{l + 1}"])
    h.backward(gout)
    assert fp.max_rel(fw["out"], h) <= 1e-10
    for l in (0, 1):
        assert fp.max_rel(fw[f"run_mean{l}"], rm[l]) <= 1e-10 and fp.max_rel(fw[f"run_var{l}"], rv[l]) <= 1e-10
    got = hr.backward(P, x, fw, gout, p)
    want = {k: Pa[k].grad for k in hr.GRAD_NAMES if k != "x"}
    want["x"] = xa.grad
    errs = hr.grad_errors(got, want)
    assert max(errs.values()) <= 1e-10, errs


@pytest.mark.parametrize("fault", hr.FAULTS)
def test_head_faults_exceed_pinned_bounds(fault):
    chans, p = [1000, 128, 128, 4], (0.5 if fault == "H3" else 0.0)
    P, x, masks, gout = _head_problem(12, chans, p)
    fw = hr.forward(P, x, masks, p)
    base = hr.backward(P, x, fw, gout, p)
    bfw = hr.forward(P, x, masks, p, fault=fault if fault == "H2" else None)
    bad = hr.backward(P, x, bfw, gout, p, fault=None if fault == "H2" else fault)
    e = hr.grad_errors(bad, base)
    e["out"] = fp.max_rel(bfw["out"], fw["out"])
    sep = max(v / hr.GPU_TOL[k] for k, v in e.items())
    print(fault, {k: f"{v:.2e}" for k, v in e.items()})
    assert sep > 3.0, (fault, e)
