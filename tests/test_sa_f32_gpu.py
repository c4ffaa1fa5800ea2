"""The fp32 set-abstraction kernels (csrc/sa_simt.cu) level by level against the decision-pinned float64 reference
(oracle/sa_f32_pinned.py), fed the kernels' own saved state: stored h1 / h2 (exactly 0 on invalid slots), all four
BatchNorm rows and the running statistics, out and arg (as a decision), and every gradient.  Each case prints its
errors and bounds, how far the nearest injected fault (F1-F7) lies from the kernels in tolerances, and the simt kernel
instances it launched (from the profiler); the last test asserts that every simt kernel of the library ran in some
case.  Tolerances: oracle/sa_f32_pinned.py GPU_TOL."""
import re
import subprocess

import pytest
import torch

from oracle import ref
from oracle import sa_f32_pinned as fp
from dl_biomass_b200 import _lib, sa
from dl_biomass_b200.data import Batch, synthetic_clouds
from dl_biomass_b200.pointnet2_regressor import MLP

F64 = torch.float64
TOL = fp.GPU_TOL

# every kernel of csrc/sa_simt.cu as the symbol table names it (without arguments and spaces); a CPU test checks this
# list against libb2pn.so
SIMT_KERNELS = sorted(
    [f"b2pn::simt::rows_gemm_kernel<{bn},b2pn::simt::{ld},b2pn::simt::{ep}>" for bn in (64, 128) for ld, ep in (
        ("GatherLoader", "StoreStatsEp"), ("BnActLoader", "StoreStatsEp"), ("BnActLoader", "SlotMaxEp"),
        ("BnActLoader", "CloudMaxEp"), ("ArgGradLoader", "MaskStoreSumsEp"), ("PlainLoader", "MaskStoreSumsEp"),
        ("PlainLoader", "ScatterEp"))]
    + [f"b2pn::simt::dw_gemm_kernel<b2pn::simt::{y},b2pn::simt::WithOnes<b2pn::simt::{a}>>" for y, a in (
        ("ArgGradLoader", "BnActLoader"), ("PlainLoader", "BnActLoader"), ("PlainLoader", "GatherLoader"))]
    + [f"b2pn::simt::{k}" for k in ("unpack_keys_kernel", "dw_reduce_kernel", "transpose_kernel", "set_double_kernel",
                                     "count_valid_kernel", "bn_fwd_finalize_kernel", "bn_bwd_finalize_kernel",
                                     "bn_bwd_apply_kernel")])

SEEN = set()        # simt kernels launched by the cases of this file so far


def kernel_key(name: str) -> str:
    """A kernel's demangled name without return type, arguments and spaces."""
    name = name.split("(")[0].replace(" ", "")
    return name[4:] if name.startswith("void") else name


def simt_symbols(lib_path: str):
    """The simt kernels in the library's symbol table (nm -C)."""
    out = subprocess.run(["nm", "-C", lib_path], capture_output=True, text=True, check=True).stdout
    keys = set()
    for line in out.splitlines():
        m = re.match(r"^[0-9a-f]+ [TtWw] (.*)$", line)
        if m and "b2pn::simt::" in m.group(1):
            k = kernel_key(m.group(1))
            if k.startswith("b2pn::simt::") and k.split("<")[0].endswith("_kernel"):
                keys.add(k)
    return keys


def _profiled(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    names = {kernel_key(e.name) for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA}
    simt = {n for n in names if n.startswith("b2pn::simt::")}
    SEEN.update(simt)
    return res, simt


def saved_state(out):
    saved = out.grad_fn.saved_tensors
    assert len(saved) == len(fp.SAVED_NAMES) == 31, len(saved)
    st = {k: (None if t is None else t.detach().cpu().clone()) for k, t in zip(fp.SAVED_NAMES, saved)}
    assert all(st[k] is None for k in ("rgrp", "row_src", "num_rows", "row_valid", "a1", "a2", "g1"))
    return st


def _mlp(chans, seed, dev, act="ReLU"):
    mref = ref.seeded_init_(ref.MLPRef(chans, act="ReLU"), seed)
    m = MLP(chans, act=act)
    m.load_state_dict(mref.state_dict())
    return m.to(dev)


def _grads(m, xg):
    g = {}
    for i in range(3):
        g[f"w{i + 1}"], g[f"b{i + 1}"] = m.lins[i].weight.grad, m.lins[i].bias.grad
    for i in range(2):
        g[f"gamma{i + 1}"], g[f"beta{i + 1}"] = m.norms[i].weight.grad, m.norms[i].bias.grad
    g["x"] = None if xg is None else xg.grad
    return {k: (None if v is None else v.detach().cpu().clone()) for k, v in g.items()}


class Report:
    def __init__(self, name):
        self.name, self.rows, self.kernels = name, [], set()

    def add(self, what, value, bound, sep=None):
        self.rows.append((what, float(value), float(bound), sep))

    def finish(self, check=True):
        print(f"\n[{self.name}]")
        for what, v, b, sep in self.rows:
            s = "" if sep is None else f"  nearest fault {sep[0]} at {sep[1]:9.1f}x tol"
            print(f"  {what:<14} {v:11.3e}  bound {b:9.2e}{s}")
        for k in sorted(self.kernels):
            print(f"  kernel {k}")
        bad = [(w, v, b) for w, v, b, _ in self.rows if not v <= b]
        if check:
            assert not bad, (self.name, bad)
        return bad


def check_level(name, st, before, out, gout, got, *, chans, train, relu, n_dst, K, kernels=(), zero_b3=False):
    """Pin one fp32 level: `st` its saved state, `before` its BatchNorm buffers before the call, `out` its output,
    `gout` the gradient that reached it, `got` the gradients it produced (`x` may be what the previous level
    received).  zero_b3: `gout` has vanishing column sums (fp.grad_errors)."""
    rep = Report(name)
    rep.kernels = set(kernels)
    kw = dict(training=train, relu=relu, n_dst=n_dst, K=K)
    st_pre = dict(st)
    for l in (1, 2):
        st_pre[f"rm{l}"], st_pre[f"rv{l}"] = before[f"norms.{l - 1}.running_mean"], before[f"norms.{l - 1}.running_var"]
    fw = fp.pinned_forward(st_pre, eps=1e-5, momentum=0.1, **kw)
    lay = fw["layout"]
    cmax = max(chans[1], chans[2])
    assert st["bn"].shape == (2, 4, cmax)
    assert st["h1"].shape == (lay.rows, chans[1]) and st["h2"].shape == (lay.rows, chans[2])
    # ---- forward
    kern = {"out": out.to(F64)}
    for l in (1, 2):
        kern[f"h{l}"] = lay.stored(st[f"h{l}"])
        kern[f"bn{l}"] = st["bn"][l - 1, :, : chans[l]].to(F64)
        if train:
            kern[f"run_mean{l}"], kern[f"run_var{l}"] = st[f"rm{l}"], st[f"rv{l}"]
        inval = torch.ones(lay.rows, dtype=torch.bool)
        inval[lay.R] = False
        rep.add(f"h{l} invalid", float(st[f"h{l}"][inval].abs().max()) if inval.any() else 0.0, 0.0)
    errs = fp.forward_errors(kern, fw, train)
    # ---- arg as a decision: the kernel's row holds the maximum up to tol, and it is the reference's row wherever that
    # leads every other row by more than tol
    v3, arg = fw["v3"], st["arg"].to(torch.int64)
    ar = lay.arg_rows(arg)
    has = fw["arg"] >= 0
    assert torch.equal(arg >= 0, has), "targets with / without rows"
    assert torch.equal(ar >= 0, has), "an arg that names an invalid slot"
    scale = float(fw["out"].abs().max()) if fw["out"].numel() else 1.0
    thr = TOL["arg"] * scale
    at_arg = torch.where(has, v3.gather(0, ar.clamp_min(0)) if v3.shape[0] else torch.zeros_like(fw["out"]),
                         fw["out"])
    rep.add("arg maximiser", float((fw["out"] - at_arg).abs().max()) / scale if has.any() else 0.0, TOL["arg"])
    near = torch.zeros(fw["out"].shape, dtype=torch.int64)
    if v3.shape[0]:
        near.scatter_add_(0, lay.cent[:, None].expand_as(v3), (v3 >= fw["out"][lay.cent] - thr).long())
    rep.add("arg != clear", float(((near == 1) & (arg != fw["arg"])).sum()), 0)
    rep.add("tie -> first", float(fp.tie_errors(arg, fw)), 0)
    # ---- backward
    want = fp.pinned_backward(st, gout, **kw)
    errs.update(fp.grad_errors(got, want, train, zero_b3))
    # ---- faults: each that moves the reference past 3 tolerances must lie more than 3 tolerances from the kernels
    faults = {}
    for f in fp.FAULTS:
        bfw, bbw = fp.with_fault(st_pre, gout, f, eps=1e-5, momentum=0.1, **kw)
        moved = fp.forward_errors(bfw, fw, train)
        moved.update(fp.grad_errors(bbw, want, train, zero_b3))
        moved = {k: v for k, v in moved.items() if k in errs}    # e.g. no x: the fault's grad_x is not checked
        ties = fp.tie_errors(bfw["arg"], fw)
        if max(v / TOL[fp.tol_key(k)] for k, v in moved.items()) < 3.0 and ties == 0:
            continue      # the fault does not show at this state (no split, no tie, no saturated neighbourhood ...)
        dist = fp.forward_errors(kern, bfw, train)
        dist.update(fp.grad_errors(got, bbw, train, zero_b3))
        faults[f] = (dist, ties)
    for k, e in errs.items():
        t = TOL[fp.tol_key(k)]
        near_f = [(f, d[k] / t) for f, (d, _) in faults.items() if d[k] > 2 * e]
        rep.add(k, e, t, min(near_f, key=lambda p: p[1]) if near_f else None)
    for f, (d, ties) in faults.items():
        sep = max(v / TOL[fp.tol_key(k)] for k, v in d.items())
        if ties:      # F6: a wrong tie is a discrete decision the tie check above rejects
            sep = max(sep, float("inf"))
        rep.add(f"{f} sep (1/x)", 3.0 / sep, 1.0)
    for k, v in got.items():
        if v is not None:
            assert torch.isfinite(v).all(), k
    assert torch.isfinite(out).all()
    rep.fw, rep.want = fw, want
    return rep


def run_level(name, dev, *, chans, problem, K, clouds=None, train=True, act="ReLU", seed=3):
    """One level of a standalone MLP through sa_apply(PREC_F32) + backward, pinned against the reference."""
    m = _mlp(chans, seed, dev, act)
    m.train(train)
    if not train:
        with torch.no_grad():
            g = torch.Generator().manual_seed(seed + 7)
            for nm in m.norms:
                nm.running_mean.copy_((torch.rand(nm.running_mean.shape, generator=g) - 0.5).to(dev))
                nm.running_var.copy_((torch.rand(nm.running_var.shape, generator=g) + 0.5).to(dev))
    before = {k: v.detach().cpu().clone() for k, v in m.named_buffers()}
    if clouds is None:
        x, pos_src, pos_dst, nbr, cnt = problem
        n_dst, seg = pos_dst.shape[0], sa.SEG_SLOTS
        args = (pos_src.to(dev), pos_dst.to(dev), nbr.to(dev), cnt.to(dev), None)
    else:
        x, pos_src, batch = problem
        n_dst, seg, K = clouds, sa.SEG_CLOUDS, 0
        args = (pos_src.to(dev), None, None, None, batch.to(dev))
    xg = None if x is None else x.to(dev).requires_grad_(True)
    gout = torch.randn(n_dst, chans[3], generator=torch.Generator().manual_seed(seed + 2))

    def call():
        out, _ = sa.sa_apply(m, xg, *args, seg_mode=seg, K=K, n_dst=n_dst, precision=sa.PREC_F32)
        st = saved_state(out)
        out.backward(gout.to(dev))
        return out, st

    (out, st), kernels = _profiled(call)
    rep = check_level(name, st, before, out.detach().cpu(), gout, _grads(m, xg), chans=chans, train=train,
                      relu=act is not None, n_dst=n_dst, K=K, kernels=kernels)
    rep.module, rep.x = m, xg
    return rep


def _slots_problem(c_in, K, B, n, r, seed):
    b = Batch.from_data_list(synthetic_clouds(seed, B, n, max(c_in, 1), True))
    x = None if c_in == 0 else torch.randn(b.pos.size(0), c_in, generator=torch.Generator().manual_seed(seed + 1))
    idx = ref.fps_ref(b.pos, b.ptr, 0.2)
    qptr = ref.sample_ptr(b.ptr, 0.2)
    nbr, cnt = ref.ball_query_ref(b.pos, b.pos[idx], b.ptr, qptr, r, K)
    return x, b.pos, b.pos[idx].contiguous(), nbr, cnt


def _crafted_problem(c_in, n_dst, cnt_fn, K, seed):
    """Targets with chosen neighbour counts."""
    g = torch.Generator().manual_seed(seed)
    n_src = 4 * n_dst + K + 64
    pos = torch.randn(n_src, 3, generator=g) * 2
    x = None if c_in == 0 else torch.randn(n_src, c_in, generator=g)
    nbr = torch.full((n_dst, K), -1, dtype=torch.int32)
    cnts = [cnt_fn(m) for m in range(n_dst)]
    for m, c in enumerate(cnts):
        nbr[m, :c] = torch.randperm(n_src, generator=g)[:c].sort().values.to(torch.int32)
    return x, pos, torch.randn(n_dst, 3, generator=g), nbr, torch.tensor(cnts, dtype=torch.int32)


def _clouds_problem(sizes, c_in, seed, dup=False):
    g = torch.Generator().manual_seed(seed)
    n = sum(sizes)
    x = torch.randn(n, c_in, generator=g)
    pos = torch.randn(n, 3, generator=g) * 3
    if dup:   # every third row repeats the row before it: exact ties, the first row must win
        x[2::3], pos[2::3] = x[1::3][: x[2::3].shape[0]], pos[1::3][: pos[2::3].shape[0]]
    batch = torch.repeat_interleave(torch.arange(len(sizes)), torch.tensor(sizes))
    return x, pos, batch


# K, channel widths and the GEMM instance each layer reaches (rows_gemm_kernel<64> for N <= 64, <128> above)
SLOTS_CASES = {
    "K8": dict(c_in=1, chans=[4, 32, 48, 40], K=8, B=3, n=600, r=1.5),
    "K16": dict(c_in=16, chans=[19, 32, 48, 42], K=16, B=3, n=600, r=2.0),
    "K32": dict(c_in=0, chans=[3, 64, 64, 64], K=32, B=3, n=600, r=2.5),
    "K64": dict(c_in=128, chans=[131, 128, 128, 200], K=64, B=3, n=600, r=2.5),
}


@pytest.mark.gpu
@pytest.mark.parametrize("case", list(SLOTS_CASES))
def test_f32_slots_level(cuda_device, case):
    c = SLOTS_CASES[case]
    prob = _slots_problem(c["c_in"], c["K"], c["B"], c["n"], c["r"], 21)
    run_level(case, cuda_device, chans=c["chans"], problem=prob, K=c["K"]).finish()


@pytest.mark.gpu
def test_f32_slots_k128_crafted(cuda_device):
    """K = 128: one target per 128-row tile, with empty (cnt = 0) and saturated (cnt = K) neighbourhoods."""
    prob = _crafted_problem(16, 40, lambda m: [0, 128, 1, 77, 128, 8, 9, 127][m % 8], 128, 5)
    run_level("K128", cuda_device, chans=[19, 64, 96, 128], problem=prob, K=128).finish()


@pytest.mark.gpu
@pytest.mark.parametrize("n_dst", [159, 160, 161])
def test_f32_rows_near_tile_multiple(cuda_device, n_dst):
    """n_dst * K = 1272, 1280, 1288 rows: 8 rows short of, exactly at and 8 rows past a 128-row tile edge."""
    prob = _crafted_problem(1, n_dst, lambda m: [8, 3, 0, 5][m % 4], 8, 7)
    run_level(f"rows/{n_dst * 8}", cuda_device, chans=[4, 64, 64, 128], problem=prob, K=8).finish()


@pytest.mark.gpu
def test_f32_two_dw_splits(cuda_device):
    """150 x 32 = 4 800 rows: two dW splits, the second one short; a third of the neighbourhoods saturated."""
    assert fp.dw_splits(150 * 32)[0] == 2
    prob = _crafted_problem(16, 150, lambda m: [32, 17, 32, 5, 32, 0][m % 6], 32, 9)
    run_level("splits=2", cuda_device, chans=[19, 64, 64, 128], problem=prob, K=32).finish()


@pytest.mark.gpu
@pytest.mark.parametrize("sizes,chans,dup", [
    ([130, 1, 0, 3, 5, 257, 64], [15, 32, 48, 40], False),    # one-row clouds, an empty cloud, boundaries in 8-row groups
    ([1, 7, 9, 0, 120, 130, 1, 255], [35, 128, 96, 200], True),  # duplicated rows: exact ties; boundaries across tiles
    ([500] * 12, [259, 256, 512, 1024], False),                # the reference's global level
])
def test_f32_clouds_level(cuda_device, sizes, chans, dup):
    prob = _clouds_problem(sizes, chans[0] - 3, 5, dup)
    rep = run_level(f"clouds/{chans[3]}{'/dup' if dup else ''}", cuda_device, chans=chans, problem=prob, K=0,
                    clouds=len(sizes))
    if dup:
        assert any(r[0] == "F6 sep (1/x)" for r in rep.rows), "the duplicated rows produced no exact tie"
    rep.finish()


@pytest.mark.gpu
@pytest.mark.parametrize("act", ["ReLU", None])
def test_f32_eval_mode(cuda_device, act):
    """Eval-mode BatchNorm with non-trivial running statistics, a backward through it; also without an activation."""
    c = SLOTS_CASES["K16"]
    prob = _slots_problem(c["c_in"], c["K"], c["B"], c["n"], c["r"], 21)
    run_level(f"eval/act={act}", cuda_device, chans=c["chans"], problem=prob, K=c["K"], train=False, act=act).finish()
    sizes = [130, 1, 0, 257]
    run_level(f"eval/clouds/act={act}", cuda_device, chans=[15, 64, 96, 200],
              problem=_clouds_problem(sizes, 12, 6), K=0, clouds=len(sizes), train=False, act=act).finish()


@pytest.mark.gpu
@pytest.mark.parametrize("kind", ["slots", "clouds"])
def test_f32_nan_prefilled_buffers(cuda_device, monkeypatch, kind):
    """Every floating-point buffer sa.py allocates for the level (h1, h2, out, bn, the gradients) starts as NaN, and
    every workspace byte as 0xFF: the results are finite and equal to a run on clean buffers (bit for bit, except the
    SLOTS grad_x, whose scatter adds in arrival order)."""
    dev = cuda_device
    if kind == "slots":
        c = SLOTS_CASES["K16"]
        x, pos_src, pos_dst, nbr, cnt = _slots_problem(c["c_in"], c["K"], c["B"], c["n"], c["r"], 21)
        chans, K, n_dst, seg = c["chans"], c["K"], pos_dst.shape[0], sa.SEG_SLOTS
        args = (pos_src.to(dev), pos_dst.to(dev), nbr.to(dev), cnt.to(dev), None)
    else:
        sizes = [130, 1, 0, 3, 5, 257, 64]
        x, pos_src, batch = _clouds_problem(sizes, 12, 5)
        chans, K, n_dst, seg = [15, 64, 96, 200], 0, len(sizes), sa.SEG_CLOUDS
        args = (pos_src.to(dev), None, None, None, batch.to(dev))
    real_empty, real_empty_like = torch.empty, torch.empty_like

    def poison(t):
        if t.is_floating_point():
            return t.fill_(float("nan"))
        if t.dtype == torch.int32:
            return t.fill_(0x7FFFFFFF)
        return t.fill_(255) if t.dtype == torch.uint8 else t

    res = []
    for poisoned in (False, True):
        m = _mlp(chans, 3, dev)
        xg = x.to(dev).requires_grad_(True)
        if poisoned:
            monkeypatch.setattr(torch, "empty", lambda *a, **k: poison(real_empty(*a, **k)))
            monkeypatch.setattr(torch, "empty_like", lambda *a, **k: poison(real_empty_like(*a, **k)))
        out, arg = sa.sa_apply(m, xg, *args, seg_mode=seg, K=K, n_dst=n_dst, precision=sa.PREC_F32)
        st = saved_state(out)
        out.backward(torch.randn(out.shape, generator=torch.Generator().manual_seed(2)).to(dev))
        torch.cuda.synchronize()
        monkeypatch.undo()
        r = _grads(m, xg)
        # (bn rows past a layer's width are never written nor read)
        r.update(out=out.detach().cpu(), arg=arg.cpu(), h1=st["h1"], h2=st["h2"], bn1=st["bn"][0, :, : chans[1]],
                 bn2=st["bn"][1, :, : chans[2]],
                 rm=m.norms[0].running_mean.cpu(), rv=m.norms[1].running_var.cpu())
        res.append(r)
    for k, v in res[1].items():
        if v.is_floating_point():
            assert torch.isfinite(v).all(), k
        if kind == "slots" and k == "x":
            assert fp.max_rel(v, res[0][k]) <= 1e-6, k
        else:
            assert torch.equal(v, res[0][k]), k


@pytest.mark.gpu
@pytest.mark.parametrize("B,n", [(3, 640), (5, 10000)])
def test_f32_net_train_step_per_level(cuda_device, monkeypatch, B, n):
    """One fp32 Net train step, each level pinned on the inputs and the incoming gradient it really received.  At
    5 x 10 000 points level 1 has 10 000 x 64 = 640 000 rows: the dW GEMMs run at their 296-split cap."""
    from dl_biomass_b200.pointnet2_regressor import Net
    dev = cuda_device
    b = Batch.from_data_list(synthetic_clouds(4321, B, n, 1, True)).to(dev)
    net = ref.seeded_init_(Net(1, "ReLU", 0, 0.0, precision="fp32"), seed=7).to(dev).set_random_start(False)
    net.train()
    levels = []
    real = sa.sa_apply

    def spy(mlp, x, *args, **kw):
        before = {k: v.detach().cpu().clone() for k, v in mlp.named_buffers()}
        res = real(mlp, x, *args, **kw)
        out = res[0]
        lv = dict(mlp=mlp, before=before, state=saved_state(out), out=out.detach().cpu().clone(), kw=kw)
        out.register_hook(lambda g, lv=lv: lv.__setitem__("dout", g.detach().cpu().clone()))
        levels.append(lv)
        return res

    monkeypatch.setattr(sa, "sa_apply", spy)
    net.zero_grad(set_to_none=True)

    def step():
        ref.weighted_mse(net(b), b.y).backward()

    _, kernels = _profiled(step)
    monkeypatch.undo()
    assert len(levels) == 3
    if n == 10000:
        assert fp.dw_splits(levels[0]["kw"]["n_dst"] * levels[0]["kw"]["K"])[0] == 296
    failed = []
    for i, lv in enumerate(levels):
        mlp = lv["mlp"]
        got = _grads(mlp, None)
        got["x"] = levels[i - 1]["dout"] if i > 0 else None
        kw = lv["kw"]
        rep = check_level(f"net{B}x{n}/level{i + 1}", lv["state"], lv["before"], lv["out"], lv["dout"], got,
                          chans=mlp.channel_list, train=True, relu=True, n_dst=kw["n_dst"], K=kw["K"],
                          kernels=kernels if i == 0 else (), zero_b3=True)
        failed += rep.finish(check=False)
    assert not failed, failed


@pytest.mark.gpu
def test_f32_every_simt_kernel_ran():
    """Runs last: every simt kernel of the library was launched by some case of this file."""
    if not SEEN:
        pytest.skip("no case of this file ran before this one")
    missing = sorted(set(SIMT_KERNELS) - SEEN)
    print("\nsimt kernels launched:", len(SEEN & set(SIMT_KERNELS)), "of", len(SIMT_KERNELS))
    for k in sorted(SEEN):
        print("  ", k)
    assert not missing, missing
    assert SEEN <= set(SIMT_KERNELS), sorted(SEEN - set(SIMT_KERNELS))


def test_simt_kernel_list_matches_library():
    """CPU: SIMT_KERNELS is exactly the set of simt kernels libb2pn.so contains."""
    _lib.build()
    assert simt_symbols(_lib.LIB_PATH) == set(SIMT_KERNELS)
