"""The 16-bit set-abstraction kernels layer by layer against the decision-pinned float64 reference (oracle/sa_pinned.py),
fed the kernels' own saved state: stored zhat / a in fp16 ulps, BatchNorm buffers and running statistics, out / arg,
the layer-1 operand, and every gradient with all roundings emulated.  Each case also proves that its bounds separate
the injected faults M1-M5 from real kernel noise at that shape.  Tolerances: oracle/sa_pinned.py GPU_TOL."""
import pytest
import torch

from oracle import ref
from oracle import sa_pinned as sp
from dl_biomass_b200 import sa
from dl_biomass_b200.data import Batch, synthetic_clouds
from dl_biomass_b200.pointnet2_regressor import MLP

pytestmark = pytest.mark.gpu
F64 = torch.float64
TOL = sp.GPU_TOL


def saved_state(out):
    """_SAFunction's saved tensors by name, on the CPU.  A change to its save list fails here."""
    saved = out.grad_fn.saved_tensors
    assert len(saved) == len(sp.SAVED_NAMES) == 31, len(saved)
    return {k: (None if t is None else t.detach().cpu().clone()) for k, t in zip(sp.SAVED_NAMES, saved)}


def _mlp_pair(chans, seed, dev):
    mref = ref.seeded_init_(ref.MLPRef(chans, act="ReLU"), seed)
    m = MLP(chans, act="ReLU")
    m.load_state_dict(mref.state_dict())
    return m.to(dev)


def _grads(m, xg):
    g = {}
    for i in range(3):
        g[f"w{i + 1}"], g[f"b{i + 1}"] = m.lins[i].weight.grad, m.lins[i].bias.grad
    for i in range(2):
        g[f"gamma{i + 1}"], g[f"beta{i + 1}"] = m.norms[i].weight.grad, m.norms[i].bias.grad
    g["x"] = None if xg is None else xg.grad
    return {k: (None if v is None else v.detach().cpu()) for k, v in g.items()}


def _ulp_err(got, want):
    """max |got - want| in fp16 ulps of want (ulp floored at that of 2^-10: fp32 evaluation noise of values near 0)."""
    return float(((got.to(F64) - want).abs() / sp.ulp16(want.abs().clamp_min(2.0 ** -10))).max())


class Report:
    def __init__(self, name):
        self.name, self.rows = name, []

    def add(self, what, value, bound, sep=None):
        self.rows.append((what, float(value), float(bound), sep))

    def finish(self, check=True):
        print(f"\n[{self.name}]")
        for what, v, b, sep in self.rows:
            s = "" if sep is None else f"  nearest fault moving it {sep:8.1f}x tol"
            print(f"  {what:<14} {v:11.3e}  bound {b:9.2e}{s}")
        bad = [(w, v, b) for w, v, b, _ in self.rows if not v <= b]
        if check:
            assert not bad, (self.name, bad)
        return bad


def _slots_problem(c_in, chans, K, B, n, r, seed, dev):
    b = Batch.from_data_list(synthetic_clouds(seed, B, n, max(c_in, 1), True))
    x = None if c_in == 0 else torch.randn(b.pos.size(0), c_in, generator=torch.Generator().manual_seed(seed + 1))
    idx = ref.fps_ref(b.pos, b.ptr, 0.2)
    qptr = ref.sample_ptr(b.ptr, 0.2)
    nbr, cnt = ref.ball_query_ref(b.pos, b.pos[idx], b.ptr, qptr, r, K)
    return x, b.pos, b.pos[idx].contiguous(), nbr, cnt


def _crafted_problem(c_in, n_dst, cnt_fn, K, seed):
    """Targets with chosen neighbour counts: the compacted row count is set by construction."""
    g = torch.Generator().manual_seed(seed)
    n_src = 4 * n_dst + 64
    pos = torch.randn(n_src, 3, generator=g) * 2
    x = None if c_in == 0 else torch.randn(n_src, c_in, generator=g)
    nbr = torch.full((n_dst, K), -1, dtype=torch.int32)
    cnts = [cnt_fn(m) for m in range(n_dst)]
    for m, c in enumerate(cnts):
        nbr[m, :c] = torch.randperm(n_src, generator=g)[:c].sort().values.to(torch.int32)
    return x, pos, torch.randn(n_dst, 3, generator=g), nbr, torch.tensor(cnts, dtype=torch.int32)


def run_level(name, dev, *, c_in, chans, K, problem, clouds=None, train=True, deterministic=False, sm_limit=0,
              seed=3, mutations=True, gout_scale=1.0):
    """One level of a standalone MLP through sa_apply(PREC_BF16) + backward, checked against the pinned reference."""
    m = _mlp_pair(chans, seed, dev)
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
    with sa.options(sm_limit=sm_limit, deterministic=deterministic):
        out, arg = sa.sa_apply(m, xg, *args, seg_mode=seg, K=K, n_dst=n_dst, precision=sa.PREC_BF16)
        st = saved_state(out)
        gout = torch.randn(out.shape, generator=torch.Generator().manual_seed(seed + 2)) * gout_scale
        out.backward(gout.to(dev))
    torch.cuda.synchronize()
    got = _grads(m, xg)
    return check_level(name, st, before, out.detach().cpu(), gout, got, chans=chans, train=train, n_dst=n_dst, K=K,
                       clouds=clouds is not None, mutations=mutations)


def check_level(name, st, before, out, gout, got, *, chans, train, n_dst, K, clouds, mutations=True):
    """Pin one level: `st` its saved state (saved_state), `before` its BatchNorm buffers before the call (names of
    MLP.named_buffers), `out` its output, `gout` the gradient that reached it, `got` the gradients it produced
    (_grads keys; "x" may be the gradient the previous level received)."""
    rep = Report(name)
    kw = dict(training=train, relu=True, n_dst=n_dst, K=K)
    # the forward is pinned against the buffers as they were BEFORE the call
    st_pre = dict(st)
    for l in (1, 2):
        st_pre[f"rm{l}"], st_pre[f"rv{l}"] = before[f"norms.{l - 1}.running_mean"], before[f"norms.{l - 1}.running_var"]
    fw = sp.pinned_forward(st_pre, eps=1e-5, momentum=0.1, **kw)
    lay = fw["layout"]
    cmax = max(chans[1], chans[2])
    assert st["bn"].shape == (2, 4, cmax)
    # ---- forward, stored tensors
    for l in (1, 2):
        zs = st[f"h{l}"][:, lay.V].t()
        rep.add(f"z{l} ulp", _ulp_err(zs.to(F64), fw[f"z{l}"]), TOL["z_ulp"])
        a_st = st[f"a{l}"]
        if a_st is not None:
            rep.add(f"a{l} ulp", _ulp_err(a_st[:, lay.V].t().to(F64), fw[f"a{l}"]), TOL["a_ulp"])
            inval = torch.ones(lay.rows_used, dtype=torch.bool)
            inval[lay.V] = False
            rep.add(f"a{l} invalid", float(a_st[:, : lay.rows_used][:, inval].abs().max()) if inval.any() else 0.0, 0.0)
        c = chans[l]
        bn = st["bn"][l - 1].to(F64)
        ga, be = st[f"gamma{l}"].to(F64), st[f"beta{l}"].to(F64)
        scale = ga * fw[f"rstd{l}"]          # the weight of the BatchNorm backward (bn_bwd_apply) ...
        shift = be - fw[f"mean{l}"] * scale  # ... and the folded affine of the evaluation kernel
        rep.add(f"bn{l} mean", sp.max_rel(bn[0, :c], fw[f"mean{l}"]), 1e-5)
        rep.add(f"bn{l} rstd", sp.max_rel(bn[1, :c], fw[f"rstd{l}"]), 1e-5)
        rep.add(f"bn{l} scale", sp.max_rel(bn[2, :c], scale), 1e-5)
        rep.add(f"bn{l} shift", sp.max_rel(bn[3, :c], shift), 1e-5)
        if train:
            rep.add(f"run_mean{l}", sp.max_rel(st[f"rm{l}"], fw[f"run_mean{l}"]), 1e-6)
            rep.add(f"run_var{l}", sp.max_rel(st[f"rv{l}"], fw[f"run_var{l}"]), 1e-6)
    o = out.to(F64)
    ar = lay.arg_rows(st["arg"])
    has = ar >= 0
    v3 = fw["v3"]
    at_arg = torch.where(has, v3.gather(0, ar.clamp_min(0)), torch.zeros_like(o))
    oscale = float(fw["out"].abs().max())
    rep.add("out@arg", float((o - at_arg).abs().max()) / oscale, 1e-5)
    rep.add("arg maximiser", float((fw["out"] - at_arg).abs().max()) / oscale, 1e-5)
    # exact ties in the reference: the kernel names the lowest slot
    ties = torch.zeros_like(has)
    if v3.shape[0]:
        nmax = torch.zeros(o.shape, dtype=torch.int64).scatter_add_(
            0, lay.cent[:, None].expand_as(v3), (v3 == fw["out"][lay.cent]).long())
        ties = nmax > 1
    rep.add("tie -> lowest", float((ties & (st["arg"].long() != fw["arg"])).sum()), 0)
    if st["g1"] is not None and st["xs"] is not None and st["xs"].dtype == torch.float32:
        G = st["g1"][:, lay.V].to(F64)
        ci = st["xs"].shape[1]
        xr = G[:ci] + G[ci:2 * ci]
        xw = st["xs"][lay.src].t().to(F64)
        rep.add("g1 x hi+lo", float(((xr - xw).abs() / xw.abs().clamp_min(0.25)).max()), 2.0 ** -21)
    if st["g1"] is not None:
        G = st["g1"][:, lay.V].to(F64)
        nx = G.shape[0] - 7
        d = (st["pos_src"][lay.src] - st["pos_dst"][lay.cent]).t().to(F64)
        dr = G[nx:nx + 3] + G[nx + 3:nx + 6]
        rep.add("g1 dpos hi+lo", float(((dr - d).abs() / d.abs().clamp_min(0.25)).max()), 2.0 ** -21)
    # ---- backward: against the exact sums (deterministic mode too: its fixed-point rounding must stay in tolerance)
    want = sp.pinned_backward(st, gout, **kw)
    errs = sp.grad_errors(got, want, train)
    mut = {}
    if mutations:
        for mu in ("M1", "M2", "M3", "M4", "M5"):
            if (not train and mu in ("M1", "M2")) or (clouds and mu == "M2"):
                continue      # eval mode: no batch statistics; CLOUDS levels: every row is an edge
            bad = sp.pinned_backward(st, gout, mutate=mu, **kw)
            if max(e / TOL[k] for k, e in sp.grad_errors(bad, want, train).items()) < 3.0:
                continue      # the fault does not show at this state (e.g. M3 with beta = 0): nothing to separate
            mut[mu] = sp.grad_errors(got, bad, train)
    for k, e in errs.items():
        # this tensor's distance from the nearest fault that moves it beyond the kernel's own error, in tolerances
        moved = [m[k] / TOL[k] for m in mut.values() if m[k] > 2 * e]
        rep.add(f"d{k}", e, TOL[k], min(moved) if moved else None)
    for mu, e in mut.items():
        rep.add(f"{mu} sep (1/x)", 3.0 / max(e[k] / TOL[k] for k in e), 1.0)   # kernel > 3x tolerance from every fault
    for k, v in got.items():
        if v is not None:
            assert torch.isfinite(v).all(), k
    rep.got, rep.state, rep.want = got, st, want
    return rep


# every case reaches a distinct code path (csrc/sa_chain.cuh, csrc/sa_tc.cu)
SLOTS_CASES = {
    # first reference level: unrolled chained instances, dup64 weight images, split (hi+lo) input, grad_x scatter
    "ref_l1": dict(c_in=1, chans=[4, 64, 64, 128], K=64, B=3, n=600, r=2.5),
    # second reference level: unrolled chained instances, fp16 features, dW MTA=2
    "ref_l2": dict(c_in=128, chans=[131, 128, 128, 256], K=64, B=3, n=600, r=2.5),
    # run-time-shaped chained instances
    "chain_rt": dict(c_in=8, chans=[11, 64, 128, 256], K=40, B=3, n=600, r=2.5),
    # multi-pass forward (not chain-eligible), LineFillK X sides of dW
    "multipass": dict(c_in=16, chans=[19, 32, 48, 40], K=16, B=3, n=600, r=2.5),
    # c3 = 42: the routed gradient's scalar (non-quad) loads
    "scalar_route": dict(c_in=4, chans=[7, 32, 32, 42], K=16, B=3, n=600, r=2.5),
    # no features: c_in = 0, no grad_x
    "no_feat": dict(c_in=0, chans=[3, 64, 64, 128], K=32, B=3, n=600, r=2.5),
}


@pytest.mark.parametrize("case", list(SLOTS_CASES))
def test_pinned_slots_level(cuda_device, case):
    c = dict(SLOTS_CASES[case])
    prob = _slots_problem(c["c_in"], c["chans"], c["K"], c["B"], c["n"], c["r"], 21, cuda_device)
    if c["c_in"] > 16:   # wide feature maps enter as fp16
        prob = (prob[0].half().float(),) + prob[1:]
    run_level(case, cuda_device, c_in=c["c_in"], chans=c["chans"], K=c["K"], problem=prob).finish()


@pytest.mark.parametrize("case,opts", [
    ("ref_l1", dict(train=False)),             # eval-mode BatchNorm with a backward: sbar = 0, running statistics
    ("ref_l1", dict(deterministic=True)),      # fixed-order dW reduction + fixed-point grad_x
    ("ref_l2", dict(deterministic=True)),
    ("ref_l2", dict(sm_limit=3)),              # few persistent CTAs: rings and parities wrap many times
    ("multipass", dict(sm_limit=3)),
])
def test_pinned_slots_options(cuda_device, case, opts):
    c = dict(SLOTS_CASES[case])
    prob = _slots_problem(c["c_in"], c["chans"], c["K"], c["B"], c["n"], c["r"], 21, cuda_device)
    if c["c_in"] > 16:
        prob = (prob[0].half().float(),) + prob[1:]
    name = case + "/" + ",".join(f"{k}={v}" for k, v in opts.items())
    run_level(name, cuda_device, c_in=c["c_in"], chans=c["chans"], K=c["K"], problem=prob, **opts).finish()


@pytest.mark.parametrize("n_dst,tail", [(160, "rows = 20 x 64, last 128-row tile full"),
                                        (161, "rows = 21 x 64, last 128-row tile half used"),
                                        (159, "rows = 20 x 64, last group of the last tile short")])
def test_pinned_row_count_near_tile_multiple(cuda_device, n_dst, tail):
    # 8 targets of <= 8 neighbours fill one 64-row block: the row count in use follows n_dst
    prob = _crafted_problem(1, n_dst, lambda m: 8 if (m % 5) else 7, 64, 31)
    run_level(f"rows/{n_dst}", cuda_device, c_in=1, chans=[4, 64, 64, 128], K=64, problem=prob).finish()


def _clouds_problem(sizes, c_in, seed):
    g = torch.Generator().manual_seed(seed)
    n = sum(sizes)
    x = torch.randn(n, c_in, generator=g).half().float()
    pos = torch.randn(n, 3, generator=g) * 3
    batch = torch.repeat_interleave(torch.arange(len(sizes)), torch.tensor(sizes))
    return x, pos, batch


@pytest.mark.parametrize("sizes,chans", [([130, 1, 257, 64], [35, 64, 96, 200]),      # a cloud of one row
                                         ([500] * 12, [259, 256, 512, 1024])])        # the reference's global level
def test_pinned_clouds_level(cuda_device, sizes, chans):
    prob = _clouds_problem(sizes, chans[0] - 3, 5)
    run_level(f"clouds/{chans[3]}", cuda_device, c_in=chans[0] - 3, chans=chans, K=0, problem=prob,
              clouds=len(sizes), seed=9).finish()


def test_pinned_headline_levels(cuda_device):
    """Level 1 of 4 x 10 000 points, and a level-2 call on the geometry that follows it (level 1's sampled points, FPS
    and ball query) with random non-negative fp16 features in place of level 1's output.  The real hand-over of level
    1's fp16 output is pinned in test_pinned_net_train_step_per_level."""
    b = Batch.from_data_list(synthetic_clouds(4321, 4, 10000, 1, False))
    idx = ref.fps_ref(b.pos, b.ptr, 0.2)
    qptr = ref.sample_ptr(b.ptr, 0.2)
    nbr, cnt = ref.ball_query_ref(b.pos, b.pos[idx], b.ptr, qptr, 2.0, 64)
    pos1 = b.pos[idx].contiguous()
    run_level("headline_l1", cuda_device, c_in=1, chans=[4, 64, 64, 128], K=64,
              problem=(b.x, b.pos, pos1, nbr, cnt), mutations=False).finish()
    idx2 = ref.fps_ref(pos1, qptr, 0.25)
    qptr2 = ref.sample_ptr(qptr, 0.25)
    nbr2, cnt2 = ref.ball_query_ref(pos1, pos1[idx2], qptr, qptr2, 8.0, 64)
    x2 = torch.randn(pos1.shape[0], 128, generator=torch.Generator().manual_seed(4)).abs().half().float()
    run_level("headline_l2", cuda_device, c_in=128, chans=[131, 128, 128, 256], K=64,
              problem=(x2, pos1, pos1[idx2].contiguous(), nbr2, cnt2), mutations=False).finish()


@pytest.mark.parametrize("deterministic", [False, True])
def test_unused_tail_is_never_read(cuda_device, monkeypatch, deterministic):
    """Every floating-point buffer the level allocates (sa.py's torch.empty / empty_like: h1, h2, a1, a2, g1, bn, out,
    the gradients) starts as NaN.  The forward writes whole 128-row tiles: up to round_up(num_rows[0], 128) the stored
    tensors must be finite (a and g1 zero past the valid rows); rows past the last tile in use stay unwritten and must
    never be read: every gradient finite and, in deterministic mode, bit-identical to a run on clean buffers.  Only
    floating-point data is poisoned; index tensors are left alone."""
    c = SLOTS_CASES["ref_l1"]
    x, pos_src, pos_dst, nbr, cnt = _slots_problem(c["c_in"], c["chans"], c["K"], 3, 600, 2.5, 21, cuda_device)
    dev = cuda_device
    real_empty, real_empty_like = torch.empty, torch.empty_like

    def nan_empty(*a, **k):
        t = real_empty(*a, **k)
        return t.fill_(float("nan")) if t.is_floating_point() else t

    def nan_empty_like(*a, **k):
        t = real_empty_like(*a, **k)
        return t.fill_(float("nan")) if t.is_floating_point() else t

    res = []
    for poison in (False, True):
        m = _mlp_pair(c["chans"], 3, dev)
        xg = x.to(dev).requires_grad_(True)
        with sa.options(deterministic=deterministic):
            if poison:
                monkeypatch.setattr(torch, "empty", nan_empty)
                monkeypatch.setattr(torch, "empty_like", nan_empty_like)
            out, _ = sa.sa_apply(m, xg, pos_src.to(dev), pos_dst.to(dev), nbr.to(dev), cnt.to(dev), None,
                                 seg_mode=sa.SEG_SLOTS, K=c["K"], n_dst=pos_dst.shape[0], precision=sa.PREC_BF16)
            saved = dict(zip(sp.SAVED_NAMES, out.grad_fn.saved_tensors))
            used = int(saved["num_rows"][0])
            tiles_end = (used + 127) // 128 * 128
            for k in ("h1", "h2", "a1", "a2", "g1"):
                t = saved[k]
                assert t is not None and tiles_end <= t.shape[1], k
                assert torch.isfinite(t[:, :tiles_end]).all(), k      # every row of every tile in use was written
                if k != "h1" and k != "h2":
                    valid = torch.zeros(tiles_end, dtype=torch.bool, device=dev)
                    rs = saved["row_src"][:tiles_end]
                    valid[: rs.numel()] = rs >= 0
                    body = t[:-1] if k == "g1" else t               # g1's last line is the ones line
                    assert torch.all(body[:, :tiles_end][:, ~valid] == 0), k
            assert torch.isfinite(out).all() and torch.isfinite(saved["bn"]).all()
            out.backward(torch.randn(out.shape, generator=torch.Generator().manual_seed(2)).to(dev))
            torch.cuda.synchronize()
            monkeypatch.undo()
        res.append(_grads(m, xg))
    for k, v in res[1].items():
        assert torch.isfinite(v).all(), k
        if deterministic:
            assert torch.equal(v, res[0][k]), k


def test_deterministic_grad_x_accumulator_range(cuda_device):
    """grad_out scaled by 2^s: the deterministic grad_x (64-bit fixed point, unit 2^-40, include/b2pn.h) stays within
    tolerance of the EXACT pinned sums (no fixed-point rounding in the reference) from 2^-24 to 2^12.  The addends a
    real training step produces are measured in test_pinned_net_train_step_per_level."""
    c = SLOTS_CASES["ref_l2"]
    prob = _slots_problem(c["c_in"], c["chans"], c["K"], 3, 600, 2.5, 21, cuda_device)
    prob = (prob[0].half().float(),) + prob[1:]
    for s in (-24, -16, -8, 0, 8, 12):
        rep = run_level(f"fixed/2^{s}", cuda_device, c_in=c["c_in"], chans=c["chans"], K=c["K"], problem=prob,
                        deterministic=True, mutations=False, gout_scale=2.0 ** s)
        if s == 0:   # the per-row addends of the scatter (dh1 W1^T) at unit scale
            add = (rep.want["dz1"] @ sp.bf16(rep.state["w1"][:, : c["c_in"]])).abs()
            nz = add[add > 0]
            print(f"\n  grad_x addends at unit grad_out scale: min {float(nz.min()):.3e} max {float(nz.max()):.3e}")
        rep.finish()


@pytest.mark.parametrize("deterministic", [False, True])
def test_pinned_net_train_step_per_level(cuda_device, monkeypatch, deterministic):
    """One bf16 Net train step at 3 x 640 points, each level pinned with the gradient that really reached it: the
    precomputed grouping and layer-1 operand of net.sample() (the forward does not build g1), the fp16 hand-over of
    each level's output to the next (x_bf16), and gradients written into the ParamArena of make_optimizer(net).
    The feature gradient of level 2 (3) is what level 1 (2) received."""
    from dl_biomass_b200.optim import ParamArena
    from dl_biomass_b200.pointnet2_regressor import Net
    from dl_biomass_b200.train import make_optimizer
    dev = cuda_device
    b = Batch.from_data_list(synthetic_clouds(4321, 3, 640, 1, True)).to(dev)
    net = ref.seeded_init_(Net(1, "ReLU", 0, 0.0, precision="bf16"), seed=7)   # gamma != 1, beta != 0
    net = net.to(dev).set_random_start(False)
    net.train()
    opt = make_optimizer(net)
    arena = ParamArena.of(net)
    assert arena is not None
    levels = []
    real = sa.sa_apply

    def spy(mlp, x, *args, **kw):
        before = {k: v.detach().cpu().clone() for k, v in mlp.named_buffers()}
        res = real(mlp, x, *args, **kw)
        out = res[0]
        lv = dict(mlp=mlp, before=before, state=saved_state(out), out=out.detach().cpu().clone(), kw=kw,
                  has_rowmap=kw.get("rowmap") is not None, has_l1op=kw.get("l1op") is not None,
                  has_x16=kw.get("x_bf16") is not None)
        out.register_hook(lambda g, lv=lv: lv.__setitem__("dout", g.detach().cpu().clone()))
        levels.append(lv)
        return res

    monkeypatch.setattr(sa, "sa_apply", spy)
    with sa.options(deterministic=deterministic):
        samp = net.sample(b)
        opt.zero_grad(set_to_none=True)
        loss = ref.weighted_mse(net(b, sampling=samp), b.y)
        loss.backward()
        torch.cuda.synchronize()
    monkeypatch.undo()
    assert len(levels) == 3
    assert levels[0]["has_rowmap"] and levels[0]["has_l1op"] and levels[0]["state"]["g1"] is not None
    assert levels[1]["has_x16"] and levels[2]["has_x16"]
    assert levels[1]["state"]["xs"].dtype == torch.float16 and levels[2]["state"]["xs"].dtype == torch.float16
    failed = []
    for i, lv in enumerate(levels):
        mlp = lv["mlp"]
        for p in mlp.parameters():      # the backward wrote straight into the arena
            assert p.grad is not None and p.grad.data_ptr() == arena.grad_views[p].data_ptr()
        got = _grads(mlp, None)
        got["x"] = levels[i - 1]["dout"] if i > 0 else None
        kw = lv["kw"]
        clouds = kw["seg_mode"] == sa.SEG_CLOUDS
        rep = check_level(f"net/level{i + 1}", lv["state"], lv["before"], lv["out"], lv["dout"], got,
                          chans=mlp.channel_list, train=True, n_dst=kw["n_dst"], K=kw["K"], clouds=clouds)
        if i == 1:   # the addends of the level-2 -> level-1 scatter in a real step
            c_in = lv["state"]["xs"].shape[1]
            add = (rep.want["dz1"] @ sp.bf16(lv["state"]["w1"][:, :c_in])).abs()
            nz = add[add > 0]
            lo, med, hi = float(nz.min()), float(nz.median()), float(nz.max())
            print(f"\n  level-2 grad_x addends of a real step: min {lo:.3e} median {med:.3e} max {hi:.3e}")
            rep.add("addend median", 1e-10 / med, 1.0)      # typical addend above the accumulator's accuracy floor
            rep.add("addend max", hi, 2.0 ** 20)             # far from the 2^23 range limit
        failed += rep.finish(check=False)
    assert not failed, failed
