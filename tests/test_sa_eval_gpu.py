"""The evaluation path level by level against the float64 reference of its own roundings (oracle/sa_eval_ref.py): the
single-launch evaluation kernel at each of its instances (csrc/sa_chain.cuh, tc_chain_eval_kernel), the multi-pass
kernels with eval-mode BatchNorm, the fp32 path, the regression head and a whole Net in eval mode.  Every case names
the kernel instance it reached (from the profiler's kernel list), compares `out` in fp16 ulps of the reference, as
max-abs error over max |want| and as rms error over rms |want|, checks the fp16 copy `out16` bit for bit against
fp16(out), and prints how far the nearest injected fault (E1-E7) lies, in tolerances.  Every allocation of the level
starts as NaN.
Tolerances: oracle/sa_eval_ref.py GPU_TOL."""
import ctypes
import re

import pytest
import torch

from oracle import ref
from oracle import sa_eval_ref as er
from dl_biomass_b200 import _lib, head, sa
from dl_biomass_b200.data import Batch, synthetic_clouds
from dl_biomass_b200.pointnet2_regressor import MLP

pytestmark = pytest.mark.gpu
F64 = torch.float64
TOL = er.GPU_TOL
FUSED_L1, FUSED_L2, FUSED_RT = "<1, 1, 1, 1, 1>", "<3, 1, 2, 2, 2>", "<-1, -1, -1, -1, -1>"
MULTIPASS = "multi-pass"


def _launches():
    return int(_lib.lib().b2pn_launch_count())


def _kernel_names(fn):
    """Run fn() under the profiler: (its result, names of the CUDA kernels it launched)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        res = fn()
        torch.cuda.synchronize()
    names = [e.name for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA]
    return res, names


def _instance(names):
    """The tc_chain_eval_kernel instance among the kernels, or MULTIPASS when none ran."""
    found = {m.group(1) for n in names for m in [re.search(r"tc_chain_eval_kernel<([^>]*)>", n)] if m}
    assert len(found) <= 1, found
    return "<" + ", ".join(s.strip() for s in next(iter(found)).split(",")) + ">" if found else MULTIPASS


def _probe_fused(x, chans, K, seg=sa.SEG_SLOTS):
    """b2pn_sa_eval_fused for these shapes, with the probe sa.py builds."""
    c_in = 0 if x is None else x.shape[1]
    p = sa.SaArgs()
    p.precision, p.training, p.seg_mode, p.K, p.c_in = sa.PREC_BF16, 0, seg, K, c_in
    p.x_dtype = 0 if (x is not None and x.dtype == torch.float32 and c_in <= 16) else 1
    for i in range(4):
        p.mlp.c[i] = chans[i]
    return int(_lib.lib().b2pn_sa_eval_fused(ctypes.byref(p)))


@pytest.fixture
def nan_alloc(monkeypatch):
    """A context manager under which every floating-point torch.empty / empty_like starts as NaN."""
    from contextlib import contextmanager
    real_empty, real_empty_like = torch.empty, torch.empty_like

    def nan_empty(*a, **k):
        t = real_empty(*a, **k)
        return t.fill_(float("nan")) if t.is_floating_point() else t

    def nan_empty_like(*a, **k):
        t = real_empty_like(*a, **k)
        return t.fill_(float("nan")) if t.is_floating_point() else t

    @contextmanager
    def poisoned():
        monkeypatch.setattr(torch, "empty", nan_empty)
        monkeypatch.setattr(torch, "empty_like", nan_empty_like)
        try:
            yield
        finally:
            monkeypatch.setattr(torch, "empty", real_empty)
            monkeypatch.setattr(torch, "empty_like", real_empty_like)
    return poisoned


class Report:
    def __init__(self, name, instance):
        self.name, self.instance, self.rows = name, instance, []

    def add(self, what, value, bound, sep=None):
        self.rows.append((what, float(value), float(bound), sep))

    def finish(self):
        print(f"\n[{self.name}]  instance {self.instance}")
        for what, v, b, sep in self.rows:
            s = "" if sep is None else f"  nearest fault {sep[0]} at {sep[1]:9.1f}x tol"
            print(f"  {what:<16} {v:11.3e}  bound {b:9.2e}{s}")
        bad = [(w, v, b) for w, v, b, _ in self.rows if not v <= b]
        assert not bad, (self.name, bad)


def _dist(got, want):
    """distance of `got` from `want` in tolerances (out), the largest of the three measures"""
    return max(er.ulp_err(got, want) / TOL["out_ulp"], er.rel_err(got, want) / TOL["out_rel"],
               er.rms_err(got, want) / TOL["out_rms"])


def pin_level(rep, out, out16, want, ref_fn):
    """Compare a level's out / out16 with the reference and separate the kernel from every injected fault that shows
    (a fault shows when it moves the reference by 3 tolerances or, for E7, changes out16)."""
    out = out.detach().cpu()
    assert torch.isfinite(out).all(), rep.name                  # every target written
    seps = []
    faults = {f: ref_fn(f) for f in er.FAULTS}
    for f, bad in faults.items():
        if f == "E7":
            if out16 is not None and bool((bad["out16"] != want["out16"]).any()):
                # the kernel's out16 is fp16(out) bit for bit; the faulted copy differs from fp16(its own out)
                n = int((out16.detach().cpu().to(F64) != bad["out16"]).sum())
                rep.add("E7 out16 diffs", 1.0 / max(n, 1e-300), 1.0)
                seps.append((f, float("inf")))
            continue
        if _dist(bad["out"], want["out"]) < 3.0:
            continue        # this fault does not show at this case (e.g. E3 without split inputs)
        d = _dist(out, bad["out"])
        rep.add(f"{f} sep (1/x)", 3.0 / d, 1.0)                 # kernel more than 3 tolerances from the fault
        seps.append((f, d))
    nearest = min(seps, key=lambda t: t[1]) if seps else None
    rep.add("out ulp", er.ulp_err(out, want["out"]), TOL["out_ulp"], nearest)
    rep.add("out rel", er.rel_err(out, want["out"]), TOL["out_rel"])
    rep.add("out rms", er.rms_err(out, want["out"]), TOL["out_rms"])
    if out16 is not None:
        o16 = out16.detach().cpu()
        assert torch.isfinite(o16).all(), rep.name
        rep.add("out16 != fp16", float((o16 != out.half()).sum()), 0)
    return rep


def _eval_mlp(chans, seed, dev):
    """A product MLP with the weights of ref.MLPRef(seed) and non-trivial running statistics, in eval mode."""
    mref = ref.seeded_init_(ref.MLPRef(chans, act="ReLU"), seed)
    m = MLP(chans, act="ReLU")
    m.load_state_dict(mref.state_dict())
    with torch.no_grad():
        g = torch.Generator().manual_seed(seed + 7)
        for n in m.norms:
            n.running_mean.copy_(torch.rand(n.running_mean.shape, generator=g) - 0.5)
            n.running_var.copy_(torch.rand(n.running_var.shape, generator=g) + 0.5)
    return m.to(dev).eval()


def _slots_problem(c_in, K, B, n, r, seed):
    b = Batch.from_data_list(synthetic_clouds(seed, B, n, max(c_in, 1), True))
    x = None if c_in == 0 else torch.randn(b.pos.size(0), c_in, generator=torch.Generator().manual_seed(seed + 1))
    idx = ref.fps_ref(b.pos, b.ptr, 0.2)
    qptr = ref.sample_ptr(b.ptr, 0.2)
    nbr, cnt = ref.ball_query_ref(b.pos, b.pos[idx], b.ptr, qptr, r, K)
    return x, b.pos, b.pos[idx].contiguous(), nbr, cnt


def _crafted_problem(c_in, n_dst, cnt_fn, K, seed):
    """Targets with chosen neighbour counts: the compacted row count (and which tile a target lands in) is set by
    construction -- with cnt <= 8 every target owns 8 rows, eight targets per 64-row tile."""
    g = torch.Generator().manual_seed(seed)
    n_src = 4 * n_dst + 64
    pos = torch.randn(n_src, 3, generator=g) * 2
    x = None if c_in == 0 else torch.randn(n_src, c_in, generator=g)
    nbr = torch.full((n_dst, K), -1, dtype=torch.int32)
    cnts = [cnt_fn(m) for m in range(n_dst)]
    for m, c in enumerate(cnts):
        nbr[m, :c] = torch.randperm(n_src, generator=g)[:c].sort().values.to(torch.int32)
    return x, pos, torch.randn(n_dst, 3, generator=g), nbr, torch.tensor(cnts, dtype=torch.int32)


def run_slots(name, dev, nan_alloc, problem, chans, K, *, expect, x16=False, sm_limit=0, seed=3):
    """One SLOTS level through sa_apply(PREC_BF16) in evaluation under no_grad, pinned against the reference.
    x16: hand the features over as fp16 (x_bf16), as the previous level's epilogue does."""
    x, pos_src, pos_dst, nbr, cnt = problem
    m = _eval_mlp(chans, seed, dev)
    n_dst = pos_dst.shape[0]
    xd = None if x is None else x.to(dev)
    x_bf16 = xd.half() if (x16 and xd is not None) else None
    args = (pos_src.to(dev), pos_dst.to(dev), nbr.to(dev), cnt.to(dev), None)
    rowmap = sa.pack_rows(args[2], args[3], K)
    fused = _probe_fused(x_bf16 if x_bf16 is not None else xd, chans, K)
    assert fused == (expect != MULTIPASS), (name, fused)

    def call():
        with torch.no_grad(), sa.options(sm_limit=sm_limit), nan_alloc():
            l0 = _launches()
            res = sa.sa_apply(m, xd, *args, seg_mode=sa.SEG_SLOTS, K=K, n_dst=n_dst, precision=sa.PREC_BF16,
                              rowmap=rowmap, x_bf16=x_bf16, want_bf16_out=True)
            return res, _launches() - l0
    ((out, arg, out16), launches), names = _kernel_names(call)
    inst = _instance(names)
    assert inst == expect, (name, inst, names)
    if expect != MULTIPASS:
        assert arg.numel() == 0 and launches == 2, (name, arg.numel(), launches)   # weight packing + the level
    else:
        assert arg.shape == out.shape and launches > 2, (name, launches)
    rep = Report(name, inst)
    rep.add("launches", launches, 2 if expect != MULTIPASS else 99)
    p = er.params_of(m)
    rows = er.Rows(n_dst, nbr=nbr, cnt=cnt)
    xin = x_bf16.cpu() if x_bf16 is not None else x
    bn = "multipass" if expect == MULTIPASS else "fused"
    f = lambda fault=None: er.eval_level(xin, pos_src, p, rows, pos_dst=pos_dst, bn=bn, fault=fault)  # noqa: E731
    pin_level(rep, out, out16, f(), f)
    rep.out, rep.out16 = out.detach().cpu(), out16.detach().cpu()
    return rep


# ------------------------------------------------------------------------------------------------------------------
#  the single-launch evaluation kernel, instance by instance
# ------------------------------------------------------------------------------------------------------------------
INSTANCE_CASES = {
    # reference level 1: fp32 intensity split into hi + lo
    "ref_l1": dict(c_in=1, chans=[4, 64, 64, 128], K=64, expect=FUSED_L1),
    # reference level 2: fp16 features from the previous level's epilogue (x_bf16) ...
    "ref_l2_x16": dict(c_in=128, chans=[131, 128, 128, 256], K=64, x16=True, expect=FUSED_L2),
    # ... and fp32 features wider than 16 channels, converted to fp16 by sa._l1_input
    "ref_l2_x32": dict(c_in=128, chans=[131, 128, 128, 256], K=64, expect=FUSED_L2),
    # neuron_multiplier = 2, level 1: c1c = c2c = mt3 = 2 picks the run-time-shaped instance
    "nm2_l1": dict(c_in=1, chans=[4, 128, 128, 256], K=64, expect=FUSED_RT),
    "rt_k40": dict(c_in=8, chans=[11, 64, 128, 256], K=40, expect=FUSED_RT),
    # no features: its image (6 columns) fits the unrolled level-1 instance
    "no_feat": dict(c_in=0, chans=[3, 64, 64, 128], K=32, expect=FUSED_L1),
    # c3 = 42: a partial warp of output channels (ch3 < c3 guards)
    "c3_42": dict(c_in=4, chans=[7, 64, 128, 42], K=16, expect=FUSED_RT),
}


@pytest.mark.parametrize("case", list(INSTANCE_CASES))
def test_eval_fused_instances(cuda_device, nan_alloc, case):
    c = INSTANCE_CASES[case]
    prob = _slots_problem(c["c_in"], c["K"], 3, 600, 2.5, 21)
    run_slots(case, cuda_device, nan_alloc, prob, c["chans"], c["K"], expect=c["expect"],
              x16=c.get("x16", False)).finish()


# tiles of 64 rows: with cnt <= 8 every target owns one 8-row group, eight targets per tile
TILE_CASES = {
    "1 tile, 3 targets": dict(n_dst=3),
    "1 tile, full": dict(n_dst=8),
    "20 tiles (rows = 10 x 128)": dict(n_dst=160),
    "21 tiles (odd: slot 1 one fewer)": dict(n_dst=168),
    "203 tiles, sm_limit=1": dict(n_dst=1621, sm_limit=1),
    "203 tiles, sm_limit=3": dict(n_dst=1621, sm_limit=3),
}


@pytest.mark.parametrize("shape", ["l1", "rt"])
@pytest.mark.parametrize("case", list(TILE_CASES))
def test_eval_fused_tiles_and_grid(cuda_device, nan_alloc, case, shape):
    c = TILE_CASES[case]
    chans, expect = ([4, 64, 64, 128], FUSED_L1) if shape == "l1" else ([4, 128, 128, 256], FUSED_RT)
    prob = _crafted_problem(1, c["n_dst"], lambda m: 1 + (m * 5) % 8, 64, 31)
    run_slots(f"{shape}/{case}", cuda_device, nan_alloc, prob, chans, 64, expect=expect,
              sm_limit=c.get("sm_limit", 0)).finish()


# ------------------------------------------------------------------------------------------------------------------
#  empty neighbourhoods: every path gives 0
# ------------------------------------------------------------------------------------------------------------------
EMPTY = {16, 28} | set(range(40, 48))   # first target of tile 2, mid-tile in tile 3, every target of tile 5


@pytest.mark.parametrize("c_in,chans,x16,expect", [(1, [4, 64, 64, 128], False, FUSED_L1),
                                                   (128, [131, 128, 128, 256], True, FUSED_L2),
                                                   (1, [4, 128, 128, 256], False, FUSED_RT)])
def test_empty_neighbourhood_is_zero_on_every_path(cuda_device, nan_alloc, c_in, chans, x16, expect):
    dev = cuda_device
    K = 64
    prob = _crafted_problem(c_in, 64, lambda m: 0 if m in EMPTY else 1 + (m * 3) % 8, K, 41)
    x, pos_src, pos_dst, nbr, cnt = prob
    if x16:
        x = x.abs().half().float()
    prob = (x, pos_src, pos_dst, nbr, cnt)
    empty = torch.tensor(sorted(EMPTY))
    rep = run_slots(f"empty/{expect}", dev, nan_alloc, prob, chans, K, expect=expect, x16=x16)
    rep.add("fused empty", float(rep.out[empty].abs().max()), 0)
    rep.add("out16 empty", float(rep.out16[empty].float().abs().max()), 0)
    rep.finish()
    # the same inputs through the multi-pass kernels (grad enabled: a backward could follow) and the fp32 path, each
    # against the reference of its own roundings (fp32: none, at the fp32 path's 1e-4 parity bound)
    m = _eval_mlp(chans, 3, dev)
    p = er.params_of(m)
    rows = er.Rows(64, nbr=nbr, cnt=cnt)
    args = (pos_src.to(dev), pos_dst.to(dev), nbr.to(dev), cnt.to(dev), None)
    xg = x.to(dev).requires_grad_(True)
    for prec, name in ((sa.PREC_BF16, "multi-pass"), (sa.PREC_F32, "fp32")):
        with nan_alloc():
            out, arg = sa.sa_apply(m, xg, *args, seg_mode=sa.SEG_SLOTS, K=K, n_dst=64, precision=prec)
        out, arg = out.detach().cpu(), arg.cpu()
        assert torch.isfinite(out).all()
        if prec == sa.PREC_BF16:
            want, bound = er.eval_level(x, pos_src, p, rows, pos_dst=pos_dst, bn="multipass")["out"], TOL["out_rel"]
        else:
            want, bound = er.eval_level(x, pos_src, p, rows, pos_dst=pos_dst, rnd=er.ROUND_NONE)["out"], 1e-4
        r = Report(f"empty/{expect}/{name}", name)
        r.add("out empty", float(out[empty].abs().max()), 0)
        r.add("arg empty = -1", float((arg[empty] != -1).sum()), 0)
        r.add("out rel", er.rel_err(out, want), bound)
        r.finish()


# ------------------------------------------------------------------------------------------------------------------
#  the multi-pass kernels with eval-mode BatchNorm (levels the single launch cannot take)
# ------------------------------------------------------------------------------------------------------------------
def test_eval_multipass_slots_levels(cuda_device, nan_alloc):
    prob = _slots_problem(16, 16, 3, 600, 2.5, 21)
    run_slots("multipass/[19,32,48,40]", cuda_device, nan_alloc, prob, [19, 32, 48, 40], 16,
              expect=MULTIPASS).finish()
    # neuron_multiplier = 2, level 2: fp16 features of 256 channels
    x, pos, pos_dst, nbr, cnt = _slots_problem(1, 64, 3, 600, 2.5, 21)
    g = torch.Generator().manual_seed(4)
    x2 = torch.randn(pos.shape[0], 256, generator=g).abs()
    run_slots("multipass/nm2_l2", cuda_device, nan_alloc, (x2, pos, pos_dst, nbr, cnt), [259, 256, 256, 512], 64,
              expect=MULTIPASS, x16=True).finish()


@pytest.mark.parametrize("sizes,chans", [([130, 1, 257, 64], [35, 64, 96, 200]),       # a cloud of one row
                                         ([500] * 12, [259, 256, 512, 1024]),          # the reference's global level
                                         ([120] * 6, [515, 512, 1024, 2048])])         # neuron_multiplier = 2
def test_eval_multipass_clouds_levels(cuda_device, nan_alloc, sizes, chans):
    dev = cuda_device
    g = torch.Generator().manual_seed(5)
    n = sum(sizes)
    x = torch.randn(n, chans[0] - 3, generator=g).abs()
    pos = torch.randn(n, 3, generator=g) * 3
    batch = torch.repeat_interleave(torch.arange(len(sizes)), torch.tensor(sizes))
    m = _eval_mlp(chans, 9, dev)
    xh = x.half().to(dev)
    assert _probe_fused(xh, chans, 0, sa.SEG_CLOUDS) == 0

    def call():
        with torch.no_grad(), nan_alloc():
            return sa.sa_apply(m, x.to(dev), pos.to(dev), None, None, None, batch.to(dev), seg_mode=sa.SEG_CLOUDS,
                               K=0, n_dst=len(sizes), precision=sa.PREC_BF16, x_bf16=xh)
    (out, arg), names = _kernel_names(call)
    inst = _instance(names)
    assert inst == MULTIPASS
    rep = Report(f"clouds/{chans}", inst)
    p = er.params_of(m)
    rows = er.Rows(len(sizes), batch=batch)
    f = lambda fault=None: er.eval_level(xh.cpu(), pos, p, rows, bn="multipass", fault=fault)  # noqa: E731
    pin_level(rep, out, None, f(), f).finish()


# ------------------------------------------------------------------------------------------------------------------
#  the regression head in evaluation
# ------------------------------------------------------------------------------------------------------------------
def _head_mlp(nm, dev):
    m = MLP([1024 * nm, 128 * nm, 128 * nm, 4], act=None, dropout=0.0)
    ref.seeded_init_(m, 13)
    with torch.no_grad():
        g = torch.Generator().manual_seed(14)
        for n in m.norms:
            n.running_mean.copy_(torch.rand(n.running_mean.shape, generator=g) - 0.5)
            n.running_var.copy_(torch.rand(n.running_var.shape, generator=g) + 0.5)
    return m.to(dev).eval()


@pytest.mark.parametrize("nm", [1, 2])
def test_eval_head_chunks(cuda_device, nm):
    dev = cuda_device
    m = _head_mlp(nm, dev)
    p = er.params_of(m)
    counter = torch.zeros((), dtype=torch.int64, device=dev)
    rep = Report(f"head/nm={nm}", "fused head")
    for B in (1, 31, 32, 33, 70, 512):
        x = torch.randn(B, 1024 * nm, generator=torch.Generator().manual_seed(B)).abs().to(dev)
        assert head.supported(m, x)
        with torch.no_grad():
            out = head.head_apply(m, x, counter, 5)
        rep.add(f"B={B}", er.rel_err(out, er.eval_head(x, p)), TOL["head_rel"])
    rep.finish()


def test_eval_head_too_wide_falls_back_to_aten(cuda_device):
    """neuron_multiplier = 3: hidden width 384 is past the fused head's 256; Net runs the head through ATen."""
    dev = cuda_device
    m = _head_mlp(3, dev)
    x = torch.randn(40, 3072, generator=torch.Generator().manual_seed(1)).abs().to(dev)
    assert not head.supported(m, x)
    with torch.no_grad():
        out = m(x)
    rep = Report("head/nm=3", "ATen")
    rep.add("B=40", er.rel_err(out, er.eval_head(x, er.params_of(m))), TOL["head_rel"])
    rep.finish()


# ------------------------------------------------------------------------------------------------------------------
#  a whole Net in eval mode, level by level
# ------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("nm", [1, 2])
@pytest.mark.parametrize("B,n", [(64, 2000), (12, 10000)])
def test_eval_net_per_level(cuda_device, monkeypatch, nm, B, n):
    """Each level pinned against the reference fed that level's actual inputs (the fp16 hand-over x_bf16 included), so
    errors do not compound; the head pinned on the recorded global-level output.  Running statistics from two
    train-mode passes of the float32 oracle."""
    from dl_biomass_b200.pointnet2_regressor import Net
    dev = cuda_device
    netr = ref.seeded_init_(ref.NetRef(1, "ReLU", nm, 0.0), seed=7)
    netr.train()
    with torch.no_grad():
        for i in range(2):
            netr(Batch.from_data_list(synthetic_clouds(500 + i, 4, 600, 1, True)))
    net = Net(1, "ReLU", nm, 0.0, precision="bf16")
    net.load_state_dict(netr.state_dict())
    net = net.to(dev).set_random_start(False).eval()
    b = Batch.from_data_list(synthetic_clouds(99, B, n, 1, True)).to(dev)
    levels, real = [], sa.sa_apply

    def spy(mlp, x, pos_src, pos_dst, nbr, cnt, batch, **kw):
        res = real(mlp, x, pos_src, pos_dst, nbr, cnt, batch, **kw)
        levels.append(dict(mlp=mlp, x=x, x_bf16=kw.get("x_bf16"), pos_src=pos_src, pos_dst=pos_dst, nbr=nbr, cnt=cnt,
                           batch=batch, kw=kw, out=res[0], out16=res[2] if len(res) > 2 else None))
        return res

    monkeypatch.setattr(sa, "sa_apply", spy)
    with torch.no_grad():
        (y, launches), names = _kernel_names(lambda: (net(b), None))
    monkeypatch.undo()
    assert len(levels) == 3
    insts = [i for i in (_instance([nm_]) for nm_ in names) if i != MULTIPASS]
    want_inst = [FUSED_L1, FUSED_L2] if nm == 1 else [FUSED_RT]
    assert insts == want_inst, insts
    failed = []
    for i, lv in enumerate(levels):
        kw = lv["kw"]
        clouds = kw["seg_mode"] == sa.SEG_CLOUDS
        x = lv["x"]
        used16 = lv["x_bf16"] is not None and x is not None and x.shape[1] > 16
        xin = None if x is None else (lv["x_bf16"] if used16 else x).detach().cpu()
        if i > 0:
            assert used16 and lv["x_bf16"].dtype == torch.float16
        p = er.params_of(lv["mlp"])
        if clouds:
            rows, inst, bn = er.Rows(kw["n_dst"], batch=lv["batch"]), MULTIPASS, "multipass"
        else:
            rows = er.Rows(kw["n_dst"], nbr=lv["nbr"], cnt=lv["cnt"])
            inst = want_inst[i] if i < len(want_inst) else MULTIPASS
            bn = "multipass" if inst == MULTIPASS else "fused"
        pos_dst = None if lv["pos_dst"] is None else lv["pos_dst"].cpu()
        f = lambda fault=None: er.eval_level(xin, lv["pos_src"].cpu(), p, rows, pos_dst=pos_dst, bn=bn,  # noqa: E731
                                             fault=fault)
        rep = pin_level(Report(f"net nm={nm} {B}x{n}/level{i + 1}", inst), lv["out"], lv["out16"], f(), f)
        try:
            rep.finish()
        except AssertionError as e:
            failed.append(str(e))
    rep = Report(f"net nm={nm} {B}x{n}/head", "fused head")
    rep.add("head", er.rel_err(y, er.eval_head(levels[2]["out"], er.params_of(net.mlp))), TOL["head_rel"])
    try:
        rep.finish()
    except AssertionError as e:
        failed.append(str(e))
    assert not failed, failed
