"""GPU parity of Kernel 3 (set-abstraction MLP + max, forward and backward) and of the whole Net
against the CPU oracle.  fp32 mode: 1e-4 relative (north_star); bf16 mode: 2e-2 on the outputs."""
import os

import pytest
import torch

from oracle import ref
from dl_biomass_b200 import ops, sa
from dl_biomass_b200.data import Batch, Data, synthetic_clouds
from dl_biomass_b200.pointnet2_regressor import MLP, Net

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")
# run-to-run spread allowed on the bf16 level-1 weight gradients in the DEFAULT (atomic) mode, relative to the largest
# level-1 gradient: measured over 20 runs in profiles/r02_grad_spread.md; the deterministic mode is held to bit-equality
SA1_SPREAD_BOUND = 5e-3   # measured worst over 20 runs: 9.2e-4 (3 x 640 points), 2.8e-4 (12 x 10 000 points)


def rel_err(got, want):
    got, want = got.detach().double().cpu(), want.detach().double().cpu()
    return float((got - want).abs().max() / want.abs().max().clamp_min(1e-12))


def _mlp_pair(chans, seed, dev):
    mref = ref.seeded_init_(ref.MLPRef(chans, act="ReLU"), seed)
    m = MLP(chans, act="ReLU")
    m.load_state_dict(mref.state_dict())
    return mref, m.to(dev)


@pytest.mark.parametrize("c_in,chans,K,train", [(1, [4, 64, 64, 128], 64, True), (1, [4, 64, 64, 128], 64, False),
                                                (16, [19, 32, 48, 40], 16, True), (0, [3, 64, 64, 128], 32, True),
                                                (128, [131, 128, 128, 256], 64, True)])
def test_sa_slots_level_fp32(cuda_device, c_in, chans, K, train):
    b = Batch.from_data_list(synthetic_clouds(21, 3, 600, max(c_in, 1), True))
    x = None if c_in == 0 else (torch.randn(b.pos.size(0), c_in, generator=torch.Generator().manual_seed(1)))
    idx = ref.fps_ref(b.pos, b.ptr, 0.2)
    qptr = ref.sample_ptr(b.ptr, 0.2)
    nbr, cnt = ref.ball_query_ref(b.pos, b.pos[idx], b.ptr, qptr, 2.5, K)
    row, col = ref.slots_to_edges(nbr, cnt)
    mref, m = _mlp_pair(chans, 3, cuda_device)
    mref.train(train)
    m.train(train)
    xr = None if x is None else x.clone().requires_grad_(True)
    want = ref.point_conv_ref(mref, xr, b.pos, b.pos[idx], row, col)
    gout = torch.randn(want.shape, generator=torch.Generator().manual_seed(2))
    want.backward(gout)

    xg = None if x is None else x.to(cuda_device).requires_grad_(True)
    out, arg = sa.sa_apply(m, xg, b.pos.to(cuda_device), b.pos[idx].to(cuda_device), nbr.to(cuda_device),
                           cnt.to(cuda_device), None, seg_mode=sa.SEG_SLOTS, K=K, n_dst=idx.numel(),
                           precision=sa.PREC_F32)
    out.backward(gout.to(cuda_device))
    torch.cuda.synchronize()
    assert rel_err(out, want) < 1e-4
    for (k, p), (_, pr) in zip(m.named_parameters(), mref.named_parameters()):
        if k in ("lins.0.bias", "lins.1.bias") and train:
            assert float(p.grad.abs().max()) < 1e-3 * float(gout.abs().sum())  # BN cancels these biases
            continue
        assert rel_err(p.grad, pr.grad) < 2e-4, k
    if x is not None:
        assert rel_err(xg.grad, xr.grad) < 2e-4
    if train:
        for (k, v), (_, vr) in zip(m.named_buffers(), mref.named_buffers()):
            assert rel_err(v.float(), vr.float()) < 1e-4, k


def test_global_sa_level_fp32(cuda_device):
    g = torch.Generator().manual_seed(5)
    sizes = [130, 257, 64]
    n = sum(sizes)
    x = torch.randn(n, 32, generator=g)
    pos = torch.randn(n, 3, generator=g) * 3
    batch = torch.repeat_interleave(torch.arange(3), torch.tensor(sizes))
    chans = [35, 64, 96, 200]
    mref, m = _mlp_pair(chans, 9, cuda_device)
    xr = x.clone().requires_grad_(True)
    want, _, _ = ref.GlobalSAModuleRef(mref)(xr, pos, batch, 3)
    gout = torch.randn(want.shape, generator=g)
    want.backward(gout)
    xg = x.to(cuda_device).requires_grad_(True)
    out, arg = sa.sa_apply(m, xg, pos.to(cuda_device), None, None, None, batch.to(cuda_device),
                           seg_mode=sa.SEG_CLOUDS, K=0, n_dst=3, precision=sa.PREC_F32)
    out.backward(gout.to(cuda_device))
    assert rel_err(out, want) < 1e-4
    assert rel_err(xg.grad, xr.grad) < 2e-4
    for (k, p), (_, pr) in zip(m.named_parameters(), mref.named_parameters()):
        if k in ("lins.0.bias", "lins.1.bias"):
            continue
        assert rel_err(p.grad, pr.grad) < 2e-4, k


def _net_pair(dev, precision="fp32", train=True):
    netr = ref.seeded_init_(ref.NetRef(1, "ReLU", 0, 0.0), seed=7)
    net = Net(1, "ReLU", 0, 0.0, precision=precision)
    net.load_state_dict(netr.state_dict())
    net = net.to(dev).set_random_start(False)
    netr.train(train)
    net.train(train)
    return netr, net


@pytest.mark.parametrize("train", [True, False])
def test_net_forward_backward_fp32_vs_oracle(cuda_device, train):
    b = Batch.from_data_list(synthetic_clouds(4321, 3, 768, 1, True))
    netr, net = _net_pair(cuda_device, "fp32", train)
    want = netr(b)
    lw = ref.weighted_mse(want, b.y)
    lw.backward()
    out = net(b.to(cuda_device))
    loss = ref.weighted_mse(out, b.y.to(cuda_device))
    loss.backward()
    torch.cuda.synchronize()
    assert rel_err(out, want) < 1e-4
    assert rel_err(loss, lw) < 1e-4
    worst = 0.0
    for (k, p), (_, pr) in zip(net.named_parameters(), netr.named_parameters()):
        if pr.grad.abs().max() < 1e-6 * max(1.0, float(lw.detach())):  # biases in front of a BatchNorm: exactly 0 in theory
            continue
        e = rel_err(p.grad, pr.grad)
        worst = max(worst, e)
        assert e < 1e-3, (k, e)
    print("worst grad rel err", worst)
    if train:
        for (k, v), (_, vr) in zip(net.named_buffers(), netr.named_buffers()):
            assert rel_err(v.float(), vr.float()) < 1e-4, k


def test_net_matches_golden_fixture(cuda_device):
    gold = torch.load(os.path.join(GOLD, "net_oracle.pt"))
    b = Batch.from_data_list([Data(**c) for c in gold["clouds"]])   # the stored clouds
    for mode in ("train", "eval"):
        _, net = _net_pair(cuda_device, "fp32", mode == "train")
        out = net(b.to(cuda_device))
        assert rel_err(out, gold["modes"][mode]["out"]) < 1e-4


def test_training_steps_track_oracle(cuda_device):
    """Three Adam steps (main.py:84,171-172) on both sides stay together."""
    b = Batch.from_data_list(synthetic_clouds(99, 2, 512, 1, False))
    netr, net = _net_pair(cuda_device, "fp32", True)
    optr, opt = ref.make_adam(netr.parameters()), ref.make_adam(net.parameters())
    bg = b.to(cuda_device)
    for step in range(3):
        optr.zero_grad()
        lr_ = ref.weighted_mse(netr(b), b.y)
        lr_.backward()
        optr.step()
        opt.zero_grad()
        lg = ref.weighted_mse(net(bg), bg.y)
        lg.backward()
        opt.step()
        # step 0 sees identical weights; later steps drift because Adam turns the (theoretically zero)
        # gradients of biases in front of a BatchNorm into +-lr updates whose sign is rounding noise
        assert rel_err(lg, lr_) < (1e-4 if step == 0 else 3e-2), (step, float(lg), float(lr_))


# ---------------------------------------------------------------------------------------------------
#  bf16 tensor-core mode (tcgen05): tolerance 2e-2 on outputs (north_star)
# ---------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("c_in,chans,K,train", [(1, [4, 64, 64, 128], 64, True), (1, [4, 64, 64, 128], 64, False),
                                                (16, [19, 32, 48, 40], 16, True), (0, [3, 64, 64, 128], 32, True),
                                                (128, [131, 128, 128, 256], 64, True), (8, [11, 64, 128, 256], 40, True),
                                                (2, [5, 64, 64, 64], 8, True)])
def test_sa_slots_level_bf16_forward(cuda_device, c_in, chans, K, train):
    b = Batch.from_data_list(synthetic_clouds(21, 3, 600, max(c_in, 1), True))
    x = None if c_in == 0 else (torch.randn(b.pos.size(0), c_in, generator=torch.Generator().manual_seed(1)))
    idx = ref.fps_ref(b.pos, b.ptr, 0.2)
    qptr = ref.sample_ptr(b.ptr, 0.2)
    nbr, cnt = ref.ball_query_ref(b.pos, b.pos[idx], b.ptr, qptr, 2.5, K)
    row, col = ref.slots_to_edges(nbr, cnt)
    mref, m = _mlp_pair(chans, 3, cuda_device)
    mref.train(train)
    m.train(train)
    with torch.no_grad():
        want = ref.point_conv_ref(mref, x, b.pos, b.pos[idx], row, col)
        xg = None if x is None else x.to(cuda_device)
        out, arg = sa.sa_apply(m, xg, b.pos.to(cuda_device), b.pos[idx].to(cuda_device), nbr.to(cuda_device),
                               cnt.to(cuda_device), None, seg_mode=sa.SEG_SLOTS, K=K, n_dst=idx.numel(),
                               precision=sa.PREC_BF16)
    torch.cuda.synchronize()
    err = rel_err(out, want)
    print("bf16 SA level rel err", err)
    assert err < 2e-2
    if train:
        a = arg.cpu().long()
        assert int(a.min()) >= 0 and bool((a < cnt.long()[:, None]).all())
        for (k, v), (_, vr) in zip(m.named_buffers(), mref.named_buffers()):
            assert rel_err(v.float(), vr.float()) < 2e-2, k
    else:   # evaluation without grad: the single-launch kernel, which records no arg-max slots (no backward can follow)
        assert arg.numel() == 0


@pytest.mark.parametrize("K,n,r", [(64, 600, 2.5), (64, 3000, 1.0), (40, 600, 2.5), (8, 600, 9.0), (16, 50, 0.01)])
def test_pack_rows_structure(cuda_device, K, n, r):
    """b2pn_pack_rows: every centroid owns max(8, round_up(cnt, 8)) consecutive rows inside one 64-row block,
    rows carry the neighbour slots in order, the device-side row count covers exactly the rows in use."""
    b = Batch.from_data_list(synthetic_clouds(77, 4, n, 1, True))
    idx = ref.fps_ref(b.pos, b.ptr, 0.2)
    qptr = ref.sample_ptr(b.ptr, 0.2)
    nbr, cnt = ref.ball_query_ref(b.pos, b.pos[idx], b.ptr, qptr, r, K)
    rgrp, row_src, num_rows, cap, row_valid = sa.pack_rows(nbr.to(cuda_device), cnt.to(cuda_device), K)
    torch.cuda.synchronize()
    rows, edges = (int(v) for v in num_rows.tolist())
    assert edges == int(cnt.clamp(0, K).sum())
    assert rows % 64 == 0 and 0 < rows <= cap
    g = rgrp.cpu().numpy().astype("uint32")
    src = row_src.cpu().numpy()
    seg = (g & 0xFFFFFF).astype("int64")
    slot0 = ((g >> 24) & 7).astype("int64") * 8
    nv = ((g >> 27) & 15).astype("int64")
    last = (g >> 31).astype("int64")
    none = seg == 0xFFFFFF
    assert none[rows // 8:].all() and (src[rows:] == -1).all()
    import numpy as np
    used = np.nonzero(~none[: rows // 8])[0]
    cntn, nbrn = cnt.numpy(), nbr.numpy()
    seen = np.zeros(cnt.numel(), dtype=bool)
    # walk the groups centroid by centroid
    i = 0
    while i < len(used):
        gi = used[i]
        m = seg[gi]
        assert slot0[gi] == 0 and not seen[m]
        seen[m] = True
        c8 = max(8, (int(cntn[m]) + 7) // 8 * 8)
        ng = c8 // 8
        assert (gi * 8) // 64 == (gi * 8 + c8 - 1) // 64, "centroid crosses a 64-row boundary"
        for j in range(ng):
            assert used[i + j] == gi + j and seg[gi + j] == m and slot0[gi + j] == 8 * j
            want_nv = min(8, max(0, int(cntn[m]) - 8 * j))
            assert nv[gi + j] == want_nv and last[gi + j] == (1 if j == ng - 1 else 0)
            want_src = np.full(8, -1, dtype=np.int64)
            want_src[:want_nv] = nbrn[m, 8 * j: 8 * j + want_nv]
            assert (src[(gi + j) * 8: (gi + j) * 8 + 8] == want_src).all()
        i += ng
    assert seen.all()
    rv = row_valid.float().cpu().numpy()
    assert ((rv == 1.0) == (src >= 0)).all() and ((rv == 0.0) | (rv == 1.0)).all()
    # centroids keep their order
    firsts = used[slot0[used] == 0]
    assert (np.diff(seg[firsts]) > 0).all()


def test_bf16_rejects_wide_slots(cuda_device):
    m = MLP([4, 64, 64, 128], act="ReLU").to(cuda_device)
    pos = torch.randn(200, 3, device=cuda_device)
    x = torch.randn(200, 1, device=cuda_device)
    nbr = torch.zeros(10, 128, dtype=torch.int32, device=cuda_device)
    cnt = torch.ones(10, dtype=torch.int32, device=cuda_device)
    with pytest.raises(RuntimeError):
        sa.sa_apply(m, x, pos, pos[:10].contiguous(), nbr, cnt, None, seg_mode=sa.SEG_SLOTS, K=128, n_dst=10,
                    precision=sa.PREC_BF16)


def test_global_sa_level_bf16_forward(cuda_device):
    g = torch.Generator().manual_seed(5)
    sizes = [130, 257, 64]
    n = sum(sizes)
    x = torch.randn(n, 32, generator=g)
    pos = torch.randn(n, 3, generator=g) * 3
    batch = torch.repeat_interleave(torch.arange(3), torch.tensor(sizes))
    for chans in ([35, 64, 96, 200], [35, 256, 512, 1024]):
        mref, m = _mlp_pair(chans, 9, cuda_device)
        with torch.no_grad():
            want, _, _ = ref.GlobalSAModuleRef(mref)(x, pos, batch, 3)
            out, arg = sa.sa_apply(m, x.to(cuda_device), pos.to(cuda_device), None, None, None, batch.to(cuda_device),
                                   seg_mode=sa.SEG_CLOUDS, K=0, n_dst=3, precision=sa.PREC_BF16)
        err = rel_err(out, want)
        print("bf16 global SA rel err", err)
        assert err < 2e-2


@pytest.mark.parametrize("train", [True, False])
def test_net_forward_bf16_vs_oracle(cuda_device, train):
    """north_star: 2e-2 on the regression outputs in the bf16 tensor-core mode (batch of 12 clouds, the
    reference's batch size: the head's train-mode BatchNorm normalises ACROSS clouds, so tiny batches
    amplify any rounding; see DESIGN.md)."""
    b = Batch.from_data_list(synthetic_clouds(4321, 12, 640, 1, True))
    netr, net = _net_pair(cuda_device, "bf16", train)
    feats = {}
    netr.sa3_module.register_forward_hook(lambda m, i, o: feats.__setitem__("ref", o[0].detach()))
    with torch.no_grad():
        want = netr(b)
        out = net(b.to(cuda_device))
    err = rel_err(out, want)
    print("bf16 Net rel err", err, "train" if train else "eval")
    assert err < 2e-2


def _grad_errs(m, mref, skip_bn_biases=True):
    errs = {}
    for (k, p), (_, pr) in zip(m.named_parameters(), mref.named_parameters()):
        if skip_bn_biases and k in ("lins.0.bias", "lins.1.bias"):
            continue
        errs[k] = rel_err(p.grad, pr.grad)
    return errs


@pytest.mark.parametrize("c_in,chans,K", [(1, [4, 64, 64, 128], 64), (16, [19, 32, 48, 40], 16),
                                          (128, [131, 128, 128, 256], 64), (0, [3, 64, 64, 128], 32),
                                          (8, [11, 64, 128, 256], 40),
                                          (4, [7, 32, 32, 42], 16)])   # 42: the routed gradient's scalar (non-quad) loads
def test_sa_slots_level_bf16_backward(cuda_device, c_in, chans, K):
    """bf16 gradients against the oracle run with bf16 rounding emulated at the same points (weights, post-BN
    values).  Against the un-rounded oracle they differ by ~10 % because rounding flips a few arg-max / ReLU
    decisions (the same deviation the emulation shows on the CPU)."""
    b = Batch.from_data_list(synthetic_clouds(21, 3, 600, max(c_in, 1), True))
    x = None if c_in == 0 else (torch.randn(b.pos.size(0), c_in, generator=torch.Generator().manual_seed(1)))
    if x is not None and c_in > 16:
        x = x.to(torch.float16).float()   # wide feature maps enter the kernel as fp16 (forward-domain operand format)
    idx = ref.fps_ref(b.pos, b.ptr, 0.2)
    qptr = ref.sample_ptr(b.ptr, 0.2)
    nbr, cnt = ref.ball_query_ref(b.pos, b.pos[idx], b.ptr, qptr, 2.5, K)
    row, col = ref.slots_to_edges(nbr, cnt)
    mref, m = _mlp_pair(chans, 3, cuda_device)
    mref.emulate_bf16 = True
    xr = None if x is None else x.clone().requires_grad_(True)
    want = ref.point_conv_ref(mref, xr, b.pos, b.pos[idx], row, col)
    gout = torch.randn(want.shape, generator=torch.Generator().manual_seed(2))
    want.backward(gout)
    xg = None if x is None else x.to(cuda_device).requires_grad_(True)
    out, arg = sa.sa_apply(m, xg, b.pos.to(cuda_device), b.pos[idx].to(cuda_device), nbr.to(cuda_device),
                           cnt.to(cuda_device), None, seg_mode=sa.SEG_SLOTS, K=K, n_dst=idx.numel(),
                           precision=sa.PREC_BF16)
    out.backward(gout.to(cuda_device))
    torch.cuda.synchronize()
    assert rel_err(out, want) < 1e-2
    errs = _grad_errs(m, mref)
    print("bf16 grads vs emulated oracle", {k: round(v, 4) for k, v in errs.items()})
    # residual differences come from arg-max / ReLU decisions that flip on last-bit differences between the
    # emulation and the kernel (fp32 summation order); narrow layers (32-48 channels) average them least
    assert max(errs.values()) < 8e-2, errs
    if x is not None:
        assert rel_err(xg.grad, xr.grad) < 0.15


def test_global_sa_level_bf16_backward(cuda_device):
    g = torch.Generator().manual_seed(5)
    sizes = [130, 257, 64]
    n = sum(sizes)
    x = (torch.randn(n, 32, generator=g)).to(torch.float16).float()
    pos = torch.randn(n, 3, generator=g) * 3
    batch = torch.repeat_interleave(torch.arange(3), torch.tensor(sizes))
    for chans in ([35, 64, 96, 200], [35, 256, 512, 1024]):
        mref, m = _mlp_pair(chans, 9, cuda_device)
        mref.emulate_bf16 = True
        xr = x.clone().requires_grad_(True)
        want, _, _ = ref.GlobalSAModuleRef(mref)(xr, pos, batch, 3)
        gout = torch.randn(want.shape, generator=g)
        want.backward(gout)
        xg = x.to(cuda_device).requires_grad_(True)
        out, arg = sa.sa_apply(m, xg, pos.to(cuda_device), None, None, None, batch.to(cuda_device),
                               seg_mode=sa.SEG_CLOUDS, K=0, n_dst=3, precision=sa.PREC_BF16)
        out.backward(gout.to(cuda_device))
        assert rel_err(out, want) < 1e-2
        errs = _grad_errs(m, mref)
        errs["x"] = rel_err(xg.grad, xr.grad)
        print("bf16 global grads vs emulated oracle", {k: round(v, 4) for k, v in errs.items()})
        assert max(errs.values()) < 6e-2, errs


def test_net_train_step_bf16_vs_oracle(cuda_device):
    """Whole training step in bf16 mode: outputs within 2e-2 of the fp32 oracle (north_star); gradients are
    only required to be sane here (level-wise gradient parity is checked above against the emulation)."""
    b = Batch.from_data_list(synthetic_clouds(4321, 12, 640, 1, True))
    netr, net = _net_pair(cuda_device, "bf16", True)
    want = netr(b)
    lw = ref.weighted_mse(want, b.y)
    lw.backward()
    out = net(b.to(cuda_device))
    loss = ref.weighted_mse(out, b.y.to(cuda_device))
    loss.backward()
    torch.cuda.synchronize()
    print("bf16 net out err", rel_err(out, want), "loss err", rel_err(loss, lw))
    assert rel_err(out, want) < 2e-2
    cos = []
    for (k, p), (_, pr) in zip(net.named_parameters(), netr.named_parameters()):
        if pr.grad.abs().max() < 1e-6 * max(1.0, float(lw.detach())):
            continue
        a, r = p.grad.detach().double().cpu().flatten(), pr.grad.double().flatten()
        cos.append(float((a @ r) / (a.norm() * r.norm()).clamp_min(1e-30)))
        assert torch.isfinite(a).all()
    print("bf16 net grad cosine min/mean", min(cos), sum(cos) / len(cos))
    assert min(cos) > 0.7 and sum(cos) / len(cos) > 0.95, cos


def _make_opt(kind, net, graph):
    from dl_biomass_b200.train import make_optimizer
    # "flat": optim.FlatAdam over the parameter arena (one libb2pn launch); "torch": ATen's fused Adam
    return make_optimizer(net) if kind == "flat" else make_optimizer(net.parameters(), capturable=graph)


@pytest.mark.parametrize("opt_kind", ["flat", "torch"])
def test_graphed_train_step_matches_eager(cuda_device, opt_kind):
    """train.GraphedTrainStep (one CUDA-graph replay per iteration) walks the same trajectory as eager launches, and
    BUILDING it does not train: warm-up and capture leave weights, BatchNorm buffers and optimiser state untouched."""
    from dl_biomass_b200.train import GraphedTrainStep, train_step
    batches = [Batch.from_data_list(synthetic_clouds(900 + 7 * i, 4, 512, 1, False)).to(cuda_device) for i in range(3)]
    losses = {}
    for mode in ("eager", "graph"):
        torch.manual_seed(3)
        net = Net(1, "ReLU", 0, 0.0, precision="bf16").to(cuda_device).set_random_start(False)
        net.train()
        opt = _make_opt(opt_kind, net, mode == "graph")
        if mode == "graph":
            state = {k: v.clone() for k, v in net.state_dict().items()}
            step = GraphedTrainStep(net, opt, batches[0], warmup=2)
            for k, v in net.state_dict().items():
                assert torch.equal(v, state[k]), f"building the stepper changed {k}"
            assert step.launches_per_replay > 20
            losses[mode] = [float(step(b)) for b in batches]
        else:
            losses[mode] = [float(train_step(net, opt, b)) for b in batches]
    print(losses)
    for a, b in zip(losses["eager"], losses["graph"]):
        assert abs(a - b) <= 2e-3 * max(abs(a), 1e-6)


@pytest.mark.parametrize("graph,opt_kind,deterministic", [(False, "flat", False), (True, "flat", False), (True, "torch", False),
                                                         (True, "flat", True)])
def test_pipelined_train_step_matches_eager(cuda_device, graph, opt_kind, deterministic):
    """train.PipelinedTrainStep (FPS of the next batch on a second stream, optionally one CUDA graph per step)
    trains exactly like the plain loop, one call later; building it does not train; flush() trains the last batch, so
    every batch is trained on exactly once (/root/reference/main.py:150-172).

    Default mode: the level gradients are summed with atomics, so two runs of the SAME loop differ by ~1e-5 after a step, and
    this batch shape (BatchNorm over 4 rows in the head) amplifies that to <= 8e-4 of the loss one step later (measured over
    repeated runs, profiles/r02_backward_ncu.md): steps 1-3 are held to 2e-3, step 4 to 5e-3.  Deterministic mode
    (b2pn_sa_args::deterministic) removes the atomics: every step within 2e-4."""
    from dl_biomass_b200 import sa
    from dl_biomass_b200.train import PipelinedTrainStep, train_step
    batches = [Batch.from_data_list(synthetic_clouds(500 + 11 * i, 4, 512, 1, False)).to(cuda_device) for i in range(4)]
    with sa.options(deterministic=deterministic):

        def fresh():
            torch.manual_seed(5)
            net = Net(1, "ReLU", 0, 0.0, precision="bf16").to(cuda_device).set_random_start(False)
            net.train()
            return net

        net = fresh()
        opt = _make_opt(opt_kind, net, False)
        want = [float(train_step(net, opt, b)) for b in batches]
        want_state = {k: v.clone() for k, v in net.state_dict().items()}

        net = fresh()
        opt = _make_opt(opt_kind, net, graph)
        state = {k: v.clone() for k, v in net.state_dict().items()}
        stepper = PipelinedTrainStep(net, opt, batches[0], graph=graph, warmup=1)
        try:
            for k, v in net.state_dict().items():
                assert torch.equal(v, state[k]), f"building the stepper changed {k}"
            got = [float(stepper.step(b)) for b in batches[1:4]]
            assert stepper.launches_per_step > 20
            got.append(float(stepper.flush()))
            with pytest.raises(RuntimeError):
                stepper.step(batches[0])
        finally:
            stepper.close()
        print(want, got)
        for i, (a, b) in enumerate(zip(want, got)):
            tol = 2e-4 if deterministic else (2e-3 if i < 3 else 5e-3)
            assert abs(a - b) <= tol * max(abs(a), 1e-6), (i, a, b)
        for k, v in net.state_dict().items():     # same trajectory: BatchNorm step counters agree exactly, weights closely
            if "num_batches_tracked" in k:
                assert torch.equal(v, want_state[k]), k
    assert sa.launch_options()[0] == 0


def test_pipelined_eager_step_takes_ragged_batches(cuda_device):
    """graph=False: batches may change their cloud sizes from step to step (augmented data)."""
    from dl_biomass_b200.train import PipelinedTrainStep, make_optimizer, train_step
    batches = [Batch.from_data_list(synthetic_clouds(700 + 13 * i, 3, 512, 1, True)).to(cuda_device) for i in range(3)]
    assert len({tuple(b.cloud_sizes) for b in batches}) == 3

    def fresh():
        torch.manual_seed(9)
        net = Net(1, "ReLU", 0, 0.0, precision="bf16").to(cuda_device).set_random_start(False)
        net.train()
        return net

    net = fresh()
    opt = make_optimizer(net.parameters())
    want = [float(train_step(net, opt, b)) for b in batches[:2]]
    net = fresh()
    opt = make_optimizer(net.parameters())
    with PipelinedTrainStep(net, opt, batches[0], graph=False) as stepper:
        got = [float(stepper.step(b)) for b in batches[1:3]]
    for a, b in zip(want, got):
        assert abs(a - b) <= 2e-3 * max(abs(a), 1e-6)


@pytest.mark.parametrize("precision", ["fp32", "bf16"])
def test_precomputed_grouping_gives_identical_results(cuda_device, precision):
    """Net.sample(grouping=True) (FPS + ball query + row compaction + gathered level-1 operand ahead of time) feeds
    forward/backward the very same numbers as computing them inside forward."""
    b = Batch.from_data_list(synthetic_clouds(321, 3, 640, 1, True)).to(cuda_device)
    torch.manual_seed(11)
    net = Net(1, "ReLU", 0, 0.0, precision=precision).to(cuda_device).set_random_start(False)
    net.train()
    state = {k: v.clone() for k, v in net.state_dict().items()}
    outs, grads = [], []
    for pre in (False, True):
        net.load_state_dict(state)
        net.zero_grad(set_to_none=True)
        samp = net.sample(b) if pre else None
        if pre:
            assert samp.group1 is not None and (samp.group1[2] is not None) == (precision == "bf16")
            assert (samp.group1[3] is not None) == (precision == "bf16") and samp.group2[3] is None
            assert len(samp.clone().tensors()) == len(samp.tensors())
        out = net(b, sampling=samp)
        out.square().sum().backward()
        outs.append(out.detach().clone())
        grads.append([p.grad.detach().clone() for p in net.parameters()])
    assert torch.equal(outs[0], outs[1])
    names = [n for n, _ in net.named_parameters()]
    scale = max(float(g.abs().max()) for g in grads[0])
    scale1 = max(float(g.abs().max()) for n, g in zip(names, grads[0]) if n.startswith("sa1_module"))
    for n, ga, gb in zip(names, *grads):
        # same products; the order of the partial sums (fp32 atomics) may differ in the last bits.  Level 1 sits below
        # level 2's atomic scatter-add, and its BatchNorm backward (differences of nearly equal sums) amplifies that
        # rounding freedom (bf16 path; the fp32 path keeps the tight bound)
        if precision == "bf16" and n.startswith("sa1_module"):
            assert float((ga - gb).abs().max()) <= SA1_SPREAD_BOUND * scale1, n
        else:
            assert float((ga - gb).abs().max()) <= 1e-4 * float(ga.abs().max()) + 1e-6 * scale, n


def test_deterministic_mode_gives_bit_identical_gradients(cuda_device):
    """b2pn_sa_args::deterministic: the dW split partials are summed in a fixed order and the feature gradient a level
    scatters into its source points is accumulated in 64-bit fixed point (integer atomics are order-independent), so
    EVERY gradient of the network is bit-identical from run to run -- level 1 included, which sits below level 2's
    scatter.  The default mode (fp32 atomics) agrees with it to rounding; its measured run-to-run spread is in
    profiles/r02_grad_spread.md."""
    from dl_biomass_b200 import sa
    b = Batch.from_data_list(synthetic_clouds(77, 3, 1024, 1, False)).to(cuda_device)
    torch.manual_seed(2)
    net = Net(1, "ReLU", 0, 0.0, precision="bf16").to(cuda_device).set_random_start(False)
    net.train()
    state = {k: v.clone() for k, v in net.state_dict().items()}
    names = [n for n, _ in net.named_parameters()]

    def grads():
        net.load_state_dict(state)
        net.zero_grad(set_to_none=True)
        net(b).square().sum().backward()
        return [p.grad.detach().clone() for p in net.parameters()]

    with sa.options(deterministic=True):
        g1, g2, g2b = grads(), grads(), grads()
    assert sa.launch_options() == (0, 0)
    g3 = grads()
    scale = max(float(g.abs().max()) for g in g1)
    scale1 = max(float(g.abs().max()) for n, g in zip(names, g1) if n.startswith("sa1_module"))
    for n, a, c, c2, e in zip(names, g1, g2, g2b, g3):
        assert torch.equal(a, c) and torch.equal(a, c2), n
        if n.startswith("sa1_module"):
            # default mode: level 1 sits downstream of level 2's fp32 atomic scatter-add (see the spread table)
            assert float((a - e).abs().max()) <= SA1_SPREAD_BOUND * scale1, n
        else:
            assert float((a - e).abs().max()) <= 1e-4 * float(a.abs().max()) + 1e-6 * scale, n


@pytest.mark.parametrize("B,n", [(5, 700), (40, 1500)])
def test_eval_mode_single_launch_levels_vs_oracle(cuda_device, B, n):
    """Evaluation (BatchNorm on running statistics, no grad: /root/reference/testing_model.py:56-64): every SLOTS level
    is ONE launch (csrc/sa_chain.cuh: gather -> MMA1 -> MMA2 -> MMA3 -> max, no hidden activation stored) and the head
    takes any number of clouds.  Outputs within 2e-2 of the fp32 oracle (measured ~2e-3), equal to the multi-pass
    kernels' to 16-bit rounding, and the launch count per level drops from 7 to 2 (weight packing + the level)."""
    from dl_biomass_b200 import _lib
    b = Batch.from_data_list(synthetic_clouds(99, B, n, 1, True))
    netr, net = _net_pair(cuda_device, "bf16", False)
    # give the running statistics something non-trivial: a few training steps' worth of updates on the oracle
    netr.train()
    with torch.no_grad():
        for i in range(2):
            netr(Batch.from_data_list(synthetic_clouds(500 + i, 4, 600, 1, True)))
    netr.eval()
    net.load_state_dict(netr.state_dict())
    net.eval()
    with torch.no_grad():
        want = netr(b)
        bg = b.to(cuda_device)
        l0 = _lib.lib().b2pn_launch_count()
        out = net(bg)
        fused_launches = _lib.lib().b2pn_launch_count() - l0
    with torch.enable_grad():      # the multi-pass kernels (hidden activations stored): same numbers to rounding
        l0 = _lib.lib().b2pn_launch_count()
        bg2 = b.to(cuda_device)
        bg2.x = bg2.x.clone().requires_grad_(True)
        out2 = net(bg2)
        multi_launches = _lib.lib().b2pn_launch_count() - l0
    torch.cuda.synchronize()
    err = rel_err(out, want)
    print("eval fused rel err", err, "vs multi-pass", rel_err(out, out2), "launches", fused_launches, multi_launches)
    assert err < 2e-2
    assert rel_err(out, out2) < 5e-3
    assert fused_launches <= multi_launches - 10
