"""The fused regression head (csrc/head.cu) in training mode against its float64 restatement (oracle/head_ref.py),
replaying the dropout masks the kernel saved: output, x.grad, every parameter gradient, the running statistics and
num_batches_tracked, at both head_lin0_kernel instances (<16> for B <= 16, <32> above), with staged and unstaged
weights, and at input widths whose last column slice of the backward is short.  Each case prints its errors, bounds, the distance of
the nearest injected fault (H1-H4) and the kernels it launched.  Tolerances: oracle/head_ref.py gpu_tol(B)."""
import pytest
import torch

from oracle import head_ref as hr
from dl_biomass_b200 import head
from dl_biomass_b200.pointnet2_regressor import MLP

F64 = torch.float64


def _head(chans, p, dev, seed=3):
    torch.manual_seed(seed)
    m = MLP(chans, act=None, dropout=p).to(dev)
    for n in m.norms:  # non-trivial affine + running stats
        n.weight.data.uniform_(0.5, 1.5)
        n.bias.data.uniform_(-0.5, 0.5)
        n.running_mean.uniform_(-0.2, 0.2)
        n.running_var.uniform_(0.5, 2.0)
    return m


def _params(m):
    P = {}
    for i, lin in enumerate(m.lins):
        P[f"w{i}"], P[f"b{i}"] = lin.weight.detach().cpu(), lin.bias.detach().cpu()
    for i, n in enumerate(m.norms):
        P[f"gamma{i}"], P[f"beta{i}"] = n.weight.detach().cpu(), n.bias.detach().cpu()
        P[f"rm{i}"], P[f"rv{i}"] = n.running_mean.detach().cpu().clone(), n.running_var.detach().cpu().clone()
    return P


def _kernel_names(fn):
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        # the profiler's kernel list on the B200 misses the first kernel launched inside the profiled region: a
        # throw-away kernel goes first so that head_lin0_kernel is listed
        torch.ones(1, device="cuda").add_(1)
        res = fn()
        torch.cuda.synchronize()
    return res, sorted({e.name.split("(")[0] for e in prof.events() if e.device_type == torch.autograd.DeviceType.CUDA})


def _grads(m, x):
    g = {}
    for i, lin in enumerate(m.lins):
        g[f"w{i}"], g[f"b{i}"] = lin.weight.grad, lin.bias.grad
    for i, n in enumerate(m.norms):
        g[f"gamma{i}"], g[f"beta{i}"] = n.weight.grad, n.bias.grad
    g["x"] = x.grad
    return {k: v.detach().cpu() for k, v in g.items()}


CHANS = {"1024": [1024, 128, 128, 4],    # the reference head: weights staged in shared memory
         "2048": [2048, 256, 256, 4],    # too wide to stage: weights read from global memory
         "300": [300, 128, 128, 4],      # 5 column slices of 60: the slices divide c0 evenly
         "1000": [1000, 128, 128, 4]}    # 16 slices of 63: the last one has 55 columns


@pytest.mark.gpu
@pytest.mark.parametrize("shape", list(CHANS))
@pytest.mark.parametrize("p", [0.0, 0.5])
@pytest.mark.parametrize("B", [2, 5, 16, 17, 31, 32])
def test_head_train_pinned_f64(cuda_device, B, p, shape):
    chans = CHANS[shape]
    dev = cuda_device
    TOL = hr.gpu_tol(B)
    m = _head(chans, p, dev)
    m.train()
    P = _params(m)
    g = torch.Generator().manual_seed(B)
    x = torch.randn(B, chans[0], generator=g).to(dev).requires_grad_(True)
    gout = torch.randn(B, chans[3], generator=g)
    counter = torch.zeros((), dtype=torch.int64, device=dev)
    assert head.supported(m, x)

    def step():
        out = head.head_apply(m, x, counter, 11)
        saved = [t.detach().cpu() for t in out.grad_fn.saved_tensors]
        out.backward(gout.to(dev))
        return out, saved

    (out, saved), names = _kernel_names(step)
    masks = saved[3:5]
    if p == 0.0:
        assert all(bool((mk == 1).all()) for mk in masks)
    else:   # the kernel really dropped about half of the values
        frac = float(torch.cat([mk.flatten() for mk in masks]).float().mean())
        assert 0.3 < frac < 0.7, frac
    fw = hr.forward(P, x.detach().cpu(), masks, p)
    want = hr.backward(P, x.detach().cpu(), fw, gout, p)
    got = _grads(m, x)
    errs = hr.grad_errors(got, want)
    errs["out"] = float((out.detach().cpu().to(F64) - fw["out"]).abs().max() / fw["out"].abs().max())
    for l, n in enumerate(m.norms):
        errs[f"run_mean{l}"] = float((n.running_mean.cpu().to(F64) - fw[f"run_mean{l}"]).abs().max()
                                     / fw[f"run_mean{l}"].abs().max())
        errs[f"run_var{l}"] = float((n.running_var.cpu().to(F64) - fw[f"run_var{l}"]).abs().max()
                                    / fw[f"run_var{l}"].abs().max())
        assert int(n.num_batches_tracked) == 1
    tol = {k: TOL["run" if k.startswith("run_") else k] for k in errs}
    # faults: each one that moves the reference past 3 tolerances must lie more than 3 tolerances from the kernel
    seps = {}
    for f in hr.FAULTS:
        bfw = hr.forward(P, x.detach().cpu(), masks, p, fault=f if f == "H2" else None)
        bad = hr.backward(P, x.detach().cpu(), bfw, gout, p, fault=None if f == "H2" else f)
        moved = hr.grad_errors(bad, want)
        moved["out"] = float((bfw["out"] - fw["out"]).abs().max() / fw["out"].abs().max())
        if max(v / TOL[k] for k, v in moved.items()) < 3.0:
            continue      # e.g. H3 without dropout
        dist = hr.grad_errors(got, bad)
        dist["out"] = float((out.detach().cpu().to(F64) - bfw["out"]).abs().max() / bfw["out"].abs().max())
        seps[f] = max(v / TOL[k] for k, v in dist.items())
    print(f"\n[head B={B} p={p} {chans}]  kernels {names}")
    for k, e in errs.items():
        print(f"  {k:<10} {e:11.3e}  bound {tol[k]:9.2e}")
    for f, s in seps.items():
        print(f"  {f} at {s:9.1f}x tol")
    lin0 = "head_lin0_kernel<16>" if B <= 16 else "head_lin0_kernel<32>"
    assert any(lin0 in n for n in names), names
    assert any("head_forward_kernel" in n for n in names) and any("head_backward_kernel" in n for n in names), names
    bad = {k: e for k, e in errs.items() if not e <= tol[k]}
    assert not bad, bad
    assert all(s > 3.0 for s in seps.values()), seps
    if p == 0.0:
        assert "H1" in seps and "H2" in seps and "H4" in seps, seps
    elif B > 2:
        assert "H3" in seps, seps


@pytest.mark.gpu
def test_head_train_single_row_raises(cuda_device):
    """BatchNorm1d refuses to train on one row (there is no variance to normalise with); so does the fused head,
    before anything is launched or any running statistic changes."""
    m = _head([64, 32, 32, 4], 0.0, cuda_device)
    m.train()
    x = torch.randn(1, 64, device=cuda_device)
    with pytest.raises(ValueError):
        m(x)                       # the layer-by-layer evaluation, i.e. torch's BatchNorm1d
    before = [b.clone() for b in m.buffers()]
    counter = torch.zeros((), dtype=torch.int64, device=cuda_device)
    with pytest.raises(ValueError, match="more than 1 value per channel"):
        head.head_apply(m, x, counter, 5)
    assert all(torch.equal(a, b) for a, b in zip(before, m.buffers()))
    # the library refuses it too (B2PN_EINVAL), on real buffers, and accepts the same call in evaluation mode
    import ctypes
    from dl_biomass_b200 import _lib
    dev = cuda_device
    out = torch.zeros(1, 4, device=dev)
    saved = (torch.zeros(1, 32, device=dev), torch.zeros(1, 32, device=dev),
             torch.zeros(1, 32, dtype=torch.uint8, device=dev), torch.zeros(1, 32, dtype=torch.uint8, device=dev),
             torch.zeros(32, device=dev), torch.zeros(32, device=dev))
    for training, rc in ((True, -1), (False, 0)):
        a = _lib.HeadArgs()
        head._fill(a, x, m, training, 0.0, out, saved, 5, counter)
        assert _lib.lib().b2pn_head_forward(ctypes.byref(a), torch.cuda.current_stream(dev).cuda_stream) == rc
        torch.cuda.synchronize()
        if training:
            assert all(torch.equal(a_, b_) for a_, b_ in zip(before, m.buffers())) and not out.any()
    m.eval()                       # evaluation normalises with the running statistics: one row is fine
    assert head.head_apply(m, x, counter, 5).shape == (1, 4)
