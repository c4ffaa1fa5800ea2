"""CPU: the oracle against the committed golden vectors (incl. the reference's own numpy FPS)."""
import os

import numpy as np
import torch

from oracle import ref
from dl_biomass_b200.data import Batch, Data, synthetic_clouds

GOLD = os.path.join(os.path.dirname(__file__), "golden")


def test_fps_matches_reference_numpy_fps():
    """Golden = /root/reference/downsampling_point_clouds.py:55-92 run in place (oracle/gen_golden.py)."""
    g = np.load(os.path.join(GOLD, "fps_reference_numpy.npz"))
    kinds = g["kinds"]
    for i, kind in enumerate(kinds):
        pos, idx = g[f"pos_{i}"], g[f"idx_{i}"]
        got64 = ref.fps_ref_f64(pos, len(idx), 0)
        assert np.array_equal(got64, idx), f"f64 case {i}"
        if kind == "dyadic":  # fp32 arithmetic is exact on these clouds -> the fp32 oracle must agree too
            p32 = torch.from_numpy(pos.astype(np.float32))
            ptr = torch.tensor([0, pos.shape[0]])
            ratio = len(idx) / pos.shape[0]
            assert ref.fps_num_samples(pos.shape[0], ratio) == len(idx)
            got32 = ref.fps_ref(p32, ptr, ratio)
            assert np.array_equal(got32.numpy(), idx), f"f32 case {i}"


def test_num_samples_rule():
    # SURVEY.md A.1: ceil(float32(n) * float32(ratio))
    assert ref.fps_num_samples(10000, 0.2) == 2000
    assert ref.fps_num_samples(2000, 0.25) == 500
    assert ref.fps_num_samples(7168, 0.2) == 1434
    assert ref.fps_num_samples(1434, 0.25) == 359
    assert ref.fps_num_samples(9999, 0.2) == 2000
    assert ref.fps_num_samples(100000, 0.2) == 20000
    assert ref.fps_num_samples(1, 0.2) == 1


def _torch_fps(pos, m, start=0):
    d = ((pos - pos[start]) ** 2).sum(1)
    out = [start]
    for _ in range(m - 1):
        a = int(d.argmax())
        out.append(a)
        d = torch.minimum(d, ((pos - pos[a]) ** 2).sum(1))
    return torch.tensor(out)


def test_fps_and_ball_query_against_torch_restatement():
    b = Batch.from_data_list(synthetic_clouds(5, 3, 400, 1, ragged=True))
    start = torch.tensor([0, 17, 3])
    idx = ref.fps_ref(b.pos, b.ptr, 0.2, start)
    qptr = ref.sample_ptr(b.ptr, 0.2)
    for c in range(3):
        p = b.pos[b.ptr[c]:b.ptr[c + 1]]
        m = int(qptr[c + 1] - qptr[c])
        assert torch.equal(_torch_fps(p, m, int(start[c])) + b.ptr[c], idx[qptr[c]:qptr[c + 1]])
    q = b.pos[idx]
    nbr, cnt = ref.ball_query_ref(b.pos, q, b.ptr, qptr, 2.0, 16)
    for c in range(3):
        s = b.pos[b.ptr[c]:b.ptr[c + 1]]
        for i in range(int(qptr[c]), int(qptr[c + 1])):
            d2 = ((s - q[i]) ** 2).sum(1)
            w = torch.nonzero(d2 < 4.0).flatten()[:16] + b.ptr[c]
            assert int(cnt[i]) == w.numel()
            assert torch.equal(nbr[i, :w.numel()].long(), w)
            assert bool((nbr[i, w.numel():] == -1).all())


def test_grouping_golden_regression():
    g = np.load(os.path.join(GOLD, "grouping_oracle.npz"))
    i = 0
    while f"spec_{i}" in g:
        r1 = g[f"spec_{i}"][4]
        pos, ptr = torch.from_numpy(g[f"pos_{i}"]), torch.from_numpy(g[f"ptr_{i}"])   # the stored clouds
        idx1 = ref.fps_ref(pos, ptr, 0.2)
        assert np.array_equal(idx1.numpy(), g[f"idx1_{i}"])
        ptr1 = ref.sample_ptr(ptr, 0.2)
        nbr1, cnt1 = ref.ball_query_ref(pos, pos[idx1], ptr, ptr1, float(r1), 64)
        assert np.array_equal(nbr1.numpy(), g[f"nbr1_{i}"]) and np.array_equal(cnt1.numpy(), g[f"cnt1_{i}"])
        i += 1
    assert i == 3


def test_segment_max_first_tie_rule():
    msg = torch.tensor([[1.0, 5.0], [2.0, 5.0], [2.0, 0.0], [0.0, 7.0]], requires_grad=True)
    seg = torch.tensor([0, 0, 0, 1])
    out, arg = ref.segment_max_first(msg, seg, 3)
    assert out.tolist() == [[2.0, 5.0], [0.0, 7.0], [0.0, 0.0]]  # empty segment -> 0 (A.3)
    out.sum().backward()
    assert msg.grad.tolist() == [[0.0, 1.0], [1.0, 0.0], [0.0, 0.0], [1.0, 1.0]]  # first arg-max row only


def test_net_oracle_golden_regression():
    """The oracle network on the stored clouds, in float64 like the fixture (oracle/gen_golden.py): in float32 its
    train-mode gradients of levels 1-2 depend on the host's summation order (thread count, CPU kernels) by up to ~0.5 %."""
    gold = torch.load(os.path.join(GOLD, "net_oracle.pt"))
    F = gold["spec"][3]
    b = Batch.from_data_list([Data(**c) for c in gold["clouds"]])
    b.x, b.pos = b.x.double(), b.pos.double()
    for mode in ("train", "eval"):
        net = ref.seeded_init_(ref.NetRef(F, "ReLU", 0, 0.0), seed=gold["init_seed"]).double()
        net.train(mode == "train")
        out = net(b)
        torch.testing.assert_close(out, gold["modes"][mode]["out"], rtol=1e-4, atol=1e-5)
        loss = ref.weighted_mse(out, b.y)
        loss.backward()
        for k, p in net.named_parameters():
            torch.testing.assert_close(p.grad.flatten()[:16], gold["modes"][mode]["grad_head"][k], rtol=2e-3, atol=1e-5)


def test_state_dict_keys_are_pyg_shaped():
    net = ref.NetRef(1, "ReLU", 0, 0.5)
    keys = set(net.state_dict().keys())
    for k in ("sa1_module.conv.local_nn.lins.0.weight", "sa2_module.conv.local_nn.norms.1.running_var",
              "sa3_module.nn.lins.2.bias", "mlp.lins.2.weight", "mlp.norms.0.num_batches_tracked"):
        assert k in keys
    assert sum(p.numel() for p in net.parameters()) == 953732  # SURVEY.md §8 a1


def test_ball_query_against_scipy_kdtree():
    """Independent cross-check of the oracle's neighbourhoods (membership, per-cloud restriction, first-K-by-index cap)
    against scipy's cKDTree -- the same family of structure torch_cluster's CPU path (nanoflann) uses.  Coordinates
    sit on a 1/16 grid so fp32 (oracle) and float64 (scipy) distances are both exact; the radius is chosen off the
    grid's distance set, and a separate case pins the strict '<' of SURVEY.md A.2."""
    from scipy.spatial import cKDTree
    rng = np.random.default_rng(3)
    sizes = [300, 1, 157, 420]
    pts = [rng.integers(-32, 32, size=(n, 3)).astype(np.float64) / 16.0 for n in sizes]
    ptr = torch.tensor(np.concatenate([[0], np.cumsum(sizes)]))
    pos = torch.from_numpy(np.concatenate(pts).astype(np.float32))
    q_idx, qptr = [], [0]
    for c, n in enumerate(sizes):
        take = np.sort(rng.choice(n, size=max(1, n // 5), replace=False))
        q_idx.append(take + int(ptr[c]))
        qptr.append(qptr[-1] + len(take))
    q_idx = torch.from_numpy(np.concatenate(q_idx))
    qptr = torch.tensor(qptr)
    r, K = 1.3, 12                                # 1.69 is not a sum of three squares of multiples of 1/16
    nbr, cnt = ref.ball_query_ref(pos, pos[q_idx], ptr, qptr, r, K)
    full = 0
    for c, n in enumerate(sizes):
        tree = cKDTree(pts[c])
        for i in range(int(qptr[c]), int(qptr[c + 1])):
            local = np.sort(np.asarray(tree.query_ball_point(pts[c][int(q_idx[i]) - int(ptr[c])], r)))
            want = local[:K] + int(ptr[c])
            full += len(local) > K
            assert int(cnt[i]) == len(want)
            assert np.array_equal(nbr[i, :len(want)].numpy(), want)
            assert bool((nbr[i, len(want):] == -1).all())
    assert full > 10                              # the cap was exercised
    # strictness: a source at distance exactly r is NOT a neighbour
    src = torch.tensor([[0.0, 0.0, 0.0], [2.0, 0.0, 0.0], [1.9375, 0.0, 0.0]])
    nbr, cnt = ref.ball_query_ref(src, src[:1], torch.tensor([0, 3]), torch.tensor([0, 1]), 2.0, 4)
    assert int(cnt[0]) == 2 and nbr[0, :2].tolist() == [0, 2]


def test_segment_max_against_torch_scatter_reduce():
    """Values of the max aggregation against torch's own scatter_reduce(amax) (the ATen op behind current
    torch_geometric's `aggr='max'`); the arg rule (first row attaining the max) against numpy."""
    g = torch.Generator().manual_seed(1)
    seg = torch.sort(torch.randint(0, 40, (500,), generator=g)).values
    msg = torch.randint(-3, 4, (500, 7), generator=g).float()          # many ties
    out, arg = ref.segment_max_first(msg, seg, 41)                    # segment 40 may be empty
    want = torch.full((41, 7), float("-inf")).scatter_reduce(0, seg[:, None].expand(-1, 7), msg, "amax", include_self=True)
    present = torch.bincount(seg, minlength=41) > 0
    assert torch.equal(out[present], want[present]) and bool((out[~present] == 0).all())
    m, s = msg.numpy(), seg.numpy()
    for k in np.nonzero(present.numpy())[0]:
        rows = np.nonzero(s == k)[0]
        assert np.array_equal(arg[k].numpy(), rows[np.argmax(m[rows], axis=0)])
