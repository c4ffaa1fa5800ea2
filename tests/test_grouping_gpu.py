"""GPU parity (bit-exact) of Kernel 1 (FPS) and Kernel 2 (ball query) against the oracle."""
import os

import numpy as np
import pytest
import torch

from oracle import ref
from dl_biomass_b200 import _lib, ops
from dl_biomass_b200.data import Batch, synthetic_clouds

pytestmark = pytest.mark.gpu
GOLD = os.path.join(os.path.dirname(__file__), "golden")


def _run_level(pos_cpu, sizes, ratio, r, dev, start=None, K=64, variant=(0, 0)):
    lv = ops.build_levels(sizes, [ratio], dev)
    pos = pos_cpu.to(dev)
    st = None if start is None else start.to(dev)
    idx, pos_out, batch_out = ops.fps(pos, lv[0], lv[1], st, cluster=variant[0], threads=variant[1])
    nbr, cnt = ops.ball_query(pos, pos_out, lv[0], lv[1], r, K)
    torch.cuda.synchronize()
    return lv, idx.cpu(), pos_out.cpu(), batch_out.cpu(), nbr.cpu(), cnt.cpu()


def _check_level(pos_cpu, ptr, ratio, r, dev, start=None, K=64, variant=(0, 0)):
    sizes = (ptr[1:] - ptr[:-1]).tolist()
    lv, idx, pos_out, batch_out, nbr, cnt = _run_level(pos_cpu, sizes, ratio, r, dev, start, K, variant)
    want_idx = ref.fps_ref(pos_cpu, ptr, ratio, start)
    assert torch.equal(idx, want_idx), f"fps mismatch at {int((idx != want_idx).nonzero()[0])}"
    assert torch.equal(pos_out, pos_cpu[want_idx])
    qptr = ref.sample_ptr(ptr, ratio)
    assert torch.equal(batch_out, torch.repeat_interleave(torch.arange(len(sizes)), qptr[1:] - qptr[:-1]))
    want_nbr, want_cnt = ref.ball_query_ref(pos_cpu, pos_cpu[want_idx], ptr, qptr, r, K)
    assert torch.equal(cnt, want_cnt)
    assert torch.equal(nbr, want_nbr)
    return idx, nbr, cnt


@pytest.mark.parametrize("B,n,ragged", [(1, 64, False), (3, 1000, False), (4, 513, True), (2, 4099, True),
                                        (12, 10000, False)])
def test_two_levels_match_oracle(cuda_device, B, n, ragged):
    b = Batch.from_data_list(synthetic_clouds(1234, B, n, 1, ragged))
    idx1, _, _ = _check_level(b.pos, b.ptr, 0.2, 2.0, cuda_device)
    ptr1 = ref.sample_ptr(b.ptr, 0.2)
    _check_level(b.pos[idx1].contiguous(), ptr1, 0.25, 8.0, cuda_device)


def test_explicit_start_and_small_k(cuda_device):
    b = Batch.from_data_list(synthetic_clouds(8, 3, 700, 1, True))
    _check_level(b.pos, b.ptr, 0.2, 3.0, cuda_device, start=torch.tensor([5, 0, 333]), K=16)


def test_ties_and_duplicates(cuda_device):
    """Dyadic grid clouds are full of exactly tied distances; duplicated points add zero distances."""
    rng = np.random.default_rng(3)
    pts = torch.from_numpy(rng.integers(-32, 32, size=(3000, 3)).astype(np.float32) / 4.0)
    pts = torch.cat([pts, pts[:500]], 0)  # duplicates
    ptr = torch.tensor([0, 1200, 3500])
    _check_level(pts, ptr, 0.25, 2.0, cuda_device)
    _check_level(pts, ptr, 0.9, 1.0, cuda_device)  # nearly exhausts the clouds


@pytest.mark.parametrize("cluster,threads", [(-2, 256), (-2, 512), (-2, 640), (-1, 512), (1, 512), (2, 256)])
def test_ties_and_duplicates_all_variants(cuda_device, cluster, threads):
    """Every FPS variant (plain register scan, Morton-sorted scans, cluster kernels) breaks ties towards the lowest
    ORIGINAL index, whatever order it keeps the points in."""
    rng = np.random.default_rng(5)
    pts = torch.from_numpy(rng.integers(-16, 16, size=(4000, 3)).astype(np.float32) / 2.0)
    pts = torch.cat([pts, pts[:700]], 0)  # duplicates
    ptr = torch.tensor([0, 1700, 4700])
    _check_level(pts, ptr, 0.3, 2.0, cuda_device, variant=(cluster, threads))   # the variant is a per-call option
    _check_level(pts, ptr, 0.95, 1.0, cuda_device, variant=(cluster, threads))


@pytest.mark.parametrize("n,r,K", [(3000, 2.0, 64), (3000, 0.3, 64), (3000, 9.0, 64), (3000, 40.0, 64), (5000, 2.0, 8),
                                   (700, 1.0, 16), (40, 2.0, 64)])
def test_grid_ball_query_equals_scan(cuda_device, n, r, K):
    """The uniform-grid kernel (large clouds) returns exactly what the ascending scan returns: sparse and dense
    radii, a radius that swallows the whole cloud (list overflow -> in-kernel fall-back), duplicates, flat clouds."""
    clouds = synthetic_clouds(321, 3, n, 1, True)
    clouds[1].pos[:, 2] = 0.25                       # a flat cloud: one layer of cells
    clouds[2].pos[: n // 3] = clouds[2].pos[n // 3: 2 * (n // 3)][: n // 3]   # duplicates
    b = Batch.from_data_list(clouds)
    sizes = b.cloud_sizes
    lv = ops.build_levels(sizes, [0.2], cuda_device)
    pos = b.pos.to(cuda_device)
    _, qpos, _ = ops.fps(pos, lv[0], lv[1])
    old = ops.GRID_MIN_SOURCES
    try:
        nbr0, cnt0 = ops.ball_query(pos, qpos, lv[0], lv[1], r, K, mode="scan")
        ops.GRID_MIN_SOURCES = 0
        nbr1, cnt1 = ops.ball_query(pos, qpos, lv[0], lv[1], r, K, mode="auto")
        torch.cuda.synchronize()
    finally:
        ops.GRID_MIN_SOURCES = old
    assert torch.equal(cnt0, cnt1)
    assert torch.equal(nbr0, nbr1)
    # and the scan itself against the oracle
    qptr = ref.sample_ptr(b.ptr, 0.2)
    idx = ref.fps_ref(b.pos, b.ptr, 0.2)
    want_nbr, want_cnt = ref.ball_query_ref(b.pos, b.pos[idx], b.ptr, qptr, r, K)
    assert torch.equal(cnt1.cpu(), want_cnt) and torch.equal(nbr1.cpu(), want_nbr)


def test_reference_numpy_fps_golden(cuda_device):
    """The reference's own FPS (downsampling_point_clouds.py:55-92) on fp32-exact clouds."""
    g = np.load(os.path.join(GOLD, "fps_reference_numpy.npz"))
    for i, kind in enumerate(g["kinds"]):
        if kind != "dyadic":
            continue
        pos, want = g[f"pos_{i}"], g[f"idx_{i}"]
        n, k = pos.shape[0], len(want)
        lv = ops.build_levels([n], [k / n], cuda_device)
        assert lv[1].total == k
        idx, _, _ = ops.fps(torch.from_numpy(pos.astype(np.float32)).to(cuda_device), lv[0], lv[1])
        assert np.array_equal(idx.cpu().numpy(), want)


def test_golden_grouping_fixture(cuda_device):
    g = np.load(os.path.join(GOLD, "grouping_oracle.npz"))
    i = 0
    while f"spec_{i}" in g:
        r1, r2 = g[f"spec_{i}"][4:6]
        pos, ptr = torch.from_numpy(g[f"pos_{i}"]), torch.from_numpy(g[f"ptr_{i}"])   # the stored clouds
        sizes = (ptr[1:] - ptr[:-1]).tolist()
        lv, idx, pos1, _, nbr, cnt = _run_level(pos, sizes, 0.2, float(r1), cuda_device)
        assert np.array_equal(idx.numpy(), g[f"idx1_{i}"])
        assert np.array_equal(nbr.numpy(), g[f"nbr1_{i}"]) and np.array_equal(cnt.numpy(), g[f"cnt1_{i}"])
        lv2, idx2, _, _, nbr2, cnt2 = _run_level(pos1, lv[1].sizes, 0.25, float(r2), cuda_device)
        assert np.array_equal(idx2.numpy(), g[f"idx2_{i}"])
        assert np.array_equal(nbr2.numpy(), g[f"nbr2_{i}"]) and np.array_equal(cnt2.numpy(), g[f"cnt2_{i}"])
        i += 1


@pytest.mark.parametrize("cluster,threads", [(-2, 512), (-2, 640), (-2, 768), (-1, 256), (-1, 512), (-1, 1024), (1, 256), (1, 512), (1, 1024), (2, 512), (4, 256), (8, 256), (8, 512),
                                             (16, 256)])
def test_fps_variants_agree(cuda_device, cluster, threads):
    b = Batch.from_data_list(synthetic_clouds(77, 5, 6000, 1, True))
    want = ref.fps_ref(b.pos, b.ptr, 0.2)
    lv = ops.build_levels((b.ptr[1:] - b.ptr[:-1]).tolist(), [0.2], cuda_device)
    idx, _, _ = ops.fps(b.pos.to(cuda_device), lv[0], lv[1], cluster=cluster, threads=threads)
    torch.cuda.synchronize()
    assert torch.equal(idx.cpu(), want)


def test_random_start_is_drawn_in_the_kernel_and_advances(cuda_device):
    """random_start=True of torch_cluster.fps (SURVEY.md A.1): with an rng_state the kernel draws floor(u*n) per cloud
    from (seed, call counter, cloud), bumps the counter once per launch (so CUDA-graph replays draw fresh starts), and
    the result equals FPS from that explicit start."""
    b = Batch.from_data_list(synthetic_clouds(91, 4, 900, 1, True))
    sizes = b.cloud_sizes
    lv = ops.build_levels(sizes, [0.2], cuda_device)
    pos = b.pos.to(cuda_device)
    state = torch.zeros(2, dtype=torch.int64, device=cuda_device)
    seed = 123456789
    lib = _lib.lib()
    seen = []
    for call in range(3):
        idx, _, _ = ops.fps(pos, lv[0], lv[1], None, seed=seed, rng_state=state)
        torch.cuda.synchronize()
        assert state.tolist() == [call + 1, 0]
        start = torch.tensor([lib.b2pn_fps_random_start(seed, call, c, n) for c, n in enumerate(sizes)])
        assert all(0 <= int(s) < n for s, n in zip(start, sizes))
        first = idx.cpu()[lv[1].ptr.cpu()[:-1]] - b.ptr[:-1]
        assert torch.equal(first, start)
        assert torch.equal(idx.cpu(), ref.fps_ref(b.pos, b.ptr, 0.2, start))
        seen.append(tuple(start.tolist()))
    assert len(set(seen)) == 3          # fresh starts every call
    # CUDA-graph replays advance the counter too
    g = torch.cuda.CUDAGraph()
    s = torch.cuda.Stream(cuda_device)
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        ops.fps(pos, lv[0], lv[1], None, seed=seed, rng_state=state)
    torch.cuda.current_stream().wait_stream(s)
    with torch.cuda.graph(g):
        gidx, _, _ = ops.fps(pos, lv[0], lv[1], None, seed=seed, rng_state=state)
    firsts = []
    for _ in range(2):
        g.replay()
        torch.cuda.synchronize()
        firsts.append(tuple((gidx.cpu()[lv[1].ptr.cpu()[:-1]] - b.ptr[:-1]).tolist()))
    assert state.tolist() == [6, 0] and firsts[0] != firsts[1]


def test_dense_cloud_properties(cuda_device):
    """100k-point cloud (BASELINE config 4): too slow for a full oracle pass in CI, so check
    size-independent properties + an oracle prefix."""
    b = Batch.from_data_list(synthetic_clouds(11, 2, 100000, 1, False))
    lv = ops.build_levels([100000, 100000], [0.2], cuda_device)
    pos = b.pos.to(cuda_device)
    idx, pos_out, _ = ops.fps(pos, lv[0], lv[1])
    nbr, cnt = ops.ball_query(pos, pos_out, lv[0], lv[1], 4.0, 64)
    idx_c = idx.cpu()
    for c in range(2):
        seg = idx_c[c * 20000:(c + 1) * 20000]
        assert seg.unique().numel() == 20000 and int(seg.min()) >= c * 100000 and int(seg.max()) < (c + 1) * 100000
    # oracle on the first cloud only, first 300 samples (prefix of FPS is independent of the total count)
    ptr = torch.tensor([0, 100000])
    want = ref.fps_ref(b.pos[:100000], ptr, 300 / 100000)
    assert torch.equal(idx_c[:300], want)
    # neighbour slots: ascending, in range, within radius, and the centroid's own cloud
    nbr_c, cnt_c = nbr.cpu().long(), cnt.cpu().long()
    assert int(cnt_c.min()) >= 1
    q = torch.randint(0, 40000, (200,))
    for m in q.tolist():
        k = int(cnt_c[m])
        row = nbr_c[m, :k]
        assert bool((row[1:] > row[:-1]).all()) and bool((nbr_c[m, k:] == -1).all())
        d2 = ((b.pos[row] - b.pos[idx_c[m]]) ** 2).sum(1)
        assert bool((d2 < 16.0).all())
        want_n, want_c = ref.ball_query_ref(b.pos, b.pos[idx_c[m]][None], torch.tensor([0, 100000, 200000]),
                                            torch.tensor([0, 1, 1]) if m < 20000 else torch.tensor([0, 0, 1]), 4.0, 64)
        assert int(want_c[0]) == k and torch.equal(want_n[0, :k].long(), row)


# ---------------------------------------------------------------------------------------------------
#  offline resampler (SURVEY 8 f1): float64 FPS == the reference's numpy farthest_point_sampling
# ---------------------------------------------------------------------------------------------------
def test_resampler_matches_reference_numpy_golden(cuda_device):
    """Every golden case of /root/reference/downsampling_point_clouds.py:55-92 (run in place by oracle/gen_golden.py):
    dyadic, float64, raw UTM coordinates, duplicates that exhaust the cloud -- bit-exact, singly and as one batch."""
    from dl_biomass_b200 import resample
    g = np.load(os.path.join(GOLD, "fps_reference_numpy.npz"))
    n_cases = len(g["kinds"])
    for i in range(n_cases):
        got = resample.farthest_point_sampling(g[f"pos_{i}"], len(g[f"idx_{i}"]))
        assert np.array_equal(got, g[f"idx_{i}"]), (i, str(g["kinds"][i]))
    # batched: clouds that share k
    same_k = [i for i in range(n_cases) if len(g[f"idx_{i}"]) == 300]
    assert len(same_k) >= 2
    outs = resample.farthest_point_sampling_batch([g[f"pos_{i}"] for i in same_k], 300)
    for i, got in zip(same_k, outs):
        assert np.array_equal(got, g[f"idx_{i}"])


def test_resampler_matches_oracle_on_large_plot(cuda_device):
    from dl_biomass_b200 import resample
    rng = np.random.default_rng(11)
    pts = rng.normal(size=(20000, 3)) * np.array([5.0, 5.0, 9.0]) + np.array([431234.5, 5312345.25, 250.0])
    got = resample.farthest_point_sampling(pts, 2048)
    want = ref.fps_ref_f64(pts, 2048, 0)
    assert np.array_equal(got, want)
    assert len(set(got.tolist())) == 2048
    with pytest.raises(ValueError):
        resample.farthest_point_sampling(pts[:100], 200)
