"""The float64 evaluation reference (oracle/sa_eval_ref.py) is right: with every rounding switched off it equals the
float64 modules of oracle/ref.py in eval mode (point_conv_ref, GlobalSAModuleRef, MLPRef) to 1e-10, in both BatchNorm
variants, empty neighbourhoods included; and each injected fault E1, E2, E4, E5, E6 moves some output by more than 3x
the bounds of tests/test_sa_eval_gpu.py, E7 every out16 value.  E3 (the lo half of split inputs lost, a 2^-12 relative
input error) is reported only: at these shapes it moves the output by about one bound, the size of a correct kernel's
16-bit rounding noise.  The test also reports which faults the older evaluation bounds let through."""
import pytest
import torch

from oracle import ref
from oracle import sa_eval_ref as er

F64 = torch.float64
TOL = er.GPU_TOL


def _eval_mlp(chans, seed, act="ReLU"):
    mlp = ref.seeded_init_(ref.MLPRef(chans, act=act), seed).double()
    with torch.no_grad():   # non-trivial running statistics
        g = torch.Generator().manual_seed(seed + 7)
        for n in mlp.norms:
            n.running_mean.copy_(torch.rand(n.running_mean.shape, generator=g, dtype=F64) - 0.5)
            n.running_var.copy_(torch.rand(n.running_var.shape, generator=g, dtype=F64) + 0.5)
    return mlp.eval()


def _slots_problem(c_in, cnts, seed, dtype=F64, K=None):
    g = torch.Generator().manual_seed(seed)
    K = K or max(max(cnts), 1)
    n_src = 3 * K + 17
    pos = (torch.randn(n_src, 3, generator=g, dtype=F64) * 2).to(dtype)
    x = None if c_in == 0 else torch.randn(n_src, c_in, generator=g, dtype=F64).to(dtype)
    pos_dst = torch.randn(len(cnts), 3, generator=g, dtype=F64).to(dtype)
    nbr = torch.full((len(cnts), K), -1, dtype=torch.int32)
    for m, c in enumerate(cnts):
        nbr[m, :c] = torch.randperm(n_src, generator=g)[:c].sort().values.to(torch.int32)
    return x, pos, pos_dst, nbr, torch.tensor(cnts, dtype=torch.int32)


# neighbour counts 1, 8, 9 and 64 (one row, one whole 8-row group, a group and a row, a whole 64-row block) and an
# empty neighbourhood in the middle
CNTS = [1, 8, 9, 64, 0, 5, 64, 17, 1, 33]


@pytest.mark.parametrize("bn", ["fused", "multipass"])
@pytest.mark.parametrize("c_in,chans", [(0, [3, 16, 16, 24]), (1, [4, 16, 24, 40]), (16, [19, 32, 16, 24]),
                                        (128, [131, 32, 32, 24])])
def test_eval_slots_match_point_conv_f64(c_in, chans, bn):
    x, pos, pos_dst, nbr, cnt = _slots_problem(c_in, CNTS, 3)
    mlp = _eval_mlp(chans, 4)
    with torch.no_grad():
        want = ref.point_conv_ref(mlp, x, pos, pos_dst, *ref.slots_to_edges(nbr, cnt))
    rows = er.Rows(len(CNTS), nbr=nbr, cnt=cnt)
    got = er.eval_level(x, pos, er.params_of(mlp), rows, pos_dst=pos_dst, bn=bn, rnd=er.ROUND_NONE)
    assert er.rel_err(got["out"], want) <= 1e-10
    assert torch.all(got["out"][CNTS.index(0)] == 0)


@pytest.mark.parametrize("bn", ["fused", "multipass"])
def test_eval_clouds_match_global_module_f64(bn):
    g = torch.Generator().manual_seed(5)
    sizes = [130, 1, 257, 64]          # ragged, one cloud of a single row
    n = sum(sizes)
    x = torch.randn(n, 12, generator=g, dtype=F64)
    pos = torch.randn(n, 3, generator=g, dtype=F64) * 3
    batch = torch.repeat_interleave(torch.arange(len(sizes)), torch.tensor(sizes))
    mlp = _eval_mlp([15, 32, 48, 40], 9)
    with torch.no_grad():
        want, _, _ = ref.GlobalSAModuleRef(mlp)(x, pos, batch, len(sizes))
    got = er.eval_level(x, pos, er.params_of(mlp), er.Rows(len(sizes), batch=batch), bn=bn, rnd=er.ROUND_NONE)
    assert er.rel_err(got["out"], want) <= 1e-10


def test_eval_head_matches_mlp_f64():
    mlp = _eval_mlp([1024, 128, 128, 4], 6, act=None)
    x = torch.randn(70, 1024, generator=torch.Generator().manual_seed(2), dtype=F64)
    with torch.no_grad():
        want = mlp(x)
    assert er.rel_err(er.eval_head(x, er.params_of(mlp)), want) <= 1e-10


def test_rounding_switches_are_the_only_difference():
    """Each rounding switch on its own moves the output (so each is wired), and all of them together stay within a few
    fp16 ulps of the exact value."""
    x, pos, pos_dst, nbr, cnt = _slots_problem(1, CNTS, 3, dtype=torch.float32)
    p = er.params_of(_eval_mlp([4, 64, 64, 128], 4))
    rows = er.Rows(len(CNTS), nbr=nbr, cnt=cnt)
    exact = er.eval_level(x, pos, p, rows, pos_dst=pos_dst, rnd=er.ROUND_NONE)["out"]
    for k in ("w16", "split", "act16"):
        one = er.EvalRounding(**{f: f == k for f in ("w16", "split", "x16", "act16")})
        assert er.rel_err(er.eval_level(x, pos, p, rows, pos_dst=pos_dst, rnd=one)["out"], exact) > 0, k
    x2 = torch.randn(x.shape[0], 40, generator=torch.Generator().manual_seed(8))
    p2 = er.params_of(_eval_mlp([43, 64, 64, 128], 4))
    e2 = er.eval_level(x2, pos, p2, rows, pos_dst=pos_dst, rnd=er.ROUND_NONE)["out"]
    only_x = er.EvalRounding(False, False, True, False)
    assert er.rel_err(er.eval_level(x2, pos, p2, rows, pos_dst=pos_dst, rnd=only_x)["out"], e2) > 0
    assert er.rel_err(er.eval_level(x, pos, p, rows, pos_dst=pos_dst)["out"], exact) < 2e-3


def fault_distance(bad, good):
    """How far a faulted reference lies from the correct one, in units of the GPU bounds (out), or as the number of
    differing out16 values (whose bound is bit equality)."""
    d = max(er.ulp_err(bad["out"], good["out"]) / TOL["out_ulp"], er.rel_err(bad["out"], good["out"]) / TOL["out_rel"],
            er.rms_err(bad["out"], good["out"]) / TOL["out_rms"])
    n16 = int((bad["out16"] != good["out16"]).sum())
    return d, n16


# the two reference levels' shapes: fp32 x split into hi + lo, and fp16 features from the previous level
FAULT_CASES = {"level1": dict(c_in=1, chans=[4, 64, 64, 128], x16=False),
               "level2": dict(c_in=128, chans=[131, 128, 128, 256], x16=True)}


@pytest.mark.parametrize("case", list(FAULT_CASES))
@pytest.mark.parametrize("fault", list(er.FAULTS))
def test_eval_faults_exceed_bounds(case, fault):
    c = FAULT_CASES[case]
    g = torch.Generator().manual_seed(11)
    cnts = torch.randint(1, 65, (160,), generator=g).tolist()
    x, pos, pos_dst, nbr, cnt = _slots_problem(c["c_in"], cnts, 21, dtype=torch.float32)
    if c["x16"]:
        x = x.abs().half()      # a previous level's non-negative fp16 output
    p = er.params_of(_eval_mlp(c["chans"], 4))
    rows = er.Rows(len(cnts), nbr=nbr, cnt=cnt)
    good = er.eval_level(x, pos, p, rows, pos_dst=pos_dst)
    bad = er.eval_level(x, pos, p, rows, pos_dst=pos_dst, fault=fault)
    d, n16 = fault_distance(bad, good)
    rel = er.rel_err(bad["out"], good["out"])
    accepted = [k for k, b in er.OLD_TOL.items() if rel < b]
    print(f"{case} {fault} ({er.FAULTS[fault]}): {d:.1f}x the new bounds, rel {rel:.2e}, "
          f"rms {er.rms_err(bad['out'], good['out']):.2e}, ulp {er.ulp_err(bad['out'], good['out']):.1f}, out16 differs in {n16}; "
          f"accepted by the old bounds: {accepted or 'none'}")
    if fault == "E7":
        assert d == 0 and n16 > 0.5 * good["out16"].numel()
    elif fault != "E3":
        assert d > 3.0, (fault, d)
