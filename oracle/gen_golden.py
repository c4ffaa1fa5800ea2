"""Generate the committed golden fixtures under tests/golden/ (run in THIS container only).

1. fps_reference_numpy.npz -- produced by the reference's OWN numpy farthest_point_sampling
   (/root/reference/downsampling_point_clouds.py:55-92), executed in place: the function's source is
   pulled out of the reference file with ``ast`` at run time (its module cannot be imported because
   it needs laspy) and never copied into this repo.  Pins oracle_fps_f64 on float64 clouds and
   oracle_fps_f32 on dyadic-grid clouds where fp32 and fp64 arithmetic agree exactly.
2. grouping_oracle.npz / net_oracle.pt -- outputs of the oracle itself on seeded clouds (regression
   anchors for the oracle and expected values for the GPU parity tests; PARITY UNPINNED, see
   oracle/ref.py).
"""
import ast
import os
import sys

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from oracle import ref  # noqa: E402
from dl_biomass_b200.data import Batch, synthetic_clouds  # noqa: E402

GOLD = os.path.join(ROOT, "tests", "golden")
REF_FILE = "/root/reference/downsampling_point_clouds.py"


def reference_numpy_fps():
    tree = ast.parse(open(REF_FILE).read())
    fn = [n for n in tree.body if isinstance(n, ast.FunctionDef) and n.name == "farthest_point_sampling"][0]
    ns = {"np": np}
    exec(compile(ast.Module(body=[fn], type_ignores=[]), REF_FILE, "exec"), ns)
    return ns["farthest_point_sampling"]


def dyadic_cloud(rng, n):
    """coordinates k/16 in [-16,16): every difference, square and sum is exact in fp32 and fp64."""
    return rng.integers(-256, 256, size=(n, 3)).astype(np.float64) / 16.0


def gen_fps_reference():
    fps_np = reference_numpy_fps()
    rng = np.random.default_rng(20221018)
    out = {}
    cases = []
    for i, (n, k, kind) in enumerate([(300, 60, "dyadic"), (1000, 200, "dyadic"), (2048, 410, "dyadic"),
                                      (777, 156, "float64"), (1500, 300, "float64"), (64, 64, "dyadic"),
                                      (1200, 300, "utm"), (600, 400, "dups"), (5000, 1024, "float64")]):
        if kind == "dyadic":
            pts = dyadic_cloud(rng, n)
            if k == n:  # avoid exhausting duplicates: make the points distinct
                pts = np.unique(pts, axis=0)
                rng.shuffle(pts)
                n = k = pts.shape[0]
        elif kind == "utm":     # raw lidar coordinates: UTM easting / northing, ellipsoidal height
            pts = rng.normal(size=(n, 3)) * np.array([4.0, 4.0, 8.0]) + np.array([512345.67, 5412345.89, 312.5])
        elif kind == "dups":    # 200 distinct points three times over, more samples than distinct points
            base = rng.normal(size=(n // 3, 3)) * np.array([4.0, 4.0, 8.0])
            pts = np.concatenate([base, base, base], 0)
            rng.shuffle(pts)
        else:
            pts = rng.normal(size=(n, 3)) * np.array([4.0, 4.0, 8.0])
        idx = fps_np(pts, k)
        out[f"pos_{i}"] = pts
        out[f"idx_{i}"] = np.asarray(idx, dtype=np.int64)
        cases.append(kind)
    out["kinds"] = np.array(cases)
    np.savez_compressed(os.path.join(GOLD, "fps_reference_numpy.npz"), **out)
    print("fps_reference_numpy.npz:", len(cases), "cases")


def gen_grouping_oracle():
    out = {}
    specs = [(1234, 3, 1000, False, 2.0, 8.0), (99, 4, 513, True, 2.0, 8.0), (7, 2, 2048, True, 4.0, 16.0)]
    for i, (seed, B, n, ragged, r1, r2) in enumerate(specs):
        b = Batch.from_data_list(synthetic_clouds(seed, B, n, 1, ragged))
        idx1 = ref.fps_ref(b.pos, b.ptr, 0.2)
        ptr1 = ref.sample_ptr(b.ptr, 0.2)
        nbr1, cnt1 = ref.ball_query_ref(b.pos, b.pos[idx1], b.ptr, ptr1, r1, 64)
        pos1 = b.pos[idx1]
        idx2 = ref.fps_ref(pos1, ptr1, 0.25)
        ptr2 = ref.sample_ptr(ptr1, 0.25)
        nbr2, cnt2 = ref.ball_query_ref(pos1, pos1[idx2], ptr1, ptr2, r2, 64)
        # the clouds themselves are stored: torch's CPU normal sampler gives different bits on different CPUs (vector
        # vs scalar kernels), so re-drawing them from the seed would make the fixture depend on the host
        out.update({f"spec_{i}": np.array([seed, B, n, int(ragged), r1, r2]), f"pos_{i}": b.pos.numpy(),
                    f"ptr_{i}": b.ptr.numpy(), f"idx1_{i}": idx1.numpy(),
                    f"cnt1_{i}": cnt1.numpy(), f"nbr1_{i}": nbr1.numpy(), f"idx2_{i}": idx2.numpy(),
                    f"cnt2_{i}": cnt2.numpy(), f"nbr2_{i}": nbr2.numpy()})
    np.savez_compressed(os.path.join(GOLD, "grouping_oracle.npz"), **out)
    print("grouping_oracle.npz:", len(specs), "specs")


def gen_net_oracle():
    # the input clouds are stored (see gen_grouping_oracle), and the network runs in float64: in float32 its train-mode
    # gradients of levels 1-2 (BatchNorm backward over few rows) move by up to ~0.5 % with the host's summation order
    # (thread count, CPU kernels), which a fixture must not pin
    torch.manual_seed(0)
    clouds = synthetic_clouds(4321, 3, 768, 1, True)
    b = Batch.from_data_list(clouds)
    b.x, b.pos = b.x.double(), b.pos.double()
    res = {}
    for mode in ("train", "eval"):
        net = ref.seeded_init_(ref.NetRef(1, "ReLU", 0, 0.0), seed=7).double()
        net.train(mode == "train")
        out = net(b)
        loss = ref.weighted_mse(out, b.y)
        loss.backward()
        res[mode] = {"out": out.detach().clone(), "loss": loss.detach().clone(),
                     "grads": {k: p.grad.clone() for k, p in net.named_parameters()},
                     "buffers": {k: v.clone() for k, v in net.named_buffers()}}
    # keep the fixture small: store grads as per-tensor (sum, abs-sum, first 8 values) digests + full small ones
    def digest(t):
        f = t.flatten().double()
        return torch.tensor([f.sum(), f.abs().sum(), (f * torch.arange(1, f.numel() + 1).double()).sum()])
    small = {}
    for mode, r in res.items():
        small[mode] = {"out": r["out"], "loss": r["loss"],
                       "grad_digest": {k: digest(v) for k, v in r["grads"].items()},
                       "grad_head": {k: v.flatten()[:16].clone() for k, v in r["grads"].items()},
                       "buf_digest": {k: digest(v.float()) for k, v in r["buffers"].items()}}
    torch.save({"spec": (4321, 3, 768, 1, True), "init_seed": 7, "modes": small,
                "clouds": [{"x": c.x, "pos": c.pos, "y": c.y} for c in clouds]}, os.path.join(GOLD, "net_oracle.pt"))
    print("net_oracle.pt: out(train) =", res["train"]["out"].flatten()[:4])


if __name__ == "__main__":
    os.makedirs(GOLD, exist_ok=True)
    gen_fps_reference()
    gen_grouping_oracle()
    gen_net_oracle()
