#!/usr/bin/env python
"""bench.py -- train tree-clouds/sec of the PointNet++ biomass regressor hot path on B200.

    python bench.py --gpus N --steps K --warmup W [--precision bf16|fp32] [--impl reference]
                    [--config train|eval|dense] [--dump-outputs DIR]

A "step" is one pass of /root/reference/main.py:150-172 over one batch of synthetic tree clouds
(forward + weighted MSE + backward + gradient all-reduce + Adam), BASELINE.json configs[1]:
10,000-point clouds, 12 clouds per GPU.  Rank 0 prints ONE JSON line (contract in the task brief):
value = device-resident throughput, e2e = through Net.forward with host buffers (H2D + loss D2H inside
the timed region), roofline = Kernel 1 (FPS, level 1) timed alone against the measured HBM peak,
cpu_baseline = the CPU oracle on this box's host cores.  `--impl reference` times the reference's CPU
path (its third-party kernels restated by oracle/) instead.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)
# the benchmark writes nothing into the tree it runs from (which may be read-only), bytecode caches included
sys.dont_write_bytecode = True

import torch  # noqa: E402

METRIC = "train tree-clouds/sec @10k pts"
UNIT = "tree-clouds/s"
DUMP_LIMIT_BYTES = 64 * 2 ** 20


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--precision", default=None, choices=["bf16", "fp32"])
    ap.add_argument("--batch", type=int, default=12, help="tree clouds per GPU per step")
    ap.add_argument("--points", type=int, default=10000)
    ap.add_argument("--pool", type=int, default=4, help="distinct batches rotated through")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-graph", action="store_true", help="eager launches instead of one CUDA graph per step")
    ap.add_argument("--join", default="end", choices=["backward", "end"], help="where the sampling branch joins")
    ap.add_argument("--no-uncap-l1", action="store_true", help="keep the SM cap through the level-1 backward")
    ap.add_argument("--no-cap", action="store_true", help="do not cap persistent kernels while the branch runs")
    ap.add_argument("--no-pregroup", action="store_true", help="ball query / row packing inside forward")
    ap.add_argument("--no-aux", dest="aux", action="store_false",
                    help="level-1 grouping behind the level-2 sampling instead of beside it on a third stream")
    ap.add_argument("--side-priority", type=int, default=0, help="CUDA priority of the sampling branch's stream (-1: high)")
    ap.add_argument("--no-pipeline", action="store_true",
                    help="sample (FPS) every batch inside its own step instead of one step ahead on a second stream")
    ap.add_argument("--config", default="train", choices=["train", "eval", "dense"],
                    help="train: BASELINE configs[1]/[4] (the headline); eval: configs[2] (inference, --batch 64..512); "
                         "dense: configs[3] (8 x 100k points, radii 4/16, train step)")
    ap.add_argument("--dp-mode", default="graph", choices=["graph", "split", "eager"],
                    help="N>1: all-reduce + Adam inside the step graph / eager after a forward+backward graph / no graph")
    ap.add_argument("--no-dp-overlap", dest="dp_overlap", action="store_false",
                    help="N>1: all-reduce the buckets after backward on the training stream instead of on a side stream as "
                         "backward finishes them (measured at N=2: 2.38 ms/step overlapped, 2.41 serial)")
    ap.add_argument("--no-fp32", action="store_true", help="skip the fp32-mode sibling measurement (N=1, train config)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step computed as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.config == "dense":
        if args.batch == 12:
            args.batch = 8
        if args.points == 10000:
            args.points = 100000
    if args.config == "eval" and args.batch == 12:
        args.batch = 256
    return args


# ------------------------------------------------------------------------------------------------
#  helpers
# ------------------------------------------------------------------------------------------------
def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), float(d.get("bf16_tflops", 1590.0)), "measured"
    return 6650.0, 1590.0, "fallback"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled every 100 ms while the timed region runs."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.proc, self.lines, self.thread = None, [], None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={gpu_index}", f"--query-gpu={self.Q}",
                                          "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except (OSError, ValueError):
            self.proc = None

    def _pump(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 6:
                continue
            try:
                sm.append(float(parts[0]))
                mx.append(float(parts[1]))
            except ValueError:
                continue
            for n, v in zip(names, parts[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def make_pool(args, rank, pin):
    """`pool` distinct batches of `batch` clouds for this rank (seeds as SURVEY.md 8(d): S + rank*1e6 + c)."""
    from dl_biomass_b200.data import Batch, synthetic_clouds
    pool = []
    for i in range(args.pool):
        clouds = synthetic_clouds(1234 + rank * 1_000_000 + i * args.batch, args.batch, args.points, 1, False)
        b = Batch.from_data_list(clouds)
        pool.append(b.pin_memory() if pin else b)
    return pool


def batch_h2d_bytes(b, with_batch_vector=True):
    ts = (b.x, b.pos, b.batch, b.y) if with_batch_vector else (b.x, b.pos, b.y)
    return sum(t.numel() * t.element_size() for t in ts if t is not None)


def dump_outputs(out_dir, arrays):
    """Write every tensor of `arrays` as out_dir/<name>.npy, float64 as float64 and everything else as float32.  The
    inputs depend on the arguments only, so two builds run with the same arguments can be compared file by file.

    A training step hands its caller the loss, so the training configs write that and not the parameters: those differ
    between two runs of the same build by far more than the loss does (DESIGN.md section 6)."""
    import numpy as np
    host = {}
    for name, t in arrays.items():
        t = t.detach().cpu()
        host[name] = (t if t.dtype == torch.float64 else t.float()).numpy()
    total = sum(a.nbytes for a in host.values())
    if total > DUMP_LIMIT_BYTES:
        raise RuntimeError(f"--dump-outputs: {total} bytes exceed the {DUMP_LIMIT_BYTES}-byte limit")
    os.makedirs(out_dir, exist_ok=True)
    for name, a in host.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


# ------------------------------------------------------------------------------------------------
#  CPU arm: the reference's CPU path as restated by oracle/ (torch CPU + C fps/radius)
# ------------------------------------------------------------------------------------------------
def cpu_train_steps(args, steps, warmup):
    """`steps` timed training steps of the oracle network on ALL host cores, every step on the FULL configured batch."""
    from oracle import ref
    torch.set_num_threads(os.cpu_count() or 1)
    from dl_biomass_b200.data import Batch, synthetic_clouds
    net = ref.seeded_init_(ref.NetRef(1, "ReLU", 0, 0.5), seed=7)
    net.train()
    if args.config == "dense":
        net.sa1_module.r, net.sa2_module.r = 4.0, 16.0
    opt = ref.make_adam(net.parameters())
    last = {}

    def one(i):
        b = Batch.from_data_list(synthetic_clouds(1234 + i * args.batch, args.batch, args.points, 1, False))
        t0 = time.perf_counter()
        opt.zero_grad()
        loss = ref.weighted_mse(net(b), b.y)
        loss.backward()
        opt.step()
        last["loss"] = loss
        return time.perf_counter() - t0

    for i in range(max(warmup, 1)):
        one(i)
    ts = [one(100 + i) for i in range(steps)]
    total = sum(ts)
    return {"value": args.batch * steps / total, "ms_per_step": 1e3 * total / steps, "steps": steps,
            "clouds_per_step": args.batch, "cores": torch.get_num_threads(), "host_cores": os.cpu_count(),
            "oracle_threads": ref.num_threads(), "loss": last["loss"]}


def workload_name(args, precision=None):
    if args.config == "eval":
        return (f"PointNet++ regressor inference (eval mode, no grad), {args.points}-pt clouds, batch {args.batch}/GPU, F=1 "
                f"(BASELINE configs[2])")
    if args.config == "dense":
        return (f"PointNet++ regressor train step, dense clouds: {args.points} pts, batch {args.batch}/GPU, radii (4, 16), "
                f"F=1 (BASELINE configs[3])")
    return (f"PointNet++ regressor train step (fwd + weighted MSE + bwd + all-reduce + Adam), {args.points}-pt clouds, "
            f"batch {args.batch}/GPU, F=1 (BASELINE configs[1]; configs[4] at N>1)")


def shared_config(args, world):
    """`config` of the JSON line: the WORKLOAD, identical for both arms (--impl b200 / reference) so that the driver
    compares like with like; what is specific to an arm lives in `impl_notes` / `cpu_baseline.sample`."""
    return {"workload": workload_name(args), "global_batch": world * args.batch, "points_per_cloud": args.points,
            "parallelism": f"dp{world}", "l2": "256 MB buffer rewritten before every timed step (GPU arm)",
            "timing": "GPU arm: per-step CUDA events on the launching stream, summed, max over ranks; CPU arm: "
                      "perf_counter around each step"}


def metric_name(args):
    if args.config == "eval":
        return f"inference tree-clouds/sec @{args.points // 1000}k pts"
    if args.config == "dense":
        return f"train tree-clouds/sec @{args.points // 1000}k pts"
    return METRIC


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    r = cpu_train_steps(args, args.steps, args.warmup)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {"loss": r["loss"].reshape(1)})
    sample = (f"{r['steps']} timed steps (after {args.warmup} warm-up), each a full train step (fwd+loss+bwd+Adam) on "
              f"{r['clouds_per_step']} clouds x {args.points} pts")
    line = {"impl": "reference", "metric": metric_name(args) if args.config != "eval" else METRIC,
            "value": round(r["value"], 4), "unit": UNIT, "n_gpus": args.gpus,
            "steps": r["steps"], "warmup": args.warmup, "ms_per_step": round(r["ms_per_step"], 3),
            "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": shared_config(args, max(1, args.gpus)),
            "impl_notes": "reference CPU path (BASELINE configs[0]): torch_cluster/torch_scatter/PyG are not installable "
                          "here, so their kernels are the oracle's restatement (oracle/ref.py, oracle/b2pn_oracle.c); "
                          "rank 0 alone runs it, on one GPU's share of the batch",
            "cpu_baseline": {"value": round(r["value"], 4), "unit": UNIT, "cores": r["cores"], "kind": "port",
                             "sample": sample},
            "e2e": {"value": round(r["value"], 4), "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------
#  B200 arm
# ------------------------------------------------------------------------------------------------
def sa_mlp_flops(net, counts):
    """Algorithmic FLOPs of one FORWARD pass of the three set-abstraction MLPs: 2 * rows * sum_l K_l * N_l with rows =
    real edges of levels 1 / 2 (padded slots do not count) and level-2 points for the global level (SURVEY 8(d))."""
    total = 0
    for mod, rows in zip((net.sa1_module.conv.local_nn, net.sa2_module.conv.local_nn, net.sa3_module.nn), counts):
        c = mod.channel_list
        total += 2 * rows * sum(a * b for a, b in zip(c[:-1], c[1:]))
    return total


def event_time(fn, reps, flush):
    evs = []
    for _ in range(reps):
        flush.zero_()
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        evs.append((a, b))
    torch.cuda.synchronize()
    return sum(a.elapsed_time(b) for a, b in evs) / reps


def profile_json(name):
    f = os.path.join(ROOT, "profiles", name)
    if os.path.exists(f):
        try:
            return json.load(open(f))
        except (OSError, ValueError):
            return None
    return None


def run_b200(args):
    import torch.distributed as dist
    from dl_biomass_b200 import _lib, ops, sa
    from dl_biomass_b200.parallel import GradReducer
    from dl_biomass_b200.pointnet2_regressor import Net
    from dl_biomass_b200.train import GraphedTrainStep, PipelinedTrainStep, make_optimizer, train_step

    if not torch.cuda.is_available():
        raise RuntimeError("bench.py needs a B200: no CUDA device (the product path has no CPU fallback)")
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    # ---- CPU baseline first (N=1 only): nothing else of this job is running yet, so the host cores are its own
    cpu = None
    if world == 1 and not args.no_cpu_baseline and args.config != "eval":
        r = cpu_train_steps(args, steps=2 if args.config == "train" else 1, warmup=1)
        cpu = {"value": round(r["value"], 4), "unit": UNIT, "cores": r["cores"], "kind": "port",
               "sample": f"1 warm-up + {r['steps']} timed full train steps of {r['clouds_per_step']} clouds x {args.points} pts "
                         f"(oracle NetRef: torch CPU + C fps/radius, {r['oracle_threads']} threads), timed before any GPU work"}

    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        # the collectives are captured into the step's CUDA graph: the process group's watchdog must not query events
        # of a capturing stream (PyTorch's documented requirement for whole-network capture with NCCL)
        os.environ.setdefault("TORCH_NCCL_ASYNC_ERROR_HANDLING", "0")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    torch.cuda.set_device(dev)
    lib = _lib.lib()

    precision = args.precision
    if precision is None:
        precision = "bf16" if getattr(sa, "bf16_available", lambda: False)() else "fp32"

    pool_host = make_pool(args, rank, pin=True)
    pool_dev = [b.to(dev) for b in pool_host]
    flush = torch.empty(256 * 1024 * 1024, dtype=torch.uint8, device=dev)  # > 126 MB L2

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    def timed(step_fn, steps):
        """Per-step CUDA events on the current stream, L2 flushed (untimed) before every step.  Returns the summed time
        and what the last step returned."""
        evs, last = [], None
        barrier()
        for i in range(steps):
            flush.zero_()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            last = step_fn(i)
            b.record()
            evs.append((a, b))
        barrier()
        ms = sum(a.elapsed_time(b) for a, b in evs)
        t = torch.tensor([ms], dtype=torch.float64, device=dev)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item()), last

    use_graph = not args.no_graph and not (world > 1 and args.dp_mode == "eager")
    # dense clouds (100k points): farthest-point sampling runs one 16-CTA cluster per cloud -- 128 of the 148 SMs for
    # ~46 ms, 0.85 of the HBM roofline in scan-equivalent bytes -- so there is no idle machine to overlap the training
    # kernels with: the step is one graph, sampling first
    pipeline = not args.no_pipeline and args.config == "train"

    def build_training(prec):
        """model + optimiser + reducer + stepper for one precision mode"""
        torch.manual_seed(7)
        net = Net(1, "ReLU", 0, 0.5, precision=prec).to(dev)
        net.train()
        if args.config == "dense":
            net.sa1_module.r, net.sa2_module.r = 4.0, 16.0   # the reference's "..._w_doubled_radius" runs
        opt = make_optimizer(net)   # FlatAdam over one parameter arena: one libb2pn launch per step
        reducer = GradReducer(net) if world > 1 else None
        graphed = stepper = None
        if pipeline:
            stepper = PipelinedTrainStep(net, opt, pool_dev[0], reducer, graph=use_graph, join=args.join,
                                         cap=not args.no_cap, grouping=not args.no_pregroup, aux=args.aux,
                                         uncap_level1_backward=not args.no_uncap_l1,
                                         capture_collective=args.dp_mode == "graph", overlap_collective=args.dp_overlap,
                                         side_priority=args.side_priority)
        elif use_graph:
            graphed = GraphedTrainStep(net, opt, pool_dev[0], reducer)

        def run_step(batch):
            if stepper is not None:
                return stepper.step(batch)
            return graphed(batch) if graphed is not None else train_step(net, opt, batch, reducer)
        return net, opt, reducer, stepper, graphed, run_step

    def measure_training(run_step, stepper, graphed, steps, warmup, sample_clocks, dump=None):
        def step_resident(i):
            return run_step(pool_dev[(i + 1) % len(pool_dev)])
        for i in range(warmup):
            step_resident(i)
        sampler = ClockSampler(local_rank) if (sample_clocks and rank == 0) else None
        l0 = lib.b2pn_launch_count()
        total_ms, last_loss = timed(step_resident, steps)
        launches = lib.b2pn_launch_count() - l0
        clocks = sampler.stop() if sampler else None
        if dump is not None:   # before the e2e steps below train the model further
            dump(last_loss)
        if stepper is not None and use_graph:  # replayed kernels do not pass through the library's launch counter
            launches = stepper.launches_per_step * steps
        elif graphed is not None:
            launches = graphed.launches_per_replay * steps
        loss_host = torch.empty((), dtype=torch.float32).pin_memory()

        def step_e2e(i):
            hb = pool_host[(i + 1) % len(pool_host)]
            if stepper is not None or graphed is not None:
                loss = run_step(hb)  # pinned host tensors are copied straight into the step's input buffers
            else:
                loss = run_step(hb.to(dev, non_blocking=True))
            loss_host.copy_(loss, non_blocking=True)
        for i in range(3):
            step_e2e(i)
        e2e_ms, _ = timed(step_e2e, steps)
        return total_ms, e2e_ms, int(launches), clocks

    hbm_peak, tc_peak, peak_kind = measured_peaks()
    peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json"))) if peak_kind == "measured" else {}
    tc_sustained = float(peaks.get("bf16_tflops_sustained", 1400.0))
    warmup = max(args.warmup, 3)

    # =============================================================================================================
    if args.config == "eval":
        torch.manual_seed(7)
        net = Net(1, "ReLU", 0, 0.5, precision=precision).to(dev).eval().set_random_start(False)
        out_host = torch.empty(args.batch, 4, dtype=torch.float32).pin_memory()

        def fwd(i):
            with torch.no_grad():
                return net(pool_dev[i % len(pool_dev)])

        def fwd_e2e(i):
            with torch.no_grad():
                out = net(pool_host[i % len(pool_host)].to(dev, non_blocking=True))
            out_host.copy_(out, non_blocking=True)
        for i in range(warmup):
            fwd(i)
        torch.cuda.reset_peak_memory_stats(dev)
        sampler = ClockSampler(local_rank) if rank == 0 else None
        l0 = lib.b2pn_launch_count()
        total_ms, out = timed(fwd, args.steps)
        launches = int(lib.b2pn_launch_count() - l0)
        clocks = sampler.stop() if sampler else None
        peak_gb = torch.cuda.max_memory_allocated(dev) / 2 ** 30
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, {"out": out})
        for i in range(2):
            fwd_e2e(i)
        e2e_ms, _ = timed(fwd_e2e, args.steps)
        if rank == 0:
            value = world * args.batch * args.steps / (total_ms * 1e-3)
            line = {"metric": metric_name(args), "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": args.steps,
                    "warmup": warmup, "ms_per_step": round(total_ms / args.steps, 4), "higher_is_better": True,
                    "scaling": "weak", "vs_baseline": None, "dtype": "bf16" if precision == "bf16" else "f32",
                    "data": "synthetic",
                    "config": shared_config(args, world),
                    "impl_notes": {"mlp_precision": precision},
                    "clocks": clocks, "gpu_launches": launches, "peak_memory_GB": round(peak_gb, 2),
                    "e2e": {"value": round(world * args.batch * args.steps / (e2e_ms * 1e-3), 2), "unit": UNIT,
                            "ms_per_step": round(e2e_ms / args.steps, 4),
                            "h2d_bytes_per_step": batch_h2d_bytes(pool_host[0]), "d2h_bytes_per_step": args.batch * 16},
                    "roofline": None, "cpu_baseline": None}
            print(json.dumps(line), flush=True)
        if world > 1:
            shutdown_dist(dist)
        return

    # =============================================================================================================
    net, opt, reducer, stepper, graphed, run_step = build_training(precision)

    def dump(loss):
        dump_outputs(args.dump_outputs, {"loss": loss.reshape(1)})
    total_ms, e2e_ms, launches, clocks = measure_training(run_step, stepper, graphed, args.steps, warmup, True,
                                                          dump if args.dump_outputs and rank == 0 else None)
    value = world * args.batch * args.steps / (total_ms * 1e-3)
    e2e_value = world * args.batch * args.steps / (e2e_ms * 1e-3)
    sm_limit_note = stepper.sm_limit if stepper is not None else 0
    dp = None
    if reducer is not None:
        torch.cuda.synchronize(dev)
        spread = reducer.replicas_identical()
        per_step = stepper.allreduce_per_step if stepper is not None else len(reducer.flat)
        dp = {"allreduce_calls_per_step": int(per_step), "buckets": [int(f.numel()) for f in reducer.flat],
              "wire_bytes_per_step_per_gpu": reducer.wire_bytes_per_step(), "mode": args.dp_mode,
              "overlap_with_backward": bool(args.dp_overlap),
              "max_abs_param_diff_across_ranks": spread}
        if spread != 0.0:
            raise RuntimeError(f"data-parallel replicas diverged: max |param - rank 0's| = {spread}")
    if stepper is not None:
        stepper.close()
        if world > 1 and use_graph:
            stepper.release_graphs()   # graphs holding NCCL plans must die before the communicator can

    # ---- rooflines: each kernel timed alone with CUDA events, L2 flushed --------------------------------------------
    b0 = pool_dev[0]
    ratios = [net.sa1_module.ratio, net.sa2_module.ratio]
    lv = ops.build_levels(b0.cloud_sizes, ratios, dev)
    torch.cuda.synchronize(dev)
    for _ in range(3):
        s1 = ops.fps(b0.pos, lv[0], lv[1])
    fps_ms = event_time(lambda: ops.fps(b0.pos, lv[0], lv[1]), 10, flush)
    scan_bytes = sum(16 * n * m for n, m in zip(lv[0].sizes, lv[1].sizes))  # m*n*16 per cloud, SURVEY 8(d)
    achieved = scan_bytes / 1e9 / (fps_ms * 1e-3)
    traffic = (profile_json("fps_dram_bytes.json") or {}).get("dram_bytes_per_launch")
    step_ms = total_ms / args.steps
    roofline = {"bound": "hbm", "kernel": f"fps_kernel (Kernel 1, SA1: {args.points}->{lv[1].sizes[0]} per cloud)",
                "achieved": round(achieved, 1), "peak": hbm_peak, "unit": "GB/s", "frac": round(achieved / hbm_peak, 4),
                "traffic": traffic, "peak_kind": f"{peak_kind} (burst copy bandwidth)",
                "bytes_model": "scan-equivalent m*n*16 B per cloud (SURVEY 8(d)); register-resident, so DRAM traffic is "
                               "the compulsory n*12+m*8 B",
                "compulsory_bytes": sum(12 * n + 8 * m for n, m in zip(lv[0].sizes, lv[1].sizes)),
                "ms_per_launch": round(fps_ms, 4), "share_of_step": round(fps_ms / step_ms, 3),
                "note": "timed alone here; inside the step it runs on the sampling branch of the graph, concurrently with "
                        "the training kernels" if stepper is not None else "timed alone"}
    # ball query, level 1
    r1 = float(net.sa1_module.r)
    for _ in range(3):
        ops.ball_query(b0.pos, s1[1], lv[0], lv[1], r1, 64)
    bq_ms = event_time(lambda: ops.ball_query(b0.pos, s1[1], lv[0], lv[1], r1, 64), 10, flush)
    bq_scan = sum(12 * n * m for n, m in zip(lv[0].sizes, lv[1].sizes))
    bq_comp = sum(12 * n + 12 * m + 64 * 4 * m + 4 * m for n, m in zip(lv[0].sizes, lv[1].sizes))
    bq_traffic = (profile_json("bq_dram_bytes.json") or {}).get("dram_bytes_per_launch")
    roof_bq = {"bound": "hbm", "kernel": f"ball query (Kernel 2, SA1: r={r1}, K=64)", "achieved": round(bq_scan / 1e9 / (bq_ms * 1e-3), 1),
               "peak": hbm_peak, "unit": "GB/s", "frac": round(bq_scan / 1e9 / (bq_ms * 1e-3) / hbm_peak, 4),
               "traffic": bq_traffic, "bytes_model": "scan-equivalent m*n*12 B per cloud (SURVEY 8(d)): what the reference's "
               "brute-force kernel streams; the grid kernel visits ~1 % of it, so the fraction exceeds 1",
               "compulsory_bytes": bq_comp, "compulsory_GBps": round(bq_comp / 1e9 / (bq_ms * 1e-3), 1),
               "ms_per_launch": round(bq_ms, 4)}
    # SA MLPs: algorithmic FLOPs of the three levels, forward + backward (3x forward), over the WHOLE training stream
    roof_mlp = None
    if precision == "bf16":
        samp = net.sample(b0, grouping=True)
        torch.cuda.synchronize(dev)
        e1 = int(samp.group1[2][2][1].item())
        e2 = int(samp.group2[2][2][1].item())
        fwd_flops = sa_mlp_flops(net, (e1, e2, lv[2].total))
        tf = 3 * fwd_flops / 1e12 / (step_ms * 1e-3)
        mlp_prof = profile_json("sa_mlp_dram_bytes.json") or {}
        roof_mlp = {"bound": "tensor", "kernel": "SA MLP kernels (Kernel 3: tc_rows_gemm / tc_dw, three levels, fwd + bwd)",
                    "achieved": round(tf, 1), "peak": tc_sustained, "unit": "TFLOP/s", "frac": round(tf / tc_sustained, 4),
                    "peak_kind": f"{peak_kind} (sustained cuBLAS bf16)", "edges": [e1, e2, lv[2].total],
                    "flops_model": "3 x forward FLOPs, forward = 2*E*sum(K_l*N_l) over real edges (SURVEY 8(d)); divided by "
                                   "the whole step time (the training stream also holds head, loss, Adam)",
                    "traffic": mlp_prof.get("dram_bytes_per_step"), "compulsory_plus_saved_bytes": mlp_prof.get("floor_bytes"),
                    "tensor_pipe_pct": mlp_prof.get("tensor_pipe_pct")}

    # ---- the other half of configs[1]: the fp32-accuracy mode, same step, measured in the same run (N=1) ---------------
    fp32 = None
    if world == 1 and args.config == "train" and precision == "bf16" and not args.no_fp32:
        del net, opt, stepper, graphed, run_step
        torch.cuda.empty_cache()
        netf, optf, _, stepf, graphf, runf = build_training("fp32")
        k = args.steps
        t_ms, e_ms, lf, _ = measure_training(runf, stepf, graphf, k, 3, False)
        if stepf is not None:
            stepf.close()
        fp32 = {"dtype": "f32", "steps": k, "ms_per_step": round(t_ms / k, 4), "value": round(args.batch * k / (t_ms * 1e-3), 2),
                "unit": UNIT, "e2e": {"value": round(args.batch * k / (e_ms * 1e-3), 2), "ms_per_step": round(e_ms / k, 4)},
                "gpu_launches": lf, "workload": workload_name(args, "fp32")}

    if rank != 0:
        if world > 1:
            shutdown_dist(dist)
        return

    line = {"metric": metric_name(args), "value": round(value, 2), "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": warmup, "ms_per_step": round(step_ms, 4), "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "bf16" if precision == "bf16" else "f32",
            "data": "synthetic",
            "config": shared_config(args, world),
            "impl_notes": {"mlp_precision": precision,
                       "launch": "one CUDA graph replay per step" if use_graph else "eager kernel launches",
                       "optimizer": "FlatAdam: one b2pn_adam_step launch over the flat parameter arena",
                       "pipeline": ("FPS" + (" + ball query + row compaction + level-1 gather" if stepper_grouping(args) else "")
                                    + " of batch i+1 on a second stream during step i (every timed step contains one "
                                    f"full sampling and one full training pass); join at {args.join}; persistent "
                                    f"kernels capped at {sm_limit_note} CTAs" + ("" if args.no_uncap_l1 else " until the level-1 backward"))
                                   if pipeline else "none"},
            "clocks": clocks, "gpu_launches": int(launches),
            "e2e": {"value": round(e2e_value, 2), "unit": UNIT, "ms_per_step": round(e2e_ms / args.steps, 4),
                    "h2d_bytes_per_step": batch_h2d_bytes(pool_host[0], with_batch_vector=not use_graph),
                    "d2h_bytes_per_step": 4},
            "roofline": roofline, "rooflines": [r for r in (roofline, roof_bq, roof_mlp) if r is not None],
            "cpu_baseline": cpu}
    if fp32 is not None:
        line["fp32"] = fp32
    if dp is not None:
        line["data_parallel"] = dp
        line["allreduce_calls_per_step"] = dp["allreduce_calls_per_step"]
    print(json.dumps(line), flush=True)
    if world > 1:
        shutdown_dist(dist)


def stepper_grouping(args):
    return not args.no_pregroup


def shutdown_dist(dist):
    """Leave the process group.  The JSON line is already out; a communicator that refuses to die must not turn a
    finished measurement into a hung job, so a watchdog ends the process after 30 s."""
    sys.stdout.flush()
    t = threading.Timer(30.0, lambda: os._exit(0))
    t.daemon = True
    t.start()
    try:
        dist.barrier()
        dist.destroy_process_group()
    finally:
        t.cancel()


def main():
    args = parse_args()
    if args.impl == "reference":
        run_reference(args)
    else:
        run_b200(args)


if __name__ == "__main__":
    main()
