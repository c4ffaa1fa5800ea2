"""GPU: the data-parallel training step (dl_biomass_b200/parallel.py + train.py) over NCCL -- the replacement of the
reference's DataParallel wrapper (/root/reference/main.py:140,153,171-172).

* world size 1 (always runs): a graph-replayed step issues one all-reduce per bucket on EVERY step (round-1 bug: only on
  the first), in both the split mode (collective eager after the replay) and the captured mode (collective inside the
  graph), and trains exactly like the step without a reducer.
* world size 2 (skipped with fewer than 2 GPUs): averaged gradients == mean of the per-rank gradients, replicas
  bit-identical after several graph-replayed steps.
"""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from dl_biomass_b200.data import Batch, synthetic_clouds

pytestmark = pytest.mark.gpu


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _batches(rank, n=5, clouds=3, pts=512):
    return [Batch.from_data_list(synthetic_clouds(7000 + 100 * rank + 11 * i, clouds, pts, 1, False)) for i in range(n)]


def _fresh(dev, dropout=0.0):
    from dl_biomass_b200.pointnet2_regressor import Net
    torch.manual_seed(5)
    net = Net(1, "ReLU", 0, dropout, precision="bf16").to(dev).set_random_start(False)
    net.train()
    return net


@pytest.mark.timeout(600)
@pytest.mark.parametrize("mode", ["split", "captured", "captured_overlap"])
def test_world1_graph_step_all_reduces_every_step(cuda_device, mode):
    from dl_biomass_b200.parallel import GradReducer
    from dl_biomass_b200.train import PipelinedTrainStep, make_optimizer, train_step
    os.environ.setdefault("TORCH_NCCL_ASYNC_ERROR_HANDLING", "0")
    batches = [b.to(cuda_device) for b in _batches(0)]
    net = _fresh(cuda_device)
    opt = make_optimizer(net)
    want = [float(train_step(net, opt, b)) for b in batches[:4]]

    dist.init_process_group("nccl", store=dist.HashStore(), rank=0, world_size=1, device_id=cuda_device)
    try:
        net = _fresh(cuda_device)
        opt = make_optimizer(net)
        red = GradReducer(net)
        assert len(red.flat) == 3
        stepper = PipelinedTrainStep(net, opt, batches[0], red, graph=True, warmup=1,
                                     capture_collective=mode != "split", overlap_collective=mode == "captured_overlap")
        got = []
        with stepper:
            assert stepper.allreduce_per_step == 3
            for b in batches[1:4]:
                c0 = red.allreduce_calls
                got.append(float(stepper.step(b)))
                # split mode: the collectives are issued from the host after every replay; captured: they are graph nodes
                assert red.allreduce_calls - c0 == (3 if mode == "split" else 0)
            got.append(float(stepper.flush()))
        torch.cuda.synchronize()
        assert red.replicas_identical() == 0.0
        stepper.release_graphs()
    finally:
        dist.destroy_process_group()
    print(mode, want, got)
    for a, b in zip(want, got):          # world size 1: averaging is the identity, the trajectory is the plain one
        assert abs(a - b) <= 2e-3 * max(abs(a), 1e-6)


def _rank_worker(rank, world, port, out_dir, mode):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    os.environ.setdefault("TORCH_NCCL_ASYNC_ERROR_HANDLING", "0")
    dev = torch.device("cuda", rank)
    torch.cuda.set_device(dev)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    from dl_biomass_b200.parallel import GradReducer
    from dl_biomass_b200.train import PipelinedTrainStep, forward_backward, make_optimizer
    batches = [b.to(dev) for b in _batches(rank)]
    # 1. one eager step: the reduced gradients (arena) are what every rank sees
    net = _fresh(dev)
    if rank != 0:   # replicas start different on purpose: the reducer broadcasts rank 0's parameters
        with torch.no_grad():
            for p in net.parameters():
                p.add_(0.01)
    opt = make_optimizer(net)
    red = GradReducer(net)
    forward_backward(net, opt, batches[0], red)
    red.finish()
    torch.cuda.synchronize()
    reduced = red.arena.flat_grads.clone().cpu()
    # 2. graph-replayed steps
    stepper = PipelinedTrainStep(net, opt, batches[0], red, graph=True, warmup=1, capture_collective=(mode == "captured"))
    with stepper:
        for b in batches[1:5]:
            stepper.step(b)
    torch.cuda.synchronize()
    spread = red.replicas_identical()
    torch.save({"reduced": reduced, "params": red.arena.flat_params.clone().cpu(), "spread": spread,
                "per_step": stepper.allreduce_per_step}, os.path.join(out_dir, f"rank{rank}.pt"))
    stepper.release_graphs()       # graphs holding NCCL plans must die before the communicator can
    dist.barrier()
    dist.destroy_process_group()


def _local_grads(rank, dev):
    """Gradients of rank `rank`'s first batch computed WITHOUT a reducer, from rank 0's initial parameters."""
    from dl_biomass_b200.optim import ParamArena
    from dl_biomass_b200.train import forward_backward, make_optimizer
    net = _fresh(dev)
    opt = make_optimizer(net)
    forward_backward(net, opt, _batches(rank)[0].to(dev))
    opt.arena.collect()
    torch.cuda.synchronize()
    return ParamArena.of(net).flat_grads.clone().cpu()


@pytest.mark.timeout(900)
@pytest.mark.parametrize("mode", ["split", "captured"])
def test_world2_nccl_replicas_stay_identical(cuda_device, tmp_path, mode):
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    ctx = mp.start_processes(_rank_worker, args=(2, _free_port(), str(tmp_path), mode), nprocs=2, join=False,
                             start_method="spawn")
    import time
    t0 = time.time()
    while not ctx.join(timeout=5):
        if time.time() - t0 > 240:
            for p in ctx.processes:
                p.kill()
            pytest.fail("2-rank NCCL step did not finish in 240 s")
    r0, r1 = torch.load(tmp_path / "rank0.pt"), torch.load(tmp_path / "rank1.pt")
    assert r0["spread"] == 0.0 and r1["spread"] == 0.0
    assert torch.equal(r0["params"], r1["params"])                 # bit-identical replicas after 4 graph-replayed steps
    assert torch.equal(r0["reduced"], r1["reduced"])
    assert r0["per_step"] == 3
    want = 0.5 * (_local_grads(0, cuda_device) + _local_grads(1, cuda_device))
    scale = float(want.abs().max())
    # bf16 level-1 gradients carry run-to-run rounding freedom (profiles/r02_grad_spread.md); elsewhere fp32 rounding
    assert float((r0["reduced"] - want).abs().max()) <= 2e-2 * scale
