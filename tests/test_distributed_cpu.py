"""N>1 host logic on CPU (gloo, world_size 2): window sharding covers the dataset exactly like
DistributedSampler, the flat-bucket gradient all-reduce equals the mean of per-rank gradients, and
replicas stay bit-identical after an optimizer step."""
import os
import socket

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from pytorch_geometric_temporal_b200 import distributed as D
from pytorch_geometric_temporal_b200.signal import shard_indices


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank))
    r, w, dev = D.init_process_group("gloo")
    assert (r, w) == (rank, world) and dev.type == "cpu"
    torch.manual_seed(100 + rank)  # different init per rank on purpose
    model = torch.nn.Sequential(torch.nn.Linear(6, 5), torch.nn.Tanh(), torch.nn.Linear(5, 2))
    D.broadcast_parameters(model, src=0)
    sync = D.FlatGradSync(model.parameters())
    opt = torch.optim.Adam(model.parameters(), lr=1e-2)
    torch.manual_seed(0)
    data, target = torch.randn(20, 6), torch.randn(20, 2)
    mine = shard_indices(20, world, rank, shuffle=True, seed=3, epoch=1)
    loss = (model(data[mine]) - target[mine]).square().mean()
    loss.backward()
    local_grad = sync.flat.clone()
    sync.all_reduce()
    opt.step()
    v = D.reduce_scalar(torch.tensor([float(rank + 1), 1.0]))
    # plain lists: tensors sent through a spawn Queue die with the worker's shared-memory handles
    q.put((rank, mine, local_grad.tolist(), sync.flat.tolist(), torch.cat([p.data.reshape(-1) for p in model.parameters()]).tolist(), v.tolist()))
    dist.destroy_process_group()


def test_two_rank_gloo_flat_allreduce_and_sharding(monkeypatch):
    # the CPU path on any machine: with a GPU visible, init_process_group would put rank r on cuda:r, and a one-GPU
    # machine has no cuda:1 (the spawned workers read this environment; CUDA in this process is unaffected)
    monkeypatch.setenv("CUDA_VISIBLE_DEVICES", "")
    world, port = 2, _free_port()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, q)) for r in range(world)]
    for p in procs:
        p.start()
    try:
        res = sorted([q.get(timeout=120) for _ in range(world)], key=lambda t: t[0])
        for p in procs:
            p.join(timeout=60)
            assert p.exitcode == 0
    finally:
        for p in procs:                     # a rank left waiting for a failed peer must not outlive the test
            if p.is_alive():
                p.kill()
                p.join()
    (_, idx0, g0, avg0, w0, v0), (_, idx1, g1, avg1, w1, v1) = res
    assert sorted(idx0 + idx1) == list(range(20))                     # the shards partition the windows
    g0, g1, avg0, avg1 = (torch.tensor(t) for t in (g0, g1, avg0, avg1))
    assert torch.allclose(avg0, (g0 + g1) / 2) and torch.equal(avg0, avg1)
    assert w0 == w1                                                    # replicas identical after the step
    assert v0 == [3.0, 2.0]                                            # reduce(SUM) lands on rank 0


def test_flat_grad_views_accumulate_in_place():
    m = torch.nn.Linear(3, 2)
    sync = D.FlatGradSync(m.parameters())
    m(torch.ones(4, 3)).sum().backward()
    assert sync.flat.abs().sum() > 0 and m.weight.grad.data_ptr() == sync.flat.data_ptr()
    assert sync.nbytes == (6 + 2) * 4
    sync.zero()
    assert m.bias.grad.abs().sum() == 0
    assert sync.all_reduce() is None  # world size 1: no collective


def test_masked_mae():
    y, t = torch.tensor([1.0, 2.0, 3.0, 4.0]), torch.tensor([0.0, 2.5, 0.0, 3.0])
    # mask = [0,1,0,1]/0.5 ; |diff| = [1,.5,3,1] -> mean([0,1,0,2]) = 0.75
    assert abs(float(D.masked_mae_loss(y, t)) - 0.75) < 1e-6


def _mae_inputs(zero_frac):
    """(prediction, target) of one masked-MAE case; a `zero_frac` share of the targets is 0 (missing)."""
    rs = np.random.RandomState(int(zero_frac * 10))
    y = rs.standard_normal((64, 207)).astype(np.float32)
    y[rs.random_sample((64, 207)) < zero_frac] = 0.0
    return torch.from_numpy(rs.standard_normal((64, 207)).astype(np.float32)), torch.from_numpy(y)


def test_masked_mae_matches_reference_example_util(golden_dir):
    """The op-for-op form (the checker of the fused CUDA loss) against the unmodified reference function
    examples/indexBatching/DCRNN/utils.py:10-18, whose results are stored in tests/golden/reference_data.pt
    (tests/golden/make_goldens_parity.py)."""
    ref = torch.load(os.path.join(golden_dir, "reference_data.pt"), weights_only=False)["masked_mae"]
    for zero_frac in (0.0, 0.3, 1.0):
        p, y = _mae_inputs(zero_frac)
        b = ref[zero_frac]
        assert torch.equal(D.masked_mae_loss_reference(p, y), b)
        assert torch.equal(D.masked_mae_loss(p, y), b)          # CPU tensors take the op-for-op form
