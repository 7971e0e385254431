"""N > 1 host logic on CPU (gloo, world_size 2): ray sharding and the flat-gradient all-reduce of
hypernerf_torch_b200.train (the reference delegates this to Lightning ddp_sharded, train.py:224-229).

The per-ray kernels need a GPU, so a small torch module stands in for the model here: what is under test is that
(a) contiguous shards cover the batch exactly once, (b) every .grad is a view of ONE flat buffer, (c) one
all_reduce(sum) of that buffer with the 1/global_rays loss scaling reproduces the single-process global-mean
gradient.  Rendezvous on 127.0.0.1."""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from hypernerf_torch_b200 import train as hn_train


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _toy_model():
    torch.manual_seed(0)
    return torch.nn.Sequential(torch.nn.Linear(6, 17), torch.nn.ReLU(), torch.nn.Linear(17, 3), torch.nn.Sigmoid())


def _local_step(model, fg, rays, rgbs, global_rays, chunk):
    """Same accumulation rule as train.train_step (sum-MSE / (3 * global_rays), chunked), on a toy model."""
    fg.zero()
    for i in range(0, rays.shape[0], chunk):
        out = model(rays[i:i + chunk, :6])
        loss = 2 * torch.nn.functional.mse_loss(out, rgbs[i:i + chunk], reduction='sum') / (3.0 * global_rays)
        loss.backward()
    fg.all_reduce()


def _worker(rank, world, port, n_rays, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        g = torch.Generator().manual_seed(7)
        rays, rgbs = torch.randn(n_rays, 9, generator=g), torch.rand(n_rays, 3, generator=g)
        lo, hi = hn_train.shard_bounds(n_rays, rank, world)
        model = _toy_model()
        fg = hn_train.FlatGrads(model.parameters())
        _local_step(model, fg, rays[lo:hi], rgbs[lo:hi], n_rays, chunk=5)
        q.put((rank, lo, hi, fg.flat.clone()))
    finally:
        dist.destroy_process_group()


@pytest.mark.parametrize("n_rays", [37, 64])
def test_two_rank_flat_gradient_matches_single_process(n_rays):
    world, port = 2, _free_port()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, world, port, n_rays, q)) for r in range(world)]
    for p in procs:
        p.start()
    got = sorted(q.get(timeout=120) for _ in range(world))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    # shards are contiguous, disjoint and cover the batch
    assert got[0][1] == 0 and got[0][2] == got[1][1] and got[1][2] == n_rays
    # single-process reference on the whole batch
    g = torch.Generator().manual_seed(7)
    rays, rgbs = torch.randn(n_rays, 9, generator=g), torch.rand(n_rays, 3, generator=g)
    model = _toy_model()
    fg = hn_train.FlatGrads(model.parameters())
    _local_step(model, fg, rays, rgbs, n_rays, chunk=n_rays)
    for _, _, _, flat in got:
        torch.testing.assert_close(flat, fg.flat, rtol=1e-5, atol=1e-7)


def test_flat_grads_are_views_of_one_buffer():
    model = _toy_model()
    fg = hn_train.FlatGrads(model.parameters())
    base = fg.flat.data_ptr()
    for p, off in zip(fg.params, fg.offsets):
        assert p.grad.data_ptr() == base + 4 * off and off % 4 == 0
    model(torch.randn(4, 6)).sum().backward()
    assert fg.flat.abs().sum() > 0
    fg.zero()
    assert all(float(p.grad.abs().sum()) == 0 for p in fg.params)


@pytest.mark.parametrize("n,world", [(65536, 1), (65536, 8), (10, 4), (3, 8), (0, 2)])
def test_shard_bounds_partition(n, world):
    spans = [hn_train.shard_bounds(n, r, world) for r in range(world)]
    assert spans[0][0] == 0 and spans[-1][1] == n
    for a, b in zip(spans, spans[1:]):
        assert a[1] == b[0]
    assert all(lo <= hi for lo, hi in spans)


# ------------------------------------------------------------------------------------------------------------------------
# hardware: 2 NCCL ranks, the real model (VERDICT r1 item 7).  Skips cleanly on a host with fewer than 2 GPUs.
# ------------------------------------------------------------------------------------------------------------------------
def _nccl_worker(rank, world, port, n_rays, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    torch.cuda.set_device(rank)
    dev = torch.device("cuda", rank)
    dist.init_process_group("nccl", rank=rank, world_size=world, device_id=dev)
    try:
        from hypernerf_torch_b200 import synthetic
        from hypernerf_torch_b200.models import NerfModel
        from oracle import ref_loader
        model = NerfModel(ref_loader.EMBEDDINGS, **ref_loader.cfg1_kwargs(n_fine=64, noise_std=1.0))
        model.load_state_dict(synthetic.make_state_dict(model, seed=0, boosted=True))
        model = model.to(dev)
        fg = hn_train.FlatGrads(model.parameters())
        model.attach_flat_grads(fg)
        rays, rgbs = synthetic.train_rays(n_rays, seed=2, device=dev)
        rel = hn_train.dp_parity_check(model, fg, rays, rgbs, tol=1e-4)
        q.put((rank, rel))
    finally:
        dist.destroy_process_group()


@pytest.mark.gpu
def test_two_gpu_train_step_equals_one_gpu_step():
    """train.train_step on the two halves of a 4 096-ray batch (globally drawn, rank-sliced u / noise tensors, one flat
    NCCL all-reduce) == the 1-GPU step on the whole batch, to 1e-4 relative (SURVEY.md §4, §8(e))."""
    if torch.cuda.device_count() < 2:
        pytest.skip("needs 2 GPUs")
    world, port = 2, _free_port()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_nccl_worker, args=(r, world, port, 4096, q)) for r in range(world)]
    for p in procs:
        p.start()
    got = sorted(q.get(timeout=300) for _ in range(world))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    print("2-GPU vs 1-GPU flat gradient, relative L2:", got)
    assert all(rel <= 1e-4 for _, rel in got)


@pytest.mark.gpu
def test_dp_parity_check_single_rank_is_exact():
    """The helper itself on one GPU (world 1): sharded == whole by construction, to accumulation-order noise."""
    from hypernerf_torch_b200 import synthetic
    from hypernerf_torch_b200.models import NerfModel
    from oracle import ref_loader
    model = NerfModel(ref_loader.EMBEDDINGS, **ref_loader.cfg1_kwargs(n_fine=64, noise_std=1.0))
    model.load_state_dict(synthetic.make_state_dict(model, seed=0, boosted=True))
    model = model.to("cuda")
    fg = hn_train.FlatGrads(model.parameters())
    model.attach_flat_grads(fg)
    rays, rgbs = synthetic.train_rays(2048, seed=2, device="cuda")
    assert hn_train.dp_parity_check(model, fg, rays, rgbs, tol=1e-5) <= 1e-5
