"""world_size-2 (and 3) gloo tests of the multi-GPU host logic (masic_b200/sharding.py), on CPU.

The device side of the claim — a pair's result is bit-identical whatever batch/rank it runs in — is
tests/test_hsic_gpu.py::test_determinism_and_batch_sharding_invariance; here the N>1 plumbing itself runs:
pair assignment, the gather of per-pair rows to rank 0 (ragged tails included), and the gradient
all-reduce that config 5 (data-parallel training) uses, against a single-process run of the concatenated batch.
"""
import os
import socket

import pytest
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from masic_b200.sharding import GradBuckets, evaluate_sharded, gather_pair_results, shard_pairs


def _free_port():
    with socket.socket() as s:
        s.bind(("127.0.0.1", 0))
        return s.getsockname()[1]


def _spawn(fn, world, *args):
    port = _free_port()
    mp.spawn(_entry, args=(world, port, fn, args), nprocs=world, join=True)


def _entry(rank, world, port, fn, args):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    try:
        fn(rank, world, *args)
    finally:
        dist.destroy_process_group()


def _pair_row(i):
    """Deterministic stand-in for (bpp, psnr1, psnr2) of pair i: depends on the pair only."""
    g = torch.Generator().manual_seed(1000 + i)
    return torch.rand(3, generator=g, dtype=torch.float64).tolist()


def test_shard_pairs_partitions_every_pair_once():
    for n in (0, 1, 7, 64):
        for world in (1, 2, 3, 8):
            owned = [shard_pairs(n, r, world) for r in range(world)]
            flat = sorted(i for o in owned for i in o)
            assert flat == list(range(n))
            assert max(len(o) for o in owned) - min(len(o) for o in owned) <= 1
    with pytest.raises(ValueError):
        shard_pairs(4, 2, 2)


def _w_eval(rank, world, n_pairs, tmp):
    table = evaluate_sharded(n_pairs, lambda i: (i,), _pair_row, 3)
    if rank == 0:
        torch.save(table, tmp)
    else:
        assert table is None


@pytest.mark.parametrize("world,n_pairs", [(2, 8), (2, 7), (3, 4), (2, 1)])
def test_sharded_eval_is_independent_of_world_size(world, n_pairs, tmp_path):
    f = str(tmp_path / "t.pt")
    _spawn(_w_eval, world, n_pairs, f)
    got = torch.load(f)
    want = torch.tensor([_pair_row(i) for i in range(n_pairs)], dtype=torch.float64)
    assert torch.equal(got, want)                                 # bit-identical to the 1-process table
    assert torch.equal(evaluate_sharded(n_pairs, lambda i: (i,), _pair_row, 3), want)


def _w_dup(rank, world):
    # both ranks claim pair 0 -> rank 0 must refuse the table
    try:
        gather_pair_results({0: [1.0, 2.0]}, 2, 2)
    except ValueError as e:
        assert rank == 0 and "missing or duplicated" in str(e)
    else:
        assert rank != 0


def test_gather_rejects_duplicates_and_holes():
    _spawn(_w_dup, 2)
    with pytest.raises(ValueError):
        gather_pair_results({0: [1.0]}, 2, 1)                     # pair 1 missing (world 1)
    with pytest.raises(ValueError):
        gather_pair_results({0: [1.0, 2.0]}, 1, 1)                # wrong row width


def _toy():
    torch.manual_seed(5)
    return torch.nn.Sequential(torch.nn.Conv2d(3, 8, 3, padding=1), torch.nn.ReLU(), torch.nn.Conv2d(8, 3, 3, padding=1))


def _loss(net, x):
    # normalised by the LOCAL batch like RateDistortionLoss (newtrain_codec_real.py:76)
    return ((net(x) - x) ** 2).mean()


def _w_grad(rank, world, tmp):
    net = _toy()
    g = torch.Generator().manual_seed(9)
    x = torch.rand(2 * world, 3, 16, 16, generator=g)
    _loss(net, x[2 * rank:2 * rank + 2]).backward()               # batch 2 per rank (config 5)
    gb = GradBuckets(net.parameters(), bucket_bytes=512)          # tiny buckets: several all-reduces
    assert len(gb.buckets) > 1
    gb.allreduce_()
    if rank == 0:
        torch.save([p.grad for p in net.parameters()], tmp)


@pytest.mark.parametrize("world", [2, 3])
def test_gradient_allreduce_matches_concatenated_batch(world, tmp_path):
    f = str(tmp_path / "g.pt")
    _spawn(_w_grad, world, f)
    got = torch.load(f)
    net = _toy()
    g = torch.Generator().manual_seed(9)
    x = torch.rand(2 * world, 3, 16, 16, generator=g)
    _loss(net, x).backward()
    for a, p in zip(got, net.parameters()):
        assert torch.allclose(a, p.grad, rtol=1e-5, atol=1e-7)


def test_grad_buckets_single_process_is_identity():
    net = _toy()
    _loss(net, torch.rand(2, 3, 8, 8)).backward()
    before = [p.grad.clone() for p in net.parameters()]
    GradBuckets(net.parameters()).allreduce_()
    for a, p in zip(before, net.parameters()):
        assert torch.equal(a, p.grad)


def _w_mean(rank, world, tmp):
    from masic_b200.sharding import all_reduce_mean_
    g = torch.Generator().manual_seed(40 + rank)
    flat = torch.rand(1000, generator=g)
    # the training step's two forms: the whole flat gradient buffer at once, or a prefix started asynchronously
    # (while the rest of the backward pass would run) and the suffix afterwards
    whole = flat.clone()
    assert all_reduce_mean_(whole) is not None
    split = flat.clone()
    h0 = all_reduce_mean_(split[:512], async_op=True)
    h1 = all_reduce_mean_(split[512:], async_op=True)
    h0.wait(); h1.wait()
    h0.wait()                                                    # idempotent
    # (three or more ranks: the backend may add the ranks' values in another order for another buffer size)
    assert torch.allclose(whole, split, rtol=1e-6, atol=1e-7)
    if rank == 0:
        torch.save(whole, tmp)


@pytest.mark.parametrize("world", [2, 3])
def test_all_reduce_mean_whole_and_split_buffer(world, tmp_path):
    """HSICTrainer.train_step's collective (sharding.all_reduce_mean_): the mean over the ranks, in place, identical
    whether the flat buffer is reduced at once or as an asynchronous prefix + suffix."""
    f = str(tmp_path / "m.pt")
    _spawn(_w_mean, world, f)
    want = torch.stack([torch.rand(1000, generator=torch.Generator().manual_seed(40 + r)) for r in range(world)]).mean(0)
    assert torch.allclose(torch.load(f), want, rtol=1e-6, atol=1e-7)


def test_all_reduce_mean_single_process_is_identity():
    from masic_b200.sharding import all_reduce_mean_
    t = torch.arange(8.0)
    all_reduce_mean_(t).wait()
    assert torch.equal(t, torch.arange(8.0))
