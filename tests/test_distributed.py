"""Gradient all-reduce of the fine-tuning configuration (SURVEY 8(a) A19) on CPU: world_size-2 gloo against the
arithmetic of the reference's LegacyDistributedDataParallel.all_reduce_grads
(fairseq/fairseq/distributed/legacy_distributed_data_parallel.py:76-165): mean over ranks, missing gradients count
as zeros and receive the mean, `expert` parameters are skipped, no_sync() postpones, parameters larger than the
bucket are reduced on their own."""
import os
import socket

import torch
import torch.distributed as dist
import torch.multiprocessing as mp

from multimodalvc_b200.distributed import GradientAllReducer


def _free_port():
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    p = s.getsockname()[1]
    s.close()
    return p


def _make_params():
    torch.manual_seed(0)
    shapes = [(7, 5), (3,), (64, 33), (1,), (10, 10), (2500,)]
    return [torch.nn.Parameter(torch.randn(*s)) for s in shapes]


def _grads_for(rank, params):
    g = torch.Generator().manual_seed(100 + rank)
    return [torch.randn(p.shape, generator=g) for p in params]


def _by_value(arrays):
    """Workers send results as numpy arrays, which a queue pickles by value.  A CPU tensor would travel as a file
    descriptor that the parent fetches from the worker while unpickling, and rank 0 may have exited by then."""
    return [None if a is None else torch.from_numpy(a) for a in arrays]


def _worker(rank, world, port, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    params = _make_params()
    params[3].requires_grad_(False)                      # frozen: never touched
    params[4].expert = True                              # unshared: skipped (reference :131-133)
    grads = _grads_for(rank, params)
    for i, (p, g) in enumerate(zip(params, grads)):
        if i == 3:
            continue
        if i == 1 and rank == 1:
            continue                                      # rank 1 has no gradient for param 1
        p.grad = g.clone()
    red = GradientAllReducer(params, buffer_size=2 ** 28, bucket_bytes=4 * 700)      # 700-element buckets: several
    with red.no_sync():
        assert red.all_reduce_grads() == 0
        assert torch.equal(params[0].grad, grads[0])     # untouched inside no_sync
    n = red.all_reduce_grads()
    out = [None if p.grad is None else p.grad.numpy().copy() for p in params]
    if rank == 0:
        q.put((n, out))        # numpy arrays: see _by_value
    dist.barrier()
    dist.destroy_process_group()


def test_gradient_all_reduce_two_ranks_gloo():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    n, out = q.get(timeout=120)
    out = _by_value(out)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    params = _make_params()
    g0, g1 = _grads_for(0, params), _grads_for(1, params)
    assert n >= 3                                         # several buckets + the big parameter on its own
    torch.testing.assert_close(out[0], (g0[0] + g1[0]) / 2)
    torch.testing.assert_close(out[1], g0[1] / 2)         # rank 1 contributed zeros
    torch.testing.assert_close(out[2], (g0[2] + g1[2]) / 2)
    assert out[3] is None                                 # frozen parameter
    assert torch.equal(out[4], g0[4])                     # expert parameter: local gradient kept
    torch.testing.assert_close(out[5], (g0[5] + g1[5]) / 2)


def test_single_process_is_identity_and_fills_missing_grads():
    params = _make_params()
    grads = _grads_for(0, params)
    for p, g in zip(params[:-1], grads[:-1]):
        p.grad = g.clone()
    red = GradientAllReducer(params)
    red.all_reduce_grads()
    for p, g in zip(params[:-1], grads[:-1]):
        assert torch.equal(p.grad, g)
    assert params[-1].grad is not None and not params[-1].grad.any()     # reference :124-125: zeros_like


def _worker_presynced(rank, world, port, q):
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    params = _make_params()
    grads = _grads_for(rank, params)
    for p, g in zip(params, grads):
        p.grad = g.clone()
    red = GradientAllReducer(params)
    # the device backward reports what it already averaged (mark_reduced): those gradients must not be reduced twice
    red.mark_reduced([params[0], params[2]])
    n1 = red.all_reduce_grads()
    first = [p.grad.numpy().copy() for p in params]
    n2 = red.all_reduce_grads()                           # the mark is per step: the next call reduces everything again
    second = [p.grad.numpy().copy() for p in params]
    # off an NCCL group (gloo here) the bucketed overlap declines and leaves the work to all_reduce_grads
    declined = red.reduce_buckets(None, None, torch.zeros(4)) is False
    if rank == 0:
        q.put((n1, n2, first, second, declined))        # numpy arrays: see _by_value
    dist.barrier()
    dist.destroy_process_group()


def test_gradients_reduced_during_the_backward_are_skipped_once():
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = _free_port()
    procs = [ctx.Process(target=_worker_presynced, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    n1, n2, first, second, declined = q.get(timeout=120)
    first, second = _by_value(first), _by_value(second)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    params = _make_params()
    g0, g1 = _grads_for(0, params), _grads_for(1, params)
    assert declined and n1 >= 1 and n2 >= 1
    for i in (0, 2):
        assert torch.equal(first[i], g0[i])                                  # skipped in the first call ...
        torch.testing.assert_close(second[i], (g0[i] + g1[i]) / 2)           # ... reduced by the second
    for i in (1, 3, 4, 5):
        torch.testing.assert_close(first[i], (g0[i] + g1[i]) / 2)
        torch.testing.assert_close(second[i], (g0[i] + g1[i]) / 2)           # averages of identical values stay put
