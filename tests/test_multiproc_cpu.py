"""world_size-2 gloo tests (CPU) of the N>1 host logic of bench.py: per-rank seeding of the
batch shard, MAX-over-ranks timing, whole-job throughput, and the reference arm's
"rank 0 alone runs" rule."""
import os
import subprocess
import sys

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _np(x):
    """Results cross the queue BY VALUE (numpy): a torch tensor would be handed over through the sender's fd-sharing
    socket, which is gone if the worker exits before the parent unpickles."""
    if torch.is_tensor(x):
        return x.detach().numpy().copy()
    if isinstance(x, (tuple, list)):
        return tuple(_np(v) for v in x)
    return x


def _pt(x):
    if isinstance(x, np.ndarray):
        return torch.from_numpy(x)
    if isinstance(x, tuple):
        return tuple(_pt(v) for v in x)
    return x


def _worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world),
                      LOCAL_RANK=str(rank))
    sys.path.insert(0, ROOT)
    import bench
    from cgg_b200 import synth
    dist.init_process_group('gloo', rank=rank, world_size=world)
    assert bench.dist_env() == (rank, rank, world)
    # each rank draws its own shard of the global batch (per-rank seed), no collective on the data path
    mf, _ = synth.make_inputs(rank, 1, 64, 64)
    ms_local = 10.0 + 5.0 * rank                       # rank 1 is the slow one
    ms = bench.reduce_max(ms_local, world, torch.device('cpu'))
    val = bench.whole_job_value(world, 16, 10, ms)
    q.put((rank, float(mf.sum()), ms, val))
    dist.barrier()
    dist.destroy_process_group()


def test_two_rank_timing_and_sharding():
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    (r0, s0, ms0, v0), (r1, s1, ms1, v1) = res
    assert s0 != s1                                   # different shards
    assert ms0 == ms1 == 15.0                         # MAX over ranks
    assert abs(v0 - 2 * 16 * 10 / 15e-3) < 1e-6 and v0 == v1


def _gather_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    sys.path.insert(0, ROOT)
    from cgg_b200.grounding import gather_captions_and_preds
    from oracle import cgg_oracle as O
    dist.init_process_group('gloo', rank=rank, world_size=world)
    pred_all, cap_all, mask_all = _gather_data(world)
    B = 2
    sl = slice(rank * B, (rank + 1) * B)
    pred = pred_all[:, sl].clone().requires_grad_(True)              # (L, B, Q, D): all head calls stacked
    embs, mask, preds = gather_captions_and_preds(list(cap_all[sl]), list(mask_all[sl]), pred)
    loss = sum(O.grounding_loss(preds[l], embs, mask, 10.0, 2.0) for l in range(preds.shape[0]))
    loss.backward()
    q.put(_np((rank, embs, mask, preds, float(loss), pred.grad)))
    dist.barrier()
    dist.destroy_process_group()


def _gather_data(world, L=3, B=2, Q=5, T=4, D=8):
    g = torch.Generator().manual_seed(5)
    pred = torch.randn((L, world * B, Q, D), generator=g)
    cap = torch.randn((world * B, T, D), generator=g)
    mask = torch.tensor([[1, 1, 0, 0], [1, 1, 1, 1], [0, 0, 0, 0], [1, 0, 0, 0]])[:world * B]
    return pred, cap, mask


def test_batched_caption_gather_matches_single_process():
    """mask2former_head.py:650-684: rank-major concatenation, cross-rank negatives in the loss, gradient only
    into the local slot -- with the 10 head calls' predictions travelling in one collective."""
    sys.path.insert(0, ROOT)
    from oracle import cgg_oracle as O
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = 31500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_gather_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted((_pt(q.get(timeout=120)) for _ in range(2)), key=lambda r: r[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    pred_all, cap_all, mask_all = _gather_data(2)
    full = pred_all.clone().requires_grad_(True)
    want = sum(O.grounding_loss(full[l], cap_all, mask_all, 10.0, 2.0) for l in range(full.shape[0]))
    want.backward()
    for rank, embs, mask, preds, loss, grad in res:
        assert torch.equal(embs, cap_all) and torch.equal(mask, mask_all) and mask.dtype == mask_all.dtype
        assert torch.equal(preds, pred_all)
        assert abs(loss - float(want)) < 1e-5 * max(1.0, abs(float(want)))
        torch.testing.assert_close(grad, full.grad[:, rank * 2:(rank + 1) * 2], rtol=1e-5, atol=1e-7)


def _reducer_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    sys.path.insert(0, ROOT)
    from cgg_b200.train import GradReducer
    dist.init_process_group('gloo', rank=rank, world_size=world)
    torch.manual_seed(0)
    net = torch.nn.Sequential(torch.nn.Linear(16, 2048), torch.nn.ReLU(), torch.nn.Linear(2048, 512), torch.nn.Linear(512, 4))
    red = GradReducer(net.parameters(), bucket_mb=1.0)
    x = torch.randn((8, 16), generator=torch.Generator().manual_seed(10 + rank))
    for _ in range(2):                      # two steps: buckets are reusable
        for p in net.parameters():
            p.grad = None
        net(x).pow(2).mean().backward()
        red.finish()
    red.zero()                              # third step: gradients accumulate straight into the bucket views
    assert all(p.grad.data_ptr() == red.buckets[red.index[p][0]]['flat'].data_ptr() + 4 * red.index[p][1] for p in net.parameters())
    net(x).pow(2).mean().backward()
    red.finish()
    q.put(_np((rank, len(red.buckets), [p.grad for p in net.parameters()])))
    dist.barrier()
    dist.destroy_process_group()


def test_bucketed_grad_reducer_two_ranks_gloo():
    """Host logic of the gradient all-reduce (train.py GradReducer): buckets in reverse parameter order, hooks fire the
    collective when a bucket is complete, the result is the mean over ranks and lands in .grad."""
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = 33500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_reducer_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted((_pt(q.get(timeout=120)) for _ in range(2)), key=lambda r: r[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    torch.manual_seed(0)
    net = torch.nn.Sequential(torch.nn.Linear(16, 2048), torch.nn.ReLU(), torch.nn.Linear(2048, 512), torch.nn.Linear(512, 4))
    total = 0.0
    for rank in range(2):
        x = torch.randn((8, 16), generator=torch.Generator().manual_seed(10 + rank))
        total = total + net(x).pow(2).mean()
    (total / 2).backward()
    assert res[0][1] > 1
    for rank, nb, grads in res:
        for g, p in zip(grads, net.parameters()):
            torch.testing.assert_close(g, p.grad, rtol=1e-5, atol=1e-7)


class _FusedLinear(torch.autograd.Function):
    """A stand-in for the fused weight-gradient path of cgg_b200.train._Linear: dW is accumulated straight into the
    parameter's .grad (the reducer's bucket view), the reducer is told so, and autograd gets None for it."""

    @staticmethod
    def forward(ctx, x, W, red):
        ctx.save_for_backward(x, W)
        ctx.red = red
        return x @ W.t()

    @staticmethod
    def backward(ctx, dy):
        x, W = ctx.saved_tensors
        W.grad.add_(dy.t() @ x)
        ctx.red.param_done(W, None)
        ctx.red._hook(W)          # ... and the second report autograd's post-accumulate hook adds on the GPU path (seen with
        #                           an empty Python stack right after param_done: the engine still runs the accumulation node)
        for bk in ctx.red.buckets:                  # (a collective launched too early is made to finish now, so that the
            if bk['work'] is not None:              #  outcome does not depend on a race with the rest of the backward)
                bk['work'].wait()
        return dy @ W, None, None


def _fused_reducer_worker(rank, world, port, q):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank), WORLD_SIZE=str(world))
    sys.path.insert(0, ROOT)
    from cgg_b200.train import GradReducer
    dist.init_process_group('gloo', rank=rank, world_size=world)
    torch.manual_seed(0)
    W1, W2 = torch.nn.Parameter(torch.randn(64, 16)), torch.nn.Parameter(torch.randn(8, 64))
    b2 = torch.nn.Parameter(torch.randn(8))
    red = GradReducer([W1, W2, b2], bucket_mb=1.0)              # one bucket: b2 (autograd hook) is produced FIRST in the backward
    x = torch.randn((8, 16), generator=torch.Generator().manual_seed(10 + rank))
    for _ in range(2):
        red.zero()
        h = torch.relu(_FusedLinear.apply(x, W1, red))
        (_FusedLinear.apply(h, W2, red) + b2).pow(2).mean().backward()
        red.finish()
    q.put(_np((rank, [p.grad for p in (W1, W2, b2)])))
    dist.barrier()
    dist.destroy_process_group()


def test_grad_reducer_counts_a_fused_parameter_once():
    """Regression test of a 2-GPU failure: a parameter whose gradient is written outside autograd reports through
    `param_done`, and autograd's post-accumulate hook may fire for it as well -- the bucket's all-reduce must still wait for
    EVERY parameter of the bucket (here W1, produced last) and the result must be the mean over the ranks."""
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = 36500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_fused_reducer_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted((_pt(q.get(timeout=120)) for _ in range(2)), key=lambda r: r[0])
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    torch.manual_seed(0)
    W1, W2 = torch.nn.Parameter(torch.randn(64, 16)), torch.nn.Parameter(torch.randn(8, 64))
    b2 = torch.nn.Parameter(torch.randn(8))
    total = 0.0
    for rank in range(2):
        x = torch.randn((8, 16), generator=torch.Generator().manual_seed(10 + rank))
        total = total + (torch.relu(x @ W1.t()) @ W2.t() + b2).pow(2).mean()
    (total / 2).backward()
    for rank, grads in res:
        for g, p in zip(grads, (W1, W2, b2)):
            torch.testing.assert_close(g, p.grad, rtol=1e-5, atol=1e-7)


def test_reference_arm_runs_on_rank0_only():
    env = dict(os.environ, RANK='1', LOCAL_RANK='1', WORLD_SIZE='2')
    r = subprocess.run([sys.executable, os.path.join(ROOT, 'bench.py'), '--impl', 'reference', '--gpus', '2', '--steps', '1',
                        '--warmup', '0'], env=env, capture_output=True, text=True, timeout=120)
    assert r.returncode == 0 and r.stdout.strip() == ''


def test_flop_model_matches_survey():
    sys.path.insert(0, ROOT)
    import bench
    assert abs(bench.flops_per_image(100) / 1e9 - 60.57) < 0.05      # SURVEY.md section 8d
    assert abs(bench.flops_per_image(200) / 1e9 - 104.4) < 0.1
