"""CPU, world_size 2 over gloo: the data-parallel exchange step of NeRF training (SURVEY.md 8e) -- one mean
all-reduce of the flat gradient buffers -- and the ray sharding of rendering (no collective)."""
import os
import socket

import torch
import torch.distributed as td
import torch.multiprocessing as mp


def _free_port() -> int:
    with socket.socket() as s:
        s.bind(('127.0.0.1', 0))
        return s.getsockname()[1]


def _worker(rank: int, world: int, port: int, out) -> None:
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    td.init_process_group('gloo', rank=rank, world_size=world)
    from nerficg_b200 import dist
    try:
        n = 595848
        torch.manual_seed(100 + rank)
        grads = [torch.randn(n), torch.randn(n)]
        local = [g.clone() for g in grads]
        dist.allreduce_mean_(grads)
        # reference: gather every rank's local gradient and average by hand
        ok = True
        for g, l in zip(grads, local):
            gathered = [torch.empty_like(l) for _ in range(world)]
            td.all_gather(gathered, l)
            ok &= torch.allclose(g, torch.stack(gathered).mean(0), atol=1e-7)
        # parameters: rank 0's weights win
        p = [torch.full((16,), float(rank + 1))]
        dist.broadcast_parameters_(p)
        ok &= bool((p[0] == 1.0).all())
        # rendering shards: disjoint, complete, no communication needed to know one's share
        mine = list(dist.shard_range(200))
        gathered = [None] * world
        td.all_gather_object(gathered, mine)
        ok &= sorted(sum(gathered, [])) == list(range(200))
        # data-parallel equivalence: mean of per-rank mean-gradients == gradient of the mean over the union batch
        w = torch.ones(8, requires_grad=True)
        torch.manual_seed(7)
        x_all = torch.randn(world * 32, 8)
        x = x_all[rank * 32:(rank + 1) * 32]
        ((x @ w) ** 2).mean().backward()
        g_local = [w.grad.clone()]
        dist.allreduce_mean_(g_local)
        w2 = torch.ones(8, requires_grad=True)
        ((x_all @ w2) ** 2).mean().backward()
        ok &= torch.allclose(g_local[0], w2.grad, atol=1e-6)
        # the captured step's flavour: SUM all-reduce, 1/world folded into the optimiser's gradient read (K7 grad_mult)
        g_sum = [local[0].clone()]
        dist.allreduce_sum_(g_sum)
        ok &= torch.allclose(g_sum[0] * (1.0 / world), grads[0], atol=1e-6)
        # the NeRF trainer's autograd path under data parallelism: identical start (rank 0's weights), per-rank batches,
        # all-reduced gradients -> identical weights on every rank after the step (no CUDA kernel involved: CPU Adam on a stand-in loss)
        from nerficg_b200 import Framework
        Framework.load_config(None, {'GLOBAL.LOG_LEVEL': 0})
        from nerficg_b200.Methods.NeRF.Model import NeRF
        torch.manual_seed(50 + rank)                         # ranks build DIFFERENT weights
        model = NeRF('ddp').build()
        dist.broadcast_parameters_([b.flat_params for b in model.blocks()])
        opt = torch.optim.Adam(model.parameters(), lr=1e-3)
        torch.manual_seed(60 + rank)                         # ... and see different data
        loss = sum(((p * torch.randn_like(p)).sum()) ** 2 for p in model.parameters())
        loss.backward()
        dist.allreduce_mean_([p.grad for p in model.parameters() if p.grad is not None])
        opt.step()
        flat = torch.cat([b.flat_params.detach() for b in model.blocks()])
        both = [torch.empty_like(flat) for _ in range(world)]
        td.all_gather(both, flat)
        ok &= torch.equal(both[0], both[1])
        out[rank] = bool(ok)
    finally:
        td.destroy_process_group()


def test_allreduce_mean_and_sharding_world2():
    world = 2
    # the result server is spawned, not forked: earlier tests in the same process may have initialised CUDA and its threads
    mgr = mp.get_context('spawn').Manager()
    out = mgr.dict()
    mp.spawn(_worker, args=(world, _free_port(), out), nprocs=world, join=True)
    assert dict(out) == {0: True, 1: True}


def test_single_process_is_identity():
    from nerficg_b200 import dist
    g = [torch.arange(4.0)]
    dist.allreduce_mean_(g)
    assert g[0].tolist() == [0.0, 1.0, 2.0, 3.0]
    assert dist.world_size() == 1 and dist.rank() == 0 and list(dist.shard_range(5)) == [0, 1, 2, 3, 4]
