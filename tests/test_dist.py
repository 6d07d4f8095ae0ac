"""Data-parallel host logic on CPU: two gloo ranks shard the global batch, each
computes loss_b / global_bs gradients (compute = the oracle here; the CUDA path
is covered by the -m gpu tests), ONE all-reduce(SUM) through
trainvali.Strategy reproduces the single-process global-batch gradient
(nlt/trainvali.py:277-284)."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CFG = dict(depth0=16, depth=16, kernel=2, stride=2, norm='None', act='leakyrelu', pool='None', use_obs=True,
           skip_connect_base=True, imh=16, imw=16, uvh=16, uvw=16)
GLOBAL_BS = 4


def _flat_grad(params, batch):
    from oracle import nlt_oracle as O
    ps = {k: v.clone().requires_grad_(True) for k, v in params.items()}
    O.train_loss(ps, CFG, batch, GLOBAL_BS).backward()
    return torch.cat([ps[k].grad.reshape(-1) for k in sorted(ps)])


def _shard(batch, rank, world):
    n = batch[1].shape[0] // world
    sl = slice(rank * n, (rank + 1) * n)
    return tuple(t[sl] if torch.is_tensor(t) else t[sl] for t in batch)


def _worker(rank, world, port, q):
    for p in (ROOT, os.path.join(ROOT, 'neural-light-transport_b200')):
        if p not in sys.path:
            sys.path.insert(0, p)
    # the ranks compute on the CPU: with a GPU visible, Strategy would bind rank r to cuda:r, which a machine with
    # fewer GPUs than ranks does not have
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR='127.0.0.1',
                      MASTER_PORT=str(port), CUDA_VISIBLE_DEVICES='')
    import trainvali
    from oracle import nlt_oracle as O
    from util import synth
    torch.set_num_threads(1)
    strategy = trainvali.Strategy(backend='gloo')
    assert strategy.num_replicas_in_sync == world
    params = O.init_params(CFG, seed=1, dtype=torch.float64)
    batch = synth.make_batch(GLOBAL_BS, 16, 16, seed=77)
    batch = tuple(t.double() if torch.is_tensor(t) else t for t in batch)
    g = _flat_grad(params, _shard(batch, rank, world))
    strategy.all_reduce_sum_(g)
    loss = O.train_loss(params, CFG, _shard(batch, rank, world), GLOBAL_BS).detach().clone()
    strategy.all_reduce_sum_(loss)
    strategy.barrier()
    if rank == 0:
        q.put((g.numpy(), float(loss)))
    torch.distributed.destroy_process_group()


@pytest.mark.timeout(300)
def test_two_rank_gradient_allreduce_equals_global_batch():
    from oracle import nlt_oracle as O
    from util import synth
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    g2, loss2 = q.get(timeout=240)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    params = O.init_params(CFG, seed=1, dtype=torch.float64)
    batch = synth.make_batch(GLOBAL_BS, 16, 16, seed=77)
    batch = tuple(t.double() if torch.is_tensor(t) else t for t in batch)
    g1 = _flat_grad(params, batch).numpy()
    loss1 = float(O.train_loss(params, CFG, batch, GLOBAL_BS))
    np.testing.assert_allclose(g2, g1, rtol=1e-10, atol=1e-14)
    assert abs(loss2 - loss1) < 1e-12


def test_strategy_single_process_is_identity():
    import trainvali
    for k in ('RANK', 'WORLD_SIZE', 'LOCAL_RANK'):
        os.environ.pop(k, None)
    s = trainvali.Strategy()
    t = torch.arange(4.0)
    assert s.num_replicas_in_sync == 1 and torch.equal(s.all_reduce_sum_(t), torch.arange(4.0))
    with pytest.raises(NotImplementedError):
        trainvali.get_strategy('cpu')
    with pytest.raises(NotImplementedError):
        trainvali.get_strategy('tpu')
    with pytest.raises(NotImplementedError):
        trainvali.Adam(amsgrad=False)
