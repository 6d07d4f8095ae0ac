"""Host logic of the train step added in round 2: flat-bucket layout in backward-production order, the two-part
gradient all-reduce with the loss riding along (gloo, world size 2), checkpoints, optimiser guards.  CPU only."""
import os
import sys

import numpy as np
import pytest
import torch
import torch.multiprocessing as mp

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _cpu_model(uv=64, **over):
    """A Model whose parameters live on the CPU (no kernel is ever launched): enough for the layout / checkpoint
    logic, which only touches torch tensors."""
    import models
    from util import io as ioutil
    cfg = ioutil.make_config(uvh=uv, uvw=uv, imh=uv, imw=uv, **over)
    model = models.get_model_class('nlt')(cfg)
    model.register_trainable()
    model.device = torch.device('cpu')
    model.build(5, 3)
    return model


def test_bucket_layout_follows_backward_production_order():
    model = _cpu_model()
    b = model.bucket
    names = {id(c): n for n, c in model.named_convs()}
    order = [names[id(L)] for L, _ in b.layout_ends]
    # decoder top-down (second conv of a block first), then encoder levels bottom-up: query block, then obs block
    assert order[:3] == ['query.13.0', 'query.12.1', 'query.12.0']
    i6 = order.index('query.6.1')
    assert order[i6:i6 + 4] == ['query.6.1', 'query.6.0', 'obs.6.1', 'obs.6.0']
    assert order[-2:] == ['query.0.0', 'obs.0.0']
    # registration order of variables()/gradients() is unchanged and every view aliases the flat buffers
    assert [tuple(v.shape) for v in model.trainable_variables][:2] == [(1, 1, 5, 16), (16,)]
    for g, v in zip(model.gradients, model.trainable_variables):
        assert v._base is b.flat and g._base is b._grad_all and g.shape == v.shape
    # offsets: disjoint, 16-byte aligned kernels, ends increasing
    spans = sorted((ko, ko + ks) for ko, ks, _, _ in b.slices)
    assert all(a[1] <= c[0] for a, c in zip(spans, spans[1:])) and all(ko % 4 == 0 for ko, _ in spans)
    L, off = b.split_point(0.9)
    assert L is not None and 0.9 * b.n <= off < b.n
    # the head holds the deep levels: nothing of levels 0-3 lies in front of the split
    head = {names[id(l)] for l, end in b.layout_ends if end <= off}
    assert not any(n.split('.')[1] in ('0', '1', '2', '3') and n.startswith('obs') for n in head)
    assert b.grad_with_loss().numel() == b.n + 1 and b.loss_slot.data_ptr() == b.grad.data_ptr() + 4 * b.n


def _reducer_worker(rank, world, port, q):
    for p in (ROOT, os.path.join(ROOT, 'neural-light-transport_b200')):
        if p not in sys.path:
            sys.path.insert(0, p)
    # CPU-only ranks (see tests/test_dist.py): no rank may bind a GPU that a one-GPU machine does not have
    os.environ.update(RANK=str(rank), WORLD_SIZE=str(world), LOCAL_RANK=str(rank), MASTER_ADDR='127.0.0.1',
                      MASTER_PORT=str(port), CUDA_VISIBLE_DEVICES='')
    import engine
    import trainvali
    torch.set_num_threads(1)
    strategy = trainvali.Strategy(backend='gloo')
    engine.USE_SIDE_STREAM = False
    model = _cpu_model()
    b = model.bucket
    out = []
    for overlap in (True, False):
        g = torch.Generator().manual_seed(100 + rank)
        b.grad.copy_(torch.rand(b.n, generator=g))
        red = trainvali.GradReducer(strategy, model, overlap=overlap)
        red.begin()
        assert (engine.WGRAD_HOOK is not None) == overlap
        if overlap:
            for L, _ in b.layout_ends:          # backward issues the weight gradients in layout order
                engine.WGRAD_HOOK(L)
            assert red.work is not None and red.split > 0
        loss = red.finish(torch.tensor(0.25 * (rank + 1)))
        assert engine.WGRAD_HOOK is None
        out.append((b.grad.clone().numpy(), float(loss)))
    strategy.barrier()
    if rank == 0:
        q.put(out)
    torch.distributed.destroy_process_group()


@pytest.mark.timeout(300)
def test_two_part_allreduce_with_loss_slot_equals_plain_sum():
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = 31500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_reducer_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    out = q.get(timeout=240)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    n = out[0][0].shape[0]
    want = sum(torch.rand(n, generator=torch.Generator().manual_seed(100 + r)) for r in range(2)).numpy()
    for grad, loss in out:
        np.testing.assert_allclose(grad, want, rtol=0, atol=1e-6)
        assert abs(loss - 0.75) < 1e-6


def test_checkpoint_round_trip_and_manager(tmp_path):
    import trainvali
    from util import ckpt
    model = _cpu_model()
    opt = trainvali.Adam(learning_rate=1e-3, amsgrad=True)
    g = torch.Generator().manual_seed(3)
    model.flat_params.copy_(torch.randn(model.flat_params.numel(), generator=g))
    opt.m, opt.v, opt.vhat = (torch.rand(model.flat_params.numel(), generator=g) for _ in range(3))
    opt.iterations = 17
    mgr = ckpt.CheckpointManager(str(tmp_path / 'checkpoints'), max_to_keep=2)
    assert mgr.latest_checkpoint is None and mgr.restore_latest(model, opt) is None
    paths = [mgr.save(model, opt, step=s) for s in (5, 6, 7)]
    assert [os.path.basename(p) for p in paths] == ['ckpt-1.npz', 'ckpt-2.npz', 'ckpt-3.npz']
    assert sorted(os.listdir(mgr.dir)) == ['ckpt-2.npz', 'ckpt-3.npz']      # max_to_keep
    with np.load(paths[-1]) as z:
        keys = set(z.files)
    assert 'net/net_query_layer0/conv0/kernel' in keys and 'net/net_obs_layer6/conv1/bias' in keys
    assert 'optimizer/vhat/net_query_layer7/conv0/kernel' in keys and 'optimizer/iterations' in keys
    # a DIFFERENT flat layout restores to the same named tensors
    other = _cpu_model()
    other_opt = trainvali.Adam(learning_rate=1e-3, amsgrad=True)
    step = mgr.restore_latest(other, other_opt)
    assert step == 7 and other_opt.iterations == 17 and int(other_opt.step_dev) == 17
    for (n1, c1), (n2, c2) in zip(model.named_convs(), other.named_convs()):
        assert n1 == n2 and torch.equal(c1.kernel, c2.kernel) and torch.equal(c1.bias, c2.bias)
    for slot in ('m', 'v', 'vhat'):      # per-layer views (the alignment gaps of the flat buffer are not state)
        a, b = ckpt._slot_views(model, getattr(opt, slot)), ckpt._slot_views(other, getattr(other_opt, slot))
        assert a.keys() == b.keys() and all(torch.equal(a[k], b[k]) for k in a)
    # shape mismatch and missing tensors are errors unless expect_partial
    state = ckpt.state_dict(model, opt, 1)
    bad = dict(state)
    bad['net/net_query_layer0/conv0/kernel'] = np.zeros((1, 1, 6, 16), np.float32)
    with pytest.raises(ValueError):
        ckpt.load_state(other, bad)
    del state['net/net_obs_layer2/conv1/bias']
    with pytest.raises(KeyError):
        ckpt.load_state(other, state)
    ckpt.load_state(other, state, expect_partial=True)


def test_optimizer_guards():
    import trainvali
    from util import io as ioutil
    with pytest.raises(NotImplementedError):
        trainvali.make_optimizer(ioutil.make_config(mgm=1.0))        # clipnorm is refused, not ignored
    opt = trainvali.make_optimizer(ioutil.make_config(lr=2.5e-4))
    assert opt.lr == 2.5e-4
    model = _cpu_model()
    with pytest.raises(ValueError):                                   # foreign tensors are not views of the buckets
        opt.apply_gradients([(torch.zeros(3), torch.zeros(3))])


def test_extract_feat_refuses_unbuilt_model():
    import models
    import nlt_test
    from util import io as ioutil
    model = models.get_model_class('nlt')(ioutil.make_config(uvh=64, uvw=64, imh=64, imw=64))
    model.register_trainable()
    with pytest.raises(RuntimeError):
        nlt_test.extract_feat(model, [])


def test_tf_tensor_bundle_round_trip_and_restore(tmp_path):
    """util/tf_ckpt.py: a bundle written in the reference's object-graph key layout restores into the model through
    util.ckpt.restore(prefix) / nlt_test.restore_model; table framing (footer magic, block handles, prefix-compressed
    keys over several blocks), snappy block decoding and the proto fields are exercised."""
    import trainvali
    from util import ckpt, tf_ckpt
    model = _cpu_model()
    opt = trainvali.Adam(learning_rate=1e-3, amsgrad=True)
    g = torch.Generator().manual_seed(9)
    model.flat_params.copy_(torch.randn(model.flat_params.numel(), generator=g))
    opt.m, opt.v, opt.vhat = (torch.rand(model.flat_params.numel(), generator=g) for _ in range(3))
    opt.iterations = 43
    prefix = str(tmp_path / 'checkpoints' / 'ckpt-43')
    tf_ckpt.save_nlt_state(prefix, ckpt.state_dict(model, opt, step=43))
    raw = tf_ckpt.load_bundle(prefix)
    assert 'net/net_query_layer0/kernel/.ATTRIBUTES/VARIABLE_VALUE' in raw                       # bare Conv2D
    assert 'net/net_obs_layer4/layer_with_weights-1/bias/.ATTRIBUTES/VARIABLE_VALUE' in raw       # Sequential block
    assert raw['net/net_query_layer7/layer_with_weights-0/kernel/.ATTRIBUTES/VARIABLE_VALUE'].shape == (2, 2, 128, 1024)
    assert len(tf_ckpt.read_index(prefix + '.index')) == len(raw) > 150                          # many blocks
    other = _cpu_model()
    other_opt = trainvali.Adam(learning_rate=1e-3, amsgrad=True)
    assert ckpt.restore(prefix, other, other_opt) == 43 and other_opt.iterations == 43
    for (n1, c1), (n2, c2) in zip(model.named_convs(), other.named_convs()):
        assert torch.equal(c1.kernel, c2.kernel) and torch.equal(c1.bias, c2.bias)
    a, b = ckpt._slot_views(model, opt.vhat), ckpt._slot_views(other, other_opt.vhat)
    assert all(torch.equal(a[k], b[k]) for k in a)
    # snappy-compressed blocks decode too (literal + copy elements)
    payload = b'abcdabcdabcdabcdXYZ' * 3
    comp = bytes([len(payload)]) + bytes([(4 - 1) << 2]) + b'abcd' + bytes([((12 - 1) << 2) | 2, 4, 0]) + \
        bytes([(3 - 1) << 2]) + b'XYZ' + bytes([((38 - 1) << 2) | 2, 19, 0])
    assert tf_ckpt._snappy_decompress(comp) == payload
    with pytest.raises(ValueError):
        tf_ckpt.read_index(__file__)
