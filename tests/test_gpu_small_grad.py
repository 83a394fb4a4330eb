"""spw_backward_towers / Engine.gradients_towers / the small_batches=True facade: the backward pass of the one-CTA-per-tower path.

A. fp64 parity of dobj and drel (obj_grad_ref / rel_grad_ref): kink-free weights with bar 1e-5 of max |ref| per column on C1
   towers through the predict glue, 128 fully connected 10-block towers, one 32-block fully connected tower and the golden
   dicts; init_weights(nonzero_bias=True) with bar max(2e-5, 4 x the oracle's own fp32 autograd error).
B. The tiled spw_backward_obj / spw_backward_rel agree within the parity bar under the same seed; logits are forward_towers' bits.
C. Batch invariance, bit for bit: 64 mixed towers alone, in order and in two shuffled batches; through the facade, packed
   score_removals-style candidates equal one batch-1 stability_gradients call each.
D. Reruns are bit-identical and one launch each; nothing is written outside logits, dobj, drel and the workspace; a call between a
   training forward and its backward leaves the weight gradients alone.
E. Facade routing: inside the limits equals gradients_towers (1/170 for poses); outside them, and on a default network, the
   tiled path bit for bit.
"""
import ctypes

import numpy as np
import pytest
import torch

from oracle import propnet as O
from obj_grad_ref import obj_grads
from rel_grad_ref import rel_grads

pytestmark = pytest.mark.gpu
BAR = 1e-5


@pytest.fixture(scope='module')
def eng():
    from spwgnn_b200.engine import Engine
    assert torch.cuda.is_available()
    return Engine('cuda:0', seed=4)


def _bits(a):
    a = np.ascontiguousarray(a.detach().cpu().numpy() if torch.is_tensor(a) else a)
    return a.view(np.uint64 if a.dtype == np.float64 else np.uint32)


def colwise(got, ref):
    got = np.asarray(got, np.float64).reshape(len(ref), -1)
    ref = np.asarray(ref, np.float64).reshape(len(ref), -1)
    out = [0.0]
    for c in range(ref.shape[1]):
        m, d = np.abs(ref[:, c]).max(), np.abs(got[:, c] - ref[:, c]).max()
        out.append(d / m if m > 0 else (0.0 if d == 0 else np.inf))
    return max(out)


def _batch(kind, count=1, seed=0):
    from spwgnn_b200 import synth
    from spwgnn_b200.graph import TowerBatch
    if kind == 'C1':
        towers = synth.make_towers('tower', count, 3 + seed, n=7)
        return TowerBatch.from_towers(towers, inference_glue=True), towers
    if kind == 'fc10':
        towers = synth.make_towers('jenga', count, 40 + seed, n=10)
        return TowerBatch.from_towers(towers, fully_connected=True), towers
    if kind == 'fc32':
        towers = synth.make_towers('jenga', count, 70 + seed, n=32)
        return TowerBatch.from_towers(towers, fully_connected=True), towers
    if kind.startswith('golden'):
        import os
        from spwgnn_b200.graph import TowerBatch
        d = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'predict_jenga_n%s.npz' % kind[-1]))
        return TowerBatch.from_dense_relations(d['objects'], d['sender_relations'], d['receiver_relations']), None
    raise ValueError(kind)


def _reference(w, batch, seed, dtype=torch.float64):
    E = batch.n_edges
    snd, rcv = batch.in_snd[:E].long().cpu(), batch.in_rcv[:E].long().cpu()
    o = batch.obj.cpu().to(dtype)
    s = torch.as_tensor(seed, dtype=dtype)
    dobj, _, _ = obj_grads(w, o, snd, rcv, s)
    drel, _, _ = rel_grads(w, o, snd, rcv, s)
    return dobj.numpy(), drel.numpy()


def _seed(batch, rng):
    return torch.as_tensor(rng.standard_normal(batch.n_nodes).astype(np.float32)).cuda()


PARITY = [('C1', 64), ('fc10', 128), ('fc32', 1), ('golden5', 1), ('golden9', 1)]


@pytest.mark.parametrize('kind,count', PARITY)
def test_parity_kinkfree(eng, kind, count):
    w64 = O.kinkfree_weights(7)
    eng.params.load_dict(w64)
    batch, _ = _batch(kind, count)
    dl = _seed(batch, np.random.default_rng(1))
    logits, dobj, drel = eng.gradients_towers(batch, dlogits=dl, want_drel=True)
    rd, rr = _reference(w64, batch, dl.cpu().double())
    bar_rel = BAR
    if kind == 'fc32':   # drel is small against its per-step terms here: within 4x the tiled path's error on the same input
        tiled, _ = eng.relation_gradients(batch, dl)
        bar_rel = max(BAR, 4 * colwise(tiled.cpu().numpy(), rr))
    assert colwise(dobj.cpu().numpy(), rd) <= BAR
    assert colwise(drel.cpu().numpy(), rr) <= bar_rel, (colwise(drel.cpu().numpy(), rr), bar_rel)
    lf, _ = eng.forward_towers(batch, want_probs=False)
    assert torch.equal(logits, lf)


@pytest.mark.parametrize('kind', ['C1', 'fc10'])
def test_parity_nonzero_bias(eng, kind):
    """Glorot weights with nonzero biases: relu units can sit near their kink, so the bar is the oracle's own fp32 autograd
    error times 4 (at least 2e-5), as for spw_backward_obj."""
    w64 = O.init_weights(31, nonzero_bias=True)
    eng.params.load_dict(w64)
    batch, _ = _batch(kind, 16, seed=5)
    dl = _seed(batch, np.random.default_rng(2))
    _, dobj, drel = eng.gradients_towers(batch, dlogits=dl, want_drel=True)
    rd, rr = _reference(w64, batch, dl.cpu().double())
    w32 = {k: v.float() for k, v in w64.items()}
    fd, fr = _reference(w32, batch, dl.cpu().float(), dtype=torch.float32)
    assert colwise(dobj.cpu().numpy(), rd) <= max(2e-5, 4 * colwise(fd, rd))
    assert colwise(drel.cpu().numpy(), rr) <= max(2e-5, 4 * colwise(fr, rr))


def test_agrees_with_the_tiled_path_and_seeds(eng):
    eng.params.load_dict(O.kinkfree_weights(8))
    batch, _ = _batch('C1', 32, seed=1)
    rng = np.random.default_rng(3)
    dl, dp = _seed(batch, rng), _seed(batch, rng)
    logits, dobj, drel = eng.gradients_towers(batch, dlogits=dl, dprobs=dp, want_drel=True)

    def tiled_seed(z):
        p = torch.sigmoid(z)
        return dl + dp * (p * (1 - p))
    tr, to = eng.relation_gradients(batch, tiled_seed)
    assert colwise(dobj.cpu().numpy(), to.cpu().numpy()) <= BAR
    assert colwise(drel.cpu().numpy(), tr.cpu().numpy()) <= BAR
    # dlogits only and dprobs only add up to both
    _, d1, r1 = eng.gradients_towers(batch, dlogits=dl, want_drel=True)
    _, d2, r2 = eng.gradients_towers(batch, dprobs=dp, want_drel=True)
    assert colwise((d1 + d2).cpu().numpy(), dobj.cpu().numpy()) <= BAR
    assert colwise((r1 + r2).cpu().numpy(), drel.cpu().numpy()) <= BAR


def test_batch_invariance_bit_for_bit(eng):
    from spwgnn_b200 import synth
    from spwgnn_b200.graph import TowerBatch
    eng.params.load_dict(O.init_weights(33, nonzero_bias=True))
    rng = np.random.default_rng(4)
    towers = []
    for i in range(64):
        nb = int(rng.integers(1, 32))                          # a 'tower' layout of n blocks has up to n + 1
        towers += synth.make_towers('jenga' if i % 2 else 'tower', 1, 100 + i, n=nb)

    def run(order):
        b = TowerBatch.from_towers([towers[i] for i in order], thr=330.0)
        ones = torch.ones(b.n_nodes, device='cuda')
        z, d, r = eng.gradients_towers(b, dprobs=ones, want_drel=True)
        off, eo = b.node_off_host, b.in_off[:b.n_nodes + 1].cpu().numpy()
        out = {}
        for k, t in enumerate(order):
            a, c = int(off[k]), int(off[k + 1])
            out[t] = (_bits(z[a:c]), _bits(d[a:c]), _bits(r[eo[a]:eo[c]]))
        return out
    ref = run(list(range(64)))
    for order in (rng.permutation(64), rng.permutation(64)):
        got = run(list(order))
        for t in range(64):
            assert all(np.array_equal(x, y) for x, y in zip(got[t], ref[t])), t
    for t in range(0, 64, 7):
        got = run([t])
        assert all(np.array_equal(x, y) for x, y in zip(got[t], ref[t])), t


def test_facade_demolish_candidates_equal_batch1_calls():
    from spwgnn_b200.Networks import PropagationNetwork
    from spwgnn_b200 import synth
    net = PropagationNetwork(device='cuda:0', seed=5, small_batches=True)
    tower = synth.make_towers('jenga', 1, 21, n=9)[0]
    m = net.getModel(len(tower) - 1)
    net.engine.params.load_dict(O.init_weights(35, nonzero_bias=True))
    cands = [np.delete(tower, c, axis=0) for c in range(len(tower))]
    packed = m.stability_gradients(cands)
    packed_rel = m.relation_gradients(cands)
    for c, t in enumerate(cands):
        assert np.array_equal(_bits(packed[c]), _bits(m.stability_gradients([t])[0])), c
        one = m.relation_gradients([t])[0]
        assert np.array_equal(packed_rel[c][0], one[0]) and np.array_equal(_bits(packed_rel[c][1]), _bits(one[1])), c


def _c_call(eng, batch, dl, guard, drel=True, logits=True):
    """spw_backward_towers through the C ABI with guard bands of `guard` bytes around every output and the workspace"""
    api, n, E = eng.api, batch.n_nodes, batch.n_edges
    G = 256
    nb = int(api.dll.spw_backward_towers_bytes(n, E))
    bufs = {k: torch.full((G + sz + G,), guard, dtype=torch.uint8, device='cuda')
            for k, sz in (('logits', 4 * n), ('dobj', 12 * n), ('drel', 4 * max(E, 1)), ('ws', nb))}
    p = lambda k: bufs[k].data_ptr() + G
    before = api.dll.spw_launch_count()
    wp = eng.params.c_struct()
    api.check(api.dll.spw_backward_towers(ctypes.byref(wp), ctypes.byref(batch.c_graph), int(batch.max_nodes), batch.obj.data_ptr(),
                                          dl.data_ptr(), None, p('logits') if logits else None, p('dobj'),
                                          p('drel') if drel else None, p('ws'), nb, torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return bufs, api.dll.spw_launch_count() - before, G


@pytest.mark.parametrize('kind', ['C1', 'fc32'])
def test_reruns_launches_and_write_footprint(eng, kind):
    eng.params.load_dict(O.kinkfree_weights(9))
    batch, _ = _batch(kind, 8 if kind == 'C1' else 1)
    dl = _seed(batch, np.random.default_rng(5))
    outs = []
    for guard in (0x00, 0xFF):
        bufs, launches, G = _c_call(eng, batch, dl, guard)
        assert launches == 1
        for k, b in bufs.items():
            h = b.cpu().numpy()
            assert (h[:G] == guard).all() and (h[len(h) - G:] == guard).all(), (k, guard)
        outs.append({k: bufs[k][G:len(bufs[k]) - G].clone() for k in ('logits', 'dobj', 'drel')})
    for k in ('logits', 'dobj', 'drel'):
        assert torch.equal(outs[0][k], outs[1][k]), k
    # without logits and drel: nothing written there, the same dobj
    bufs, _, G = _c_call(eng, batch, dl, 0x5A, drel=False, logits=False)
    assert (bufs['logits'].cpu().numpy() == 0x5A).all() and (bufs['drel'].cpu().numpy() == 0x5A).all()
    assert torch.equal(bufs['dobj'][G:len(bufs['dobj']) - G], outs[0]['dobj'])


def test_isolation_from_a_training_step_in_flight(eng):
    eng.params.load_dict(O.init_weights(37, nonzero_bias=True))
    bx, _ = _batch('C1', 40, seed=2)
    by, _ = _batch('fc10', 50, seed=3)
    tgt = torch.as_tensor((np.random.default_rng(5).random(bx.n_nodes) > 0.5).astype(np.float32)).cuda()

    def step(interleave):
        logits, _ = eng.forward(bx, training=True, want_probs=False, dropout_rate=0.1, dropout_seed=99)
        logits = logits.clone()
        if interleave:
            eng.gradients_towers(by, dprobs=torch.ones(by.n_nodes, device='cuda'), want_drel=True)
        dl, _ = eng.bce_seed(logits, tgt, bx.n_nodes)
        eng.backward(dl)
        torch.cuda.synchronize()
        return eng.grads.flat.clone()
    assert torch.equal(step(False), step(True))


def test_facade_routing():
    from spwgnn_b200 import synth
    from spwgnn_b200.graph import TowerBatch
    from spwgnn_b200.Networks import PropagationNetwork
    on = PropagationNetwork(device='cuda:0', seed=6, small_batches=True)
    off = PropagationNetwork(device='cuda:0', seed=6)
    m_on, m_off = on.getModel(0), off.getModel(0)
    w = O.init_weights(38, nonzero_bias=True)
    on.engine.params.load_dict(w)
    off.engine.params.load_dict(w)
    towers = synth.make_towers('tower', 8, 9, n=7)
    batch = TowerBatch.from_towers(towers, inference_glue=True, device=on.engine.device)
    _, dobj, drel = on.engine.gradients_towers(batch, dprobs=torch.ones(batch.n_nodes, device='cuda'), want_drel=True)
    g = m_on.stability_gradients(towers)
    ref = dobj.cpu().numpy().astype(np.float64) / 170.0
    off_h = batch.node_off_host
    for t in range(len(towers)):
        assert np.array_equal(_bits(g[t]), _bits(ref[off_h[t]:off_h[t + 1]]))
    rg = m_on.relation_gradients(towers)
    assert sum(len(v) for _, v in rg) == batch.n_edges
    assert np.array_equal(np.sort(_bits(np.concatenate([v for _, v in rg]))), np.sort(_bits(drel.cpu().numpy().astype(np.float64))))
    # inside the limits the two networks agree to fp32 rounding
    assert colwise(np.concatenate(g), np.concatenate(m_off.stability_gradients(towers))) <= 1e-5
    # outside the limits, and on the default network, the tiled path bit for bit
    for ts in (synth.make_towers('tower', on.small_max_towers + 1, 7, n=7), synth.make_towers('jenga', 3, 8, n=on.small_max_nodes + 1)):
        a, b = m_on.stability_gradients(ts), m_off.stability_gradients(ts)
        assert all(np.array_equal(_bits(x), _bits(y)) for x, y in zip(a, b))
        a, b = m_on.relation_gradients(ts), m_off.relation_gradients(ts)
        assert all(np.array_equal(x[0], y[0]) and np.array_equal(_bits(x[1]), _bits(y[1])) for x, y in zip(a, b))
