"""spw_forward_towers / Engine.forward_towers / PropagationNetwork(small_batches=True): inference with one CTA per tower.

A. fp64 parity.  Logits and probs against oracle.propnet.forward_sparse on the same fp32 inputs and weights, max|d| / max|ref|
   <= 1e-5 per batch, on C1 towers (7-block TowerCreator layouts, predict glue and contact edges), 10-block fully connected
   towers, a ragged batch of 0, 1, 2, 7, 13 and 32 blocks and one 32-block fully connected tower (in-degree 31), with Glorot
   weights, init_weights(nonzero_bias=True) after load_dict, and the weights after an adam_step.
B. Probabilities: test_gpu_inference.prob_check on the kernel's own logits, head bias spreading them over [-120, 120].
C. Batch invariance, bit for bit: every tower alone, first and last in a batch of 32, in a permuted batch, on a rerun.
D. The tiled path (Engine.forward) agrees within 2e-5 normwise on a 1000-tower C1 batch.
E. Facade: golden fixtures through predict; score_removals / score_drops sums bit-equal to sequential batch-1 predicts summed
   in float64 in block order, same argmin; batches outside the limits get the tiled path's bits; with the flag off a
   predict_towers call launches what it launched before.
F. One launch per call (none for an empty batch); write footprints between guard bands with 0x00 and 0xFF fills;
   isolation from a training step in flight; CUDA-graph capture and replay.

The worst ratio of A is written to $SPW_SMALL_OUT (default: small_parity.json in the temporary directory).
"""
import ctypes
import json
import os
import tempfile

import numpy as np
import pytest
import torch

from oracle import propnet as O

pytestmark = pytest.mark.gpu
SMALL_OUT = os.environ.get('SPW_SMALL_OUT', os.path.join(tempfile.gettempdir(), 'small_parity.json'))
TOL = 1e-5
_WORST = {}


@pytest.fixture(scope='module')
def eng():
    from spwgnn_b200.engine import Engine
    assert torch.cuda.is_available()
    e = Engine('cuda:0', seed=3)
    yield e
    if _WORST:
        try:
            with open(SMALL_OUT, 'w') as f:
                json.dump({'device': torch.cuda.get_device_name(0), 'max|d|/max|ref|': _WORST}, f, indent=1, sort_keys=True)
                f.write('\n')
        except OSError:
            pass


def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint64 if a.dtype == np.float64 else np.uint32)


def _rel(got, ref):
    ref = np.asarray(ref, dtype=np.float64)
    return float(np.abs(np.asarray(got, dtype=np.float64) - ref).max() / max(np.abs(ref).max(), 1e-30))


def _batch(kind, count=1, seed=0):
    from spwgnn_b200 import synth
    from spwgnn_b200.graph import TowerBatch
    if kind == 'C1':                        # latency_probe.py's shape: predict glue, every pair related
        towers = synth.make_towers('tower', count, 3 + seed, n=7)
        return TowerBatch.from_towers(towers, inference_glue=True), towers
    if kind == 'C1 contact':                # the same layouts, relations by the distance test on raw pixels
        towers = synth.make_towers('tower', count, 3 + seed, n=7)
        return TowerBatch.from_towers(towers), towers
    if kind == 'fc10':
        towers = synth.make_towers('jenga', count, 40 + seed, n=10)
        return TowerBatch.from_towers(towers, fully_connected=True), towers
    if kind == 'ragged':
        towers = []
        for i, nb in enumerate([0, 1, 2, 7, 13, 32]):
            towers += synth.make_towers('jenga', 1, 60 + seed + i, n=nb) if nb else [np.zeros((0, 3))]
        return TowerBatch.from_towers(towers, thr=330.0), towers
    if kind == 'fc32':
        towers = synth.make_towers('jenga', count, 70 + seed, n=32)
        return TowerBatch.from_towers(towers, fully_connected=True), towers
    raise ValueError(kind)


def _oracle(w64, batch):
    E = batch.n_edges
    snd = batch.in_snd[:E].long().cpu()
    rcv = batch.in_rcv[:E].long().cpu()
    o64 = batch.obj.double().cpu()
    p, z = O.forward_sparse(w64, o64, snd, rcv, return_logits=True)
    return z.numpy(), p.numpy()


def _weights64(eng):
    return {k: v.detach().double().cpu() for k, v in eng.params.to_dict().items()}


PARITY = ['C1', 'C1 contact', 'fc10', 'ragged', 'fc32']


def _parity(eng, label, fails):
    w64 = _weights64(eng)
    for kind in PARITY:
        batch, _ = _batch(kind, {'C1': 64, 'C1 contact': 64, 'fc10': 32, 'fc32': 1}.get(kind, 1))
        z, p = eng.forward_towers(batch)
        z64, p64 = _oracle(w64, batch)
        rz, rp = _rel(z.cpu().numpy(), z64), _rel(p.cpu().numpy(), p64)
        key = '%s / %s' % (kind, label)
        _WORST[key] = max(rz, rp)
        if not (rz <= TOL and rp <= TOL):
            fails.append('%s: logits %.3g, probs %.3g' % (key, rz, rp))


def test_fp64_parity(eng):
    from spwgnn_b200.params import ParamBuffer
    fails = []
    eng.params.load_dict(ParamBuffer('cpu').glorot_init(9).to_dict())
    _parity(eng, 'glorot', fails)
    eng.params.load_dict(O.init_weights(31, nonzero_bias=True))
    _parity(eng, 'init_weights nonzero_bias, load_dict', fails)
    batch, _ = _batch('C1 contact', 16, seed=5)
    tgt = torch.as_tensor((np.random.default_rng(1).random(batch.n_nodes) > 0.5).astype(np.float32)).cuda()
    eng.loss_and_grads(batch, tgt)
    eng.adam_step(lr=1e-2)
    _parity(eng, 'after adam_step', fails)
    eng._adam = None
    assert not fails, '\n'.join(fails)


def test_probabilities_elementwise(eng):
    import test_gpu_inference as I
    eng.params.load_dict(O.init_weights(32, nonzero_bias=True))
    batch, _ = _batch('C1 contact', 32)
    zs, ps = [], []
    for b in np.linspace(-120.0, 120.0, 97):
        eng.params.views['omp.b1'][0] = float(b)
        z, p = eng.forward_towers(batch)
        zs.append(z.clone())
        ps.append(p.clone())
    z, p = torch.cat(zs), torch.cat(ps)
    assert float(z.min()) < -100 and float(z.max()) > 100
    msgs, worst = I.prob_check(z, p)
    _WORST['probs: |p - sigma| / (6 u sigma)'] = worst
    assert not msgs, '\n'.join(msgs)


def test_batch_invariance_bit_for_bit(eng):
    from spwgnn_b200 import synth
    from spwgnn_b200.graph import TowerBatch
    eng.params.load_dict(O.init_weights(33, nonzero_bias=True))
    rng = np.random.default_rng(4)
    towers = [synth.make_towers('tower', 1, 100 + i, n=int(rng.integers(2, 11)))[0] for i in range(16)] + \
             [synth.make_towers('jenga', 1, 200 + i, n=int(rng.integers(1, 33)))[0] for i in range(16)]

    def run(ts):
        b = TowerBatch.from_towers(ts, thr=330.0)
        z, p = eng.forward_towers(b)
        off = b.node_off_host
        z, p = z.cpu().numpy(), p.cpu().numpy()
        return [(z[off[t]:off[t + 1]], p[off[t]:off[t + 1]]) for t in range(len(ts))]

    ref = run(towers)
    fails = []

    def same(a, b, what):
        if not (np.array_equal(_bits(a[0]), _bits(b[0])) and np.array_equal(_bits(a[1]), _bits(b[1]))):
            fails.append(what)

    for t, tw in enumerate(towers):
        same(run([tw])[0], ref[t], 'tower %d alone' % t)
        others = towers[:t] + towers[t + 1:]
        same(run([tw] + others)[0], ref[t], 'tower %d first' % t)
        same(run(others + [tw])[-1], ref[t], 'tower %d last' % t)
    perm = rng.permutation(len(towers))
    got = run([towers[i] for i in perm])
    for j, i in enumerate(perm):
        same(got[j], ref[i], 'tower %d permuted to %d' % (i, j))
    for t, r in enumerate(run(towers)):
        same(r, ref[t], 'tower %d rerun' % t)
    assert not fails, '\n'.join(fails)


def test_agrees_with_the_tiled_path(eng):
    eng.params.load_dict(O.init_weights(34, nonzero_bias=True))
    batch, _ = _batch('C1', 1000)
    z0, p0 = eng.forward(batch, training=False)
    z1, p1 = eng.forward_towers(batch)
    for a, b, what in ((z1, z0, 'logits'), (p1, p0, 'probs')):
        r = float((a.double() - b.double()).norm() / b.double().norm())
        _WORST['tiled vs small, 1000 C1 towers, normwise %s' % what] = r
        assert r <= 2e-5, (what, r)


def test_one_launch_per_call(eng):
    from spwgnn_b200.graph import TowerBatch
    api = eng.api
    for kind, count in (('C1', 1), ('C1', 32), ('fc10', 128), ('ragged', 1)):
        batch, _ = _batch(kind, count)
        before = api.dll.spw_launch_count()
        eng.forward_towers(batch)
        eng.forward_towers(batch, want_probs=False)
        assert api.dll.spw_launch_count() - before == 2, kind
    empty = TowerBatch.from_towers([])
    before = api.dll.spw_launch_count()
    z, p = eng.forward_towers(empty)
    assert api.dll.spw_launch_count() == before and z.numel() == 0 and p.numel() == 0
    big = TowerBatch.from_towers([np.zeros((33, 3))], fully_connected=True)
    from spwgnn_b200 import SpwError
    with pytest.raises(SpwError):
        eng.forward_towers(big)


def test_oversized_tower_gets_nan_rows(eng):
    """max_nodes_per_tower below a tower's size: that tower's rows are NaN, the others are computed"""
    api = eng.api
    batch, _ = _batch('ragged')
    off = batch.node_off_host
    n = batch.n_nodes
    ws = torch.empty(api.dll.spw_forward_towers_bytes(n, batch.n_edges) + 16, dtype=torch.uint8, device='cuda')
    z_ref, _ = eng.forward_towers(batch)
    z = torch.zeros(n, device='cuda')
    p = torch.zeros(n, device='cuda')
    wp = eng.params.c_struct()
    api.check(api.dll.spw_forward_towers(ctypes.byref(wp), ctypes.byref(batch.c_graph), 13, batch.obj.data_ptr(), z.data_ptr(),
                                         p.data_ptr(), ws.data_ptr(), ws.numel(), torch.cuda.current_stream().cuda_stream))
    big = slice(int(off[5]), int(off[6]))                     # the 32-block tower
    assert off[6] - off[5] == 32
    assert bool(torch.isnan(z[big]).all()) and bool(torch.isnan(p[big]).all())
    assert torch.equal(z[:big.start], z_ref[:big.start])


# ---- E. facade ---------------------------------------------------------------------------------------------------------------------
def _dense_dict(raw, n):
    boxes = (raw / 170.0)[None]
    rs, rr = O.build_relations_dense(boxes[:, :, :2], 170.0)
    return {'objects': boxes, 'sender_relations': rs, 'receiver_relations': rr, 'propagation': np.zeros((1, n, 100))}


def test_golden_fixtures_through_facade(golden_dir):
    from spwgnn_b200.Networks import PropagationNetwork
    wz = np.load(os.path.join(golden_dir, 'weights.npz'))
    pn = PropagationNetwork(small_batches=True)
    api = None
    for name in ['train_n2', 'train_n4', 'train_n7', 'train_n9', 'predict_jenga_n5', 'predict_jenga_n9']:
        g = np.load(os.path.join(golden_dir, name + '.npz'))
        model = pn.getModel(int(g['n_objects']), 3)
        model.set_weights_dict({k: wz[k] for k in wz.files})
        api = pn.engine.api
        x = {'objects': g['objects'], 'sender_relations': g['sender_relations'], 'receiver_relations': g['receiver_relations'],
             'propagation': np.zeros(g['objects'].shape[:2] + (100,))}
        before = api.dll.spw_launch_count()
        out = model.predict(x)
        assert out.shape == g['probs'].shape and out.dtype == np.float32
        assert _rel(out, g['probs']) < TOL, name
        if g['objects'].shape[0] <= pn.small_max_towers and g['objects'].shape[1] <= pn.small_max_nodes:
            assert api.dll.spw_launch_count() - before == 1, name      # the dense-dict batch is built with torch ops


def test_demolish_searches_equal_sequential_batch1_predicts():
    import test_gpu_inference as I
    from spwgnn_b200.Networks import PropagationNetwork
    from spwgnn_b200 import synth
    net = PropagationNetwork(device='cuda', seed=5, small_batches=True)
    tower = synth.make_towers('jenga', 1, 21, n=9)[0]
    N = len(tower)
    full, less = net.getModel(N), net.getModel(N - 1)
    net.engine.params.load_dict(O.init_weights(35, nonzero_bias=True))
    sums, idx = full.score_removals(tower)
    probs = np.concatenate([less.predict(_dense_dict(np.delete(tower, c, axis=0), N - 1)).reshape(-1) for c in range(N)])
    ref = I.tower_sums_reference(probs, np.arange(N + 1) * (N - 1))
    assert np.array_equal(_bits(sums), _bits(ref)), (sums, ref)
    assert idx == int(np.argmin(ref))
    base = synth.make_towers('tower', 1, 4, n=6)[0][1:]
    K = 100
    rng = np.random.default_rng(3)
    poses = np.stack([rng.random(K) * 700 + 400, rng.random(K) * 300 + 300], 1)
    m = net.getModel(len(base) + 1)                                   # candidate c: a block dropped at poses[c] on top of `base`
    sums, idx = m.score_drops(base, poses)
    probs = np.concatenate([m.predict(_dense_dict(np.concatenate([[[poses[c, 0], poses[c, 1], 150.0]], base]), len(base) + 1)).reshape(-1)
                            for c in range(K)])
    ref = I.tower_sums_reference(probs, np.arange(K + 1) * (len(base) + 1))
    assert np.array_equal(_bits(sums), _bits(ref))
    assert idx == int(np.argmin(ref))


def test_outside_the_limits_gives_the_tiled_bits():
    from spwgnn_b200.Networks import PropagationNetwork
    from spwgnn_b200 import synth
    on = PropagationNetwork(device='cuda', seed=6, small_batches=True)
    off = PropagationNetwork(device='cuda', seed=6)
    m_on, m_off = on.getModel(0), off.getModel(0)
    for towers in (synth.make_towers('tower', on.small_max_towers + 1, 7, n=7),          # too many towers
                   synth.make_towers('jenga', 3, 8, n=on.small_max_nodes + 1)):           # towers above the block limit
        a, b = m_on.predict_towers(towers), m_off.predict_towers(towers)
        assert all(np.array_equal(_bits(x), _bits(y)) for x, y in zip(a, b))
    # inside the limits the small path is taken: its bits differ from the tiled path's somewhere, but not by more than fp32
    towers = synth.make_towers('tower', 8, 9, n=7)
    a, b = np.concatenate(m_on.predict_towers(towers)), np.concatenate(m_off.predict_towers(towers))
    assert _rel(a, b) < 1e-5


def test_flag_off_launches_what_it_launched_before():
    from spwgnn_b200.Networks import PropagationNetwork
    from spwgnn_b200.graph import TowerBatch
    from spwgnn_b200 import synth
    net = PropagationNetwork(device='cuda', seed=7)
    model = net.getModel(7)
    eng, api = net.engine, net.engine.api
    for count in (1, 32, 300):
        towers = synth.make_towers('tower', count, 11, n=7)
        model.predict_towers(towers)                                  # capture graphs, set attributes
        before = api.dll.spw_launch_count()
        model.predict_towers(towers)
        facade = api.dll.spw_launch_count() - before
        before = api.dll.spw_launch_count()
        eng.forward(TowerBatch.from_towers(towers, inference_glue=True, device=eng.device), training=False)
        direct = api.dll.spw_launch_count() - before
        assert facade == direct, (count, facade, direct)


# ---- F. footprints, isolation, capture -----------------------------------------------------------------------------------------
@pytest.mark.parametrize('kind', ['C1', 'ragged', 'fc32'])
def test_write_footprint(eng, kind):
    import test_gpu_inference as I
    api = eng.api
    batch, _ = _batch(kind, 32 if kind == 'C1' else 1)
    n, E = batch.n_nodes, batch.n_edges
    eng.params.load_dict(O.init_weights(36, nonzero_bias=True))
    allocs = {'logits': I.Guarded('logits', 4 * n), 'probs': I.Guarded('probs', 4 * n),
              'workspace': I.Guarded('workspace', api.dll.spw_forward_towers_bytes(n, E))}
    inputs = {'weights': eng.params.flat, 'obj': batch.obj, 'node_off': batch.node_off, 'in_off': batch.in_off,
              'in_snd': batch.in_snd, 'in_rcv': batch.in_rcv}
    before = {k: v.clone() for k, v in inputs.items()}
    wp = eng.params.c_struct()
    st = torch.cuda.current_stream().cuda_stream
    runs, fails = [], []
    for want_probs in (True, False):
        snaps = []
        for fill in (0x00, 0xFF):
            for g in allocs.values():
                g.raw.fill_(fill)
            api.check(api.dll.spw_forward_towers(ctypes.byref(wp), ctypes.byref(batch.c_graph), int(batch.max_nodes),
                                                 batch.obj.data_ptr(), allocs['logits'].ptr,
                                                 allocs['probs'].ptr if want_probs else None, allocs['workspace'].ptr,
                                                 allocs['workspace'].nbytes, st))
            torch.cuda.synchronize()
            snaps.append({k: g.raw.clone() for k, g in allocs.items()})
        for k, g in allocs.items():
            fails += I.footprint_violations('%s (probs %s)' % (k, want_probs), [s[k] for s in snaps], [0x00, 0xFF], I.GUARD)
        for k in ('logits', 'probs'):
            p0, p1 = snaps[0][k][I.GUARD:I.GUARD + 4 * n], snaps[1][k][I.GUARD:I.GUARD + 4 * n]
            written = int(((p0 != 0x00) | (p1 != 0xFF)).sum())
            if k == 'probs' and not want_probs:
                if written:
                    fails.append('probs = NULL: %d bytes of the probs buffer written' % written)
                continue
            if not torch.equal(p0, p1):
                fails.append('%s differs between the 0x00 and the 0xFF run' % k)
            if written != 4 * n:
                fails.append('%s: %d of %d bytes written' % (k, written, 4 * n))
        runs.append(snaps[0]['logits'][I.GUARD:I.GUARD + 4 * n])
    if not torch.equal(runs[0], runs[1]):
        fails.append('logits differ with and without probs')
    for k, v in inputs.items():
        if not torch.equal(before[k], v):
            fails.append('input %s changed' % k)
    assert not fails, '\n'.join(fails)


def test_between_training_forward_and_backward(eng):
    eng.params.load_dict(O.init_weights(37, nonzero_bias=True))
    bx, _ = _batch('C1 contact', 40, seed=2)
    by, _ = _batch('fc10', 50, seed=3)
    tgt = torch.as_tensor((np.random.default_rng(5).random(bx.n_nodes) > 0.5).astype(np.float32)).cuda()

    def step(interleave):
        logits, _ = eng.forward(bx, training=True, want_probs=False, dropout_rate=0.1, dropout_seed=99)
        logits = logits.clone()
        if interleave:
            eng.forward_towers(by)
            eng.forward_towers(bx, want_probs=False)
        dl, _ = eng.bce_seed(logits, tgt, bx.n_nodes)
        eng.backward(dl)
        torch.cuda.synchronize()
        return logits, eng.grads.flat.clone()

    l0, g0 = step(False)
    l1, g1 = step(True)
    assert torch.equal(l0, l1) and torch.equal(g0, g1), int((g0 != g1).sum())


def test_cuda_graph_capture_replays_bit_identically(eng):
    api = eng.api
    eng.params.load_dict(O.init_weights(38, nonzero_bias=True))
    batch, _ = _batch('ragged')
    n = batch.n_nodes
    z_ref, p_ref = [t.clone() for t in eng.forward_towers(batch)]
    z = torch.full((n,), float('nan'), device='cuda')
    p = torch.full((n,), float('nan'), device='cuda')
    ws = torch.empty(api.dll.spw_forward_towers_bytes(n, batch.n_edges), dtype=torch.uint8, device='cuda')
    wp = eng.params.c_struct()
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g):
        api.check(api.dll.spw_forward_towers(ctypes.byref(wp), ctypes.byref(batch.c_graph), int(batch.max_nodes), batch.obj.data_ptr(),
                                             z.data_ptr(), p.data_ptr(), ws.data_ptr(), ws.numel(),
                                             torch.cuda.current_stream().cuda_stream))
    for _ in range(3):
        z.fill_(float('nan'))
        g.replay()
        torch.cuda.synchronize()
        assert torch.equal(z, z_ref) and torch.equal(p, p_ref)
