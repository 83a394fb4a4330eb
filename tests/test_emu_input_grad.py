"""spw_backward_inputs (the gradients with respect to the dense relation tensors, the propagation input and the objects;
spw_input_grad.cuh) under the host emulator (tools/cuemu) against the fp64 reference, its host-side argument checks, and the
reference itself: input_grad_ref.input_grads equals autograd of oracle.propnet.forward_dense with respect to all four inputs
(objects, sender_relations, receiver_relations, propagation) on the reference's own dicts, and central differences.  CPU only;
tests/test_gpu_input_grad.py checks the real binary."""
import ctypes
import os

import numpy as np
import pytest
import torch

from oracle import propnet as O
from input_grad_ref import input_grads
from test_emu_obj_grad import _ragged, backward_obj, dropout_scales

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, 'spwgnn_b200', 'csrc')
GOLDEN = os.path.join(ROOT, 'tests', 'golden')


@pytest.fixture(scope='module')
def emu():
    import emu_harness
    from emu_harness import Emu, EMU_LIB, build_emu
    # the harness tracks the sources it knew of; the headers below are included by spwgnn.cu but not listed there
    srcs = [os.path.join(CSRC, f) for f in ('spw_input_grad.cuh', 'spw_rel_grad.cuh', 'spw_obj_grad.cuh', 'spw_small.cuh',
                                            'spw_kernels.cuh', 'spwgnn.cu')]
    if os.path.exists(EMU_LIB) and os.path.getmtime(EMU_LIB) < max(os.path.getmtime(s) for s in srcs):
        build_emu(force=True)
    assert emu_harness.EMU_LIB == EMU_LIB
    return Emu()


def _aligned(count, fill=np.nan):
    buf = np.full(count + 8, fill, np.float32)
    off = (-buf.ctypes.data // 4) % 4
    return buf[off:off + count]


def backward_inputs(emu, g, dlogits, max_nodes, with_dobj=True):
    """spw_backward_inputs on the state of the last emu.forward(training=True); every output is NaN-filled first.
    Returns (drs (E, max_nodes), drr, drr_free (n,), dprop (n, 100), dobj (n, 3) or None, launches)."""
    api = emu.api
    wl, wp, keep, obj, ws, wsv, nbytes = emu._state
    dl = np.ascontiguousarray(dlogits, np.float32)
    E, n = g.E, g.n
    drs, drr = _aligned(max(E * max_nodes, 1)), _aligned(max(E * max_nodes, 1))
    free, dprop, dobj = _aligned(max(n, 1)), _aligned(100 * max(n, 1)), _aligned(3 * max(n, 1))
    sb = api.dll.spw_backward_inputs_bytes(n, E)
    scratch = _aligned(sb // 4 + 1)
    before = api.dll.spw_launch_count()
    api.check(api.dll.spw_backward_inputs(ctypes.byref(wp), ctypes.byref(g.c), max_nodes, obj.ctypes.data, dl.ctypes.data,
                                          wsv.ctypes.data, nbytes, emu._rate, scratch.ctypes.data, sb,
                                          drs.ctypes.data if E else None, drr.ctypes.data if E else None, free.ctypes.data,
                                          dprop.ctypes.data, dobj.ctypes.data if with_dobj else None, None))
    launches = api.dll.spw_launch_count() - before
    return (drs[:E * max_nodes].reshape(E, max_nodes).copy(), drr[:E * max_nodes].reshape(E, max_nodes).copy(), free[:n].copy(),
            dprop[:100 * n].reshape(n, 100).copy(), dobj[:3 * n].reshape(n, 3).copy() if with_dobj else None, launches)


def normwise(got, ref):
    """max |delta| / max |ref|; an all-zero reference must be matched exactly"""
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    if ref.size == 0:
        return 0.0
    m, d = np.abs(ref).max(), np.abs(got - ref).max()
    return float(d / m) if m > 0 else (0.0 if d == 0 else np.inf)


# ---- the reference --------------------------------------------------------------------------------------------------------------
def dense_edges(rs, rr):
    """active columns of dense (B, N, R) one-hots -> (snd, rcv, batch, slot), global block ids, slot order"""
    B, N, _ = rs.shape
    bi, ri = np.nonzero((rs != 0).any(1) | (rr != 0).any(1))
    return rs[bi, :, ri].argmax(1) + bi * N, rr[bi, :, ri].argmax(1) + bi * N, bi, ri


def dense_grads(w, objects, rs, rr, dl):
    """autograd of oracle.propnet.forward_dense with respect to (objects, sender_relations, receiver_relations, propagation)"""
    B, N, _ = objects.shape
    ins = [torch.as_tensor(a, dtype=torch.float64).clone().requires_grad_(True)
           for a in (objects, rs, rr, np.zeros((B, N, O.PROP_DIM)))]
    _, z = O.forward_dense(w, *ins, return_logits=True)
    return [g.numpy() for g in torch.autograd.grad((z.reshape(B, N) * torch.as_tensor(dl)).sum(), ins)]


def compact_to_dense(drs, drr, free, snd, rcv, bi, ri, B, N, R):
    """the compact rows scattered into (B, N, R) as PropagationModel.input_gradients does: inactive columns get 0 / drr_free"""
    Drs = np.zeros((B, N, R)); Drr = np.repeat(np.asarray(free).reshape(B, N)[:, :, None], R, 2)
    Drs[bi, :, ri] = np.asarray(drs)[:, :N]
    Drr[bi, :, ri] = np.asarray(drr)[:, :N]
    return Drs, Drr


def _dicts():
    out = {}
    for name in ('predict_jenga_n5', 'predict_jenga_n9', 'train_n2', 'train_n4', 'train_n7', 'train_n9'):
        d = np.load(os.path.join(GOLDEN, name + '.npz'))
        out[name] = (d['objects'], d['sender_relations'], d['receiver_relations'])
    d = np.load(os.path.join(GOLDEN, 'train_n4.npz'))
    B, N, R = d['sender_relations'].shape
    out['relation_free'] = (d['objects'], np.zeros((B, N, R)), np.zeros((B, N, R)))
    # active columns moved off the leading slots: the slots of each tower are permuted
    perm = np.random.default_rng(3).permutation(R)
    out['permuted_slots'] = (d['objects'], d['sender_relations'][:, :, perm], d['receiver_relations'][:, :, perm])
    return out


DICTS = _dicts()


@pytest.mark.parametrize('name', sorted(DICTS))
def test_reference_equals_dense_autograd(name):
    """input_grads, scattered into the dense shapes, equals autograd of oracle.propnet.forward_dense with respect to all four
    inputs to 1e-12 of each tensor's largest value (at the inactive slots too)."""
    objects, rs, rr = DICTS[name]
    B, N, R = rs.shape
    w = O.init_weights(7, nonzero_bias=True)
    dl = np.random.default_rng(B * N + R).standard_normal(B * N)
    snd, rcv, bi, ri = dense_edges(rs, rr)
    drs, drr, free, dprop, dobj, _, _ = input_grads(w, torch.as_tensor(objects.reshape(B * N, 3), dtype=torch.float64),
                                                 np.arange(B + 1) * N, snd, rcv, dl)
    refs = dense_grads(w, objects, rs, rr, dl.reshape(B, N))
    Drs, Drr = compact_to_dense(drs.numpy(), drr.numpy(), free.numpy(), snd, rcv, bi, ri, B, N, R)
    for got, ref in ((dobj.numpy().reshape(B, N, 3), refs[0]), (Drs, refs[1]), (Drr, refs[2]),
                     (dprop.numpy().reshape(B, N, 100), refs[3])):
        assert normwise(got, ref) <= 1e-12
    if name == 'relation_free':
        assert not Drs.any() and np.abs(Drr).max() > 0


def test_reference_matches_central_differences():
    """Every input of a 4-block tower with three active relations, differentiated by fp64 central differences of
    oracle.propnet.forward_dense (kink-free weights at full Glorot scale, every relu unit further from its kink than 100
    steps): the active and inactive slots of both relation tensors, propagation and objects."""
    rng = np.random.default_rng(11)
    N, R = 4, 12
    objects = np.stack([rng.uniform(2, 5, N), rng.uniform(0.6, 3, N), rng.uniform(0.3, 1.7, N)], 1)[None]
    rs, rr = np.zeros((1, N, R)), np.zeros((1, N, R))
    for slot, (s, r) in zip((0, 4, 9), ((0, 1), (1, 2), (3, 0))):
        rs[0, s, slot] = rr[0, r, slot] = 1.0
    w = O.kinkfree_weights(7, scale=1.0)
    snd, rcv, bi, ri = dense_edges(rs, rr)
    assert O.min_relu_margin(w, torch.as_tensor(objects[0]), torch.as_tensor(snd), torch.as_tensor(rcv)) > 100 * 1e-6
    dl = rng.standard_normal(N)
    drs, drr, free, dprop, dobj, _, _ = input_grads(w, torch.as_tensor(objects[0]), [0, N], snd, rcv, dl)
    Drs, Drr = compact_to_dense(drs.numpy(), drr.numpy(), free.numpy(), snd, rcv, bi, ri, 1, N, R)
    got = [dobj.numpy()[None], Drs, Drr, dprop.numpy()[None]]
    base = [objects, rs, rr, np.zeros((1, N, O.PROP_DIM))]

    def f(vals):
        _, z = O.forward_dense(w, *[torch.as_tensor(v) for v in vals], return_logits=True)
        return float((z.reshape(-1) * torch.as_tensor(dl)).sum())
    h = 1e-6
    for k, idxs in ((0, [(0, 1, 0), (0, 2, 2)]), (1, [(0, 0, 0), (0, 2, 0), (0, 3, 5)]), (2, [(0, 1, 0), (0, 3, 0), (0, 2, 7)]),
                    (3, [(0, 0, 3), (0, 2, 50)])):
        for idx in idxs:
            vals = []
            for sgn in (1, -1):
                v = [b.copy() for b in base]
                v[k][idx] += sgn * h
                vals.append(f(v))
            fd = (vals[0] - vals[1]) / (2 * h)
            assert abs(got[k][idx] - fd) <= 1e-6 * max(1.0, abs(fd)), (k, idx, got[k][idx], fd)


def test_reference_on_a_given_relu_branch(monkeypatch):
    """With the relu states of the oracle's own sparse forward (recorded at O._relu), input_grads forced onto that branch is
    input_grads unforced, to 1e-12, with no unit flipped: the padding of the per-tower restatement takes its states right."""
    rng = np.random.default_rng(1)
    node_off, pos, wid = _ragged(rng, [5, 0, 4, 1])
    eo, snd, rcv, slot = O.edge_list(pos, node_off, thr=330.0)
    o = np.argsort(rcv, kind='stable')                               # receiver-major, as the saved states are
    snd, rcv = snd[o], rcv[o]
    obj = torch.as_tensor(np.concatenate([pos, wid[:, None]], 1) / 170.0)
    w = O.init_weights(2, nonzero_bias=True)
    rec = []
    with monkeypatch.context() as m:
        m.setattr(O, '_relu', lambda x: (rec.append(x.detach() > 0), torch.relu(x))[1])
        O.forward_sparse(w, obj, torch.as_tensor(snd), torch.as_tensor(rcv))
    assert len(rec) == 21
    dl = rng.standard_normal(len(obj))
    free = input_grads(w, obj, node_off, snd, rcv, dl)
    forced = input_grads(w, obj, node_off, snd, rcv, dl, masks=rec)
    assert sum(f[0] for f in forced[6]) == 0
    for a, b in zip(free[:5], forced[:5]):
        assert normwise(b.numpy(), a.numpy()) <= 1e-12


# ---- the FFMA kernels under the emulator ---------------------------------------------------------------------------------------
CASES = {
    # name: (tower sizes, threshold, fully connected)
    'two_relations': ([2], 1e9, False),
    'c1_tower_7': ([7], 330.0, False),
    'fully_connected_5x2': ([5, 5], 0.0, True),
    'ragged_0_1_2_7': ([0, 1, 2, 7], 330.0, False),
    'no_relations': ([3, 4], 0.0, False),
    'tower_64': ([64, 3], 200.0, False),
}


@pytest.mark.parametrize('rate', [0.0, 0.1])
@pytest.mark.parametrize('case', sorted(CASES))
def test_emu_input_grad_matches_reference(emu, case, rate):
    sizes, thr, fc = CASES[case]
    rng = np.random.default_rng(sum(map(ord, case)) + 2)
    node_off, pos, wid = _ragged(rng, sizes)
    g = emu.edges(pos, node_off, thr=thr, fully_connected=fc)
    if case == 'no_relations':
        assert g.E == 0
    obj = np.concatenate([pos, wid[:, None]], 1) / 170.0
    w64 = O.kinkfree_weights(3)
    wnp = {k: v.numpy() for k, v in w64.items()}
    seed = 0x13579BDF2468ACE0
    emu.forward(wnp, g, obj, training=True, dropout_rate=rate, dropout_seed=seed)
    dl = rng.standard_normal(g.n).astype(np.float32)
    dobj_ref, _ = backward_obj(emu, g, dl)
    cs, qs = (None, None)
    if rate > 0:   # the reference on the receiver-major relation list: row k's dropout elements are k * 160 + c
        g_rm = type('G', (), {'out_pos': np.arange(g.E, dtype=np.int64), 'n': g.n})
        cs, qs = dropout_scales(g_rm, seed, rate)
    o64 = torch.as_tensor(obj.astype(np.float32).astype(np.float64))
    ref = input_grads(w64, o64, node_off, g.in_snd, g.in_rcv, dl.astype(np.float64), c_scale=cs, q_scale=qs)
    max_n = min(max(sizes) + 2, 64)                              # rows wider than the largest tower: the tail is written as 0
    drs, drr, free, dprop, dobj, launches = backward_inputs(emu, g, dl, max_n)
    for got in (drs, drr, free, dprop):
        assert np.isfinite(got).all()
    Nm = ref[0].shape[1]
    assert not drs[:, Nm:].any() and not drr[:, Nm:].any()
    for k, got in enumerate((drs[:, :Nm], drr[:, :Nm], free, dprop)):
        r = normwise(got, ref[k].numpy())
        assert r <= 1e-5, (case, rate, k, r)
    assert np.array_equal(dobj.view(np.uint32), dobj_ref.view(np.uint32))
    # rerun, and without dobj: the same bits
    again = backward_inputs(emu, g, dl, max_n, with_dobj=False)
    for a, b in zip(again[:4], (drs, drr, free, dprop)):
        assert np.array_equal(a.view(np.uint32), b.view(np.uint32))


def test_emu_input_grad_leaves_weight_gradients_alone(emu):
    """A backward_inputs between the forward and spw_backward: the weight gradients are the same bits as without it."""
    rng = np.random.default_rng(6)
    node_off, pos, wid = _ragged(rng, [5, 6])
    g = emu.edges(pos, node_off, thr=330.0)
    obj = np.concatenate([pos, wid[:, None]], 1) / 170.0
    wnp = {k: v.numpy() for k, v in O.kinkfree_weights(4).items()}
    dl = rng.standard_normal(g.n).astype(np.float32)
    emu.forward(wnp, g, obj, training=True)
    g0 = emu.backward(g, dl)
    emu.forward(wnp, g, obj, training=True)
    backward_inputs(emu, g, dl, 6)
    g1 = emu.backward(g, dl)
    for k in g0:
        assert np.array_equal(g0[k].view(np.uint32), g1[k].view(np.uint32)), k


def test_emu_input_grad_tower_beyond_declared_size_is_nan(emu):
    """A tower larger than max_nodes_per_tower gets NaN in its rows and its drr_free, and the other towers are unaffected."""
    rng = np.random.default_rng(8)
    node_off, pos, wid = _ragged(rng, [4, 7])
    g = emu.edges(pos, node_off, thr=330.0)
    obj = np.concatenate([pos, wid[:, None]], 1) / 170.0
    wnp = {k: v.numpy() for k, v in O.kinkfree_weights(4).items()}
    dl = rng.standard_normal(g.n).astype(np.float32)
    emu.forward(wnp, g, obj, training=True)
    full = backward_inputs(emu, g, dl, 7)
    small = backward_inputs(emu, g, dl, 4)
    big = np.arange(g.E) >= g.in_off[4]                           # receiver-major rows of the second tower
    assert np.isnan(small[0][big]).all() and np.isnan(small[1][big]).all() and np.isnan(small[2][4:]).all()
    assert np.array_equal(small[0][~big], full[0][~big, :4]) and np.array_equal(small[2][:4], full[2][:4])


def test_backward_inputs_host_side_argument_checks():
    """Host-side errors on the sm_100a library, without a GPU: null outputs, a misaligned output, scratch or workspace, a bad
    rate or tower size, a scratch that is too small, a misaligned weight.  An empty batch launches nothing, and a batch without
    relations accepts null drs / drr."""
    from spwgnn_b200 import build
    from spwgnn_b200._capi import CApi, SpwGraph
    api = CApi(build.build())
    p = CApi.params([16 * (i + 1) for i in range(22)])
    g = SpwGraph(1, 4, 12, 16, 16, 16, 16, 16, 16)                       # non-null, aligned fake device pointers
    big = 1 << 40
    f = api.dll.spw_backward_inputs

    def call(mx=4, obj=16, ws=16, rate=0.0, sc=16, sb=big, drs=16, drr=16, free=16, dprop=16, dobj=None, graph=g):
        return f(ctypes.byref(p), ctypes.byref(graph), mx, obj, 16, ws, big, rate, sc, sb, drs, drr, free, dprop, dobj, None)
    err = lambda: api.dll.spw_last_error()
    assert call(drs=None) == -1 and b'null' in err()
    assert call(free=None) == -1 and b'null' in err()
    assert call(obj=None) == -1 and b'null' in err()
    assert call(drr=18) == -1 and b'aligned' in err()
    assert call(dprop=20) == -1 and b'dprop' in err()
    assert call(dobj=20) == -1 and b'dobj' in err()
    assert call(ws=24) == -1 and b'workspace' in err()
    assert call(sc=24) == -1 and b'scratch' in err()
    assert call(sc=None) == -1 and b'scratch' in err()
    for mx in (-1, 65):
        assert call(mx=mx) == -1 and b'max_nodes_per_tower' in err()
    for rate in (-0.1, 1.0):
        assert call(rate=rate) == -1 and b'rate' in err()
    need = api.dll.spw_backward_inputs_bytes(4, 12)
    assert need > 0 and api.dll.spw_backward_inputs_bytes(-1, 0) == 0
    assert call(sb=need - 1) == -3 and b'scratch' in err()
    p.p[3] = 20                                                          # a misaligned weight tensor
    assert call() == -1 and b'tensor 3' in err()
    p.p[3] = 64
    before = api.dll.spw_launch_count()
    empty = SpwGraph(0, 0, 0, None, None, None, None, None, None)
    assert f(ctypes.byref(p), ctypes.byref(empty), 0, None, None, None, 0, 0.0, None, 0, None, None, None, None, None, None) == 0
    assert api.dll.spw_launch_count() == before
