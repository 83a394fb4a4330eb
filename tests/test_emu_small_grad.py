"""spw_backward_towers (the backward pass of the one-CTA-per-tower path, k_tower_backward in spw_small_grad.cuh) under the host
emulator (tools/cuemu) against the fp64 references of the pose and relation gradients, and its host-side argument checks.
CPU only; tests/test_gpu_small_grad.py checks the real binary."""
import ctypes
import os

import numpy as np
import pytest
import torch

from oracle import propnet as O
from obj_grad_ref import obj_grads
from rel_grad_ref import rel_grads

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, 'spwgnn_b200', 'csrc')
GOLDEN = os.path.join(ROOT, 'tests', 'golden')
BAR = 1e-5


@pytest.fixture(scope='module')
def emu():
    import emu_harness
    from emu_harness import Emu, EMU_LIB, build_emu
    # the harness tracks the sources it knew of; the headers below are included by spwgnn.cu but not listed there
    srcs = [os.path.join(CSRC, f) for f in ('spw_small_grad.cuh', 'spw_small.cuh', 'spwgnn.cu')]
    if os.path.exists(EMU_LIB) and os.path.getmtime(EMU_LIB) < max(os.path.getmtime(s) for s in srcs):
        build_emu(force=True)
    assert emu_harness.EMU_LIB == EMU_LIB
    return Emu()


def _aligned(n, fill):
    buf = np.full(n + 8, fill, np.float32)
    off = (-buf.ctypes.data // 4) % 4
    return buf, buf[off:off + n]


def backward_towers(emu, w, g, obj, max_nodes, dlogits=None, dprobs=None, want_drel=True, want_logits=True, fill=np.nan):
    """spw_backward_towers on host arrays; returns (logits or None, dobj (n, 3), drel (E,) or None, launches)"""
    api = emu.api
    wl, wp, keep = emu.pack_params(w)
    obj = np.ascontiguousarray(obj, dtype=np.float32)
    nbytes = int(api.dll.spw_backward_towers_bytes(g.n, g.E))
    _, wsv = _aligned(nbytes // 4, fill)
    _, lv = _aligned(max(g.n, 1), fill)
    _, dv = _aligned(3 * max(g.n, 1), fill)
    _, rv = _aligned(max(g.E, 1), fill)
    dl = None if dlogits is None else np.ascontiguousarray(dlogits, np.float32)
    dp = None if dprobs is None else np.ascontiguousarray(dprobs, np.float32)
    before = api.dll.spw_launch_count()
    api.check(api.dll.spw_backward_towers(ctypes.byref(wp), ctypes.byref(g.c), int(max_nodes), obj.ctypes.data,
                                          None if dl is None else dl.ctypes.data, None if dp is None else dp.ctypes.data,
                                          lv.ctypes.data if want_logits else None, dv.ctypes.data,
                                          rv.ctypes.data if want_drel else None, wsv.ctypes.data, nbytes, None))
    launches = api.dll.spw_launch_count() - before
    return (lv[:g.n].copy() if want_logits else None, dv[:3 * g.n].reshape(g.n, 3).copy(),
            rv[:g.E].copy() if want_drel else None, launches)


class _Graph:
    pass


def graph_from_edges(emu, node_off, snd, rcv):
    """SpwGraph of the relations snd[k] -> rcv[k] (global block indices): receiver-major rows, out-CSR rows ascending"""
    node_off = np.ascontiguousarray(node_off, np.int32)
    n, E = int(node_off[-1]), len(snd)
    snd, rcv = np.asarray(snd, np.int64), np.asarray(rcv, np.int64)
    order = np.lexsort((snd, rcv))
    g = _Graph()
    g.T, g.n, g.E, g.node_off = len(node_off) - 1, n, E, node_off
    g.in_snd = np.zeros(max(E, 1), np.int32); g.in_snd[:E] = snd[order]
    g.in_rcv = np.zeros(max(E, 1), np.int32); g.in_rcv[:E] = rcv[order]
    g.in_off = np.searchsorted(g.in_rcv[:E], np.arange(n + 1)).astype(np.int32)
    o = np.lexsort((np.arange(E), g.in_snd[:E]))
    g.out_pos = np.zeros(max(E, 1), np.int32); g.out_pos[:E] = o
    g.out_off = np.searchsorted(g.in_snd[:E][o], np.arange(n + 1)).astype(np.int32)
    g.c = emu.api.graph(g.T, n, E, *[a.ctypes.data for a in (node_off, g.in_off, g.in_snd, g.in_rcv, g.out_off, g.out_pos)])
    return g


def _ragged(rng, sizes):
    node_off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)
    n = int(node_off[-1])
    pos = np.stack([rng.integers(300, 900, n).astype(np.float64), 110 + 80 * rng.integers(0, 5, n)], 1)
    wid = rng.integers(50, 300, n).astype(np.float64)
    return node_off, np.concatenate([pos, wid[:, None]], 1) / 170.0


def _contact_edges(obj, node_off, thr=330.0, fully_connected=False):
    _, snd, rcv, _ = O.edge_list(obj[:, :2] * 170.0, node_off, thr=thr, fully_connected=fully_connected)
    return np.asarray(snd), np.asarray(rcv)


def _golden(name):
    d = np.load(os.path.join(GOLDEN, name))
    obj = np.asarray(d['objects'][0], np.float64)
    rs, rr = np.asarray(d['sender_relations'][0]), np.asarray(d['receiver_relations'][0])
    act = (rs.sum(0) > 0) & (rr.sum(0) > 0)
    snd, rcv = rs.argmax(0)[act], rr.argmax(0)[act]
    return np.array([0, obj.shape[0]], np.int32), obj, snd, rcv


def reference(w64, obj, g, dlogits, dprobs):
    """fp64 (dobj, drel, logits) of sum(dlogits*z + dprobs*sigmoid(z)), relations in g's receiver-major order"""
    o64 = torch.as_tensor(np.asarray(obj, np.float32).astype(np.float64))
    snd, rcv = torch.as_tensor(g.in_snd[:g.E].astype(np.int64)), torch.as_tensor(g.in_rcv[:g.E].astype(np.int64))
    _, z = O.forward_sparse(w64, o64, snd, rcv, return_logits=True)
    p = torch.sigmoid(z)
    seed = torch.zeros_like(z)
    if dlogits is not None:
        seed += torch.as_tensor(np.asarray(dlogits, np.float32).astype(np.float64))
    if dprobs is not None:
        seed += torch.as_tensor(np.asarray(dprobs, np.float32).astype(np.float64)) * p * (1 - p)
    dobj, _, _ = obj_grads(w64, o64, snd, rcv, seed)
    drel, _, _ = rel_grads(w64, o64, snd, rcv, seed)
    return dobj.numpy(), drel.numpy(), z.numpy()


def colwise(got, ref):
    """max |delta| / max |ref| per column; an all-zero reference column must be matched exactly"""
    got, ref = np.atleast_2d(got.T).T, np.atleast_2d(ref.T).T
    out = []
    for c in range(ref.shape[1]):
        m = np.abs(ref[:, c]).max() if len(ref) else 0.0
        d = np.abs(got[:, c] - ref[:, c]).max() if len(ref) else 0.0
        out.append(d / m if m > 0 else (0.0 if d == 0 else np.inf))
    return max(out) if out else 0.0


def _case(emu, name, rng):
    if name.startswith('golden'):
        node_off, obj, snd, rcv = _golden('predict_jenga_n%s.npz' % name[-1])
        return node_off, obj, graph_from_edges(emu, node_off, snd, rcv)
    sizes, thr, fc = {'n1': ([1], 330.0, False), 'n2': ([2], 1e9, False), 'no_relations': ([3, 4], 0.0, False),
                      'fc32': ([32], 0.0, True), 'ragged': ([3, 0, 1, 2, 7, 13, 5], 330.0, False)}[name]
    node_off, obj = _ragged(rng, sizes)
    snd, rcv = _contact_edges(obj, node_off, thr, fc)
    return node_off, obj, graph_from_edges(emu, node_off, snd, rcv)


SEEDS = ('dlogits', 'dprobs', 'both')
CASES = [('golden5', 'both'), ('golden9', 'dprobs'), ('n1', 'both'), ('n2', 'dlogits'), ('n2', 'dprobs'), ('n2', 'both'),
         ('no_relations', 'dprobs'), ('fc32', 'both'), ('ragged', 'dlogits'), ('ragged', 'dprobs'), ('ragged', 'both')]


@pytest.mark.parametrize('case,seed', CASES)
def test_emu_backward_towers_matches_reference(emu, case, seed):
    """dobj and drel against the fp64 references (kink-free weights, bar 1e-5 of max |ref| per column), logits bit-equal to
    spw_forward_towers, one launch; the 32-block tower is fully connected (992 relations, in-degree 31, 31 chunks)."""
    from test_emu_small import forward_towers
    rng = np.random.default_rng(sum(map(ord, case)) + 3)
    node_off, obj, g = _case(emu, case, rng)
    if case == 'fc32':
        assert g.E == 32 * 31
    if case == 'no_relations':
        assert g.E == 0
    w64 = O.kinkfree_weights(5)
    wnp = {k: v.numpy() for k, v in w64.items()}
    dl = rng.standard_normal(g.n).astype(np.float32) if seed in ('dlogits', 'both') else None
    dp = rng.standard_normal(g.n).astype(np.float32) if seed in ('dprobs', 'both') else None
    mx = int(np.diff(node_off).max())
    logits, dobj, drel, launches = backward_towers(emu, wnp, g, obj, mx, dl, dp)
    assert launches == 1
    ref_dobj, ref_drel, _ = reference(w64, obj, g, dl, dp)
    assert np.isfinite(dobj).all() and np.isfinite(drel).all()
    assert colwise(dobj, ref_dobj) <= BAR, (case, seed, colwise(dobj, ref_dobj))
    bar_rel = BAR
    if case == 'fc32':
        # drel of a fully connected 32-block tower is small (max 2e-5) against its per-step terms, so the fp32 cancellation
        # approaches 1e-5 on the tiled path too: bound it by 4x that path's error on the same input and seed
        from test_emu_rel_grad import backward_rel
        p = 1.0 / (1.0 + np.exp(-logits.astype(np.float64)))
        s = np.zeros(g.n, np.float64) + (dl if dl is not None else 0) + (dp * (p * (1 - p)) if dp is not None else 0)
        emu.forward(wnp, g, obj, training=True)
        tiled, _, _ = backward_rel(emu, g, s.astype(np.float32))
        bar_rel = max(BAR, 4 * colwise(tiled, ref_drel))
    assert colwise(drel, ref_drel) <= bar_rel, (case, seed, colwise(drel, ref_drel), bar_rel)
    lf, _, _ = forward_towers(emu, wnp, g, obj, mx)
    assert np.array_equal(logits.view(np.uint32), lf.view(np.uint32))
    # without logits and drel: the same dobj bits
    l2, d2, r2, _ = backward_towers(emu, wnp, g, obj, mx, dl, dp, want_drel=False, want_logits=False, fill=0.0)
    assert l2 is None and r2 is None and np.array_equal(d2.view(np.uint32), dobj.view(np.uint32))


def test_emu_backward_towers_is_batch_invariant(emu):
    """Every tower of a ragged batch alone, with its own node capacity, and the batch rerun: the same bits."""
    rng = np.random.default_rng(21)
    node_off, obj, g = _case(emu, 'ragged', rng)
    wnp = {k: v.numpy() for k, v in O.init_weights(13, nonzero_bias=True).items()}
    dl, dp = rng.standard_normal(g.n).astype(np.float32), rng.standard_normal(g.n).astype(np.float32)
    logits, dobj, drel, _ = backward_towers(emu, wnp, g, obj, 32, dl, dp)
    for t in range(len(node_off) - 1):
        a, b = int(node_off[t]), int(node_off[t + 1])
        if a == b:
            continue
        ea, eb = int(g.in_off[a]), int(g.in_off[b])
        gt = graph_from_edges(emu, np.array([0, b - a], np.int32), g.in_snd[ea:eb] - a, g.in_rcv[ea:eb] - a)
        lt, dt, rt, _ = backward_towers(emu, wnp, gt, obj[a:b], b - a, dl[a:b], dp[a:b])
        assert np.array_equal(lt.view(np.uint32), logits[a:b].view(np.uint32)), t
        assert np.array_equal(dt.view(np.uint32), dobj[a:b].view(np.uint32)), t
        assert np.array_equal(rt.view(np.uint32), drel[ea:eb].view(np.uint32)), t
    l2, d2, r2, _ = backward_towers(emu, wnp, g, obj, 32, dl, dp, fill=0.0)
    for x, y in ((l2, logits), (d2, dobj), (r2, drel)):
        assert np.array_equal(x.view(np.uint32), y.view(np.uint32))


def test_emu_backward_towers_oversized_and_malformed(emu):
    """A tower larger than max_nodes_per_tower gets NaN logits, dobj rows and drel of its relations, and its neighbours keep
    their bits; a relation between two towers gives both of them NaN logits and dobj rows, and the tower between keeps its
    values."""
    rng = np.random.default_rng(22)
    node_off, obj = _ragged(rng, [4, 9, 5])
    snd, rcv = _contact_edges(obj, node_off, 1e9)
    g = graph_from_edges(emu, node_off, snd, rcv)
    wnp = {k: v.numpy() for k, v in O.kinkfree_weights(6).items()}
    dl = rng.standard_normal(g.n).astype(np.float32)
    logits, dobj, drel, _ = backward_towers(emu, wnp, g, obj, 8, dl, None, fill=0.0)
    e4, e13 = int(g.in_off[4]), int(g.in_off[13])
    assert np.isnan(logits[4:13]).all() and np.isnan(dobj[4:13]).all() and np.isnan(drel[e4:e13]).all()
    fl, fd, fr, _ = backward_towers(emu, wnp, g, obj, 9, dl, None)
    for x, y in ((logits, fl), (dobj, fd)):
        assert np.array_equal(x[:4].view(np.uint32), y[:4].view(np.uint32))
        assert np.array_equal(x[13:].view(np.uint32), y[13:].view(np.uint32))
    assert np.array_equal(drel[:e4].view(np.uint32), fr[:e4].view(np.uint32))
    assert np.array_equal(drel[e13:].view(np.uint32), fr[e13:].view(np.uint32))
    # a relation of tower 2 whose sender lies in tower 0
    bad_snd = g.in_snd[:g.E].copy()
    k = int(g.in_off[13])
    bad_snd[k] = 0
    gb = graph_from_edges(emu, node_off, bad_snd, g.in_rcv[:g.E])
    lb, db, _, _ = backward_towers(emu, wnp, gb, obj, 9, dl, None, fill=0.0)
    for a, b in ((0, 4), (13, 18)):
        assert np.isnan(lb[a:b]).all() and np.isnan(db[a:b]).all()
    assert np.array_equal(lb[4:13].view(np.uint32), fl[4:13].view(np.uint32))
    assert np.array_equal(db[4:13].view(np.uint32), fd[4:13].view(np.uint32))


def test_backward_towers_host_side_argument_checks():
    """Host-side errors on the sm_100a library, without a GPU: a tower limit above SPW_SMALL_MAX_NODES, a null obj or dobj,
    two null seeds, a misaligned dobj, a short workspace, a misaligned weight.  An empty batch launches nothing."""
    from spwgnn_b200 import build
    from spwgnn_b200._capi import CApi, SpwGraph
    api = CApi(build.build())
    p = CApi.params([16 * (i + 1) for i in range(22)])
    g = SpwGraph(1, 4, 12, 16, 16, 16, 16, 16, 16)                       # non-null, aligned fake device pointers
    f = api.dll.spw_backward_towers
    need = api.dll.spw_backward_towers_bytes(4, 12)
    assert need == (2 * 12 * 152 + 4 * 2820) * 4 and api.dll.spw_backward_towers_bytes(-1, 0) == 0
    big = 1 << 40
    rc = f(ctypes.byref(p), ctypes.byref(g), 33, 16, 16, None, None, 16, 16, 16, big, None)
    assert rc == -2 and b'limit' in api.dll.spw_last_error()
    rc = f(ctypes.byref(p), ctypes.byref(g), -1, 16, 16, None, None, 16, 16, 16, big, None)
    assert rc == -1 and b'max_nodes' in api.dll.spw_last_error()
    rc = f(ctypes.byref(p), ctypes.byref(g), 4, None, 16, None, None, 16, 16, 16, big, None)
    assert rc == -1 and b'null' in api.dll.spw_last_error()
    rc = f(ctypes.byref(p), ctypes.byref(g), 4, 16, 16, None, None, None, 16, 16, big, None)
    assert rc == -1 and b'null' in api.dll.spw_last_error()
    rc = f(ctypes.byref(p), ctypes.byref(g), 4, 16, None, None, None, 16, 16, 16, big, None)
    assert rc == -1 and b'seed' in api.dll.spw_last_error()
    rc = f(ctypes.byref(p), ctypes.byref(g), 4, 16, None, 16, None, 20, 16, 16, big, None)
    assert rc == -1 and b'aligned' in api.dll.spw_last_error()
    rc = f(ctypes.byref(p), ctypes.byref(g), 4, 16, 16, 16, 16, 16, 16, 16, need - 1, None)
    assert rc == -3 and b'workspace' in api.dll.spw_last_error()
    rc = f(ctypes.byref(p), ctypes.byref(g), 4, 16, 16, 16, 16, 16, 16, 24, need, None)
    assert rc == -1 and b'workspace' in api.dll.spw_last_error()
    p.p[3] = 20                                                          # a misaligned weight tensor
    rc = f(ctypes.byref(p), ctypes.byref(g), 4, 16, 16, None, None, 16, 16, 16, big, None)
    assert rc == -1 and b'tensor 3' in api.dll.spw_last_error()
    p.p[3] = 64
    before = api.dll.spw_launch_count()
    empty = SpwGraph(0, 0, 0, None, None, None, None, None, None)
    assert f(ctypes.byref(p), ctypes.byref(empty), 4, None, None, None, None, None, None, None, 0, None) == 0
    assert api.dll.spw_launch_count() == before
