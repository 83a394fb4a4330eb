"""spw_backward_rel (the gradient with respect to the relation weights, k_rel_grad_step / k_rel_grad_enc in spw_rel_grad.cuh)
under the host emulator (tools/cuemu) against the fp64 reference, its host-side argument checks, and the reference itself:
rel_grad_ref.forward_weighted is oracle.propnet.forward_sparse bit for bit without weights, and rel_grads equals the Keras
gradients with respect to the two nonzero entries of each relation column (autograd of oracle.propnet.forward_dense) and
central differences.  CPU only; tests/test_gpu_rel_grad.py checks the real binary."""
import ctypes
import os

import numpy as np
import pytest
import torch

from oracle import propnet as O
from rel_grad_ref import forward_weighted, rel_grads
from test_emu_obj_grad import _ragged, backward_obj, dropout_scales

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, 'spwgnn_b200', 'csrc')


@pytest.fixture(scope='module')
def emu():
    import emu_harness
    from emu_harness import Emu, EMU_LIB, build_emu
    # the harness tracks the sources it knew of; the headers below are included by spwgnn.cu but not listed there
    srcs = [os.path.join(CSRC, f) for f in ('spw_rel_grad.cuh', 'spw_obj_grad.cuh', 'spw_small.cuh', 'spw_kernels.cuh', 'spwgnn.cu')]
    if os.path.exists(EMU_LIB) and os.path.getmtime(EMU_LIB) < max(os.path.getmtime(s) for s in srcs):
        build_emu(force=True)
    assert emu_harness.EMU_LIB == EMU_LIB
    return Emu()


def backward_rel(emu, g, dlogits, with_dobj=True):
    """spw_backward_rel on the state of the last emu.forward(training=True); drel and dobj are NaN-filled.
    Returns (drel (E,), dobj (n, 3) or None, launches)."""
    api = emu.api
    wl, wp, keep, obj, ws, wsv, nbytes = emu._state
    dl = np.ascontiguousarray(dlogits, np.float32)
    drel = np.full(max(g.E, 1), np.nan, np.float32)
    buf = np.full(3 * max(g.n, 1) + 8, np.nan, np.float32)
    off = (-buf.ctypes.data // 4) % 4
    dobj = buf[off:off + 3 * max(g.n, 1)]
    before = api.dll.spw_launch_count()
    api.check(api.dll.spw_backward_rel(ctypes.byref(wp), ctypes.byref(g.c), obj.ctypes.data, dl.ctypes.data, wsv.ctypes.data,
                                       nbytes, emu._rate, drel.ctypes.data if g.E else None,
                                       dobj.ctypes.data if with_dobj else None, None))
    launches = api.dll.spw_launch_count() - before
    return drel[:g.E].copy(), dobj[:3 * g.n].reshape(g.n, 3).copy() if with_dobj else None, launches


def normwise(got, ref):
    """max |delta| / max |ref|; an all-zero reference must be matched exactly"""
    if len(ref) == 0:
        return 0.0
    m, d = np.abs(ref).max(), np.abs(got - ref).max()
    return float(d / m) if m > 0 else (0.0 if d == 0 else np.inf)


# ---- the reference --------------------------------------------------------------------------------------------------------------
def _graph(seed, B, N, thr):
    rng = np.random.default_rng(seed)
    node_off = np.arange(B + 1) * N
    pos = np.stack([rng.integers(300, 900, B * N).astype(np.float64), 110 + 80 * rng.integers(0, 5, B * N)], 1)
    wid = rng.integers(50, 300, B * N).astype(np.float64)
    eo, snd, rcv, slot = O.edge_list(pos, node_off, thr=thr)
    obj = torch.as_tensor(np.concatenate([pos, wid[:, None]], 1) / 170.0)
    return rng, node_off, obj, eo, snd, rcv, slot


def test_weighted_forward_is_the_oracle():
    """Without weights (and with all weights 1) forward_weighted gives oracle.propnet.forward_sparse's logits bit for bit."""
    _, _, obj, _, snd, rcv, _ = _graph(1, 3, 6, 330.0)
    snd, rcv = torch.as_tensor(snd), torch.as_tensor(rcv)
    w = O.init_weights(2, nonzero_bias=True)
    _, ref = O.forward_sparse(w, obj, snd, rcv, return_logits=True)
    for scale in (None, torch.ones(len(snd), dtype=torch.float64)):
        _, z = forward_weighted(w, obj, snd, rcv, scale)
        assert torch.equal(z, ref)


@pytest.mark.parametrize('B,N,thr', [(2, 4, 1e9), (3, 5, 330.0), (2, 6, 250.0)])
def test_rel_grads_equal_the_dense_gradients(B, N, thr):
    """rel_grads[e] = dRs[s, e] + dRr[r, e] from autograd of oracle.propnet.forward_dense (the reference graph line by line)
    with the relation tensors as inputs, to 1e-12 of the largest value."""
    rng, node_off, obj, eo, snd, rcv, slot = _graph(10 * B + N, B, N, thr)
    assert len(snd) > 0
    w = O.init_weights(5, nonzero_bias=True)
    dl = rng.standard_normal(B * N)
    got, _, _ = rel_grads(w, obj, torch.as_tensor(snd), torch.as_tensor(rcv), torch.as_tensor(dl))
    rs, rr = O.relations_from_edges(N, eo, snd, rcv, slot, node_off)
    rs = torch.as_tensor(rs).requires_grad_(True)
    rr = torch.as_tensor(rr).requires_grad_(True)
    _, z = O.forward_dense(w, obj.reshape(B, N, 3), rs, rr, return_logits=True)
    drs, drr = torch.autograd.grad((z.reshape(-1) * torch.as_tensor(dl)).sum(), [rs, rr])
    t = np.repeat(np.arange(B), np.diff(eo))
    ref = drs[t, snd - node_off[t], slot] + drr[t, rcv - node_off[t], slot]
    assert float((got - ref).abs().max()) <= 1e-12 * float(ref.abs().max())


def test_rel_grads_match_central_differences():
    """rel_grads against fp64 central differences of sum dlogits*logits in every relation weight, on a fully connected
    4-block tower with kink-free weights at full Glorot scale (every relu unit further from its kink than 100 steps)."""
    rng, node_off, obj, eo, snd, rcv, slot = _graph(9, 1, 4, 1e9)
    snd, rcv = torch.as_tensor(snd), torch.as_tensor(rcv)
    w = O.kinkfree_weights(3, scale=1.0)
    h = 1e-6
    assert O.min_relu_margin(w, obj, snd, rcv) > 100 * h
    dl = torch.as_tensor(rng.standard_normal(4))
    got, _, _ = rel_grads(w, obj, snd, rcv, dl)
    E = len(snd)
    fd = torch.zeros(E, dtype=torch.float64)
    for e in range(E):
        vals = []
        for sgn in (1, -1):
            sc = torch.ones(E, dtype=torch.float64)
            sc[e] += sgn * h
            vals.append(float((forward_weighted(w, obj, snd, rcv, sc)[1] * dl).sum()))
        fd[e] = (vals[0] - vals[1]) / (2 * h)
    assert normwise(got.numpy(), fd.numpy()) < 1e-5, (got, fd)


# ---- the FFMA kernels under the emulator ---------------------------------------------------------------------------------------
CASES = {
    # name: (tower sizes, threshold, fully connected)
    'two_relations': ([2], 1e9, False),
    'c1_tower_7': ([7], 330.0, False),
    'fully_connected_5x2': ([5, 5], 0.0, True),
    'ragged_0_1_2_7': ([0, 1, 2, 7], 330.0, False),
    'no_relations': ([3, 4], 0.0, False),
}


@pytest.mark.parametrize('rate', [0.0, 0.1])
@pytest.mark.parametrize('case', sorted(CASES))
def test_emu_rel_grad_matches_reference(emu, case, rate):
    sizes, thr, fc = CASES[case]
    rng = np.random.default_rng(sum(map(ord, case)) + 1)
    node_off, pos, wid = _ragged(rng, sizes)
    g = emu.edges(pos, node_off, thr=thr, fully_connected=fc)
    if case == 'two_relations':
        assert g.E == 2
    if case == 'no_relations':
        assert g.E == 0
    obj = np.concatenate([pos, wid[:, None]], 1) / 170.0
    w64 = O.kinkfree_weights(3)
    wnp = {k: v.numpy() for k, v in w64.items()}
    seed = 0x2468ACE013579BDF
    emu.forward(wnp, g, obj, training=True, dropout_rate=rate, dropout_seed=seed)
    dl = rng.standard_normal(g.n).astype(np.float32)
    dobj_ref, _ = backward_obj(emu, g, dl)
    # the reference on the receiver-major relation list: row k's dropout elements are k * 160 + c
    cs, qs = (None, None)
    if rate > 0:
        g_rm = type('G', (), {'out_pos': np.arange(g.E, dtype=np.int64), 'n': g.n})
        cs, qs = dropout_scales(g_rm, seed, rate)
    o64 = torch.as_tensor(obj.astype(np.float32).astype(np.float64))
    ref, _, _ = rel_grads(w64, o64, torch.as_tensor(g.in_snd), torch.as_tensor(g.in_rcv), torch.as_tensor(dl.astype(np.float64)),
                          c_scale=cs, q_scale=qs)
    drel, dobj, launches = backward_rel(emu, g, dl)
    assert np.isfinite(drel).all()
    r = normwise(drel, ref.numpy())
    assert r <= 1e-5, (case, rate, r)
    assert np.array_equal(dobj.view(np.uint32), dobj_ref.view(np.uint32))
    # rerun, and without dobj: the same bits
    again, _, _ = backward_rel(emu, g, dl, with_dobj=False)
    assert np.array_equal(again.view(np.uint32), drel.view(np.uint32))
    if g.E == 0:
        _, _, launches = backward_rel(emu, g, dl, with_dobj=False)
        assert launches == 0


def test_emu_rel_grad_leaves_weight_gradients_alone(emu):
    """A backward_rel between the forward and spw_backward: the weight gradients are the same bits as without it."""
    rng = np.random.default_rng(6)
    node_off, pos, wid = _ragged(rng, [5, 6])
    g = emu.edges(pos, node_off, thr=330.0)
    obj = np.concatenate([pos, wid[:, None]], 1) / 170.0
    wnp = {k: v.numpy() for k, v in O.kinkfree_weights(4).items()}
    dl = rng.standard_normal(g.n).astype(np.float32)
    emu.forward(wnp, g, obj, training=True)
    g0 = emu.backward(g, dl)
    emu.forward(wnp, g, obj, training=True)
    backward_rel(emu, g, dl)
    g1 = emu.backward(g, dl)
    for k in g0:
        assert np.array_equal(g0[k].view(np.uint32), g1[k].view(np.uint32)), k


def test_backward_rel_host_side_argument_checks():
    """Host-side errors on the sm_100a library, without a GPU: null drel (with relations), null obj, misaligned drel, dobj or
    workspace, a bad rate, a workspace that is too small, a misaligned weight.  An empty batch launches nothing, and a batch
    without relations accepts a null drel."""
    from spwgnn_b200 import build
    from spwgnn_b200._capi import CApi, SpwGraph
    api = CApi(build.build())
    p = CApi.params([16 * (i + 1) for i in range(22)])
    g = SpwGraph(1, 4, 12, 16, 16, 16, 16, 16, 16)                       # non-null, aligned fake device pointers
    big = 1 << 40
    f = api.dll.spw_backward_rel
    rc = f(ctypes.byref(p), ctypes.byref(g), 16, 16, 16, big, 0.0, None, None, None)
    assert rc == -1 and b'null' in api.dll.spw_last_error()
    rc = f(ctypes.byref(p), ctypes.byref(g), None, 16, 16, big, 0.0, 16, None, None)
    assert rc == -1 and b'null' in api.dll.spw_last_error()
    rc = f(ctypes.byref(p), ctypes.byref(g), 16, 16, 16, big, 0.0, 18, None, None)
    assert rc == -1 and b'drel' in api.dll.spw_last_error()
    rc = f(ctypes.byref(p), ctypes.byref(g), 16, 16, 16, big, 0.0, 20, 20, None)
    assert rc == -1 and b'dobj' in api.dll.spw_last_error()
    rc = f(ctypes.byref(p), ctypes.byref(g), 16, 16, 24, big, 0.0, 16, None, None)
    assert rc == -1 and b'workspace' in api.dll.spw_last_error()
    for rate in (-0.1, 1.0):
        rc = f(ctypes.byref(p), ctypes.byref(g), 16, 16, 16, big, rate, 16, None, None)
        assert rc == -1 and b'rate' in api.dll.spw_last_error()
    need = api.dll.spw_workspace_bytes(4, 12, 1)
    rc = f(ctypes.byref(p), ctypes.byref(g), 16, 16, 16, need - 1, 0.0, 16, 16, None)
    assert rc == -3 and b'workspace' in api.dll.spw_last_error()
    p.p[3] = 20                                                          # a misaligned weight tensor
    rc = f(ctypes.byref(p), ctypes.byref(g), 16, 16, 16, big, 0.0, 16, None, None)
    assert rc == -1 and b'tensor 3' in api.dll.spw_last_error()
    p.p[3] = 64
    before = api.dll.spw_launch_count()
    empty = SpwGraph(0, 0, 0, None, None, None, None, None, None)
    assert f(ctypes.byref(p), ctypes.byref(empty), None, None, None, 0, 0.0, None, None, None) == 0
    no_rel = SpwGraph(1, 4, 0, 16, 16, 16, 16, 16, 16)
    assert f(ctypes.byref(p), ctypes.byref(no_rel), 16, 16, 16, big, 0.0, None, None, None) == 0
    assert api.dll.spw_launch_count() == before
