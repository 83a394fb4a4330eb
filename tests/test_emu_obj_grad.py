"""spw_backward_obj (the gradient with respect to obj = [x, y, width] / 170, k_obj_grad_c in spw_obj_grad.cuh) under the host
emulator (tools/cuemu) against the fp64 oracle, its host-side argument checks, and the fp64 reference obj_grads (tests/obj_grad_ref.py) against central
differences.  CPU only; tests/test_gpu_obj_grad.py checks the real binary."""
import ctypes
import os

import numpy as np
import pytest
import torch

from oracle import propnet as O
from obj_grad_ref import obj_grads

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
CSRC = os.path.join(ROOT, 'spwgnn_b200', 'csrc')


@pytest.fixture(scope='module')
def emu():
    import emu_harness
    from emu_harness import Emu, EMU_LIB, build_emu
    # the harness tracks the sources it knew of; spw_obj_grad.cuh (and spw_small.cuh) are included by spwgnn.cu but not listed
    srcs = [os.path.join(CSRC, f) for f in ('spw_obj_grad.cuh', 'spw_small.cuh', 'spw_kernels.cuh', 'spwgnn.cu')]
    if os.path.exists(EMU_LIB) and os.path.getmtime(EMU_LIB) < max(os.path.getmtime(s) for s in srcs):
        build_emu(force=True)
    assert emu_harness.EMU_LIB == EMU_LIB
    return Emu()


def backward_obj(emu, g, dlogits, rate=None):
    """spw_backward_obj on the state of the last emu.forward(training=True); dobj is 16-byte aligned and NaN-filled."""
    api = emu.api
    wl, wp, keep, obj, ws, wsv, nbytes = emu._state
    dl = np.ascontiguousarray(dlogits, np.float32)
    buf = np.full(3 * max(g.n, 1) + 8, np.nan, np.float32)
    off = (-buf.ctypes.data // 4) % 4
    dobj = buf[off:off + 3 * max(g.n, 1)]
    before = api.dll.spw_launch_count()
    api.check(api.dll.spw_backward_obj(ctypes.byref(wp), ctypes.byref(g.c), obj.ctypes.data, dl.ctypes.data, wsv.ctypes.data,
                                       nbytes, emu._rate if rate is None else rate, dobj.ctypes.data, None))
    return dobj[:3 * g.n].reshape(g.n, 3).copy(), api.dll.spw_launch_count() - before


def _ragged(rng, sizes):
    node_off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)
    n = int(node_off[-1])
    pos = np.stack([rng.integers(300, 900, n).astype(np.float64), 110 + 80 * rng.integers(0, 5, n)], 1)
    wid = rng.integers(50, 300, n).astype(np.float64)
    return node_off, pos, wid


def dropout_scales(g, seed, rate):
    """The kernels' dropout masks restated (test_emu_kernels.test_emu_dropout_matches_oracle_with_same_mask) as oracle factors."""
    sc, sq = O.dropout_seeds(seed)
    keep = float(1.0 / (1.0 - np.float32(rate)))
    epos = g.out_pos.astype(np.uint64)
    c_keep = O.dropout_keep_mask(sc, epos[:, None] * np.uint64(160) + np.arange(150, dtype=np.uint64)[None, :], rate)
    q_keep = O.dropout_keep_mask(sq, np.arange(g.n, dtype=np.uint64)[:, None] * np.uint64(128) + np.arange(100, dtype=np.uint64)[None, :], rate)
    return torch.as_tensor(c_keep * keep), torch.as_tensor(q_keep * keep)


def normwise(got, ref):
    """max |delta| / max |ref| per column (x, y, width); a column whose reference is all zero must be exactly zero"""
    out = []
    for c in range(3):
        m = np.abs(ref[:, c]).max() if len(ref) else 0.0
        d = np.abs(got[:, c] - ref[:, c]).max() if len(ref) else 0.0
        out.append(d / m if m > 0 else (0.0 if d == 0 else np.inf))
    return out


CASES = {
    # name: (tower sizes, threshold, fully connected)
    'two_relations': ([2], 1e9, False),
    'c1_tower_7': ([7], 330.0, False),
    'ragged_0_1_2_7': ([0, 1, 2, 7], 330.0, False),
    'no_relations': ([3, 4], 0.0, False),
}


@pytest.mark.parametrize('rate', [0.0, 0.1])
@pytest.mark.parametrize('case', sorted(CASES))
def test_emu_obj_grad_matches_oracle(emu, case, rate):
    sizes, thr, fc = CASES[case]
    rng = np.random.default_rng(sum(map(ord, case)))
    node_off, pos, wid = _ragged(rng, sizes)
    g = emu.edges(pos, node_off, thr=thr, fully_connected=fc)
    eo, snd, rcv, _ = O.edge_list(pos, node_off, thr=thr, fully_connected=fc)
    if case == 'two_relations':
        assert g.E == 2
    if case == 'no_relations':
        assert g.E == 0
    obj = np.concatenate([pos, wid[:, None]], 1) / 170.0
    w64 = O.kinkfree_weights(3)
    wnp = {k: v.numpy() for k, v in w64.items()}
    seed = 0x2468ACE013579BDF
    logits, _ = emu.forward(wnp, g, obj, training=True, dropout_rate=rate, dropout_seed=seed)
    cs, qs = dropout_scales(g, seed, rate) if rate > 0 else (None, None)
    o64 = torch.as_tensor(obj.astype(np.float32).astype(np.float64))
    dl = rng.standard_normal(g.n).astype(np.float32)
    ref, l64, _ = obj_grads(w64, o64, torch.as_tensor(snd), torch.as_tensor(rcv), torch.as_tensor(dl.astype(np.float64)),
                              c_scale=cs, q_scale=qs)
    if g.n:
        assert np.abs(logits - l64.numpy()).max() / np.abs(l64.numpy()).max() < 1e-5
    dobj, launches = backward_obj(emu, g, dl)
    assert np.isfinite(dobj).all()
    for c, r in enumerate(normwise(dobj, ref.numpy())):
        assert r <= 1e-5, (case, rate, 'xyw'[c], r)
    if g.E == 0:
        assert np.all(dobj[:, 0] == 0)
    # rerun: the same bits; the forward state is left for another backward
    again, _ = backward_obj(emu, g, dl)
    assert np.array_equal(again.view(np.uint32), dobj.view(np.uint32))
    if g.n == 0:
        assert launches == 0


def test_emu_obj_grad_leaves_weight_gradients_alone(emu):
    """A backward_obj between the forward and spw_backward: the weight gradients are the same bits as without it."""
    rng = np.random.default_rng(5)
    node_off, pos, wid = _ragged(rng, [5, 6])
    g = emu.edges(pos, node_off, thr=330.0)
    obj = np.concatenate([pos, wid[:, None]], 1) / 170.0
    wnp = {k: v.numpy() for k, v in O.kinkfree_weights(4).items()}
    dl = rng.standard_normal(g.n).astype(np.float32)
    emu.forward(wnp, g, obj, training=True)
    g0 = emu.backward(g, dl)
    emu.forward(wnp, g, obj, training=True)
    backward_obj(emu, g, dl)
    g1 = emu.backward(g, dl)
    for k in g0:
        assert np.array_equal(g0[k].view(np.uint32), g1[k].view(np.uint32)), k


def test_backward_obj_host_side_argument_checks():
    """Host-side errors on the sm_100a library, without a GPU: null dobj, a misaligned dobj or workspace, a bad rate, a
    workspace that is too small.  An empty batch launches nothing."""
    from spwgnn_b200 import build
    from spwgnn_b200._capi import CApi, SpwGraph
    api = CApi(build.build())
    p = CApi.params([16 * (i + 1) for i in range(22)])
    g = SpwGraph(1, 4, 12, 16, 16, 16, 16, 16, 16)                       # non-null, aligned fake device pointers
    big = 1 << 40
    f = api.dll.spw_backward_obj
    rc = f(ctypes.byref(p), ctypes.byref(g), 16, 16, 16, big, 0.0, None, None)
    assert rc == -1 and b'null' in api.dll.spw_last_error()
    rc = f(ctypes.byref(p), ctypes.byref(g), 16, 16, 16, big, 0.0, 20, None)
    assert rc == -1 and b'aligned' in api.dll.spw_last_error()
    rc = f(ctypes.byref(p), ctypes.byref(g), 16, 16, 24, big, 0.0, 16, None)
    assert rc == -1 and b'workspace' in api.dll.spw_last_error()
    for rate in (-0.1, 1.0):
        rc = f(ctypes.byref(p), ctypes.byref(g), 16, 16, 16, big, rate, 16, None)
        assert rc == -1 and b'rate' in api.dll.spw_last_error()
    need = api.dll.spw_workspace_bytes(4, 12, 1)
    rc = f(ctypes.byref(p), ctypes.byref(g), 16, 16, 16, need - 1, 0.0, 16, None)
    assert rc == -3 and b'workspace' in api.dll.spw_last_error()
    p.p[3] = 20                                                          # a misaligned weight tensor
    rc = f(ctypes.byref(p), ctypes.byref(g), 16, 16, 16, big, 0.0, 16, None)
    assert rc == -1 and b'tensor 3' in api.dll.spw_last_error()
    p.p[3] = 64
    before = api.dll.spw_launch_count()
    empty = SpwGraph(0, 0, 0, None, None, None, None, None, None)
    assert f(ctypes.byref(p), ctypes.byref(empty), None, None, None, 0, 0.0, None, None) == 0
    assert api.dll.spw_launch_count() == before


def test_obj_grads_reference_matches_central_differences():
    """obj_grads against fp64 central differences of sum dlogits*logits on a 4-block tower, per column.  Kink-free weights at
    full Glorot scale: every relu unit is further from its kink than 100 steps, and the x column is not negligible (at the
    default scale 0.1 it is 1e-7 of the others)."""
    rng = np.random.default_rng(9)
    node_off, pos, wid = _ragged(rng, [4])
    eo, snd, rcv, _ = O.edge_list(pos, node_off, thr=1e9)
    snd, rcv = torch.as_tensor(snd), torch.as_tensor(rcv)
    obj = torch.as_tensor(np.concatenate([pos, wid[:, None]], 1) / 170.0)
    w64 = O.kinkfree_weights(3, scale=1.0)
    h = 1e-6
    assert O.min_relu_margin(w64, obj, snd, rcv) > 100 * h
    dl = torch.as_tensor(rng.standard_normal(4))
    got, _, _ = obj_grads(w64, obj, snd, rcv, dl)

    def f(o):
        _, z = O.forward_sparse(w64, o, snd, rcv, return_logits=True)
        return float((z * dl).sum())
    fd = torch.zeros_like(obj)
    for i in range(4):
        for c in range(3):
            a, b = obj.clone(), obj.clone()
            a[i, c] += h; b[i, c] -= h
            fd[i, c] = (f(a) - f(b)) / (2 * h)
    for c, r in enumerate(normwise(got.numpy(), fd.numpy())):
        assert r < 1e-5, ('xyw'[c], r, got[:, c], fd[:, c])
    assert float(got[:, 0].abs().max()) > 1e-3 * float(got.abs().max())
