"""spw_forward_towers (one CTA per tower, spw_small.cuh) under the host emulator (tools/cuemu) against the fp64 oracle, and its
host-side argument checks.  CPU only; tests/test_gpu_small.py checks the real binary."""
import ctypes
import os

import numpy as np
import pytest
import torch

from oracle import propnet as O

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SMALL_SRC = os.path.join(ROOT, 'spwgnn_b200', 'csrc', 'spw_small.cuh')


@pytest.fixture(scope='module')
def emu():
    import emu_harness
    from emu_harness import Emu, EMU_LIB, build_emu
    # the harness tracks the sources it knew of; spw_small.cuh is included by spwgnn.cu but not in its list
    if os.path.exists(EMU_LIB) and os.path.getmtime(EMU_LIB) < os.path.getmtime(SMALL_SRC):
        build_emu(force=True)
    assert emu_harness.EMU_LIB == EMU_LIB
    return Emu()


def forward_towers(emu, w, g, obj, max_nodes, want_probs=True, fill=np.nan):
    """spw_forward_towers on host arrays; returns (logits, probs or None, workspace)"""
    api = emu.api
    wl, wp, keep = emu.pack_params(w)
    obj = np.ascontiguousarray(obj, dtype=np.float32)
    nbytes = int(api.dll.spw_forward_towers_bytes(g.n, g.E))
    ws = np.full(nbytes // 4 + 8, fill, np.float32)
    off = (-ws.ctypes.data // 4) % 4
    wsv = ws[off:off + nbytes // 4]
    logits = np.full(max(g.n, 1) + 4, fill, np.float32)
    probs = np.full(max(g.n, 1) + 4, fill, np.float32)
    lo, po = (-logits.ctypes.data // 4) % 4, (-probs.ctypes.data // 4) % 4
    lv, pv = logits[lo:lo + max(g.n, 1)], probs[po:po + max(g.n, 1)]
    before = api.dll.spw_launch_count()
    api.check(api.dll.spw_forward_towers(ctypes.byref(wp), ctypes.byref(g.c), int(max_nodes), obj.ctypes.data, lv.ctypes.data,
                                         pv.ctypes.data if want_probs else None, wsv.ctypes.data, nbytes, None))
    launches = api.dll.spw_launch_count() - before
    return lv[:g.n].copy(), (pv[:g.n].copy() if want_probs else None), launches


def _ragged(rng, sizes, fully_connected):
    node_off = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int32)
    n = int(node_off[-1])
    pos = np.stack([rng.integers(300, 900, n).astype(np.float64), 110 + 80 * rng.integers(0, 5, n)], 1)
    wid = rng.integers(50, 300, n).astype(np.float64)
    return node_off, pos, wid


def _oracle(w64, obj, snd, rcv):
    o64 = torch.as_tensor(np.asarray(obj, np.float32).astype(np.float64))
    p, z = O.forward_sparse(w64, o64, torch.as_tensor(snd), torch.as_tensor(rcv), return_logits=True)
    return z.numpy(), p.numpy()


def test_emu_forward_towers_matches_oracle_and_is_batch_invariant(emu):
    """A ragged batch of 0 .. 32 blocks (contact edges; the 32-block tower fully connected: in-degree 31, 992 edges, 31
    chunks) against the oracle, then every tower alone: the same bits."""
    rng = np.random.default_rng(7)
    sizes = [3, 0, 1, 2, 7, 13, 32]
    node_off, pos, wid = _ragged(rng, sizes, False)
    obj = np.concatenate([pos, wid[:, None]], 1) / 170.0
    w64 = O.init_weights(11, nonzero_bias=True)
    wnp = {k: v.numpy() for k, v in w64.items()}
    # contact edges for the small towers, all pairs for the 32-block one (a threshold above every distance in it)
    g = emu.edges(pos, node_off, thr=330.0)
    a32 = int(node_off[-2])
    gf = emu.edges(pos[a32:], np.array([0, 32], np.int32), fully_connected=True)
    assert gf.E == 32 * 31
    logits, probs, launches = forward_towers(emu, wnp, g, obj, 32)
    assert launches == 1
    eo, snd, rcv, _ = O.edge_list(pos, node_off, thr=330.0)
    z64, p64 = _oracle(w64, obj, snd, rcv)
    assert np.abs(logits - z64).max() / np.abs(z64).max() <= 1e-5
    assert np.abs(probs - p64).max() / np.abs(p64).max() <= 1e-5
    lf, pf, _ = forward_towers(emu, wnp, gf, obj[a32:], 32)
    eo, snd, rcv, _ = O.edge_list(pos[a32:], np.array([0, 32]), fully_connected=True)
    z64, p64 = _oracle(w64, obj[a32:], snd, rcv)
    assert np.abs(lf - z64).max() / np.abs(z64).max() <= 1e-5
    assert np.abs(pf - p64).max() / np.abs(p64).max() <= 1e-5
    # every tower alone, with a different node capacity: the same bits
    for t, nt in enumerate(sizes):
        a, b = int(node_off[t]), int(node_off[t + 1])
        if nt == 0:
            continue
        gt = emu.edges(pos[a:b], np.array([0, nt], np.int32), thr=330.0)
        lt, pt, _ = forward_towers(emu, wnp, gt, obj[a:b], nt)
        assert np.array_equal(lt.view(np.uint32), logits[a:b].view(np.uint32)), t
        assert np.array_equal(pt.view(np.uint32), probs[a:b].view(np.uint32)), t
    # a rerun: the same bits
    l2, p2, _ = forward_towers(emu, wnp, g, obj, 32, fill=0.0)
    assert np.array_equal(l2.view(np.uint32), logits.view(np.uint32))


def test_emu_forward_towers_oversized_tower_and_no_probs(emu):
    """A tower larger than max_nodes_per_tower gets NaN rows; its neighbours are computed; probs = NULL writes no probs."""
    rng = np.random.default_rng(8)
    sizes = [4, 9, 5]
    node_off, pos, wid = _ragged(rng, sizes, False)
    obj = np.concatenate([pos, wid[:, None]], 1) / 170.0
    w64 = O.init_weights(12, nonzero_bias=True)
    wnp = {k: v.numpy() for k, v in w64.items()}
    g = emu.edges(pos, node_off, thr=330.0)
    logits, probs, _ = forward_towers(emu, wnp, g, obj, 8, fill=0.0)
    assert np.all(np.isnan(logits[4:13])) and np.all(np.isnan(probs[4:13]))
    full, _, _ = forward_towers(emu, wnp, g, obj, 9)
    assert np.array_equal(logits[:4], full[:4]) and np.array_equal(logits[13:], full[13:])
    l0, p0, launches = forward_towers(emu, wnp, g, obj, 9, want_probs=False)
    assert p0 is None and launches == 1 and np.array_equal(l0, full)


def test_forward_towers_host_side_argument_checks():
    """The three host-side errors, on the sm_100a library, without a GPU: a null tensor, a tower limit above
    SPW_SMALL_MAX_NODES, a workspace that is too small.  An empty batch launches nothing."""
    from spwgnn_b200 import build
    from spwgnn_b200._capi import CApi, SpwParams, SpwGraph
    api = CApi(build.build())
    p = SpwParams()
    g = SpwGraph(1, 4, 12, 16, 16, 16, 16, 16, 16)                       # non-null, aligned fake device pointers
    rc = api.dll.spw_forward_towers(ctypes.byref(p), ctypes.byref(g), 4, 16, 16, None, 16, 1 << 20, None)
    assert rc == -1 and b'tensor 0' in api.dll.spw_last_error()
    p = CApi.params([16 * (i + 1) for i in range(22)])
    p.p[5] = 20                                                          # misaligned
    rc = api.dll.spw_forward_towers(ctypes.byref(p), ctypes.byref(g), 4, 16, 16, None, 16, 1 << 20, None)
    assert rc == -1 and b'tensor 5' in api.dll.spw_last_error()
    p.p[5] = 96
    rc = api.dll.spw_forward_towers(ctypes.byref(p), ctypes.byref(g), 33, 16, 16, None, 16, 1 << 20, None)
    assert rc == -2 and b'limit' in api.dll.spw_last_error()
    need = api.dll.spw_forward_towers_bytes(4, 12)
    assert need == 12 * 152 * 4 and api.dll.spw_forward_towers_bytes(4, 0) == 0
    rc = api.dll.spw_forward_towers(ctypes.byref(p), ctypes.byref(g), 4, 16, 16, None, 16, need - 1, None)
    assert rc == -3 and b'workspace' in api.dll.spw_last_error()
    before = api.dll.spw_launch_count()
    empty = SpwGraph(0, 0, 0, None, None, None, None, None, None)
    assert api.dll.spw_forward_towers(ctypes.byref(p), ctypes.byref(empty), 4, None, None, None, None, 0, None) == 0
    assert api.dll.spw_launch_count() == before
