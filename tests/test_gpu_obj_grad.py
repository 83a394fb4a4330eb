"""spw_backward_obj / PropNetObjFunction / PropagationModel.stability_gradients: the gradient of the predictions with respect
to the block features obj = [x, y, width] / 170, the relations held fixed.

A. fp64 parity against obj_grad_ref.obj_grads (autograd of oracle.propnet.forward_sparse), normwise max|d| / max|ref| per batch and per column (x, y, width), seeded
   with a fixed random dlogits and with the BCE seed.  Kink-free weights, bar 1e-5: C1 (predict glue and contact relations),
   512 fully connected 10-block towers, a ragged 0/1/2/7/13/32/64-block batch, a batch without relations, 64 Jenga-18 towers.
   Glorot weights at scale on the GPU's relu branch (masks from Engine.saved_relu_states() of a training forward of the same
   batch, whose logits PropNetObjFunction must equal bit for bit): C2 full size, C3 at 1024 towers, a 512-tower C4 slice; every
   unit whose state differs from fp64's has |pre-activation| < 2e-5; bar max(2e-5, 4 e32) with e32 the error of a plain fp32
   CPU evaluation of the same branch.  Dropout 0.1 with the mask injected into the oracle, kink-free weights, bar 1e-5.
B. Stage check of k_obj_grad_c on the workspace's own fp32 D_e (GB) and dQ1, elementwise |got - ref| <= tau absref, with absref
   the same formula on absolute values.  The kernel computes u_e as a chain of 150 fused multiply-adds (error <= gamma_150 of
   its absolute sum, gamma_k = k u / (1 - k u), u = 2^-24), adds the u_e of the k <= d in-edges and of the out-edges in two
   sequential chains (gamma_d more), subtracts them (one rounding) and, for y, adds v_i, a 100-term FMA chain (<= gamma_100 <
   gamma_150), with one more rounding.  Every term of the result therefore carries at most 150 + d + 2 roundings:
   tau = gamma_{152 + d}, d = the largest in- or out-degree of the batch.
C. Exact properties: seeding one tower leaves every other tower's rows exactly 0; without relations the x column is exactly 0;
   horizontal translation invariance per tower, |sum_i d/dx_i| <= tau' sum_e |u_e.0|: every edge's u_e (the same bits from
   both ends) enters once with + and once with -, so only the roundings of the two sums and the subtraction are left, and each
   edge is in two nodes' sums: tau' = 2 gamma_{d + 1} (times 1 + gamma_150 for taking |u_e| from fp64); reruns are bit-identical;
   n = 0 launches nothing.
D. No weight gradient: fewer launches than spw_backward, and no k_wgrad_*, k_skinny_c or k_reduce_* tag.
E. Isolation: PropNetObjFunction and stability_gradients between Engine.forward(training=True) and Engine.backward leave the
   weight gradients bit-identical.
F. Write footprint between guard bands with 0x00 and 0xFF fills (test_gpu_inference.footprint_violations): no guard byte of
   dobj or the workspace is written, workspace writes lie in the backward pass's data-gradient arrays, the forward state and the
   inputs are unchanged, both runs give the same bits.
G. Facade: stability_gradients against obj_grads with respect to raw pixels on C1 towers (predict glue, contact relations)
   and on the candidate towers of one score_removals call; bar 1e-5 over the whole matrix and, per column, max(1e-5, 4 e32)
   (the test's docstring says why).

The worst ratio per case is written to $SPW_OBJ_GRAD_OUT (default: obj_grad_parity.json in the temporary directory).
"""
import ctypes
import json
import os
import tempfile

import numpy as np
import pytest
import torch

from oracle import propnet as O
from obj_grad_ref import obj_grads

pytestmark = pytest.mark.gpu
OUT = os.environ.get('SPW_OBJ_GRAD_OUT', os.path.join(tempfile.gettempdir(), 'obj_grad_parity.json'))
TOL = 1e-5
BRANCH_TOL = 2e-5
FLIP_MARGIN = 2e-5
U32 = 2.0 ** -24
_WORST = {}


def gamma(k):
    return k * U32 / (1 - k * U32)


@pytest.fixture(scope='module')
def eng():
    from spwgnn_b200.engine import Engine
    assert torch.cuda.is_available()
    e = Engine('cuda:0', seed=3)
    e.w_kinkfree = O.kinkfree_weights(3)
    e.w_glorot = O.init_weights(3, nonzero_bias=True)
    yield e
    if _WORST:
        try:
            with open(OUT, 'w') as f:
                json.dump({'device': torch.cuda.get_device_name(0), 'max|d|/max|ref| per column (x, y, width)': _WORST}, f,
                          indent=1, sort_keys=True)
                f.write('\n')
        except OSError:
            pass


def _use(eng, which):
    eng.w64 = eng.w_glorot if which == 'glorot' else eng.w_kinkfree
    eng.params.load_dict(eng.w64)


def _batch(kind, seed=0):
    from spwgnn_b200 import synth
    from spwgnn_b200.graph import TowerBatch
    if kind == 'C1':
        return TowerBatch.from_towers(synth.make_towers('tower', 32, 3 + seed, n=7), inference_glue=True)
    if kind == 'C1 contact':
        return TowerBatch.from_towers(synth.make_towers('tower', 32, 3 + seed, n=7))
    if kind == 'fc10 x512':
        return TowerBatch.from_towers(synth.make_towers('jenga', 512, 40 + seed, n=10), fully_connected=True)
    if kind == 'ragged':
        towers = []
        for i, nb in enumerate([0, 1, 2, 7, 13, 32, 64]):
            towers += synth.make_towers('jenga', 1, 60 + seed + i, n=nb) if nb else [np.zeros((0, 3))]
        return TowerBatch.from_towers(towers, thr=330.0)
    if kind == 'no relations':
        return TowerBatch.from_towers(synth.make_towers('jenga', 6, 80 + seed, n=5), thr=0.0)
    if kind == 'jenga18 x64':
        return TowerBatch.from_towers(synth.make_towers('jenga18', 64, 90 + seed))
    if kind == 'C2':
        return TowerBatch.from_towers(synth.make_towers('jenga', 4096, 1235, n=10), fully_connected=True)
    if kind == 'C3':
        return TowerBatch.from_towers(synth.make_towers('jenga18', 1024, 31))
    if kind == 'C4 x512':
        return TowerBatch.from_towers(synth.make_towers('uniform', 512, 32, lo=6, hi=32))
    raise ValueError(kind)


def _edges(batch):
    E = batch.n_edges
    return batch.in_snd[:E].cpu().long(), batch.in_rcv[:E].cpu().long()


def _seed(eng, batch, which, rng):
    n = batch.n_nodes
    if which == 'random':
        return torch.as_tensor(rng.standard_normal(n).astype(np.float32)).cuda()
    logits, _ = eng.forward(batch, training=False, want_probs=False)
    tgt = torch.as_tensor((rng.random(n) > 0.5).astype(np.float32)).cuda()
    dl, _ = eng.bce_seed(logits.contiguous(), tgt, max(n, 1))
    return dl.clone()


def obj_grad(eng, batch, dl):
    """PropNetObjFunction forward + backward; returns (logits, dobj) on the device"""
    from spwgnn_b200.engine import PropNetObjFunction
    obj = batch.obj.detach().clone().requires_grad_(True)
    logits = PropNetObjFunction.apply(obj, eng, batch)
    logits.backward(dl)
    return logits.detach(), obj.grad


def percol(got, ref):
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    out = []
    for c in range(3):
        m = np.abs(ref[:, c]).max() if len(ref) else 0.0
        d = np.abs(got[:, c] - ref[:, c]).max() if len(ref) else 0.0
        out.append(float(d / m) if m > 0 else (0.0 if d == 0 else float('inf')))
    return out


def _record(name, errs, extra=None):
    _WORST[name] = dict(zip(('x', 'y', 'width'), errs), **(extra or {}))


# ---- A. fp64 parity -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('seed_kind', ['random', 'bce'])
@pytest.mark.parametrize('kind', ['C1', 'C1 contact', 'fc10 x512', 'ragged', 'no relations', 'jenga18 x64'])
def test_parity_kinkfree(eng, kind, seed_kind):
    _use(eng, 'kinkfree')
    batch = _batch(kind)
    if kind == 'no relations':
        assert batch.n_edges == 0
    dl = _seed(eng, batch, seed_kind, np.random.default_rng(11))
    logits, dobj = obj_grad(eng, batch, dl)
    snd, rcv = _edges(batch)
    ref, l64, _ = obj_grads(eng.w64, batch.obj.cpu().double(), snd, rcv, dl.cpu().double())
    assert np.abs(logits.cpu().numpy() - l64.numpy()).max() <= TOL * np.abs(l64.numpy()).max()
    errs = percol(dobj.cpu().numpy(), ref.numpy())
    _record('%s, kinkfree, %s seed' % (kind, seed_kind), errs)
    assert max(errs) <= TOL, errs


@pytest.mark.parametrize('kind', ['C2', 'C3', 'C4 x512'])
def test_parity_glorot_on_gpu_branch(eng, kind):
    _use(eng, 'glorot')
    batch = _batch(kind)
    n = batch.n_nodes
    lt, _ = eng.forward(batch, training=True, want_probs=False)
    lt = lt.clone()
    masks = [m.cpu() for m in eng.saved_relu_states()]
    dl = _seed(eng, batch, 'random', np.random.default_rng(12))
    logits, dobj = obj_grad(eng, batch, dl)
    assert torch.equal(logits, lt)
    snd, rcv = _edges(batch)
    obj32 = batch.obj.cpu()
    ref, _, flips = obj_grads(eng.w64, obj32.double(), snd, rcv, dl.cpu().double(), masks=masks)
    w32 = {k: v.float() for k, v in eng.w64.items()}
    g32, _, _ = obj_grads(w32, obj32, snd, rcv, dl.cpu(), masks=masks)
    maxpre = max(f[1] for f in flips)
    assert maxpre < FLIP_MARGIN, maxpre
    errs = percol(dobj.cpu().numpy(), ref.numpy())
    e32 = percol(g32.numpy(), ref.numpy())
    _record('%s, glorot, GPU branch' % kind, errs, {'plain_fp32_same_branch': e32, 'blocks': n, 'relations': batch.n_edges,
                                                     'relu_units_flipped_vs_fp64': sum(f[0] for f in flips)})
    for c in range(3):
        assert errs[c] <= max(BRANCH_TOL, 4 * e32[c]), (c, errs, e32)


def _c_api_obj(eng, batch, dl, rate=0.0, seed=0, fill=None):
    """training spw_forward + spw_backward_obj through the C ABI on a workspace of our own (optionally pre-filled with the byte
    `fill`); returns (logits, dobj, workspace bytes, the workspace right after the forward)"""
    from spwgnn_b200.graph import _stream_ptr
    api, n, E = eng.api, batch.n_nodes, batch.n_edges
    nbytes = int(api.dll.spw_workspace_bytes(n, E, 1))
    ws = torch.full((nbytes,), fill if fill is not None else 0xFF, dtype=torch.uint8, device='cuda')
    if fill is None:
        ws.view(torch.float32).fill_(float('nan'))
    logits = torch.empty(max(n, 1), device='cuda')
    dobj = torch.full((max(n, 1), 3), float('nan'), device='cuda')
    wp = eng.params.c_struct()
    st = _stream_ptr(torch.device('cuda:0'))
    api.check(api.dll.spw_forward(ctypes.byref(wp), ctypes.byref(batch.c_graph), batch.obj.data_ptr(), logits.data_ptr(), None,
                                  ws.data_ptr(), nbytes, 1, float(rate), int(seed), st))
    after_fwd = ws.clone()
    api.check(api.dll.spw_backward_obj(ctypes.byref(wp), ctypes.byref(batch.c_graph), batch.obj.data_ptr(), dl.data_ptr(),
                                       ws.data_ptr(), nbytes, float(rate), dobj.data_ptr(), st))
    torch.cuda.synchronize()
    return logits[:n], dobj[:n], ws, after_fwd


def test_dropout_matches_oracle_with_same_mask(eng):
    _use(eng, 'kinkfree')
    batch = _batch('C1 contact')
    n, E = batch.n_nodes, batch.n_edges
    rate, seed = 0.1, 0x1234567855AA77
    dl = _seed(eng, batch, 'random', np.random.default_rng(13))
    logits, dobj, _, _ = _c_api_obj(eng, batch, dl, rate, seed)
    sc, sq = O.dropout_seeds(seed)
    keep = float(1.0 / (1.0 - np.float32(rate)))
    # the oracle runs on the receiver-major edge list: edge row p's mask elements are p * 160 + c
    c_keep = O.dropout_keep_mask(sc, np.arange(E, dtype=np.uint64)[:, None] * np.uint64(160) + np.arange(150, dtype=np.uint64)[None, :], rate)
    q_keep = O.dropout_keep_mask(sq, np.arange(n, dtype=np.uint64)[:, None] * np.uint64(128) + np.arange(100, dtype=np.uint64)[None, :], rate)
    snd, rcv = _edges(batch)
    ref, l64, _ = obj_grads(eng.w64, batch.obj.cpu().double(), snd, rcv, dl.cpu().double(),
                              c_scale=torch.as_tensor(c_keep * keep), q_scale=torch.as_tensor(q_keep * keep))
    assert np.abs(logits.cpu().numpy() - l64.numpy()).max() <= TOL * np.abs(l64.numpy()).max()
    errs = percol(dobj.cpu().numpy(), ref.numpy())
    _record('C1 contact, kinkfree, dropout 0.1', errs)
    assert max(errs) <= TOL, errs


# ---- B. stage check of k_obj_grad_c -------------------------------------------------------------------------------------------
def _stage_inputs(eng, batch, ws):
    n, E = batch.n_nodes, batch.n_edges
    lay = eng.api.workspace_layout(n, E, 1)
    f = ws.view(torch.float32)
    gb, dq1 = lay['GB'] // 4, lay['dQ1'] // 4
    D = f[gb:gb + 38 * E * 4].view(38, E, 4).permute(1, 0, 2).reshape(E, 152)[:, :150].double().cpu()
    Q = f[dq1:dq1 + 25 * n * 4].view(25, n, 4).permute(1, 0, 2).reshape(n, 100).double().cpu()
    return D, Q


def _formula(D, Q, rw, ow, batch):
    """d obj from D_e and dQ1 in fp64 (the kernel's formula); returns (dobj, per-edge u)"""
    n = batch.n_nodes
    snd, rcv = _edges(batch)
    u = D @ rw.T                                  # (E, 2)
    v = Q @ ow.T                                  # (n, 2)
    out = torch.zeros(n, 3, dtype=torch.float64)
    out[:, 0:2].index_add_(0, rcv, u).index_add_(0, snd, -u)
    out[:, 1] += v[:, 0]
    out[:, 2] = v[:, 1]
    return out, u


@pytest.mark.parametrize('kind', ['C1 contact', 'fc10 x512', 'ragged', 'jenga18 x64'])
def test_stage_k_obj_grad_c(eng, kind):
    _use(eng, 'glorot')
    batch = _batch(kind)
    dl = _seed(eng, batch, 'random', np.random.default_rng(14))
    _, dobj, ws, _ = _c_api_obj(eng, batch, dl)
    D, Q = _stage_inputs(eng, batch, ws)
    rw, ow = eng.w64['rm.w0'].double(), eng.w64['om.w0'].double()            # Keras [2][k]: row 0 -> x (resp. y), row 1 -> y (width)
    ref, _ = _formula(D, Q, rw, ow, batch)
    snd, rcv = _edges(batch)
    au, av = D.abs() @ rw.abs().T, Q.abs() @ ow.abs().T
    absref = torch.zeros(batch.n_nodes, 3, dtype=torch.float64)
    absref[:, 0:2].index_add_(0, rcv, au).index_add_(0, snd, au)
    absref[:, 1] += av[:, 0]
    absref[:, 2] = av[:, 1]
    n = batch.n_nodes
    deg = 0
    if batch.n_edges:
        deg = int(max(torch.bincount(rcv, minlength=n).max(), torch.bincount(snd, minlength=n).max()))
    tau = gamma(152 + deg)
    got = dobj.cpu().double()
    assert torch.isfinite(got).all()
    viol = (got - ref).abs() > tau * absref
    assert not bool(viol.any()), (int(viol.sum()), float(((got - ref).abs() / absref.clamp_min(1e-300)).max()), tau)


# ---- C. exact properties --------------------------------------------------------------------------------------------------------
def test_exact_properties(eng):
    _use(eng, 'glorot')
    batch = _batch('C1 contact')
    n = batch.n_nodes
    off = batch.node_off_host
    dl = _seed(eng, batch, 'random', np.random.default_rng(15))
    # one tower seeded: every other row exactly 0
    t = 5
    one = torch.zeros_like(dl)
    one[off[t]:off[t + 1]] = dl[off[t]:off[t + 1]]
    _, d1 = obj_grad(eng, batch, one)
    d1 = d1.cpu().numpy()
    mask = np.ones(n, bool)
    mask[off[t]:off[t + 1]] = False
    assert np.all(d1[mask] == 0) and np.abs(d1[~mask]).max() > 0
    # no relations: x column exactly 0
    nb = _batch('no relations')
    _, d0 = obj_grad(eng, nb, _seed(eng, nb, 'random', np.random.default_rng(16)))
    assert torch.all(d0[:, 0] == 0) and float(d0[:, 1:].abs().max()) > 0
    # horizontal translation invariance per tower
    for kind in ('C1', 'fc10 x512', 'jenga18 x64'):
        b = _batch(kind)
        dlk = _seed(eng, b, 'random', np.random.default_rng(17))
        _, dobj, ws, _ = _c_api_obj(eng, b, dlk)
        D, _ = _stage_inputs(eng, b, ws)
        snd, rcv = _edges(b)
        u0 = (D @ eng.w64['rm.w0'].double()[0]).abs()
        tower_of = torch.as_tensor(np.repeat(np.arange(b.n_towers), np.diff(b.node_off_host)))
        su = torch.zeros(b.n_towers, dtype=torch.float64).index_add_(0, tower_of[rcv], u0)
        sx = torch.zeros(b.n_towers, dtype=torch.float64).index_add_(0, tower_of, dobj[:, 0].cpu().double())
        deg = int(max(torch.bincount(rcv).max(), torch.bincount(snd).max()))
        tau = 2 * gamma(deg + 1) * (1 + gamma(150))
        assert bool((sx.abs() <= tau * su).all()), (kind, float((sx.abs() / su).max()), tau)
        assert float(dobj[:, 0].abs().max()) > 0
    # reruns: the same bits
    a1 = _c_api_obj(eng, batch, dl)[1].clone()
    a2 = _c_api_obj(eng, batch, dl)[1].clone()
    assert torch.equal(a1.view(torch.int32), a2.view(torch.int32))
    _, d3 = obj_grad(eng, batch, dl)
    assert torch.equal(d3.view(torch.int32), a1.view(torch.int32))
    # n = 0 launches nothing
    api = eng.api
    from spwgnn_b200._capi import SpwGraph
    empty = SpwGraph(0, 0, 0, None, None, None, None, None, None)
    before = api.dll.spw_launch_count()
    wp = eng.params.c_struct()
    assert api.dll.spw_backward_obj(ctypes.byref(wp), ctypes.byref(empty), None, None, None, 0, 0.0, None, None) == 0
    assert api.dll.spw_launch_count() == before


# ---- D. no weight gradient ------------------------------------------------------------------------------------------------------
def _profiled(api, fn):
    buf = ctypes.create_string_buffer(1 << 16)
    api.check(api.dll.spw_profile_report(buf, len(buf)))
    api.check(api.dll.spw_profile(1))
    try:
        before = api.dll.spw_launch_count()
        fn()
        torch.cuda.synchronize()
        launches = api.dll.spw_launch_count() - before
        api.check(api.dll.spw_profile_report(buf, len(buf)))
    finally:
        api.dll.spw_profile(0)
    return launches, [ln.split()[0] for ln in buf.value.decode().splitlines() if ln.strip()]


def test_weight_gradients_are_skipped(eng):
    from spwgnn_b200.graph import _stream_ptr
    _use(eng, 'glorot')
    api = eng.api
    batch = _batch('C1 contact')
    dl = _seed(eng, batch, 'random', np.random.default_rng(18))
    eng.forward(batch, training=True, want_probs=False)
    _, ws, _, _ = eng._fwd
    n = batch.n_nodes
    dobj = torch.empty(n, 3, device='cuda')
    wp = eng.params.c_struct()
    st = _stream_ptr(torch.device('cuda:0'))
    nb, tb = _profiled(api, lambda: eng.backward(dl))
    no, to = _profiled(api, lambda: api.check(api.dll.spw_backward_obj(
        ctypes.byref(wp), ctypes.byref(batch.c_graph), batch.obj.data_ptr(), dl.data_ptr(), ws.data_ptr(), ws.numel(), 0.0,
        dobj.data_ptr(), st)))
    assert no < nb, (no, nb)
    assert 'k_obj_grad_c' in to and 'k_obj_grad_c' not in tb
    assert any(t.startswith('k_wgrad') for t in tb)
    bad = [t for t in to if t.startswith('k_wgrad') or t.startswith('k_skinny_c') or t.startswith('k_reduce')]
    assert not bad, bad


# ---- E. isolation -------------------------------------------------------------------------------------------------------------
def test_isolation_from_a_training_step_in_flight(eng):
    from spwgnn_b200 import synth
    from spwgnn_b200.Networks import PropagationNetwork
    _use(eng, 'glorot')
    batch = _batch('C1 contact')
    dl = _seed(eng, batch, 'random', np.random.default_rng(19))
    eng.forward(batch, training=True, want_probs=False, dropout_rate=0.1, dropout_seed=7)
    ref = eng.backward(dl).flat.clone()
    net = PropagationNetwork()
    net._engine = eng
    model = net.getModel(7)
    other = _batch('fc10 x512')
    eng.forward(batch, training=True, want_probs=False, dropout_rate=0.1, dropout_seed=7)
    obj_grad(eng, other, _seed(eng, other, 'random', np.random.default_rng(20)))
    model.stability_gradients(synth.make_towers('tower', 4, 5, n=7))
    got = eng.backward(dl).flat.clone()
    assert torch.equal(got, ref)


# ---- F. write footprint ---------------------------------------------------------------------------------------------------------
BACKWARD_ARRAYS = ('dU', 'dG', 'T', 'dS', 'dR', 'dH2S', 'DP', 'dQ', 'dQ1', 'dA', 'DH1', 'GB')


def test_write_footprint(eng):
    from test_gpu_inference import footprint_violations
    from spwgnn_b200.graph import _stream_ptr
    _use(eng, 'glorot')
    api = eng.api
    batch = _batch('C1 contact')
    n, E = batch.n_nodes, batch.n_edges
    dl = _seed(eng, batch, 'random', np.random.default_rng(21))
    nbytes = int(api.dll.spw_workspace_bytes(n, E, 1))
    lay = api.workspace_layout(n, E, 1)
    ends = sorted(set(v for k, v in lay.items() if k in api.dll.spw_workspace_layout_names().decode().split(',')[:40]) | {nbytes})
    spans = [(k, lay[k], min(e for e in ends if e > lay[k])) for k in BACKWARD_ARRAYS]
    G = 4096
    inputs = [batch.obj, dl, batch.in_off, batch.out_off, batch.out_pos, batch.in_snd, batch.in_rcv, batch.node_off]
    snap = [t.clone() for t in inputs]
    res, wsruns, wsfills, oruns = [], [], [], []
    wp = eng.params.c_struct()
    st = _stream_ptr(torch.device('cuda:0'))
    for fill in (0x00, 0xFF):
        wsb = torch.full((nbytes + 2 * G,), fill, dtype=torch.uint8, device='cuda')
        ob = torch.full((n * 12 + 2 * G,), fill, dtype=torch.uint8, device='cuda')
        logits = torch.empty(n, device='cuda')
        api.check(api.dll.spw_forward(ctypes.byref(wp), ctypes.byref(batch.c_graph), batch.obj.data_ptr(), logits.data_ptr(), None,
                                      wsb.data_ptr() + G, nbytes, 1, 0.0, 0, st))
        before = wsb.clone()
        api.check(api.dll.spw_backward_obj(ctypes.byref(wp), ctypes.byref(batch.c_graph), batch.obj.data_ptr(), dl.data_ptr(),
                                           wsb.data_ptr() + G, nbytes, 0.0, ob.data_ptr() + G, st))
        torch.cuda.synchronize()
        wsruns.append(wsb); wsfills.append(before); oruns.append(ob)
        res.append(ob[G:G + n * 12].view(torch.float32).clone())
    msgs = footprint_violations('dobj', oruns, (0x00, 0xFF), G)
    msgs += footprint_violations('workspace', wsruns, wsfills, G, spans)
    assert not msgs, msgs
    assert torch.equal(res[0].view(torch.int32), res[1].view(torch.int32))
    for a, b in zip(inputs, snap):
        assert torch.equal(a, b)


# ---- G. facade --------------------------------------------------------------------------------------------------------------
def _facade_ref(w64, towers, inference_glue, dtype=torch.float64, thr=170.0):
    from spwgnn_b200 import synth
    raw, node_off = synth.pack_towers(towers)
    pos = raw[:, :2] / 170.0 if inference_glue else raw[:, :2]
    eo, snd, rcv, _ = O.edge_list(pos, node_off, thr=thr)
    w = {k: v.to(dtype) for k, v in w64.items()}
    obj = torch.as_tensor((raw / 170.0).astype(np.float32)).to(dtype)
    _, z = O.forward_sparse(w, obj, torch.as_tensor(snd), torch.as_tensor(rcv), return_logits=True)
    p = torch.sigmoid(z)
    g, _, _ = obj_grads(w, obj, torch.as_tensor(snd), torch.as_tensor(rcv), p * (1 - p))
    return g.double().numpy() / 170.0


@pytest.mark.parametrize('case', ['C1 glue', 'C1 contact', 'score_removals candidates'])
def test_stability_gradients_facade(eng, case):
    """Bars of A, per column max(1e-5, 4 e32) with e32 the error of a plain fp32 CPU evaluation, and 1e-5 over the whole
    matrix.  The e32 term matters for the x column of fully connected (predict glue) towers: with the kink-free weights and the
    score's seed p (1 - p), which is nearly the same for every block, the x derivatives cancel to ~1e-12 of the y and width
    ones, so that column is rounding noise in any fp32 evaluation (e32 ~ 1 there)."""
    from spwgnn_b200 import synth
    from spwgnn_b200.Networks import PropagationNetwork
    _use(eng, 'kinkfree')
    net = PropagationNetwork()
    net._engine = eng
    model = net.getModel(7)
    towers = synth.make_towers('tower', 16, 23, n=7)
    glue = case != 'C1 contact'
    if case == 'score_removals candidates':
        tower = towers[0]
        model.score_removals(tower)
        towers = [np.delete(tower, c, 0) for c in range(len(tower))]
    got = model.stability_gradients(towers, inference_glue=glue)
    ref = _facade_ref(eng.w64, towers, glue)
    e32 = percol(_facade_ref(eng.w64, towers, glue, torch.float32), ref)
    assert len(got) == len(towers) and all(g.dtype == np.float64 and g.shape == (len(t), 3) for g, t in zip(got, towers))
    got = np.concatenate(got)
    errs = percol(got, ref)
    whole = float(np.abs(got - ref).max() / np.abs(ref).max())
    _record('stability_gradients, %s' % case, errs, {'whole_matrix': whole, 'plain_fp32': e32})
    assert whole <= TOL, whole
    for c in range(3):
        assert errs[c] <= max(TOL, 4 * e32[c]), (c, errs, e32)
