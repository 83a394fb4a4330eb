"""spw_backward_rel / Engine.relation_gradients / PropagationModel.relation_gradients: the gradient of the predictions with
respect to the relation weights (relation e = s -> r scaled by w_e in both of its one-hot entries, d/dw_e at w = 1).

A. fp64 parity against rel_grad_ref.rel_grads (autograd of the weighted oracle forward), max|d| / max|ref| per batch, seeded
   with a fixed random dlogits and with the BCE seed.  Kink-free weights, bar 1e-5: C1 (predict glue and contact relations),
   512 fully connected 10-block towers, a ragged 0/1/2/7/13/32/64-block batch, 64 Jenga-18 towers.  Glorot weights at scale
   on the GPU's relu branch (masks from Engine.saved_relu_states() of a training forward of the same batch, whose logits the
   gradient's own forward must equal bit for bit): C2 full size, C3 at 1024 towers, a 512-tower C4 slice; every unit whose
   state differs from fp64's has |pre-activation| < 2e-5; bar max(2e-5, 4 e32) with e32 the error of a plain fp32 CPU
   evaluation of the same branch.  Dropout 0.1 with the mask injected into the reference, kink-free weights, bar 1e-5.
B. Stage check of k_rel_grad_step + k_rel_grad_enc, elementwise |got - ref| <= tau absref, ref the kernels' formula in fp64 on
   the workspace's own fp32 A, S, R, dG (every step), D_e (GB) and the saved relu bits, absref the same formula on absolute
   values.  The kernels read DH1 and dSh2 of each step before the next step overwrites them; the test rebuilds them in fp64
   from the GPU's own dG (dSh2 = dG.W3^T, one k_lin with K = 100; DH1 = relu'(h1) * ((relu'(h2) * dSh2[r]).W2^T),
   k_edge_dgrad_c with K = 150), so, as for the composite stages of test_gpu_stages.py, their bars tau_lin(100) and
   tau_lin(150) are added, with absref carried through on absolute values.  The kernels' own arithmetic: per step one
   sequential chain of 150 + 150 + 100 fused multiply-adds, whose factor A + 2 (S + R) carries two roundings (the add and
   the fma), and one add into drel per launch: five step launches and the encoder term, itself a 150-term fma chain (u_e)
   and two roundings.  Every term of the result carries at most 400 + 2 + 6 roundings: tau_k = gamma_408; the bar is
   tau = tau_lin(100) + tau_lin(150) + gamma_408.
C. Exact properties: dobj from spw_backward_rel is torch.equal to spw_backward_obj's on the same forward; seeding one tower
   leaves every other tower's relations exactly 0; reruns are bit-identical; n = 0 launches nothing; a batch without
   relations launches nothing for drel (nothing at all without dobj, spw_backward_obj's launches with it).
D. No weight gradient: spw_backward_obj's launches plus five k_rel_grad_step and one k_rel_grad_enc, and no k_wgrad_*,
   k_skinny_c or k_reduce_* tag.
E. Isolation: Engine.relation_gradients and PropagationModel.relation_gradients between Engine.forward(training=True) and
   Engine.backward leave the weight gradients bit-identical.
F. Write footprint between guard bands with 0x00 and 0xFF fills (test_gpu_inference.footprint_violations): drel writes
   exactly n_edges floats, no guard byte of drel, dobj or the workspace is written, workspace writes lie in the backward
   pass's data-gradient arrays, the forward state and the inputs are unchanged, both runs give the same bits.
G. Facade: on C1 towers (predict glue and contact relations) the pairs equal a numpy restatement of main.py:66-81 and the
   values match rel_grads in fp64 with the seed p (1 - p); bar 1e-5, or 4 e32 where a plain fp32 evaluation is worse.

The worst ratio per case is written to $SPW_REL_GRAD_OUT (default: rel_grad_parity.json in the temporary directory).
"""
import ctypes
import json
import os
import tempfile

import numpy as np
import pytest
import torch

from oracle import propnet as O
from rel_grad_ref import rel_grads
from test_gpu_obj_grad import _batch, _edges, _profiled, _seed, _use, gamma

pytestmark = pytest.mark.gpu
OUT = os.environ.get('SPW_REL_GRAD_OUT', os.path.join(tempfile.gettempdir(), 'rel_grad_parity.json'))
TOL = 1e-5
BRANCH_TOL = 2e-5
FLIP_MARGIN = 2e-5
U32 = 2.0 ** -24
_WORST = {}


def tau_lin(K):
    """test_gpu_stages.tau_lin: the elementwise bar of one k_lin / k_edge_dgrad_c contraction of length K"""
    return 2.5 * 2.0 ** -21 + np.ceil(K / 8) * 2.0 ** -22 + 4 * U32


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
                json.dump({'device': torch.cuda.get_device_name(0), 'max|d|/max|ref|': _WORST}, f, indent=1, sort_keys=True)
                f.write('\n')
        except OSError:
            pass


def ratio(got, ref):
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    if ref.size == 0:
        return 0.0
    m, d = np.abs(ref).max(), np.abs(got - ref).max()
    return float(d / m) if m > 0 else (0.0 if d == 0 else float('inf'))


def _c_api_rel(eng, batch, dl, rate=0.0, seed=0, ws=None, with_dobj=True):
    """training spw_forward (unless ws, the workspace of one, is given) + spw_backward_rel through the C ABI; drel and dobj are
    NaN-filled.  Returns (logits or None, drel, dobj or None, workspace)"""
    from spwgnn_b200.graph import _stream_ptr
    api, n, E = eng.api, batch.n_nodes, batch.n_edges
    nbytes = int(api.dll.spw_workspace_bytes(n, E, 1))
    wp = eng.params.c_struct()
    st = _stream_ptr(torch.device('cuda:0'))
    logits = None
    if ws is None:
        ws = torch.full((nbytes,), 0xFF, dtype=torch.uint8, device='cuda')
        logits = torch.empty(max(n, 1), device='cuda')
        api.check(api.dll.spw_forward(ctypes.byref(wp), ctypes.byref(batch.c_graph), batch.obj.data_ptr(), logits.data_ptr(), None,
                                      ws.data_ptr(), nbytes, 1, float(rate), int(seed), st))
        logits = logits[:n]
    drel = torch.full((max(E, 1),), float('nan'), device='cuda')
    dobj = torch.full((max(n, 1), 3), float('nan'), device='cuda')
    api.check(api.dll.spw_backward_rel(ctypes.byref(wp), ctypes.byref(batch.c_graph), batch.obj.data_ptr(), dl.data_ptr(),
                                       ws.data_ptr(), ws.numel(), float(rate), drel.data_ptr(),
                                       dobj.data_ptr() if with_dobj else None, st))
    torch.cuda.synchronize()
    return logits, drel[:E], dobj[:n] if with_dobj else None, ws


# ---- A. fp64 parity -----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('seed_kind', ['random', 'bce'])
@pytest.mark.parametrize('kind', ['C1', 'C1 contact', 'fc10 x512', 'ragged', 'jenga18 x64'])
def test_parity_kinkfree(eng, kind, seed_kind):
    _use(eng, 'kinkfree')
    batch = _batch(kind)
    dl = _seed(eng, batch, seed_kind, np.random.default_rng(11))
    drel, _ = eng.relation_gradients(batch, dl)
    snd, rcv = _edges(batch)
    ref, _, _ = rel_grads(eng.w64, batch.obj.cpu().double(), snd, rcv, dl.cpu().double())
    err = ratio(drel.cpu().numpy(), ref.numpy())
    _record('%s, kinkfree, %s seed' % (kind, seed_kind), err)
    assert err <= TOL, err


def _record(name, err, extra=None):
    _WORST[name] = dict({'drel': err}, **(extra or {}))


@pytest.mark.parametrize('kind', ['C2', 'C3', 'C4 x512'])
def test_parity_glorot_on_gpu_branch(eng, kind):
    _use(eng, 'glorot')
    batch = _batch(kind)
    lt, _ = eng.forward(batch, training=True, want_probs=False)
    lt = lt.clone()
    masks = [m.cpu() for m in eng.saved_relu_states()]
    dl = _seed(eng, batch, 'random', np.random.default_rng(12))
    logits, drel, _, _ = _c_api_rel(eng, batch, dl, with_dobj=False)
    assert torch.equal(logits, lt)
    snd, rcv = _edges(batch)
    obj32 = batch.obj.cpu()
    ref, _, flips = rel_grads(eng.w64, obj32.double(), snd, rcv, dl.cpu().double(), masks=masks)
    w32 = {k: v.float() for k, v in eng.w64.items()}
    g32, _, _ = rel_grads(w32, obj32, snd, rcv, dl.cpu(), masks=masks)
    maxpre = max(f[1] for f in flips)
    assert maxpre < FLIP_MARGIN, maxpre
    err = ratio(drel.cpu().numpy(), ref.numpy())
    e32 = ratio(g32.numpy(), ref.numpy())
    _record('%s, glorot, GPU branch' % kind, err, {'plain_fp32_same_branch': e32, 'blocks': batch.n_nodes,
                                                   'relations': batch.n_edges,
                                                   'relu_units_flipped_vs_fp64': sum(f[0] for f in flips)})
    assert err <= max(BRANCH_TOL, 4 * e32), (err, e32)


def test_dropout_matches_reference_with_same_mask(eng):
    _use(eng, 'kinkfree')
    batch = _batch('C1 contact')
    n, E = batch.n_nodes, batch.n_edges
    rate, seed = 0.1, 0x1234567855AA77
    dl = _seed(eng, batch, 'random', np.random.default_rng(13))
    _, drel, _, _ = _c_api_rel(eng, batch, dl, rate, seed)
    sc, sq = O.dropout_seeds(seed)
    keep = float(1.0 / (1.0 - np.float32(rate)))
    # the reference runs on the receiver-major relation list: row p's mask elements are p * 160 + c
    c_keep = O.dropout_keep_mask(sc, np.arange(E, dtype=np.uint64)[:, None] * np.uint64(160) + np.arange(150, dtype=np.uint64)[None, :], rate)
    q_keep = O.dropout_keep_mask(sq, np.arange(n, dtype=np.uint64)[:, None] * np.uint64(128) + np.arange(100, dtype=np.uint64)[None, :], rate)
    snd, rcv = _edges(batch)
    ref, _, _ = rel_grads(eng.w64, batch.obj.cpu().double(), snd, rcv, dl.cpu().double(),
                          c_scale=torch.as_tensor(c_keep * keep), q_scale=torch.as_tensor(q_keep * keep))
    err = ratio(drel.cpu().numpy(), ref.numpy())
    _record('C1 contact, kinkfree, dropout 0.1', err)
    assert err <= TOL, err


# ---- B. stage check of k_rel_grad_step / k_rel_grad_enc -------------------------------------------------------------------------
@pytest.mark.parametrize('kind', ['C1 contact', 'fc10 x512', 'ragged', 'jenga18 x64'])
def test_stage_k_rel_grad(eng, kind):
    _use(eng, 'glorot')
    api = eng.api
    batch = _batch(kind)
    n, E = batch.n_nodes, batch.n_edges
    dl = _seed(eng, batch, 'random', np.random.default_rng(14))
    eng.forward(batch, training=True, want_probs=False)
    masks = [m.double() for m in eng.saved_relu_states()]
    _, ws, _, _ = eng._fwd
    _, drel, _, _ = _c_api_rel(eng, batch, dl, ws=ws, with_dobj=False)
    lay = api.workspace_layout(n, E, 1)
    f = ws[:ws.numel() // 4 * 4].view(torch.float32)                  # Engine.ws is grow-only: any byte count

    def arr(name, quads, rows, row0, nrows, cols):
        o = lay[name] // 4
        return f[o:o + quads * rows * 4].view(quads, rows, 4)[:, row0:row0 + nrows].permute(1, 0, 2).reshape(nrows, 4 * quads)[:, :cols].double()
    W = {k: v.double().cuda() for k, v in eng.w64.items()}
    Wa = {k: v.abs() for k, v in W.items()}
    snd, rcv = batch.in_snd[:E].long(), batch.in_rcv[:E].long()
    A = arr('A', 38, E, 0, E, 150)
    ref = torch.zeros(E, dtype=torch.float64, device='cuda')
    absref = torch.zeros_like(ref)
    for l in range(5):
        S, R = arr('S', 38, 5 * n, l * n, n, 150), arr('R', 38, 5 * n, l * n, n, 150)
        dG = arr('dG', 26, 5 * n, l * n, n, 100)
        m1, m2 = masks[6 + 3 * l].cuda(), masks[7 + 3 * l].cuda()
        dH, dHa = dG @ W['rmp.w2'].T, dG.abs() @ Wa['rmp.w2'].T
        G, Ga = m2 * dH[rcv], m2 * dHa[rcv]
        DH1, DH1a = m1 * (G @ W['rmp.w1'].T), m1 * (Ga @ Wa['rmp.w1'].T)
        v = A + 2 * (S[snd] + R[rcv])
        va = A.abs() + 2 * (S[snd].abs() + R[rcv].abs())
        ref += (DH1 * v).sum(1) + G @ W['rmp.b1'] + dG[rcv] @ W['rmp.b2']
        absref += (DH1a * va).sum(1) + Ga @ Wa['rmp.b1'] + dG[rcv].abs() @ Wa['rmp.b2']
    D = arr('GB', 38, E, 0, E, 150)
    obj = batch.obj
    dpos = (obj[rcv, :2] - obj[snd, :2]).double()                      # fp32 difference, as the kernel forms it
    ref += ((D @ W['rm.w0'].T) * dpos).sum(1)
    absref += ((D.abs() @ Wa['rm.w0'].T) * dpos.abs()).sum(1)
    tau = tau_lin(100) + tau_lin(150) + gamma(408)
    got = drel.double()
    assert torch.isfinite(got).all()
    viol = (got - ref).abs() > tau * absref
    assert not bool(viol.any()), (int(viol.sum()), float(((got - ref).abs() / absref.clamp_min(1e-300)).max()), tau)
    _record('stage, %s' % kind, float(((got - ref).abs() / absref.clamp_min(1e-300)).max()), {'tau': tau})


# ---- C. exact properties --------------------------------------------------------------------------------------------------------
def test_exact_properties(eng):
    from spwgnn_b200.graph import _stream_ptr
    from spwgnn_b200._capi import SpwGraph
    _use(eng, 'glorot')
    api = eng.api
    batch = _batch('C1 contact')
    n, E = batch.n_nodes, batch.n_edges
    dl = _seed(eng, batch, 'random', np.random.default_rng(15))
    # dobj equals spw_backward_obj's on the same forward
    _, drel, dobj, ws = _c_api_rel(eng, batch, dl)
    ref_obj = torch.full((n, 3), float('nan'), device='cuda')
    wp = eng.params.c_struct()
    st = _stream_ptr(torch.device('cuda:0'))
    api.check(api.dll.spw_backward_obj(ctypes.byref(wp), ctypes.byref(batch.c_graph), batch.obj.data_ptr(), dl.data_ptr(),
                                       ws.data_ptr(), ws.numel(), 0.0, ref_obj.data_ptr(), st))
    torch.cuda.synchronize()
    assert torch.equal(dobj, ref_obj)
    # reruns, through the C ABI and the Engine: the same bits
    again = _c_api_rel(eng, batch, dl)[1]
    assert torch.equal(again.view(torch.int32), drel.view(torch.int32))
    d_eng, o_eng = eng.relation_gradients(batch, dl)
    assert torch.equal(d_eng.view(torch.int32), drel.view(torch.int32)) and torch.equal(o_eng, dobj)
    # one tower seeded: every other tower's relations exactly 0
    off = batch.node_off_host
    t = 5
    one = torch.zeros_like(dl)
    one[off[t]:off[t + 1]] = dl[off[t]:off[t + 1]]
    d1, _ = eng.relation_gradients(batch, one)
    rcv = batch.in_rcv[:E].long().cpu().numpy()
    mine = (rcv >= off[t]) & (rcv < off[t + 1])
    d1 = d1.cpu().numpy()
    assert np.all(d1[~mine] == 0) and np.abs(d1[mine]).max() > 0
    # n = 0 launches nothing
    empty = SpwGraph(0, 0, 0, None, None, None, None, None, None)
    before = api.dll.spw_launch_count()
    assert api.dll.spw_backward_rel(ctypes.byref(wp), ctypes.byref(empty), None, None, None, 0, 0.0, None, None, None) == 0
    assert api.dll.spw_launch_count() == before
    # no relations: nothing for drel
    nb = _batch('no relations')
    assert nb.n_edges == 0
    dln = _seed(eng, nb, 'random', np.random.default_rng(16))
    eng.forward(nb, training=True, want_probs=False)
    _, wsn, _, _ = eng._fwd
    args = (ctypes.byref(wp), ctypes.byref(nb.c_graph), nb.obj.data_ptr(), dln.data_ptr(), wsn.data_ptr(), wsn.numel(), 0.0)
    launches, _ = _profiled(api, lambda: api.check(api.dll.spw_backward_rel(*args, None, None, st)))
    assert launches == 0
    o1 = torch.empty(nb.n_nodes, 3, device='cuda')
    o2 = torch.empty(nb.n_nodes, 3, device='cuda')
    lo, to = _profiled(api, lambda: api.check(api.dll.spw_backward_obj(*args, o1.data_ptr(), st)))
    lr, tr = _profiled(api, lambda: api.check(api.dll.spw_backward_rel(*args, None, o2.data_ptr(), st)))
    assert lr == lo and not any(x.startswith('k_rel_grad') for x in tr)
    assert torch.equal(o1, o2)


# ---- D. no weight gradient ------------------------------------------------------------------------------------------------------
def test_weight_gradients_are_skipped(eng):
    from spwgnn_b200.graph import _stream_ptr
    _use(eng, 'glorot')
    api = eng.api
    batch = _batch('C1 contact')
    dl = _seed(eng, batch, 'random', np.random.default_rng(18))
    eng.forward(batch, training=True, want_probs=False)
    _, ws, _, _ = eng._fwd
    n, E = batch.n_nodes, batch.n_edges
    dobj = torch.empty(n, 3, device='cuda')
    drel = torch.empty(E, device='cuda')
    wp = eng.params.c_struct()
    st = _stream_ptr(torch.device('cuda:0'))
    args = (ctypes.byref(wp), ctypes.byref(batch.c_graph), batch.obj.data_ptr(), dl.data_ptr(), ws.data_ptr(), ws.numel(), 0.0)
    no, to = _profiled(api, lambda: api.check(api.dll.spw_backward_obj(*args, dobj.data_ptr(), st)))
    nr, tr = _profiled(api, lambda: api.check(api.dll.spw_backward_rel(*args, drel.data_ptr(), dobj.data_ptr(), st)))
    assert nr == no + 6, (nr, no)
    assert 'k_rel_grad_step' in tr and 'k_rel_grad_enc' in tr and 'k_rel_grad_step' not in to
    bad = [t for t in tr if t.startswith('k_wgrad') or t.startswith('k_skinny_c') or t.startswith('k_reduce')]
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
    eng.relation_gradients(other, _seed(eng, other, 'random', np.random.default_rng(20)))
    model.relation_gradients(synth.make_towers('tower', 4, 5, n=7))
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
    res, wsruns, wsfills, rruns, oruns = [], [], [], [], []
    wp = eng.params.c_struct()
    st = _stream_ptr(torch.device('cuda:0'))
    for fill in (0x00, 0xFF):
        wsb = torch.full((nbytes + 2 * G,), fill, dtype=torch.uint8, device='cuda')
        rb = torch.full((E * 4 + 2 * G,), fill, dtype=torch.uint8, device='cuda')
        ob = torch.full((n * 12 + 2 * G,), fill, dtype=torch.uint8, device='cuda')
        logits = torch.empty(n, device='cuda')
        api.check(api.dll.spw_forward(ctypes.byref(wp), ctypes.byref(batch.c_graph), batch.obj.data_ptr(), logits.data_ptr(), None,
                                      wsb.data_ptr() + G, nbytes, 1, 0.0, 0, st))
        before = wsb.clone()
        api.check(api.dll.spw_backward_rel(ctypes.byref(wp), ctypes.byref(batch.c_graph), batch.obj.data_ptr(), dl.data_ptr(),
                                           wsb.data_ptr() + G, nbytes, 0.0, rb.data_ptr() + G, ob.data_ptr() + G, st))
        torch.cuda.synchronize()
        wsruns.append(wsb); wsfills.append(before); rruns.append(rb); oruns.append(ob)
        res.append(rb[G:G + E * 4].view(torch.float32).clone())
    msgs = footprint_violations('drel', rruns, (0x00, 0xFF), G)
    msgs += footprint_violations('dobj', oruns, (0x00, 0xFF), G)
    msgs += footprint_violations('workspace', wsruns, wsfills, G, spans)
    assert not msgs, msgs
    # every float of drel is written: the two fills leave no byte at its fill value in both runs
    assert bool(((rruns[0][G:G + E * 4] != 0x00) | (rruns[1][G:G + E * 4] != 0xFF)).all())
    assert torch.equal(res[0].view(torch.int32), res[1].view(torch.int32))
    for a, b in zip(inputs, snap):
        assert torch.equal(a, b)


# ---- G. facade --------------------------------------------------------------------------------------------------------------
def _main_py_pairs(raw, thr, glue):
    """main.py:66-81 restated on one tower: the (sender m, receiver j) of every active relation column, in column order"""
    pos = raw[:, :2] / 170.0 if glue else raw[:, :2]
    N = len(raw)
    out = []
    for m in range(N):
        for j in range(N):
            if m != j and np.linalg.norm(pos[m] - pos[j]) < thr:
                out.append((m, j))
    return np.array(out, np.int64).reshape(-1, 2)


@pytest.mark.parametrize('case', ['C1 glue', 'C1 contact'])
def test_relation_gradients_facade(eng, case):
    from spwgnn_b200 import synth
    from spwgnn_b200.Networks import PropagationNetwork
    _use(eng, 'kinkfree')
    net = PropagationNetwork()
    net._engine = eng
    model = net.getModel(7)
    towers = synth.make_towers('tower', 16, 23, n=7)
    glue = case == 'C1 glue'
    got = model.relation_gradients(towers, inference_glue=glue)
    assert len(got) == len(towers)
    refs, r32 = [], []
    for (pairs, vals), tw in zip(got, towers):
        exp = _main_py_pairs(np.asarray(tw, np.float64), 170.0, glue)
        assert pairs.dtype == np.int64 and vals.dtype == np.float64 and vals.shape == (len(exp),)
        assert np.array_equal(pairs, exp)
        for dt, acc in ((torch.float64, refs), (torch.float32, r32)):
            w = {k: v.to(dt) for k, v in eng.w64.items()}
            obj = torch.as_tensor((np.asarray(tw, np.float64) / 170.0).astype(np.float32)).to(dt)
            s, r = torch.as_tensor(exp[:, 0]), torch.as_tensor(exp[:, 1])
            _, z = O.forward_sparse(w, obj, s, r, return_logits=True)
            p = torch.sigmoid(z)
            acc.append(rel_grads(w, obj, s, r, p * (1 - p))[0].double().numpy())
    got = np.concatenate([v for _, v in got])
    ref = np.concatenate(refs)
    err, e32 = ratio(got, ref), ratio(np.concatenate(r32), ref)
    _record('relation_gradients, %s' % case, err, {'plain_fp32': e32})
    assert err <= max(TOL, 4 * e32), (err, e32)
