"""spw_backward_inputs / Engine.input_gradients / PropagationModel.input_gradients: the gradient of the predictions with
respect to every input of the reference's model (objects, sender_relations, receiver_relations, propagation).

A. fp64 parity against input_grad_ref.input_grads (autograd of the per-tower restatement of oracle.propnet.forward_dense),
   max|d| / max|ref| per output tensor (drs, drr, drr_free, dprop), kink-free weights, bar 1e-5: the reference's own dicts
   (tests/golden), C1 (predict glue and contact relations), 512 fully connected 10-block towers, a ragged 0/1/2/7/13/32/64-block
   batch and 64 Jenga-18 towers, each with a fixed random seed and with the BCE seed.  Glorot weights on the GPU's relu branch
   (the 21 saved relu states of a training forward of the same batch, whose logits the gradient's forward equals bit for bit):
   a 512-tower C2 slice, a 256-tower C3 slice and a 512-tower C4 slice; every unit whose state differs from fp64's has
   |pre-activation| < 2e-5; bar max(2e-5, 4 e32) per tensor, e32 the error of a plain fp32 evaluation of the same branch.
A2. Stage check, elementwise |got - ref| <= tau absref (absref: the same contraction on absolute values).
   * The h2 recompute (k_lin<150, 150> on the kept h1, masked by the saved bits), step 0, which the scratch holds after the
     pass, on its own fp32 input H1: tau_lin(150).  It lies on the saved relu branch: exactly 0 where the bit is clear, and
     positive where it is set except at units whose fp64 value is itself within that bar of 0 (a recompute cannot reproduce
     the sign of a unit the forward found within rounding of its kink; their count is recorded).
   * drs, drr and drr_free against the formula of spw_input_grad.cuh in fp64 on the workspace's own fp32 S, R, dG (every step),
     H1, D_e (GB), obj and h2_0 (the scratch) and the saved relu bits.  dSh2 and DH1 of each step are overwritten by the next
     step, so they are rebuilt in fp64 from dG (dSh2 = dG.W3^T, one k_lin with K = 100; DH1 = relu'(h1) * ((relu'(h2) *
     dSh2[r]).W2^T), k_edge_dgrad_c with K = 150), and h2 from H1 (k_lin with K = 150): tau_lin(100) + 2 tau_lin(150).  The
     kernels' own arithmetic: per step one sequential chain of at most 450 fmas (150 for drs, 300 for drr) plus the add of
     <dG, b3> (itself a 100-fma chain), one add into the output per step launch (five), and the encoder term (a 150-fma chain
     u_e, one fma, one add): every term carries at most 450 + 100 + 5 + 153 roundings, gamma_708.  Bar:
     tau = tau_lin(100) + 2 tau_lin(150) + gamma_708.
   * drs[s_e, e] + drr[r_e, e] against spw_backward_rel's drel on the same workspace, elementwise: both are within their own
     bars of fp64 evaluations that differ by <DH1, H1 - (A + S + R)> (two roundings of the stored h1), so
     |sum - drel| <= (tau + gamma_1) absref_inputs + (tau_rel + gamma_2) absref_rel, tau_rel the bar of test_gpu_rel_grad.
B. Exact properties: dobj equals spw_backward_obj's bit for bit on the same forward; reruns are bit-identical; n = 0 launches
   nothing.
C. No weight gradient: spw_backward_obj's launches plus 17 (one k_zero_message; per step the h2 recompute and
   k_input_grad_step; in step 0 the V1c product, the sender / receiver sums and two products into d prop; k_input_grad_enc;
   k_dprop_rows), and no k_wgrad_*, k_skinny_c or k_reduce_* tag.
D. Isolation and memory: Engine.input_gradients between Engine.forward(training=True) and Engine.backward leaves the weight
   gradients bit-identical.  Write footprints (test_gpu_inference.footprint_violations) with 0x00 / 0xFF fills: every output,
   the scratch and the workspace lie between guard bands nobody writes; every float of every output is written and both runs
   give the same bits; inside the workspace every written byte lies in the backward pass's data-gradient arrays
   (BACKWARD_ARRAYS), among them the ones this pass uses beyond spw_backward_obj's: DH1 (also written in step 0) and the dS / dR
   slot 0 (step 0's sender / receiver sums); every other byte, the forward state included, is unchanged.
E. Facade: PropagationModel.input_gradients on the reference's dicts, and on one whose active columns are not the leading
   slots, against autograd of oracle.propnet.forward_dense with respect to all four inputs (K.gradients with grad_ys = dprobs),
   bar max(1e-5, 4 e32) with e32 the error of a plain fp32 evaluation; a nonzero propagation and a wrongly shaped dprobs raise.

The worst ratios are written to $SPW_INPUT_GRAD_OUT (default: input_grad_parity.json in the temporary directory).
"""
import ctypes
import json
import os
import tempfile

import numpy as np
import pytest
import torch

from oracle import propnet as O
from input_grad_ref import input_grads
from test_gpu_obj_grad import _batch, _edges, _profiled, _seed, _use

pytestmark = pytest.mark.gpu
OUT = os.environ.get('SPW_INPUT_GRAD_OUT', os.path.join(tempfile.gettempdir(), 'input_grad_parity.json'))
TOL = 1e-5
BRANCH_TOL = 2e-5
FLIP_MARGIN = 2e-5
U32 = 2.0 ** -24
_WORST = {}
GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden')
NAMES = ('drs', 'drr', 'drr_free', 'dprop')


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
                json.dump({'device': torch.cuda.get_device_name(0), 'worst': _WORST}, f, indent=1, sort_keys=True)
                f.write('\n')
        except OSError:
            pass


def gamma(k):
    return k * U32 / (1 - k * U32)


def tau_lin(K):
    """test_gpu_stages.tau_lin: the elementwise bar of one k_lin / k_edge_dgrad_c contraction of length K"""
    return 2.5 * 2.0 ** -21 + np.ceil(K / 8) * 2.0 ** -22 + 4 * U32


def ratio(got, ref):
    got, ref = np.asarray(got, np.float64), np.asarray(ref, np.float64)
    if ref.size == 0:
        return 0.0
    m, d = np.abs(ref).max(), np.abs(got - ref).max()
    return float(d / m) if m > 0 else (0.0 if d == 0 else float('inf'))


def _golden_batch(name):
    from spwgnn_b200.graph import TowerBatch
    d = np.load(os.path.join(GOLDEN, name + '.npz'))
    return TowerBatch.from_dense_relations(d['objects'], d['sender_relations'], d['receiver_relations'])


def _c_api(eng, batch, dl, ws, nbytes, outs, scratch, with_dobj=True):
    from spwgnn_b200.graph import _stream_ptr
    api, E = eng.api, batch.n_edges
    drs, drr, free, dprop, dobj = outs
    wp = eng.params.c_struct()
    api.check(api.dll.spw_backward_inputs(ctypes.byref(wp), ctypes.byref(batch.c_graph), batch.max_nodes, batch.obj.data_ptr(),
                                          dl.data_ptr(), ws.data_ptr(), nbytes, 0.0, scratch.data_ptr(), scratch.numel(),
                                          drs.data_ptr() if E else None, drr.data_ptr() if E else None, free.data_ptr(),
                                          dprop.data_ptr(), dobj.data_ptr() if with_dobj else None, _stream_ptr(torch.device('cuda:0'))))
    torch.cuda.synchronize()


def _training_forward(eng, batch):
    from spwgnn_b200.graph import _stream_ptr
    api, n, E = eng.api, batch.n_nodes, batch.n_edges
    nbytes = int(api.dll.spw_workspace_bytes(n, E, 1))
    ws = torch.full((nbytes,), 0xFF, dtype=torch.uint8, device='cuda')
    logits = torch.empty(max(n, 1), device='cuda')
    wp = eng.params.c_struct()
    api.check(api.dll.spw_forward(ctypes.byref(wp), ctypes.byref(batch.c_graph), batch.obj.data_ptr(), logits.data_ptr(), None,
                                  ws.data_ptr(), nbytes, 1, 0.0, 0, _stream_ptr(torch.device('cuda:0'))))
    torch.cuda.synchronize()
    _training_forward.logits = logits[:n]
    return ws, nbytes


def _outputs(batch):
    n, E, mx = batch.n_nodes, batch.n_edges, batch.max_nodes
    nan = lambda *shape: torch.full(shape, float('nan'), device='cuda')
    return [nan(max(E, 1), mx), nan(max(E, 1), mx), nan(n), nan(n, 100), nan(n, 3)]


def _backward_obj(eng, batch, dl, ws, nbytes):
    from spwgnn_b200.graph import _stream_ptr
    dobj = torch.full((max(batch.n_nodes, 1), 3), float('nan'), device='cuda')
    wp = eng.params.c_struct()
    eng.api.check(eng.api.dll.spw_backward_obj(ctypes.byref(wp), ctypes.byref(batch.c_graph), batch.obj.data_ptr(), dl.data_ptr(),
                                               ws.data_ptr(), nbytes, 0.0, dobj.data_ptr(), _stream_ptr(torch.device('cuda:0'))))
    torch.cuda.synchronize()
    return dobj[:batch.n_nodes]


# ---- A. fp64 parity -----------------------------------------------------------------------------------------------------------
KINDS = ['golden predict_jenga_n5', 'golden predict_jenga_n9', 'golden train_n7', 'golden train_n9',
         'C1', 'C1 contact', 'fc10 x512', 'ragged', 'jenga18 x64']


@pytest.mark.parametrize('seed_kind', ['random', 'bce'])
@pytest.mark.parametrize('kind', KINDS)
def test_parity_kinkfree(eng, kind, seed_kind):
    _use(eng, 'kinkfree')
    batch = _golden_batch(kind.split()[1]) if kind.startswith('golden') else _batch(kind)
    dl = _seed(eng, batch, seed_kind, np.random.default_rng(11))
    got = eng.input_gradients(batch, dl)
    snd, rcv = _edges(batch)
    ref = input_grads(eng.w64, batch.obj.cpu().double(), batch.node_off_host, snd.numpy(), rcv.numpy(), dl.cpu().double().numpy())
    Nm = ref[0].shape[1]
    for k in range(4):
        g = got[k].cpu().numpy()
        if k < 2:
            assert not g[:, Nm:].any()
            g = g[:, :Nm]
        err = ratio(g, ref[k].numpy())
        _WORST.setdefault('%s, kinkfree' % kind, {})[NAMES[k]] = max(err, _WORST.get('%s, kinkfree' % kind, {}).get(NAMES[k], 0.0))
        assert err <= TOL, (kind, NAMES[k], err)


def _slice(kind):
    from spwgnn_b200 import synth
    from spwgnn_b200.graph import TowerBatch
    if kind == 'C2 x512':
        return TowerBatch.from_towers(synth.make_towers('jenga', 512, 1235, n=10), fully_connected=True)
    if kind == 'C3 x256':
        return TowerBatch.from_towers(synth.make_towers('jenga18', 256, 31))
    return _batch(kind)


@pytest.mark.parametrize('kind', ['C2 x512', 'C3 x256', 'C4 x512'])
def test_parity_glorot_on_gpu_branch(eng, kind):
    _use(eng, 'glorot')
    batch = _slice(kind)
    lt, _ = eng.forward(batch, training=True, want_probs=False)
    lt = lt.clone()
    masks = [m.cpu() for m in eng.saved_relu_states()]
    dl = _seed(eng, batch, 'random', np.random.default_rng(12))
    ws, nbytes = _training_forward(eng, batch)
    assert torch.equal(_training_forward.logits, lt)
    outs = _outputs(batch)
    scratch = torch.empty(int(eng.api.dll.spw_backward_inputs_bytes(batch.n_nodes, batch.n_edges)), dtype=torch.uint8, device='cuda')
    _c_api(eng, batch, dl, ws, nbytes, outs, scratch)
    snd, rcv = _edges(batch)
    obj32 = batch.obj.cpu()
    args = (batch.node_off_host, snd.numpy(), rcv.numpy())
    ref = input_grads(eng.w64, obj32.double(), *args, dl.cpu().double().numpy(), masks=masks)
    w32 = {k: v.float() for k, v in eng.w64.items()}
    r32 = input_grads(w32, obj32, *args, dl.cpu().numpy(), masks=masks)
    maxpre = max(f[1] for f in ref[6])
    assert maxpre < FLIP_MARGIN, maxpre
    Nm = ref[0].shape[1]
    rec = {'relu_units_flipped_vs_fp64': sum(f[0] for f in ref[6]), 'blocks': batch.n_nodes, 'relations': batch.n_edges}
    bad = []
    for k in range(4):
        g = outs[k][:batch.n_edges].cpu().numpy() if k < 2 else outs[k].cpu().numpy()
        if k < 2:
            g = g[:, :Nm]
        err, e32 = ratio(g, ref[k].numpy()), ratio(r32[k].double().numpy(), ref[k].numpy())
        rec[NAMES[k]] = err; rec[NAMES[k] + '_plain_fp32_same_branch'] = e32
        if not err <= max(BRANCH_TOL, 4 * e32):
            bad.append((NAMES[k], err, e32))
    _WORST['%s, glorot, GPU branch' % kind] = rec
    assert not bad, bad


# ---- A2. stage check ------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('kind', ['C1 contact', 'fc10 x512', 'ragged', 'jenga18 x64'])
def test_stage_input_grad(eng, kind):
    from spwgnn_b200.graph import _stream_ptr
    _use(eng, 'glorot')
    api = eng.api
    batch = _batch(kind)
    n, E, mx = batch.n_nodes, batch.n_edges, batch.max_nodes
    dl = _seed(eng, batch, 'random', np.random.default_rng(14))
    eng.forward(batch, training=True, want_probs=False)
    masks = [m.double().cuda() for m in eng.saved_relu_states()]
    _, ws, _, _ = eng._fwd
    nbytes = ws.numel()
    outs = _outputs(batch)
    sb = int(api.dll.spw_backward_inputs_bytes(n, E))
    scratch = torch.empty(sb, dtype=torch.uint8, device='cuda')
    _c_api(eng, batch, dl, ws, nbytes, outs, scratch, with_dobj=False)
    drel = torch.full((max(E, 1),), float('nan'), device='cuda')
    wp = eng.params.c_struct()
    api.check(api.dll.spw_backward_rel(ctypes.byref(wp), ctypes.byref(batch.c_graph), batch.obj.data_ptr(), dl.data_ptr(),
                                       ws.data_ptr(), nbytes, 0.0, drel.data_ptr(), None, _stream_ptr(torch.device('cuda:0'))))
    torch.cuda.synchronize()
    lay = api.workspace_layout(n, E, 1)
    f = ws[:ws.numel() // 4 * 4].view(torch.float32)
    sf = scratch.view(torch.float32)

    def slab(base, off, quads, rows, row0, nrows, cols):
        return base[off:off + quads * rows * 4].view(quads, rows, 4)[:, row0:row0 + nrows].permute(1, 0, 2).reshape(nrows, 4 * quads)[:, :cols].double()

    def arr(name, quads, rows, row0, nrows, cols, extra=0):
        return slab(f, lay[name] // 4 + extra, quads, rows, row0, nrows, cols)
    W = {k: v.double().cuda() for k, v in eng.w64.items()}
    Wa = {k: v.abs() for k, v in W.items()}
    snd, rcv = batch.in_snd[:E].long(), batch.in_rcv[:E].long()
    off = torch.as_tensor(batch.node_off_host, device='cuda')
    t_e = torch.searchsorted(off, rcv, right=True) - 1
    t_n = torch.searchsorted(off, torch.arange(n, device='cuda'), right=True) - 1
    Nt = (off[1:] - off[:-1])[t_e]
    jj = torch.arange(mx, device='cuda')
    valid = jj[None, :] < Nt[:, None]                                            # (E, mx)
    blk = torch.where(valid, off[t_e][:, None] + jj[None, :], torch.zeros((), dtype=torch.long, device='cuda'))
    h_ld = 38 * E * 4 + 64                                                       # floats per H1 slot
    # the h2 recompute of step 0 (the scratch keeps the last step processed) on its own fp32 input, and its sign pattern
    h2 = slab(sf, 0, 38, E, 0, E, 150)
    H1 = arr('H1', 38, E, 0, E, 152)
    hr = masks[7] * (H1[:, :150] @ W['rmp.w1'] + W['rmp.b1'])
    ha = masks[7] * (H1[:, :150].abs() @ Wa['rmp.w1'] + Wa['rmp.b1'])
    hv = (h2 - hr).abs() > tau_lin(150) * ha
    assert not bool(hv.any()), int(hv.sum())
    on = masks[7] > 0
    assert bool((h2[~on] == 0).all())                                           # exactly 0 off the saved branch
    kink = on & (h2 <= 0)                                                        # on it: positive, but for units within rounding of 0
    assert bool((hr[kink].abs() <= tau_lin(150) * ha[kink]).all())
    sign_kinks = int(kink.sum())
    # h2_0 (k_zero_message, plain fp32 chains) against fp64
    h20_off = (38 * E * 4 + 64 + 63) // 64 * 64
    h20 = sf[h20_off:h20_off + 150].double()
    x = torch.relu(W['rm.b0'])
    for li in (1, 2, 3):
        x = torch.relu(x @ W['rm.w%d' % li] + W['rm.b%d' % li])
    x = torch.relu(torch.relu(x @ W['rmp.w0'][:150] + W['rmp.b0']) @ W['rmp.w1'] + W['rmp.b1'])
    assert ratio(h20.cpu().numpy(), x.cpu().numpy()) <= 1e-5
    # drs, drr, drr_free: the kernels' formula on the workspace's own inputs
    rs = torch.zeros(E, mx, dtype=torch.float64, device='cuda'); rr = torch.zeros_like(rs)
    rsa, rra = torch.zeros_like(rs), torch.zeros_like(rs)
    fr, fra = torch.zeros(n, dtype=torch.float64, device='cuda'), torch.zeros(n, dtype=torch.float64, device='cuda')
    rel, rela = torch.zeros(E, dtype=torch.float64, device='cuda'), torch.zeros(E, dtype=torch.float64, device='cuda')
    A = arr('A', 38, E, 0, E, 150)
    for l in range(5):
        S, R = arr('S', 38, 5 * n, l * n, n, 150), arr('R', 38, 5 * n, l * n, n, 150)
        dG = arr('dG', 26, 5 * n, l * n, n, 100)
        m1, m2 = masks[6 + 3 * l].cuda(), masks[7 + 3 * l].cuda()
        dH, dHa = dG @ W['rmp.w2'].T, dG.abs() @ Wa['rmp.w2'].T
        G, Ga = m2 * dH[rcv], m2 * dHa[rcv]
        DH1, DH1a = m1 * (G @ W['rmp.w1'].T), m1 * (Ga @ Wa['rmp.w1'].T)
        H1l = arr('H1', 38, E, 0, E, 150, extra=l * h_ld)
        h2l = m2 * (H1l @ W['rmp.w1'] + W['rmp.b1'])
        h2la = m2 * (H1l.abs() @ Wa['rmp.w1'] + Wa['rmp.b1'])
        gb, gba = dG @ W['rmp.b2'], dG.abs() @ Wa['rmp.b2']
        rs += torch.einsum('ec,ejc->ej', DH1, S[blk]); rsa += torch.einsum('ec,ejc->ej', DH1a, S[blk].abs())
        rr += torch.einsum('ec,ejc->ej', DH1, R[blk]) + torch.einsum('ec,ejc->ej', h2l, dH[blk]) + gb[blk]
        rra += (torch.einsum('ec,ejc->ej', DH1a, R[blk].abs()) + torch.einsum('ec,ejc->ej', h2la, dHa[blk]) + gba[blk])
        fr += dH @ h20 + gb; fra += dHa @ h20.abs() + gba
        v = A + 2 * (S[snd] + R[rcv]); va = A.abs() + 2 * (S[snd].abs() + R[rcv].abs())
        rel += (DH1 * v).sum(1) + G @ W['rmp.b1'] + dG[rcv] @ W['rmp.b2']
        rela += (DH1a * va).sum(1) + Ga @ Wa['rmp.b1'] + dG[rcv].abs() @ Wa['rmp.b2']
    D = arr('GB', 38, E, 0, E, 150)
    u, ua = D @ W['rm.w0'].T, D.abs() @ Wa['rm.w0'].T                          # (E, 2)
    xy = batch.obj[:, :2].double()
    enc, enca = torch.einsum('ek,ejk->ej', u, xy[blk]), torch.einsum('ek,ejk->ej', ua, xy[blk].abs())
    rs -= enc; rr += enc; rsa += enca; rra += enca
    dpos = (batch.obj[rcv, :2] - batch.obj[snd, :2]).double()
    rel += (u * dpos).sum(1); rela += (ua * dpos.abs()).sum(1)
    zero = torch.zeros((), dtype=torch.float64, device='cuda')
    rs, rr, rsa, rra = [torch.where(valid, t, zero) for t in (rs, rr, rsa, rra)]
    tau = tau_lin(100) + 2 * tau_lin(150) + gamma(708)
    worst = {}
    for name, got, ref, absref in (('drs', outs[0][:E], rs, rsa), ('drr', outs[1][:E], rr, rra), ('drr_free', outs[2], fr, fra)):
        got = got.double()
        assert torch.isfinite(got).all(), name
        viol = (got - ref).abs() > tau * absref
        assert not bool(viol.any()), (name, int(viol.sum()), tau)
        worst[name] = float(((got - ref).abs() / absref.clamp_min(1e-300)).max()) if got.numel() else 0.0
    if E:
        k = torch.arange(E, device='cuda')
        sl, rl = snd - off[t_e], rcv - off[t_e]
        s = outs[0][k, sl].double() + outs[1][k, rl].double()
        sa = rsa[k, sl] + rra[k, rl]
        tau_rel = tau_lin(100) + tau_lin(150) + gamma(408)
        bar = (tau + gamma(1)) * sa + (tau_rel + gamma(2)) * rela
        viol = (s - drel[:E].double()).abs() > bar
        assert not bool(viol.any()), ('drs + drr vs drel', int(viol.sum()))
        worst['drs+drr vs drel, share of bar'] = float(((s - drel[:E].double()).abs() / bar.clamp_min(1e-300)).max())
    worst['tau'] = tau
    worst['h2 units on the saved branch within rounding of 0'] = sign_kinks
    _WORST['stage, %s' % kind] = worst


# ---- B. exact properties ----------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize('kind', ['C1 contact', 'ragged', 'no relations'])
def test_exact_properties(eng, kind):
    from spwgnn_b200.engine import PropNetObjFunction
    _use(eng, 'glorot')
    batch = _batch(kind)
    dl = _seed(eng, batch, 'random', np.random.default_rng(13))
    a = eng.input_gradients(batch, dl)
    b = eng.input_gradients(batch, dl)
    for x, y in zip(a, b):
        assert torch.equal(x.view(torch.int32), y.view(torch.int32))
    obj = batch.obj.detach().clone().requires_grad_(True)
    PropNetObjFunction.apply(obj, eng, batch).backward(dl)
    assert torch.equal(a[4].view(torch.int32), obj.grad.view(torch.int32))


def test_empty_batch_launches_nothing(eng):
    from spwgnn_b200._capi import SpwGraph
    api = eng.api
    p = eng.params.c_struct()
    empty = SpwGraph(0, 0, 0, None, None, None, None, None, None)
    before = api.dll.spw_launch_count()
    assert api.dll.spw_backward_inputs(ctypes.byref(p), ctypes.byref(empty), 0, None, None, None, 0, 0.0, None, 0, None, None,
                                       None, None, None, None) == 0
    assert api.dll.spw_launch_count() == before


# ---- C. no weight gradient, launch count ----------------------------------------------------------------------------------------
def test_no_weight_gradient_launches(eng):
    _use(eng, 'glorot')
    batch = _batch('C1 contact')
    assert batch.n_edges > 0
    dl = _seed(eng, batch, 'random', np.random.default_rng(18))
    ws, nbytes = _training_forward(eng, batch)
    n, E, mx = batch.n_nodes, batch.n_edges, batch.max_nodes
    outs = [torch.empty(E, mx, device='cuda'), torch.empty(E, mx, device='cuda'), torch.empty(n, device='cuda'),
            torch.empty(n, 100, device='cuda'), torch.empty(n, 3, device='cuda')]
    scratch = torch.empty(int(eng.api.dll.spw_backward_inputs_bytes(n, E)), dtype=torch.uint8, device='cuda')
    no, to = _profiled(eng.api, lambda: _backward_obj(eng, batch, dl, ws, nbytes))
    ni, ti = _profiled(eng.api, lambda: _c_api(eng, batch, dl, ws, nbytes, outs, scratch))
    assert ni == no + 17, (no, ni)
    for tag in ti:
        assert not tag.startswith(('k_wgrad', 'k_skinny', 'k_reduce')), tag
    for tag in ('k_zero_message', 'k_input_grad_step', 'k_input_grad_enc', 'k_dprop_rows', 'k_lin:h2'):
        assert tag in ti, (tag, ti)


# ---- D. isolation and memory -------------------------------------------------------------------------------------------------------
def test_isolation_from_training_step(eng):
    from spwgnn_b200.Networks import PropagationNetwork
    _use(eng, 'glorot')
    batch = _batch('C1 contact')
    dl = _seed(eng, batch, 'random', np.random.default_rng(19))
    eng.forward(batch, training=True, want_probs=False, dropout_rate=0.1, dropout_seed=7)
    g0 = eng.backward(dl).flat.clone()
    net = PropagationNetwork()
    net._engine = eng
    d = np.load(os.path.join(GOLDEN, 'train_n7.npz'))
    other = _batch('fc10 x512')
    eng.forward(batch, training=True, want_probs=False, dropout_rate=0.1, dropout_seed=7)
    eng.input_gradients(other, _seed(eng, other, 'random', np.random.default_rng(20)))
    net.getModel(7).input_gradients({'objects': d['objects'], 'sender_relations': d['sender_relations'],
                                     'receiver_relations': d['receiver_relations']})
    g1 = eng.backward(dl).flat.clone()
    assert torch.equal(g0.view(torch.int32), g1.view(torch.int32))


BACKWARD_ARRAYS = ('dU', 'dG', 'T', 'dS', 'dR', 'dH2S', 'DP', 'dQ', 'dQ1', 'dA', 'DH1', 'GB')


@pytest.mark.parametrize('kind', ['C1 contact', 'ragged'])
def test_write_footprints(eng, kind):
    from test_gpu_inference import footprint_violations
    from spwgnn_b200.graph import _stream_ptr
    _use(eng, 'glorot')
    api = eng.api
    batch = _batch(kind)
    dl = _seed(eng, batch, 'random', np.random.default_rng(20))
    n, E, mx = batch.n_nodes, batch.n_edges, batch.max_nodes
    nbytes = int(api.dll.spw_workspace_bytes(n, E, 1))
    lay = api.workspace_layout(n, E, 1)
    ends = sorted(set(v for k, v in lay.items() if k in api.dll.spw_workspace_layout_names().decode().split(',')[:40]) | {nbytes})
    spans = [(k, lay[k], min(e for e in ends if e > lay[k])) for k in BACKWARD_ARRAYS]
    G = 4096
    names = ('drs', 'drr', 'drr_free', 'dprop', 'dobj', 'scratch')
    sizes = [E * mx * 4, E * mx * 4, n * 4, n * 400, n * 12, int(api.dll.spw_backward_inputs_bytes(n, E))]
    inputs = [batch.obj, dl, batch.in_off, batch.out_off, batch.out_pos, batch.in_snd, batch.in_rcv, batch.node_off]
    snap = [t.clone() for t in inputs]
    wp = eng.params.c_struct()
    st = _stream_ptr(torch.device('cuda:0'))
    runs, wsruns, wsfills = [], [], []
    for fill in (0x00, 0xFF):
        wsb = torch.full((nbytes + 2 * G,), fill, dtype=torch.uint8, device='cuda')
        logits = torch.empty(max(n, 1), device='cuda')
        api.check(api.dll.spw_forward(ctypes.byref(wp), ctypes.byref(batch.c_graph), batch.obj.data_ptr(), logits.data_ptr(), None,
                                      wsb.data_ptr() + G, nbytes, 1, 0.0, 0, st))
        torch.cuda.synchronize()
        before = wsb.clone()
        bufs = [torch.full((sz + 2 * G,), fill, dtype=torch.uint8, device='cuda') for sz in sizes]
        views = [b[G:G + sz].view(torch.float32).reshape(shape) for b, sz, shape in
                 zip(bufs, sizes, [(E, mx), (E, mx), (n,), (n, 100), (n, 3), (-1,)])]
        _c_api(eng, batch, dl, wsb[G:G + nbytes], nbytes, views[:5], bufs[5][G:G + sizes[5]])
        runs.append((bufs, [v.clone() for v in views[:5]]))
        wsruns.append(wsb); wsfills.append(before)
    msgs = []
    for i, name in enumerate(names):
        msgs += footprint_violations(name, [r[0][i] for r in runs], (0x00, 0xFF), G)
    # the workspace: every written byte lies in the data-gradient arrays; the forward state and the rest are unchanged
    msgs += footprint_violations('workspace', wsruns, wsfills, G, spans)
    assert not msgs, msgs
    for i in range(5):   # every byte of every output is written: no byte keeps its fill in both runs; both runs give the same bits
        assert bool(((runs[0][0][i][G:G + sizes[i]] != 0x00) | (runs[1][0][i][G:G + sizes[i]] != 0xFF)).all()), names[i]
        assert torch.equal(runs[0][1][i].view(torch.int32), runs[1][1][i].view(torch.int32)), names[i]
    # the arrays this pass writes beyond spw_backward_obj's are among the spans: DH1 (step 0) and dS / dR slot 0
    written = (wsruns[0][G:G + nbytes] != wsfills[0][G:G + nbytes]) | (wsruns[1][G:G + nbytes] != wsfills[1][G:G + nbytes])
    if E:
        for k in ('DH1', 'dS', 'dR'):
            assert bool(written[lay[k]:lay[k] + 16 * n].any()), k
    for a, b in zip(inputs, snap):
        assert torch.equal(a, b)


# ---- E. facade ----------------------------------------------------------------------------------------------------------------
def _dense_ref(w, objects, rs, rr, dprobs, dt):
    B, N, _ = objects.shape
    ins = [torch.as_tensor(a).to(dt).clone().requires_grad_(True) for a in (objects, rs, rr, np.zeros((B, N, O.PROP_DIM)))]
    wd = {k: v.to(dt) for k, v in w.items()}
    p = O.forward_dense(wd, *ins)
    return [g.double().numpy() for g in torch.autograd.grad((p * torch.as_tensor(dprobs).to(dt)).sum(), ins)]


@pytest.mark.parametrize('name', ['predict_jenga_n5', 'predict_jenga_n9', 'train_n4', 'train_n7', 'train_n7 permuted slots'])
def test_input_gradients_facade(eng, name):
    from spwgnn_b200.Networks import PropagationNetwork
    from spwgnn_b200._lib import SpwError
    _use(eng, 'kinkfree')
    d = np.load(os.path.join(GOLDEN, name.split()[0] + '.npz'))
    objects, rs, rr = d['objects'], d['sender_relations'], d['receiver_relations']
    if name.endswith('permuted slots'):    # active columns off the leading slots: the device scatter goes through slot_list
        perm = np.random.default_rng(3).permutation(rs.shape[2])
        rs, rr = rs[:, :, perm], rr[:, :, perm]
        assert not np.array_equal(rs, d['sender_relations'])
    B, N, R = rs.shape
    net = PropagationNetwork()
    net._engine = eng
    model = net.getModel(N)
    x = {'objects': objects, 'sender_relations': rs, 'receiver_relations': rr, 'propagation': np.zeros((B, N, 100))}
    dprobs = np.random.default_rng(5).standard_normal((B, N, 1))
    got = model.input_gradients(x, dprobs)
    assert sorted(got) == sorted(x)
    o32 = objects.astype(np.float32)
    ref = _dense_ref(eng.w64, o32.astype(np.float64), rs, rr, dprobs, torch.float64)
    r32 = _dense_ref(eng.w64, o32, rs, rr, dprobs, torch.float32)
    for k, key in enumerate(('objects', 'sender_relations', 'receiver_relations', 'propagation')):
        assert got[key].dtype == np.float32 and got[key].shape == x[key].shape
        err, e32 = ratio(got[key], ref[k]), ratio(r32[k], ref[k])
        _WORST.setdefault('facade, %s' % name, {})[key] = err
        assert err <= max(TOL, 4 * e32), (key, err, e32)
    ones = model.input_gradients({k: v for k, v in x.items() if k != 'propagation'})
    assert np.array_equal(ones['objects'], model.input_gradients(x, np.ones((B, N)))['objects'])
    with pytest.raises(SpwError):
        model.input_gradients(dict(x, propagation=np.ones((B, N, 100))))
    with pytest.raises(SpwError):
        model.input_gradients(x, np.ones((B, N + 1, 1)))
