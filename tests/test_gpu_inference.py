"""The inference path against the checked training forward, the head's probabilities and the loss statistics element by
element, the demolish kernels bit for bit, and the bytes every entry point writes against the outputs it declares.

A. Inference = training forward, bit for bit.  spw_forward(training = 0) runs the same kernels, grids and operand order as
   a training forward with dropout rate 0; only the workspace layout differs (the relation encoder ping-pongs X0 = X2 = A,
   X1 = C; [g | p] has two slots, gp_slot(l) = l & 1; U, S, R and H2S one slot; no sign bits or h1).  So logits and probs
   must be torch.equal, and every array inference leaves must equal, byte for byte, the training array it corresponds to:
   Q1, Q, QV, degf, C, A by name, U / S / R / H2S slot 0 = training slot 4, GP slot 0 = training slot 4 ([g^4 | p^4]),
   GP slot 1 = training slot 3.  Both workspaces are filled with 0xFF first, so pad and ones columns and bytes nobody
   writes are compared too.  Checked for direct launches, CUDA-graph replay (also after load_dict and adam_step changed
   the weights in place), predict_towers, a dropout rate passed to inference (ignored: dropout applies only when
   training), and an inference between a training forward and its backward (the gradients must not change).

B. Probabilities.  k_logit_c computes p = 1 / (1 + expf(-z)) in fp32 from its own fp32 logit z.  With u = 2^-24:
   expf is within 2 ulp (CUDA C Programming Guide, single-precision functions), a relative error <= 4 u of e = exp(-z);
   1 + e and the IEEE division are one rounding each, u + u.  sigma = 1 / (1 + e) has relative sensitivity e / (1 + e) <= 1
   to e, so  |p - sigma(z)| <= 6 u sigma(z)  for sigma(z) >= 2^-126 (a normal fp32 result), with sigma(z) evaluated in
   fp64 from the GPU's own logit.  Below that p is subnormal or 0 (expf(-z) overflows for z < -88.72): p must lie in
   [0, 2^-125].  Everywhere 0 <= p <= 1 and no NaN.  And p must lie in test_gpu_stages.prob_interval(z): the fp32 results
   of the add and the division at the smallest and largest fp32 value expf may return (they are correctly rounded, hence
   monotone), which near p = 1 is the fp32 grid itself.  The head bias omp.b1[0] spreads the logits over [-120, 120].

C. Loss statistics (k_bce_grad).  The kernel forms the same p, clips it to [1e-7f, 1.f - 1e-7f] (fp32 constants; the
   upper one is 1 - 2^-23), adds -(y log pc + (1 - y) log(1 - pc)) (logf, 1 ulp: <= 2 u relative) into stats[0] and
   [(p > 0.5) == (y > 0.5)] into stats[1], and writes dlogits.  The kernel's p lies in prob_interval(z) (see B); a relative
   bar cannot decide the upper clip, since 6 u is three times 1 - (1 - 2^-23), but the interval can: p < 1 - 2^-23 exactly
   when fl(1 + expf(-z)) >= 1 + 2^-22, so at most one fp32 logit near z = 15.537 (and one near the lower edge) leaves the
   branch open, and every larger logit must clip.  The per-element loss is monotone in pc, so it lies between its fp64
   values at the two clipped ends of the interval, widened by logf's 2 u |log| and, for y = 0, by the rounding of 1.f - pc
   (u relative, 1.01 u absolute after the log).  The sum adds the double-precision summation term
   (n + 64) 2^-53 (|seed| + sum |loss|).  stats[1] is exact, except for an element whose interval straddles 0.5 (none of
   the crafted ones); z = 0 gives p = 1 / (1 + 1) = 0.5 exactly and counts as not > 0.5.  dlogits: the stage test's bar
   8 u (p + |p - y|) / count, with the branch fixed by the interval (test_gpu_stages.bce_seed_reference).  A CPU test runs
   k_bce_grad restated in fp32 through these references: they must accept it, and reject it without the upper clip of the
   gradient or with the upper clip at 1 - 2e-7.

D. Demolish kernels, bit-exact: the candidate builders against a numpy restatement (a double division by 170 rounded once
   to fp32), spw_tower_sums against a sequential float64 accumulation in block order, its argmin against np.argmin (first
   minimum) with exact ties placed in the same thread, in neighbouring threads and at both ends.

E. Write footprints.  Every output is allocated at exactly its documented size between guard bands of GUARD bytes; the
   sequence forward (inference), forward (training), BCE, backward, edges count and fill runs twice, after filling
   everything with 0x00 and then with 0xFF.  A byte is written if it differs from its fill in either run.  No guard byte
   may be written; every written workspace byte must lie in a named array of its mode or in the packed tensor-core
   operands [0, W2hi); a training forward must leave the backward-only arrays untouched; inputs must be unchanged; and
   every result must be identical between the two runs (a difference means a launch read bytes nobody wrote).

The worst measured ratio (error over bar) of every check of B and C, summaries of A, D and E, and the module's wall time
are written to $SPW_INFER_OUT (default: infer_r04.json in the temporary directory; committed copy: profiles/infer_r04.json).
"""
import contextlib
import ctypes
import json
import os
import tempfile
import time

import numpy as np
import pytest
import torch

from oracle import propnet as O

INFER_OUT = os.environ.get('SPW_INFER_OUT', os.path.join(tempfile.gettempdir(), 'infer_r04.json'))
U = 2.0 ** -24
P_REL = 6 * U
TINY = 2.0 ** -126
GUARD = 4096                      # bytes before and after every output (a multiple of 16: the payload stays aligned)
_RECORD = {}

INF_VS_TRAIN = [('Q1', 'Q1', 0), ('Q', 'Q', 0), ('QV', 'QV', 0), ('degf', 'degf', 0), ('C', 'C', 0), ('A', 'A', 0),
                ('U', 'U', 4), ('S', 'S', 4), ('R', 'R', 4), ('H2S', 'H2S', 4), ('GP', 'GP', 4), ('GP:1', 'GP', 3)]
NODE_QUADS = {'Q1': 26, 'Q': 26, 'QV': 26, 'U': 26, 'S': 38, 'R': 38, 'H2S': 38, 'GP': 50}
BACKWARD_ONLY = ['dU', 'dG', 'T', 'dS', 'dR', 'dH2S', 'DP', 'dQ', 'dQ1', 'dA', 'DH1', 'GB', 'partE', 'part0', 'partN']
FORWARD_TRAINING_ONLY = ['H1', 'EB', 'M1', 'M2']


def _record(section, name, value):
    _RECORD.setdefault(section, {})[name] = value


def _worst(section, name, ratio):
    d = _RECORD.setdefault(section, {})
    d[name] = max(d.get(name, 0.0), float(ratio))


# ---- footprint checker (plain tensors, any device) ---------------------------------------------------------------------------
def workspace_spans(L, n, E, training):
    """(name, first byte, end byte) of every array a workspace of this mode may hold, plus the packed tensor-core operands"""
    from test_host_logic import _workspace_array_floats
    size = _workspace_array_floats(L, n, E)
    spans = [('packed operands', 0, L['W2hi'])]
    for k, floats in size.items():
        if not training and k in BACKWARD_ONLY + FORWARD_TRAINING_ONLY:
            assert L[k] == 0, k
            continue
        spans.append((k, L[k], L[k] + 4 * floats))
    return spans


def footprint_violations(name, runs, fills, guard, spans=None, limit=6):
    """runs: one allocation (uint8: guard, payload, guard) after each run, fills: the byte it was filled with before that run.
    A byte counts as written if it differs from its fill in any run.  Returns messages for written guard bytes and, with
    spans ((name, start, end) byte ranges of the payload), for written payload bytes outside every span; offsets are bytes
    from the start of the payload."""
    written = torch.zeros(runs[0].shape, dtype=torch.bool, device=runs[0].device)
    for r, f in zip(runs, fills):
        written |= r != f
    size = runs[0].numel() - 2 * guard
    out = []
    head = torch.nonzero(written[:guard]).flatten()
    if head.numel():
        out.append('%s: %d bytes written in the guard before the start (first at offset %d)'
                   % (name, head.numel(), int(head[0]) - guard))
    tail = torch.nonzero(written[guard + size:]).flatten()
    if tail.numel():
        out.append('%s: %d bytes written in the guard after the end (first at offset %d, %d bytes past the %d-byte output)'
                   % (name, tail.numel(), size + int(tail[0]), int(tail[0]), size))
    if spans is not None:
        allowed = torch.zeros(size, dtype=torch.bool, device=written.device)
        for _, a, b in spans:
            allowed[a:b] = True
        stray = torch.nonzero(written[guard:guard + size] & ~allowed).flatten()
        if stray.numel():
            brk = torch.nonzero(stray[1:] - stray[:-1] > 1).flatten()
            starts = torch.cat([stray[:1], stray[brk + 1]]).tolist()
            ends = torch.cat([stray[brk], stray[-1:]]).tolist()
            for s, e in list(zip(starts, ends))[:limit]:
                before = [(b, k) for k, a, b in spans if b <= s]
                where = ('%d bytes after the end of %s' % (s - max(before)[0], max(before)[1])) if before else 'before every array'
                out.append('%s: %d bytes written outside every array at offset %d (%s)' % (name, e - s + 1, s, where))
            if len(starts) > limit:
                out.append('%s: %d more stray runs' % (name, len(starts) - limit))
    return out


def test_footprint_checker_names_the_array_and_offset():
    """CPU: a written byte in a gap between two arrays, or in either guard, is reported with the array and the offset."""
    g = 64
    spans = [('packed operands', 0, 32), ('Q', 64, 128), ('U', 128, 160)]
    clean = [torch.full((2 * g + 192,), f, dtype=torch.uint8) for f in (0x00, 0xFF)]
    for r in clean:
        r[g + 64:g + 160] = 7                       # the arrays themselves may be written
    assert footprint_violations('ws', clean, [0x00, 0xFF], g, spans) == []
    gap = [r.clone() for r in clean]
    gap[1][g + 40] = 0                              # a gap byte written in the 0xFF run only
    gap[0][g + 170:g + 174] = 1                     # four bytes after the last array, in the 0x00 run only
    msg = footprint_violations('ws', gap, [0x00, 0xFF], g, spans)
    assert msg == ['ws: 1 bytes written outside every array at offset 40 (8 bytes after the end of packed operands)',
                   'ws: 4 bytes written outside every array at offset 170 (10 bytes after the end of U)'], msg
    grd = [r.clone() for r in clean]
    grd[0][g + 192 + 3] = 9                         # guard after the end
    grd[1][g - 2] = 0                               # guard before the start
    msg = footprint_violations('logits', grd, [0x00, 0xFF], g)
    assert msg == ['logits: 1 bytes written in the guard before the start (first at offset -2)',
                   'logits: 1 bytes written in the guard after the end (first at offset 195, 3 bytes past the 192-byte output)'], msg
    # a span list restated from the layout covers [0, total) with gaps only where the alignment leaves them
    from spwgnn_b200 import build
    from spwgnn_b200._capi import CApi
    api = CApi(build.build())
    for training in (0, 1):
        L = api.workspace_layout(129, 257, training)
        sp = workspace_spans(L, 129, 257, training)
        assert max(b for _, _, b in sp) <= L['total_bytes']
        assert all(a % 16 == 0 for _, a, _ in sp)


# ---- graphs and weights ---------------------------------------------------------------------------------------------------------
def _batch(name):
    """(batch, dropout rate of the stage test) for the stage test's graphs and three more"""
    from spwgnn_b200.graph import TowerBatch
    from spwgnn_b200 import synth
    import test_gpu_stages as S
    if name in S.GRAPHS:
        return S._graph(name)
    if name == 'C5':                        # BASELINE config 5's shape: 8-64 blocks, fully connected, predict glue
        return TowerBatch.sample_jenga(2000, 8, 64, 0xC5, fully_connected=True, inference_glue=True), 0.0
    if name == 'E0':                        # single-block towers only: no relations at all
        return TowerBatch.from_towers(synth.make_towers('jenga', 300, 41, n=1)), 0.0
    if name == 'n1':
        return TowerBatch.from_towers(synth.make_towers('jenga', 1, 42, n=1)), 0.0
    raise ValueError(name)


@pytest.fixture(scope='module', autouse=True)
def _module_record():
    """wall time from the first to the last test of this module; the record is written when a GPU test ran"""
    t0 = time.perf_counter()
    yield
    if not _RECORD:
        return
    _RECORD['_head'] = {'device': torch.cuda.get_device_name(0), 'module_seconds': round(time.perf_counter() - t0, 1)}
    try:
        os.makedirs(os.path.dirname(os.path.abspath(INFER_OUT)), exist_ok=True)
        with open(INFER_OUT, 'w') as f:
            json.dump(_RECORD, f, indent=1, sort_keys=True)
            f.write('\n')
    except OSError:
        pass


@pytest.fixture(scope='module')
def eng():
    from spwgnn_b200.engine import Engine
    assert torch.cuda.is_available()
    return Engine('cuda:0', seed=5)


@contextlib.contextmanager
def graph_limit(eng, limit):
    """Engine.graph_max_edges = limit inside the block (0: direct launches only), restored after it"""
    old = eng.graph_max_edges
    eng.graph_max_edges = limit
    try:
        yield
    finally:
        eng.graph_max_edges = old


def _load(eng, seed):
    eng.params.load_dict(O.init_weights(seed, nonzero_bias=True))
    eng._adam = None


# ---- A. inference = training forward -----------------------------------------------------------------------------------------
def _slot(raw, L, name, n, s, quads, slots):
    o = L[name]
    return raw[o:o + quads * slots * n * 16].view(quads, slots, n * 16)[:, s]


def compare_inference_arrays(api, n, E, ws_inf, ws_train):
    """byte-for-byte comparison of every array inference leaves with its training counterpart: list of messages"""
    Li, Lt = api.workspace_layout(n, E, 0), api.workspace_layout(n, E, 1)
    earr = 4 * Lt['edge_stride_floats']
    out = []
    for inf_name, tr_name, tr_slot in INF_VS_TRAIN:
        if tr_name == 'degf':
            a, b = ws_inf[Li['degf']:Li['degf'] + 4 * n], ws_train[Lt['degf']:Lt['degf'] + 4 * n]
        elif tr_name in ('C', 'A'):
            if E == 0:
                continue
            a, b = ws_inf[Li[tr_name]:Li[tr_name] + earr], ws_train[Lt[tr_name]:Lt[tr_name] + earr]
        else:
            q = NODE_QUADS[tr_name]
            slots = lambda L: 1 if tr_name in ('Q1', 'Q', 'QV') else L['slotsGP'] if tr_name == 'GP' else L['slots']
            a = _slot(ws_inf, Li, tr_name, n, 1 if inf_name == 'GP:1' else 0, q, slots(Li))
            b = _slot(ws_train, Lt, tr_name, n, tr_slot, q, slots(Lt))
        if not torch.equal(a, b):
            d = torch.nonzero(a != b)
            first = d[0].tolist()
            if a.dim() == 2:        # (quad, byte of the slot): name the row and column
                first = 'quad %d row %d column %d' % (first[0], first[1] // 16, 4 * first[0] + first[1] % 16 // 4)
            out.append('%s (training %s slot %d): %d bytes differ, first at %s' % (inf_name, tr_name, tr_slot, d.shape[0], first))
    return out


def _training_reference(eng, api, batch):
    """logits, probs and the workspace of a training forward with dropout rate 0 (workspace pre-filled with 0xFF)"""
    eng.ws.get(api.dll.spw_workspace_bytes(batch.n_nodes, batch.n_edges, 1)).fill_(0xFF)
    logits, probs = eng.forward(batch, training=True, want_probs=True, dropout_rate=0.0)
    return logits.clone(), probs.clone(), eng._fwd[1]


def _check_inference(eng, api, batch, how, label, fails, ref=None):
    """one inference of `batch` (how: 'direct' or 'graph') against the training forward on the current weights"""
    n, E, T = batch.n_nodes, batch.n_edges, batch.n_towers
    tl, tp, tws = ref if ref is not None else _training_reference(eng, api, batch)
    if how == 'direct':
        with graph_limit(eng, 0):
            eng.ws_inf.get(api.dll.spw_workspace_bytes(n, E, 0)).fill_(0xFF)
            logits, probs = eng.forward(batch, training=False, want_probs=True)
        ws = eng.ws_inf.buf
    else:
        assert 0 < E <= 8192
        key = (T, n, E, True)
        with graph_limit(eng, 8192):
            if key not in eng._graphs:
                eng.forward(batch, training=False, want_probs=True)            # capture
            eng._graphs[key][4].fill_(0xFF)
            logits, probs = eng.forward(batch, training=False, want_probs=True)   # replay
        ws = eng._graphs[key][4]
    torch.cuda.synchronize()
    msgs = []
    if not torch.equal(logits, tl):
        msgs.append('logits: %d of %d differ' % (int((logits != tl).sum()), n))
    if not torch.equal(probs, tp):
        msgs.append('probs: %d of %d differ' % (int((probs != tp).sum()), n))
    msgs += compare_inference_arrays(api, n, E, ws, tws)
    fails += ['%s, %s: %s' % (label, how, m) for m in msgs]
    _record('A', '%s %s' % (label, how), 'equal' if not msgs else '%d mismatches' % len(msgs))


A_GRAPHS = ['fc2', 'fc3+1', 'tails', 'fc64', 'contact', 'C2', 'C5', 'E0']


@pytest.mark.gpu
@pytest.mark.parametrize('graph', A_GRAPHS)
def test_inference_equals_the_training_forward(eng, graph):
    from spwgnn_b200._lib import lib
    api = lib()
    batch, _ = _batch(graph)
    n = batch.n_nodes
    hows = ['direct'] + (['graph'] if 0 < batch.n_edges <= 8192 else [])
    fails = []
    _load(eng, 21)
    for how in hows:
        _check_inference(eng, api, batch, how, '%s weights 21' % graph, fails)
    _load(eng, 22)                                      # a second weight set, in place: stale packed operands would show
    for how in hows:
        _check_inference(eng, api, batch, how, '%s weights 22 (load_dict)' % graph, fails)
    tgt = torch.as_tensor((np.random.default_rng(n).random(n) > 0.5).astype(np.float32)).cuda()
    eng.loss_and_grads(batch, tgt)
    eng.adam_step()
    for how in hows:
        _check_inference(eng, api, batch, how, '%s after adam_step' % graph, fails)
    del batch
    torch.cuda.empty_cache()
    assert not fails, '\n'.join(fails)


@pytest.mark.gpu
def test_predict_towers_and_inference_dropout_equal_the_training_forward(eng):
    """predict_towers (inference_glue) through graph replay and direct launches; spw_forward(training = 0) with a dropout
    rate: equal to the training forward at rate 0"""
    from spwgnn_b200 import synth
    from spwgnn_b200.graph import TowerBatch
    from spwgnn_b200.Networks import PropagationNetwork, PropagationModel
    _load(eng, 23)
    net = PropagationNetwork()
    net._engine = eng
    model = PropagationModel(net, 0)
    towers = synth.make_towers('jenga', 7, 51, n=6) + synth.make_towers('jenga', 3, 52, n=11) + synth.make_towers('jenga', 2, 53, n=1)
    batch = TowerBatch.from_towers(towers, inference_glue=True)
    assert 0 < batch.n_edges <= 8192
    _, tp = eng.forward(batch, training=True, want_probs=True)
    tp = tp.cpu().numpy()
    off = batch.node_off_host
    fails = []
    for gme in (8192, 0):
        with graph_limit(eng, gme):
            got = model.predict_towers(towers, inference_glue=True)
        for t, p in enumerate(got):
            if not np.array_equal(p, tp[off[t]:off[t + 1]]):
                fails.append('predict_towers (graph_max_edges %d): tower %d differs' % (gme, t))
    b2, _ = _batch('tails')
    with graph_limit(eng, 0):
        l0, p0 = [x.clone() for x in eng.forward(b2, training=False, want_probs=True)]
        l1, p1 = eng.forward(b2, training=False, want_probs=True, dropout_rate=0.1, dropout_seed=0x1234567)
    tl, tp2 = eng.forward(b2, training=True, want_probs=True, dropout_rate=0.0)
    if not (torch.equal(l0, l1) and torch.equal(p0, p1)):
        fails.append('inference with dropout_rate 0.1 differs from rate 0')
    if not (torch.equal(l0, tl) and torch.equal(p0, tp2)):
        fails.append('tails: direct inference differs from the training forward')
    assert not fails, '\n'.join(fails)


@pytest.mark.gpu
def test_inference_between_forward_and_backward_leaves_the_step_alone(eng):
    """Engine keeps a separate inference workspace so that a predict between a training forward and its backward cannot
    touch the saved state: the gradients must be bit-identical to the same step without the inference calls"""
    bx, rate = _batch('tails')
    by_graph, _ = _batch('fc3+1')
    by_direct, _ = _batch('fc64')
    n = bx.n_nodes
    tgt = torch.as_tensor((np.random.default_rng(3).random(n) > 0.5).astype(np.float32)).cuda()
    _load(eng, 24)

    def step(interleave):
        logits, _ = eng.forward(bx, training=True, want_probs=False, dropout_rate=rate, dropout_seed=77)
        logits = logits.clone()
        if interleave:
            with graph_limit(eng, 8192):
                eng.forward(by_graph, training=False)
                eng.forward(by_direct, training=False)
            with graph_limit(eng, 0):
                eng.forward(by_graph, training=False)
        dl, stats = eng.bce_seed(logits, tgt, n)
        eng.backward(dl)
        torch.cuda.synchronize()
        return logits, eng.grads.flat.clone(), stats.clone()

    l0, g0, s0 = step(False)
    l1, g1, s1 = step(True)
    assert torch.equal(l0, l1)
    assert torch.equal(g0, g1), '%d gradient elements differ after an inference between forward and backward' % int((g0 != g1).sum())
    assert torch.equal(s0[1], s1[1])


# ---- B. probabilities ----------------------------------------------------------------------------------------------------------
def prob_check(z, p):
    """z: fp32 logits, p: fp32 probs (any device).  Returns (messages, worst |p - sigma| / (6 u sigma) over normal sigma)."""
    z64, p64 = z.double(), p.double()
    s = torch.sigmoid(z64)
    msgs = []
    if bool(torch.isnan(p).any()):
        msgs.append('%d NaN probabilities' % int(torch.isnan(p).sum()))
    if bool(((p64 < 0) | (p64 > 1)).any()):
        msgs.append('%d probabilities outside [0, 1]' % int(((p64 < 0) | (p64 > 1)).sum()))
    normal = s >= TINY
    d = (p64 - s).abs()
    ratio = d[normal] / (P_REL * s[normal])
    worst = float(ratio.max()) if ratio.numel() else 0.0
    over = torch.nonzero(normal & (d > P_REL * s)).flatten()
    if over.numel():
        i = int(over[0])
        msgs.append('%d probabilities over 6 u sigma (worst ratio %.3g; first z %r: p %r, sigma %r)'
                    % (over.numel(), worst, float(z[i]), float(p[i]), float(s[i])))
    sub = ~normal & ((p64 < 0) | (p64 > 2 * TINY))
    if bool(sub.any()):
        i = int(torch.nonzero(sub).flatten()[0])
        msgs.append('%d probabilities of sigma < 2^-126 outside [0, 2^-125] (first z %r: p %r)' % (int(sub.sum()), float(z[i]), float(p[i])))
    import test_gpu_stages as S
    p_lo, p_hi = S.prob_interval(z)
    out = (p64 < p_lo) | (p64 > p_hi)
    if bool(out.any()):
        i = int(torch.nonzero(out).flatten()[0])
        msgs.append('%d probabilities outside the interval of the fp32 arithmetic (first z %r: p %r, interval [%r, %r])'
                    % (int(out.sum()), float(z[i]), float(p[i]), float(p_lo[i]), float(p_hi[i])))
    return msgs, worst


@pytest.mark.gpu
@pytest.mark.parametrize('graph', ['contact', 'fc3+1'])
def test_probabilities_elementwise(eng, graph):
    """head bias omp.b1[0] from -120 to 120: every probability against fp64 sigmoid of the GPU's own logit"""
    batch, _ = _batch(graph)
    _load(eng, 25)
    zs, ps = [], []
    with graph_limit(eng, 0 if graph == 'contact' else 8192):          # direct launches / graph replay
        for b in np.linspace(-120.0, 120.0, 97):
            eng.params.views['omp.b1'][0] = float(b)
            logits, probs = eng.forward(batch, training=False, want_probs=True)
            zs.append(logits.clone())
            ps.append(probs.clone())
    z, p = torch.cat(zs), torch.cat(ps)
    msgs, worst = prob_check(z, p)
    _worst('B', 'max |p - sigma| / (6 u sigma), sigma >= 2^-126', worst)
    _record('B', 'elements %s' % graph, {'total': int(z.numel()), 'sigma < 2^-126': int((torch.sigmoid(z.double()) < TINY).sum()),
                                          'p == 0': int((p == 0).sum()), 'p == 1': int((p == 1).sum())})
    assert float(z.min()) < -100 and float(z.max()) > 100
    assert not msgs, '\n'.join(msgs)


# ---- C. BCE statistics -------------------------------------------------------------------------------------------------------
def _bce_logits(n, seed):
    """crafted logits (fp32) and 0 / 1 targets: zeros, +-2^-20, both clip edges, +-100, the rest random"""
    rng = np.random.default_rng(seed)
    special = np.concatenate([np.zeros(16), np.repeat([2.0 ** -20, -2.0 ** -20], 8),
                              np.linspace(-16.14, -16.10, 400), np.linspace(15.50, 15.58, 200), np.linspace(15.93, 16.13, 800),
                              np.repeat([100.0, -100.0, 50.0, -50.0, 20.0, -20.0], 4)])
    z = np.concatenate([special, rng.normal(0, 4, n - special.size)]).astype(np.float32)
    t = np.concatenate([np.arange(special.size) % 2, rng.random(n - special.size) > 0.5]).astype(np.float32)
    t[:16] = np.arange(16) >= 12        # z = 0: 12 targets 0 (counted correct) and 4 targets 1
    return z, t


def _loss64(pc, y):
    return -(y * torch.log(pc) + (1 - y) * torch.log1p(-pc))


def bce_stats_reference(z, t):
    """(loss interval lo, hi, summation magnitude, correct count of the unambiguous elements, ambiguous count) for fp32 logits
    z and 0 / 1 targets t, both float64 tensors; see the module docstring"""
    import test_gpu_stages as S
    p_lo, p_hi = S.prob_interval(z)
    c = lambda p: p.clamp(S.CLIP_LO, S.CLIP_HI)
    la, lb = _loss64(c(p_lo), t), _loss64(c(p_hi), t)
    lmin, lmax = torch.minimum(la, lb), torch.maximum(la, lb)
    e = 2 * U * lmax + torch.where(t > 0.5, torch.zeros_like(z), torch.full_like(z, 1.01 * U))
    lo, hi = float((lmin - e).sum()), float((lmax + e).sum())
    amb = (p_lo <= 0.5) & (p_hi > 0.5)
    correct = ((p_lo > 0.5) == (t > 0.5)) & ~amb
    return lo, hi, float(lmax.abs().sum()), int(correct.sum()), int(amb.sum())


def dlogit_violations(z, t, count, dl):
    """(elements over the bar 8 u absref of test_gpu_stages.bce_seed_reference or NaN, worst |d| / (8 u absref), ambiguous
    clip branches) of the loss seed dl for fp32 logits z and targets t (float64 tensors)"""
    import test_gpu_stages as S
    ref, ab, amb = S.bce_seed_reference(z, t, count, dl)
    d = (dl.double() - ref).abs()
    pos = ab > 0
    worst = float((d[pos] / (8 * U * ab[pos])).max()) if bool(pos.any()) else 0.0
    over = torch.nonzero(torch.isnan(dl) | (d > 8 * U * ab)).flatten()
    return over, worst, int(amb.sum())


def _emulate_bce(z, t, count, hi_clip=None, upper_clip=True):
    """k_bce_grad restated in numpy fp32 (expf as the correctly rounded exp): (dlogits, loss sum, correct count).  hi_clip and
    upper_clip=False give the wrong kernels the CPU test must reject."""
    f32 = np.float32
    eps = f32(1e-7)
    hi = f32(1) - eps if hi_clip is None else f32(hi_clip)
    with np.errstate(over='ignore'):
        e = np.exp(-z.astype(np.float64)).astype(f32)
    p = f32(1) / (f32(1) + e)
    pc = np.minimum(np.maximum(p, eps), hi)
    log32 = lambda x: np.log(x.astype(np.float64)).astype(f32).astype(np.float64)
    loss = -(t * log32(pc) + (1.0 - t) * log32(f32(1) - pc))
    inside = (p > eps) & (p < hi) if upper_clip else (p > eps)
    dl = np.where(inside, ((pc - t.astype(f32)).astype(np.float64) * (1.0 / count)).astype(f32), f32(0))
    return dl, float(loss.sum()), int(((p > 0.5) == (t > 0.5)).sum())


def test_loss_references_reject_a_wrong_clip():
    """CPU: the dlogits and stats references accept k_bce_grad restated in fp32 on the crafted logits and reject it without
    the upper clip of the gradient, or with the upper clip at 1 - 2e-7"""
    n, count = 3000, 3005.0
    z, t = _bce_logits(n, n)
    z64, t64 = torch.from_numpy(z).double(), torch.from_numpy(t).double()
    lo, hi, _, correct, amb = bce_stats_reference(z64, t64)
    dl, loss, right = _emulate_bce(z, t, count)
    over, _, namb = dlogit_violations(z64, t64, count, torch.from_numpy(dl))
    assert over.numel() == 0 and lo <= loss <= hi and correct <= right <= correct + amb
    assert namb <= 2, namb                                          # at most one fp32 logit per edge is ambiguous
    dl, _, _ = _emulate_bce(z, t, count, upper_clip=False)
    over, _, _ = dlogit_violations(z64, t64, count, torch.from_numpy(dl))
    assert over.numel() >= 400 and float(z64[over].min()) > 15.5     # the upper-edge logits, +20, +50 and +100 with y = 0
    _, loss, _ = _emulate_bce(z, t, count, hi_clip=1 - 2e-7)
    assert not lo <= loss <= hi, (lo, loss, hi)


@pytest.mark.gpu
@pytest.mark.parametrize('n', [3000, 1500])
def test_bce_statistics_at_the_clip_edges(eng, n):
    """n > 256 rows of one CTA (12 and 6 CTAs), stats pre-seeded: the call adds into them"""
    import test_gpu_stages as S
    from spwgnn_b200._lib import lib
    api = lib()
    z, t = _bce_logits(n, n)
    zg, tg = torch.from_numpy(z).cuda(), torch.from_numpy(t).cuda()
    seed = torch.tensor([12.375, 7.0], dtype=torch.float64, device='cuda')
    stats = seed.clone()
    dl = torch.full((n,), float('nan'), dtype=torch.float32, device='cuda')
    count = float(n + 5)
    api.check(api.dll.spw_bce_grad(zg.data_ptr(), tg.data_ptr(), n, count, dl.data_ptr(), stats.data_ptr(),
                                   torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    z64, t64 = zg.double(), tg.double()
    lo, hi, mag, correct, amb = bce_stats_reference(z64, t64)
    got0, got1 = float(stats[0]), float(stats[1])
    summ = (n + 64) * 2.0 ** -53 * (abs(float(seed[0])) + mag)
    lo, hi = lo + float(seed[0]) - summ, hi + float(seed[0]) + summ
    mid, half = (lo + hi) / 2, (hi - lo) / 2
    _worst('C', 'stats[0], crafted + bulk: |got - mid| / half-width', abs(got0 - mid) / half)
    _worst('C', 'stats[0]: interval half-width / loss sum', half / mag)
    assert lo <= got0 <= hi, 'stats[0] = %r outside [%r, %r]' % (got0, lo, hi)
    base = float(seed[1]) + correct
    _record('C', 'stats[1] n=%d' % n, {'got': got1, 'exact part': base, 'ambiguous': amb})
    assert base <= got1 <= base + amb, (got1, base, amb)
    # z = 0 exactly: p = 0.5, not > 0.5; the count of the z = 0 elements alone
    z0 = z == 0
    assert z0.sum() == 16
    one = torch.zeros(2, dtype=torch.float64, device='cuda')
    api.check(api.dll.spw_bce_grad(zg.data_ptr(), tg.data_ptr(), 16, count, dl.data_ptr(), one.data_ptr(),
                                   torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    assert float(one[1]) == float((t[:16] < 0.5).sum()), ('z = 0 must count as p = 0.5, not > 0.5', float(one[1]))
    # dlogits (the stage test's bar, fp32 clip constants, either branch near an edge)
    api.check(api.dll.spw_bce_grad(zg.data_ptr(), tg.data_ptr(), n, count, dl.data_ptr(), stats.data_ptr(),
                                   torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    over, worst, namb = dlogit_violations(z64, t64, count, dl)
    _worst('C', 'dlogits: max |d| / (8 u absref)', worst)
    _record('C', 'dlogits: ambiguous clip branch, n=%d' % n, namb)
    assert over.numel() == 0, ('dlogits over the bar', over.numel(), float(z[int(over[0])]), float(dl[int(over[0])]))
    # a reference with the clip at 1 - 1e-7 in double passes the gradient where the kernel (1 - 2^-23) clips it
    p = torch.sigmoid(z64)
    old = (p > 1e-7) & (p < 1 - 1e-7) & (dl == 0)
    _record('C', 'elements a clip at 1 - 1e-7 (double) gets wrong, n=%d' % n, int(old.sum()))
    # the unclipped bulk alone (the clip-edge elements dominate the interval above): a sharper stats[0]
    S0 = 1456                                               # crafted logits first (_bce_logits); 1456 * 4 bytes keeps 16-byte alignment
    bulk = torch.zeros(2, dtype=torch.float64, device='cuda')
    api.check(api.dll.spw_bce_grad(zg.data_ptr() + 4 * S0, tg.data_ptr() + 4 * S0, n - S0, count, dl.data_ptr(), bulk.data_ptr(),
                                   torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    lo, hi, mag, correct, amb = bce_stats_reference(z64[S0:], t64[S0:])
    summ = (n + 64) * 2.0 ** -53 * mag
    lo, hi = lo - summ, hi + summ
    got0 = float(bulk[0])
    _worst('C', 'stats[0], unclipped bulk: |got - mid| / half-width', abs(got0 - (lo + hi) / 2) / ((hi - lo) / 2))
    assert lo <= got0 <= hi, ('stats[0] of the bulk', got0, lo, hi)
    assert correct <= float(bulk[1]) <= correct + amb


# ---- D. demolish kernels ---------------------------------------------------------------------------------------------------------
def _bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint64 if a.dtype == np.float64 else np.uint32)


def _raw(N, seed):
    rng = np.random.default_rng(seed)
    return np.stack([rng.integers(400, 1100, N) + rng.random(N), rng.integers(40, 600, N) + rng.random(N),
                     rng.integers(50, 300, N).astype(np.float64)], 1)


@pytest.mark.gpu
@pytest.mark.parametrize('N', [2, 9, 64])
def test_candidates_remove_bit_exact(N):
    from spwgnn_b200._lib import lib
    api = lib()
    raw = _raw(N, N)
    idx = np.array([[k if k < c else k + 1 for k in range(N - 1)] for c in range(N)], dtype=np.int64).reshape(-1)
    for glue in (0, 1):
        obj = torch.full((N * (N - 1), 3), float('nan'), dtype=torch.float32, device='cuda')
        pos = torch.full((N * (N - 1), 2), float('nan'), dtype=torch.float64, device='cuda')
        r = torch.from_numpy(raw).cuda()
        api.check(api.dll.spw_candidates_remove(r.data_ptr(), N, obj.data_ptr(), pos.data_ptr(), glue, torch.cuda.current_stream().cuda_stream))
        src = raw[idx]
        assert np.array_equal(_bits(obj.cpu().numpy()), _bits((src / 170.0).astype(np.float32)))
        assert np.array_equal(_bits(pos.cpu().numpy()), _bits(src[:, :2] / 170.0 if glue else src[:, :2]))


@pytest.mark.gpu
@pytest.mark.parametrize('N,K', [(5, 1), (9, 100), (63, 5000)])
def test_candidates_drop_bit_exact(N, K):
    """(63, 5000): 320 000 items, more than one pass of the grid-stride loop (grid_for caps the grid at 8 CTAs per SM)"""
    from spwgnn_b200._lib import lib
    api = lib()
    raw = _raw(N, N + K)
    rng = np.random.default_rng(K)
    poses = np.stack([rng.random(K) * 700 + 400, rng.random(K) * 600], 1)
    width = 150.0
    ref = np.concatenate([np.concatenate([[[poses[c, 0], poses[c, 1], width]], raw]) for c in range(K)])
    for glue in (0, 1):
        obj = torch.full((K * (N + 1), 3), float('nan'), dtype=torch.float32, device='cuda')
        pos = torch.full((K * (N + 1), 2), float('nan'), dtype=torch.float64, device='cuda')
        r, ps = torch.from_numpy(raw).cuda(), torch.from_numpy(poses).cuda()
        api.check(api.dll.spw_candidates_drop(r.data_ptr(), N, ps.data_ptr(), K, width, obj.data_ptr(), pos.data_ptr(), glue,
                                              torch.cuda.current_stream().cuda_stream))
        assert np.array_equal(_bits(obj.cpu().numpy()), _bits((ref / 170.0).astype(np.float32)))
        assert np.array_equal(_bits(pos.cpu().numpy()), _bits(ref[:, :2] / 170.0 if glue else ref[:, :2]))


def tower_sums_reference(probs, node_off):
    """sequential float64 accumulation in block order per tower (not np.sum, which adds pairwise); 0.0 for an empty tower"""
    out = np.zeros(len(node_off) - 1)
    for t in range(len(node_off) - 1):
        a, b = node_off[t], node_off[t + 1]
        if b > a:
            out[t] = np.add.accumulate(probs[a:b].astype(np.float64))[-1]
    return out


def _tower_sums(api, probs, node_off, want_argmin=True):
    p = torch.from_numpy(np.ascontiguousarray(probs, dtype=np.float32)).cuda()
    no = torch.from_numpy(np.asarray(node_off, dtype=np.int32)).cuda()
    T = len(node_off) - 1
    sums = torch.full((T,), float('nan'), dtype=torch.float64, device='cuda')
    amin = torch.full((1,), -7, dtype=torch.int32, device='cuda')
    api.check(api.dll.spw_tower_sums(p.data_ptr(), no.data_ptr(), T, sums.data_ptr(), amin.data_ptr() if want_argmin else None,
                                     torch.cuda.current_stream().cuda_stream))
    return sums.cpu().numpy(), int(amin.item())


@pytest.mark.gpu
def test_tower_sums_bit_exact():
    from spwgnn_b200._lib import lib
    api = lib()
    rng = np.random.default_rng(11)
    sizes = rng.integers(0, 65, 3000)
    sizes[:5] = 0                       # empty towers, including the first
    sizes[-1] = 0
    node_off = np.concatenate([[0], np.cumsum(sizes)])
    # magnitudes from 1e-30 to 1: the sum's rounding depends on the order of the additions
    probs = (rng.random(node_off[-1]) * 10.0 ** rng.integers(-30, 1, node_off[-1])).astype(np.float32)
    probs[rng.random(probs.size) < 0.05] = 1.0
    got, amin = _tower_sums(api, probs, node_off)
    ref = tower_sums_reference(probs, node_off)
    assert np.array_equal(_bits(got), _bits(ref)), int((got != ref).sum())
    assert amin == int(np.argmin(ref))
    assert np.all(got[sizes == 0] == 0.0)
    pairwise = np.array([probs[a:b].astype(np.float64).sum() for a, b in zip(node_off[:-1], node_off[1:])])
    _record('D', 'towers where np.sum (pairwise) differs from the block-order sum', int((pairwise != ref).sum()))


@pytest.mark.gpu
@pytest.mark.parametrize('T', [1, 2, 255, 256, 257, 5000])
def test_argmin_first_minimum_with_ties(T):
    """one block per tower, so sums[t] = probs[t]; exact ties in the same thread (t, t + 256), in neighbouring threads
    (t, t + 1) and at both ends (0, T - 1)"""
    from spwgnn_b200._lib import lib
    api = lib()
    rng = np.random.default_rng(T)
    node_off = np.arange(T + 1)
    places = [(0, T - 1)] + [(t, t + 1) for t in (0, 37, 127, 128, 254, T - 2)] + [(t, t + 256) for t in (0, 3, 200, T - 257)]
    places += [(T - 1, T - 1)]
    for a, b in places:
        if not (0 <= a < T and 0 <= b < T):
            continue
        for pattern in ('pair', 'pair + later'):
            v = (0.5 + 0.5 * rng.random(T)).astype(np.float32)
            v[a] = v[b] = 0.25
            if pattern == 'pair + later' and b + 1 < T:
                v[b + 1:][rng.random(T - b - 1) < 0.1] = 0.25      # more copies of the minimum after the pair
            got, amin = _tower_sums(api, v, node_off)
            assert amin == int(np.argmin(got)) == int(np.argmin(v.astype(np.float64))) == a, (T, a, b, pattern, amin)


@pytest.mark.gpu
def test_score_removals_ties_and_sums(eng):
    """score_removals end to end: its sums bit-identical to the block-order restatement on the engine's own probabilities of
    the same candidate batch; two identical neighbouring blocks give two identical candidates (a real tie), and a tower of
    identical blocks ties every candidate, so the argmin must be 0.  33 blocks: each candidate has 32 * 31 = 992 relations,
    a multiple of 32, so every candidate's relations start at the same offset within the edge step's 32-row chunks."""
    from spwgnn_b200._lib import lib
    from spwgnn_b200.graph import TowerBatch
    from spwgnn_b200.Networks import PropagationNetwork, PropagationModel
    api = lib()
    _load(eng, 26)
    net = PropagationNetwork()
    net._engine = eng
    model = PropagationModel(net, 0)
    N = 33
    base = _raw(N, 99)
    base[7] = base[6]
    for label, tower in (('two identical blocks', base), ('all blocks identical', np.repeat(base[:1], N, 0))):
        sums, amin = model.score_removals(tower, inference_glue=True)
        raw = torch.from_numpy(np.ascontiguousarray(tower)).cuda()
        obj = torch.empty(N * (N - 1), 3, dtype=torch.float32, device='cuda')
        pos = torch.empty(N * (N - 1), 2, dtype=torch.float64, device='cuda')
        api.check(api.dll.spw_candidates_remove(raw.data_ptr(), N, obj.data_ptr(), pos.data_ptr(), 1, torch.cuda.current_stream().cuda_stream))
        node_off = np.arange(N + 1) * (N - 1)
        batch = TowerBatch.from_poses(obj, node_off, pos, max_nodes=N - 1)
        _, probs = eng.forward(batch, training=False)
        ref = tower_sums_reference(probs.cpu().numpy(), node_off)
        assert np.array_equal(_bits(sums), _bits(ref)), label
        assert amin == int(np.argmin(ref)), label
        if label == 'two identical blocks':
            assert sums[6] == sums[7], (label, sums[6], sums[7])
        else:
            assert np.all(sums == sums[0]) and amin == 0, (label, amin)


# ---- E. write footprints ----------------------------------------------------------------------------------------------------------
class Guarded:
    """a device allocation of exactly `nbytes` between two guard bands; .ptr is the payload (16-byte aligned)"""

    def __init__(self, name, nbytes, spans=None):
        self.name, self.nbytes, self.spans = name, int(nbytes), spans
        self.raw = torch.empty(2 * GUARD + self.nbytes, dtype=torch.uint8, device='cuda')
        self.ptr = self.raw.data_ptr() + GUARD
        assert self.ptr % 16 == 0

    @property
    def payload(self):
        return self.raw[GUARD:GUARD + self.nbytes]


def _run_footprint(api, eng, batch, rate, tgt, allocs, fill, grads_struct):
    """one pass of the sequence with every allocation filled with `fill`; returns (snapshots, messages)"""
    n, E, T = batch.n_nodes, batch.n_edges, batch.n_towers
    a = allocs
    st = torch.cuda.current_stream().cuda_stream
    for g in a.values():
        g.raw.fill_(fill)
    a['stats'].payload.zero_()                                       # spw_bce_grad adds into stats: zeroed by the caller
    wp = eng.params.c_struct()
    gr = batch.c_graph
    msgs = []
    inputs = {'weights': eng.params.flat, 'obj': batch.obj, 'target': tgt, 'node_off': batch.node_off, 'in_off': batch.in_off,
              'in_snd': batch.in_snd, 'in_rcv': batch.in_rcv, 'out_off': batch.out_off, 'out_pos': batch.out_pos,
              'pos': batch._keep[0]}
    before = {k: v.clone() for k, v in inputs.items()}
    api.check(api.dll.spw_forward(ctypes.byref(wp), ctypes.byref(gr), batch.obj.data_ptr(), a['logits (inference)'].ptr,
                                  a['probs (inference)'].ptr, a['workspace (inference)'].ptr, a['workspace (inference)'].nbytes,
                                  0, 0.0, 0, st))
    wst = a['workspace (training)']
    api.check(api.dll.spw_forward(ctypes.byref(wp), ctypes.byref(gr), batch.obj.data_ptr(), a['logits'].ptr, a['probs'].ptr,
                                  wst.ptr, wst.nbytes, 1, float(rate), 0x9E3779B97F4A7C15, st))
    torch.cuda.synchronize()
    L = api.workspace_layout(n, E, 1)
    from test_host_logic import _workspace_array_floats
    size = _workspace_array_floats(L, n, E)
    for k in BACKWARD_ONLY:
        seg = wst.payload[L[k]:L[k] + 4 * size[k]]
        if bool((seg != fill).any()):
            msgs.append('training forward wrote %d bytes of the backward-only array %s' % (int((seg != fill).sum()), k))
    api.check(api.dll.spw_bce_grad(a['logits'].ptr, tgt.data_ptr(), n, float(n), a['dlogits'].ptr, a['stats'].ptr, st))
    torch.cuda.synchronize()
    dl_before = a['dlogits'].payload.clone()
    api.check(api.dll.spw_backward(ctypes.byref(wp), ctypes.byref(gr), batch.obj.data_ptr(), a['dlogits'].ptr, wst.ptr, wst.nbytes,
                                   ctypes.byref(grads_struct), float(rate), st))
    pos = batch._keep[0]
    ptr = lambda k: a[k].ptr
    api.check(api.dll.spw_edges_count(pos.data_ptr(), batch.node_off.data_ptr(), T, n, batch.max_nodes, 170.0, 0, ptr('deg_out'),
                                      ptr('deg_in'), ptr('edge_off'), st))
    api.check(api.dll.spw_edges_fill(pos.data_ptr(), batch.node_off.data_ptr(), T, n, batch.max_nodes, 170.0, 0, ptr('edge_off'),
                                     ptr('snd'), ptr('rcv'), ptr('slot'), ptr('in_off'), ptr('in_snd'), ptr('in_rcv'), ptr('out_off'),
                                     ptr('out_pos'), st))
    torch.cuda.synchronize()
    if not torch.equal(dl_before, a['dlogits'].payload):
        msgs.append('spw_backward changed its input dlogits')
    for k, v in inputs.items():
        if not torch.equal(before[k], v):
            msgs.append('input %s changed' % k)
    return {k: g.raw.clone() for k, g in a.items()}, msgs


FOOTPRINT_SHAPES = ['fc2', 'fc3+1', 'tails', 'E0', 'n1', 'fc64', 'C2']


@pytest.mark.gpu
@pytest.mark.parametrize('shape', FOOTPRINT_SHAPES)
def test_write_footprints(eng, shape):
    from spwgnn_b200._lib import lib
    from spwgnn_b200._capi import CApi, PARAM_SPECS
    api = lib()
    batch, rate = _batch(shape)
    n, E, T = batch.n_nodes, batch.n_edges, batch.n_towers
    _load(eng, 27)
    tgt = torch.as_tensor((np.random.default_rng(n).random(n) > 0.5).astype(np.float32)).cuda()
    # edge count of the distance test (the outputs of spw_edges_fill are sized from it)
    pos = batch._keep[0]
    eo = torch.empty(T + 1, dtype=torch.int32, device='cuda')
    dg = torch.empty(max(n, 1), dtype=torch.int32, device='cuda')
    api.check(api.dll.spw_edges_count(pos.data_ptr(), batch.node_off.data_ptr(), T, n, batch.max_nodes, 170.0, 0, dg.data_ptr(),
                                      dg.data_ptr(), eo.data_ptr(), torch.cuda.current_stream().cuda_stream))
    Ef = int(eo[T].item())
    allocs = {}

    def add(name, nbytes, spans=None):
        allocs[name] = Guarded(name, nbytes, spans)

    for training, name in ((0, 'workspace (inference)'), (1, 'workspace (training)')):
        L = api.workspace_layout(n, E, training)
        add(name, api.dll.spw_workspace_bytes(n, E, training), workspace_spans(L, n, E, training))
    for k in ('logits (inference)', 'probs (inference)', 'logits', 'probs', 'dlogits'):
        add(k, 4 * n)
    add('stats', 16)
    for k, shp in PARAM_SPECS:
        add('grad ' + k, 4 * int(np.prod(shp)))
    for k in ('deg_out', 'deg_in'):
        add(k, 4 * n)
    add('edge_off', 4 * (T + 1))
    for k in ('snd', 'rcv', 'slot', 'in_snd', 'in_rcv', 'out_pos'):
        add(k, 4 * Ef)
    for k in ('in_off', 'out_off'):
        add(k, 4 * (n + 1))
    gs = CApi.params([allocs['grad ' + k].ptr for k, _ in PARAM_SPECS])
    runs, fails = [], []
    for fill in (0x00, 0xFF):
        snap, msgs = _run_footprint(api, eng, batch, rate, tgt, allocs, fill, gs)
        runs.append(snap)
        fails += ['fill 0x%02X: %s' % (fill, m) for m in msgs]
    written = {}
    for k, g in allocs.items():
        fails += footprint_violations(k, [r[k] for r in runs], [0x00, 0xFF], GUARD, g.spans)
        if g.spans is None:
            p0, p1 = runs[0][k][GUARD:GUARD + g.nbytes], runs[1][k][GUARD:GUARD + g.nbytes]
            if k == 'stats':        # stats[0]: a double atomicAdd per CTA, in no fixed order; stats[1] counts exactly
                s0, s1 = p0.view(torch.float64), p1.view(torch.float64)
                same = bool(s0[1] == s1[1]) and abs(float(s0[0] - s1[0])) <= 1e-12 * abs(float(s0[0]))
            else:
                same = torch.equal(p0, p1)
            if not same:
                fails.append('%s differs between the 0x00 and the 0xFF run (%d bytes): a launch read bytes nobody wrote'
                             % (k, int((p0 != p1).sum())))
            written[k] = int(((p0 != 0x00) | (p1 != 0xFF)).sum())
    for k in ('workspace (inference)', 'workspace (training)'):
        written[k] = int(((runs[0][k] != 0x00) | (runs[1][k] != 0xFF)).sum())
    _record('E', shape, {'n': n, 'E': E, 'edges_fill_E': Ef, 'violations': len(fails),
                         'workspace bytes written (inference, training)': [written['workspace (inference)'], written['workspace (training)']]})
    # every exactly-sized output that must be written in full was
    for k in ('logits', 'probs', 'logits (inference)', 'probs (inference)', 'dlogits'):
        if written[k] != 4 * n:
            fails.append('%s: %d of %d bytes written' % (k, written[k], 4 * n))
    del runs, allocs
    torch.cuda.empty_cache()
    assert not fails, '\n'.join(fails)
