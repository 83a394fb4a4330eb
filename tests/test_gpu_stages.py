"""Every launch of a training step against an fp64 evaluation of that one launch on the GPU's own fp32 inputs.

A training step leaves almost all of its intermediates in the caller-owned workspace (spw_workspace_layout names them).  Each
array is the output of one launch, or of a short chain of launches, applied to arrays that are also in the workspace.  So
every launch is checked in isolation, at its real shape, grid, layout and PDL overlap, against the same operation evaluated
in float64 on the device from the GPU's fp32 inputs, relu states and saved sign bits.  Relu kinks cannot amplify anything
here, so no kink escapes are needed, and the bars are close to fp32 rounding.  The workspace is filled with 0xFF bytes
(NaN) before every checked step: a NaN in a checked array means a launch read memory nobody wrote, and fails the test
naming the array.  The forward arrays are read again after the backward pass and must be unchanged.

Bars (u = 2^-24, the fp32 unit roundoff; absref = the same contraction on absolute values, times the post-factor):

* bit-exact where the launch is a fixed sequence of fp32 adds, relus or single multiplies: h1 = relu((A + S[snd]) + R[rcv])
  (k_edge_step_c's operand build), dU_4 (k_logit_bwd_c), DP = (((dU_0 + dU_1) + dU_2) + dU_3) + dU_4 (k_sum_slots_c), the
  ones and pad columns, sign bits against the GPU's own stored values, dropout zeros, S_0 = R_0 = p_0 = 0.
* fma: the layer-0 encoders are two fused multiply-adds, two roundings: |d| <= 2 u sum|terms|.  The head (k_logit_c) is a
  chain of 100 fmas and one add: |d| <= 101 u sum|terms| (the worst-case bound of a sequential sum).
* GEMM (k_lin, 3xTF32 on tcgen05): |got - ref| <= tau_lin(K) absref elementwise, and got == 0 exactly where absref == 0.
  tau_lin(K) = 2.5 * 2^-21 + ceil(K / 8) * 2^-22 + 4 u, from the accumulation structure:
    - split: hi = rna_tf32(x), lo = x - hi with |lo| <= 2^-11 |x|; the tensor core truncates lo to tf32 (split_fast), an error
      <= 2^-21 |x| on either operand, and the dropped lo.lo product is <= 2^-22 |a b|: 2.5 * 2^-21 of sum|a b|;
    - the MMAs of one k-step (8 products) are added into the fp32 accumulator with truncation: assuming the tensor core's
      internal sum of the products loses at most one more truncation, 2 * 2^-23 = 2^-22 of the magnitude of the partial sum
      (<= absref) per k-step of the main (hi.hi) pass; the correction pass works on values 2^-11 smaller and is covered by
      the slack below;
    - epilogue: bias (or rowscale fma), addend, post-scale and accumulate are one round-to-nearest each: 4 u.
  K = 100 / 150 / 200 gives tau = 4.6e-6 / 6.1e-6 / 7.6e-6.  tanh epilogues add 4 u |ref| (tanhf is within 2 ulp), and a
  (1 - m^2) multiplier adds 2 u of the pre-multiplier magnitude (1 - fl(m m) is off by <= u m^2 + u |1 - m^2| <= 2 u).
  The forward GEMM stages must also hold max|d| / max|ref| < 2e-6, the bar test_gpu_csl.py holds k_lin to.  For the two
  tanh stages (g, p) the denominator is the largest pre-activation: the bar belongs to the GEMM, and tanh is 1-Lipschitz, so
  an error of the product shows in g at most at its own size.  (g sums up to 63 relations, its pre-activations reach ~10
  where tanh saturates; measured against max|g| <= 1 the ratio is 1e-5 with every element inside its elementwise bar.)
* segmented sum (H2S, k_edge_step_c + k_seg_fix_c): the GEMM bar plus (5 + chunks + 1) u for the warp scan (5 levels) and
  k_seg_fix_c's chunk sum (chunks = ceil(max in-degree / 32) + 1).  A sign bit of h2 may differ from fp64 only where
  |pre| <= tau_lin(150) (|h1| |W2| + |b2|).  The sums over the in- / out-edges of d h1 (k_gather_dsr_c) are sequential:
  max degree u.
* wgrad (k_wgrad_c / k_wgrad_pair + the fixed-order reduction): tau_wg(M) = 2.5 * 2^-21 + 16 * 2^-22 + (t + launches + 27) u:
  the split as above; 16 truncating k-steps per 128-row tile (the tile sums are then added with round-to-nearest, so the
  truncations of the tiles add up to 16 * 2^-22 of sum|x dy|); t = ceil(tiles / 74) round-to-nearest running-sum adds per
  CTA (74 = row streams of the CTA-pair kernel, the fewest); one add per launch into the partials (the five step launches of
  rmp layer 1); the reduction of <= 148 partials in 8 sub-sums of <= 19 and one sum of the 8: 27 adds.
* skinny weight gradients (k_skinny_c + reduction): 8 fmas per lane, 5 shuffle levels, ceil(warps / 8) + 8 reduction adds:
  tau_sk(M) = (22 + ceil(ceil(M / 256) / 8)) u.
* composite (a stage whose input the step overwrote, rebuilt here in fp64 from the GPU's own earlier array): the sum of the
  stages' tau, with absref carried through the chain on absolute values.

Per stage and graph (the worst layer and step) the maximum |d| / absref, tau, the normwise error and the mean least-squares
shrink 1 - (got.ref)/(ref.ref) are written to $SPW_STAGES_OUT (default: stages_r03.json in the temporary directory;
committed copy: profiles/stages_r03.json), one line per stage.  The shrink is recorded, not asserted.
"""
import json
import math
import os
import re
import tempfile
import time

import numpy as np
import pytest
import torch

from oracle import propnet as O

pytestmark = pytest.mark.gpu
STAGES_OUT = os.environ.get('SPW_STAGES_OUT', os.path.join(tempfile.gettempdir(), 'stages_r03.json'))
U = 2.0 ** -24
TANH_REL = 4 * U
FWD_NORMWISE = 2e-6
_RECORD = {}
_CHECKED = set()          # stage names checked in this run (the coverage guard reads it)


def tau_lin(K):
    return 2.5 * 2.0 ** -21 + math.ceil(K / 8) * 2.0 ** -22 + 4 * U


def tau_wg(M, launches=1):
    tiles = math.ceil(math.ceil(M / 128) / 74)
    return 2.5 * 2.0 ** -21 + 16 * 2.0 ** -22 + (tiles + launches + 27) * U


def tau_sk(M):
    return (22 + math.ceil(math.ceil(M / 256) / 8)) * U


# ---- readers ---------------------------------------------------------------------------------------------------------------
class Workspace:
    """Views of the workspace the last training forward used (Engine._fwd), as (rows, cols) tensors."""

    def __init__(self, api, eng):
        batch, ws, _, _ = eng._fwd
        self.n, self.E = batch.n_nodes, batch.n_edges
        self.L = api.workspace_layout(self.n, self.E, 1)
        self.raw = ws
        self.f = ws[:ws.numel() // 4 * 4].view(torch.float32)
        n = self.n
        self.rows = {'Q1': n, 'Q': n, 'QV': n, 'DP': n, 'dQ': n, 'dQ1': n, 'dH2S': n, 'GP': 5 * n, 'U': 5 * n, 'S': 5 * n,
                     'R': 5 * n, 'H2S': 5 * n, 'dU': 5 * n, 'dG': 5 * n, 'T': 4 * n, 'dS': 4 * n, 'dR': 4 * n}

    def _csl(self, base, rows_alloc, row0, nrows, col0, cols):
        q0, q1 = col0 // 4, (col0 + cols + 3) // 4
        a = self.f[base + q0 * rows_alloc * 4:base + q1 * rows_alloc * 4].view(q1 - q0, rows_alloc, 4)[:, row0:row0 + nrows]
        return a.permute(1, 0, 2).reshape(nrows, 4 * (q1 - q0))[:, :cols].clone()

    def node(self, name, cols, slot=0, col0=0):
        """slot `slot` (rows slot * n ..) of a node array [quads][rows_alloc][4]"""
        return self._csl(self.L[name] // 4, self.rows[name], slot * self.n, self.n, col0, cols)

    def edge(self, name, cols=152, step=None):
        base = self.L[name] // 4 + (step * self.L['edge_stride_floats'] if step is not None else 0)
        return self._csl(base, self.E, 0, self.E, 0, cols)

    def bits(self, name, i, nbytes=19):
        """sign-bit array i of a group: byte-slab u8 [20][bits_rows] -> bool (E, 8 * nbytes)"""
        rows = self.L['bits_rows']
        off = self.L[name] + i * 4 * self.L['bits_floats']
        b = self.raw[off:off + 20 * rows].view(20, rows)[:nbytes, :self.E]
        sh = torch.arange(8, device=b.device, dtype=torch.uint8)
        return ((b.unsqueeze(-1) >> sh) & 1).bool().permute(1, 0, 2).reshape(self.E, 8 * nbytes)

    def forward_state(self):
        """raw bytes of every array the forward pass leaves for the backward pass"""
        out = {}
        for k, nq in [('Q1', 25), ('Q', 26), ('QV', 26), ('GP', 50), ('U', 26), ('S', 38), ('R', 38), ('H2S', 38)]:
            o = self.L[k]
            out[k] = self.raw[o:o + nq * self.rows[k] * 16].clone()
        es = 4 * self.L['edge_stride_floats']
        for k, cnt in [('X0', 1), ('X1', 1), ('X2', 1), ('C', 1), ('A', 1), ('H1', 5)]:
            o = self.L[k]
            out[k] = self.raw[o:o + cnt * es - 256].clone()
        bb = 4 * self.L['bits_floats']
        for k, cnt in [('EB', 4), ('M1', 5), ('M2', 5)]:
            o = self.L[k]
            out[k] = torch.cat([self.raw[o + i * bb:o + i * bb + 19 * self.L['bits_rows']] for i in range(cnt)])
        return out


# ---- checks ----------------------------------------------------------------------------------------------------------------
class Checker:
    def __init__(self, case):
        self.case = case
        self.fail = []
        self.rec = _RECORD.setdefault(case, {})

    def _nan(self, name, got):
        if got.dtype.is_floating_point:
            k = int(torch.isnan(got).sum())
            if k:
                self.fail.append('%s: %d NaN (a launch read workspace memory no launch wrote, or an MMA barrier timed out)' % (name, k))
                return True
        return False

    def exact(self, name, got, ref):
        _CHECKED.add(name.split('[')[0])
        if self._nan(name, got):
            return
        bad = int((got != ref).sum())
        self.rec[name] = {'bit_exact': True, 'mismatches': bad}
        if bad:
            idx = torch.nonzero(got != ref)[0].tolist()
            self.fail.append('%s: %d of %d elements differ from the bit-exact reference (first at %s: %r vs %r)'
                             % (name, bad, got.numel(), idx, got[tuple(idx)].item(), ref[tuple(idx)].item()))

    def bar(self, name, got, ref, absref, tau, extra=None, normwise=None, norm_ref=None):
        """|got - ref| <= tau absref (+ extra) elementwise; got == ref exactly where the bound is 0.  normwise: also
        max|got - ref| / max|norm_ref| < normwise (norm_ref defaults to ref; a tanh stage passes its pre-activation)"""
        _CHECKED.add(name.split('[')[0])
        if self._nan(name, got):
            return
        g = got.double()
        d = (g - ref).abs()
        bound = tau * absref if extra is None else tau * absref + extra
        pos = absref > 0
        worst = float((d[pos] / absref[pos]).max()) if bool(pos.any()) else 0.0
        rn = float(ref.norm())
        nw = float(d.norm()) / rn if rn > 0 else float(d.norm())
        rr = float((ref * ref).sum())
        shrink = 1.0 - float((g * ref).sum()) / rr if rr > 0 else 0.0
        self.rec[name] = {'max_err_over_absref': worst, 'tau': tau, 'normwise': nw, 'shrink_1_minus_scale': shrink,
                          'elements': int(ref.numel())}
        over = d > bound
        if bool(over.any()):
            i = torch.nonzero(over)[0].tolist()
            self.fail.append('%s: %d of %d elements over the bar (worst |d|/absref %.3g, tau %.3g; first at %s: got %r, ref %r, absref %r)'
                             % (name, int(over.sum()), ref.numel(), worst, tau, i, g[tuple(i)].item(), ref[tuple(i)].item(),
                                absref[tuple(i)].item()))
        if normwise is not None:
            r = float(d.max()) / max(float((ref if norm_ref is None else norm_ref).abs().max()), 1e-300)
            self.rec[name]['max_err_over_max_ref'] = r
            if r >= normwise:
                self.fail.append('%s: max|d| / max|ref| = %.3g >= %.3g' % (name, r, normwise))


_PER_STEP = re.compile(r'^(S|R|G|U|P|dU|dG|T|dS|dR|H2S_)\d$')     # one check per propagation step: recorded as one stage


def _write_record(seconds):
    """stage -> graph -> [max |d| / absref, tau, normwise, mean shrink] over the layers and steps; one line per stage"""
    acc = {}
    for case, stages in _RECORD.items():
        graph = case.split()[0]
        for name, v in stages.items():
            if 'tau' not in v:
                continue
            a = acc.setdefault(_PER_STEP.sub(r'\1l', name), {}).setdefault(graph, [0.0, 0.0, 0.0, []])
            a[0], a[1], a[2] = max(a[0], v['max_err_over_absref']), max(a[1], v['tau']), max(a[2], v['normwise'])
            a[3].append(v['shrink_1_minus_scale'])
    g3 = lambda x: float('%.3g' % x)
    lines = ['  %s: {%s}' % (json.dumps(st), ', '.join('%s: %s' % (json.dumps(g), json.dumps([g3(a[0]), g3(a[1]), g3(a[2]), g3(sum(a[3]) / len(a[3]))]))
                                                   for g, a in per.items())) for st, per in sorted(acc.items())]
    head = {'device': torch.cuda.get_device_name(0), 'file_seconds': round(seconds, 1),
            'columns': ['max_err_over_absref', 'tau', 'normwise', 'shrink_1_minus_scale (mean)']}
    text = '{\n' + ''.join('  %s: %s,\n' % (json.dumps(k), json.dumps(v)) for k, v in head.items())
    text += '  "stages": {\n' + ',\n'.join('  ' + ln for ln in lines) + '\n  }\n}\n'
    try:
        os.makedirs(os.path.dirname(os.path.abspath(STAGES_OUT)), exist_ok=True)
        with open(STAGES_OUT, 'w') as f:
            f.write(text)
    except OSError:
        pass


# ---- loss seed (restatement of k_bce_grad's clip) ----------------------------------------------------------------------------
# k_bce_grad clips at the fp32 constants 1e-7f and 1.f - 1e-7f; the second rounds to 1 - 2^-23 (1 - 1e-7 in double is
# 1.9e-8 closer to 1, and logits 15.94 .. 16.12 fall between the two)
CLIP_LO = float(np.float32(1e-7))
CLIP_HI = float(np.float32(1.0) - np.float32(1e-7))


def prob_interval(z):
    """[p_lo, p_hi] (float64, on z's device) containing the kernels' fp32 p = 1 / (1 + expf(-z)) for fp32 logits z.
    expf is within 2 ulp of exp(-z) (4 u relative; exact at 0, where it returns 1); the add and the division are correctly
    rounded, hence monotone, so p lies between the values this arithmetic gives at the smallest and the largest fp32 number
    expf may return.  Near p = 1 this is the fp32 grid itself (p < 1 - 2^-23 exactly when fl(1 + e) >= 1 + 2^-22, i.e.
    e >= 3 * 2^-24, z <= ~15.537), which a relative bar on p cannot resolve."""
    zz = z.detach().cpu().numpy().astype(np.float32)
    e64 = np.exp(-zz.astype(np.float64))
    e64 = np.where(zz == 0, 1.0, e64)
    slack = np.where(zz == 0, 0.0, 4 * U)
    f32 = np.float32
    with np.errstate(over='ignore'):
        lo, hi = e64 * (1 - slack), e64 * (1 + slack)
        elo = lo.astype(f32)
        elo = np.where(elo.astype(np.float64) < lo, np.nextafter(elo, f32(np.inf)), elo)
        ehi = hi.astype(f32)
        ehi = np.where(ehi.astype(np.float64) > hi, np.nextafter(ehi, f32(0)), ehi)
        ehi = np.where(hi > np.finfo(f32).max, f32(np.inf), ehi)          # expf may overflow
        p_hi, p_lo = f32(1) / (f32(1) + elo), f32(1) / (f32(1) + ehi)
    to = lambda a: torch.from_numpy(a.astype(np.float64)).to(z.device)
    return to(p_lo), to(p_hi)


def bce_seed_reference(z, t, count, got):
    """fp64 d(mean clipped BCE)/d logit of fp32 logits z with targets t: (ref, absref, ambiguous).  The gradient passes only
    strictly inside the clip.  `ambiguous` marks the elements whose probability interval (prob_interval) straddles a clip
    edge, where the kernel's fp32 probability may fall on either side: there the reference follows the branch `got` took
    (exactly 0 outside, the inside value otherwise).  Everywhere else the branch is fixed."""
    p = torch.sigmoid(z)
    p_lo, p_hi = prob_interval(z)
    inside_sure = (p_lo > CLIP_LO) & (p_hi < CLIP_HI)
    outside_sure = (p_hi <= CLIP_LO) | (p_lo >= CLIP_HI)
    amb = ~inside_sure & ~outside_sure
    inside = torch.where(amb, got.double() != 0, inside_sure)
    ref = torch.where(inside, (p - t) / count, torch.zeros_like(p))
    ab = torch.where(inside, (p + (p - t).abs()) / count, torch.zeros_like(p))
    return ref, ab, amb


# ---- dropout masks (restatement of dropout_hash, spw_common.cuh, on the device) -----------------------------------------
def _keep(seed32, rows, stride, cols, rate, device):
    idx = torch.arange(rows, device=device, dtype=torch.int64)[:, None] * stride + torch.arange(cols, device=device)[None, :]
    M = 0xffffffff
    h = (idx * 0x9E3779B9 + seed32) & M
    h ^= h >> 16
    h = (h * 0x85EBCA6B) & M                   # int64 products wrap; the low 32 bits are exact
    h ^= h >> 13
    h = (h * 0xC2B2AE35) & M
    h ^= h >> 16
    return (h >> 8) >= int(np.float32(rate) * np.float32(16777216.0))


def _scale(seed32, rows, stride, cols, rate, device):
    """0 or 1/keep per element (inverted dropout); None without dropout"""
    if rate <= 0:
        return None
    inv = float(np.float32(1.0) / (np.float32(1.0) - np.float32(rate)))
    return _keep(seed32, rows, stride, cols, rate, device).double() * inv


# ---- one checked training step ---------------------------------------------------------------------------------------------
def _prefilled_step(api, eng, batch, tgt, rate, seed):
    n, E = batch.n_nodes, batch.n_edges
    eng.ws.get(api.dll.spw_workspace_bytes(n, E, 1)).fill_(0xFF)
    logits, _ = eng.forward(batch, training=True, want_probs=False, dropout_rate=rate, dropout_seed=seed)
    torch.cuda.synchronize()
    ws = Workspace(api, eng)
    fwd = ws.forward_state()
    logits = logits.clone()
    dl, _ = eng.bce_seed(logits, tgt, n)
    eng.backward(dl)
    torch.cuda.synchronize()
    return ws, fwd, logits, dl.clone()


def check_step(api, eng, batch, tgt, rate, seed, case):
    chk = Checker(case)
    ws, fwd_before, logits, dl = _prefilled_step(api, eng, batch, tgt, rate, seed)
    n, E, dev = batch.n_nodes, batch.n_edges, tgt.device
    W = {k: v.double() for k, v in eng.params.views.items()}
    Wa = {k: v.abs() for k, v in W.items()}
    relu = torch.relu
    seed_c, seed_q = O.dropout_seeds(seed)
    inv_keep = float(np.float32(1.0) / (np.float32(1.0) - np.float32(rate))) if rate > 0 else 1.0
    obj = batch.obj[:n]
    snd, rcv = batch.in_snd[:E].long(), batch.in_rcv[:E].long()
    in_off = batch.in_off[:n + 1].long()
    deg = (in_off[1:] - in_off[:-1]).double()
    maxdeg = int(deg.max()) if n else 0
    out_deg = torch.bincount(snd, minlength=n)
    max_outdeg = int(out_deg.max()) if E else 0
    d64 = lambda t: t.double()

    def mm(X, w, wa):
        X = X.double()
        return X @ w, X.abs() @ wa

    def index_sum(vals, idx):
        return torch.zeros(n, vals.shape[1], dtype=torch.float64, device=dev).index_add_(0, idx, vals)

    zeros2 = lambda rows: torch.zeros(rows, 2, dtype=torch.float32, device=dev)

    # ================= forward =================
    # object encoder layer 0 (k_obj_enc0_c): relu(fma(w, W[1], fma(y, W[0], b)))
    y, wv = d64(obj[:, 1])[:, None], d64(obj[:, 2])[:, None]
    pre = y * W['om.w0'][0] + wv * W['om.w0'][1] + W['om.b0']
    ab = (y * W['om.w0'][0]).abs() + (wv * W['om.w0'][1]).abs() + Wa['om.b0']
    Q1 = ws.node('Q1', 100)
    chk.bar('Q1', Q1, relu(pre), ab, 2 * U)
    # q = drop(relu(q1 . om.w1 + b))  (k_lin:node)
    ref, ab = mm(Q1, W['om.w1'], Wa['om.w1'])
    ref, ab = relu(ref + W['om.b1']), ab + Wa['om.b1']
    sq = _scale(seed_q, n, 128, 100, rate, dev)
    if sq is not None:
        ref, ab = ref * sq, ab * sq
    Q = ws.node('Q', 104)
    chk.bar('Q', Q[:, :100], ref, ab, tau_lin(100), normwise=FWD_NORMWISE)
    if sq is not None:
        chk.exact('Q[dropped]', Q[:, :100][sq == 0], torch.zeros_like(Q[:, :100][sq == 0]))
    # qv = q . V1a + c1
    ref, ab = mm(Q[:, :100], W['omp.w0'][:100], Wa['omp.w0'][:100])
    QV = ws.node('QV', 100)
    chk.bar('QV', QV, ref + W['omp.b0'], ab + Wa['omp.b0'], tau_lin(100), normwise=FWD_NORMWISE)

    if E > 0:
        # relation encoder layer 0 (k_edge_enc0_c) on [dx, dy] = (obj[rcv] - obj[snd])[:2], fp32 differences as the kernel forms them
        dx, dy = d64(obj[rcv, 0] - obj[snd, 0])[:, None], d64(obj[rcv, 1] - obj[snd, 1])[:, None]
        pre = dx * W['rm.w0'][0] + dy * W['rm.w0'][1] + W['rm.b0']
        ab = (dx * W['rm.w0'][0]).abs() + (dy * W['rm.w0'][1]).abs() + Wa['rm.b0']
        X = [ws.edge(k) for k in ('X0', 'X1', 'X2', 'C')]
        EB = [ws.bits('EB', i) for i in range(4)]
        chk.bar('X0', X[0][:, :150], relu(pre), ab, 2 * U)
        ones_pad = torch.cat([torch.ones(E, 1, device=dev), torch.zeros(E, 1, device=dev)], 1)
        chk.exact('X0[ones,pad]', X[0][:, 150:], ones_pad)
        # layers 1..3 (k_lin:enc_fwd): relu, ones column, sign bits; dropout on c_e (element index row * 160 + column)
        sc = _scale(seed_c, E, 160, 150, rate, dev)
        for i in range(1, 4):
            ref, ab = mm(X[i - 1][:, :150], W['rm.w%d' % i], Wa['rm.w%d' % i])
            ref, ab = relu(ref + W['rm.b%d' % i]), ab + Wa['rm.b%d' % i]
            if i == 3 and sc is not None:
                ref, ab = ref * sc, ab * sc
            name = 'X%d' % i if i < 3 else 'C'
            chk.bar(name, X[i][:, :150], ref, ab, tau_lin(150), normwise=FWD_NORMWISE)
            chk.exact(name + '[ones,pad]', X[i][:, 150:], ones_pad)
            if i == 3 and sc is not None:
                chk.exact('C[dropped]', X[3][:, :150][sc == 0], torch.zeros_like(X[3][:, :150][sc == 0]))
        for i in range(4):
            chk.exact('EB%d' % i, EB[i][:, :152], torch.cat([X[i][:, :150] > 0, torch.zeros(E, 2, dtype=torch.bool, device=dev)], 1))
        # A = c . W1a + b1
        ref, ab = mm(X[3][:, :150], W['rmp.w0'][:150], Wa['rmp.w0'][:150])
        A = ws.edge('A')
        chk.bar('A', A[:, :150], ref + W['rmp.b0'], ab + Wa['rmp.b0'], tau_lin(150), normwise=FWD_NORMWISE)
        chk.exact('A[pad]', A[:, 150:], zeros2(E))

    W1b, W1c = W['rmp.w0'][150:250], W['rmp.w0'][250:350]
    W1ba, W1ca = Wa['rmp.w0'][150:250], Wa['rmp.w0'][250:350]
    V1bc, V1bca = W['omp.w0'][100:300], Wa['omp.w0'][100:300]
    V2p, V2pa = W['omp.w1'][:, 1:], Wa['omp.w1'][:, 1:]
    chk.exact('P0', ws.node('GP', 100, 0, 100), torch.zeros(n, 100, device=dev))
    steps = []
    for l in range(5):
        st = {}
        GP = ws.node('GP', 200, l)
        P = GP[:, 100:]
        S, R = ws.node('S', 152, l), ws.node('R', 152, l)
        if l == 0:
            chk.exact('S0', S, torch.zeros_like(S))
            chk.exact('R0', R, torch.zeros_like(R))
        else:
            for nm, t, w, wa in (('S', S, W1b, W1ba), ('R', R, W1c, W1ca)):
                ref, ab = mm(P, w, wa)
                chk.bar('%s%d' % (nm, l), t[:, :150], ref, ab, tau_lin(100), normwise=FWD_NORMWISE)
                chk.exact('%s%d[pad]' % (nm, l), t[:, 150:], zeros2(n))
        H2S = ws.node('H2S', 152, l)
        if E > 0:
            # h1 (k_edge_step_c's operand build): bit-exact, same fp32 order
            H1 = ws.edge('H1', step=l)
            h1 = relu((A[:, :150] + S[snd, :150]) + R[rcv, :150])
            chk.exact('H1_%d' % l, H1[:, :150], h1)
            chk.exact('H1_%d[ones,pad]' % l, H1[:, 150:], ones_pad)
            M1 = ws.bits('M1', l)
            chk.exact('M1_%d' % l, M1[:, :152], torch.cat([h1 > 0, torch.zeros(E, 2, dtype=torch.bool, device=dev)], 1))
            # h2 and its receiver sums (k_edge_step_c + k_seg_fix_c), on the GPU's relu states
            M2 = ws.bits('M2', l)
            pre, abp = mm(H1[:, :150], W['rmp.w1'], Wa['rmp.w1'])
            pre, abp = pre + W['rmp.b1'], abp + Wa['rmp.b1']
            m2 = M2[:, :150]
            flips = (m2 != (pre > 0)) & (pre.abs() > tau_lin(150) * abp)
            chk.exact('M2_%d[vs fp64 outside rounding]' % l, flips, torch.zeros_like(flips))
            chk.exact('M2_%d[pad]' % l, M2[:, 150:152], torch.zeros(E, 2, dtype=torch.bool, device=dev))
            ref = index_sum(pre * m2, rcv)
            ab = index_sum(abp * m2, rcv)
            chunks = math.ceil(maxdeg / 32) + 1
            chk.bar('H2S_%d' % l, H2S[:, :150], ref, ab, tau_lin(150) + (6 + chunks) * U)
            st.update(H1=H1, M1=M1, M2=M2)
        else:
            chk.exact('H2S_%d' % l, H2S[:, :150], torch.zeros(n, 150, device=dev))
        chk.exact('H2S_%d[pad]' % l, H2S[:, 150:], zeros2(n))
        # g = tanh(H2S . W3 + deg b3)
        ref, ab = mm(H2S[:, :150], W['rmp.w2'], Wa['rmp.w2'])
        pre, ab = ref + deg[:, None] * W['rmp.b2'], ab + deg[:, None] * Wa['rmp.b2']
        ref = torch.tanh(pre)
        G = GP[:, :100]
        chk.bar('G%d' % l, G, ref, ab, tau_lin(150), extra=TANH_REL * ref.abs(), normwise=FWD_NORMWISE, norm_ref=pre)
        # u = relu([g | p] . [V1b ; V1c] + qv)
        ref, ab = mm(GP, V1bc, V1bca)
        ref, ab = relu(ref + d64(QV)), ab + d64(QV).abs()
        Uu = ws.node('U', 104, l)
        chk.bar('U%d' % l, Uu[:, :100], ref, ab, tau_lin(200), normwise=FWD_NORMWISE)
        if l < 4:   # p' = tanh(u . V2p + c2[1:] + p)
            ref, ab = mm(Uu[:, :100], V2p, V2pa)
            pre, ab = ref + W['omp.b1'][1:] + d64(P), ab + Wa['omp.b1'][1:] + d64(P).abs()
            ref = torch.tanh(pre)
            chk.bar('P%d' % (l + 1), ws.node('GP', 100, l + 1, 100), ref, ab, tau_lin(100), extra=TANH_REL * ref.abs(),
                    normwise=FWD_NORMWISE, norm_ref=pre)
        st.update(G=G, P=P, GP=GP, U=Uu[:, :100], H2S=H2S)
        steps.append(st)
    # head (k_logit_c)
    U4 = d64(steps[4]['U'])
    terms = U4 * W['omp.w1'][:, 0]
    ref = terms.sum(1) + W['omp.b1'][0]
    ab = terms.abs().sum(1) + Wa['omp.b1'][0]
    chk.bar('logits', logits[:n], ref, ab, 101 * U)
    # loss seed (k_bce_grad): d(mean clipped BCE)/d logit on the GPU's logits
    ref, ab, _ = bce_seed_reference(d64(logits[:n]), d64(tgt[:n]), n, dl[:n])
    chk.bar('dlogits', dl[:n], ref, ab, 8 * U)

    # ================= backward =================
    # dU_4 = dlogit (x) V2[:, 0] * [u_4 > 0]  (k_logit_bwd_c): one fp32 multiply
    dU = [ws.node('dU', 100, l) for l in range(5)]
    dG = [ws.node('dG', 100, l) for l in range(5)]
    v20 = eng.params.views['omp.w1'][:, 0]
    chk.exact('dU4', dU[4], torch.where(steps[4]['U'] > 0, dl[:n, None] * v20[None, :], torch.zeros_like(dU[4])))
    T = [ws.node('T', 100, l) for l in range(4)]
    dS = [ws.node('dS', 152, l) for l in range(4)]
    dR = [ws.node('dR', 152, l) for l in range(4)]
    W3T, W3Ta = W['rmp.w2'].t(), Wa['rmp.w2'].t()
    W2T, W2Ta = W['rmp.w1'].t(), Wa['rmp.w1'].t()
    dA_ref = torch.zeros(E, 150, dtype=torch.float64, device=dev)
    dA_abs = torch.zeros_like(dA_ref)
    dh2 = [None] * 5
    for l in range(4, -1, -1):
        st = steps[l]
        if l < 4:   # dUpre = (T . V2p^T) * [u > 0]
            ref, ab = mm(T[l], V2p.t(), V2pa.t())
            m = (st['U'] > 0).double()
            chk.bar('dU%d' % l, dU[l], ref * m, ab * m, tau_lin(100))
        # dg_pre = (dUpre . V1b^T) * (1 - g^2)
        ref, ab = mm(dU[l], W['omp.w0'][100:200].t(), Wa['omp.w0'][100:200].t())
        f = 1 - d64(st['G']) ** 2
        chk.bar('dG%d' % l, dG[l], ref * f, ab * f.abs(), tau_lin(100), extra=2 * U * ab)
        # d(sum h2) = dg_pre . W3^T (only step 0's survives the pass), rebuilt in fp64 for the edge stages
        dH, dHa = mm(dG[l], W3T, W3Ta)
        if l == 0:
            got = ws.node('dH2S', 152)
            chk.bar('dH2S0', got[:, :150], dH, dHa, tau_lin(100))
            chk.exact('dH2S0[pad]', got[:, 150:], zeros2(n))
        if E > 0:
            m2, m1 = st['M2'][:, :150].double(), st['M1'][:, :150].double()
            g2, g2a = dH[rcv] * m2, dHa[rcv] * m2
            dh2[l] = (g2, g2a)
            h1, h1a = g2 @ W2T * m1, g2a @ W2Ta * m1
            dA_ref += h1
            dA_abs += h1a
            if l > 0:   # dS / dR of step l (k_edge_dgrad_c -> DH1 -> k_gather_dsr_c), composite
                tau = tau_lin(100) + tau_lin(150)
                chk.bar('dR%d' % (l - 1), dR[l - 1][:, :150], index_sum(h1, rcv), index_sum(h1a, rcv), tau + maxdeg * U)
                chk.bar('dS%d' % (l - 1), dS[l - 1][:, :150], index_sum(h1, snd), index_sum(h1a, snd), tau + max_outdeg * U)
        elif l > 0:
            chk.exact('dR%d' % (l - 1), dR[l - 1][:, :150], torch.zeros(n, 150, device=dev))
            chk.exact('dS%d' % (l - 1), dS[l - 1][:, :150], torch.zeros(n, 150, device=dev))
        if l > 0:
            # T^{l-1} = (dU_l . V1c^T [+ T_l] + dS . W1b^T + dR . W1c^T) * (1 - p_l^2): three k_lin launches through DP
            r1, a1 = mm(dU[l], W['omp.w0'][200:300].t(), Wa['omp.w0'][200:300].t())
            r2, a2 = mm(dS[l - 1][:, :150], W1b.t(), W1ba.t())
            r3, a3 = mm(dR[l - 1][:, :150], W1c.t(), W1ca.t())
            ref, ab = r1 + r2 + r3, a1 + a2 + a3
            if l < 4:
                ref, ab = ref + d64(T[l]), ab + d64(T[l]).abs()
            f = 1 - d64(st['P']) ** 2
            chk.bar('T%d' % (l - 1), T[l - 1], ref * f, ab * f.abs(), tau_lin(100) + 2 * tau_lin(150), extra=2 * U * ab)
    # DP = sum of the steps' dUpre (k_sum_slots_c): bit-exact
    DP = ws.node('DP', 100)
    s = torch.zeros_like(dU[0])
    for l in range(5):
        s = s + dU[l]
    chk.exact('DP', DP, s)
    # dq = (DP . V1a^T) * [q > 0] / keep ; dq1 = (dq . om.w1^T) * [q1 > 0]
    ref, ab = mm(DP, W['omp.w0'][:100].t(), Wa['omp.w0'][:100].t())
    m = (Q[:, :100] > 0).double() * inv_keep
    dQ = ws.node('dQ', 100)
    chk.bar('dQ', dQ, ref * m, ab * m, tau_lin(100))
    ref, ab = mm(dQ, W['om.w1'].t(), Wa['om.w1'].t())
    m = (Q1 > 0).double()
    dQ1 = ws.node('dQ1', 100)
    chk.bar('dQ1', dQ1, ref * m, ab * m, tau_lin(100))
    if E > 0:
        chk.bar('dA', ws.edge('dA')[:, :150], dA_ref, dA_abs, tau_lin(100) + tau_lin(150) + 5 * U)
        # relation-encoder data gradients (k_lin:enc_bwd); the first two are overwritten by the last two and rebuilt here
        dA = d64(ws.edge('dA')[:, :150])
        enc, enca = [], []
        src, srca = dA, dA.abs()
        for i, wn in enumerate(['rmp.w0', 'rm.w3', 'rm.w2', 'rm.w1']):
            w = W[wn][:150] if i == 0 else W[wn]
            wa = w.abs()
            m = EB[3 - i][:, :150].double() * (inv_keep if i == 0 else 1.0)
            r, a = (src @ w.t()) * m, (srca @ wa.t()) * m
            enc.append(r)
            enca.append(a)
            src, srca = r, a
        DH1 = ws.edge('DH1')
        GB = ws.edge('GB')
        chk.bar('DH1[enc2]', DH1[:, :150], enc[2], enca[2], 3 * tau_lin(150))
        ref, ab = mm(DH1[:, :150], W['rm.w1'].t(), Wa['rm.w1'].t())
        m = EB[0][:, :150].double()
        chk.bar('GB[enc3]', GB[:, :150], ref * m, ab * m, tau_lin(150))

    # ================= the 22 gradients =================
    gv = eng.grads.views

    def wg(name, got, X, dY, tau, rowscale=None, Xa=None, dYa=None, bias=None):
        """got = [X^T dY ; sum rowscale dY] as a contraction of saved arrays"""
        X, dY = X.double(), dY.double()
        Xa = X.abs() if Xa is None else Xa
        dYa = dY.abs() if dYa is None else dYa
        chk.bar(name, got, X.t() @ dY, Xa.t() @ dYa, tau)
        if bias is not None:
            rs = torch.ones(X.shape[0], dtype=torch.float64, device=dev) if rowscale is None else rowscale
            chk.bar(bias[0], bias[1], rs @ dY, rs.abs() @ dYa, tau)

    GPall = torch.cat([st['GP'] for st in steps])
    wg('grad omp.w0[:100]', gv['omp.w0'][:100], Q[:, :100], DP, tau_wg(n), bias=('grad omp.b0', gv['omp.b0']))
    wg('grad omp.w0[100:]', gv['omp.w0'][100:], GPall, torch.cat(dU), tau_wg(5 * n))
    wg('grad omp.w1[:,1:]', gv['omp.w1'][:, 1:], torch.cat([st['U'] for st in steps[:4]]), torch.cat(T), tau_wg(4 * n),
       bias=('grad omp.b1[1:]', gv['omp.b1'][1:]))
    wg('grad omp.w1[:,0]', gv['omp.w1'][:, :1], steps[4]['U'], dl[:n, None], tau_sk(n), bias=('grad omp.b1[0]', gv['omp.b1'][:1]))
    wg('grad rmp.w2', gv['rmp.w2'], torch.cat([st['H2S'][:, :150] for st in steps]), torch.cat(dG), tau_wg(5 * n),
       rowscale=deg.repeat(5), bias=('grad rmp.b2', gv['rmp.b2']))
    Pall = torch.cat([st['P'] for st in steps[1:]])
    wg('grad rmp.w0[150:250]', gv['rmp.w0'][150:250], Pall, torch.cat([t[:, :150] for t in dS]), tau_wg(4 * n))
    wg('grad rmp.w0[250:]', gv['rmp.w0'][250:], Pall, torch.cat([t[:, :150] for t in dR]), tau_wg(4 * n))
    wg('grad om.w1', gv['om.w1'], Q1, dQ, tau_wg(n), bias=('grad om.b1', gv['om.b1']))
    wg('grad om.w0', gv['om.w0'], obj[:, 1:3], dQ1, tau_sk(n), bias=('grad om.b0', gv['om.b0']))
    if E > 0:
        H1all = torch.cat([st['H1'][:, :150] for st in steps])
        wg('grad rmp.w1', gv['rmp.w1'], H1all, torch.cat([d[0] for d in dh2]), tau_wg(E, 5) + tau_lin(100),
           dYa=torch.cat([d[1] for d in dh2]), bias=('grad rmp.b1', gv['rmp.b1']))
        wg('grad rmp.w0[:150]', gv['rmp.w0'][:150], X[3][:, :150], dA, tau_wg(E), bias=('grad rmp.b0', gv['rmp.b0']))
        wg('grad rm.w3', gv['rm.w3'], X[2][:, :150], enc[0], tau_wg(E) + tau_lin(150), dYa=enca[0],
           bias=('grad rm.b3', gv['rm.b3']))
        wg('grad rm.w2', gv['rm.w2'], X[1][:, :150], enc[1], tau_wg(E) + 2 * tau_lin(150), dYa=enca[1],
           bias=('grad rm.b2', gv['rm.b2']))
        wg('grad rm.w1', gv['rm.w1'], X[0][:, :150], DH1[:, :150], tau_wg(E), bias=('grad rm.b1', gv['rm.b1']))
        dxy = torch.cat([obj[rcv, 0:1] - obj[snd, 0:1], obj[rcv, 1:2] - obj[snd, 1:2]], 1)
        wg('grad rm.w0', gv['rm.w0'], dxy, GB[:, :150], tau_sk(E), bias=('grad rm.b0', gv['rm.b0']))
    else:
        for k in ['rmp.w1', 'rmp.b1', 'rm.w0', 'rm.b0', 'rm.w1', 'rm.b1', 'rm.w2', 'rm.b2', 'rm.w3', 'rm.b3']:
            chk.exact('grad ' + k, gv[k], torch.zeros_like(gv[k]))
        chk.exact('grad rmp.w0[:150]', gv['rmp.w0'][:150], torch.zeros_like(gv['rmp.w0'][:150]))
        chk.exact('grad rmp.b0', gv['rmp.b0'], torch.zeros_like(gv['rmp.b0']))

    # the backward pass never writes forward state
    after = ws.forward_state()
    for k, v in fwd_before.items():
        if not torch.equal(v, after[k]):
            chk.fail.append('%s: the backward pass wrote forward state (%d bytes changed)' % (k, int((v != after[k]).sum())))
    return chk


# ---- graphs ----------------------------------------------------------------------------------------------------------------
def _graph(name):
    from spwgnn_b200.graph import TowerBatch
    from spwgnn_b200 import synth
    if name == 'fc2':                       # one 2-block tower: E = 2
        return TowerBatch.from_towers(synth.make_towers('jenga', 1, 11, n=2), fully_connected=True), 0.0
    if name == 'fc3+1':                     # a 3-block tower next to a 1-block tower (a node without in-edges)
        return TowerBatch.from_towers(synth.make_towers('jenga', 1, 12, n=3) + synth.make_towers('jenga', 1, 13, n=1),
                                      fully_connected=True), 0.0
    if name == 'tails':                     # n = 129 = 1 (mod 128), E = 257 = 1 (mod 32): one edge of 43 3-block towers removed
        b = TowerBatch.from_towers(synth.make_towers('jenga', 43, 14, n=3), fully_connected=True, want_slot_list=True)
        s, r = b.slot_list[0][:b.n_edges].long(), b.slot_list[1][:b.n_edges].long()
        keep = torch.ones(b.n_edges, dtype=torch.bool, device=s.device)
        keep[100] = False
        b._set_edges(s[keep], r[keep])
        assert b.n_nodes % 128 == 1 and b.n_edges % 32 == 1
        return b, 0.1
    if name == 'fc64':                      # in-degree 63 (segments over three 32-row chunks); E = 96 768 > 4 * 148 * 128
        b = TowerBatch.from_towers(synth.make_towers('jenga', 24, 15, n=64), fully_connected=True)
        assert b.n_edges == 96768
        return b, 0.0
    if name == 'contact':                   # Jenga-18 towers with runs of 40+ single-block towers between them
        towers = []
        for k in range(6):
            towers += synth.make_towers('jenga18', 1, 20 + k) + synth.make_towers('jenga', 40 + 3 * k, 30 + k, n=1)
        return TowerBatch.from_towers(towers), 0.0
    if name == 'C2':                        # BASELINE config 2 at full size, dropout 0.1
        b = TowerBatch.from_towers(synth.make_towers('jenga', 4096, 1235, n=10), fully_connected=True)
        assert b.n_nodes == 40960 and b.n_edges == 368640
        return b, 0.1
    raise ValueError(name)


GRAPHS = ['fc2', 'fc3+1', 'tails', 'fc64', 'contact', 'C2']


@pytest.fixture(scope='module')
def eng():
    from spwgnn_b200.engine import Engine
    assert torch.cuda.is_available()
    t0 = time.perf_counter()
    e = Engine('cuda:0', seed=5)
    yield e
    _write_record(time.perf_counter() - t0)


def test_dropout_mask_restatement_matches_the_oracle():
    for seed, rate in [(0x12345678, 0.1), (7, 0.5)]:
        got = _keep(seed, 64, 160, 150, rate, 'cuda').cpu().numpy()
        idx = np.arange(64)[:, None] * 160 + np.arange(150)[None, :]
        assert np.array_equal(got, O.dropout_keep_mask(seed, idx, rate))


@pytest.mark.parametrize('graph', GRAPHS)
def test_stages(eng, graph):
    from spwgnn_b200._lib import lib
    api = lib()
    batch, rate = _graph(graph)
    n = batch.n_nodes
    tgt = torch.as_tensor((np.random.default_rng(n).random(n) > 0.5).astype(np.float32)).cuda()
    eng.params.load_dict(O.init_weights(21, nonzero_bias=True))
    eng._adam = None
    seed = 0x9e3779b97f4a7c15 if rate > 0 else 0
    chks = [check_step(api, eng, batch, tgt, rate, seed, '%s step 1' % graph)]
    # a second step after the weights were changed in place (stale packed operands would show): Adam, then a new weight set
    eng.adam_step()
    chks.append(check_step(api, eng, batch, tgt, rate, seed + 1, '%s step 2 (after adam_step)' % graph))
    if graph != 'C2':
        eng.params.load_dict(O.init_weights(22, nonzero_bias=True))
        chks.append(check_step(api, eng, batch, tgt, rate, seed + 2, '%s step 3 (after load_dict)' % graph))
    fails = [f for c in chks for f in c.fail]
    assert not fails, '\n'.join(fails)


# launch tag (spw_profile_report) -> the stage checks that cover it
TAG_CHECKS = {
    'k_pack_tc': ['Q', 'QV', 'S', 'G', 'U', 'P', 'dU', 'dG', 'T', 'dQ', 'dQ1', 'dH2S0'],
    'k_pack_umma': ['H2S', 'dR', 'DH1', 'GB'],
    'k_deg_to_float': ['G', 'grad rmp.b2'],
    'k_obj_enc0_c': ['Q1'],
    'k_edge_enc0_c': ['X0', 'EB0'],
    'k_lin:node': ['Q', 'QV', 'S', 'R', 'G', 'U', 'P', 'dU', 'dG', 'T', 'dH2S0', 'dQ', 'dQ1'],
    'k_lin:enc_fwd': ['X1', 'X2', 'C', 'A', 'EB1', 'EB2', 'EB3'],
    'k_edge_step_c': ['H1_', 'M1_', 'M2_', 'H2S_'],
    'k_seg_fix_c': ['H2S_'],
    'k_logit_c': ['logits'],
    'k_bce_grad': ['dlogits'],
    'k_logit_bwd_c': ['dU4'],
    'k_edge_dgrad_c': ['dA', 'dR', 'dS'],
    'k_gather_dsr_c': ['dR', 'dS'],
    'k_sum_slots_c': ['DP'],
    'k_lin:enc_bwd': ['DH1', 'GB'],
    'k_wgrad_c:step': ['grad rmp.w1', 'grad rmp.b1'],
    'k_wgrad_c:node': ['grad omp.w0', 'grad omp.b0', 'grad omp.w1', 'grad omp.b1', 'grad rmp.w2', 'grad rmp.b2', 'grad om.w1',
                       'grad om.b1', 'grad rmp.w0'],
    'k_wgrad_c:enc': ['grad rmp.w0', 'grad rmp.b0', 'grad rm.w3', 'grad rm.b3', 'grad rm.w2', 'grad rm.b2', 'grad rm.w1', 'grad rm.b1'],
    'k_skinny_c': ['grad omp.w1', 'grad omp.b1', 'grad om.w0', 'grad om.b0', 'grad rm.w0', 'grad rm.b0'],
    'k_reduce_parts': ['grad omp.w0', 'grad rmp.w1', 'grad rm.w0', 'grad om.w0'],
}


def test_every_launch_of_a_training_step_has_a_stage_check(eng):
    """One extra profiled step (event brackets change the PDL overlap, so it is not one of the checked steps): every launch tag
    of a training step must map to stage checks that ran in this module -- a kernel added later without one fails here."""
    from spwgnn_b200._lib import lib
    import ctypes
    api = lib()
    batch, _ = _graph('contact')
    n = batch.n_nodes
    tgt = torch.zeros(n, device='cuda')
    buf = ctypes.create_string_buffer(1 << 16)
    api.check(api.dll.spw_profile_report(buf, len(buf)))          # clears anything recorded before
    api.check(api.dll.spw_profile(1))
    try:
        eng.loss_and_grads(batch, tgt)
        torch.cuda.synchronize()
        api.check(api.dll.spw_profile_report(buf, len(buf)))
    finally:
        api.dll.spw_profile(0)
    tags = [ln.split()[0] for ln in buf.value.decode().splitlines() if ln.strip()]
    assert 'k_edge_step_c' in tags and 'k_wgrad_c:step' in tags, tags
    missing = [t for t in tags if t not in TAG_CHECKS]
    assert not missing, 'launch tags without a stage check: %s' % missing
    if _CHECKED:        # with the stage tests in the same run: every mapped check actually ran
        for t in tags:
            for c in TAG_CHECKS[t]:
                assert any(k == c or k.startswith(c) for k in _CHECKED), (t, c)
