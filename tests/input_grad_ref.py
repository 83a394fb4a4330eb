"""TEST INFRASTRUCTURE: the fp64 reference of spw_backward_inputs, on top of oracle.propnet (which it uses unchanged).

forward_towers restates oracle.propnet.forward_dense per tower on the compact relation tensors: tower t gets sender / receiver
matrices Ms, Mr (N_max, E_max + 1) whose columns are the tower's active relations (one-hot) plus one all-zero column, and blocks
past N_t as zero padding (no relation touches them, and their logits get no weight).  The all-zero column carries the message of
a zero input, as every inactive slot of the dense input does (Networks.py:75,86-88 run on every column), so its receiver
gradient is the value of every inactive slot.  It calls the oracle's own _mlp and _relu; c_scale / q_scale inject the dropout
of a training forward as obj_grad_ref does (the all-zero column gets none).  input_grads differentiates it with torch autograd
with respect to Ms, Mr, the propagation input (at 0) and the objects.  Given the 21 relu states of a forward on the active
relations (Engine.saved_relu_states), it evaluates that linear branch through the oracle's relu-forcing hook: the all-zero and
padding columns and the padding blocks keep their own states (those of the zero-input message and of a zero block without
relations, which depend on the weights alone)."""
import numpy as np
import torch

from oracle import propnet as O


def forward_towers(w, objp, Ms, Mr, prop, c_scale=None, q_scale=None):
    """forward_dense(w, objp, Ms, Mr, prop, return_logits=True)[1] with inverted-dropout factors c_scale (T, R, 150) on the
    relation encoding and q_scale (T, N, 100) on the object encoding; returns logits (T, N)."""
    rs_t, rr_t = Ms.permute(0, 2, 1), Mr.permute(0, 2, 1)
    diff_rs = (rr_t @ objp)[:, :, 0:2] - (rs_t @ objp)[:, :, 0:2]
    rel_enc = O._relu(O._mlp(w, 'rm', diff_rs))
    obj_enc = O._relu(O._mlp(w, 'om', torch.cat([objp[:, :, 1:2], objp[:, :, 2:3]], dim=-1)))
    if c_scale is not None:
        rel_enc = rel_enc * c_scale
    if q_scale is not None:
        obj_enc = obj_enc * q_scale
    p, x = prop, None
    for _ in range(O.N_STEPS):
        x = O._mlp(w, 'rmp', torch.cat([rel_enc, rs_t @ p, rr_t @ p], dim=-1))
        eff = torch.tanh(Mr @ x)
        x = O._mlp(w, 'omp', torch.cat([obj_enc, eff, p], dim=-1))
        p = torch.tanh(x[:, :, 1:] + p)
    return x[:, :, 0]


def zero_message_states(w):
    """relu states of the message of an all-zero relation column: rm layers 0..3 and rmp layers 0, 1 (150 each)"""
    x, out = torch.zeros(1, 2, dtype=w['rm.w0'].dtype), []
    for li in range(4):
        x = x @ w['rm.w%d' % li] + w['rm.b%d' % li]
        out.append(x[0] > 0); x = torch.relu(x)
    x = x @ w['rmp.w0'][:150] + w['rmp.b0']
    out.append(x[0] > 0); x = torch.relu(x)
    x = x @ w['rmp.w1'] + w['rmp.b1']
    out.append(x[0] > 0)
    return out


def zero_block_states(w):
    """relu states of a padding block (zero features, no relations): om layers 0, 1, then omp layer 0 of the five steps"""
    x, out = torch.zeros(1, 2, dtype=w['om.w0'].dtype), []
    x = x @ w['om.w0'] + w['om.b0']
    out.append(x[0] > 0)
    x = torch.relu(x) @ w['om.w1'] + w['om.b1']
    out.append(x[0] > 0)
    q, p = torch.relu(x), torch.zeros(1, O.PROP_DIM, dtype=x.dtype)
    for _ in range(O.N_STEPS):
        h = torch.cat([q, torch.zeros_like(p), p], dim=-1) @ w['omp.w0'] + w['omp.b0']
        out.append(h[0] > 0)
        z = torch.relu(h) @ w['omp.w1'] + w['omp.b1']
        p = torch.tanh(z[:, 1:] + p)
    return out


def input_grads(w, obj, node_off, snd, rcv, dlogits, c_scale=None, q_scale=None, masks=None):
    """Gradient of sum_i dlogits[i]*logit[i] with respect to the four inputs of the reference's model, for the towers
    node_off (T+1,) with the active relations snd[e] -> rcv[e] (GLOBAL block ids, any order).  c_scale (E, 150) / q_scale
    (n, 100): dropout factors in the order of the relations / blocks.  masks: None, or the 21 relu states of a forward with the
    relations in the order given (rm 0..3 and per step rmp 0, 1 [E][150]; om 0..1 and per step omp 0 [n][100]).  Returns, in
    obj's dtype, (drs (E, N_max), drr (E, N_max), drr_free (n,), dprop (n, 100), dobj (n, 3), logits (n,), flips): row e of
    drs / drr is relation e's column, entry j local block j of its tower (0 for j >= N_t), as spw_backward_inputs lays them
    out; flips as oracle.propnet.loss_and_grads_forced (None without masks)."""
    dt = obj.dtype
    node_off = np.asarray(node_off, np.int64)
    snd, rcv = np.asarray(snd, np.int64), np.asarray(rcv, np.int64)
    T, n, E = len(node_off) - 1, int(node_off[-1]), len(snd)
    Nt = np.diff(node_off)
    Nm = max(int(Nt.max()) if T else 0, 1)
    ti = np.repeat(np.arange(T), Nt)                              # block -> tower, local index
    ji = np.arange(n) - node_off[ti]
    te = ti[rcv] if E else np.zeros(0, np.int64)                  # relation -> tower, column within the tower
    order = np.argsort(te, kind='stable')                         # column within the tower: rank among its relations
    ke = np.empty(E, np.int64)
    cnt = np.bincount(te, minlength=T) if E else np.zeros(T, np.int64)
    ke[order] = np.arange(E) - np.repeat(np.cumsum(cnt) - cnt, cnt)
    R = int(cnt.max() if T else 0) + 1                            # column R - 1 is all-zero in every tower
    Ms = torch.zeros(T, Nm, R, dtype=dt); Mr = torch.zeros(T, Nm, R, dtype=dt)
    Ms[te, snd - node_off[te], ke] = 1.0
    Mr[te, rcv - node_off[te], ke] = 1.0
    objp = torch.zeros(T, Nm, 3, dtype=dt); objp[ti, ji] = obj.detach()
    prop = torch.zeros(T, Nm, O.PROP_DIM, dtype=dt)
    cs = qs = None
    if c_scale is not None:
        cs = torch.ones(T, R, 150, dtype=dt); cs[te, ke] = torch.as_tensor(c_scale, dtype=dt)
    if q_scale is not None:
        qs = torch.ones(T, Nm, 100, dtype=dt); qs[ti, ji] = torch.as_tensor(q_scale, dtype=dt)
    if masks is not None:
        zs, zb = zero_message_states(w), zero_block_states(w)
        edge_state = [0, 1, 2, 3] + [4, 5] * 5             # which zero-message state each [E][150] layer takes
        padded, k, kb = [], 0, 0
        for m in masks:
            m = torch.as_tensor(m).to(dt)
            if m.shape[1] == 150:
                pm = zs[edge_state[k]].to(dt).expand(T, R, 150).clone(); pm[te, ke] = m; k += 1
            else:
                pm = zb[kb].to(dt).expand(T, Nm, 100).clone(); pm[ti, ji] = m; kb += 1
            padded.append(pm)
        O._FORCED, O._FLIPS = padded, []
    try:
        ins = [t.requires_grad_(True) for t in (Ms, Mr, prop, objp)]
        z = forward_towers(w, objp, Ms, Mr, prop, cs, qs)
        assert not O._FORCED, 'unused masks'
        dl = torch.zeros(T, Nm, dtype=dt); dl[ti, ji] = torch.as_tensor(dlogits, dtype=dt)
        gMs, gMr, gp, go = torch.autograd.grad((z * dl).sum(), ins)
        flips = O._FLIPS
    finally:
        O._FORCED, O._FLIPS = None, None
    valid = torch.as_tensor(np.arange(Nm)[None, :] < Nt[te][:, None])       # (E, N_max): j < N_t of the relation's tower
    drs = torch.where(valid, gMs[te, :, ke], torch.zeros((), dtype=dt))
    drr = torch.where(valid, gMr[te, :, ke], torch.zeros((), dtype=dt))
    return (drs.detach(), drr.detach(), gMr[ti, ji, R - 1].detach(), gp[ti, ji].detach(), go[ti, ji].detach(),
            z[ti, ji].detach(), flips)
