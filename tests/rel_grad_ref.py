"""TEST INFRASTRUCTURE: the fp64 reference of spw_backward_rel, on top of oracle.propnet (which it uses unchanged).

forward_weighted restates oracle.propnet.forward_sparse with a weight per relation, rel_scale (E,), multiplying diff, p[snd],
p[rcv] and x before index_add: where the dense graph's one-hot entries act (Networks.py:32-33,84-85,88).  With rel_scale None it
is forward_sparse operation for operation (test_emu_rel_grad pins that bit for bit), and it calls the oracle's own _mlp and
_relu, so the oracle's relu-forcing hook (_FORCED / _FLIPS) evaluates a given linear branch of it.  rel_grads differentiates it
with torch autograd with respect to rel_scale at 1."""
import torch

from oracle import propnet as O


def forward_weighted(w, obj, snd, rcv, rel_scale=None, c_scale=None, q_scale=None):
    """oracle.propnet.forward_sparse(..., return_logits=True) with relation e scaled by rel_scale[e]; returns (probs, logits)"""
    n = obj.shape[0]
    snd = snd.long(); rcv = rcv.long()
    sc = (lambda t: t) if rel_scale is None else (lambda t: t * rel_scale[:, None])
    diff = sc(obj[rcv, 0:2] - obj[snd, 0:2])
    c = O._relu(O._mlp(w, 'rm', diff))
    q = O._relu(O._mlp(w, 'om', obj[:, 1:3]))
    if c_scale is not None:
        c = c * c_scale
    if q_scale is not None:
        q = q * q_scale
    p = torch.zeros(n, O.PROP_DIM, dtype=obj.dtype)
    z = None
    for _ in range(O.N_STEPS):
        x = sc(O._mlp(w, 'rmp', torch.cat([c, sc(p[snd]), sc(p[rcv])], dim=-1)))
        agg = torch.zeros(n, O.PROP_DIM, dtype=obj.dtype).index_add(0, rcv, x)
        g = torch.tanh(agg)
        z = O._mlp(w, 'omp', torch.cat([q, g, p], dim=-1))
        p = torch.tanh(z[:, 1:] + p)
    logits = z[:, 0]
    return torch.sigmoid(logits), logits


def rel_grads(w, obj, snd, rcv, dlogits, masks=None, c_scale=None, q_scale=None):
    """Gradient of sum_i dlogits[i]*logit[i] with respect to the relation weights at 1, in obj's dtype, for the relations
    snd[e] -> rcv[e] in the order given.  masks / c_scale / q_scale: as obj_grad_ref.obj_grads.
    Returns (drel (E,), logits (n,), flips)."""
    if masks is not None:
        O._FORCED, O._FLIPS = [m for m in masks], []
    try:
        ws = torch.ones(len(snd), dtype=obj.dtype, requires_grad=True)
        _, logits = forward_weighted(w, obj.detach(), snd, rcv, ws, c_scale=c_scale, q_scale=q_scale)
        assert not O._FORCED, 'unused masks'
        dl = torch.as_tensor(dlogits, dtype=obj.dtype)
        (g,) = torch.autograd.grad((logits * dl).sum(), [ws], allow_unused=True)
        if g is None:
            g = torch.zeros_like(ws)
        return g.detach(), logits.detach(), O._FLIPS
    finally:
        O._FORCED, O._FLIPS = None, None
