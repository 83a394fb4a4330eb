"""TEST INFRASTRUCTURE: the fp64 reference of spw_backward_obj, on top of oracle.propnet (which it uses unchanged).

obj_grads differentiates oracle.propnet.forward_sparse with torch autograd with respect to obj, the relations held fixed.  It
can evaluate a given linear branch of the network through the oracle's relu-forcing hook (_FORCED / _FLIPS, the mechanism
oracle.propnet.loss_and_grads_forced uses)."""
import torch

from oracle import propnet as O


def obj_grads(w, obj, snd, rcv, dlogits, masks=None, c_scale=None, q_scale=None):
    """Gradient of sum_i dlogits[i]*logit[i] with respect to obj (n, 3) = [x, y, width] / 170, in obj's dtype.
    masks: optional 21 relu masks (the order of O.loss_and_grads_forced) to evaluate on that linear branch; c_scale / q_scale:
    dropout factors as in O.forward_sparse.  Returns (dobj (n, 3), logits (n,), flips): flips as O.loss_and_grads_forced gives
    them when masks are passed, else None."""
    if masks is not None:
        O._FORCED, O._FLIPS = [m for m in masks], []
    try:
        o = obj.detach().clone().requires_grad_(True)
        _, logits = O.forward_sparse(w, o, snd, rcv, return_logits=True, c_scale=c_scale, q_scale=q_scale)
        assert not O._FORCED, 'unused masks'
        dl = torch.as_tensor(dlogits, dtype=o.dtype)
        (g,) = torch.autograd.grad((logits * dl).sum(), [o], allow_unused=True)
        if g is None:
            g = torch.zeros_like(o)
        return g.detach(), logits.detach(), O._FLIPS
    finally:
        O._FORCED, O._FLIPS = None, None
