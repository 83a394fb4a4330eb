"""Host-side driver of the CUDA hot path: forward, loss seed, backward, Keras-form Adam.

Everything numerical happens inside libspwgnn.so (include/spwgnn.h); torch supplies device
memory, streams and (for data parallelism) torch.distributed.  No CPU fallback exists.
"""
import ctypes
import os

import torch

from ._capi import CApi
from ._lib import lib, require_cuda, SpwError
from .graph import TowerBatch, _stream_ptr
from .params import ParamBuffer, FLAT_SIZE, STATS_TAIL

SMALL_MAX_NODES = 32      # SPW_SMALL_MAX_NODES (include/spwgnn.h): blocks per tower of forward_towers


class Workspace:
    """Grow-only device scratch shared by forward and backward (caller-owned, see spwgnn.h)."""

    def __init__(self, device):
        self.device = device
        self.buf = None

    def get(self, nbytes):
        if self.buf is None or self.buf.numel() < nbytes:
            self.buf = None
            self.buf = torch.empty(int(nbytes * 1.1) + 256, dtype=torch.uint8, device=self.device)
        return self.buf


def keras_adam_update_(params, grads, state, lr=5e-4, beta1=0.9, beta2=0.999, eps=1e-7):
    """One step of Keras 2.2 Adam (the optimiser main.py trains with: `optimizers.Adam(lr=0.0005)`, Networks.py:101) on flat
    tensors, in place:  t += 1;  lr_t = lr sqrt(1 - b2^t) / (1 - b1^t);  m = b1 m + (1 - b1) g;  v = b2 v + (1 - b2) g^2;
    p -= lr_t m / (sqrt(v) + eps)  with eps = K.epsilon() = 1e-7 OUTSIDE the square root and no bias-corrected m, v (that is
    what distinguishes it from torch.optim.Adam).  state: dict(t, m, v)."""
    state['t'] += 1
    t = state['t']
    state['m'].mul_(beta1).add_(grads, alpha=1 - beta1)
    state['v'].mul_(beta2).addcmul_(grads, grads, value=1 - beta2)
    lr_t = lr * (1 - beta2 ** t) ** 0.5 / (1 - beta1 ** t)
    params.addcdiv_(state['m'], state['v'].sqrt().add_(eps), value=-lr_t)
    return params


class Engine:
    """One replica of the network on one GPU."""

    def __init__(self, device='cuda', seed=0):
        require_cuda()
        self.api = lib()
        self.device = torch.device(device)
        self.params = ParamBuffer(self.device).glorot_init(seed)
        self.grads_buffer = torch.zeros(FLAT_SIZE + STATS_TAIL, dtype=torch.float32, device=self.device)   # gradients + stats tail
        self.grads = ParamBuffer(self.device, flat=self.grads_buffer[:FLAT_SIZE])
        self.ws = Workspace(self.device)        # training: must survive until backward
        self.ws_inf = Workspace(self.device)    # inference: separate, so a predict() between forward and
                                                # backward of a training step cannot clobber saved state
        self.ws_small = Workspace(self.device)  # forward_towers: separate from both for the same reason
        self._adam = None
        self._fwd = None
        # small inference batches are launch-bound (~60 launches for microseconds of work: the reference's GUI loops predict
        # one tower at a time, JengaBuilder.py:328): the forward pass of a given (towers, blocks, relations) shape is
        # captured once as a CUDA graph over static buffers and replayed
        self._graphs = {}
        self.graph_max_edges = 0 if os.environ.get('SPW_NO_GRAPHS') else 8192

    # ---- forward ------------------------------------------------------------------------------
    def _forward_graph(self, batch, want_probs):
        """Inference forward of a small batch through a captured CUDA graph (one per shape, least recently used evicted)."""
        api, n, E, T = self.api, batch.n_nodes, batch.n_edges, batch.n_towers
        key = (T, n, E, bool(want_probs))
        srcs = (batch.obj, batch.node_off, batch.in_off, batch.in_snd, batch.in_rcv, batch.out_off, batch.out_pos)
        ent = self._graphs.get(key)
        if ent is None:
            if len(self._graphs) >= 64:
                self._graphs.pop(next(iter(self._graphs)))
            with torch.cuda.device(self.device):
                st = [torch.empty_like(t) for t in srcs]
                logits = torch.empty(max(n, 1), dtype=torch.float32, device=self.device)
                probs = torch.empty(max(n, 1), dtype=torch.float32, device=self.device) if want_probs else None
                ws = torch.empty(int(api.dll.spw_workspace_bytes(n, E, 0)) + 256, dtype=torch.uint8, device=self.device)
                cg = CApi.graph(T, n, E, *[t.data_ptr() for t in st[1:]])
                wp = self.params.c_struct()

                def run():
                    api.check(api.dll.spw_forward(ctypes.byref(wp), ctypes.byref(cg), st[0].data_ptr(), logits.data_ptr(),
                                                  probs.data_ptr() if want_probs else None, ws.data_ptr(), ws.numel(), 0, 0.0, 0,
                                                  _stream_ptr(self.device)))
                for d, t in zip(st, srcs):
                    d.copy_(t)
                side = torch.cuda.Stream(self.device)
                side.wait_stream(torch.cuda.current_stream(self.device))
                with torch.cuda.stream(side):
                    run()                                   # un-captured once: function attributes, lazy statics
                torch.cuda.current_stream(self.device).wait_stream(side)
                g = torch.cuda.CUDAGraph()
                with torch.cuda.graph(g):
                    run()
            ent = (g, st, logits, probs, ws, cg, wp)
            self._graphs[key] = ent
        else:
            self._graphs[key] = self._graphs.pop(key)       # most recently used last
        g, st, logits, probs = ent[0], ent[1], ent[2], ent[3]
        with torch.cuda.device(self.device):
            for d, t in zip(st, srcs):
                d.copy_(t, non_blocking=True)
            g.replay()
            return logits[:n].clone(), (probs[:n].clone() if want_probs else None)   # the static buffers are reused by the next replay

    def forward(self, batch: TowerBatch, training=False, want_probs=True, dropout_rate=0.0, dropout_seed=0):
        """Per-block logits (and sigmoid probabilities) for a packed batch (Networks.py:58-96)."""
        api, n = self.api, batch.n_nodes
        if not training and 0 < batch.n_edges <= self.graph_max_edges and n > 0 and not torch.cuda.is_current_stream_capturing():
            return self._forward_graph(batch, want_probs)
        with torch.cuda.device(self.device):        # kernels launch on the current device: make it this engine's
            logits = torch.empty(max(n, 1), dtype=torch.float32, device=self.device)
            probs = torch.empty(max(n, 1), dtype=torch.float32, device=self.device) if want_probs else None
            nbytes = api.dll.spw_workspace_bytes(n, batch.n_edges, int(training))
            ws = (self.ws if training else self.ws_inf).get(nbytes)
            wp = self.params.c_struct()
            api.check(api.dll.spw_forward(ctypes.byref(wp), ctypes.byref(batch.c_graph), batch.obj.data_ptr(),
                                          logits.data_ptr(), probs.data_ptr() if want_probs else None, ws.data_ptr(),
                                          ws.numel(), int(training), float(dropout_rate), int(dropout_seed),
                                          _stream_ptr(self.device)))
        if training:
            self._fwd = (batch, ws, logits, float(dropout_rate))
        return logits[:n], (probs[:n] if want_probs else None)

    def forward_towers(self, batch: TowerBatch, want_probs=True):
        """Inference with one CTA per tower in ONE kernel launch (spw_forward_towers): the function of `forward(training=False)`
        for towers of at most SMALL_MAX_NODES blocks, computed in plain fp32 with every sum in a fixed order.  A tower's
        results are the same bits whatever else is in the batch.  Returns (logits[:n], probs[:n] or None)."""
        if batch.max_nodes > SMALL_MAX_NODES:
            raise SpwError('forward_towers: towers of up to %d blocks, this batch allows %d' % (SMALL_MAX_NODES, batch.max_nodes))
        api, n = self.api, batch.n_nodes
        with torch.cuda.device(self.device):
            logits = torch.empty(max(n, 1), dtype=torch.float32, device=self.device)
            probs = torch.empty(max(n, 1), dtype=torch.float32, device=self.device) if want_probs else None
            ws = self.ws_small.get(api.dll.spw_forward_towers_bytes(n, batch.n_edges))
            wp = self.params.c_struct()
            api.check(api.dll.spw_forward_towers(ctypes.byref(wp), ctypes.byref(batch.c_graph), int(batch.max_nodes),
                                                 batch.obj.data_ptr(), logits.data_ptr(), probs.data_ptr() if want_probs else None,
                                                 ws.data_ptr(), ws.numel(), _stream_ptr(self.device)))
        return logits[:n], (probs[:n] if want_probs else None)

    # ---- loss seed + backward -------------------------------------------------------------------
    def bce_seed(self, logits, target, count):
        """Keras binary_crossentropy (Networks.py:102).  Returns (dlogits, stats) with stats a device
        double[2] = [sum of per-block losses, number of correct predictions]."""
        api, n = self.api, logits.numel()
        with torch.cuda.device(self.device):
            dlogits = torch.empty(max(n, 1), dtype=torch.float32, device=self.device)
            stats = torch.zeros(2, dtype=torch.float64, device=self.device)
            api.check(api.dll.spw_bce_grad(logits.data_ptr(), target.data_ptr(), n, float(count), dlogits.data_ptr(),
                                           stats.data_ptr(), _stream_ptr(self.device)))
        return dlogits[:n], stats

    def backward(self, dlogits):
        """Gradients of sum(dlogits*logits) w.r.t. all 22 tensors -> self.grads (overwritten)."""
        if self._fwd is None:
            raise SpwError('backward without a training forward')
        batch, ws, _, rate = self._fwd
        api = self.api
        wp, gp = self.params.c_struct(), self.grads.c_struct()
        dl = dlogits.contiguous()
        with torch.cuda.device(self.device):
            api.check(api.dll.spw_backward(ctypes.byref(wp), ctypes.byref(batch.c_graph), batch.obj.data_ptr(),
                                           dl.data_ptr(), ws.data_ptr(), ws.numel(), ctypes.byref(gp), rate,
                                           _stream_ptr(self.device)))
        return self.grads

    def relation_gradients(self, batch, dlogits):
        """Gradient of sum(dlogits*logits) with respect to the relation weights and the block features, from one pass of
        spw_backward_rel: (drel (n_edges,), dobj (n_nodes, 3)), fp32 on the device.  drel[k] belongs to the receiver-major
        relation batch.in_snd[k] -> batch.in_rcv[k] (include/spwgnn.h says how to reach the slot order); dobj equals
        PropNetObjFunction's gradient bit for bit.  dlogits: (n_nodes,) tensor, or a function of the forward's fp32 logits that
        returns one (for a seed such as p (1 - p)).  The forward pass is PropNetObjFunction's (a training forward at dropout
        rate 0 into a workspace owned by this call), so a training step in flight on this Engine is left alone."""
        api, n, E = self.api, batch.n_nodes, batch.n_edges
        logits, ws, nbytes = _gradient_forward(self, batch, batch.obj.contiguous())
        dl = (dlogits(logits) if callable(dlogits) else dlogits).detach().to(torch.float32).contiguous()
        if dl.shape != (n,) or dl.device != self.device:
            raise SpwError('relation_gradients: dlogits must be (%d,) on %s, got %s on %s' % (n, self.device, tuple(dl.shape), dl.device))
        with torch.cuda.device(self.device):
            drel = torch.empty(E, dtype=torch.float32, device=self.device)
            dobj = torch.empty(n, 3, dtype=torch.float32, device=self.device)
            wp = self.params.c_struct()
            api.check(api.dll.spw_backward_rel(ctypes.byref(wp), ctypes.byref(batch.c_graph), batch.obj.data_ptr(), dl.data_ptr(),
                                               ws.data_ptr(), nbytes, 0.0, drel.data_ptr() if E else None, dobj.data_ptr(),
                                               _stream_ptr(self.device)))
        return drel, dobj

    def saved_relu_states(self):
        """The relu states the last training forward left for the backward pass, in the oracle's order of relu layers
        (Networks.py:75-76, then :84-90 per step): a list of 21 bool tensors -- rm layers 0..3 [E][150], om layers 0..1
        [n][100], then per propagation step rmp layer 0, rmp layer 1 [E][150] and omp layer 0 [n][100].  Edge rows are in
        receiver-major order (batch.in_snd / batch.in_rcv).  Parity tests evaluate the fp64 oracle on the same linear branch."""
        if self._fwd is None:
            raise SpwError('saved_relu_states without a training forward')
        batch, ws, _, _ = self._fwd
        n, E = batch.n_nodes, batch.n_edges
        lay = (ctypes.c_int64 * 8)()
        self.api.check(self.api.dll.spw_saved_state_layout(n, E, lay))
        rows, stride, eb, m1, m2, u_off, q_off, q1_off = [int(v) for v in lay]

        def bits(off):                      # byte-slab u8 [20][rows] -> bool [E][150]
            b = ws[off:off + 20 * rows].view(20, rows)[:19, :E]
            return ((b.unsqueeze(-1) >> torch.arange(8, device=b.device, dtype=torch.uint8)) & 1).bool().permute(1, 0, 2).reshape(E, 152)[:, :150]

        def pos(off, rows_alloc, row0):     # float column-slab [25 quads][rows_alloc][4] -> bool [n][100]
            a = ws[off:off + 25 * rows_alloc * 16].view(torch.float32).view(25, rows_alloc, 4)[:, row0:row0 + n]
            return (a.permute(1, 0, 2).reshape(n, 100) > 0)

        out = [bits(eb + i * stride) for i in range(4)] + [pos(q1_off, n, 0), pos(q_off, n, 0)]
        for l in range(5):
            out += [bits(m1 + l * stride), bits(m2 + l * stride), pos(u_off, 5 * n, l * n)]
        return out

    def loss_and_grads(self, batch, target, count=None, dropout_rate=0.0, dropout_seed=0):
        """forward(training) + BCE + backward.  `count` = number of blocks the mean runs over
        (global count under data parallelism).  Returns stats (device double[2])."""
        logits, _ = self.forward(batch, training=True, want_probs=False, dropout_rate=dropout_rate,
                                 dropout_seed=dropout_seed)
        dl, stats = self.bce_seed(logits, target, count if count is not None else max(batch.n_nodes, 1))
        self.backward(dl)
        return stats

    # ---- optimiser (host-side torch on the flat buffers) ----------------------------------------
    def adam_step(self, lr=5e-4, beta1=0.9, beta2=0.999, eps=1e-7):
        """Keras 2.2 Adam (Networks.py:101): lr_t = lr*sqrt(1-b2^t)/(1-b1^t); p -= lr_t*m/(sqrt(v)+eps)."""
        if self._adam is None:
            self._adam = dict(t=0, m=torch.zeros(FLAT_SIZE, device=self.device), v=torch.zeros(FLAT_SIZE, device=self.device))
        keras_adam_update_(self.params.flat, self.grads.flat, self._adam, lr, beta1, beta2, eps)


class PropNetFunction(torch.autograd.Function):
    """torch.autograd bridge: logits = PropNetFunction.apply(flat_params, engine, batch)."""

    @staticmethod
    def forward(ctx, flat_params, engine, batch):
        assert flat_params.data_ptr() == engine.params.flat.data_ptr(), 'pass engine.params.flat'
        logits, _ = engine.forward(batch, training=True, want_probs=False)
        ctx.engine = engine
        ctx.saved = engine._fwd              # the engine keeps ONE training step's state (workspace) in flight
        return logits.clone()

    @staticmethod
    def backward(ctx, dlogits):
        if ctx.engine._fwd is not ctx.saved:
            raise SpwError('PropNetFunction.backward: a later training forward on the same Engine overwrote the state '
                           'saved for this one (one Engine keeps one training step in flight)')
        g = ctx.engine.backward(dlogits)
        return g.flat.clone(), None, None


def _gradient_forward(engine, batch, obj):
    """The forward pass of the input gradients: a training spw_forward at dropout rate 0 of `batch` with features `obj` (n, 3)
    (contiguous fp32 on the engine's device), into a workspace of its own.  Returns (logits, workspace, its size in bytes)."""
    api, n = engine.api, batch.n_nodes
    with torch.cuda.device(engine.device):
        logits = torch.empty(n, dtype=torch.float32, device=engine.device)
        nbytes = api.dll.spw_workspace_bytes(n, batch.n_edges, 1)
        ws = torch.empty(max(nbytes, 1), dtype=torch.uint8, device=engine.device)
        wp = engine.params.c_struct()
        api.check(api.dll.spw_forward(ctypes.byref(wp), ctypes.byref(batch.c_graph), obj.data_ptr(), logits.data_ptr(), None,
                                      ws.data_ptr(), nbytes, 1, 0.0, 0, _stream_ptr(engine.device)))
    return logits, ws, nbytes


class PropNetObjFunction(torch.autograd.Function):
    """torch.autograd bridge for the gradient with respect to the block features: logits = PropNetObjFunction.apply(obj,
    engine, batch).  obj: (n, 3) fp32 on the engine's device, [x, y, width] / 170, used in place of batch.obj; the relations
    of `batch` and the weights are constants (no gradient flows to them, and the weights must not change before backward).

    The forward pass is a training spw_forward at dropout rate 0, whose logits are the inference logits bit for bit, into a
    workspace owned by this call and kept until the autograd graph is freed.  It never touches Engine.ws, so it does not
    disturb a training step in flight, and several calls may be in flight at once.  The backward pass is spw_backward_obj:
    the data gradients of the network without any weight gradient."""

    @staticmethod
    def forward(ctx, obj, engine, batch):
        n = batch.n_nodes
        if obj.shape != (n, 3) or obj.dtype != torch.float32 or obj.device != engine.device:
            raise SpwError('PropNetObjFunction: obj must be (%d, 3) float32 on %s, got %s %s on %s'
                           % (n, engine.device, tuple(obj.shape), obj.dtype, obj.device))
        obj = obj.detach().contiguous()
        logits, ws, nbytes = _gradient_forward(engine, batch, obj)
        ctx.engine, ctx.batch, ctx.obj, ctx.ws, ctx.nbytes = engine, batch, obj, ws, nbytes
        return logits

    @staticmethod
    def backward(ctx, dlogits):
        engine, batch = ctx.engine, ctx.batch
        api, n = engine.api, batch.n_nodes
        dl = dlogits.detach().to(torch.float32).contiguous()
        with torch.cuda.device(engine.device):
            dobj = torch.empty(n, 3, dtype=torch.float32, device=engine.device)
            wp = engine.params.c_struct()
            api.check(api.dll.spw_backward_obj(ctypes.byref(wp), ctypes.byref(batch.c_graph), ctx.obj.data_ptr(), dl.data_ptr(),
                                               ctx.ws.data_ptr(), ctx.nbytes, 0.0, dobj.data_ptr(), _stream_ptr(engine.device)))
        return dobj, None, None
