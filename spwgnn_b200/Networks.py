"""Drop-in for /root/reference/src/Networks.py: `PropagationNetwork().getModel(n_objects, object_dim)`
returns an object with the Keras calls the reference's callers make -- `.fit(x_dict, y_dict,
batch_size=, epochs=, validation_split=, shuffle=, verbose=)` (main.py:92-98) and `.predict(x_dict)`
-> ndarray (B, N, 1) (TowerCreator.py:430-431, JengaBuilder.py:328-329) -- backed by the sm_100a
kernels in libspwgnn.so.  Differences by design:
  * one set of weights serves every n_objects (the reference re-wires shared MLPs per N,
    Networks.py:17-18,40-56); `getModel` still caches one facade per N like `self.Nets`;
  * besides the dense one-hot dict, `predict_towers` / `fit_towers` take ragged raw poses and build
    the relations on the GPU (no O(N^3) tensors);
  * logits are exposed (`predict_logits`); `predict_tower_sums` returns the per-tower sum of block
    probabilities the demolish searches use (JengaBuilder.py:254-256, TowerCreator.py:299-300), and
    `score_removals` / `score_drops` run a whole demolish search (candidate towers, scores, argmin)
    as one packed inference instead of N or 100 batch-1 predicts;
  * `PropagationNetwork(small_batches=True)` sends inference on small batches of small towers through
    `Engine.forward_towers` (one CTA per tower, one launch) instead of the tiled `Engine.forward`;
  * `stability_gradients` differentiates each tower's demolish score with respect to its block poses, and
    `relation_gradients` with respect to the weights of its relations (which contacts hold the tower up);
  * `input_gradients` differentiates predict with respect to all four inputs of the reference's dict (K.gradients).
"""
import os
import sys

import numpy as np
import torch

try:
    from .engine import Engine, PropNetObjFunction
    from .graph import TowerBatch, REL_THRESHOLD
    from ._lib import SpwError
    from .Blocks import RelationalModel, ObjectModel
except ImportError:      # imported as top-level `Networks` (reference style: `from Networks import *`)
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    from spwgnn_b200.engine import Engine, PropNetObjFunction
    from spwgnn_b200.graph import TowerBatch, REL_THRESHOLD
    from spwgnn_b200._lib import SpwError
    from spwgnn_b200.Blocks import RelationalModel, ObjectModel

__all__ = ['PropagationNetwork', 'PropagationModel', 'History', 'RelationalModel', 'ObjectModel']


class History:
    def __init__(self):
        self.history = {}
        self.epoch = []

    def _add(self, epoch, **kv):
        self.epoch.append(epoch)
        for k, v in kv.items():
            self.history.setdefault(k, []).append(v)


class PropagationNetwork:
    """Networks.py:12-104.  Holds the shared weights (one Engine, created when a model first computes) and a per-N facade
    cache like the reference's `self.Nets`; `relnet / objnet / relnetp / objnetp` are the four shared MLPs (Networks.py:40-56)
    as Blocks descriptors.

    small_batches=True: every inference call of the models (predict, predict_logits, predict_towers, predict_tower_sums,
    score_removals, score_drops, evaluate and the validation pass of fit / fit_towers) uses Engine.forward_towers when the
    batch's towers have at most `small_max_nodes` blocks and there are at most `small_max_towers` of them, and the tiled
    Engine.forward otherwise; stability_gradients and relation_gradients use Engine.gradients_towers (the backward pass of
    the same kernel's forward, one launch) under the same limits, so predictions and their gradients come from one fp32
    function.  Training and input_gradients are unchanged.  On that path a tower's probabilities and gradients do not depend
    on the rest of the batch, bit for bit: a packed demolish search (score_removals, score_drops) gives exactly the sums of
    one batch-1 predict per candidate, and a packed stability_gradients call the gradients of one batch-1 call per tower.
    Off by default: the two paths agree to fp32 rounding, not bit for bit, and the tiled path is faster."""

    # The limits keep forward_towers where its cost stays within about 2x of the tiled path.  It wins nowhere yet: measured
    # on one B200 at a 1000 W power limit (tools/bench_small.py, profiles/small_r05.json), device time per call, tiled vs
    # forward_towers: C1 (8-block TowerCreator towers) 248 vs 408 us at 1 tower, 276 vs 402 us at 32; fully connected 10-block
    # towers 249 vs 533 us at 1, 281 vs 530 us at 128, then 385 vs 2097 us at 512 and 883 vs 7385 us at 2048; one fully
    # connected tower of 16 / 24 / 32 blocks 249 vs 1194 / 2548 / 4366 us.  What the flag buys is batch invariance.
    small_max_nodes = 10
    small_max_towers = 128

    def __init__(self, device='cuda', seed=0, small_batches=False):
        self.Nets = {}
        self.small_batches = bool(small_batches)
        self.set_weights = False
        self._device, self._seed = device, seed
        self._engine = None
        self.relnet = self.objnet = self.relnetp = self.objnetp = None

    @property
    def engine(self):
        if self._engine is None:                        # deferred: getModel() itself needs no GPU (main.py:36-37 runs before any data exists)
            self._engine = Engine(self._device, self._seed)
        return self._engine

    def getModel(self, n_objects, object_dim=3, relation_dim=1):
        if n_objects in self.Nets:                      # Networks.py:17-18
            return self.Nets[n_objects]
        if object_dim != 3:
            raise SpwError('object_dim=%d: only object_dim=3 is well defined in the reference (with 2 the object '
                           'encoder is declared 2-wide but fed 1 feature, Networks.py:42,47,70-73)' % object_dim)
        n_relations = n_objects * (n_objects - 1)       # Networks.py:20
        if not self.set_weights:                        # Networks.py:46-56: the four MLPs are created once and shared by every model size
            self.relnet = RelationalModel((n_relations,), 2, [150, 150, 150, 150], prefix='rm', network=self).getRelnet()
            self.objnet = ObjectModel((n_objects,), 2, [100, 100], prefix='om', network=self).getObjnet()
            self.relnetp = RelationalModel((n_relations,), 350, [150, 150, 100], prefix='rmp', network=self).getRelnet()
            self.objnetp = ObjectModel((n_objects,), 300, [100, 101], prefix='omp', network=self).getObjnet()
            self.set_weights = True
        model = PropagationModel(self, n_objects)
        self.Nets[n_objects] = model
        return model


class PropagationModel:
    """The compiled-model facade: Adam(lr=5e-4) + binary_crossentropy + binary_accuracy (Networks.py:101-102)."""

    def __init__(self, network, n_objects):
        self.network = network
        self.n_objects = n_objects
        self.lr = 5e-4               # optimizers.Adam(lr=0.0005), Networks.py:101
        self.dropout_rate = 0.1      # Dropout(0.1) on both encodings, train only, Networks.py:77-78
        self._drop_seed = 0x5EED0001

    @property
    def engine(self):
        return self.network.engine

    # ---- inference -----------------------------------------------------------------------------
    def _small(self, batch):
        """True when the batch takes the per-tower kernels: small_batches=True and the batch inside the network's limits."""
        net = self.network
        return net.small_batches and batch.max_nodes <= net.small_max_nodes and batch.n_towers <= net.small_max_towers

    def _infer(self, batch, want_probs=True):
        """The inference forward of every call below: forward_towers for small batches of small towers when the network
        was built with small_batches=True, the tiled forward otherwise."""
        eng = self.engine
        if self._small(batch):
            return eng.forward_towers(batch, want_probs=want_probs)
        return eng.forward(batch, training=False, want_probs=want_probs)

    def _batch_from_dict(self, x, sel=None):
        obj = np.asarray(x['objects'])
        rs, rr = np.asarray(x['sender_relations']), np.asarray(x['receiver_relations'])
        if sel is not None:
            obj, rs, rr = obj[sel], rs[sel], rr[sel]
        if obj.shape[1] != self.n_objects:
            raise SpwError('model built for %d objects, got %d' % (self.n_objects, obj.shape[1]))
        return TowerBatch.from_dense_relations(obj, rs, rr, device=self.engine.device)

    def predict(self, x, batch_size=None, verbose=0):
        """x: the reference's dict ('objects', 'sender_relations', 'receiver_relations', 'propagation';
        the all-zero 'propagation' seed is implied and ignored).  Returns float32 (B, N, 1)."""
        B, N = np.asarray(x['objects']).shape[:2]
        batch = self._batch_from_dict(x)
        _, probs = self._infer(batch)
        return probs.reshape(B, N, 1).cpu().numpy()

    def predict_logits(self, x):
        B, N = np.asarray(x['objects']).shape[:2]
        logits, _ = self._infer(self._batch_from_dict(x))
        return logits.reshape(B, N, 1).cpu().numpy()

    def predict_towers(self, towers, inference_glue=True, thr=REL_THRESHOLD, fully_connected=False):
        """Fast path: list of (N_t, 3) RAW [x, y, width] arrays (mixed sizes allowed).  With
        inference_glue=True the relations are built as the reference's predict_stabilities does
        (positions/170 thresholded against 170, i.e. fully connected).  Returns a list of (N_t,) arrays."""
        batch = TowerBatch.from_towers(towers, thr=thr, fully_connected=fully_connected,
                                       inference_glue=inference_glue, device=self.engine.device)
        _, probs = self._infer(batch)
        p = probs.cpu().numpy()
        off = batch.node_off_host
        return [p[off[t]:off[t + 1]] for t in range(batch.n_towers)]

    def _tower_sums(self, batch, probs, want_argmin=True):
        """Per-tower sum of block probabilities (double, block order) and the index of the first minimum, on the GPU."""
        api, dev = self.engine.api, self.engine.device
        sums = torch.empty(max(batch.n_towers, 1), dtype=torch.float64, device=dev)
        amin = torch.zeros(1, dtype=torch.int32, device=dev)
        with torch.cuda.device(dev):
            api.check(api.dll.spw_tower_sums(probs.data_ptr(), batch.node_off.data_ptr(), batch.n_towers, sums.data_ptr(),
                                             amin.data_ptr() if want_argmin else None, torch.cuda.current_stream(dev).cuda_stream))
        return sums[:batch.n_towers], amin

    def predict_tower_sums(self, towers, **kw):
        """Per-tower sum of block probabilities (the demolish searches' score, JengaBuilder.py:254-256), computed on the GPU."""
        batch = TowerBatch.from_towers(towers, device=self.engine.device, **kw)
        _, probs = self._infer(batch)
        return self._tower_sums(batch, probs, want_argmin=False)[0].cpu().numpy()

    def _score_candidates(self, obj, pos, n_cand, n_each, inference_glue, thr):
        node_off = np.arange(n_cand + 1, dtype=np.int64) * n_each
        batch = TowerBatch.from_poses(obj, node_off, pos, thr=thr, fully_connected=False, device=self.engine.device, max_nodes=n_each)
        _, probs = self._infer(batch)
        sums, amin = self._tower_sums(batch, probs)
        return sums.cpu().numpy(), int(amin.item())

    def score_removals(self, tower, inference_glue=True, thr=REL_THRESHOLD):
        """JengaBuilder.remove_to_demolish (JengaBuilder.py:236-269) as ONE packed inference: candidate c is `tower`
        ((N, 3) raw [x, y, width]) without block c.  The candidates are built on the device, scored together, summed per
        candidate and arg-minimised by kernels.  Returns (box_stabilities (N,) float64, remove_index) -- the reference's
        `box_stabilities` and `np.argmin(box_stabilities)`.  inference_glue=True builds the relations as the reference's
        predict glue does (positions / 170 against the threshold 170: fully connected, JengaBuilder.py:309-323)."""
        api, dev = self.engine.api, self.engine.device
        raw = torch.as_tensor(np.ascontiguousarray(np.asarray(tower, dtype=np.float64).reshape(-1, 3))).to(dev)
        N = raw.shape[0]
        if N < 2:
            raise SpwError('score_removals needs at least two blocks')
        obj = torch.empty(N * (N - 1), 3, dtype=torch.float32, device=dev)
        pos = torch.empty(N * (N - 1), 2, dtype=torch.float64, device=dev)
        with torch.cuda.device(dev):
            api.check(api.dll.spw_candidates_remove(raw.data_ptr(), N, obj.data_ptr(), pos.data_ptr(), int(bool(inference_glue)),
                                                    torch.cuda.current_stream(dev).cuda_stream))
        return self._score_candidates(obj, pos, N, N - 1, inference_glue, thr)

    def score_drops(self, tower, poses, width=150.0, inference_glue=True, thr=REL_THRESHOLD):
        """TowerCreator.drop_to_demolish (TowerCreator.py:276-319) as ONE packed inference: candidate c is `tower`
        ((N, 3) raw) plus a dropped block at poses[c] = [x, y], which becomes object 0 (TowerCreator.py:451).
        Returns (stability sums (K,) float64, index_min)."""
        api, dev = self.engine.api, self.engine.device
        raw = torch.as_tensor(np.ascontiguousarray(np.asarray(tower, dtype=np.float64).reshape(-1, 3))).to(dev)
        ps = torch.as_tensor(np.ascontiguousarray(np.asarray(poses, dtype=np.float64).reshape(-1, 2))).to(dev)
        N, K = raw.shape[0], ps.shape[0]
        obj = torch.empty(max(K * (N + 1), 1), 3, dtype=torch.float32, device=dev)
        pos = torch.empty(max(K * (N + 1), 1), 2, dtype=torch.float64, device=dev)
        with torch.cuda.device(dev):
            api.check(api.dll.spw_candidates_drop(raw.data_ptr(), N, ps.data_ptr(), K, float(width), obj.data_ptr(), pos.data_ptr(),
                                                  int(bool(inference_glue)), torch.cuda.current_stream(dev).cuda_stream))
        return self._score_candidates(obj[:K * (N + 1)], pos[:K * (N + 1)], K, N + 1, inference_glue, thr)

    def stability_gradients(self, towers, inference_glue=True, thr=REL_THRESHOLD, fully_connected=False):
        """Gradient of each tower's demolish score sum_i p_i (JengaBuilder.py:254-256) with respect to its blocks' RAW
        [x, y, width]: a list of (N_t, 3) float64 arrays, in pixels.  `towers` and the relation options are those of
        predict_towers; the relations are held fixed (they come from a distance threshold, which is piecewise constant).
        Towers are independent, so one packed backward pass of the batch's total gives every tower the gradient of its own
        sum.  p = sigmoid(logits) in fp32; the factor 1/170 of the feature normalisation is applied in float64.  The path is
        the one predict takes: Engine.gradients_towers (seed dprobs = 1) when _infer would use forward_towers, else the tiled
        PropNetObjFunction."""
        if not towers:
            return []
        eng = self.engine
        batch = TowerBatch.from_towers(towers, thr=thr, fully_connected=fully_connected, inference_glue=inference_glue,
                                       device=eng.device)
        if self._small(batch):
            ones = torch.ones(batch.n_nodes, dtype=torch.float32, device=eng.device)
            _, g, _ = eng.gradients_towers(batch, dprobs=ones)
        else:
            obj = batch.obj.detach().clone().requires_grad_(True)
            with torch.enable_grad():
                p = torch.sigmoid(PropNetObjFunction.apply(obj, eng, batch))
                (g,) = torch.autograd.grad(p.sum(), [obj])
        g = g.cpu().numpy().astype(np.float64) / REL_THRESHOLD
        off = batch.node_off_host
        return [g[off[t]:off[t + 1]] for t in range(batch.n_towers)]

    def relation_gradients(self, towers, inference_glue=True, thr=REL_THRESHOLD, fully_connected=False):
        """Gradient of each tower's demolish score sum_i p_i with respect to the weights of its relations: relation e = (s -> r)
        gets a weight w_e multiplying both of its one-hot entries in the reference's sender_relations / receiver_relations, and
        the value is d(sum_i p_i)/dw_e at w = 1 (the sum of the Keras gradients with respect to those two entries).  Returns, per
        tower, (pairs, grads): pairs (E_t, 2) int64 local (sender, receiver) block indices of the tower's active relations in
        the reference's slot order (main.py:69-81: sender outer, receiver inner), grads (E_t,) float64.  Weights are
        dimensionless, so no 1/170 factor applies.  `towers` and the relation options are those of predict_towers; one packed
        pass of Engine.relation_gradients with the seed p (1 - p) serves the whole batch, or of Engine.gradients_towers with
        dprobs = 1 when _infer would use forward_towers (small_batches=True)."""
        if not towers:
            return []
        eng = self.engine
        batch = TowerBatch.from_towers(towers, thr=thr, fully_connected=fully_connected, inference_glue=inference_glue,
                                       device=eng.device)

        def seed(z):
            p = torch.sigmoid(z)
            return p * (1 - p)
        if self._small(batch):
            ones = torch.ones(batch.n_nodes, dtype=torch.float32, device=eng.device)
            _, _, drel = eng.gradients_towers(batch, dprobs=ones, want_drel=True)
        else:
            drel, _ = eng.relation_gradients(batch, seed)
        E, off = batch.n_edges, batch.node_off_host
        if E == 0:
            return [(np.zeros((0, 2), np.int64), np.zeros(0, np.float64)) for _ in range(batch.n_towers)]
        o = batch.out_pos[:E].long()                      # slot (sender-major) order -> receiver-major row
        snd = batch.in_snd[:E].long()[o].cpu().numpy()
        rcv = batch.in_rcv[:E].long()[o].cpu().numpy()
        val = drel[o].cpu().numpy().astype(np.float64)
        eo = batch.out_off[:batch.n_nodes + 1].cpu().numpy().astype(np.int64)[off]
        return [(np.stack([snd[eo[t]:eo[t + 1]], rcv[eo[t]:eo[t + 1]]], 1) - off[t], val[eo[t]:eo[t + 1]])
                for t in range(batch.n_towers)]

    def input_gradients(self, x, dprobs=None):
        """The gradient of sum(dprobs * p) with respect to the four inputs of the reference's model, p = predict(x): what
        K.gradients(model.output, model.inputs, grad_ys=dprobs) returns for the reference's Keras model (Networks.py:22-99).
        x: the reference's dict; dprobs: (B, N, 1) or (B, N), default ones.  Returns a dict with the keys and shapes of x
        ('objects' (B, N, 3), 'sender_relations' / 'receiver_relations' (B, N, R), 'propagation' (B, N, 100)), float32: the
        gradients at every entry of the relation tensors, zero and inactive ones included, and at propagation = 0 (the forward
        implies that seed, so a nonzero 'propagation' raises).  One packed pass of Engine.input_gradients with the seed
        dprobs * p (1 - p), p = sigmoid(logits) in fp32."""
        obj = np.asarray(x['objects'])
        B, N = obj.shape[:2]
        R = np.asarray(x['sender_relations']).shape[2]
        if x.get('propagation') is not None and np.any(np.asarray(x['propagation']) != 0):
            raise SpwError('input_gradients: the forward pass implies propagation = 0; a nonzero propagation input is not supported')
        eng = self.engine
        if dprobs is None:
            dp = torch.ones(B * N, dtype=torch.float32, device=eng.device)
        else:
            dp = torch.as_tensor(np.asarray(dprobs, dtype=np.float32))
            if tuple(dp.shape) not in ((B, N, 1), (B, N)):
                raise SpwError('input_gradients: dprobs must be (%d, %d, 1) or (%d, %d), got %s' % (B, N, B, N, tuple(dp.shape)))
            dp = dp.reshape(B * N).to(eng.device)
        batch = self._batch_from_dict(x)

        def seed(z):
            p = torch.sigmoid(z)
            return dp * (p * (1 - p))
        drs, drr, free, dprop, dobj = eng.input_gradients(batch, seed)
        d_rs = torch.zeros(B, N, R, dtype=torch.float32, device=eng.device)
        d_rr = free.reshape(B, N, 1).expand(B, N, R).contiguous()        # inactive slots: 0 and drr_free
        E = batch.n_edges
        if E:
            snd, _, slot = batch.slot_list                                  # slot (sender-major) order
            o, b, sl = batch.out_pos[:E].long(), snd[:E].long() // N, slot[:E].long()
            d_rs[b, :, sl] = drs[o, :N]
            d_rr[b, :, sl] = drr[o, :N]
        return {'objects': dobj.reshape(B, N, 3).cpu().numpy(), 'sender_relations': d_rs.cpu().numpy(),
                'receiver_relations': d_rr.cpu().numpy(), 'propagation': dprop.reshape(B, N, 100).cpu().numpy()}

    # ---- training ------------------------------------------------------------------------------
    def train_on_batch(self, batch, target):
        """One optimiser step on a packed batch; returns (mean loss, binary accuracy)."""
        eng = self.engine
        self._drop_seed = (self._drop_seed * 6364136223846793005 + 1442695040888963407) & 0xFFFFFFFFFFFFFFFF
        stats = eng.loss_and_grads(batch, target, dropout_rate=self.dropout_rate, dropout_seed=self._drop_seed)
        eng.adam_step(lr=self.lr)
        s = stats.cpu().numpy() / max(batch.n_nodes, 1)
        return float(s[0]), float(s[1])

    def test_on_batch(self, batch, target):
        eng = self.engine
        logits, _ = self._infer(batch, want_probs=False)
        _, stats = eng.bce_seed(logits, target, max(batch.n_nodes, 1))
        s = stats.cpu().numpy() / max(batch.n_nodes, 1)
        return float(s[0]), float(s[1])

    def fit(self, x, y, batch_size=32, epochs=1, validation_split=0.0, shuffle=True, verbose=1, seed=None):
        """Keras semantics: the LAST `validation_split` fraction is held out before shuffling; each epoch
        shuffles the rest and steps once per mini-batch; epoch metrics are sample-weighted means."""
        tgt_all = np.asarray(y['target'] if isinstance(y, dict) else y, dtype=np.float32)
        B = tgt_all.shape[0]
        n_tr = int(B * (1. - validation_split)) if validation_split else B     # Keras: split_at = int(len(x) * (1 - split))
        n_val = B - n_tr
        rng = np.random.default_rng(seed)
        dev = self.engine.device
        hist = History()
        for ep in range(epochs):
            order = rng.permutation(n_tr) if shuffle else np.arange(n_tr)
            tl = ta = 0.0
            for s0 in range(0, n_tr, batch_size):
                sel = np.sort(order[s0:s0 + batch_size]) if not shuffle else order[s0:s0 + batch_size]
                batch = self._batch_from_dict(x, sel)
                tgt = torch.as_tensor(tgt_all[sel].reshape(-1)).to(dev)
                l, a = self.train_on_batch(batch, tgt)
                tl += l * len(sel); ta += a * len(sel)
            rec = dict(loss=tl / max(n_tr, 1), binary_accuracy=ta / max(n_tr, 1))
            if n_val:
                vl = va = 0.0
                for s0 in range(n_tr, B, batch_size):
                    sel = np.arange(s0, min(s0 + batch_size, B))
                    batch = self._batch_from_dict(x, sel)
                    tgt = torch.as_tensor(tgt_all[sel].reshape(-1)).to(dev)
                    l, a = self.test_on_batch(batch, tgt)
                    vl += l * len(sel); va += a * len(sel)
                rec.update(val_loss=vl / n_val, val_binary_accuracy=va / n_val)
            hist._add(ep, **rec)
            if verbose:
                print('Epoch %d/%d - ' % (ep + 1, epochs) + ' - '.join('%s: %.4f' % kv for kv in rec.items()))
        return hist

    def fit_towers(self, towers, labels, batch_size=32, epochs=1, validation_split=0.0, shuffle=True, verbose=1,
                   seed=None, thr=REL_THRESHOLD, fully_connected=False):
        """Fast-path training: `towers` = list of (N_t, 3) RAW [x, y, width] arrays (mixed sizes allowed),
        `labels` = list of (N_t,) 0/1 arrays.  Relations are built on the GPU from the raw positions exactly as
        main.py:66-81 does (threshold 170 on raw pixels); everything else follows `fit`."""
        B = len(towers)
        n_tr = int(B * (1. - validation_split)) if validation_split else B
        n_val = B - n_tr
        rng = np.random.default_rng(seed)
        dev = self.engine.device
        hist = History()

        def make(sel):
            batch = TowerBatch.from_towers([towers[i] for i in sel], thr=thr, fully_connected=fully_connected, device=dev)
            tgt = torch.as_tensor(np.concatenate([np.asarray(labels[i], dtype=np.float32).reshape(-1) for i in sel])).to(dev)
            return batch, tgt
        for ep in range(epochs):
            order = rng.permutation(n_tr) if shuffle else np.arange(n_tr)
            tl = ta = 0.0
            nb = 0
            for s0 in range(0, n_tr, batch_size):
                sel = order[s0:s0 + batch_size]
                batch, tgt = make(sel)
                l, a = self.train_on_batch(batch, tgt)
                tl += l * batch.n_nodes; ta += a * batch.n_nodes; nb += batch.n_nodes
            rec = dict(loss=tl / max(nb, 1), binary_accuracy=ta / max(nb, 1))
            if n_val:
                vl = va = 0.0
                nv = 0
                for s0 in range(n_tr, B, batch_size):
                    batch, tgt = make(np.arange(s0, min(s0 + batch_size, B)))
                    l, a = self.test_on_batch(batch, tgt)
                    vl += l * batch.n_nodes; va += a * batch.n_nodes; nv += batch.n_nodes
                rec.update(val_loss=vl / max(nv, 1), val_binary_accuracy=va / max(nv, 1))
            hist._add(ep, **rec)
            if verbose:
                print('Epoch %d/%d - ' % (ep + 1, epochs) + ' - '.join('%s: %.4f' % kv for kv in rec.items()))
        return hist

    def evaluate(self, x, y, batch_size=32, verbose=0):
        tgt_all = np.asarray(y['target'] if isinstance(y, dict) else y, dtype=np.float32)
        B = tgt_all.shape[0]
        tl = ta = 0.0
        for s0 in range(0, B, batch_size):
            sel = np.arange(s0, min(s0 + batch_size, B))
            batch = self._batch_from_dict(x, sel)
            l, a = self.test_on_batch(batch, torch.as_tensor(tgt_all[sel].reshape(-1)).to(self.engine.device))
            tl += l * len(sel); ta += a * len(sel)
        return [tl / max(B, 1), ta / max(B, 1)]

    # ---- weights -------------------------------------------------------------------------------
    def get_weights(self):
        return [v.cpu().numpy() for v in self.engine.params.to_dict().values()]

    def set_weights_dict(self, d):
        self.engine.params.load_dict(d)
