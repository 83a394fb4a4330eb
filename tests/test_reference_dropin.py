"""Boundary tests against what the reference's own source produced, plus CPU tests of the Keras-facing host logic.

The reference (Keras / TF1, pymunk, pyglet) is not part of this repository and cannot be installed next to it, so its
outputs are stored under tests/golden/:
  * train_n*.npz: what the reference's unmodified `main.train_gnn` handed to `.fit` for a stored trajectory file (the input
    dict after frame padding, the relation loops of main.py:66-81, labelling and /170; the targets; the keyword arguments),
    written by oracle/make_golden.py.  The drop-in must rebuild that call from the same file and take it.
  * reference_layouts.npz: the layouts of JengaBuilder.create_world (JengaBuilder.py:137-192) and TowerCreator.create_world
    + drop_object (TowerCreator.py:106-213, 265-271) under seeded `random`, which the samplers of spwgnn_b200/synth.py must
    reproduce bit for bit.
  * the Keras-form Adam update and the validation split of `fit` against plain restatements.
"""
import json
import os
import random
import subprocess
import sys
import textwrap

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _run(script):
    env = dict(os.environ, PYTHONPATH='')
    res = subprocess.run([sys.executable, '-c', textwrap.dedent(script)], capture_output=True, text=True, env=env, cwd=ROOT, timeout=600)
    assert res.returncode == 0, res.stdout[-2000:] + res.stderr[-4000:]
    return json.loads(res.stdout.strip().splitlines()[-1])


def test_dropin_takes_the_fit_call_of_reference_main_py(golden_dir, tmp_path):
    """In a fresh process with the reference's import layout (main.py star-imports `Networks` and `Blocks` as top-level
    modules), the drop-in provides the names main.py uses without importing Keras or TensorFlow; the project's trajectory
    loader and relation builder rebuild, from the stored trajectory file, the dict main.train_gnn passed to `.fit`; and the
    drop-in model's `.fit` takes that call with main.py's keyword arguments."""
    out = _run('''
        import inspect, json, os, sys
        ROOT, GOLDEN, TMP = %r, %r, %r
        sys.path[:0] = [os.path.join(ROOT, 'spwgnn_b200'), ROOT]
        import numpy as np
        from Networks import *                                 # main.py:3-4
        from Blocks import *
        import Networks, Blocks
        assert os.path.dirname(os.path.abspath(Networks.__file__)) == os.path.join(ROOT, 'spwgnn_b200'), Networks.__file__
        assert os.path.dirname(os.path.abspath(Blocks.__file__)) == os.path.join(ROOT, 'spwgnn_b200'), Blocks.__file__
        assert PropagationNetwork is Networks.PropagationNetwork and RelationalModel is Blocks.RelationalModel
        assert ObjectModel is Blocks.ObjectModel
        from spwgnn_b200 import data as D
        from oracle import propnet as O
        checked, active, slots = 0, 0, 0
        for name in ('train_n2', 'train_n4', 'train_n7', 'train_n9'):
            g = np.load(os.path.join(GOLDEN, name + '.npz'))
            n_obj = int(g['n_objects'])                        # jenga: n_objects = n - 1 (main.py:30-31)
            path = os.path.join(TMP, name + '.txt')
            with open(path, 'w') as f:
                f.write(str(g['traj_json']))
            raw0, y = D.training_arrays(path, n_obj + 1, jenga=True)
            rs, rr = O.build_relations_dense(raw0[:, :, :2], 170.0)
            x = {'objects': raw0 / 170.0, 'sender_relations': rs, 'receiver_relations': rr,
                 'propagation': np.zeros((len(raw0), n_obj, 100))}
            assert np.array_equal(x['objects'], g['objects']) and np.array_equal(y, g['target']), name
            assert np.array_equal(rs, g['sender_relations']) and np.array_equal(rr, g['receiver_relations']), name
            assert list(x['propagation'].shape) == g['propagation_shape'].tolist(), name
            kw = json.loads(str(g['fit_kwargs']))
            assert kw == dict(batch_size=32, epochs=10, validation_split=0.2, shuffle=True, verbose=1), kw
            model = PropagationNetwork().getModel(n_obj)
            assert isinstance(model, Networks.PropagationModel) and model.n_objects == n_obj
            inspect.signature(model.fit).bind(x, {'target': y}, **kw)
            active += int((rs.sum(1) > 0).sum())
            slots += int(rs.shape[0] * rs.shape[2])
            checked += 1
        assert not any(m == 'keras' or m.startswith('keras.') or m.startswith('tensorflow') for m in sys.modules), 'Keras / TF got imported'
        print(json.dumps(dict(ok=True, checked=checked, active_relations=active, slots=slots)))
    ''' % (ROOT, golden_dir, str(tmp_path)))
    assert out['ok'] and out['checked'] == 4 and 0 < out['active_relations'] < out['slots']


def test_layout_samplers_are_pinned_to_the_reference(golden_dir):
    """synth.g_jenga / synth.g_tower against the reference's JengaBuilder / TowerCreator layouts for the same seeds
    (`random.seed(s)` before the reference builds a world; `random.Random(s)` here).  The stored layouts were recorded from
    synth.py as it stood when a test that ran both samplers side by side last found them equal bit for bit."""
    from spwgnn_b200 import synth
    z = np.load(os.path.join(golden_dir, 'reference_layouts.npz'))
    checked = 0
    for kind, fn, extra in (('jenga', synth.g_jenga, 0), ('tower', synth.g_tower, 1)):   # tower: + the dropped block, object 0
        refs = np.split(z[kind + '_layouts'], np.cumsum(z[kind + '_rows'])[:-1])
        for n, s, ref in zip(z[kind + '_n'], z[kind + '_seed'], refs):
            assert len(ref) == n + extra, (kind, n, s)
            got = fn(int(n), random.Random(int(s)))
            assert ref.shape == got.shape and np.array_equal(ref, got), (kind, n, s)
            checked += 1
    assert checked == 7 * 25 + 5 * 60


def test_keras_adam_matches_fp64_restatement():
    """engine.keras_adam_update_ against a numpy fp64 restatement of Keras 2.2 Adam (Networks.py:101: lr 5e-4, betas (0.9, 0.999),
    epsilon 1e-7 outside the square root, lr_t folding both bias corrections), ten steps."""
    from spwgnn_b200.engine import keras_adam_update_
    rng = np.random.default_rng(0)
    p0 = rng.standard_normal(5000)
    gs = [rng.standard_normal(5000) * 10.0 ** rng.integers(-4, 1) for _ in range(10)]
    p = torch.as_tensor(p0, dtype=torch.float32).clone()
    st = dict(t=0, m=torch.zeros(5000), v=torch.zeros(5000))
    p64, m, v = p0.astype(np.float32).astype(np.float64), np.zeros(5000), np.zeros(5000)
    lr, b1, b2, eps = 5e-4, 0.9, 0.999, 1e-7
    for t, g in enumerate(gs, 1):
        g32 = g.astype(np.float32)
        keras_adam_update_(p, torch.as_tensor(g32), st, lr, b1, b2, eps)
        g64 = g32.astype(np.float64)
        lr_t = lr * np.sqrt(1 - b2 ** t) / (1 - b1 ** t)
        m = b1 * m + (1 - b1) * g64
        v = b2 * v + (1 - b2) * g64 * g64
        p64 = p64 - lr_t * m / (np.sqrt(v) + eps)
    assert st['t'] == 10
    assert np.abs(p.numpy() - p64).max() < 2e-6
    # the first step moves every weight by lr * g / (|g| + eps sqrt(1 - b2)-ish): close to lr, the Keras signature
    p1 = torch.zeros(3)
    keras_adam_update_(p1, torch.tensor([1.0, -2.0, 1e-3]), dict(t=0, m=torch.zeros(3), v=torch.zeros(3)))
    assert np.allclose(p1.numpy(), [-5e-4, 5e-4, -5e-4], rtol=1e-2)


def test_fit_holds_out_the_last_fraction_like_keras(monkeypatch):
    """Keras: split_at = int(len(x) * (1 - validation_split)); samples [split_at:] are held out BEFORE shuffling (main.py:92-98
    relies on it).  B = 999, split 0.2 -> 799 training samples, 200 validation samples."""
    from spwgnn_b200.Networks import PropagationNetwork, PropagationModel
    model = PropagationNetwork().getModel(4)                        # no GPU needed until something computes
    trained, validated = [], []

    class _B:
        n_nodes = 1
    monkeypatch.setattr(PropagationModel, 'engine', property(lambda self: type('E', (), {'device': 'cpu'})()))
    monkeypatch.setattr(PropagationModel, '_batch_from_dict', lambda self, x, sel=None: (_B(), list(sel))[0] if not trained.append(list(sel)) else None)
    monkeypatch.setattr(PropagationModel, 'train_on_batch', lambda self, batch, tgt: (0.5, 1.0))
    monkeypatch.setattr(PropagationModel, 'test_on_batch', lambda self, batch, tgt: (validated.append(int(tgt.numel())) or 0.25, 0.5))
    B = 999
    y = {'target': np.zeros((B, 4, 1), np.float32)}
    x = {'objects': np.zeros((B, 4, 3))}
    hist = model.fit(x, y, batch_size=32, epochs=1, validation_split=0.2, shuffle=True, verbose=0, seed=1)
    calls = trained
    train_idx = sorted(i for c in calls[:25] for i in c)
    val_idx = sorted(i for c in calls[25:] for i in c)
    assert train_idx == list(range(799)) and val_idx == list(range(799, 999))
    assert hist.history['loss'] == [0.5] and hist.history['val_loss'] == [0.25]
