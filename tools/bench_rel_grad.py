"""Gradient with respect to the relation weights: device time of spw_backward_rel (drel alone, and drel with dobj from the same
pass) against spw_backward_obj, the same data gradients without the relation terms, and the public-call time of
relation_gradients.

Shapes: C2 (4096 fully connected 10-block towers), C3 (1024 Jenga-18 towers, contact relations), C1 (7-block TowerCreator
towers through the predict glue) at 1 and 32 towers.  Device time: CUDA events around back-to-back calls after every shape
was warmed up, each backward variant in a window of its own; the three windows run in three rounds with their order rotated,
and the median round is kept.  Every backward runs on the state
of one training forward, which all of them leave unchanged.  Traffic model from shapes only: the relation terms stream two
150-wide fp32 rows per relation and step (DH1, A) and one more for the encoder term (D_e), 11 x 600 bytes per relation; the
node tables they gather fit in L2.  The GPU's name and power limit are read in the same run.

Usage: python tools/bench_rel_grad.py [--out FILE.json (default profiles/rel_grad_r07.json)] [--calls 20]
"""
import argparse
import ctypes
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from spwgnn_b200.Networks import PropagationNetwork
from spwgnn_b200.graph import TowerBatch, _stream_ptr
from spwgnn_b200 import synth

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from bench_small import gpu_info, device_us      # noqa: E402


def shapes():
    yield 'C2', TowerBatch.from_towers(synth.make_towers('jenga', 4096, 1235, n=10), fully_connected=True)
    yield 'C3', TowerBatch.from_towers(synth.make_towers('jenga18', 1024, 31))
    for nb in (1, 32):
        yield 'C1 x%d' % nb, TowerBatch.from_towers(synth.make_towers('tower', nb, 3, n=7), inference_glue=True)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'profiles',
                                                  'rel_grad_r07.json'), help='where the JSON record goes')
    ap.add_argument('--calls', type=int, default=20)
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'bench_rel_grad.py measures on the GPU'
    torch.cuda.set_device(0)
    rec = {'head': gpu_info(), 'calls': args.calls, 'rows': []}
    print(json.dumps(rec['head']))
    model = PropagationNetwork(device='cuda:0', seed=0).getModel(0)
    eng = model.engine
    api, dev = eng.api, eng.device
    st = _stream_ptr(dev)
    for label, b in shapes():
        n, E = b.n_nodes, b.n_edges
        dl = torch.randn(n, device=dev)
        dobj = torch.empty(n, 3, device=dev)
        drel = torch.empty(max(E, 1), device=dev)
        wp = eng.params.c_struct()
        eng.forward(b, training=True, want_probs=False)
        _, ws, _, _ = eng._fwd
        args_ = (ctypes.byref(wp), ctypes.byref(b.c_graph), b.obj.data_ptr(), dl.data_ptr(), ws.data_ptr(), ws.numel(), 0.0)

        def bwd_obj():
            api.check(api.dll.spw_backward_obj(*args_, dobj.data_ptr(), st))

        def bwd_rel():
            api.check(api.dll.spw_backward_rel(*args_, drel.data_ptr(), None, st))

        def bwd_rel_obj():
            api.check(api.dll.spw_backward_rel(*args_, drel.data_ptr(), dobj.data_ptr(), st))
        fns = {'spw_backward_obj': bwd_obj, 'spw_backward_rel': bwd_rel, 'spw_backward_rel_with_dobj': bwd_rel_obj}
        for _ in range(3):
            for f in fns.values():
                f()
        calls = args.calls if n > 1000 else 10 * args.calls
        samples = {k: [] for k in fns}
        for rnd in range(3):
            keys = list(fns)[rnd:] + list(fns)[:rnd]
            for k in keys:
                samples[k].append(device_us(fns[k], calls))
        row = {'shape': label, 'towers': b.n_towers, 'blocks': n, 'relations': E}
        for k, v in samples.items():
            row['device_us_' + k] = sorted(v)[1]
            row['device_us_' + k + '_rounds'] = v
        row['extra_us_rel_over_obj'] = row['device_us_spw_backward_rel_with_dobj'] - row['device_us_spw_backward_obj']
        row['model_bytes_relation_terms'] = 11 * 600 * E
        row['model_us_at_7.7TBps'] = row['model_bytes_relation_terms'] / 7.7e12 * 1e6
        rec['rows'].append(row)
        print('%-6s %5d towers %6d blocks %7d relations  spw_backward_obj %9.1f us  spw_backward_rel %9.1f us  with dobj %9.1f us'
              '  (+%.1f us; traffic model %.1f us at 7.7 TB/s)'
              % (label, b.n_towers, n, E, row['device_us_spw_backward_obj'], row['device_us_spw_backward_rel'],
                 row['device_us_spw_backward_rel_with_dobj'], row['extra_us_rel_over_obj'], row['model_us_at_7.7TBps']), flush=True)
    tower = synth.make_towers('tower', 1, 3, n=7)
    for _ in range(5):
        model.relation_gradients(tower)
    calls = 10 * args.calls
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(calls):
        model.relation_gradients(tower)
    rec['wall_us_relation_gradients_C1_x1'] = (time.perf_counter() - t0) / calls * 1e6
    print('relation_gradients, one C1 tower: %.1f us per call' % rec['wall_us_relation_gradients_C1_x1'])
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            json.dump(rec, f, indent=1)
            f.write('\n')
    print(json.dumps(rec))


if __name__ == '__main__':
    main()
