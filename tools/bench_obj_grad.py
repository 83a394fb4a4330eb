"""Gradient with respect to the block features: device time of spw_backward_obj against spw_backward (the same data gradients
plus the 22 weight gradients) and the training forward both start from, and the public-call time of stability_gradients.

Shapes: C2 (4096 fully connected 10-block towers), C3 (1024 Jenga-18 towers, contact relations), C1 (7-block TowerCreator
towers through the predict glue) at 1 and 32 towers.  Device time: CUDA events around back-to-back calls after every shape
was warmed up; each backward runs on the state of one training forward (both leave it unchanged).  Wall time: one
stability_gradients call on one C1 tower, ending in the copy of the gradient to the host.  The GPU's name and power limit are
read in the same run.

Usage: python tools/bench_obj_grad.py [--out FILE.json (default profiles/obj_grad_r06.json)] [--calls 20]
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
                                                  'obj_grad_r06.json'), help='where the JSON record goes')
    ap.add_argument('--calls', type=int, default=20)
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'bench_obj_grad.py measures on the GPU'
    torch.cuda.set_device(0)
    rec = {'head': gpu_info(), 'calls': args.calls, 'rows': []}
    print(json.dumps(rec['head']))
    model = PropagationNetwork(device='cuda:0', seed=0).getModel(0)
    eng = model.engine
    api, dev = eng.api, eng.device
    st = _stream_ptr(dev)
    for label, b in shapes():
        n = b.n_nodes
        dl = torch.randn(n, device=dev)
        dobj = torch.empty(n, 3, device=dev)
        wp = eng.params.c_struct()

        def fwd():
            eng.forward(b, training=True, want_probs=False)

        def bwd():
            eng.backward(dl)

        def bwd_obj():
            _, ws, _, _ = eng._fwd
            api.check(api.dll.spw_backward_obj(ctypes.byref(wp), ctypes.byref(b.c_graph), b.obj.data_ptr(), dl.data_ptr(),
                                               ws.data_ptr(), ws.numel(), 0.0, dobj.data_ptr(), st))
        for _ in range(3):
            fwd(); bwd(); bwd_obj()
        calls = args.calls if n > 1000 else 10 * args.calls
        row = {'shape': label, 'towers': b.n_towers, 'blocks': n, 'relations': b.n_edges,
               'device_us_forward_training': device_us(fwd, calls)}
        row['device_us_spw_backward'] = device_us(bwd, calls)
        row['device_us_spw_backward_obj'] = device_us(bwd_obj, calls)
        row['obj_over_weights'] = row['device_us_spw_backward_obj'] / row['device_us_spw_backward']
        rec['rows'].append(row)
        print('%-6s %5d towers %6d blocks %7d relations  forward %9.1f us  spw_backward %9.1f us  spw_backward_obj %9.1f us (x%.2f)'
              % (label, b.n_towers, n, b.n_edges, row['device_us_forward_training'], row['device_us_spw_backward'],
                 row['device_us_spw_backward_obj'], row['obj_over_weights']), flush=True)
    tower = synth.make_towers('tower', 1, 3, n=7)
    for _ in range(5):
        model.stability_gradients(tower)
    calls = 10 * args.calls
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(calls):
        model.stability_gradients(tower)
    rec['wall_us_stability_gradients_C1_x1'] = (time.perf_counter() - t0) / calls * 1e6
    print('stability_gradients, one C1 tower: %.1f us per call' % rec['wall_us_stability_gradients_C1_x1'])
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            json.dump(rec, f, indent=1)
            f.write('\n')
    print(json.dumps(rec))


if __name__ == '__main__':
    main()
