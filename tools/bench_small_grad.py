"""Small-batch gradients: spw_backward_towers (one CTA per tower, one launch) against the tiled gradient path.

For every shape of tools/bench_small.py: device time (CUDA events around >= 200 back-to-back calls after every shape was warmed
up) of spw_backward_towers with and without drel, and of the tiled path it replaces (a rate-0 training spw_forward plus
spw_backward_obj, or plus spw_backward_rel), all on preallocated buffers; and the wall time of the public
PropagationModel.stability_gradients with small_batches on / off.  The GPU's name and power limit are read in the same run.

Usage: python tools/bench_small_grad.py [--out FILE.json] [--calls 200]
"""
import argparse
import ctypes
import json
import os
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch

from spwgnn_b200.Networks import PropagationNetwork
from spwgnn_b200.graph import TowerBatch, _stream_ptr
from spwgnn_b200 import synth

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from bench_small import SHAPES, gpu_info, device_us, wall_us


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None, help='write the JSON record here (default: print only)')
    ap.add_argument('--calls', type=int, default=200)
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'bench_small_grad.py measures on the GPU'
    torch.cuda.set_device(0)
    rec = {'head': gpu_info(), 'calls': args.calls, 'rows': []}
    print(json.dumps(rec['head']))
    tiled = PropagationNetwork(device='cuda:0', seed=0).getModel(0)
    small = PropagationNetwork(device='cuda:0', seed=0, small_batches=True)
    small.small_max_towers = 1 << 30                       # measure the small path at every batch size
    small.small_max_nodes = 32
    small = small.getModel(0)
    eng = tiled.engine
    api, dev = eng.api, eng.device
    wp = eng.params.c_struct()
    cases = []
    for label, nb, n, kind, rel in SHAPES:
        towers = synth.make_towers(kind, nb, 3 if kind == 'tower' else 11 + n, n=n)
        kw = dict(inference_glue=True) if rel == 'glue' else dict(inference_glue=False, fully_connected=True)
        b = TowerBatch.from_towers(towers, device=dev, **kw)
        N, E = b.n_nodes, b.n_edges
        ones = torch.ones(N, device=dev)
        logits, dobj, drel = torch.empty(N, device=dev), torch.empty(N, 3, device=dev), torch.empty(max(E, 1), device=dev)
        sb = api.dll.spw_backward_towers_bytes(N, E)
        ws_s = torch.empty(sb, dtype=torch.uint8, device=dev)
        tb = api.dll.spw_workspace_bytes(N, E, 1)
        ws_t = torch.empty(tb, dtype=torch.uint8, device=dev)
        st = _stream_ptr(dev)

        def towers_call(want_drel, b=b, ones=ones, logits=logits, dobj=dobj, drel=drel, ws=ws_s, nbytes=sb):
            api.check(api.dll.spw_backward_towers(ctypes.byref(wp), ctypes.byref(b.c_graph), int(b.max_nodes), b.obj.data_ptr(), None,
                                                  ones.data_ptr(), logits.data_ptr(), dobj.data_ptr(),
                                                  drel.data_ptr() if want_drel and b.n_edges else None, ws.data_ptr(), nbytes, st))

        def tiled_call(want_drel, b=b, ones=ones, logits=logits, dobj=dobj, drel=drel, ws=ws_t, nbytes=tb):
            api.check(api.dll.spw_forward(ctypes.byref(wp), ctypes.byref(b.c_graph), b.obj.data_ptr(), logits.data_ptr(), None,
                                          ws.data_ptr(), nbytes, 1, 0.0, 0, st))
            if want_drel:
                api.check(api.dll.spw_backward_rel(ctypes.byref(wp), ctypes.byref(b.c_graph), b.obj.data_ptr(), ones.data_ptr(),
                                                   ws.data_ptr(), nbytes, 0.0, drel.data_ptr() if b.n_edges else None,
                                                   dobj.data_ptr(), st))
            else:
                api.check(api.dll.spw_backward_obj(ctypes.byref(wp), ctypes.byref(b.c_graph), b.obj.data_ptr(), ones.data_ptr(),
                                                   ws.data_ptr(), nbytes, 0.0, dobj.data_ptr(), st))
        cases.append((label, nb, n, towers, kw, b, towers_call, tiled_call))
    for c in cases:                                                     # warm every shape first
        c[6](True); c[6](False); c[7](True); c[7](False)
        tiled.stability_gradients(c[3], **c[4]); small.stability_gradients(c[3], **c[4])
    torch.cuda.synchronize()
    for label, nb, n, towers, kw, b, towers_call, tiled_call in cases:
        calls = args.calls
        row = {'shape': label, 'towers': nb, 'blocks': n, 'relations': b.n_edges,
               'towers_obj_us': device_us(lambda: towers_call(False), calls),
               'towers_rel_us': device_us(lambda: towers_call(True), calls),
               'tiled_obj_us': device_us(lambda: tiled_call(False), calls),
               'tiled_rel_us': device_us(lambda: tiled_call(True), calls),
               'stability_gradients_small_wall_us': wall_us(lambda: small.stability_gradients(towers, **kw), max(calls // 4, 20)),
               'stability_gradients_tiled_wall_us': wall_us(lambda: tiled.stability_gradients(towers, **kw), max(calls // 4, 20))}
        rec['rows'].append(row)
        print(json.dumps(row))
    if args.out:
        with open(args.out, 'w') as f:
            json.dump(rec, f, indent=1)
            f.write('\n')


if __name__ == '__main__':
    main()
