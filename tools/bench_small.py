"""Small-batch inference: Engine.forward_towers (one CTA per tower, one launch) against the tiled Engine.forward.

For every shape and both paths: device time (CUDA events around >= 200 back-to-back calls after every shape was warmed up;
the tiled path replays its captured CUDA graph where it would, i.e. up to Engine.graph_max_edges relations) and the wall time
of the public call (PropagationModel.predict_towers with small_batches on / off, which ends in a device synchronise when the
probabilities are copied to the host).  The GPU's name and power limit are read in the same run.

Usage: python tools/bench_small.py [--out FILE.json] [--calls 200]
"""
import argparse
import json
import os
import subprocess
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from spwgnn_b200.Networks import PropagationNetwork
from spwgnn_b200.graph import TowerBatch
from spwgnn_b200 import synth

# (label, towers, blocks per tower, layout, relations): C1 = latency_probe.py's TowerCreator towers through the predict glue
SHAPES = ([('C1', nb, 7, 'tower', 'glue') for nb in (1, 32)]
          + [('fc10', nb, 10, 'jenga', 'fc') for nb in (1, 32, 128, 512, 2048)]
          + [('fc%d' % n, 1, n, 'jenga', 'fc') for n in (16, 24, 32)])


def gpu_info():
    try:
        out = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                             capture_output=True, text=True, timeout=30).stdout.strip().splitlines()[0]
        name, power, clock = [s.strip() for s in out.split(',')]
        return {'gpu': name, 'power_limit': power, 'max_sm_clock': clock}
    except Exception as e:      # the device name from torch is still recorded
        return {'gpu': torch.cuda.get_device_name(0), 'power_limit': 'unknown (%s)' % type(e).__name__}


def device_us(f, calls):
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    a.record()
    for _ in range(calls):
        f()
    b.record()
    torch.cuda.synchronize()
    return a.elapsed_time(b) / calls * 1e3


def wall_us(f, calls):
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(calls):
        f()
    torch.cuda.synchronize()
    return (time.perf_counter() - t0) / calls * 1e6


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=None, help='write the JSON record here (default: print only)')
    ap.add_argument('--calls', type=int, default=200)
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'bench_small.py measures on the GPU'
    torch.cuda.set_device(0)
    rec = {'head': gpu_info(), 'calls': args.calls, 'rows': []}
    print(json.dumps(rec['head']))
    tiled = PropagationNetwork(device='cuda:0', seed=0).getModel(0)
    small = PropagationNetwork(device='cuda:0', seed=0, small_batches=True)
    small.small_max_towers = 1 << 30                       # measure the small path at every batch size
    small = small.getModel(0)
    eng_t, eng_s = tiled.engine, small.engine
    cases = []
    for label, nb, n, kind, rel in SHAPES:
        towers = synth.make_towers(kind, nb, 3 if kind == 'tower' else 11 + n, n=n)
        kw = dict(inference_glue=True) if rel == 'glue' else dict(inference_glue=False, fully_connected=True)
        bt = TowerBatch.from_towers(towers, device=eng_t.device, **kw)
        bs = TowerBatch.from_towers(towers, device=eng_s.device, **kw)
        cases.append((label, nb, n, towers, kw, bt, bs))
    for _, _, _, towers, kw, bt, bs in cases:              # warm every shape: graph capture, function attributes
        for _ in range(3):
            eng_t.forward(bt)
            eng_s.forward_towers(bs)
            tiled.predict_towers(towers, **kw)
            small.predict_towers(towers, **kw)
    torch.cuda.synchronize()
    for label, nb, n, towers, kw, bt, bs in cases:
        wall_calls = max(20, min(args.calls, 20000 // nb))
        row = {'shape': label, 'towers': nb, 'blocks': n, 'relations': bt.n_edges,
               'tiled_graph_replay': bool(0 < bt.n_edges <= eng_t.graph_max_edges),
               'device_us_tiled': device_us(lambda: eng_t.forward(bt), args.calls),
               'device_us_small': device_us(lambda: eng_s.forward_towers(bs), args.calls),
               'wall_us_tiled': wall_us(lambda: tiled.predict_towers(towers, **kw), wall_calls),
               'wall_us_small': wall_us(lambda: small.predict_towers(towers, **kw), wall_calls),
               'wall_calls': wall_calls}
        row['device_speedup'] = row['device_us_tiled'] / row['device_us_small']
        row['wall_speedup'] = row['wall_us_tiled'] / row['wall_us_small']
        rec['rows'].append(row)
        print('%-5s %5d towers %3d blocks %7d relations  device tiled %9.1f us  small %9.1f us (x%.2f)   '
              'wall tiled %9.1f us  small %9.1f us (x%.2f)'
              % (label, nb, n, bt.n_edges, row['device_us_tiled'], row['device_us_small'], row['device_speedup'],
                 row['wall_us_tiled'], row['wall_us_small'], row['wall_speedup']), flush=True)
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            json.dump(rec, f, indent=1)
            f.write('\n')
    print(json.dumps(rec))


if __name__ == '__main__':
    main()
