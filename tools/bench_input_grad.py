"""Gradient with respect to every input of the reference's model: device time of spw_backward_inputs (dense relation tensors,
propagation and objects from one pass) against spw_backward_obj, the same data gradients without the input terms, and the
public-call time of PropagationModel.input_gradients.

Shapes: C2 (4096 fully connected 10-block towers), C3 (1024 Jenga-18 towers, contact relations), C1 (8-block TowerCreator
towers through the predict glue) at 1 and 32 towers.  Device time: CUDA events around back-to-back calls after every shape
was warmed up, each variant in a window of its own; the windows run in three rounds with their order rotated, and the median
round is kept.  Every backward runs on the state of one training forward, which both leave unchanged.

Model, from shapes only (not measured):
  * h2 recompute: per step one read of H1 and one write of H2, [E][152] fp32 each: 5 x 2 x 608 bytes per relation;
  * the per-tower contraction: sum over towers of E_t N_t 450 fmas per step, 5 steps, against the FP32 FFMA rate of
    148 SMs x 128 lanes x 2 FLOP x 1.9 GHz = 72 TFLOP/s (derived, not a data-sheet figure);
  * the compact outputs drs, drr: 2 x E x max N_t fp32; the dense (B, N, R) pair a caller of the facade receives:
    2 x sum over towers of N_t^2 (N_t - 1) fp32.
The GPU's name and power limit are read in the same run.

Usage: python tools/bench_input_grad.py [--out FILE.json (default profiles/input_grad_r08.json)] [--calls 20]
"""
import argparse
import ctypes
import json
import os
import sys
import time

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np
import torch

from spwgnn_b200.Networks import PropagationNetwork
from spwgnn_b200.graph import TowerBatch, _stream_ptr
from spwgnn_b200 import synth

sys.path.insert(0, os.path.dirname(os.path.abspath(__file__)))
from bench_small import gpu_info, device_us      # noqa: E402

FFMA_FLOPS = 148 * 128 * 2 * 1.9e9
HBM_BPS = 7.7e12


def shapes():
    yield 'C2', TowerBatch.from_towers(synth.make_towers('jenga', 4096, 1235, n=10), fully_connected=True)
    yield 'C3', TowerBatch.from_towers(synth.make_towers('jenga18', 1024, 31))
    for nb in (1, 32):
        yield 'C1 x%d' % nb, TowerBatch.from_towers(synth.make_towers('tower', nb, 3, n=7), inference_glue=True)


def model(b):
    off = b.node_off_host
    Nt = np.diff(off)
    in_off = b.in_off[:b.n_nodes + 1].cpu().numpy().astype(np.int64) if b.n_nodes else np.zeros(1, np.int64)
    Et = in_off[off[1:]] - in_off[off[:-1]]
    fma = float((Et * Nt).sum()) * 450 * 5
    h2_bytes = 5 * 2 * 608 * b.n_edges
    return {'model_fma_contraction': fma, 'model_us_contraction_at_72TFLOPs': 2 * fma / FFMA_FLOPS * 1e6,
            'model_bytes_h2_recompute': h2_bytes, 'model_us_h2_at_7.7TBps': h2_bytes / HBM_BPS * 1e6,
            'model_bytes_compact_outputs': 2 * 4 * b.n_edges * b.max_nodes,
            'model_bytes_dense_relation_outputs': float(2 * 4 * (Nt ** 2 * np.maximum(Nt - 1, 0)).sum())}


def kernel_times(fn):
    """device time per kernel name (us, summed over launches) of one call of fn, from torch.profiler"""
    from torch.profiler import ProfilerActivity, profile
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    out = {}
    for ev in prof.key_averages():
        if ev.device_type.name == 'CUDA' or getattr(ev, 'self_device_time_total', 0) > 0:
            t = getattr(ev, 'self_device_time_total', None)
            if t is None:
                t = ev.self_cuda_time_total
            if t > 0:
                out[ev.key[:80]] = round(float(t), 1)
    return dict(sorted(out.items(), key=lambda kv: -kv[1])[:12])


def dense_dict(raw):
    """one tower's reference dict, relations as main.py:66-81 builds them on the predict glue (positions / 170 against 170)"""
    obj = np.asarray(raw, np.float64) / 170.0
    N = len(obj)
    rs, rr = np.zeros((1, N, N * (N - 1))), np.zeros((1, N, N * (N - 1)))
    c = 0
    for m in range(N):
        for j in range(N):
            if m != j:
                if np.linalg.norm(obj[m, :2] - obj[j, :2]) < 170.0:
                    rs[0, m, c] = rr[0, j, c] = 1.0
                c += 1
    return {'objects': obj[None], 'sender_relations': rs, 'receiver_relations': rr}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default=os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), 'profiles',
                                                  'input_grad_r08.json'), help='where the JSON record goes')
    ap.add_argument('--calls', type=int, default=20)
    args = ap.parse_args()
    assert torch.cuda.is_available(), 'bench_input_grad.py measures on the GPU'
    torch.cuda.set_device(0)
    rec = {'head': gpu_info(), 'calls': args.calls, 'rows': []}
    print(json.dumps(rec['head']))
    pm = PropagationNetwork(device='cuda:0', seed=0).getModel(7)
    eng = pm.engine
    api, dev = eng.api, eng.device
    st = _stream_ptr(dev)
    for label, b in shapes():
        n, E, mx = b.n_nodes, b.n_edges, b.max_nodes
        dl = torch.randn(n, device=dev)
        dobj = torch.empty(n, 3, device=dev)
        drs, drr = torch.empty(max(E * mx, 1), device=dev), torch.empty(max(E * mx, 1), device=dev)
        free, dprop = torch.empty(n, device=dev), torch.empty(n, 100, device=dev)
        sb = api.dll.spw_backward_inputs_bytes(n, E)
        scratch = torch.empty(sb, dtype=torch.uint8, device=dev)
        wp = eng.params.c_struct()
        eng.forward(b, training=True, want_probs=False)
        _, ws, _, _ = eng._fwd

        def bwd_obj():
            api.check(api.dll.spw_backward_obj(ctypes.byref(wp), ctypes.byref(b.c_graph), b.obj.data_ptr(), dl.data_ptr(),
                                               ws.data_ptr(), ws.numel(), 0.0, dobj.data_ptr(), st))

        def bwd_inputs():
            api.check(api.dll.spw_backward_inputs(ctypes.byref(wp), ctypes.byref(b.c_graph), mx, b.obj.data_ptr(), dl.data_ptr(),
                                                  ws.data_ptr(), ws.numel(), 0.0, scratch.data_ptr(), sb, drs.data_ptr(),
                                                  drr.data_ptr(), free.data_ptr(), dprop.data_ptr(), dobj.data_ptr(), st))
        fns = {'spw_backward_obj': bwd_obj, 'spw_backward_inputs': bwd_inputs}
        for _ in range(3):
            for f in fns.values():
                f()
        calls = args.calls if n > 1000 else 10 * args.calls
        samples = {k: [] for k in fns}
        for rnd in range(3):
            keys = list(fns)[rnd % 2:] + list(fns)[:rnd % 2]
            for k in keys:
                samples[k].append(device_us(fns[k], calls))
        row = {'shape': label, 'towers': b.n_towers, 'blocks': n, 'relations': E, 'max_blocks': mx}
        for k, v in samples.items():
            row['device_us_' + k] = sorted(v)[1]
            row['device_us_' + k + '_rounds'] = v
        row['extra_us_inputs_over_obj'] = row['device_us_spw_backward_inputs'] - row['device_us_spw_backward_obj']
        row.update(model(b))
        if label in ('C2', 'C3'):   # where the time goes: device time per kernel name of one call of each, in a profiled run
            row['profile_us_per_kernel'] = {k: kernel_times(f) for k, f in fns.items()}
        rec['rows'].append(row)
        print('%-6s %5d towers %6d blocks %7d relations  spw_backward_obj %9.1f us  spw_backward_inputs %9.1f us  (+%.1f us; '
              'model: contraction %.1f us at 72 TFLOP/s, h2 recompute %.1f us at 7.7 TB/s)'
              % (label, b.n_towers, n, E, row['device_us_spw_backward_obj'], row['device_us_spw_backward_inputs'],
                 row['extra_us_inputs_over_obj'], row['model_us_contraction_at_72TFLOPs'], row['model_us_h2_at_7.7TBps']), flush=True)
    tower = synth.make_towers('tower', 1, 3, n=7)[0]
    pm = PropagationNetwork(device='cuda:0', seed=0).getModel(len(tower))
    x = dense_dict(tower)
    for _ in range(5):
        pm.input_gradients(x)
    calls = 10 * args.calls
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(calls):
        pm.input_gradients(x)
    rec['wall_us_input_gradients_C1_x1'] = (time.perf_counter() - t0) / calls * 1e6
    print('input_gradients, one C1 dict: %.1f us per call' % rec['wall_us_input_gradients_C1_x1'])
    if args.out:
        os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
        with open(args.out, 'w') as f:
            json.dump(rec, f, indent=1)
            f.write('\n')
    print(json.dumps(rec))


if __name__ == '__main__':
    main()
