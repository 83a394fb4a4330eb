"""bench.py -- SPWGNN propagation-network hot path on B200.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
  (N > 1: launched by torch.distributed.run, one rank per GPU, NCCL)

Headline workload (BASELINE.json configs[1], "C2"): 10-block towers, batch 4096 PER GPU (weak scaling), fully
connected relations, one TRAINING step = edge-index build from poses + forward (with the reference's
Dropout(0.1), Networks.py:77-78) + Keras-BCE seed + backward + (N>1: ONE NCCL all-reduce of the flat gradient
buffer, loss / accuracy sums in its tail) + Keras-form Adam.  Synthetic towers (spwgnn_b200.synth.g_jenga(10),
seed 1235), glorot weights.  One JSON line on stdout (rank 0).

`value`  : towers/s, whole job, inputs already resident in HBM, CUDA-event timed, max over ranks.
`e2e`    : same metric through the public API from PINNED HOST buffers: every step copies the
           poses/features/targets host->device and reads the loss/accuracy scalars back.
`roofline`: the dominant modelled kernel, timed with CUDA events on its stream (spw_profile).
`configs`: the other named BASELINE configurations, each device-timed in the same run:
           C1 (7 blocks, batch-32 fit step and batch-1 predict latency), C3 (Jenga-18 x 1024, contact relations),
           C4 (6-32 blocks, GLOBAL batch 65 536 split over the ranks by dp.shard_towers: strong scaling),
           C5 (8-64 blocks, fully connected, forward only, device-generated, sharded).
`cpu_baseline` / `--impl reference`: the reference formulation (dense one-hot graph of Networks.py, fp32, torch
           autograd) on the host cores -- the reference itself (Keras/TF1) cannot be installed here (DESIGN.md);
           kind = "port".
"""
import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

TOWERS_PER_GPU = 4096
N_BLOCKS = 10
SEED = 1235
FLOP_EDGE_FWD, FLOP_NODE_FWD = 1035600, 421400        # SURVEY.md section 8(d), reference formulation
# Kernels with a fixed per-edge FLOP model (DESIGN.md section 4).  The roofline entry is computed for whichever of
# them takes the largest share of the step.  algo = reference-formulation FLOPs of the layer the launch implements
# (per edge); exec = FLOPs the kernel issues (padding, 3xTF32 split: three tf32 MMAs per product).
_MMA = 2 * 128 * 160 * 8                               # FLOPs of one tcgen05.mma kind::tf32 M128 N160 K8
KERNEL_MODELS = {
    'k_wgrad_c:step': dict(algo=2 * 150 * 150, exec=6 * _MMA / 8.0, pipe='tensor'),       # 2 M-tiles (CTAs) x 3 MMAs per 8 edge rows
    'k_wgrad_c:enc': dict(algo=2 * 150 * 150, exec=6 * _MMA / 8.0, pipe='tensor'),
    'k_edge_dgrad_c': dict(algo=2 * 150 * 150, exec=57 * _MMA / 128.0, pipe='tensor'),      # 19 k-steps x 3 MMAs per 128 rows
    'k_edge_step_c': dict(algo=2 * 150 * 150, exec=57 * _MMA / 128.0, pipe='tensor'),
    'k_lin:enc_fwd': dict(algo=2 * 150 * 150, exec=57 * _MMA / 128.0, pipe='tensor'),       # one relation-encoder layer per launch
    'k_lin:enc_bwd': dict(algo=2 * 150 * 150, exec=57 * _MMA / 128.0, pipe='tensor'),
}
TF32_FLOP_PER_CLK_SM = 4096                            # dense tf32 tcgen05: 128 x 160 x 8 MACs in 80 cycles (measured, tools/probe)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--towers', type=int, default=TOWERS_PER_GPU, help='towers per GPU')
    ap.add_argument('--cpu-sample', type=int, default=512, help='towers in the bounded CPU sample')
    ap.add_argument('--no-configs', action='store_true', help='skip the C1 / C3 / C4 / C5 section (development runs)')
    ap.add_argument('--c4-towers', type=int, default=65536, help='GLOBAL towers of configuration 4')
    ap.add_argument('--c5-towers', type=int, default=200000, help='towers PER GPU of configuration 5')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write what the last timed training step computed (rank 0) to DIR/<name>.npy')
    return ap.parse_args()


def ncu_record():
    """What the committed ncu captures (profiles/r02_ncu.json, written by tools/summarize_ncu.py from the .ncu-rep files of the
    same workload) say per kernel tag: DRAM bytes per launch, tensor-pipe activity; and the DRAM bytes of one whole step."""
    p = os.path.join(ROOT, 'profiles', 'r02_ncu.json')
    return json.load(open(p)) if os.path.exists(p) else {}


def load_peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d.get('hbm_gbs', 6650.0), tf=d.get('bf16_tflops_sustained', d.get('bf16_tflops', 1590.0)),
                    src='measured (MEASURED_PEAKS.json, bf16 sustained)')
    return dict(hbm=6650.0, tf=1590.0, src='fallback (B200_PROFILING.md)')


# ---------------------------------------------------------------------------------------------------
# CPU arm: the reference formulation on the host cores (oracle port; checker-only module)
# ---------------------------------------------------------------------------------------------------
def cpu_reference_rate(sample_towers, steps, warmup):
    import torch
    from oracle import propnet as O
    from spwgnn_b200 import synth
    threads = os.cpu_count() or 1
    torch.set_num_threads(threads)
    towers = synth.make_towers('jenga', sample_towers, SEED, n=N_BLOCKS)
    raw = np.stack(towers)                                          # (B, 10, 3)
    rs, rr = O.build_relations_dense(raw[:, :, :2] / 170.0, 170.0)   # inference-glue positions => fully connected
    obj = torch.as_tensor((raw / 170.0).astype(np.float32))
    rs_t, rr_t = torch.as_tensor(rs.astype(np.float32)), torch.as_tensor(rr.astype(np.float32))
    tgt = torch.as_tensor((np.random.default_rng(0).random((sample_towers, N_BLOCKS, 1)) > 0.5).astype(np.float32))
    w = {k: v.float().requires_grad_(True) for k, v in O.init_weights(0).items()}
    names = O.tensor_names()

    def step():
        probs = O.forward_dense(w, obj, rs_t, rr_t)
        loss = O.bce_keras(probs, tgt)
        torch.autograd.grad(loss, [w[k] for k in names])
    for _ in range(warmup):
        step()
    t0 = time.perf_counter()
    for _ in range(steps):
        step()
    dt = (time.perf_counter() - t0) / steps
    return sample_towers / dt, dt, threads


def cpu_model_name():
    try:
        for line in open('/proc/cpuinfo'):
            if line.startswith('model name'):
                return line.split(':', 1)[1].strip()
    except OSError:
        pass
    return 'unknown'


def run_reference(args, rank):
    """The reference arm: the driver's --steps / --warmup are honoured; what is bounded is the SAMPLE -- every step is one
    training step on `--cpu-sample` towers of the same shape (the CPU rate per tower does not improve with the batch,
    BASELINE.md section 2), so K steps stay within minutes."""
    if rank != 0:
        return
    steps, warmup = max(1, args.steps), max(0, args.warmup)
    rate, dt, threads = cpu_reference_rate(args.cpu_sample, steps, warmup)
    sample = ('%d ten-block fully connected towers per step (dense one-hot formulation, fp32, torch autograd), '
              '%d warm-up + %d timed steps, %s' % (args.cpu_sample, warmup, steps, cpu_model_name()))
    line = {
        'impl': 'reference', 'metric': 'towers_per_sec', 'value': rate, 'unit': 'towers/s', 'n_gpus': args.gpus,
        'steps': steps, 'warmup': warmup, 'ms_per_step': dt * 1e3, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'edges_per_sec': rate * N_BLOCKS * (N_BLOCKS - 1),
        'config': {'workload': 'C2: 10-block towers, fully connected, forward+backward; each step is a bounded sample of %d towers '
                               '(not the GPU arm\'s 4096 per GPU): towers/s is rate-normalised' % args.cpu_sample},
        'cpu_baseline': {'value': rate, 'unit': 'towers/s', 'cores': threads, 'kind': 'port', 'sample': sample},
        'e2e': {'value': rate, 'unit': 'towers/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons every 20 ms, started BEFORE the warm-up so that it is up when the timed
    region begins; stop() keeps the samples whose timestamp falls inside the timed windows."""
    Q = ('timestamp,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index):
        self.proc, self.path = None, '/tmp/spw_clocks_%d.csv' % os.getpid()
        try:
            self.f = open(self.path, 'w')
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(gpu_index), '--query-gpu=' + self.Q, '--format=csv,noheader,nounits',
                                          '-lms', '20'], stdout=self.f, stderr=subprocess.DEVNULL)
        except OSError:
            self.proc = None

    def stop(self, windows):
        import datetime
        out = {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': []}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except subprocess.TimeoutExpired:
            self.proc.kill()
        self.f.close()
        rows = []
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        for line in open(self.path):
            p = [x.strip() for x in line.split(',')]
            if len(p) < 9:
                continue
            try:
                ts = datetime.datetime.strptime(p[0], '%Y/%m/%d %H:%M:%S.%f').timestamp()
                rows.append((ts, float(p[1]), float(p[2]), [nm for nm, v in zip(names, p[5:9]) if v.lower().startswith('active')]))
            except ValueError:
                continue
        try:
            os.remove(self.path)
        except OSError:
            pass
        inside = [r for r in rows if any(a - 0.02 <= r[0] <= b + 0.02 for a, b in windows)]
        where = 'timed regions'
        if not inside and rows:        # very short timed regions: the samples closest to them (GPU still under the same load)
            mid = sum(a + b for a, b in windows) / (2 * len(windows))
            inside = sorted(rows, key=lambda r: abs(r[0] - mid))[:5]
            where = 'nearest to the timed regions'
        if inside:
            out = {'sm_mhz': float(np.median([r[1] for r in inside])), 'sm_max_mhz': float(max(r[2] for r in inside)),
                   'reasons': sorted({nm for r in inside for nm in r[3]}), 'samples': len(inside), 'sampled': where}
        return out


def timed_events(torch, dist, world, dev, fn, steps):
    """K calls of fn bracketed by barrier + synchronize; CUDA-event time, max over ranks (ms)."""
    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    out = None
    for _ in range(steps):
        out = fn()
    e1.record()
    barrier()
    ms = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms = float(t[0])
    return ms, out


def dump_outputs(path, stats, eng, n):
    """What a caller of the timed training step holds after its last call, so that two builds can be compared output for
    output on the same seeded inputs: the returned stats (float64: summed BCE loss, correct predictions), the block logits
    of the forward pass (float32, dropout applied), and every gradient and updated weight tensor (float32, after Adam)."""
    out = {'stats': stats, 'logits': eng._fwd[2][:n]}
    for k, v in eng.grads.views.items():
        out['grad.' + k] = v
    for k, v in eng.params.views.items():
        out['param.' + k] = v
    os.makedirs(path, exist_ok=True)
    for name, t in out.items():
        np.save(os.path.join(path, name + '.npy'), t.detach().cpu().numpy())


def run_configs(args, torch, dist, world, rank, dev, eng, comm):
    """The named BASELINE configurations besides the headline one; every entry is device-timed like `value`."""
    from spwgnn_b200 import synth
    from spwgnn_b200.dp import shard_towers, tower_cost, tower_edge_counts
    from spwgnn_b200.graph import TowerBatch
    from spwgnn_b200.Networks import PropagationNetwork
    out = {}

    def algo_tflops(E, n, ms, train=True):
        return (3.0 if train else 1.0) * (E * FLOP_EDGE_FWD + n * FLOP_NODE_FWD) / (ms * 1e-3) / 1e12

    def allsum(x):
        if world == 1:
            return x
        t = torch.tensor([float(x)], dtype=torch.float64, device=dev)
        dist.all_reduce(t)
        return float(t[0])

    # ---- C1: 7 blocks (6 stacked + the dropped one, main.py:27), contact relations: batch-32 fit step, batch-1 predict ----
    if rank == 0:
        towers = synth.make_towers('tower', 1000, SEED + 1, n=6)
        labels = [(np.random.default_rng(i).random(7) > 0.5).astype(np.float32) for i in range(len(towers))]
        net = PropagationNetwork(device=dev, seed=0)
        model = net.getModel(7)
        b32 = TowerBatch.from_towers(towers[:32], device=dev)
        t32 = torch.as_tensor(np.concatenate(labels[:32])).to(dev)
        for _ in range(5):
            model.train_on_batch(b32, t32)
        ms_fit, _ = timed_events(torch, None, 1, dev, lambda: model.train_on_batch(b32, t32), 20)
        one = [towers[0]]
        for _ in range(5):
            model.predict_towers(one)
        ms_pred, _ = timed_events(torch, None, 1, dev, lambda: model.predict_towers(one), 50)
        gmax, model.engine.graph_max_edges = model.engine.graph_max_edges, 0      # the same call as ~60 direct launches
        for _ in range(5):
            model.predict_towers(one)
        ms_pred_direct, _ = timed_events(torch, None, 1, dev, lambda: model.predict_towers(one), 50)
        model.engine.graph_max_edges = gmax
        t0 = time.perf_counter()
        model.fit_towers(towers, labels, batch_size=32, epochs=1, validation_split=0.2, shuffle=True, verbose=0, seed=0)
        torch.cuda.synchronize()
        epoch_s = time.perf_counter() - t0
        out['C1'] = {'workload': '7-block towers (TowerCreator layout), contact relations: fit step on a batch of 32 (edge build + fwd + bwd + Adam, '
                                 'host-synchronous like Keras), batch-1 predict through the public API (forward replayed from a CUDA graph per shape), one epoch of fit(batch 32, split 0.2) on 1000 samples',
                     'fit_step_ms': ms_fit / 20, 'fit_towers_per_sec': 32 * 20 / (ms_fit * 1e-3), 'predict_batch1_us': ms_pred / 50 * 1e3,
                     'predict_batch1_us_without_cuda_graph': ms_pred_direct / 50 * 1e3,
                     'epoch_1000_samples_s': epoch_s, 'edges_in_batch32': b32.n_edges}
    else:
        out['C1'] = None

    # ---- C3: Jenga-18 (54 blocks) x 1024 per GPU, contact relations, training step ----
    towers = synth.make_towers('jenga18', 1024, SEED + 3 + 101 * rank)
    raw, node_off = synth.pack_towers(towers)
    obj_d = torch.as_tensor((raw / 170.0).astype(np.float32)).to(dev)
    pos_d = torch.as_tensor(np.ascontiguousarray(raw[:, :2])).to(dev)
    tgt_d = torch.as_tensor((np.random.default_rng(3).random(len(raw)) > 0.5).astype(np.float32)).to(dev)
    gnodes = len(raw) * world
    state = {}

    def step_c3():
        b = TowerBatch.from_poses(obj_d, node_off, pos_d, device=dev, max_nodes=54)
        state['E'] = b.n_edges
        st = eng.loss_and_grads(b, tgt_d, count=gnodes, dropout_rate=0.1, dropout_seed=17)
        comm.allreduce_(eng.grads.flat, st, buffer=eng.grads_buffer)
        eng.adam_step()
    for _ in range(3):
        step_c3()
    ms, _ = timed_events(torch, dist, world, dev, step_c3, 10)
    E_all = allsum(state['E'])
    out['C3'] = {'workload': 'Jenga-18 (54 blocks) x 1024 towers per GPU, contact relations (threshold 170 px on raw positions), training step; weak scaling',
                 'towers_per_sec': 1024 * world * 10 / (ms * 1e-3), 'edges_per_sec': E_all * 10 / (ms * 1e-3), 'ms_per_step': ms / 10,
                 'edges': int(E_all), 'mean_edges_per_tower': E_all / (1024.0 * world),
                 'algorithmic_tflops': algo_tflops(E_all, gnodes, ms / 10)}

    # ---- C4: 6-32 blocks, GLOBAL batch split over the ranks by dp.shard_towers on the measured relation counts (strong scaling) ----
    T4 = args.c4_towers
    full = TowerBatch.sample_jenga(T4, 6, 32, SEED + 4, device=dev, want_raw=True)          # every rank draws the same towers (counter-based)
    sizes = np.diff(full.node_off_host)
    t0 = time.perf_counter()
    edges4 = tower_edge_counts(full)
    shards = shard_towers(sizes, world, edges=edges4)
    plan_ms = (time.perf_counter() - t0) * 1e3
    cost = tower_cost(sizes, edges4)
    loads = np.array([cost[sh].sum() for sh in shards])
    mine = shards[rank]
    node_sel = np.concatenate([np.arange(full.node_off_host[t], full.node_off_host[t + 1]) for t in mine]) if len(mine) else np.zeros(0, np.int64)
    sel_d = torch.as_tensor(node_sel).to(dev)
    raw4 = full.raw[sel_d]
    obj4 = (raw4 / 170.0).float().contiguous()
    pos4 = raw4[:, :2].contiguous()
    off4 = np.concatenate([[0], np.cumsum(sizes[mine])]).astype(np.int64)
    tgt4 = (torch.rand(len(node_sel), device=dev) > 0.5).float()
    gnodes4 = int(sizes.sum())
    del full

    def step_c4():
        b = TowerBatch.from_poses(obj4, off4, pos4, device=dev, max_nodes=32)
        state['E4'] = b.n_edges
        st = eng.loss_and_grads(b, tgt4, count=gnodes4, dropout_rate=0.1, dropout_seed=23)
        comm.allreduce_(eng.grads.flat, st, buffer=eng.grads_buffer)
        eng.adam_step()
    for _ in range(2):
        step_c4()
    ms, _ = timed_events(torch, dist, world, dev, step_c4, 5)
    out['C4'] = {'workload': '%d towers of 6-32 blocks (GLOBAL batch), contact relations, split over %d rank(s) by dp.shard_towers on the relation counts '
                             'spw_edges_count measured; training step + one all-reduce; strong scaling' % (T4, world),
                 'towers_per_sec': T4 * 5 / (ms * 1e-3), 'edges_per_sec': float(edges4.sum()) * 5 / (ms * 1e-3), 'ms_per_step': ms / 5,
                 'edges': int(edges4.sum()), 'blocks': gnodes4, 'load_imbalance_max_over_mean': float(loads.max() / loads.mean()),
                 'shard_plan_host_ms': plan_ms, 'algorithmic_tflops': algo_tflops(float(edges4.sum()), gnodes4, ms / 5), 'scaling': 'strong'}
    del obj4, pos4, tgt4, raw4

    # ---- C5: inference sweep, 8-64 blocks, fully connected (the reference's predict glue, SURVEY F5), generated on the device ----
    T5, chunk = args.c5_towers, 10000
    nchunks = (T5 + chunk - 1) // chunk
    counts = {'n': 0, 'E': 0}

    def sweep():
        counts['n'] = counts['E'] = 0
        acc = torch.zeros((), dtype=torch.float64, device=dev)
        for i in range(nchunks):
            b = TowerBatch.sample_jenga(min(chunk, T5 - i * chunk), 8, 64, SEED + 5 + 7919 * rank + i, device=dev, fully_connected=True,
                                        inference_glue=True)
            _, probs = eng.forward(b, training=False)
            acc += probs.double().sum()
            counts['n'] += b.n_nodes
            counts['E'] += b.n_edges
        return acc
    b = TowerBatch.sample_jenga(chunk, 8, 64, SEED + 5, device=dev, fully_connected=True, inference_glue=True)
    eng.forward(b, training=False)
    del b
    ms, acc = timed_events(torch, dist, world, dev, sweep, 1)
    E5, n5 = allsum(counts['E']), allsum(counts['n'])
    out['C5'] = {'workload': 'inference over %d device-generated towers of 8-64 blocks per GPU, FULLY CONNECTED relations, chunks of %d towers; '
                             'sampling + edge build + forward; weak scaling' % (T5, chunk),
                 'towers_per_sec': T5 * world / (ms * 1e-3), 'edges_per_sec': E5 / (ms * 1e-3), 'seconds': ms * 1e-3, 'edges': int(E5),
                 'blocks': int(n5), 'mean_probability': float(acc) / max(counts['n'], 1), 'algorithmic_tflops': algo_tflops(E5, n5, ms, train=False)}
    return out


def main():
    args = parse()
    rank = int(os.environ.get('RANK', 0))
    world = int(os.environ.get('WORLD_SIZE', 1))
    local_rank = int(os.environ.get('LOCAL_RANK', 0))
    if args.impl == 'reference':
        run_reference(args, rank)
        return

    import ctypes
    import torch
    import torch.distributed as dist
    from spwgnn_b200 import synth
    from spwgnn_b200._lib import lib
    from spwgnn_b200.engine import Engine
    from spwgnn_b200.graph import TowerBatch
    from spwgnn_b200.dp import GradientAllReduce

    assert torch.cuda.is_available(), 'bench.py needs a CUDA device; there is no CPU fallback'
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        dist.init_process_group('nccl', device_id=dev)
    api = lib()
    T = args.towers
    K, W = args.steps, max(args.warmup, 3)

    # ---- synthetic inputs: this rank's shard of the global batch (weak scaling: T towers per GPU)
    towers = synth.make_towers('jenga', T, SEED + 7919 * rank, n=N_BLOCKS)
    raw, node_off = synth.pack_towers(towers)
    n = int(node_off[-1])
    E = int(sum(len(t) * (len(t) - 1) for t in towers))
    obj_h = torch.as_tensor((raw / 170.0).astype(np.float32)).pin_memory()
    pos_h = torch.as_tensor(np.ascontiguousarray(raw[:, :2] / 170.0)).pin_memory()    # inference-glue positions (F5)
    tgt_h = torch.as_tensor((np.random.default_rng(rank).random(n) > 0.5).astype(np.float32)).pin_memory()
    off_h = torch.as_tensor(node_off.astype(np.int32)).pin_memory()
    global_nodes = n * world

    eng = Engine(dev, seed=0)
    comm = GradientAllReduce()
    comm.broadcast_(eng.params.flat, 0)
    obj_d, pos_d, tgt_d = obj_h.to(dev), pos_h.to(dev), tgt_h.to(dev)
    DROPOUT = 0.1                                     # Dropout(0.1) on both encodings while training (Networks.py:77-78)
    step_no = [0]

    def seed():
        step_no[0] += 1
        return (0x5EED0001 + 0x9E3779B97F4A7C15 * (step_no[0] * 64 + rank + 1)) & 0xFFFFFFFFFFFFFFFF

    def step_resident():
        batch = TowerBatch.from_poses(obj_d, node_off, pos_d, fully_connected=True, device=dev, max_nodes=N_BLOCKS)
        stats = eng.loss_and_grads(batch, tgt_d, count=global_nodes, dropout_rate=DROPOUT, dropout_seed=seed())
        comm.allreduce_(eng.grads.flat, stats, buffer=eng.grads_buffer)
        eng.adam_step()
        return stats

    def step_e2e():
        o = obj_h.to(dev, non_blocking=True); p = pos_h.to(dev, non_blocking=True); t = tgt_h.to(dev, non_blocking=True)
        batch = TowerBatch.from_poses(o, node_off, p, fully_connected=True, device=dev, max_nodes=N_BLOCKS)
        stats = eng.loss_and_grads(batch, t, count=global_nodes, dropout_rate=DROPOUT, dropout_seed=seed())
        comm.allreduce_(eng.grads.flat, stats, buffer=eng.grads_buffer)
        eng.adam_step()
        return stats.cpu()                      # device -> host read of the step's loss / accuracy

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    sampler = ClockSampler(local_rank) if rank == 0 else None
    for _ in range(W):
        step_resident()
    l0 = api.dll.spw_launch_count()
    tw0 = time.time()
    ms, stats_resident = timed_events(torch, dist, world, dev, step_resident, K)
    tw1 = time.time()
    launches = api.dll.spw_launch_count() - l0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, stats_resident, eng, n)

    for _ in range(2):
        step_e2e()
    tw2 = time.time()
    ms_e2e, last_stats = timed_events(torch, dist, world, dev, step_e2e, K)
    tw3 = time.time()
    clocks = sampler.stop([(tw0, tw1), (tw2, tw3)]) if sampler else None
    h2d = obj_h.numel() * 4 + pos_h.numel() * 8 + tgt_h.numel() * 4 + off_h.numel() * 4
    d2h = 16

    # ---- per-kernel CUDA-event timing of the same step (separate pass: keeps `value` free of event overhead)
    api.dll.spw_profile(1)
    prof_steps = min(K, 5)
    barrier()
    for _ in range(prof_steps):
        step_resident()
    barrier()
    api.dll.spw_profile(0)
    buf = ctypes.create_string_buffer(1 << 16)
    api.dll.spw_profile_report(buf, len(buf))
    kern = {}
    for line in buf.value.decode().splitlines():
        nm, cnt, tot = line.rsplit(' ', 2)
        kern[nm] = (int(cnt), float(tot))
    total_kernel_ms = sum(v[1] for v in kern.values()) or 1.0

    # ---- FP32 pipe peak (the honest denominator for FFMA kernels), measured on this GPU
    grid, iters = 148 * 8, 1 << 15
    outbuf = torch.empty(grid * 256, device=dev)
    st = torch.cuda.current_stream(dev).cuda_stream
    for _ in range(2):
        api.dll.spw_ffma_peak(outbuf.data_ptr(), grid, iters, st)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize(); e0.record()
    api.dll.spw_ffma_peak(outbuf.data_ptr(), grid, iters, st)
    e1.record(); torch.cuda.synchronize()
    fp32_peak_tf = 2.0 * 16 * iters * grid * 256 / (e0.elapsed_time(e1) * 1e-3) / 1e12

    configs = None if args.no_configs else run_configs(args, torch, dist, world, rank, dev, eng, comm)

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks = load_peaks()
    ncu = ncu_record()
    modelled = [(v[1], k) for k, v in kern.items() if k in KERNEL_MODELS]
    K_DOM = max(modelled)[1] if modelled else 'k_wgrad_c:step'
    model = KERNEL_MODELS[K_DOM]
    towers_per_s = T * world * K / (ms * 1e-3)
    e2e_per_s = T * world * K / (ms_e2e * 1e-3)
    dom_cnt, dom_ms = kern.get(K_DOM, (0, 0.0))
    dom_avg_s = (dom_ms / dom_cnt) * 1e-3 if dom_cnt else float('nan')
    achieved_tf = E * model['algo'] / dom_avg_s / 1e12 if dom_cnt else None
    exec_tf = E * model['exec'] / dom_avg_s / 1e12 if dom_cnt else None
    sm_mhz = (clocks or {}).get('sm_mhz') or 1965.0
    tf32_pipe_peak = TF32_FLOP_PER_CLK_SM * 148 * sm_mhz * 1e6 / 1e12          # dense tf32 tensor pipe at the sampled SM clock
    step_algo_flop = 3.0 * (E * FLOP_EDGE_FWD + n * FLOP_NODE_FWD)
    cpu_rate, cpu_dt, cpu_threads = cpu_reference_rate(args.cpu_sample, 3, 1) if world == 1 else (None, None, None)
    dom_ncu = (ncu.get('kernels') or {}).get(K_DOM) or {}

    line = {
        'metric': 'towers_per_sec', 'value': towers_per_s, 'unit': 'towers/s', 'n_gpus': world, 'steps': K, 'warmup': W,
        'ms_per_step': ms / K, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
        'data': 'synthetic',
        'edges_per_sec': towers_per_s * N_BLOCKS * (N_BLOCKS - 1),
        'config': {
            'workload': 'C2: 10-block towers, batch %d per GPU, fully connected (90 edges/tower), training step = '
                        'edge build + forward (dropout 0.1 as in Networks.py:77-78) + BCE + backward%s + Adam'
                        % (T, ' + one NCCL all-reduce (gradients + loss sums)' if world > 1 else ''),
            'towers_per_gpu': T, 'blocks_per_tower': N_BLOCKS, 'edges_per_gpu': E, 'parallelism': 'dp%d' % world, 'dropout': DROPOUT,
            'l2': 'no flush: per-step working set (per-edge activations, 16 arrays x %.0f MB, + node state) exceeds the 126 MB L2'
                  % (E * 152 * 4 / 1e6),
        },
        'clocks': clocks,
        'e2e': {'value': e2e_per_s, 'unit': 'towers/s', 'h2d_bytes_per_step': int(h2d), 'd2h_bytes_per_step': d2h,
                'ms_per_step': ms_e2e / K, 'loss': float(last_stats[0]) / global_nodes},
        'gpu_launches': int(launches),
        'roofline': {
            'bound': 'tensor', 'kernel': K_DOM, 'achieved': achieved_tf, 'peak': peaks['tf'], 'unit': 'TFLOP/s',
            'frac': (achieved_tf / peaks['tf']) if achieved_tf else None,
            'traffic': dom_ncu.get('dram_bytes_per_launch'), 'traffic_source': ncu.get('source') if dom_ncu else None,
            'peak_source': peaks['src'],
            'note': 'dominant = the kernel with a fixed FLOP model that takes the largest share of the step; achieved = algorithmic '
                    '(reference-formulation, fp32) FLOPs of the layer / launch time (CUDA events) against the measured bf16 tensor peak.  '
                    'The kernels run fp32-accurate 3xTF32 (three tf32 MMAs per product) on padded tiles: executed_tflops counts what is '
                    'issued, against the dense tf32 pipe at the sampled SM clock (4096 FLOP/clk/SM); tensor_pipe_active_ncu is the hardware '
                    'counter sm__pipe_tensor_cycles_active of the committed ncu capture of the same kernel.',
            'pipe': model['pipe'],
            'executed_tflops': exec_tf, 'tf32_pipe_peak_at_clock': tf32_pipe_peak,
            'executed_frac_of_pipe': (exec_tf / tf32_pipe_peak) if exec_tf else None,
            'tensor_pipe_active_ncu': dom_ncu.get('tensor_active_pct'),
            'launch_ms': dom_avg_s * 1e3 if dom_cnt else None, 'launches_timed': dom_cnt,
            'share_of_kernel_time': dom_ms / total_kernel_ms,
            'fp32_pipe': {'peak_tflops_measured': fp32_peak_tf},
            'step_algorithmic_tflops': step_algo_flop / (ms / K * 1e-3) / 1e12,
            'step_algorithmic_bytes': 4044.0 * n, 'step_dram_bytes': ncu.get('step_dram_bytes'),
            'hbm_algorithmic_gbs': (4044.0 * n) / (ms / K * 1e-3) / 1e9,
            'kernels': {k: {'launches': v[0], 'ms': v[1], 'share': v[1] / total_kernel_ms,
                            'tensor_active_pct_ncu': ((ncu.get('kernels') or {}).get(k) or {}).get('tensor_active_pct')}
                        for k, v in sorted(kern.items())},
        },
        'cpu_baseline': None if cpu_rate is None else {
            'value': cpu_rate, 'unit': 'towers/s', 'cores': cpu_threads, 'kind': 'port',
            'sample': '%d ten-block fully connected towers per step, dense one-hot reference formulation (fp32, torch '
                      'autograd), 1 warm-up + 3 timed steps, %s' % (args.cpu_sample, cpu_model_name())},
        'configs': configs,
    }
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == '__main__':
    main()
