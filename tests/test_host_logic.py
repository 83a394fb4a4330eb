"""CPU tests: the C ABI library loads and exports what include/spwgnn.h declares (no compute
calls without a GPU), host-side argument checks, synthetic generators, sharding, and the
world_size-2 gloo path of the gradient all-reduce."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope='module')
def built_lib():
    from spwgnn_b200 import build
    return build.build()


def test_library_exports_every_declared_symbol(built_lib):
    from spwgnn_b200._capi import CApi, EXPORTS
    header = open(os.path.join(ROOT, 'include', 'spwgnn.h')).read()
    declared = set(re.findall(r'\b(spw_[a-z0-9_]+)\s*\(', header))
    assert declared == set(EXPORTS), declared ^ set(EXPORTS)
    api = CApi(built_lib)
    for name in declared:
        assert getattr(api.dll, name) is not None
    assert api.dll.spw_version() == 1
    assert api.dll.spw_workspace_bytes(10, 90, 1) > api.dll.spw_workspace_bytes(10, 90, 0) > 0


def test_library_is_sm100a_only(built_lib):
    out = subprocess.run(['cuobjdump', '-lelf', built_lib], capture_output=True, text=True).stdout
    assert 'sm_100a' in out and 'sm_90' not in out and 'sm_80' not in out


def _workspace_array_floats(L, n, E):
    """Floats of every named workspace array, restated from the shapes (column-slab arrays: [quads][rows][4])."""
    q100, q150, q200 = 26 * n * 4, 38 * n * 4, 50 * n * 4
    earr = 38 * E * 4 + 64
    chunks = (E + 31) // 32 + 1
    bits = L['bits_floats']
    size = {'W2hi': 24320, 'W2lo': 24320, 'W2Thi': 24320, 'W2Tlo': 24320, 'ENCT': 8 * 24320, 'degf': n,
            'Q1': q100, 'Q': q100, 'QV': q100, 'GP': q200 * L['slotsGP'], 'U': q100 * L['slots'],
            'S': q150 * L['slots'], 'R': q150 * L['slots'], 'H2S': q150 * L['slots'], 'PF': chunks * 160, 'PL': chunks * 160,
            'X0': earr, 'X1': earr, 'X2': earr, 'C': earr, 'A': earr, 'H1': 5 * earr, 'EB': 4 * bits, 'M1': 5 * bits, 'M2': 5 * bits,
            'dU': 5 * q100, 'dG': 5 * q100, 'T': 4 * q100, 'dS': 4 * q150, 'dR': 4 * q150, 'dH2S': q150, 'DP': q100, 'dQ': q100,
            'dQ1': q100, 'dA': earr, 'DH1': earr, 'GB': earr, 'partE': 160 * 2 * 160 * 128,
            'part0': 3 * L['part0_stride_floats'], 'partN': 11 * L['part_stride_floats']}
    return size


@pytest.mark.parametrize('n,E', [(1, 0), (2, 2), (4, 6), (129, 257), (1000, 0), (1000, 8705), (40960, 368640)])
def test_workspace_layout_hook(built_lib, n, E):
    """spw_workspace_layout: every array in bounds of spw_workspace_bytes and 16-byte aligned (the TMA tensor maps need it),
    the training arrays pairwise disjoint, the inference aliases exactly the intended ones, agreement with
    spw_saved_state_layout.  E = 0 and E = 1 (mod 128) are the edge cases of the sign-bit rows."""
    import ctypes
    from spwgnn_b200._capi import CApi
    api = CApi(built_lib)
    names = api.dll.spw_workspace_layout_names().decode().split(',')
    assert len(names) == len(set(names))
    short = (ctypes.c_int64 * 4)()
    assert api.dll.spw_workspace_layout(n, E, 1, short, 4) == -1
    assert api.dll.spw_workspace_layout(-1, E, 1, short, 4) == -1
    for training in (1, 0):
        L = api.workspace_layout(n, E, training)
        total = L['total_bytes']
        assert total == api.dll.spw_workspace_bytes(n, E, training)
        assert L['slots'] == (5 if training else 1) and L['slotsGP'] == (5 if training else 2)
        assert L['bits_rows'] == (E + 127) // 128 * 128 + 128 and L['bits_floats'] == (20 * L['bits_rows'] + 3) // 4
        assert L['edge_stride_floats'] == 38 * E * 4 + 64
        size = _workspace_array_floats(L, n, E)
        backward = ['H1', 'EB', 'M1', 'M2', 'dU', 'dG', 'T', 'dS', 'dR', 'dH2S', 'DP', 'dQ', 'dQ1', 'dA', 'DH1', 'GB', 'partE',
                    'part0', 'partN']
        used = [k for k in size if training or k not in backward]
        if not training:
            assert all(L[k] == 0 for k in backward)
            assert L['X0'] == L['X2'] == L['A'] and L['X1'] == L['C'] and L['X0'] != L['X1']
        spans = {}
        for k in used:
            off, nbytes = L[k], 4 * size[k]
            assert off % 16 == 0, (k, off)
            assert 0 <= off and off + nbytes <= total, (k, off, nbytes, total)
            spans[k] = (off, off + nbytes)
        aliases = set() if training else {frozenset(('X0', 'X2')), frozenset(('X0', 'A')), frozenset(('X2', 'A')), frozenset(('X1', 'C'))}
        ks = sorted(spans)
        for i, a in enumerate(ks):
            for b in ks[i + 1:]:
                if frozenset((a, b)) in aliases:
                    continue
                (a0, a1), (b0, b1) = spans[a], spans[b]
                assert a1 <= b0 or b1 <= a0, ('overlap', a, spans[a], b, spans[b])
    saved = (ctypes.c_int64 * 8)()
    api.check(api.dll.spw_saved_state_layout(n, E, saved))
    L = api.workspace_layout(n, E, 1)
    assert list(saved) == [L['bits_rows'], 4 * L['bits_floats'], L['EB'], L['M1'], L['M2'], L['U'], L['Q'], L['Q1']]


def test_host_side_argument_checks(built_lib):
    """Errors that are detected before any kernel launch can be exercised without a GPU."""
    import ctypes
    from spwgnn_b200._capi import CApi, SpwError, SpwParams, SpwGraph
    api = CApi(built_lib)
    rc = api.dll.spw_edges_count(None, None, 1, 70, 70, 170.0, 0, None, None, None, None)
    assert rc == -2 and b'limit' in api.dll.spw_last_error()             # SPW_ERR_UNSUPPORTED
    with pytest.raises(SpwError):
        api.check(rc)
    assert api.dll.spw_edges_count(None, None, -1, 0, 0, 170.0, 0, None, None, None, None) == -1
    p = SpwParams()                                                       # all-null tensors
    g = SpwGraph()
    assert api.dll.spw_forward(ctypes.byref(p), ctypes.byref(g), None, None, None, None, 0, 0, 0.0, 0, None) == -1
    assert b'tensor 0' in api.dll.spw_last_error()


def test_product_fails_loudly_without_cuda():
    from spwgnn_b200 import SpwError
    from spwgnn_b200.engine import Engine
    if torch.cuda.is_available():
        pytest.skip('GPU present')
    with pytest.raises(SpwError):
        Engine('cuda')


def test_product_never_imports_the_oracle_or_emulator():
    for dirpath, _, files in os.walk(os.path.join(ROOT, 'spwgnn_b200')):
        for f in files:
            if f.endswith('.py'):
                src = open(os.path.join(dirpath, f)).read()
                assert not re.search(r'^\s*(from|import)\s+oracle', src, re.M), f
                assert 'cuemu' not in src and 'libspwgnn_emu' not in src and 'SPW_EMU' not in src, f


def test_param_buffer_layout():
    from spwgnn_b200.params import ParamBuffer, N_PARAMS, OFFSETS
    assert N_PARAMS == 209501
    assert all(o % 4 == 0 for o in OFFSETS)
    pb = ParamBuffer('cpu').glorot_init(0)
    assert pb.views['rmp.w0'].shape == (350, 150) and float(pb.views['rm.b0'].abs().max()) == 0.0
    lim = (6.0 / 500) ** 0.5
    assert float(pb.views['rmp.w0'].abs().max()) <= lim


def test_synthetic_generators_are_seeded_and_shaped():
    from spwgnn_b200 import synth
    a = synth.make_towers('jenga', 5, 3, n=10)
    b = synth.make_towers('jenga', 5, 3, n=10)
    assert all(np.array_equal(x, y) for x, y in zip(a, b))
    assert all(t.shape == (10, 3) for t in a)
    assert all(t.shape == (7, 3) for t in synth.make_towers('tower', 4, 1, n=6))
    assert all(t.shape == (54, 3) for t in synth.make_towers('jenga18', 3, 1))
    u = synth.make_towers('uniform', 50, 2, lo=6, hi=32)
    assert min(len(t) for t in u) >= 6 and max(len(t) for t in u) <= 32
    t = synth.make_towers('tower', 1, 9, n=6)[0]
    assert np.all(t[:, 2] == 150) and np.all((t[:, 1] - 110) % 80 == 0)


def test_shard_towers_balances_cost():
    from spwgnn_b200.dp import shard_towers, tower_cost, estimate_edges
    rng = np.random.default_rng(0)
    sizes = rng.integers(6, 33, size=4096)
    shards = shard_towers(sizes, 8)
    assert sorted(np.concatenate(shards).tolist()) == list(range(4096))
    cost = tower_cost(sizes, estimate_edges(sizes, False))
    loads = np.array([cost[s].sum() for s in shards])
    assert loads.max() / loads.mean() < 1.01
    assert all(np.array_equal(a, b) for a, b in zip(shards, shard_towers(sizes, 8)))
    assert all((np.diff(s) > 0).all() for s in shards)
    # real relation counts (what spw_edges_count measures) instead of the size-based estimate
    edges = rng.integers(0, 200, size=4096)
    shards = shard_towers(sizes, 8, edges=edges)
    loads = np.array([tower_cost(sizes, edges)[s].sum() for s in shards])
    assert sorted(np.concatenate(shards).tolist()) == list(range(4096)) and loads.max() / loads.mean() < 1.01


def test_shard_towers_is_cheap():
    """A 65 536-tower global batch (BASELINE config 4) is planned in a few milliseconds (round 1: 0.25 s)."""
    import time
    from spwgnn_b200.dp import shard_towers
    sizes = np.random.default_rng(1).integers(6, 33, size=65536)
    shard_towers(sizes, 8)
    t0 = time.perf_counter()
    shard_towers(sizes, 8)
    assert time.perf_counter() - t0 < 0.05


def _gloo_worker(rank, world, port, q):
    import torch.distributed as dist
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    dist.init_process_group('gloo', rank=rank, world_size=world)
    try:
        from spwgnn_b200.dp import GradientAllReduce
        from spwgnn_b200.params import FLAT_SIZE
        comm = GradientAllReduce()
        flat = torch.full((FLAT_SIZE,), float(rank + 1))
        stats = torch.tensor([1.0 * (rank + 1), 10.0], dtype=torch.float64)
        params = torch.arange(FLAT_SIZE, dtype=torch.float32) * (1 if rank == 0 else -1)
        comm.broadcast_(params, 0)
        comm.allreduce_(flat, stats)
        # the one-collective path: stats ride in the tail of the gradient buffer
        from spwgnn_b200.params import STATS_TAIL
        buf = torch.full((FLAT_SIZE + STATS_TAIL,), float(rank + 1))
        stats2 = torch.tensor([0.5 * (rank + 1), 7.0], dtype=torch.float64)
        comm.allreduce_(buf[:FLAT_SIZE], stats2, buffer=buf)
        assert float(buf[0]) == 3.0 and stats2.tolist() == [1.5, 14.0]
        q.put((rank, float(flat[0]), float(flat[-1]), stats.tolist(), float(params[5])))
    finally:
        dist.destroy_process_group()


def test_gradient_allreduce_world2_gloo():
    import torch.multiprocessing as mp
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    port = 29500 + (os.getpid() % 2000)
    procs = [ctx.Process(target=_gloo_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = sorted(q.get(timeout=120) for _ in range(2))
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    for rank, g0, g1, stats, p5 in res:
        assert g0 == 3.0 and g1 == 3.0 and stats == [3.0, 20.0] and p5 == 5.0


def test_trajectory_loader_matches_reference_main_py(golden_dir, tmp_path):
    """spwgnn_b200.data against what the reference's own main.train_gnn produced (fixtures)."""
    import json
    from spwgnn_b200 import data as D
    for name in ['train_n2', 'train_n4', 'train_n7', 'train_n9']:
        g = np.load(os.path.join(golden_dir, name + '.npz'))
        n_obj = int(g['n_objects'])
        p = tmp_path / (name + '.txt')
        p.write_text(str(g['traj_json']))
        raw0, y = D.training_arrays(str(p), n_obj + 1, jenga=True)
        assert np.array_equal(raw0 / 170.0, g['objects'])
        assert np.array_equal(y, g['target'])
        assert y.min() == 0.0 and y.max() == 1.0 or n_obj == 2
