"""Opt-in engine features that the default path does not use (file name sorts last on purpose: these were written
after the round's last GPU session and a failure here must not hide the default-path suites under ``-x``):
per-stage CUDA graphs (option ``stage_graphs``) and the gate backward that also leaves the row maxima of dg
(option ``gate_bwd_rows``)."""
import numpy as np
import pytest

from helpers import model_weights

pytestmark = pytest.mark.gpu


@pytest.fixture()
def engine():
    from sevenn_b200.engine import B200Engine, set_option
    meta, arrays = model_weights('sevennet_0')
    yield B200Engine(meta, arrays)
    set_option('stage_graphs', 0)
    set_option('gate_bwd_rows', 0)


def _si(reps, seed=0, sigma=0.05, a=5.431):
    from sevenn_b200.neighbors import diamond_si
    pos, cell, _ = diamond_si(*reps, a=a, sigma=sigma, seed=seed)
    return pos, cell


def _split_sequence(eng, T):
    """the runner's stage order with the interior / boundary split, exchanges left out (single GPU)"""
    from sevenn_b200 import engine as E
    eng.run_stage(E.STAGE_FWD_BEGIN)
    for t in range(T):
        if t == 0:
            eng.run_stage(E.STAGE_FWD_LAYER_A, t)
        else:
            eng.run_stage(E.STAGE_FWD_CONV_INTERIOR, t)
            eng.run_stage(E.STAGE_FWD_LAYER_A2, t)
        eng.run_stage(E.STAGE_FWD_LAYER_SC, t)
    eng.run_stage(E.STAGE_FWD_END)
    for t in range(T - 1, -1, -1):
        if t == 0:
            eng.run_stage(E.STAGE_BWD_LAYER_A, t)
            continue
        eng.run_stage(E.STAGE_BWD_LAYER_A1, t)
        eng.run_stage(E.STAGE_BWD_LAYER_A2, t)
        eng.run_stage(E.STAGE_BWD_LAYER_B1, t)
        eng.run_stage(E.STAGE_BWD_LAYER_B2, t)
    eng.run_stage(E.STAGE_BWD_END)


def test_stage_graphs_equal_direct_stage_launches(engine):
    """option stage_graphs: one captured graph per (stage, layer), replayed on the caller's stream; a changed
    graph key (set_interior) re-captures; an entry whose key never settles falls back to direct launches"""
    import torch
    from sevenn_b200.engine import set_option
    pos, cell = _si((3, 2, 2))
    sp = np.full(len(pos), engine.spec.type_map[14], dtype=np.int32)
    engine.set_positions(sp, pos, cell, True)
    T = engine.spec.n_layers
    engine.compute(); torch.cuda.synchronize()
    ref = {k: v.cpu().numpy().copy() for k, v in engine.results().items()}
    try:
        engine.set_interior(len(pos) // 3)
        set_option('stage_graphs', 0)
        _split_sequence(engine, T); torch.cuda.synchronize()
        direct = {k: v.cpu().numpy().copy() for k, v in engine.results().items()}
        assert engine.stage_graph_stats() == (0, 0)
        set_option('stage_graphs', 1)
        for _ in range(3):
            _split_sequence(engine, T)
        torch.cuda.synchronize()
        out = {k: v.cpu().numpy().copy() for k, v in engine.results().items()}
        captures, replays = engine.stage_graph_stats()
        assert captures == 5 + T + 6 * (T - 1) and replays == 3 * captures      # one per run_stage call of the sequence
        for res in (direct, out):
            assert abs(res['energy'][0] - ref['energy'][0]) < 1e-6
            assert np.allclose(res['forces'], ref['forces'], atol=2e-6)
            assert np.allclose(res['virial'], ref['virial'], atol=1e-5)
        engine.set_interior(len(pos) // 2)          # another split point: every stage re-captures once
        _split_sequence(engine, T); _split_sequence(engine, T); torch.cuda.synchronize()
        out2 = {k: v.cpu().numpy().copy() for k, v in engine.results().items()}
        assert engine.stage_graph_stats()[0] == 2 * captures
        assert np.allclose(out2['forces'], ref['forces'], atol=2e-6)
        for i in range(5):                          # the key changes on every step: capturing stops after three tries
            engine.set_interior(10 + i)
            _split_sequence(engine, T)
        torch.cuda.synchronize()
        out3 = {k: v.cpu().numpy().copy() for k, v in engine.results().items()}
        assert engine.stage_graph_stats()[0] <= 2 * captures + 3 * captures
        assert np.allclose(out3['forces'], ref['forces'], atol=2e-6)
    finally:
        set_option('stage_graphs', 0)


@pytest.mark.parametrize('model', ['sevennet_0', 'sevennet_l3i5'])
def test_gate_bwd_rows_option_matches_default(model):
    """option gate_bwd_rows: same forces as the default (separate row-exponent pass over dg) -- the row maxima
    are the same numbers, so the tensor-core slices and every result must be bit-identical up to RED.ADD order"""
    import torch
    from sevenn_b200.engine import B200Engine, set_option
    meta, arrays = model_weights(model)
    eng = B200Engine(meta, arrays)
    pos, cell = _si((2, 2, 3), seed=4)
    sp = np.full(len(pos), eng.spec.type_map[14], dtype=np.int32)
    try:
        set_option('gate_bwd_rows', 0)
        eng.set_positions(sp, pos, cell, True)
        eng.compute(); torch.cuda.synchronize()
        ref = {k: v.cpu().numpy().copy() for k, v in eng.results().items()}
        set_option('gate_bwd_rows', 1)
        eng.compute(); torch.cuda.synchronize()
        out = {k: v.cpu().numpy().copy() for k, v in eng.results().items()}
    finally:
        set_option('gate_bwd_rows', 0)
    # the option changes the backward only: every per-atom energy is bit-identical; the total is a double atomicAdd of
    # per-block partial sums (readout_kernel) in an order that varies from run to run, so it is equal up to the
    # rounding of a reordered sum of n terms
    assert np.array_equal(out['atomic_energy'], ref['atomic_energy'])
    n = len(ref['atomic_energy'])
    assert abs(out['energy'][0] - ref['energy'][0]) <= n * np.finfo(np.float64).eps * np.abs(ref['atomic_energy']).sum()
    assert np.allclose(out['forces'], ref['forces'], atol=2e-6)
    assert np.allclose(out['virial'], ref['virial'], atol=1e-5)


@pytest.mark.parametrize('model', ['sevennet_0'])
def test_host_staged_stage_protocol_two_ranks_on_one_gpu(model):
    """The protocol of examples/lammps/pair_e3gnn_b200_parallel.cpp through the same C entry points
    (s7b_engine_set_graph_host / read_rows_host / write_rows_host / read_scalars_host): two bricks of one cell,
    one engine each on the same GPU, ghost rows exchanged through host arrays between the stages.  Must reproduce
    the single-engine evaluation of the whole cell."""
    import torch
    from sevenn_b200 import engine as E
    from sevenn_b200.engine import B200Engine
    from sevenn_b200.neighbors import build_graph, diamond_si
    from sevenn_b200.parallel import brick_decompose
    from helpers import species_of
    meta, arrays = model_weights(model)
    pos, cell, z = diamond_si(4, 2, 2, seed=3)
    sp_all = species_of(meta, z)
    ei, ev = build_graph(pos, cell, True, 5.0)
    whole = B200Engine(meta, arrays)
    whole.set_graph(sp_all, ei, ev)
    whole.compute(); torch.cuda.synchronize()
    ref = {k: v.cpu().numpy().copy() for k, v in whole.results().items()}

    world = 2
    parts = [brick_decompose(pos, cell, sp_all, (2, 1, 1), r, 5.0) for r in range(world)]
    engs = [B200Engine(meta, arrays) for _ in range(world)]
    owner_row = {}                                   # global id -> (rank, owned row)
    for r, p in enumerate(parts):
        order = np.argsort(p['edge_index'][0], kind='stable')
        engs[r].set_graph_host(p['species'], p['edge_index'][0][order], p['edge_index'][1][order], p['edge_vec'][order], p['n_local'])
        for row, g in enumerate(p['global_ids'][:p['n_local']]):
            owner_row[int(g)] = (r, row)
    T = engs[0].spec.n_layers

    def forward(name, layer, width):                 # ghost rows <- owners' rows
        owned = [engs[r].read_rows(name, layer, 0, parts[r]['n_local'], width) for r in range(world)]
        for r, p in enumerate(parts):
            ghosts = p['global_ids'][p['n_local']:]
            if len(ghosts):
                rows = np.stack([owned[owner_row[int(g)][0]][owner_row[int(g)][1]] for g in ghosts])
                engs[r].write_rows(name, layer, p['n_local'], rows)

    def reverse(name, layer, width):                 # owners' rows += the ghost rows that stand for them
        full = [engs[r].read_rows(name, layer, 0, parts[r]['n_nodes'], width) for r in range(world)]
        acc = [full[r][:parts[r]['n_local']].astype(np.float64) for r in range(world)]
        for r, p in enumerate(parts):
            for k, g in enumerate(p['global_ids'][p['n_local']:]):
                q, row = owner_row[int(g)]
                acc[q][row] += full[r][p['n_local'] + k]
        for r in range(world):
            engs[r].write_rows(name, layer, 0, acc[r].astype(np.float32))
        return acc

    for e in engs:
        e.run_stage(E.STAGE_FWD_BEGIN)
    for t in range(T):
        for e in engs:
            e.run_stage(E.STAGE_FWD_LAYER, t)
        if t + 1 < T:
            forward('x', t + 1, engs[0].spec.layers[t + 1].dim_x)
    for e in engs:
        e.run_stage(E.STAGE_FWD_END)
    for t in range(T - 1, -1, -1):
        for e in engs:
            e.run_stage(E.STAGE_BWD_LAYER_A, t)
        if t > 0:
            reverse('dx', t, engs[0].spec.layers[t].dim_x)
            for e in engs:
                e.run_stage(E.STAGE_BWD_LAYER_B, t)
    for e in engs:
        e.run_stage(E.STAGE_BWD_END)
    forces = reverse('forces', 0, 3)
    energy = sum(e.read_scalars()[0] for e in engs)
    virial = sum(e.read_scalars()[1] for e in engs)
    f_all = np.zeros((len(pos), 3))
    for r, p in enumerate(parts):
        f_all[p['global_ids'][:p['n_local']]] = forces[r]
    assert abs(energy - ref['energy'][0]) < 2e-5
    assert np.allclose(f_all, ref['forces'], atol=5e-6)
    assert np.allclose(virial, ref['virial'], atol=5e-4)


def _stage_graph_worker(rank, world, port, q):
    import os
    import torch
    import torch.distributed as dist
    from sevenn_b200.engine import B200Engine, set_option
    from sevenn_b200.neighbors import diamond_si
    from sevenn_b200.parallel import DistributedRunner, brick_decompose
    from helpers import species_of
    os.environ['MASTER_ADDR'] = '127.0.0.1'
    os.environ['MASTER_PORT'] = str(port)
    torch.cuda.set_device(rank)
    dist.init_process_group('nccl', rank=rank, world_size=world, device_id=torch.device('cuda', rank))
    try:
        meta, arrays = model_weights('sevennet_0')
        pos, cell, z = diamond_si(4, 3, 3, seed=2)
        part = brick_decompose(pos, cell, species_of(meta, z), (2, 1, 1), rank, 5.0)
        run = DistributedRunner(B200Engine(meta, arrays, device=rank), part, cuda_graph=False, stage_graphs=False)
        run.compute()
        torch.cuda.synchronize()
        ref = run.results()
        set_option('stage_graphs', 1)       # every stage between two exchanges: captured once, then replayed
        for _ in range(3):
            run.compute()
        torch.cuda.synchronize()
        out = run.results()
        captures, replays = run.engine.stage_graph_stats()
        ok = (captures > 0 and replays == 3 * captures
              and abs(float(out['energy'].cpu()[0]) - float(ref['energy'].cpu()[0])) < 1e-9
              and bool(torch.allclose(out['forces'], ref['forces'], atol=2e-6)))
        q.put((rank, ok, captures, replays))
    finally:
        set_option('stage_graphs', 0)
        dist.destroy_process_group()


def test_stage_graphs_between_nccl_exchanges_two_gpus():
    import socket
    import torch
    import torch.multiprocessing as mp
    if torch.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs')
    s = socket.socket()
    s.bind(('127.0.0.1', 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context('spawn')
    q = ctx.Queue()
    procs = [ctx.Process(target=_stage_graph_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    try:
        res = [q.get(timeout=300) for _ in range(2)]
        for p in procs:
            p.join(timeout=120)
    finally:
        for p in procs:
            if p.is_alive():
                p.kill()
    assert all(ok for _, ok, _, _ in res), res


def test_lammps_pair_styles_in_the_mock_harness_with_the_real_library(tmp_path):
    """tests/mock_lammps/harness_parallel.cpp built with -DREAL_ENGINE: both pair styles go through settings() /
    coeff() with an exported model file and run on the GPU inside the mock LAMMPS (64 Si atoms + ~460 periodic image
    ghosts, stock Comm hooks); reference = the library's positions-in entry on the periodic cell.  (The same harness
    runs on the CPU against a toy double of the stage protocol in tests/test_host_logic.py.)"""
    import os
    import subprocess
    from helpers import ROOT
    from sevenn_b200.export import export_flat
    mock, ex = os.path.join(ROOT, 'tests', 'mock_lammps'), os.path.join(ROOT, 'examples', 'lammps')
    lib_dir = os.path.join(ROOT, 'sevenn_b200', 'lib')
    exe = str(tmp_path / 'harness_real')
    subprocess.check_call(['g++', '-std=c++17', '-O1', '-DREAL_ENGINE', '-I', mock, '-I', ex, os.path.join(mock, 'harness_parallel.cpp'),
                           os.path.join(ex, 'pair_e3gnn_b200_parallel.cpp'), os.path.join(ex, 'pair_e3gnn_b200.cpp'), '-o', exe,
                           f'-L{lib_dir}', '-lsevenn_b200', f'-Wl,-rpath,{lib_dir}'])
    meta, arrays = model_weights('sevennet_0')
    model = str(tmp_path / 'sevennet_0.s7b')
    export_flat(model, meta, arrays)
    p = subprocess.run([exe, model], capture_output=True, text=True, timeout=300)
    assert p.returncode == 0 and p.stdout.strip().endswith('OK'), p.stdout + p.stderr
