#!/usr/bin/env python
"""Benchmark of the per-MD-step energy+force hot path (BASELINE.json metric:
atom-updates/sec per MD step, SevenNet-0, 1/2/4/8 B200).

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA engine
    python bench.py --impl reference --gpus N --steps K ...   # the CPU oracle (reference arm)
    python bench.py ... --dump-outputs DIR                    # also write the last timed step's results as DIR/*.npy

One "step" = one energy+force evaluation of one periodic Si cell with a fixed neighbour list:
  N = 1 : BASELINE configs[1], SevenNet-0, Si 10x10x15 = 12 000 atoms, 336 000 edges
  N > 1 : weak scaling at ~12 500 atoms per GPU (configs[3] at N = 8: Si 25x25x20 = 100 000 atoms),
          spatial brick decomposition with NCCL ghost exchange (one rank per GPU, torchrun).
`value` is timed with inputs resident in HBM (CUDA events, L2 flushed between steps); `e2e` is
the same metric through the host-buffer C-ABI call with pinned host inputs copied in and
forces/energy copied out inside the timed region.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = 'atom_updates_per_sec'
UNIT = 'atom-updates/s'
CELLS = {1: (10, 10, 15), 2: (25, 25, 5), 4: (25, 25, 10), 8: (25, 25, 20)}
GRIDS = {1: (1, 1, 1), 2: (2, 1, 1), 4: (2, 2, 1), 8: (2, 2, 2)}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
         'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, index=0):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        self.rows = []
        try:
            self.proc = subprocess.Popen(
                ['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits', '-lms', '100',
                 '-i', str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def stop(self):
        if self.proc is None:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': ['nvidia-smi unavailable']}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm = [float(r[1]) for r in self.rows if len(r) >= 9 and r[1].replace('.', '').isdigit()]
        mx = [float(r[2]) for r in self.rows if len(r) >= 9 and r[2].replace('.', '').isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) < 9:
                continue
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), r[5:9]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        return {'sm_mhz': statistics.median(sm) if sm else None, 'sm_max_mhz': max(mx) if mx else None,
                'samples': len(sm), 'reasons': sorted(reasons)}


DUMP_LIMIT = 60 << 20      # bytes of array data written by --dump-outputs (the .npy headers stay within 64 MB)


def dump_outputs(out_dir, arrays, limit=DUMP_LIMIT):
    """--dump-outputs: every array as <out_dir>/<name>.npy in float32 or float64, so that two builds of the project
    can be compared output by output on identical inputs.  Should the arrays exceed `limit` bytes in all, the largest
    keep a fixed sample of their rows (RandomState(0), sorted): the same rows for the same shapes."""
    arrs = {}
    for name, a in arrays.items():
        a = a.detach().cpu().numpy() if hasattr(a, 'detach') else np.asarray(a)
        arrs[name] = a if a.dtype in (np.float32, np.float64) else a.astype(np.float64)
    os.makedirs(out_dir, exist_ok=True)
    left = limit
    for i, name in enumerate(sorted(arrs, key=lambda k: arrs[k].nbytes)):
        a = arrs[name]
        share = left // (len(arrs) - i)
        if a.nbytes > share:
            rows = np.random.RandomState(0).choice(len(a), share // (a.nbytes // len(a)), replace=False)
            a = a[np.sort(rows)]
        np.save(os.path.join(out_dir, f'{name}.npy'), a)
        left -= a.nbytes
    print(f'bench: wrote {", ".join(sorted(arrs))} to {out_dir}', file=sys.stderr, flush=True)


def global_results(r, n_global, dev):
    """the distributed runner's per-rank results -> energy, virial and per-atom arrays over all atoms in the global
    atom order, on every rank (collective)"""
    import torch
    import torch.distributed as dist
    gids = torch.as_tensor(np.asarray(r['global_ids']), dtype=torch.long, device=dev)
    out = {'energy': r['energy'], 'virial': r['virial']}
    for k in ('atomic_energy', 'forces'):
        full = torch.zeros((n_global,) + tuple(r[k].shape[1:]), dtype=r[k].dtype, device=dev)
        full[gids] = r[k]
        dist.all_reduce(full)
        out[k] = full
    return out


def make_system(cells):
    from sevenn_b200.neighbors import build_graph, diamond_si
    pos, cell, z = diamond_si(*cells)
    ei, ev = build_graph(pos, cell, True, 5.0)
    return pos, cell, z, ei, ev


def make_oracle():
    import torch
    from oracle.oracle import Oracle
    from sevenn_b200.checkpoint import load_weights
    meta, arrays = load_weights(os.path.join(ROOT, 'weights', 'sevennet_0.npz'))
    return Oracle(meta, arrays, dtype=torch.float32), meta


def best_thread_count(o, meta):
    """torch-CPU gets slower, not faster, with one thread per core on many-core hosts for these
    small ops: pick the thread count (<= host cores) that runs a 216-atom step fastest."""
    import torch
    tm = {int(k): int(v) for k, v in meta['type_map'].items()}
    pos, cell, z, ei, ev = make_system((3, 3, 3))
    sp = np.array([tm[int(a)] for a in z])
    ncpu = os.cpu_count() or 1
    best = (None, 1e30)
    for th in sorted({t for t in (4, 8, 16, 32, 64, ncpu) if t <= ncpu}):
        torch.set_num_threads(th)
        o.forward(sp, ei, ev)
        t0 = time.perf_counter()
        o.forward(sp, ei, ev)
        dt = time.perf_counter() - t0
        if dt < best[1]:
            best = (th, dt)
    torch.set_num_threads(best[0])
    return best[0]


def run_reference(args):
    """Reference arm: the CPU oracle (this repo's restatement of the reference torch/e3nn path; the
    reference itself cannot be imported without e3nn) on the box's host cores, bounded sample."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    import torch
    o, meta = make_oracle()
    best_thread_count(o, meta)
    tm = {int(k): int(v) for k, v in meta['type_map'].items()}
    # calibrate the sample: largest of 216 / 512 / 1000 atoms whose step stays below ~4 s
    sample = None
    for nc in (3, 4, 5):
        pos, cell, z, ei, ev = make_system((nc, nc, nc))
        sp = np.array([tm[int(a)] for a in z])
        t0 = time.perf_counter()
        o.forward(sp, ei, ev)
        dt = time.perf_counter() - t0
        sample = (nc, sp, ei, ev, len(z))
        if dt * (((nc + 1) / nc) ** 3) > 4.0:
            break
    nc, sp, ei, ev, n_atoms = sample
    for _ in range(max(args.warmup, 1)):
        o.forward(sp, ei, ev)
    times = []
    for _ in range(args.steps):
        t0 = time.perf_counter()
        out = o.forward(sp, ei, ev)
        times.append(time.perf_counter() - t0)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {k: v for k, v in out.items() if isinstance(v, torch.Tensor) and v.is_floating_point()})
    total = sum(times)
    value = n_atoms * args.steps / total
    line = {
        'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * total / args.steps,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32',
        'data': 'synthetic', 'gpu_launches': 0,
        'config': {'workload': f'SevenNet-0 energy+forces, Si {nc}x{nc}x{nc} diamond cells = {n_atoms} atoms, '
                               f'{ei.shape[1]} edges (bounded CPU sample of the 12 000-atom workload)',
                   'weights': 'SevenNet-0 (11Jul2024) converted checkpoint'},
        'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': torch.get_num_threads(), 'kind': 'port',
                         'sample': f'{n_atoms}-atom Si cell, {args.steps} steps, torch-CPU fp32 oracle, '
                                   f'{torch.get_num_threads()} of {os.cpu_count()} host threads (fastest setting)'},
        'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
    }
    print(json.dumps(line), flush=True)


def parity_tolerance(n_atoms):
    """VERDICT r1 item 2: |dE| <= 1e-4 eV * sqrt(N/64), max|dF| <= 5e-5 eV/A."""
    return 1e-4 * (max(n_atoms, 64) / 64.0) ** 0.5, 5e-5


def oracle_parity(model, species, ei, ev, energy, forces, device):
    """One-off comparison (outside every timed region) of the engine's result on the benchmark cell with
    the fp64 oracle evaluated edge-chunked (oracle/oracle.py, `edge_chunk`) on `device`."""
    import torch
    from oracle.oracle import Oracle
    from sevenn_b200.checkpoint import load_weights
    meta, arrays = load_weights(os.path.join(ROOT, 'weights', f'{model}.npz'))
    t0 = time.perf_counter()
    o = Oracle(meta, arrays, dtype=torch.float64, device=device)
    ref = o.forward(species, ei, ev, edge_chunk=32768)
    if device != 'cpu':
        torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    dE = float(energy) - float(ref['energy'])
    dF = float(np.abs(np.asarray(forces, dtype=np.float64) - ref['forces'].cpu().numpy()).max())
    tolE, tolF = parity_tolerance(len(species))
    del o, ref
    if device != 'cpu':
        torch.cuda.empty_cache()
    return {'against': f'oracle fp64 (torch on {device}, edge-chunked), same cell', 'dE_eV': dE, 'max_dF_eV_per_A': dF,
            'dE_per_atom_eV': dE / len(species), 'tol_dE_eV': tolE, 'tol_dF_eV_per_A': tolF,
            'ok': bool(abs(dE) <= tolE and dF <= tolF), 'oracle_seconds': dt}


def gpu_standin(model, cells):
    """torch-CUDA unfused stand-in of the reference GPU path (tools/gpu_standin.py), in a subprocess so
    that its ~84 GiB of autograd state never coexists with the engine's buffers."""
    try:
        r = subprocess.run([sys.executable, os.path.join(ROOT, 'tools', 'gpu_standin.py'), model] + [str(c) for c in cells] + ['--json'],
                           capture_output=True, text=True, timeout=600)
        for ln in reversed(r.stdout.strip().splitlines()):
            if ln.startswith('{'):
                return json.loads(ln)
        return {'error': (r.stderr or r.stdout)[-300:]}
    except Exception as ex:   # noqa: BLE001
        return {'error': repr(ex)[:300]}


def time_steps(torch, step, steps, flush):
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    torch.cuda.synchronize()
    for a, b in evs:
        flush.fill_(1)
        a.record()
        step()
        b.record()
    torch.cuda.synchronize()
    return sum(a.elapsed_time(b) for a, b in evs) / steps


def extra_model(args, model, cells, flush, dev, local_rank, parity_device):
    """configs[2]: the same cell with another model (SevenNet-l3i5): ms/step, roofline of its dominant
    kernel, parity against the oracle."""
    import torch
    from sevenn_b200.checkpoint import load_weights
    from sevenn_b200.engine import B200Engine
    meta, arrays = load_weights(os.path.join(ROOT, 'weights', f'{model}.npz'))
    tm = {int(k): int(v) for k, v in meta['type_map'].items()}
    pos, cell, z, ei, ev = make_system(cells)
    species = np.array([tm[int(a)] for a in z], dtype=np.int32)
    eng = B200Engine(meta, arrays, radial=args.radial, device=local_rank)
    eng.set_graph(species, ei, ev)
    for _ in range(3):
        eng.compute()
    ms = time_steps(torch, eng.compute, min(args.steps, 10), flush)
    res = eng.results()
    energy, forces = float(res['energy'].cpu()[0]), res['forces'].cpu().numpy()
    eng.set_profiling(True)
    for _ in range(3):
        flush.fill_(1)
        eng.compute()
    torch.cuda.synchronize()
    roof, breakdown = roofline_from_profile(eng, eng.profile(), ei.shape[1], len(z), 3)
    eng.set_profiling(False)
    out = {'model': model, 'atoms': len(z), 'edges': int(ei.shape[1]), 'ms_per_step': ms, 'value': len(z) / (ms * 1e-3),
           'unit': UNIT, 'roofline': roof, 'kernel_breakdown_ms': breakdown, 'energy_eV': energy}
    if parity_device != 'off':
        out['parity'] = oracle_parity(model, species, ei, ev, energy, forces, parity_device)
    del eng
    torch.cuda.empty_cache()
    return out


def run_engine(args):
    import torch
    import torch.distributed as dist
    from sevenn_b200.checkpoint import load_weights
    from sevenn_b200.engine import B200Engine

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if world != args.gpus:
        if world == 1 and args.gpus > 1:
            raise SystemExit('--gpus N > 1 must be launched with torch.distributed.run (one rank per GPU)')
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        import datetime
        dist.init_process_group('nccl', device_id=dev, timeout=datetime.timedelta(seconds=600))

    from sevenn_b200.engine import set_option
    for opt in ('concurrent_conv', 'tc_gemm', 'cuda_graph', 'tc_swizzle'):   # A/B switches: S7B_CONCURRENT_CONV=0, S7B_TC_GEMM=1, S7B_CUDA_GRAPH=0
        if os.environ.get('S7B_' + opt.upper()) is not None:
            set_option(opt, int(os.environ['S7B_' + opt.upper()]))
    meta, arrays = load_weights(os.path.join(ROOT, 'weights', f'{args.model}.npz'))
    tm = {int(k): int(v) for k, v in meta['type_map'].items()}
    cells = CELLS[args.gpus] if args.cells is None else tuple(args.cells)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)   # > 126 MB L2

    sampler = ClockSampler(local_rank)
    if world == 1:
        pos, cell, z, ei, ev = make_system(cells)
        n_atoms, n_edges = len(z), ei.shape[1]
        species = np.array([tm[int(a)] for a in z], dtype=np.int32)
        eng = B200Engine(meta, arrays, radial=args.radial, device=local_rank)
        eng.set_graph(species, ei, ev)

        def step():
            eng.compute()
        runner = None
    else:
        from sevenn_b200.parallel import DistributedRunner, brick_decompose
        from sevenn_b200.neighbors import diamond_si
        pos, cell, z = diamond_si(*cells)
        n_atoms = len(z)
        species_all = np.array([tm[int(a)] for a in z], dtype=np.int32)
        part = brick_decompose(pos, cell, species_all, GRIDS[args.gpus], rank, 5.0)
        n_edges_local = part['edge_index'].shape[1]
        eng = B200Engine(meta, arrays, radial=args.radial, device=local_rank)
        runner = DistributedRunner(eng, part)      # whole step (NCCL included) as one CUDA graph; S7B_CUDA_GRAPH=0: per-stage graphs
        t = torch.tensor([n_edges_local], device=dev, dtype=torch.int64)
        dist.all_reduce(t)
        n_edges = int(t.item())

        def step():
            runner.compute()

    # ---- device-resident timing ------------------------------------------------------------------
    def timed_run():
        """W warm-up steps, then exactly K timed steps -> (sum of the step times in ms, max over ranks; launches; clocks)"""
        for _ in range(max(args.warmup, 3)):
            step()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        (runner or eng).launch_count(reset=True)
        sampler.start()
        evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
        torch.cuda.synchronize()
        for a, b in evs:
            flush.fill_(1)          # evict L2 between timed iterations (untimed)
            if world > 1:
                dist.barrier()
            a.record()
            step()
            b.record()
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        clk = sampler.stop()
        n_launch = (runner or eng).launch_count()      # replays of the captured step count the kernels recorded in it
        ms = torch.tensor([sum(a.elapsed_time(b) for a, b in evs)], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        return float(ms.item()), n_launch, clk

    # N > 1: the direct-launch schedule (measured at N = 1..8 in round 1 and 2) is timed first, then the same K steps
    # with the whole step replayed as one CUDA graph (NCCL inside).  Should the graph phase ever hang -- NCCL capture
    # was only exercised on 2 GPUs while this was written -- a timer prints the line of the direct-launch phase
    # instead of leaving the run without one.
    direct, guard = None, None
    if runner is not None and runner.use_graph:
        runner.set_cuda_graph(False)
        d_ms, d_launch, d_clk = timed_run()
        direct = {'ms_per_step': d_ms / args.steps, 'value': n_atoms * args.steps / (d_ms * 1e-3), 'gpu_launches': int(d_launch)}
        guard = graph_phase_guard(args, rank, n_atoms, n_edges, cells, direct, d_clk)
        runner.set_cuda_graph(True)
    total_ms, launches, clocks = timed_run()
    value = n_atoms * args.steps / (total_ms * 1e-3)
    if args.dump_outputs:       # the last timed step's results, read before any later leg runs the engine again
        res = (runner or eng).results()
        if world > 1:
            res = global_results(res, n_atoms, dev)
        if rank == 0:
            dump_outputs(args.dump_outputs, res)

    # ---- per-kernel breakdown + roofline of the dominant kernel (rank 0) ---------------------------
    # (every rank runs the same steps -- the exchanges are collective; only rank 0 records events)
    roofline, breakdown = None, None
    if runner is not None:
        graph_on = runner.use_graph
        runner.set_cuda_graph(False)      # per-kernel events need the eager stage sequence
    eng.set_profiling(rank == 0)
    for _ in range(min(args.steps, 10)):
        flush.fill_(1)
        step()
    torch.cuda.synchronize()
    if rank == 0:
        prof = eng.profile()
        roofline, breakdown = roofline_from_profile(eng, prof, n_edges if world == 1 else n_edges_local, eng.n_local, min(args.steps, 10))
    eng.set_profiling(False)
    if runner is not None:
        runner.set_cuda_graph(graph_on)

    # ---- end to end through the host-buffer entry (N = 1) or the runner's host path (N > 1) -------
    if world == 1:
        def pinned(a):
            t = torch.from_numpy(np.ascontiguousarray(a)).pin_memory()
            return t, t.numpy()
        keep = [pinned(species), pinned(ei[0].astype(np.int32)), pinned(ei[1].astype(np.int32)), pinned(ev.astype(np.float32))]
        h_sp, h_c, h_n, h_v = [k[1] for k in keep]
        h2d = h_sp.nbytes + h_c.nbytes + h_n.nbytes + h_v.nbytes      # species, centre, neighbour, edge_vec
        d2h = 12 * n_atoms + 4 * n_atoms + 8 + 48

        def e2e_step():
            return eng.compute_host(h_sp, h_c, h_n, h_v)
    else:
        h2d, d2h = runner.host_bytes()

        def e2e_step():
            return runner.compute_host()
    for _ in range(3):
        e2e_step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    for _ in range(args.steps):
        out = e2e_step()
    b.record()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    e2e_ms = torch.tensor([max(a.elapsed_time(b), wall * 1e3)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(e2e_ms, op=dist.ReduceOp.MAX)
    e2e_value = n_atoms * args.steps / (float(e2e_ms.item()) * 1e-3)

    # ---- informational: positions in -> forces out (device neighbour list inside the timed region) ----
    e2e_pos = None
    if world == 1:
        for _ in range(2):
            eng.compute_positions(species, pos, cell, True)
        t0 = time.perf_counter()
        for _ in range(args.steps):
            eng.compute_positions(species, pos, cell, True)
        torch.cuda.synchronize()
        e2e_pos = {'value': n_atoms * args.steps / (time.perf_counter() - t0), 'unit': UNIT,
                   'h2d_bytes_per_step': 28 * n_atoms, 'd2h_bytes_per_step': 16 * n_atoms + 56,
                   'what': 'host positions -> device neighbour list + graph -> energy/forces -> host'}
        eng.set_graph(species, ei, ev)

    # ---- parity of the benchmarked configuration (outside the timed regions) --------------------------
    parity, extra, standin = None, None, None
    if world == 1:
        eng.compute()
        torch.cuda.synchronize()
        res = eng.results()
        if args.parity != 'off':
            parity = oracle_parity(args.model, species, ei, ev, float(res['energy'].cpu()[0]), res['forces'].cpu().numpy(), args.parity)
        if args.cells is None and args.model == 'sevennet_0' and not args.no_extras:
            extra = {'l3i5': extra_model(args, 'sevennet_l3i5', cells, flush, dev, local_rank, 'cuda' if args.parity != 'off' else 'off')}
            del flush
            torch.cuda.empty_cache()
            standin = gpu_standin(args.model, cells)
    else:
        parity = distributed_parity(runner, eng, meta, arrays, pos, cell, species_all, local_rank)

    if rank == 0:
        line = {
            'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
            'warmup': max(args.warmup, 3), 'ms_per_step': total_ms / args.steps, 'higher_is_better': True,
            'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
            'config': {
                'workload': f'{args.model} energy+forces per MD step, diamond Si {cells[0]}x{cells[1]}x{cells[2]} cells = '
                            f'{n_atoms} atoms, {n_edges} directed edges, cutoff 5.0 A, positions = lattice + N(0, 0.05 A)',
                'weights': f'{args.model} converted from the reference checkpoint', 'radial': args.radial,
                'parallelism': 'single GPU' if world == 1 else f'spatial bricks {GRIDS[args.gpus]} + NCCL ghost exchange',
                'l2': 'flushed with a 256 MiB write between timed steps',
                'cuda_graph': (bool(int(os.environ.get('S7B_CUDA_GRAPH', '1'))) and args.radial == 'table') if world == 1
                else (True if (runner.use_graph and runner.graph_replays > 0) else ('per stage' if runner.stage_graphs else False)),
                'cuda_graph_note': None if world == 1 else (
                    runner.graph_error or (f'{runner.graph_captures} capture(s), {runner.graph_replays} replays; NCCL calls inside the graph'
                                           if runner.graph_replays > 0 else
                                           'stage graphs (captures, replays) = %s; NCCL calls between the graphs' % (eng.stage_graph_stats(),))),
                'tc_gemm': bool(int(os.environ.get('S7B_TC_GEMM', '1'))),
                'energy_eV': float(out[0]) if world == 1 else float(out['energy'])},
            'e2e': {'value': e2e_value, 'unit': UNIT, 'h2d_bytes_per_step': int(h2d), 'd2h_bytes_per_step': int(d2h)},
            'e2e_positions': e2e_pos,
            'gpu_launches': int(launches), 'clocks': clocks, 'roofline': roofline, 'kernel_breakdown_ms': breakdown,
            'parity': parity,
        }
        if extra is not None:
            line['extra'] = extra
        if standin is not None:
            line['gpu_standin'] = standin
        if world == 1 and not args.no_cpu_baseline:
            line['cpu_baseline'] = cpu_baseline()
        if direct is not None:
            line['config']['direct_launch'] = direct       # the same K steps without the whole-step graph
        if guard is not None:
            guard.cancel()
        print(json.dumps(line), flush=True)
    if guard is not None:
        guard.cancel()
    if world > 1:
        shutdown(runner)


def graph_phase_guard(args, rank, n_atoms, n_edges, cells, direct, clocks, deadline_s=240.0):
    """timer armed before the first whole-step graph capture of a multi-rank run: if the rest of the run does not
    finish in time, rank 0 prints the line of the direct-launch phase (device-resident number only) and every
    rank leaves with exit code 0"""
    def expire():
        if rank == 0:
            line = {'metric': METRIC, 'value': direct['value'], 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
                    'warmup': max(args.warmup, 3), 'ms_per_step': direct['ms_per_step'], 'higher_is_better': True,
                    'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
                    'config': {'workload': f'{args.model} energy+forces per MD step, diamond Si {cells[0]}x{cells[1]}x{cells[2]} cells = '
                                           f'{n_atoms} atoms, {n_edges} directed edges, cutoff 5.0 A, positions = lattice + N(0, 0.05 A)',
                               'parallelism': f'spatial bricks {GRIDS[args.gpus]} + NCCL ghost exchange',
                               'l2': 'flushed with a 256 MiB write between timed steps', 'cuda_graph': False,
                               'cuda_graph_note': f'the whole-step graph phase did not finish within {deadline_s:.0f} s; this is the '
                                                  f'direct-launch phase of the same run (no e2e / parity legs)'},
                    'e2e': {'value': None, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0,
                            'note': 'not measured: the run ended in the fallback of the graph-phase guard'},
                    'gpu_launches': direct['gpu_launches'], 'clocks': clocks, 'roofline': None, 'parity': None}
            print(json.dumps(line), flush=True)
        os._exit(0)
    t = threading.Timer(deadline_s, expire)
    t.daemon = True
    t.start()
    return t


def shutdown(runner):
    """multi-rank teardown: the captured step graph refers to the NCCL communicator and must go first
    (ncclCommDestroy waits for such graphs); a timer guards the teardown so that a bench line that is already
    printed is never followed by a hung process"""
    import threading
    import torch
    import torch.distributed as dist
    sys.stdout.flush()
    guard = threading.Timer(90.0, lambda: os._exit(0))
    guard.daemon = True
    guard.start()
    if runner is not None:
        runner.close()
    torch.cuda.synchronize()
    dist.barrier()
    dist.destroy_process_group()
    guard.cancel()


def distributed_parity(runner, eng, meta, arrays, pos, cell, species_all, local_rank):
    """N > 1: rank 0 also evaluates the SAME global system with a single-GPU engine and compares energy
    and forces of all atoms with the distributed result (forces gathered over NCCL).  Outside the timed
    regions.  (The single-GPU engine itself is compared with the fp64 oracle in the N = 1 line.)"""
    import torch
    import torch.distributed as dist
    from sevenn_b200.engine import B200Engine
    from sevenn_b200.neighbors import build_graph
    runner.compute()
    torch.cuda.synchronize()
    r = runner.results()
    world, rank = dist.get_world_size(), dist.get_rank()
    n_global = len(species_all)
    f_all = torch.zeros(n_global, 3, dtype=torch.float32, device=eng.device)
    gids = torch.as_tensor(np.asarray(r['global_ids']), dtype=torch.long, device=eng.device)
    f_all[gids] = r['forces']
    dist.all_reduce(f_all)
    e_dist = float(r['energy'].cpu()[0])
    out = None
    if rank == 0:
        t0 = time.perf_counter()
        ei, ev = build_graph(pos, cell, True, 5.0)
        single = B200Engine(meta, arrays, radial=eng.radial, device=local_rank)
        single.set_graph(species_all, ei, ev)
        single.compute()
        torch.cuda.synchronize()
        rs = single.results()
        dE = e_dist - float(rs['energy'].cpu()[0])
        dF = float((f_all - rs['forces']).abs().max())
        tolE, tolF = parity_tolerance(n_global)
        out = {'against': 'the same global system evaluated by this engine on ONE GPU (rank 0)', 'dE_eV': dE,
               'max_dF_eV_per_A': dF, 'dE_per_atom_eV': dE / n_global, 'tol_dE_eV': tolE, 'tol_dF_eV_per_A': tolF,
               'ok': bool(abs(dE) <= tolE and dF <= tolF), 'seconds': time.perf_counter() - t0}
        del single
        torch.cuda.empty_cache()
    dist.barrier()
    return out


def run_nacl_d3(args):
    """BASELINE configs[4]: SevenNet-0 + D3 dispersion on a rocksalt NaCl cell (25x25x10 = 50 000 atoms by
    default), N GPUs: the network by spatial bricks + NCCL ghost exchange, the D3 correction by atom
    decomposition with replicated positions (three small all-gathers).  One step = both, summed."""
    import torch
    import torch.distributed as dist
    from sevenn_b200.checkpoint import load_weights
    from sevenn_b200.d3 import D3Engine, distributed_d3
    from sevenn_b200.engine import B200Engine
    from sevenn_b200.neighbors import build_graph, rocksalt_nacl
    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        import datetime
        dist.init_process_group('nccl', device_id=dev, timeout=datetime.timedelta(seconds=600))
    meta, arrays = load_weights(os.path.join(ROOT, 'weights', 'sevennet_0.npz'))
    tm = {int(k): int(v) for k, v in meta['type_map'].items()}
    cells = (25, 25, 10) if args.cells is None else tuple(args.cells)
    pos, cell, z = rocksalt_nacl(*cells, a=args.nacl_a, sigma=0.05, seed=0)
    n_atoms = len(z)
    species = np.array([tm[int(a)] for a in z], dtype=np.int32)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    eng = B200Engine(meta, arrays, radial=args.radial, device=local_rank)
    d3 = D3Engine('damp_bj', 'pbe', device=local_rank)
    if world == 1:
        ei, ev = build_graph(pos, cell, True, 5.0)
        n_edges = ei.shape[1]
        eng.set_graph(species, ei, ev)

        def step():
            eng.compute()
            d3.set_system(z, pos, cell)
            for st in (1, 2, 3):
                d3.run_stage(st)
    else:
        from sevenn_b200.parallel import DistributedRunner, brick_decompose
        part = brick_decompose(pos, cell, species, GRIDS[args.gpus], rank, 5.0)
        runner = DistributedRunner(eng, part)
        t = torch.tensor([part['edge_index'].shape[1]], device=dev, dtype=torch.int64)
        dist.all_reduce(t)
        n_edges = int(t.item())

        def step():
            runner.compute()
            distributed_d3(d3, z, pos, cell)
    for _ in range(max(args.warmup, 3)):
        step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    (eng if world == 1 else runner).launch_count(reset=True)
    total = 0.0
    t_net = t_d3 = 0.0
    for _ in range(args.steps):
        flush.fill_(1)
        if world > 1:
            dist.barrier()
        a, b, c = (torch.cuda.Event(enable_timing=True) for _ in range(3))
        a.record()
        if world == 1:
            eng.compute()
        else:
            runner.compute()
        b.record()
        if world == 1:
            d3.set_system(z, pos, cell)
            for st in (1, 2, 3):
                d3.run_stage(st)
            e_d3, f_d3, s_d3 = d3.results()
        else:
            e_d3, f_d3, s_d3 = distributed_d3(d3, z, pos, cell)
        c.record()
        torch.cuda.synchronize()
        total += a.elapsed_time(c)
        t_net += a.elapsed_time(b)
        t_d3 += b.elapsed_time(c)
    clocks = sampler.stop()
    launches = (eng if world == 1 else runner).launch_count()      # network kernels only (the D3 library entry points do not feed this counter)
    if args.dump_outputs:
        res = (eng if world == 1 else runner).results()
        if world > 1:
            res = global_results(res, n_atoms, dev)
        if rank == 0:
            dump_outputs(args.dump_outputs, {**{f'network_{k}': v for k, v in res.items()},
                                             'd3_energy': np.float64(e_d3), 'd3_forces': f_d3, 'd3_sigma': s_d3})
    tt = torch.tensor([total, t_net, t_d3], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
    total, t_net, t_d3 = (float(v) for v in tt.cpu())
    e_net = float((eng.buffer('energy', dtype='f8')).cpu()[0])
    parity = None
    if world > 1:      # rank 0: the same system on one GPU, network and D3
        f_all = torch.zeros(n_atoms, 3, dtype=torch.float32, device=dev)
        r = runner.results()
        gids = torch.as_tensor(np.asarray(r['global_ids']), dtype=torch.long, device=dev)
        f_all[gids] = r['forces']
        dist.all_reduce(f_all)
        if rank == 0:
            ei, ev = build_graph(pos, cell, True, 5.0)
            single = B200Engine(meta, arrays, radial=args.radial, device=local_rank)
            single.set_graph(species, ei, ev)
            single.compute()
            torch.cuda.synchronize()
            rs = single.results()
            e1, f1, _ = D3Engine('damp_bj', 'pbe', device=local_rank).compute(z, pos, cell)
            tolE, tolF = parity_tolerance(n_atoms)
            parity = {'against': 'the same system on ONE GPU (rank 0): SevenNet-0 and D3 separately',
                      'net_dE_eV': e_net - float(rs['energy'].cpu()[0]), 'net_max_dF': float((f_all - rs['forces']).abs().max()),
                      'd3_dE_eV': e_d3 - e1, 'd3_max_dF': float(np.abs(f_d3 - f1).max()), 'tol_dE_eV': tolE, 'tol_dF_eV_per_A': tolF}
            parity['ok'] = bool(abs(parity['net_dE_eV']) <= tolE and parity['net_max_dF'] <= tolF
                                and abs(parity['d3_dE_eV']) <= tolE and parity['d3_max_dF'] <= tolF)
        dist.barrier()
    if rank == 0:
        ms = total / args.steps
        line = {'metric': METRIC, 'value': n_atoms / (ms * 1e-3), 'unit': UNIT, 'n_gpus': args.gpus, 'steps': args.steps,
                'warmup': max(args.warmup, 3), 'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'strong',
                'vs_baseline': None, 'dtype': 'f32 (network), f32 pair terms / f64 sums (D3)', 'data': 'synthetic',
                'config': {'workload': f'SevenNet-0 + D3(BJ, pbe, 9000/1600 bohr^2) energy+forces per MD step, rocksalt NaCl a = {args.nacl_a} A, '
                                       f'{cells[0]}x{cells[1]}x{cells[2]} cells = {n_atoms} atoms, {n_edges} network edges',
                           'parallelism': 'single GPU' if world == 1 else f'network: spatial bricks {GRIDS[args.gpus]} + NCCL ghost exchange; '
                                          f'D3: atom decomposition, replicated positions, 3 all-gathers',
                           'l2': 'flushed with a 256 MiB write between timed steps',
                           'note': 'the reference D3 is single-GPU, O(N^2) and capped at 46 340 atoms; this cell exceeds it'},
                'ms_network': t_net / args.steps, 'ms_d3': t_d3 / args.steps, 'energy_network_eV': e_net, 'energy_d3_eV': e_d3,
                'gpu_launches': int(launches), 'clocks': clocks, 'parity': parity}
        print(json.dumps(line), flush=True)
    if world > 1:
        shutdown(runner)


def roofline_from_profile(eng, prof, n_edges, n_dst, steps):
    """Roofline of the dominant kernel from the engine's CUDA-event profile (DESIGN.md section 4).
    The convolution kernels keep x (23 MB) and the radial tables (23 MB/layer) L2-resident, so their
    ALGORITHMIC HBM bytes are only the streamed per-edge records/harmonics/accumulators and the per-atom
    mid-feature slice; `achieved`/`frac` (bound = hbm, as the contract asks) are therefore small by
    construction.  What actually bounds them is reported next to it: `l2_gbs` (all algorithmic bytes
    incl. the L2-served table and gather traffic) and `fp32` (flops of the generated code vs the FP32
    pipe peak 148 SM x 128 lanes x 2 x SM clock)."""
    if not prof:
        return None, None
    # per profiled STEP, not per call: the split schedule of the multi-GPU runner launches a convolution label twice
    # per step (interior + boundary range)
    breakdown = {k: v[0] / steps for k, v in sorted(prof.items(), key=lambda kv: -kv[1][0])}
    name = next(iter(breakdown))
    ms = breakdown[name]
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json')))
    except Exception:
        pass
    peak = float(peaks.get('hbm_gbs', 6650.0))
    src = 'measured (MEASURED_PEAKS.json hbm_gbs)' if 'hbm_gbs' in peaks else 'fallback 6.65 TB/s (B200_PROFILING.md)'
    sm_mhz = float(peaks.get('sm_max_mhz', 1965.0))
    fp32_peak = 148 * 128 * 2 * sm_mhz * 1e6 / 1e12
    out = {'kernel': name, 'ms': ms, 'bound': 'fp32', 'achieved': None, 'peak': fp32_peak, 'unit': 'TFLOP/s', 'frac': None,
           'traffic': None, 'peak_source': f'FP32 FMA pipe: 148 SM x 128 lanes x 2 flop x {sm_mhz:.0f} MHz (theoretical; '
                                           f'MEASURED_PEAKS.json holds no fp32 entry)'}
    if name.startswith('conv_'):
        import importlib.util
        spec_ = importlib.util.spec_from_file_location('gen_kernels', os.path.join(ROOT, 'sevenn_b200', 'csrc', 'gen_kernels.py'))
        gk = importlib.util.module_from_spec(spec_)
        spec_.loader.exec_module(gk)
        parts = name.split('.')
        t, l1 = int(parts[1][1:]), int(parts[2][1:])
        L = eng.spec.layers[t]
        mul = L.x_muls[l1]
        paths = [p for p in L.paths if p.l1 == l1]
        nacc = sum(2 * p.l3 + 1 for p in paths)
        nys = (eng.spec.n_sh - 1 + 3) // 4 * 4
        bwd = name.startswith('conv_bwd')
        f_fwd, f_bwd, npath = gk.op_counts(l1, eng.spec.lmax_filter, len(L.out_muls) - 1)
        # HBM: edge record 16 B + harmonics + (bwd) dY/dEdr read-modify-write; per atom the mid slice
        hbm = (16 + 4 * nys + ((8 * nys + 8) if bwd else 0)) * n_edges + 4 * nacc * mul * n_dst
        # L2-served: gathered x slice, radial coefficients (12 B per channel), (bwd) dx reduction
        l2 = (4 * (2 * l1 + 1) * mul + (12 if eng.radial == 'table' else 4) * npath * mul
              + (4 * (2 * l1 + 1) * mul if (bwd and t > 0) else 0)) * n_edges
        flops = ((f_bwd + 15 * npath) if bwd else (f_fwd + 6 * npath)) * mul * n_edges
        out.update(achieved=flops / (ms * 1e-3) / 1e12, algorithmic_flops=int(flops))
        out['frac'] = out['achieved'] / fp32_peak
        out['hbm'] = {'achieved_gbs': hbm / (ms * 1e-3) / 1e9, 'peak_gbs': peak, 'frac': hbm / (ms * 1e-3) / 1e9 / peak,
                      'algorithmic_bytes': int(hbm), 'peak_source': src}
        out['l2_gbs'] = (hbm + l2) / (ms * 1e-3) / 1e9
        try:   # dram bytes per launch of this kernel kind from the committed ncu --set full capture (mid layers, 12k atoms)
            tr = json.load(open(os.path.join(ROOT, 'profiles', 'ncu_traffic.json')))
            if 1 <= t <= 3 and n_dst == 12000:
                out['traffic'] = tr.get('sevennet_0' if eng.spec.lmax_filter == 2 else 'sevennet_l3i5', {}).get(f'{parts[0]}.l{l1}')
        except Exception:
            pass
        out['note'] = ('bound = the FP32 FMA pipe: the channel-wise Clebsch-Gordan product is not GEMM-shaped (DESIGN.md 4); x and the '
                       'radial tables are L2-resident, so the HBM fraction (`hbm`) is small by construction; traffic = ncu dram '
                       'bytes per launch from profiles/ncu_traffic.json')
    return out, breakdown


def cpu_baseline():
    """The oracle (CPU port of the reference torch/e3nn path) on this box's host cores, bounded sample."""
    import torch
    o, meta = make_oracle()
    best_thread_count(o, meta)
    tm = {int(k): int(v) for k, v in meta['type_map'].items()}
    pos, cell, z, ei, ev = make_system((4, 4, 4))
    sp = np.array([tm[int(a)] for a in z])
    o.forward(sp, ei, ev)
    times = []
    t_start = time.perf_counter()
    while len(times) < 3 or (time.perf_counter() - t_start < 12.0 and len(times) < 10):
        t0 = time.perf_counter()
        o.forward(sp, ei, ev)
        times.append(time.perf_counter() - t0)
    best = min(times)
    return {'value': len(z) / best, 'unit': UNIT, 'cores': torch.get_num_threads(), 'kind': 'port',
            'sample': f'SevenNet-0, {len(z)}-atom Si cell ({ei.shape[1]} edges), best of {len(times)} steps, '
                      f'torch-CPU fp32 oracle, {torch.get_num_threads()} of {os.cpu_count()} host threads (fastest setting)'}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='b200', choices=['b200', 'reference'])
    ap.add_argument('--model', default='sevennet_0')
    ap.add_argument('--radial', default='table', choices=['table', 'mlp'])
    ap.add_argument('--cells', type=int, nargs=3, default=None)
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--parity', default='cuda', choices=['cuda', 'cpu', 'off'],
                    help='where the fp64 oracle of the one-off parity check runs (it is the checker, never timed)')
    ap.add_argument('--no-extras', action='store_true', help='skip the l3i5 / gpu_standin legs of the N = 1 line')
    ap.add_argument('--workload', default='si', choices=['si', 'nacl_d3'],
                    help="'si': the headline benchmark (BASELINE configs[1]/[3]); 'nacl_d3': configs[4], SevenNet-0 + D3 on NaCl")
    ap.add_argument('--nacl-a', type=float, default=5.64,
                    help='lattice constant of the nacl_d3 workload; 4.0 is the dense variant of SURVEY 8(d).5 (about 65 neighbours per atom)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='after the timed steps, write the results of the last one as DIR/<name>.npy (float32/float64, '
                         'at most 64 MB in all); the inputs are the same on every run with the same arguments')
    args = ap.parse_args()
    if args.gpus not in CELLS:
        raise SystemExit('--gpus must be 1, 2, 4 or 8')
    if args.steps < 1:
        raise SystemExit('--steps must be at least 1')
    if args.impl == 'reference':
        run_reference(args)
    elif args.workload == 'nacl_d3':
        run_nacl_d3(args)
    else:
        run_engine(args)


if __name__ == '__main__':
    main()
