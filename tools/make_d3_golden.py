#!/usr/bin/env python
"""Generate tests/golden/d3_reference_nacl.npz: the reference's own CUDA D3 on three rocksalt NaCl cells.

Needs a GPU and oracle/_ref/libpaird3.so, the unmodified reference D3 compiled by oracle/Makefile
(``make -C oracle REF=<reference checkout>/sevenn/pair_e3gnn``).  For each case the file stores the inputs
(``<case>_numbers``, ``_positions``, ``_cell``) and the reference's results (``_energy`` eV, ``_forces`` eV/A,
``_sigma`` = its pair_get_stress, eV), all float64 except the atomic numbers.  tests/test_d3_gpu.py compares the
repository's D3 kernels with them.

    python tools/make_d3_golden.py [OUT.npz]
"""
import ctypes
import os
import sys

import numpy as np

ROOT = os.path.join(os.path.dirname(os.path.abspath(__file__)), '..')
sys.path.insert(0, ROOT)
OUT = os.path.join(ROOT, 'tests', 'golden', 'd3_reference_nacl.npz')

# (rocksalt cells, damping): 64 / 1152 / 1000 atoms, rocksalt_nacl(*cells, sigma=0.05, seed=11)
CASES = [((2, 2, 2), 'damp_bj'), ((6, 6, 4), 'damp_bj'), ((5, 5, 5), 'damp_zero')]


def case_key(cells, damping):
    return 'nacl_{}x{}x{}_{}'.format(*cells, damping)


def reference_lib(path=os.path.join(ROOT, 'oracle', '_ref', 'libpaird3.so')):
    lib = ctypes.CDLL(path)
    lib.pair_init.restype = ctypes.c_void_p
    lib.pair_get_energy.restype = ctypes.c_double
    lib.pair_get_force.restype = ctypes.POINTER(ctypes.c_double)
    lib.pair_get_stress.restype = ctypes.POINTER(ctypes.c_double * 6)
    for fn in ('pair_set_atom', 'pair_set_domain', 'pair_run_settings', 'pair_run_coeff', 'pair_run_compute', 'pair_fin'):
        getattr(lib, fn).restype = None
    lib.pair_get_energy.argtypes = lib.pair_get_force.argtypes = lib.pair_get_stress.argtypes = [ctypes.c_void_p]
    lib.pair_set_atom.argtypes = [ctypes.c_void_p, ctypes.c_int, ctypes.c_int, ctypes.c_void_p, ctypes.c_void_p]
    lib.pair_set_domain.argtypes = [ctypes.c_void_p] + [ctypes.c_int] * 3 + [ctypes.c_void_p] * 2 + [ctypes.c_double] * 3
    lib.pair_run_settings.argtypes = [ctypes.c_void_p, ctypes.c_double, ctypes.c_double, ctypes.c_char_p, ctypes.c_char_p]
    lib.pair_run_coeff.argtypes = [ctypes.c_void_p, ctypes.c_void_p]
    lib.pair_run_compute.argtypes = lib.pair_fin.argtypes = [ctypes.c_void_p]
    return lib


def run_reference_d3(lib, z, pos, cell, damping=b'damp_bj'):
    """the compiled, unmodified reference at its default cutoffs (orthogonal / lower-triangular cells only: no
    frame rotation here)"""
    uniq = list(dict.fromkeys(np.asarray(z).tolist()))
    types = np.ascontiguousarray([uniq.index(a) + 1 for a in z], dtype=np.int32)
    x = np.ascontiguousarray(pos, dtype=np.float64)
    nums = np.ascontiguousarray(uniq, dtype=np.int32)
    lo, hi = np.zeros(3), np.ascontiguousarray([cell[0, 0], cell[1, 1], cell[2, 2]], dtype=np.float64)
    p = lib.pair_init()
    lib.pair_set_atom(p, len(z), len(uniq), types.ctypes.data, x.ctypes.data)
    lib.pair_set_domain(p, 1, 1, 1, lo.ctypes.data, hi.ctypes.data, float(cell[1, 0]), float(cell[2, 0]), float(cell[2, 1]))
    lib.pair_run_settings(p, 9000.0, 1600.0, damping, b'pbe')
    lib.pair_run_coeff(p, nums.ctypes.data)
    lib.pair_run_compute(p)
    e = lib.pair_get_energy(p)
    f = np.ctypeslib.as_array(lib.pair_get_force(p), shape=(len(z) * 3,)).reshape(-1, 3).copy()
    s = np.array(lib.pair_get_stress(p).contents)
    return e, f, s


def main(out=OUT):
    from sevenn_b200.neighbors import rocksalt_nacl
    lib = reference_lib()
    data = {}
    for cells, damping in CASES:
        pos, cell, z = rocksalt_nacl(*cells, sigma=0.05, seed=11)
        e, f, s = run_reference_d3(lib, z, pos, cell, damping.encode())
        k = case_key(cells, damping)
        data.update({f'{k}_numbers': np.asarray(z, dtype=np.int32), f'{k}_positions': np.asarray(pos, dtype=np.float64),
                     f'{k}_cell': np.asarray(cell, dtype=np.float64), f'{k}_energy': np.float64(e),
                     f'{k}_forces': f.astype(np.float64), f'{k}_sigma': s.astype(np.float64)})
        print(f'{k}: {len(z)} atoms, E = {e:.10f} eV, max|F| = {np.abs(f).max():.3e} eV/A')
    os.makedirs(os.path.dirname(os.path.abspath(out)), exist_ok=True)
    np.savez_compressed(out, **data)
    print('wrote', out, os.path.getsize(out), 'bytes')


if __name__ == '__main__':
    main(*sys.argv[1:2])
