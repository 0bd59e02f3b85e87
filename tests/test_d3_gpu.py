"""GPU parity of the cell-list D3 kernels (csrc/d3_kernels.cuh through the C ABI) against the fp64 oracle
(oracle/d3_oracle.py), the reference's golden values (tests/unit_tests/test_calculator.py:192-238) and the stored
results of the reference's own CUDA D3 (tests/golden/d3_reference_nacl.npz)."""
import ctypes
import os

import numpy as np
import pytest

from test_d3_oracle import H2O_POS, H2O_REF, NACL, NACL_REF, h2o_cell

pytestmark = pytest.mark.gpu


def _rel(a, b):
    return np.abs(np.asarray(a) - np.asarray(b)).max() / (np.abs(np.asarray(b)).max() + 1e-300)


def test_reference_goldens():
    from sevenn_b200.d3 import D3Engine
    e, f, s = D3Engine().compute(NACL['numbers'], NACL['positions'], NACL['cell'])
    assert 0.0 <= e / NACL_REF['energy'] - 1.0 < 1e-4          # see tests/test_d3_oracle.py for the sign / size
    assert np.allclose(f, NACL_REF['forces'], atol=2e-7, rtol=0)
    vol = abs(np.linalg.det(np.array(NACL['cell'])))
    stress = -np.array([s[0], s[1], s[2], s[5], s[4], s[3]]) / vol
    assert np.allclose(stress, NACL_REF['stress'], rtol=5e-5, atol=5e-8)
    e, f, s = D3Engine().compute([8, 1, 1], H2O_POS, h2o_cell())
    assert abs(e / H2O_REF['energy'] - 1.0) < 5e-6
    assert np.allclose(f, H2O_REF['forces'], atol=2e-7, rtol=0)


@pytest.mark.parametrize('damping', ['damp_bj', 'damp_zero'])
@pytest.mark.parametrize('case', ['triclinic_mixed', 'slab', 'nacl_bulk'])
def test_matches_fp64_oracle(case, damping):
    from oracle.d3_oracle import d3_reference
    from sevenn_b200.d3 import D3Engine
    rng = np.random.RandomState(1)
    if case == 'triclinic_mixed':
        cell = np.array([[9.0, 0.5, 0.0], [0.3, 8.0, 0.6], [0.0, 0.4, 10.0]])
        z = rng.choice([1, 6, 8, 14, 29], size=40)
        pos = rng.uniform(0, 1, size=(40, 3)) @ cell
        pbc = (True, True, True)
    elif case == 'slab':
        cell = np.diag([8.0, 8.0, 30.0])
        z = rng.choice([13, 8], size=30)
        pos = rng.uniform(0, 1, size=(30, 3)) * np.array([8.0, 8.0, 6.0]) + np.array([0, 0, 12.0])
        pbc = (True, True, False)
    else:
        from sevenn_b200.neighbors import rocksalt_nacl
        pos, cell, z = rocksalt_nacl(2, 2, 2, sigma=0.05, seed=3)
        pbc = (True, True, True)
    kw = dict(vdw_cutoff=2500.0, cn_cutoff=900.0)                    # 26 A / 16 A: the oracle is O(N^2 images)
    ref = d3_reference(z, pos, cell, pbc, damping=damping, **kw)
    e, f, s = D3Engine(damping, 'pbe', **kw).compute(z, pos, cell, pbc)
    assert abs(e / ref['energy'] - 1.0) < 2e-6
    assert _rel(f, ref['forces']) < 2e-5
    sg = ref['sigma']
    assert _rel(s, [sg[0, 0], sg[1, 1], sg[2, 2], sg[0, 1], sg[0, 2], sg[1, 2]]) < 2e-5


def test_reference_named_entry_points():
    """pair_init ... pair_fin, called as sevenn/calculator.py:563-603 calls them (LAMMPS-style upper-triangular
    box, 1-based types)."""
    from oracle.d3_oracle import d3_reference
    from sevenn_b200.engine import load_library
    lib = load_library()
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
    rng = np.random.RandomState(5)
    cell = np.array([[7.0, 0.0, 0.0], [0.8, 6.5, 0.0], [0.4, -0.6, 8.0]])        # already lower-triangular rows = LAMMPS frame
    z = np.array([14, 8, 8, 14, 1, 1, 8, 14])
    pos = rng.uniform(0, 1, size=(8, 3)) @ cell
    uniq = list(dict.fromkeys(z.tolist()))
    types = np.ascontiguousarray([uniq.index(a) + 1 for a in z], dtype=np.int32)
    x = np.ascontiguousarray(pos, dtype=np.float64)
    nums = np.ascontiguousarray(uniq, dtype=np.int32)
    lo, hi = np.zeros(3), np.ascontiguousarray([cell[0, 0], cell[1, 1], cell[2, 2]])
    p = lib.pair_init()
    lib.pair_set_atom(p, len(z), len(uniq), types.ctypes.data, x.ctypes.data)
    lib.pair_set_domain(p, 1, 1, 1, lo.ctypes.data, hi.ctypes.data, cell[1, 0], cell[2, 0], cell[2, 1])
    lib.pair_run_settings(p, 2500.0, 900.0, b'damp_bj', b'pbe')
    lib.pair_run_coeff(p, nums.ctypes.data)
    lib.pair_run_compute(p)
    e = lib.pair_get_energy(p)
    f = np.ctypeslib.as_array(lib.pair_get_force(p), shape=(len(z) * 3,)).reshape(-1, 3).copy()
    s = np.array(lib.pair_get_stress(p).contents)
    lib.pair_fin(p)
    ref = d3_reference(z, pos, cell, vdw_cutoff=2500.0, cn_cutoff=900.0)
    assert abs(e / ref['energy'] - 1.0) < 2e-6
    assert _rel(f, ref['forces']) < 2e-5
    sg = ref['sigma']
    assert _rel(s, [sg[0, 0], sg[1, 1], sg[2, 2], sg[0, 1], sg[0, 2], sg[1, 2]]) < 2e-5


@pytest.mark.parametrize('cells,damping', [((2, 2, 2), 'damp_bj'), ((6, 6, 4), 'damp_bj'), ((5, 5, 5), 'damp_zero')])
def test_matches_compiled_reference(cells, damping):
    """The reference's own CUDA D3 at its default cutoffs on rocksalt NaCl (64 / 1152 / 1000 atoms): inputs and
    results stored in tests/golden/d3_reference_nacl.npz by tools/make_d3_golden.py.  The reference sums its
    lattice images in fp32 (see tests/test_d3_oracle.py), hence 1e-4 on the energy."""
    from sevenn_b200.d3 import D3Engine
    key = 'nacl_{}x{}x{}_{}'.format(*cells, damping)
    with np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), 'golden', 'd3_reference_nacl.npz')) as g:
        z, pos, cell = g[f'{key}_numbers'], g[f'{key}_positions'], g[f'{key}_cell']
        e_ref, f_ref, s_ref = float(g[f'{key}_energy']), g[f'{key}_forces'], g[f'{key}_sigma']
    e, f, s = D3Engine(damping, 'pbe').compute(z, pos, cell)
    assert abs(e / e_ref - 1.0) < 1e-4
    assert np.abs(f - f_ref).max() < 2e-6 + 1e-4 * np.abs(f_ref).max()
    assert _rel(s, s_ref) < 2e-4
