"""One-electron integrals (SURVEY.md 8f-3): overlap, kinetic energy, nuclear attraction, dipole, diagonal quadrupole and the
cross-basis overlap (tuna_integral.pyx:282-912).

`not gpu`: (i) the C oracle against the reference's own compiled engine (oracle/_ref) on every committed configuration,
(ii) the kernel math (tuna_b200/csrc/oneel_core.cuh, `__host__ __device__`) compiled for the CPU against the oracle.
The GPU tests of this path live in tests/test_zz_fullsize.py (they were written after the round's GPU budget was spent).
Tolerance: 1e-12 absolute, 1e-13 relative above 10 (kinetic / nuclear matrix elements of tight functions reach 1e3)."""
import ctypes
import os
import subprocess
from types import SimpleNamespace

import numpy as np
import pytest

from util import load_golden, oracle_basis

HERE = os.path.dirname(os.path.abspath(__file__))
CHARGES = {"h2_631g": (1, 1), "n2_ccpvtz": (7, 7), "co_b3lyp_ccpvtz": (6, 8), "ne2_uhf_ccpvqz": (10, 10), "et100": (7, 7)}
NAMES = ("S", "T", "V", "D", "Q")


def molecule_inputs(fb, name):
    zs = np.array(sorted(set(fb.origins[:, 2].tolist())))
    ch = np.array(CHARGES[name], dtype=np.float64)
    origin = np.array([0.0, 0.0, float((zs * ch).sum() / ch.sum())])        # on the axis, like molecule.centre_of_mass (tuna_kernel.py:289-316)
    return zs, ch, origin


def close(got, ref, what):
    ref = np.asarray(ref)
    bad = np.abs(np.asarray(got) - ref) > np.maximum(1e-12, 1e-13 * np.abs(ref))
    assert not bad.any(), f"{what}: {int(bad.sum())} elements out of tolerance, max abs diff {np.abs(np.asarray(got) - ref).max():.2e}"


def sub_basis(oracle, fb, idx):
    off = fb.offsets
    sel = np.concatenate([np.arange(off[i], off[i] + fb.nprim[i]) for i in idx])
    return oracle.FlatBasis(fb.origins[idx], fb.lmn[idx], fb.nprim[idx], fb.exps[sel], fb.coefs[sel], fb.norms[sel])


@pytest.mark.parametrize("name", list(CHARGES))
def test_oracle_vs_compiled_reference(oracle, name):
    eng = oracle.reference_engine()
    if eng is None:
        pytest.skip("oracle/_ref not built")
    g = load_golden(name)
    fb = oracle_basis(oracle, g)
    zs, ch, origin = molecule_inputs(fb, name)
    atoms = [SimpleNamespace(origin=np.array([0.0, 0.0, z]), charge=float(c)) for z, c in zip(zs, ch)]
    bfs = oracle.reference_basis_objects(fb)
    ref = eng.calculate_one_electron_integrals(fb.ncart, bfs, len(atoms), atoms, origin, 4)
    got = oracle.one_electron(fb, zs, ch, origin)
    for nm, a, b in zip(NAMES, got, ref):
        close(a, b, f"{name} {nm}")
    # the overlap matrix the reference's own SCF used (fixture) is the spherical image of S
    U = np.array(g["U"])
    assert np.abs(U @ got[0] @ U.T - np.array(g["S"])).max() < 1e-12
    assert np.abs(U @ got[1] @ U.T - np.array(g["T"])).max() < 1e-11 and np.abs(U @ got[2] @ U.T - np.array(g["V_NE"])).max() < 1e-11
    idx = np.arange(0, fb.ncart, 3)
    sub = sub_basis(oracle, fb, idx)
    refc = np.asarray(eng.calculate_cross_basis_overlap_matrix(fb.ncart, sub.ncart, bfs, oracle.reference_basis_objects(sub), 4))
    close(oracle.cross_overlap(fb, sub), refc, f"{name} S_cross")


@pytest.mark.parametrize("name", list(CHARGES))
def test_oracle_vs_reference_scf_matrices(oracle, name):
    """The spherical images of S, T and V_NE against the matrices the reference's own SCF used (fixtures), without the reference tree."""
    g = load_golden(name)
    fb = oracle_basis(oracle, g)
    S, T, V = oracle.one_electron(fb, *molecule_inputs(fb, name))[:3]
    U = np.array(g["U"])
    assert np.abs(U @ S @ U.T - np.array(g["S"])).max() < 1e-12
    assert np.abs(U @ T @ U.T - np.array(g["T"])).max() < 1e-11 and np.abs(U @ V @ U.T - np.array(g["V_NE"])).max() < 1e-11


@pytest.fixture(scope="module")
def emul():
    so = os.path.join(HERE, "host_emul", "libemul_oneel.so")
    subprocess.run(["g++", "-O2", "-fopenmp", "-fPIC", "-shared", "-x", "c++", "-o", so, os.path.join(HERE, "host_emul", "emul.cpp"), "-lm"], check=True)
    return ctypes.CDLL(so)


def c_args(fb):
    dp, ip, lp = ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int64)
    keep = (np.ascontiguousarray(fb.origins[:, 2]), np.ascontiguousarray(fb.lmn, dtype=np.int32), np.ascontiguousarray(fb.nprim, dtype=np.int32),
            np.ascontiguousarray(fb.offsets, dtype=np.int64), np.ascontiguousarray(fb.exps), np.ascontiguousarray(fb.coefs * fb.norms))
    return keep, [keep[0].ctypes.data_as(dp), keep[1].ctypes.data_as(ip), keep[2].ctypes.data_as(ip), keep[3].ctypes.data_as(lp),
                  keep[4].ctypes.data_as(dp), keep[5].ctypes.data_as(dp)]


@pytest.mark.parametrize("name", ["h2_631g", "n2_ccpvtz", "ne2_uhf_ccpvqz", "et100", "h_shells"])
def test_kernel_math_vs_oracle(emul, oracle, name):
    dp = ctypes.POINTER(ctypes.c_double)
    if name == "h_shells":          # every shell type up to H on both centres, tight and diffuse, off-axis electric origin
        from tuna_b200 import workloads as w
        from tuna_b200.basis import from_arrays
        sa = [(0, [2.1e5], [1.0]), (1, [0.9], [1.0]), (5, [6.5], [1.0]), (3, [1.0, 0.4], [0.6, 0.5])]
        sb = [(2, [0.8], [1.0]), (4, [1.2], [1.0]), (5, [1.0], [1.0]), (0, [0.1], [1.0])]
        b = w.shells_to_components([sa, sb], [0.0, 2.0787])
        fb = oracle.FlatBasis.from_reference_objects(from_arrays(b["origins"], b["lmn"], b["nprim"], b["exps"], b["raw_coefs"]))
        zs, ch, origin = np.array([0.0, 2.0787]), np.array([7.0, 8.0]), np.array([0.1, -0.2, 0.77])
    else:
        fb = oracle_basis(oracle, load_golden(name))
        zs, ch, origin = molecule_inputs(fb, name)
    n = fb.ncart
    ref = oracle.one_electron(fb, zs, ch, origin)
    out = [np.empty((n, n)), np.empty((n, n)), np.empty((n, n)), np.empty((3, n, n)), np.empty((3, n, n))]
    keep, a = c_args(fb)
    rc = emul.emul_one_electron(n, *a, len(zs), zs.ctypes.data_as(dp), ch.ctypes.data_as(dp), origin.ctypes.data_as(dp), *[x.ctypes.data_as(dp) for x in out])
    assert rc == 0
    for nm, x, y in zip(NAMES, out, ref):
        close(x, y, f"{name} {nm}")
    assert np.array_equal(out[0], out[0].T) and np.array_equal(out[2], out[2].T)
    idx = np.arange(1, n, 4)
    sub = sub_basis(oracle, fb, idx)
    S12 = np.empty((n, sub.ncart))
    keep2, a2 = c_args(sub)
    assert emul.emul_cross_overlap(n, *a, sub.ncart, *a2, S12.ctypes.data_as(dp)) == 0
    close(S12, oracle.cross_overlap(fb, sub), f"{name} S_cross")
    close(S12, out[0][:, idx], f"{name} S_cross vs S columns")
