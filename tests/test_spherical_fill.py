"""The spherical ERI tensor filled straight from the shell-quartet engine (tuna_eri_fill_sph): no Cartesian tensor on the device.

CPU: the per-quartet rotation (shell4_fill_sph) and the block-diagonal check of U (build_sph_shells) compiled for the host on top of the
fill-mode harness, against the oracle's Cartesian tensor rotated with NumPy.  GPU: eri_fill_sph against eri_fill_cart + eri_cart_to_sph,
the fallbacks (dense U, generic engine), stored J/K from the new tensor and the provider's stored-mode SCF."""
import ctypes
import os
import subprocess
import sys
from types import SimpleNamespace

import numpy as np
import pytest

from util import basis_objects, context_for, load_golden, oracle_basis

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


def _pg(lmn):
    """x/y parity code of each Cartesian component (ShellTab::pg)."""
    lmn = np.asarray(lmn)
    return (lmn[:, 0] & 1) * 2 + (lmn[:, 1] & 1)


def coverage_fb(oracle):
    """The synthetic two-centre basis with every shell type from s to h (contracted s-f shells, one uncontracted g and h)."""
    from tuna_b200 import workloads as w
    from tuna_b200.basis import from_arrays
    a = [(0, [120.0, 25.0, 7.0, 2.1, 0.6], [0.02, 0.1, 0.3, 0.45, 0.3]), (1, [18.0, 4.2, 1.2, 0.35], [0.1, 0.35, 0.5, 0.3]),
         (2, [6.0, 2.0, 0.8, 0.3], [0.15, 0.4, 0.45, 0.2]), (3, [9.0, 4.0, 1.8, 0.8], [0.05, 0.3, 0.35, 0.25]), (5, [1.1], [1.0])]
    b = [(0, [80.0, 15.0, 3.5, 0.9], [0.05, 0.25, 0.5, 0.35]), (1, [25.0, 6.0, 1.8], [0.2, 0.4, 0.35]), (4, [1.2], [1.0]), (0, [0.05], [1.0])]
    sh = w.shells_to_components([a, b], [0.0, 1.6])
    objs = from_arrays(sh["origins"], sh["lmn"], sh["nprim"], sh["exps"], sh["raw_coefs"])
    return oracle.FlatBasis.from_reference_objects(objs), objs


def shell_blocks_U(fb, seed=5):
    """A rotation with the structure of real solid harmonics: per shell of angular momentum L, 2L+1 rows, each a random combination of
    the shell's components of one x/y parity (the parity of component k for row k).  Components of a shell share centre, L and exponents."""
    rng = np.random.default_rng(seed)
    lmn = np.asarray(fb.lmn)
    L = lmn.sum(axis=1)
    pg = _pg(lmn)
    key = [(float(fb.origins[i, 2]), int(L[i]), tuple(np.asarray(fb.exps)[fb.offsets[i]:fb.offsets[i] + fb.nprim[i]])) for i in range(fb.ncart)]
    shells = {}
    for i, k in enumerate(key):
        shells.setdefault(k, []).append(i)
    rows = []
    for k, comps in shells.items():
        comps = sorted(comps, key=lambda i: (-lmn[i, 0], -lmn[i, 1]))
        for r in range(2 * k[1] + 1):
            u = np.zeros(fb.ncart)
            same = [i for i in comps if pg[i] == pg[comps[r]]]
            u[same] = rng.uniform(-1.0, 1.0, len(same))
            rows.append(u)
    return np.array(rows)


def sph_parity(U, lmn):
    pg = _pg(lmn)
    return np.array([pg[np.nonzero(row)[0][0]] for row in U])


def parity_mask(par):
    return (par[:, None, None, None] ^ par[None, :, None, None] ^ par[None, None, :, None] ^ par[None, None, None, :]) != 0


def check_tensor(got, ref, par):
    """Within 1e-13 max(1, max|ERI|) of the reference, exact parity zeros, one value in all eight images."""
    assert np.isfinite(got).all()
    assert np.abs(got - ref).max() <= 1e-13 * max(1.0, np.abs(ref).max()), np.abs(got - ref).max()
    assert (got[parity_mask(par)] == 0.0).all()
    for perm in ((1, 0, 2, 3), (0, 1, 3, 2), (2, 3, 0, 1)):
        assert np.array_equal(got, got.transpose(perm))


# ---------------------------------------------------------------------------------------------------------------------
# CPU: host build of the per-quartet rotation and of the block-diagonal check
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def emul_sph(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("emul_sph") / "libemul_sph.so")
    subprocess.run(["g++", "-O2", "-fopenmp", "-fPIC", "-shared", "-x", "c++", "-o", so, os.path.join(HERE, "host_emul", "emul_sph.cpp"), "-lm"], check=True)
    return ctypes.CDLL(so)


def _basis_args(fb):
    dp, ip, lp = ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int64)
    keep = [np.ascontiguousarray(fb.origins[:, 2]), np.ascontiguousarray(fb.lmn, dtype=np.int32), np.ascontiguousarray(fb.nprim, dtype=np.int32),
            np.ascontiguousarray(fb.offsets, dtype=np.int64), np.ascontiguousarray(fb.exps, dtype=np.float64),
            np.ascontiguousarray(fb.coefs * fb.norms)]
    types = [dp, ip, ip, lp, dp, dp]
    return keep, [a.ctypes.data_as(t) for a, t in zip(keep, types)]


def _blocks_ok(emul_sph, fb, U):
    keep, args = _basis_args(fb)
    U = np.ascontiguousarray(U, dtype=np.float64)
    return emul_sph.emul_sph_blocks_ok(fb.ncart, *args, U.shape[0], U.ctypes.data_as(ctypes.POINTER(ctypes.c_double)))


def test_block_diagonal_check(emul_sph, oracle):
    for name in ("n2_ccpvtz", "ne2_uhf_ccpvqz", "co_b3lyp_ccpvtz"):
        g = load_golden(name)
        assert _blocks_ok(emul_sph, oracle_basis(oracle, g), g["U"]) == 1, name
    g = load_golden("n2_ccpvtz")
    fb = oracle_basis(oracle, g)
    rng = np.random.default_rng(11)
    assert _blocks_ok(emul_sph, fb, rng.standard_normal(np.asarray(g["U"]).shape)) == 0
    U = np.array(g["U"])
    j = int(np.nonzero(U[0])[0][0])
    U[0, (j + 1) % fb.ncart if _pg(fb.lmn)[(j + 1) % fb.ncart] != _pg(fb.lmn)[j] else (j + 2) % fb.ncart] = 0.3      # one entry outside the shell
    assert _blocks_ok(emul_sph, fb, U) == 0
    cfb, _ = coverage_fb(oracle)
    assert _blocks_ok(emul_sph, cfb, shell_blocks_U(cfb)) == 1


@pytest.mark.parametrize("name", ["n2_ccpvtz", "coverage"])
def test_fill_sph_host_build_vs_rotated_oracle(emul_sph, oracle, name):
    if name == "coverage":
        fb, _ = coverage_fb(oracle)
        U = shell_blocks_U(fb)
    else:
        g = load_golden(name)
        fb, U = oracle_basis(oracle, g), np.array(g["U"])
    nbf = U.shape[0]
    ref = oracle.cart_to_sph_eri(oracle.eri_fill(fb), U)
    out = np.full((nbf,) * 4, np.nan)
    keep, args = _basis_args(fb)
    Uc = np.ascontiguousarray(U)
    rc = emul_sph.emul_fill_sph(fb.ncart, *args, nbf, Uc.ctypes.data_as(ctypes.POINTER(ctypes.c_double)),
                                out.ctypes.data_as(ctypes.POINTER(ctypes.c_double)))
    assert rc == 0
    check_tensor(out, ref, sph_parity(U, fb.lmn))


# ---------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def tb():
    import tuna_b200
    return tuna_b200


def _gpu_case(name, oracle):
    import tuna_b200
    from tuna_b200.basis import flatten
    if name == "coverage":
        fb, objs = coverage_fb(oracle)
        U = shell_blocks_U(fb)
    else:
        g = load_golden(name)
        objs, U = basis_objects(g), np.array(g["U"])
        fb = oracle_basis(oracle, g)

    def make():
        ctx = tuna_b200.Context(0)
        ctx.set_basis(*flatten(objs))
        ctx.set_transform(U)
        return ctx
    return make, U, fb


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["n2_ccpvtz", "ne2_uhf_ccpvqz", "coverage"])
def test_fill_sph_matches_two_step_path(tb, oracle, name):
    make, U, fb = _gpu_case(name, oracle)
    ctx = make()
    ctx.eri_fill_cart()
    ctx.eri_cart_to_sph()
    ref = ctx.eri_download(1)
    ctx.eri_fill_sph()
    got = ctx.eri_download(1)
    check_tensor(got, ref, sph_parity(U, fb.lmn))
    with pytest.raises(Exception):
        ctx.eri_download(0)                  # no Cartesian tensor was made
    ctx2 = make()
    ctx2.eri_fill_sph()
    assert np.array_equal(ctx2.eri_download(1), got)
    assert ctx2.last_kernel_ms(0) > 0.0


@pytest.mark.gpu
def test_fill_sph_dense_U_is_the_two_step_path(tb, oracle):
    g = load_golden("n2_ccpvtz")
    rng = np.random.default_rng(3)
    U = 0.1 * rng.standard_normal(np.asarray(g["U"]).shape)
    ctx = context_for(g)
    ctx.set_transform(U)
    ctx.eri_fill_cart()
    ctx.eri_cart_to_sph()
    ref = ctx.eri_download(1)
    ctx.eri_fill_sph()
    assert np.array_equal(ctx.eri_download(1), ref)


_GENERIC_CHILD = """
import sys, numpy as np
sys.path.insert(0, {root!r}); sys.path.insert(0, {tests!r})
from util import context_for, load_golden
g = load_golden("n2_ccpvtz")
a = context_for(g); a.set_transform(g["U"]); a.eri_fill_cart(); a.eri_cart_to_sph()
b = context_for(g); b.set_transform(g["U"]); b.eri_fill_sph()
assert np.array_equal(a.eri_download(1), b.eri_download(1))
print("bitwise-equal")
"""


@pytest.mark.gpu
def test_fill_sph_generic_engine_is_the_two_step_path(tb):
    env = dict(os.environ, TUNA_B200_DIRECT_ENGINE="generic")
    r = subprocess.run([sys.executable, "-c", _GENERIC_CHILD.format(root=ROOT, tests=HERE)], env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "bitwise-equal" in r.stdout, r.stdout + r.stderr


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["n2_ccpvtz", "ne2_uhf_ccpvqz"])
def test_stored_jk_from_the_spherical_fill(tb, name):
    g = load_golden(name)
    ctx = context_for(g)
    ctx.set_transform(g["U"])
    ctx.eri_fill_sph()
    P = tb.workloads.fixed_density(int(g["nbf"]))
    J, K = ctx.jk_stored(P)
    assert np.abs(J - g["Jfix"]).max() < 1e-11 * max(1.0, np.abs(g["Jfix"]).max())
    assert np.abs(K - g["Kfix"]).max() < 1e-11 * max(1.0, np.abs(g["Kfix"]).max())
    for k in sorted(k for k in g.files if k.startswith("seq") and k.endswith("_P")):
        J, K = ctx.jk_stored(g[k])
        assert np.abs((J if k.split("_")[2] == "J" else K) - g[k[:-2] + "_out"]).max() < 1e-11, k


def _provider_handles(tb, g):
    n = int(g["ncart"])
    cart = tb.calculate_two_electron_integrals(n, basis_objects(g), None)
    z, z3 = np.zeros((n, n)), np.zeros((3, n, n))
    molecule = SimpleNamespace(spherical_harmonic_transformation_matrix=np.array(g["U"]))
    return cart, lambda: tb.transform_to_spherical_harmonics(z, z, z, z3, z3, cart, molecule, None, True)[5]


@pytest.mark.gpu
def test_provider_stored_scf_through_the_spherical_fill(tb):
    from oracle import scf_oracle
    g = load_golden("ne2_uhf_ccpvqz")
    tb.configure(mode="stored")
    try:
        cart, transform = _provider_handles(tb, g)
        assert cart.pending_fill
        eri = transform()
        assert not cart.pending_fill and eri.ctx.n_stored == int(g["nbf"])
        with pytest.raises(Exception):
            eri.ctx.eri_download(0)          # filled in the spherical basis: the Cartesian tensor never existed
        calls = []

        def jk(P):
            calls.append(1)
            return tb.calculate_coulomb_matrix(P, eri), tb.calculate_exchange_matrix(P, eri)
        energy, iterations, _ = scf_oracle.run_scf(jk, g)
        assert abs(energy - float(g["energy"])) < 1e-10, (energy, float(g["energy"]))
        assert iterations == int(g["n_iterations"])
    finally:
        tb.configure(mode="auto")


@pytest.mark.gpu
def test_provider_cartesian_handle_touched_before_the_transform(tb, oracle):
    g = load_golden("n2_ccpvtz")
    tb.configure(mode="stored")
    try:
        cart, transform = _provider_handles(tb, g)
        E = np.asarray(cart)                   # the Cartesian tensor, filled on first touch
        assert not cart.pending_fill
        ref = oracle.eri_fill(oracle_basis(oracle, g))
        assert np.abs(E - ref).max() <= 1e-12 * max(1.0, np.abs(ref).max())
        eri = transform()
        Es = np.asarray(eri)
        assert np.abs(Es - oracle.cart_to_sph_eri(ref, np.array(g["U"]))).max() <= 1e-12 * max(1.0, np.abs(ref).max())
    finally:
        tb.configure(mode="auto")
