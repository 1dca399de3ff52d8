"""Schwarz screening of direct J/K against an element-wise bound from the oracle's tensor.

The engine drops a shell quartet when Q_AB Q_CD dmax < tau, with Q_AB the largest AO Schwarz factor of the pair and dmax the largest
|P_cart| of the densities screened together.  Every AO term it drops then has Q_ab Q_cd dmax < tau, so with the mask
M = [Q_ab Q_cd dmax < tau (1 + 1e-10)] on the oracle's normalised Cartesian tensor E (Q_ab = sqrt|(ab|ab)|):

    |J(tau) - J(0)|_ij <= sum_kl M_ij,kl |(ij|kl)| |P_kl| + slack_ij,     |K(tau) - K(0)|_ij <= sum_kl M_il,kj |(il|kj)| |P_kl| + slack_ij

slack_ij: the integer accumulation rounds each dropped term by at most 2^-61 and the two conversions to FP64 add a few ulp of |X(0)|.
With a transform U the engine screens P_cart = U^T P U and returns U X_cart U^T: the bound is |U| B(P_cart) |U|^T.  Both results come
from one engine (a work item's integer words do not depend on which other items run), so J(tau) - J(0) isolates the screening.

CPU: the host build of the engine (tests/host_emul/emul.cpp; pairQ, build_item_prefix and the exact test, shared with the device).
GPU: the shell engine with and without a transform, a density that reaches the Cartesian amplification of the pre-screen's margin, the
job-set cache across thresholds and density magnitudes, the per-component kernel and the provider's threshold."""
import ctypes
import os

import numpy as np
import pytest

from test_host_emul import LazyEmul
from test_kernel_variants import coverage_basis, jk_tolerance
from test_multi_device import provider_state  # noqa: F401  (fixture)
from test_spherical_fill import shell_blocks_U
from util import basis_objects, load_golden, oracle_basis

HERE = os.path.dirname(os.path.abspath(__file__))

TAUS = (1e-14, 1e-12, 1e-10, 1e-8, 1e-6)
ULP = 2.0 ** -53
FIX = 2.0 ** -61               # resolution of the low accumulator word (fixed_split)
NAMES = ["n2_ccpvtz", "coverage"]
# threshold from which the engine must drop quartets: the coverage basis spans a 1e5 and a 0.05 s exponent; N2/cc-pVTZ is compact and
# keeps every shell quartet up to 1e-6 (there the bound is checked, and a threshold that cannot drop anything must change no bit)
ENGAGES = {"coverage": 1e-10, "n2_ccpvtz": None}


# ---------------------------------------------------------------------------------------------------------------------------------
# cases and the bound
# ---------------------------------------------------------------------------------------------------------------------------------
_CASES = {}


def case(oracle, name):
    """Basis objects, FlatBasis, the oracle's Cartesian tensor E, its Schwarz factors Q (ncart x ncart), a transform U (nbf x ncart: the
    fixture's, or the solid-harmonic-like one of test_spherical_fill for the coverage basis), a recorded-like spherical density and Lmax."""
    if name not in _CASES:
        if name == "coverage":
            objs = coverage_basis()
            fb = oracle.FlatBasis.from_reference_objects(objs)
            U = shell_blocks_U(fb)
            P = None
        else:
            g = load_golden(name)
            objs, fb, U = basis_objects(g), oracle_basis(oracle, g), np.array(g["U"])
            P = np.array(g["P_final"])
        if P is None:                            # no SCF for the synthetic basis: the fixed density of the benchmarks
            from tuna_b200 import workloads as w
            P = w.fixed_density(U.shape[0])
        E = oracle.eri_fill(fb)
        n = fb.ncart
        Q = np.sqrt(np.abs(np.einsum("abab->ab", E)))
        _CASES[name] = dict(objs=objs, fb=fb, E=E, Q=Q, U=U, P_sph=P, n=n, lmax=int(np.asarray(fb.lmn).sum(axis=1).max()))
    return _CASES[name]


def stacks(c):
    """The density stacks of the Cartesian runs: the recorded density's Cartesian image, a seeded random symmetric O(1) stack of two,
    the same x 1e3 (the pre-screen's bound scales with it), and a non-symmetric stack (the plan's S / A split)."""
    n = c["n"]
    rng = np.random.default_rng(20261022)
    R = rng.standard_normal((2, n, n))
    R = (R + R.transpose(0, 2, 1)) / 2
    A = rng.standard_normal((2, n, n))
    return {"recorded": (c["U"].T @ c["P_sph"] @ c["U"])[None], "random": R, "random_x1e3": 1e3 * R, "nonsymmetric": A}


def run_stack(P):
    """The densities a direct build runs (plan_density, csrc/density_split.hpp): P, or S = (P + P^T) / 2 then A = (P - P^T) / 2."""
    if np.abs(P - P.transpose(0, 2, 1)).max() > 1e-15 * np.abs(P).max():
        return np.concatenate([(P + P.transpose(0, 2, 1)) / 2, (P - P.transpose(0, 2, 1)) / 2]), True
    return P, False


def density_passes(nrun, lmax, shell=True):
    """Mirror of direct_pass_densities (csrc/tuna_b200.cu): the run stack goes through the engine in passes small enough for the largest
    class to keep its J/K blocks in shared memory, and each pass is screened with the max |P_cart| of its own densities."""
    nd_max = 4
    if shell:
        nc = (lmax + 1) * (lmax + 2) // 2
        per_density = 4 * (nc + 4) ** 2 + 8 * nc * nc
        while nd_max > 1 and nd_max * per_density + 9000 > 27000:
            nd_max -= 1
    npass = -(-nrun // nd_max)
    per = -(-nrun // npass)
    return [list(range(d0, min(d0 + per, nrun))) for d0 in range(0, nrun, per)]


def masked_tensor(E, Q, tau, dmax):
    """|E| where the engine may drop the term: Q_ab Q_cd dmax < tau (1 + 1e-10), zero elsewhere."""
    n = Q.shape[0]
    drop = (np.multiply.outer(Q, Q) * dmax < tau * (1.0 + 1e-10)).reshape((n,) * 4)
    return np.where(drop, np.abs(E), 0.0)


def contract(W, X):
    """(sum_kl W_ijkl X_kl, sum_kl W_ilkj X_kl) for a stack X."""
    return np.einsum("ijkl,dkl->dij", W, X, optimize=True), np.einsum("ilkj,dkl->dij", W, X, optimize=True)


def screening_bound(c, P, tau, U=None, shell=True):
    """(B^J, B^K, dmax of every pass) for the caller's stack P in the caller's basis (U None: P is Cartesian).  A density of the run
    stack is screened with the dmax of its pass; when the S and A parts of a split stack share a pass, K's bound takes |P| itself."""
    E, Q = c["E"], c["Q"]
    R, split = run_stack(P)
    Rc = R if U is None else np.einsum("pa,dpq,qb->dab", U, R, U, optimize=True)
    nD = P.shape[0]
    passes = density_passes(len(R), c["lmax"], shell)
    dmax = np.empty(len(R))
    for p in passes:
        dmax[p] = np.abs(Rc[p]).max()
    W = {}
    for x in sorted(set(dmax)):
        W[x] = masked_tensor(E, Q, tau, x)
    BJ, BK = np.empty((nD,) + Rc.shape[1:]), np.empty((nD,) + Rc.shape[1:])
    for d in range(nD):
        BJ[d] = contract(W[dmax[d]], np.abs(Rc[d:d + 1]))[0][0]
        if split and dmax[d] == dmax[nD + d]:
            BK[d] = contract(W[dmax[d]], np.abs(Rc[d:d + 1] + Rc[nD + d:nD + d + 1]))[1][0]
        elif split:
            BK[d] = contract(W[dmax[d]], np.abs(Rc[d:d + 1]))[1][0] + contract(W[dmax[nD + d]], np.abs(Rc[nD + d:nD + d + 1]))[1][0]
        else:
            BK[d] = contract(W[dmax[d]], np.abs(Rc[d:d + 1]))[1][0]
    if U is not None:
        aU = np.abs(U)
        BJ, BK = aU @ BJ @ aU.T, aU @ BK @ aU.T
    return BJ, BK, sorted(set(dmax))


def fixed_slack(c, J0, K0, P, U=None):
    """Rounding of the integer accumulation: 2^-61 per dropped term (8 n^2 2^-61) and a few ulp of |X(0)| from the conversions.  With a
    transform, the two FP64 rotations of X(tau) and X(0) add up to 4 k ulp of |U| (sum |E| |P_cart|) |U|^T, k the most nonzeros in a row of U."""
    n = c["n"]
    if U is None:
        return 4 * ULP * np.abs(J0) + 8 * n * n * FIX, 4 * ULP * np.abs(K0) + 8 * n * n * FIX
    R, _ = run_stack(P)
    Rc = np.abs(np.einsum("pa,dpq,qb->dab", U, R, U, optimize=True))
    Rc = Rc[:P.shape[0]] + (Rc[P.shape[0]:] if len(Rc) > P.shape[0] else 0.0)
    k = int((U != 0).sum(axis=1).max())
    aU = np.abs(U)
    AJ, AK = contract(np.abs(c["E"]), Rc)
    rot = lambda A: aU @ (8 * n * n * FIX + 4 * k * ULP * A) @ aU.T
    return 4 * ULP * np.abs(J0) + rot(AJ), 4 * ULP * np.abs(K0) + rot(AK)


def check_bound(label, got, ref, bound, slack):
    """|got - ref| <= bound + slack element-wise.  Returns the tightness: the largest |got - ref| / bound where the bound exceeds the slack."""
    diff = np.abs(got - ref)
    lim = bound + slack
    bad = diff > lim
    assert not bad.any(), (f"{label}: {int(bad.sum())} elements outside the screening bound, worst excess "
                           f"{(diff - lim).max():.3e} (|diff| {diff[bad].max():.3e}, bound {bound[bad].max():.3e})")
    big = bound > slack
    return float((diff[big] / bound[big]).max()) if big.any() else 0.0


def print_report(rows):
    for label, value in rows:
        print(f"SCREENING {label}: {value}")


# ---------------------------------------------------------------------------------------------------------------------------------
# CPU: the margin of the pre-screen, and the host build of the engine
# ---------------------------------------------------------------------------------------------------------------------------------
def amplification(U):
    """Largest max|U^T P U| / max|P|: (max_a sum_p |U_pa|)^2, reached by P = s s^T with s_p = sign(U_pa*)."""
    return float(np.abs(U).sum(axis=0).max() ** 2)


def test_prescreen_margin_covers_the_cartesian_amplification(oracle):
    """The job lists are pre-screened with dens_bound = 1e3 max(1, max|P|), max|P| in the caller's basis, while the device screens with
    max|U^T P U|.  No quartet the device keeps is lost as long as max|U^T P U| <= 1e3 max|P|: true for every fixture's U and for the
    h-shell U of the coverage basis.  The worst-case density reaches the amplification exactly."""
    seen = {}
    for f in sorted(f for f in os.listdir(os.path.join(HERE, "golden")) if f.endswith(".npz")):
        g = np.load(os.path.join(HERE, "golden", f))
        if "U" in g.files:
            seen[f] = amplification(np.array(g["U"]))
    seen["coverage h-shell U"] = amplification(case(oracle, "coverage")["U"])
    assert len(seen) >= 8, seen
    for k, a in seen.items():
        assert a < 1e3, (k, a)
    for U in (case(oracle, "coverage")["U"], np.array(load_golden("n2_ccpvtz")["U"])):
        P = worst_case_density(U)
        assert np.abs(P).max() == 1.0
        assert np.isclose(np.abs(U.T @ P @ U).max(), amplification(U), rtol=1e-14)
    print(f"SCREENING amplification: {seen}")


def worst_case_density(U):
    a = int(np.argmax(np.abs(U).sum(axis=0)))
    s = np.where(U[:, a] < 0, -1.0, 1.0)
    return np.outer(s, s)


@pytest.fixture(scope="module")
def emul():
    return LazyEmul("")


def run_emul(emul, fb, P, tau):
    dp, ip, lp = ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int64)
    oz = np.ascontiguousarray(fb.origins[:, 2])
    lmn = np.ascontiguousarray(fb.lmn, dtype=np.int32)
    npr = np.ascontiguousarray(fb.nprim, dtype=np.int32)
    off = np.ascontiguousarray(fb.offsets, dtype=np.int64)
    ceff = np.ascontiguousarray(fb.coefs * fb.norms)
    P = np.ascontiguousarray(P)
    J, K, stats = np.zeros_like(P), np.zeros_like(P), np.zeros(8, dtype=np.int64)
    rc = emul.emul_jk_shell4(fb.ncart, oz.ctypes.data_as(dp), lmn.ctypes.data_as(ip), npr.ctypes.data_as(ip), off.ctypes.data_as(lp),
                             fb.exps.ctypes.data_as(dp), ceff.ctypes.data_as(dp), P.shape[0], P.ctypes.data_as(dp), J.ctypes.data_as(dp),
                             K.ctypes.data_as(dp), ctypes.c_double(tau), stats.ctypes.data_as(ctypes.POINTER(ctypes.c_longlong)))
    assert rc == 0
    return J, K, stats


@pytest.mark.parametrize("stack", ["recorded", "random", "random_x1e3"])
@pytest.mark.parametrize("name", NAMES)
def test_host_engine_screening_bound(emul, oracle, name, stack):
    """The host build of the engine along the threshold ladder: J(tau) - J(0) and K(tau) - K(0) within the bound; the pre-screen's kept
    items never grow, the quartets screened in all (cut by the pre-screen or dropped by the exact test) never shrink, and from 1e-10 up
    the exact test drops quartets and the result changes."""
    c = case(oracle, name)
    P = stacks(c)[stack]
    J0, K0, s0 = run_emul(emul, c["fb"], P, 0.0)
    assert s0[3] == 0
    report, kept, screened = [], [int(s0[2])], [0]
    for tau in TAUS:
        J, K, st = run_emul(emul, c["fb"], P, tau)
        BJ, BK, dm = screening_bound(c, P, tau)
        assert len(dm) == 1                     # one pass on the host
        sJ, sK = fixed_slack(c, J0, K0, P)
        rj = check_bound(f"host {name} {stack} tau {tau:g} J", J, J0, BJ, sJ)
        rk = check_bound(f"host {name} {stack} tau {tau:g} K", K, K0, BK, sK)
        kept.append(int(st[2]))
        screened.append(int(s0[2] - st[2] + st[3]))
        report.append((f"host {name} {stack} tau {tau:g} [prescreen cut, exact-test dropped, max ratio J, K]",
                       [int(s0[2] - st[2]), int(st[3]), round(rj, 4), round(rk, 4)]))
        if ENGAGES[name] is not None and tau >= ENGAGES[name]:
            assert st[3] > 0, (tau, st)
            assert not np.array_equal(J, J0) and not np.array_equal(K, K0), tau
        if not BJ.any() and not BK.any():
            assert np.array_equal(J, J0) and np.array_equal(K, K0) and st[2] == s0[2] and st[3] == 0, tau
    assert all(a >= b for a, b in zip(kept, kept[1:])), kept
    assert all(a <= b for a, b in zip(screened, screened[1:])), screened
    if ENGAGES[name] is not None:
        assert screened[-1] > screened[1], screened
    print_report(report)


# ---------------------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------------------
def make_ctx(c, U=None):
    import tuna_b200
    from tuna_b200.basis import flatten
    ctx = tuna_b200.Context(0)
    ctx.set_basis(*flatten(c["objs"]))
    ctx.set_transform(np.eye(c["n"]) if U is None else U)
    return ctx


def oracle_jk(oracle, c, P, U=None):
    Pc = P if U is None else np.einsum("pa,dpq,qb->dab", U, P, U, optimize=True)
    J = np.stack([oracle.coulomb(p, c["E"]) for p in Pc])
    K = np.stack([oracle.exchange(p, c["E"]) for p in Pc])
    if U is not None:
        J, K = U @ J @ U.T, U @ K @ U.T
    return J, K


def ladder(oracle, ctx, c, P, label, engages, U=None, shell=True, taus=TAUS, counts=True):
    """J/K along the ladder against the same context's tau = 0 build (the bound) and the oracle (the bound plus the suite's tolerance)."""
    J0, K0 = ctx.jk_direct(P, 0.0)
    if counts:
        surviving = ctx.counts()["surviving_quartets"]
        assert ctx.counts()["evaluated_last_direct"] == surviving
        evaluated = [surviving]
    Jr, Kr = oracle_jk(oracle, c, P, U)
    tol = jk_tolerance(Kr)
    report = []
    for tau in taus:
        J, K = ctx.jk_direct(P, tau)
        BJ, BK, dm = screening_bound(c, P, tau, U, shell)
        if shell:
            sJ, sK = fixed_slack(c, J0, K0, P, U)
        else:                                    # FP64 atomics: the per-element rounding bound of a sum of the terms
            Rc = np.abs(run_stack(P)[0])
            Rc = Rc[:P.shape[0]] + (Rc[P.shape[0]:] if len(Rc) > P.shape[0] else 0.0)
            AJ, AK = contract(np.abs(c["E"]), Rc)
            sJ, sK = 64 * ULP * AJ, 64 * ULP * AK
        rj = check_bound(f"{label} tau {tau:g} J", J, J0, BJ, sJ)
        rk = check_bound(f"{label} tau {tau:g} K", K, K0, BK, sK)
        for what, got, ref, B in (("J", J, Jr, BJ), ("K", K, Kr, BK)):
            err = np.abs(got - ref) - B
            assert err.max() <= tol, f"{label} tau {tau:g} {what} vs oracle: {err.max():.3e} beyond bound, tolerance {tol:.1e}"
        row = [len(dm), round(rj, 4), round(rk, 4)]
        if counts:
            ev = ctx.counts()["evaluated_last_direct"]
            row.insert(0, surviving - ev)
            assert ev <= evaluated[-1], (tau, ev, evaluated)
            if engages is not None and tau >= engages:
                assert ev < surviving, (tau, ev, surviving)
            evaluated.append(ev)
        if engages is not None and tau >= engages:
            assert not np.array_equal(J, J0) or not np.array_equal(K, K0), tau
        if shell and not BJ.any() and not BK.any():             # integer accumulation: nothing dropped, nothing changed
            assert np.array_equal(J, J0) and np.array_equal(K, K0), tau
        report.append((f"{label} tau {tau:g} [{'screened quartets, ' if counts else ''}passes, max ratio J, K]", row))
    print_report(report)


@pytest.mark.gpu
@pytest.mark.parametrize("stack", ["recorded", "random", "random_x1e3", "nonsymmetric"])
@pytest.mark.parametrize("name", NAMES)
def test_shell_engine_screening_bound(oracle, name, stack):
    """The shell engine in the Cartesian basis (U = 1), every stack along the ladder; evaluated quartets never grow along it and fall
    below the surviving count from 1e-10 up."""
    c = case(oracle, name)
    ctx = make_ctx(c)
    ladder(oracle, ctx, c, stacks(c)[stack], f"shell {name} {stack}", ENGAGES[name])
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", NAMES)
def test_shell_engine_screening_bound_with_transform(oracle, name):
    """With the fixture's U (N2/cc-pVTZ) and the h-shell U (coverage basis): the bound |U| B(U^T P U) |U|^T for the recorded density,
    a random symmetric stack, the same x 1e3, and at tau = 1e-10 the worst-case density for the pre-screen's margin (max|P| = 1,
    max|P_cart| = the amplification)."""
    c = case(oracle, name)
    U = c["U"]
    nbf = U.shape[0]
    rng = np.random.default_rng(7)
    R = rng.standard_normal((2, nbf, nbf))
    R = (R + R.transpose(0, 2, 1)) / 2
    ctx = make_ctx(c, U)
    for label, P in (("recorded", c["P_sph"][None]), ("random", R), ("random_x1e3", 1e3 * R)):
        ladder(oracle, ctx, c, P, f"shell {name} U {label}", ENGAGES[name], U)
    W = worst_case_density(U)[None]
    assert np.isclose(np.abs(np.einsum("pa,dpq,qb->dab", U, W, U)).max(), amplification(U), rtol=1e-14)
    ladder(oracle, ctx, c, W, f"shell {name} U worst case", ENGAGES[name], U, taus=(1e-10,))
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", NAMES)
def test_job_sets_across_thresholds_and_densities(oracle, name):
    """One context through the ladder up and back down, with a small, a x 1e3 and a small density in turn: every result bitwise equal to
    a fresh context's for the same (P, tau).  A cached job set pre-screened for a larger density keeps only extra items the device
    test drops; one pre-screened for a smaller density would lose quartets."""
    c = case(oracle, name)
    P = stacks(c)["random"]
    dens = [P, 1e3 * P, P]
    ctx = make_ctx(c)
    for i, tau in enumerate(TAUS + TAUS[::-1]):
        Q = dens[i % 3]
        got = ctx.jk_direct(Q, tau)
        fresh = make_ctx(c)
        ref = fresh.jk_direct(Q, tau)
        for a, b, what in zip(got, ref, "JK"):
            assert np.array_equal(a, b), f"step {i} tau {tau:g} x{np.abs(Q).max():.0f} {what}: max diff {np.abs(a - b).max():.3e}"
        assert ctx.counts()["evaluated_last_direct"] == fresh.counts()["evaluated_last_direct"], (i, tau)
        fresh.close()
    ctx.close()


@pytest.mark.gpu
@pytest.mark.parametrize("stack", ["random", "nonsymmetric"])
@pytest.mark.parametrize("name", NAMES)
def test_per_component_kernel_screening_bound(oracle, name, stack, monkeypatch):
    """k_jk_direct (TUNA_B200_DIRECT_ENGINE=generic) with its AO-level test Q_ab Q_cd dmax < tau: the same bound, with the FP64
    rounding bound 64 ulp sum |E| |P| as the slack."""
    monkeypatch.setenv("TUNA_B200_DIRECT_ENGINE", "generic")
    c = case(oracle, name)
    ctx = make_ctx(c)
    ladder(oracle, ctx, c, stacks(c)[stack], f"generic {name} {stack}", ENGAGES[name], shell=False, counts=False)
    ctx.close()


@pytest.mark.gpu
def test_provider_threshold(provider_state):
    """configure(tau=1e-10): direct J/K through the reference's signatures is bitwise Context.jk_direct(P, 1e-10)."""
    import tuna_b200
    from types import SimpleNamespace
    from util import context_for
    g = load_golden("n2_ccpvtz")
    n, U = int(g["ncart"]), np.array(g["U"])
    tuna_b200.configure(mode="direct", tau=1e-10, devices=[0])
    calc = SimpleNamespace(cartesian_harmonics=False, number_of_threads=4, method=SimpleNamespace(method_base="HF"))
    mol = SimpleNamespace(spherical_harmonic_transformation_matrix=U)
    h = tuna_b200.calculate_two_electron_integrals(n, basis_objects(g), calc)
    one = np.eye(n)
    eri = tuna_b200.transform_to_spherical_harmonics(one, one, one, np.stack([one] * 3), np.stack([one] * 3), h, mol, calc, True)[5]
    P = np.array(g["P_final"])
    J, K = tuna_b200.calculate_coulomb_matrix(P, eri), tuna_b200.calculate_exchange_matrix(P, eri)
    ctx = context_for(g)
    ctx.set_transform(U)
    Jr, Kr = ctx.jk_direct(P, 1e-10)
    assert np.array_equal(J, Jr) and np.array_equal(K, Kr)
