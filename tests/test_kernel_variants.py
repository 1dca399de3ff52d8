"""Every J/K kernel variant and launch configuration against the oracle, on the GPU.

Direct engine: each knob configuration of the launch rules (INTEGRATION.md section 5) runs in its own child process
(tests/variant_gpu_case.py) because several knobs are read once per process and job sets are cached per context.  The parent
compares J/K of a synthetic s-h coverage basis and of N2/cc-pVTZ with the oracle's dense tensor, checks that shard partials
sum to the whole and that the engine's fill mode reproduces the oracle's tensor, and asserts from the job tables the children
dump that every compiled k_shell4_one / k_shell4_multi instantiation ran at least once.

Stored mode: every (kernel, density count) cell that tuna_jk_stored_dev can dispatch to, and the TMA kernel at tile, stage and
grid geometries off their defaults, on uploaded random tensors against np.einsum with a per-element rounding bound."""
import csv
import glob
import json
import os
import subprocess
import sys

import numpy as np
import pytest

from util import context_for, eri_tolerance, load_golden, oracle_basis

pytestmark = pytest.mark.gpu

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)


# ---------------------------------------------------------------------------------------------------------------------
# coverage basis: every L from 0 to 5 on two centres; contracted s-f shells of 4-6 primitives (nppAB * nppCD > 16, so the bra and
# the ket split engage), one uncontracted g and h, a diffuse and a very tight s
# ---------------------------------------------------------------------------------------------------------------------
def coverage_shells(with_h=True):
    a = [(0, [120.0, 25.0, 7.0, 2.1, 0.6], [0.02, 0.1, 0.3, 0.45, 0.3]),
         (1, [18.0, 4.2, 1.2, 0.35], [0.1, 0.35, 0.5, 0.3]),
         (2, [6.0, 2.0, 0.8, 0.3], [0.15, 0.4, 0.45, 0.2]),
         (3, [9.0, 4.0, 1.8, 0.8, 0.4, 0.18], [0.05, 0.15, 0.3, 0.35, 0.25, 0.1]),
         (0, [1.0e5], [1.0])]
    if with_h:
        a.insert(4, (5, [1.1], [1.0]))
    b = [(0, [80.0, 15.0, 3.5, 0.9], [0.05, 0.25, 0.5, 0.35]),
         (1, [25.0, 6.0, 1.8, 0.6, 0.2], [0.05, 0.2, 0.4, 0.35, 0.15]),
         (2, [5.0, 1.9, 0.7, 0.3, 0.12], [0.1, 0.3, 0.4, 0.3, 0.1]),
         (3, [4.0, 1.5, 0.6, 0.25], [0.2, 0.4, 0.4, 0.15]),
         (4, [1.2], [1.0]),
         (0, [0.05], [1.0])]
    return [a, b], [0.0, 1.6]


def coverage_basis(with_h=True):
    """list[Basis] of the coverage basis (with_h=False: the same without the h shell, so that four densities fit one pass)."""
    from tuna_b200 import workloads as w
    from tuna_b200.basis import from_arrays
    shells, z = coverage_shells(with_h)
    b = w.shells_to_components(shells, z)
    return from_arrays(b["origins"], b["lmn"], b["nprim"], b["exps"], b["raw_coefs"])


def densities(n, seed=20261020):
    """Two random symmetric densities and one non-symmetric density."""
    rng = np.random.default_rng(seed)
    P = rng.standard_normal((3, n, n))
    P[:2] = (P[:2] + P[:2].transpose(0, 2, 1)) / 2
    return P


def jk_tolerance(K):
    """DESIGN.md section 2: J/K of a random density within 1e-11 * max(1, max|K|)."""
    return 1e-11 * max(1.0, float(np.abs(K).max()))


@pytest.fixture(scope="module")
def tb():
    import tuna_b200
    return tuna_b200


@pytest.fixture(scope="module")
def references(oracle):
    """Per basis: the oracle's dense Cartesian tensor and the FP64 J/K of densities() on it (J/K in the Cartesian basis: U = 1)."""
    from tuna_b200.basis import flatten
    out = {}
    for name in ("coverage", "n2_ccpvtz"):
        if name == "coverage":
            fb = oracle.FlatBasis.from_reference_objects(coverage_basis())
        else:
            fb = oracle_basis(oracle, load_golden(name))
        E = oracle.eri_fill(fb)
        P = densities(fb.ncart)
        J = np.stack([oracle.coulomb(p, E) for p in P])
        K = np.stack([oracle.exchange(p, E) for p in P])
        out[name] = dict(E=E, P=P, J=J, K=K, n=fb.ncart)
    return out


def _check_eri(got, ref):
    bad = np.abs(got - ref) > eri_tolerance(ref)
    assert not bad.any(), f"{int(bad.sum())} elements out of tolerance, max abs diff {np.abs(got - ref).max():.3e}"


# ---------------------------------------------------------------------------------------------------------------------
# direct engine: one child process per knob configuration
# ---------------------------------------------------------------------------------------------------------------------
_SMALL_G = {"TUNA_B200_G_DIV": "1e9", "TUNA_B200_SMEM_PER_LANE": "1e9"}      # group size set by the shared-memory limit alone
CONFIGS = {
    "default": {},
    "nb1": {"TUNA_B200_NB": "1"},
    "nb4": {"TUNA_B200_NB": "4"},
    "it_budget1500": {"TUNA_B200_IT_BUDGET": "1500"},          # multi-chunk classes
    "s_budget1500": {"TUNA_B200_S_BUDGET": "1500"},
    "term_max0": {"TUNA_B200_TERM_MAX": "0"},                  # separable digestion everywhere
    "tier2_off": {"TUNA_B200_TIER2": "0"},
    "own_launch_all": {"TUNA_B200_OWN_LAUNCH_UNITS": "0"},     # every job on its own launch
    "grouped": {"TUNA_B200_OWN_LAUNCH_UNITS": "1e9"},          # every NB = 2 job in a grouped launch
    "g_div1": {"TUNA_B200_G_DIV": "1"},
    "g_div64": {"TUNA_B200_G_DIV": "64"},
    "smem_per_lane64": {"TUNA_B200_SMEM_PER_LANE": "64"},
    "reg_tier_off": {"TUNA_B200_REG_TIER": "0"},
    "psplit0": {"TUNA_B200_PSPLIT_TARGET": "0"},
    "psplit7": {"TUNA_B200_PSPLIT_TARGET": "7"},               # ragged primitive chunks
    "psplit16_bra_only": {"TUNA_B200_PSPLIT_TARGET": "16", "TUNA_B200_KSPLIT": "0"},
    "streams1": {"TUNA_B200_STREAMS": "1"},
    # the remaining (G, NB) combinations of k_shell4_one and the group sizes of k_shell4_multi
    "small_g_nb1": dict(_SMALL_G, TUNA_B200_NB="1"),
    "small_g_nb4": dict(_SMALL_G, TUNA_B200_NB="4"),
    "small_g_own_launch": dict(_SMALL_G, TUNA_B200_OWN_LAUNCH_UNITS="0"),
    "small_g_grouped": dict(_SMALL_G, TUNA_B200_OWN_LAUNCH_UNITS="1e9"),
    "g_div1_nb1": {"TUNA_B200_G_DIV": "1", "TUNA_B200_NB": "1"},
    "g_div1_nb4": {"TUNA_B200_G_DIV": "1", "TUNA_B200_NB": "4"},
    "g_div1_grouped": {"TUNA_B200_G_DIV": "1", "TUNA_B200_OWN_LAUNCH_UNITS": "1e9"},
}
_KNOBS = ("NB", "NB_BYTES", "G_DIV", "SMEM_PER_LANE", "OWN_LAUNCH_UNITS", "IT_BUDGET", "S_BUDGET", "TERM_MAX", "TIER2", "REG_TIER",
          "PSPLIT_TARGET", "KSPLIT", "STREAMS", "DIRECT_ENGINE", "FILL_ENGINE", "DUMP_JOBS", "DBG_SKIP")


@pytest.fixture(scope="module")
def sweep(tmp_path_factory):
    """sweep(cfg) -> output directory of the child process of configuration cfg (run once per module)."""
    done = {}

    def run(cfg):
        if cfg not in done:
            out = tmp_path_factory.mktemp(cfg)
            env = {k: v for k, v in os.environ.items() if k not in {"TUNA_B200_" + x for x in _KNOBS}}
            env.update(CONFIGS[cfg])
            r = subprocess.run([sys.executable, os.path.join(HERE, "variant_gpu_case.py"), str(out)], env=env, cwd=ROOT,
                               capture_output=True, text=True, timeout=900)
            done[cfg] = (str(out), r.returncode, r.stdout[-2000:] + r.stderr[-4000:])
        out, rc, log = done[cfg]
        assert rc == 0, f"configuration {cfg} {CONFIGS[cfg]}: child failed (rc {rc}):\n{log}"
        return out
    return run


@pytest.mark.parametrize("cfg", list(CONFIGS))
def test_direct_engine_configuration_vs_oracle(sweep, references, cfg):
    """J/K at tau = 0 and 1e-16 within 1e-11 max(1, max|K|) of the oracle; shard partials sum to the whole; the engine fill equals the
    oracle's tensor within the ERI tolerance, with the same exact zeros and exact 8-fold symmetry."""
    out = sweep(cfg)
    for name, ref in references.items():
        tol = jk_tolerance(ref["K"])
        ld = lambda f: np.load(os.path.join(out, f"{name}_{f}.npy"))
        for tau in ("0", "1e-16"):
            J, K = ld(f"J_tau{tau}"), ld(f"K_tau{tau}")
            for d in range(len(ref["P"])):
                dj, dk = np.abs(J[d] - ref["J"][d]).max(), np.abs(K[d] - ref["K"][d]).max()
                assert dj <= tol and dk <= tol, f"{cfg} {name} tau {tau} density {d}: |dJ| {dj:.2e}, |dK| {dk:.2e}, tolerance {tol:.1e}"
        J0, K0 = ld("J_tau0"), ld("K_tau0")
        assert np.abs(ld("J_shard0") + ld("J_shard1") - J0).max() <= tol, (cfg, name, "J shards")
        assert np.abs(ld("K_shard0") + ld("K_shard1") - K0).max() <= tol, (cfg, name, "K shards")
        fill = os.path.join(out, f"{name}_fill.npy")
        E = np.load(fill)
        os.remove(fill)
        _check_eri(E, ref["E"])
        assert np.array_equal(E == 0.0, ref["E"] == 0.0), (cfg, name, "exact zeros")
        assert np.array_equal(E, E.transpose(1, 0, 2, 3)) and np.array_equal(E, E.transpose(0, 1, 3, 2)) and np.array_equal(E, E.transpose(2, 3, 0, 1))


def test_direct_engine_single_stream_is_bitwise_identical(sweep):
    """One stream instead of several changes only the order in which the class jobs run; the integer accumulation makes J/K bit-identical."""
    a, b = sweep("default"), sweep("streams1")
    files = sorted(os.path.basename(f) for f in glob.glob(os.path.join(a, "*_[JK]_*.npy")))
    assert len(files) == 2 * 2 * 4
    for f in files:
        assert np.array_equal(np.load(os.path.join(a, f)), np.load(os.path.join(b, f))), f


# Instantiations the launcher's switches can select (launch_shell4_jobs, csrc/tuna_b200.cu): k_shell4_one<G, NB, regs> for every G and NB
# with the default register budget (80), the 128-register builds of G = 256 with NB = 1 and 2, and k_shell4_multi<G, 2> for every G.
# Every one of them is reachable with the coverage basis and N2/cc-pVTZ under CONFIGS, so none is excluded.
GROUP_SIZES = (1, 2, 4, 8, 16, 32, 64, 128, 256)
ONE_INSTANTIATIONS = {(G, nb, 80) for G in GROUP_SIZES for nb in (1, 2, 4)} | {(256, 1, 128), (256, 2, 128)}
MULTI_INSTANTIATIONS = set(GROUP_SIZES)


def test_direct_engine_instantiation_coverage(sweep):
    """Every compiled k_shell4_one / k_shell4_multi instantiation ran in at least one configuration; the job tables also show
    term-list and separable digestion, multi-chunk classes (G >= 64 only), and bra and ket primitive splitting."""
    one, multi, seen = set(), set(), {"terms": set(), "nchunk>1": False, "ksplit>1": False, "psplit>1": False}
    for cfg in CONFIGS:
        for path in glob.glob(os.path.join(sweep(cfg), "jobs_*.csv")):
            with open(path) as f:
                for row in csv.DictReader(f):
                    G, nb = int(row["G"]), int(row["nb"])
                    if int(row["own"]):
                        one.add((G, nb, int(row["regs"])))
                    else:
                        assert nb == 2, row                       # k_shell4_multi exists for NB = 2 only
                        multi.add(G)
                    seen["terms"].add(int(row["terms"]))
                    seen["nchunk>1"] |= int(row["nchunk"]) > 1
                    seen["ksplit>1"] |= int(row["ksplit"]) > 1
                    seen["psplit>1"] |= int(row["psplit"]) > int(row["ksplit"])
                    if int(row["nchunk"]) > 1:
                        assert G >= 64, row                      # the table reload of a multi-chunk class synchronises the whole CTA
    report = json.dumps({"k_shell4_one ran": sorted(one), "k_shell4_multi ran": sorted(multi)})
    assert one <= ONE_INSTANTIATIONS and multi <= MULTI_INSTANTIATIONS, report
    missing_one, missing_multi = ONE_INSTANTIATIONS - one, MULTI_INSTANTIATIONS - multi
    assert not missing_one and not missing_multi, f"never ran: k_shell4_one {sorted(missing_one)}, k_shell4_multi {sorted(missing_multi)}; {report}"
    assert seen == {"terms": {0, 1}, "nchunk>1": True, "ksplit>1": True, "psplit>1": True}, seen


# ---------------------------------------------------------------------------------------------------------------------
# direct mode: density passes, J-only / K-only calls, zero and antisymmetric densities
# ---------------------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("engine", ["shell", "generic"])
@pytest.mark.parametrize("with_h", [True, False], ids=["h_two_per_pass", "g_four_per_pass"])
def test_direct_density_passes_and_partial_outputs(tb, oracle, references, monkeypatch, engine, with_h):
    """Non-symmetric densities double into symmetric and antisymmetric parts, cut into passes of 2 (h shells) or 4 (up to g) densities:
    nD = 3, 5, 8 give passes that mix both kinds.  J-only and K-only calls equal the halves of the full call; a zero density gives
    J = K = 0 exactly; a purely antisymmetric density gives J = 0 and the antisymmetric K of the oracle."""
    from tuna_b200.basis import flatten
    bfs = coverage_basis(with_h)
    n = len(bfs)
    E = references["coverage"]["E"] if with_h else oracle.eri_fill(oracle.FlatBasis.from_reference_objects(bfs))
    assert E.shape[0] == n
    if engine == "generic":
        monkeypatch.setenv("TUNA_B200_DIRECT_ENGINE", "generic")
    ctx = tb.Context(0)
    ctx.set_basis(*flatten(bfs))
    ctx.set_transform(np.eye(n))
    rng = np.random.default_rng(31)
    P = rng.standard_normal((8, n, n))
    Jr = np.stack([oracle.coulomb(p, E) for p in P])
    Kr = np.stack([oracle.exchange(p, E) for p in P])
    tol = jk_tolerance(Kr)
    for nD in (3, 5, 8):
        J, K = ctx.jk_direct(P[:nD], 0.0)
        for d in range(nD):
            assert np.abs(J[d] - Jr[d]).max() <= tol and np.abs(K[d] - Kr[d]).max() <= tol, (nD, d)
    J, K = ctx.jk_direct(P[:5], 0.0)
    Jo, Kn = ctx.jk_direct(P[:5], 0.0, want_k=False)
    Jn, Ko = ctx.jk_direct(P[:5], 0.0, want_j=False)
    assert Kn is None and Jn is None
    if engine == "shell":                       # integer accumulation: the same kernels give the same bits
        assert np.array_equal(Jo, J) and np.array_equal(Ko, K)
    else:
        assert np.abs(Jo - J).max() <= tol and np.abs(Ko - K).max() <= tol
    Z = np.zeros((n, n))
    Jz, Kz = ctx.jk_direct(Z, 0.0)
    assert not Jz.any() and not Kz.any()
    Jz, Kz = ctx.jk_direct(np.stack([P[0], Z, P[1]]), 1e-16)
    assert not Jz[1].any() and not Kz[1].any()
    A = (P[2] - P[2].T) / 2
    Ja, Ka = ctx.jk_direct(A, 0.0)
    assert np.abs(Ja).max() <= tol
    assert np.abs(Ka + Ka.T).max() <= tol
    assert np.abs(Ka - oracle.exchange(A, E)).max() <= tol


# ---------------------------------------------------------------------------------------------------------------------
# FockBuilder with a non-symmetric density
# ---------------------------------------------------------------------------------------------------------------------
def test_fock_builder_non_symmetric_density(tb):
    """The reference's CO/B3LYP guess density is asymmetric at ~1e-8 relative; FockBuilder.build must give the recorded K (1e-11).
    (tuna_jk_direct_dev, the device path of build_device, takes densities as symmetric and would drop K of the antisymmetric part.)"""
    from tuna_b200.distributed import FockBuilder
    g = load_golden("co_b3lyp_ccpvtz")
    P = np.array(g["seq0_1_K_P"])
    assert np.abs(P - P.T).max() > 1e-15 * np.abs(P).max()
    ctx = context_for(g)
    ctx.set_transform(g["U"])
    fb = FockBuilder(ctx, nD=1, tau=1e-16)
    J, K = fb.build(P)
    assert np.abs(K - g["seq0_1_K_out"]).max() < 1e-11
    Jd, Kd = ctx.jk_direct(P, 1e-16)
    assert np.abs(J - Jd).max() < 1e-11 and np.abs(K - Kd).max() < 1e-11
    Ps = (P + P.T) / 2                          # a symmetric density still takes the device path
    J2, K2 = fb.build(Ps)
    Jd2, Kd2 = ctx.jk_direct(Ps, 1e-16)
    assert np.abs(J2 - Jd2).max() < 1e-11 and np.abs(K2 - Kd2).max() < 1e-11


# ---------------------------------------------------------------------------------------------------------------------
# stored mode: every kernel instantiation tuna_jk_stored_dev dispatches to, on uploaded random tensors
# ---------------------------------------------------------------------------------------------------------------------
# Mirror of the rule of jk_stored_sym (csrc/tuna_b200.cu) for a pair-symmetric tensor: r = min(n, 960 / n) slab rows per tile, MT from
# ceil(n / r), 4 / 2 / 1 densities per pass for MT = 4 / 8 / 16; it declines (general kernels) for odd n, n < 16, MT > 16, more passes
# than the general kernels' 4 densities per pass, or when four ring stages do not fit 227 KB of shared memory.
def sym_launches(n, nD):
    """[(ND, MT) of every k_jk_stored_sym launch] for n x n x n x n and nD densities, or None when the general kernels run."""
    if n % 2 or n < 16 or n > 960:
        return None
    r = min(n, 960 // n)
    mt_need = -(-n // r)
    MT = 4 if mt_need <= 4 else 8 if mt_need <= 8 else 16 if mt_need <= 16 else 0
    if MT == 0:
        return None
    nd_max = {4: 4, 8: 2, 16: 1}[MT]
    if -(-nD // nd_max) > (nD + 3) // 4:
        return None
    out = []
    for d0 in range(0, nD, nd_max):
        nd = min(nd_max, nD - d0)
        if (nd * n * n + 2 * nd * r * n) * 8 + 2 * 16 * 8 + 128 + 4 * 2 * r * n * 8 > 227 * 1024:
            return None
        out.append((nd, MT))
    return out


# Shared memory of k_jk_stored_tma (tuna_jk_stored_dev): a ring of `stages` tiles of R whole slab rows, R from the tile size, next to
# the per-warp J partials and the K buffer of four densities.  The launcher lowers the stage count to what fits 227 KB; the geometries
# below are chosen to fit as given.
def tma_ring_fits(n, tile_kb, stages):
    r = max(1, 512 // n)
    q = -(-n * n * 8 // (tile_kb * 1024))
    R = -(-n // q)
    R = -(-R // r) * r
    nwarp = -(-n * r // 32)
    return stages * R * n * 8 + (2 * nwarp * 4 + 4 * r * n) * 8 + 4 * 8 + 16 <= 227 * 1024


SYM_INSTANTIATIONS = {(1, 4), (2, 4), (3, 4), (4, 4), (1, 8), (2, 8), (1, 16)}
# (n, nD) of the pair-symmetric cases; together they launch every k_jk_stored_sym<ND, MT>
SYM_CASES = [(48, 1), (48, 3), (48, 4), (48, 5), (48, 8), (60, 2), (64, 1), (64, 2), (96, 1)]
# (tile KB, stages, CTAs per SM) of the TMA kernel off the defaults (24, 3, 2)
TMA_GEOMETRIES = [(1, 3, 2), (64, 3, 2), (24, 1, 2), (24, 4, 2), (24, 3, 1), (24, 3, 4), (1, 1, 4), (64, 1, 1)]


def test_stored_rule_mirror_reaches_every_sym_instantiation():
    cells = {c for n, nD in SYM_CASES for c in (sym_launches(n, nD) or [])}
    assert cells == SYM_INSTANTIATIONS
    assert sym_launches(126, 1) is None and sym_launches(14, 1) is None and sym_launches(64, 3) is None and sym_launches(96, 2) is None
    assert not tma_ring_fits(126, 64, 4)


def _stored_reference(E, P):
    """J, K by np.einsum in FP64 and the per-element bound 64 * 2^-53 * sum_kl |E| |P| of a rounded sum of those terms."""
    J = np.einsum("ijkl,dkl->dij", E, P, optimize=True)
    K = np.einsum("ilkj,dkl->dij", E, P, optimize=True)
    aE, aP = np.abs(E), np.abs(P)
    u = 64 * 2.0 ** -53
    return J, K, u * np.einsum("ijkl,dkl->dij", aE, aP, optimize=True), u * np.einsum("ilkj,dkl->dij", aE, aP, optimize=True)


def _check_stored(tb, E, P, ref, label, want_j=True, want_k=True):
    ctx = tb.Context(0)
    ctx.eri_upload(E)
    J, K = ctx.jk_stored(P, want_j=want_j, want_k=want_k)
    ctx.close()
    Jr, Kr, bJ, bK = ref
    if want_j:
        bad = np.abs(J - Jr) > bJ
        assert not bad.any(), f"{label}: J off at {int(bad.sum())} elements, max |dJ| {np.abs(J - Jr).max():.2e}"
    else:
        assert J is None
    if want_k:
        bad = np.abs(K - Kr) > bK
        assert not bad.any(), f"{label}: K off at {int(bad.sum())} elements, max |dK| {np.abs(K - Kr).max():.2e}"
    else:
        assert K is None


_STORED_ENV = ("STORED_KERNEL", "JK_TILE_KB", "JK_STAGES", "JK_CTAS_PER_SM")


@pytest.mark.parametrize("n", [4, 8, 14, 48, 60, 64, 69, 96, 126])
def test_stored_kernel_matrix(tb, monkeypatch, n):
    """Stored J/K of every kernel and density count at dimension n: k_jk_stored_sym<ND, MT> on pair-symmetric tensors (SYM_CASES),
    k_jk_stored_tma<ND> on general tensors of even n >= 8 (also forced on a symmetric one, and at TMA_GEOMETRIES), k_jk_stored<ND> for
    odd n, n < 8 and when forced; J-only and K-only calls; several passes of 4 densities."""
    for k in _STORED_ENV:
        monkeypatch.delenv("TUNA_B200_" + k, raising=False)
    rng = np.random.default_rng(1000 + n)
    A = rng.standard_normal((n * n, n * n))
    small = n <= 14
    counts = (1, 2, 3, 4, 5, 8) if small else (1, 2, 5) if n <= 64 else (1,)
    P = rng.standard_normal((max(counts), n, n))
    Eg = A.reshape(n, n, n, n)
    refs = {nD: _stored_reference(Eg, P[:nD]) for nD in counts}
    general = "simple" if n % 2 or n < 8 else "tma"
    for nD in counts:
        _check_stored(tb, Eg, P[:nD], refs[nD], f"{general} n {n} nD {nD}")
    _check_stored(tb, Eg, P[:counts[-1]], refs[counts[-1]], f"{general} n {n} J only", want_k=False)
    _check_stored(tb, Eg, P[:counts[-1]], refs[counts[-1]], f"{general} n {n} K only", want_j=False)
    if general == "tma":
        monkeypatch.setenv("TUNA_B200_STORED_KERNEL", "simple")
        for nD in (counts if small else counts[:1]):
            _check_stored(tb, Eg, P[:nD], refs[nD], f"simple (forced) n {n} nD {nD}")
        monkeypatch.delenv("TUNA_B200_STORED_KERNEL")
        if n in (14, 64, 126):
            nD = counts[-1]
            for tile, stages, cps in TMA_GEOMETRIES:
                if not tma_ring_fits(n, tile, stages):
                    continue
                monkeypatch.setenv("TUNA_B200_JK_TILE_KB", str(tile))
                monkeypatch.setenv("TUNA_B200_JK_STAGES", str(stages))
                monkeypatch.setenv("TUNA_B200_JK_CTAS_PER_SM", str(cps))
                _check_stored(tb, Eg, P[:nD], refs[nD], f"tma n {n} tile {tile} KB, {stages} stages, {cps} CTAs/SM")
                _check_stored(tb, Eg, P[:nD], refs[nD], f"tma n {n} tile {tile} KB, {stages} stages, {cps} CTAs/SM, K only", want_j=False)
            for k in _STORED_ENV[1:]:
                monkeypatch.delenv("TUNA_B200_" + k)
    del Eg, refs
    sym = [nD for m, nD in SYM_CASES if m == n]
    if n % 2 == 0 and n >= 8 and (sym or n in (14, 126)):
        A += A.T
        A *= 0.5
        Es = A.reshape(n, n, n, n)                           # (ij|kl) = (kl|ij): pair-symmetric
        for nD in sym or [1]:
            Pd = rng.standard_normal((nD, n, n))
            ref = _stored_reference(Es, Pd)
            _check_stored(tb, Es, Pd, ref, f"n {n} nD {nD} symmetric tensor, {sym_launches(n, nD)}")
            if nD == max(sym or [1]):
                _check_stored(tb, Es, Pd, ref, f"n {n} nD {nD} symmetric tensor, J only", want_k=False)
                _check_stored(tb, Es, Pd, ref, f"n {n} nD {nD} symmetric tensor, K only", want_j=False)
                monkeypatch.setenv("TUNA_B200_STORED_KERNEL", "tma")
                _check_stored(tb, Es, Pd, ref, f"tma (forced) n {n} nD {nD} symmetric tensor")
                monkeypatch.delenv("TUNA_B200_STORED_KERNEL")
