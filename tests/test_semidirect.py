"""Semi-direct J/K: the shell-quartet engine's integral store (tuna_set_integral_store, Context.set_integral_store,
DeviceGroup.set_integral_store, configure(store_fraction=...)).

A store pass runs the direct kernels and also writes every work item's contracted integral buffer to a row in device memory; later
builds load the rows instead of evaluating phases 0-4 and digest them exactly as the direct build does.  Every work item contributes the
same integer words either way, so J and K must be BITWISE equal to the direct build whatever is stored.

CPU: the engine body with store and replay (tests/host_emul/emul_store.cpp) against the direct build, bitwise, with full and partial
stores, different chunk splits between store pass and replay, a replay density that screens differently from the store pass, and one
rank of a sharded launch whose jobs start at non-zero flat unit offsets (the grouped kernel).
GPU (`-m gpu`): recorded SCF densities, asymmetric densities, screening changes, budgets, invalidation, contexts sharded as rank r > 0
of n on one device over builds that change the job set, groups of 2/4/8 devices (skipped where fewer are visible) and the restated SCF
through the provider, including a second geometry's mode decision.  (The reference's own driver runs direct mode with the store on in test_reference_on_gpu.py, since
the store is on by default there.)"""
import ctypes
import os
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(HERE, "golden"))

from util import basis_objects, load_golden, oracle_basis  # noqa: E402

TAU = 1e-16
BIG = 1 << 50          # "everything": the library clamps the budget to the free device memory


# ---------------------------------------------------------------------------------------------------------------------------------
# CPU: host build of store and replay
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def emul_store(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("emul") / "libemul_store.so")
    src = os.path.join(HERE, "host_emul", "emul_store.cpp")
    subprocess.run(["g++", "-O2", "-fopenmp", "-fPIC", "-shared", "-x", "c++", "-o", so, src, "-lm"], check=True)
    return ctypes.CDLL(so)


def _h_shell_basis(oracle):
    from tuna_b200 import workloads as w
    from tuna_b200.basis import from_arrays
    shells_a = [(0, [1.3], [1.0]), (1, [0.9], [1.0]), (5, [1.1], [1.0])]
    shells_b = [(2, [0.8], [1.0]), (4, [1.2], [1.0]), (5, [0.7], [1.0]), (3, [1.0, 0.4], [0.6, 0.5])]
    b = w.shells_to_components([shells_a, shells_b], [0.0, 1.9])
    return oracle.FlatBasis.from_reference_objects(from_arrays(b["origins"], b["lmn"], b["nprim"], b["exps"], b["raw_coefs"]))


def _run_store(lib, fb, P1, P2, tau, select, rank=0, nranks=1, unit_shift=0):
    n = fb.ncart
    dp, ip, lp = ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int), ctypes.POINTER(ctypes.c_int64)
    oz = np.ascontiguousarray(fb.origins[:, 2])
    lmn = np.ascontiguousarray(fb.lmn, dtype=np.int32)
    npr = np.ascontiguousarray(fb.nprim, dtype=np.int32)
    off = np.ascontiguousarray(fb.offsets, dtype=np.int64)
    ceff = np.ascontiguousarray(fb.coefs * fb.norms)
    nD = P1.shape[0]
    J, K = np.full((2, nD, n, n), np.nan), np.full((2, nD, n, n), np.nan)
    stats = np.zeros(8, dtype=np.int64)
    rc = lib.emul_jk_shell4_store(n, oz.ctypes.data_as(dp), lmn.ctypes.data_as(ip), npr.ctypes.data_as(ip), off.ctypes.data_as(lp),
                                  fb.exps.ctypes.data_as(dp), ceff.ctypes.data_as(dp), nD, np.ascontiguousarray(P1).ctypes.data_as(dp),
                                  np.ascontiguousarray(P2).ctypes.data_as(dp), ctypes.c_double(tau), select, rank, nranks, unit_shift,
                                  J.ctypes.data_as(dp), K.ctypes.data_as(dp), stats.ctypes.data_as(ctypes.POINTER(ctypes.c_longlong)))
    assert rc == 0
    return J, K, stats


def _sym(rng, nD, n):
    P = rng.standard_normal((nD, n, n))
    return (P + P.transpose(0, 2, 1)) / 2


@pytest.mark.parametrize("case,nb,budget,budget_replay", [("n2_ccpvtz", "2", None, None), ("n2_ccpvtz", "1", "96", None),
                                                          ("h_shells", "2", None, "1500"), ("h_shells", "4", "700", None),
                                                          ("h_shells", "1", "1500", "700")])
def test_host_store_and_replay_bitwise(emul_store, oracle, case, nb, budget, budget_replay, monkeypatch):
    """Direct, stored-then-replayed and partially stored J/K of two builds are bitwise equal; multi-chunk classes, 1/2/4 quartets per
    batch, and chunk splits that differ between the store pass and the replay.  Every row of a stored job is written by the store pass
    and read exactly once by the replay."""
    monkeypatch.setenv("TUNA_EMUL_NB", nb)
    for var, val in (("TUNA_EMUL_IT_BUDGET", budget), ("TUNA_EMUL_IT_BUDGET_REPLAY", budget_replay)):
        if val:
            monkeypatch.setenv(var, val)
        else:
            monkeypatch.delenv(var, raising=False)
    fb = oracle_basis(oracle, load_golden(case)) if case != "h_shells" else _h_shell_basis(oracle)
    rng = np.random.default_rng(5)
    P1, P2 = _sym(rng, 2, fb.ncart), _sym(rng, 2, fb.ncart)
    Jd, Kd, sd = _run_store(emul_store, fb, P1, P2, 0.0, 0)
    assert sd[0] == 0 and not np.isnan(Jd).any() and not np.isnan(Kd).any()
    for select in (1, 2):
        J, K, st = _run_store(emul_store, fb, P1, P2, 0.0, select)
        assert np.array_equal(J, Jd) and np.array_equal(K, Kd), select
        assert st[0] > 0 and st[1] == 0 and st[2] == 0 and st[3] == 0 and st[5] == st[0] and st[6] == 0 and st[7] == 0, (select, st)
    E = oracle.eri_fill(fb)
    assert np.abs(Jd[1, 0] - oracle.coulomb(P2[0], E)).max() < 1e-11 * max(1.0, np.abs(Jd).max())
    assert np.abs(Kd[1, 1] - oracle.exchange(P2[1], E)).max() < 1e-11 * max(1.0, np.abs(Kd).max())


@pytest.mark.parametrize("rank,nranks,shift", [(1, 2, 1), (3, 4, 3), (2, 3, 1), (0, 3, 5)])
def test_host_store_sharded_with_flat_unit_offsets(emul_store, oracle, rank, nranks, shift):
    """One rank of a sharded launch that deals FLAT units (a group of jobs in one k_shell4_multi launch: job j's units start at a non-zero
    offset, so the units a rank owns in a job need not start with the job's first).  The store pass writes exactly the rows of the rank's
    share (nothing outside it, guard rows between the jobs intact), the replay digests each once, and the rank's J/K are bitwise equal to
    its direct J/K.  The ranks' shares together hold every work item once."""
    fb = _h_shell_basis(oracle)
    rng = np.random.default_rng(13)
    P1, P2 = _sym(rng, 1, fb.ncart), _sym(rng, 1, fb.ncart)
    Jd, Kd, _ = _run_store(emul_store, fb, P1, P2, 0.0, 0, rank, nranks, shift)
    for select in (1, 2):
        J, K, st = _run_store(emul_store, fb, P1, P2, 0.0, select, rank, nranks, shift)
        assert np.array_equal(J, Jd) and np.array_equal(K, Kd), select
        assert st[0] > 0 and st[1] == 0 and st[2] == 0 and st[3] == 0 and st[6] == 0 and st[7] == 0, (select, st)
    rows = [_run_store(emul_store, fb, P1, P2, 0.0, 1, r, nranks, shift)[2][0] for r in range(nranks)]
    assert sum(rows) == _run_store(emul_store, fb, P1, P2, 0.0, 1)[2][0]


def test_host_store_pass_keeps_what_its_density_screens_out(emul_store, oracle):
    """A store pass whose density screens quartets out of its own digestion still evaluates and stores them; a replay build whose
    density keeps more (or fewer) quartets digests exactly the direct build's quartets."""
    fb = oracle_basis(oracle, load_golden("n2_ccpvtz"))
    rng = np.random.default_rng(9)
    P = _sym(rng, 1, fb.ncart)
    tau = 1e-9
    for P1, P2 in ((1e-4 * P, P), (P, 1e-4 * P)):
        Jd, Kd, _ = _run_store(emul_store, fb, P1, P2, tau, 0)
        J, K, st = _run_store(emul_store, fb, P1, P2, tau, 1)
        assert np.array_equal(J, Jd) and np.array_equal(K, Kd)
        assert st[1] == 0 and st[2] == 0
        if P1 is not P:
            assert st[4] > 0                     # screened out of the store pass's digestion, stored all the same


def test_configure_store_fraction():
    import tuna_b200
    from tuna_b200 import provider
    saved = provider._store_fraction
    try:
        tuna_b200.configure(store_fraction=0.25)
        assert provider._store_fraction == 0.25
        for bad in (-0.1, 1.5):
            with pytest.raises(tuna_b200.TunaError):
                tuna_b200.configure(store_fraction=bad)
        tuna_b200.configure(store_fraction=0)
        assert provider._store_fraction == 0.0
    finally:
        provider._store_fraction = saved


# ---------------------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------------------
def _gpus():
    import torch
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


def _case(name):
    """(flattened basis, U, golden or None)."""
    from tuna_b200 import workloads as w
    from tuna_b200.basis import flatten, from_arrays
    if name.startswith("et") and name != "et100":
        b = w.even_tempered_diatomic(int(name[2:]))
        bfs = from_arrays(b["origins"], b["lmn"], b["nprim"], b["exps"], b["raw_coefs"])
        return flatten(bfs), np.eye(len(bfs)), None
    g = load_golden(name)
    return flatten(basis_objects(g)), np.array(g["U"]), g


def _ctx(flat, U, device=0, budget=0):
    import tuna_b200
    ctx = tuna_b200.Context(device)
    ctx.set_basis(*flat)
    ctx.set_transform(U)
    ctx.set_integral_store(budget)
    return ctx


def _sequence(g):
    """The recorded SCF densities, one stack per Fock build (UHF: alpha and beta together, nD = 2)."""
    keys = sorted((k for k in g.files if k.startswith("seq") and k.endswith("_J_P")), key=lambda k: (int(k.split("_")[0][3:]), k))
    builds = {}
    for k in keys:
        builds.setdefault(int(k.split("_")[0][3:]), []).append(np.array(g[k]))
    return [np.stack(v) if len(v) > 1 else v[0] for _, v in sorted(builds.items())]


def _bitwise(got, ref, what=""):
    for a, b, name in zip(got, ref, "JK"):
        assert np.array_equal(a, b), f"{what} {name}: max |semi-direct - direct| = {np.abs(a - b).max():.3e}"


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["n2_ccpvtz", "ne2_uhf_ccpvqz", "et100"])
def test_recorded_scf_densities_bitwise(name):
    flat, U, g = _case(name)
    direct, semi = _ctx(flat, U), _ctx(flat, U, budget=BIG)
    seq = _sequence(g)
    assert len(seq) >= 3
    for i, P in enumerate(seq):
        _bitwise(semi.jk_direct(P, TAU), direct.jk_direct(P, TAU), f"build {i}")
        assert semi.counts()["evaluated_last_direct"] == direct.counts()["evaluated_last_direct"]
    info = semi.integral_store_info()
    assert info["bytes"] > 0 and info["items"] > 0 and info["items"] <= info["items_last_build"], info
    assert info["replayed_builds"] == len(seq) - 1, info
    if name == "ne2_uhf_ccpvqz":
        assert seq[0].shape[0] == 2
    assert direct.integral_store_info() == {"bytes": 0, "items": 0, "items_last_build": 0, "replayed_builds": 0}


@pytest.mark.gpu
def test_asymmetric_density_and_screening_changes():
    """An asymmetric density (antisymmetric split: twice the densities, another job set), and densities whose per-build screening differs
    from the store pass's, in both directions."""
    flat, U, g = _case("n2_ccpvtz")
    nbf = U.shape[0]
    P = _sequence(g)[-1]
    A = np.random.default_rng(3).standard_normal((nbf, nbf))
    asym = P + 1e-6 * (A - A.T)
    tau = 1e-10
    direct, semi = _ctx(flat, U), _ctx(flat, U, budget=BIG)
    for i, (Q, t) in enumerate([(P, TAU), (asym, TAU), (P, TAU), (1e-3 * P, tau), (P, tau), (1e-5 * P, tau), (asym, TAU)]):
        _bitwise(semi.jk_direct(Q, t), direct.jk_direct(Q, t), f"build {i}")
        assert semi.counts()["evaluated_last_direct"] == direct.counts()["evaluated_last_direct"]
    assert semi.integral_store_info()["replayed_builds"] >= 4


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["n2_ccpvtz", "et100"])
def test_budgets(name):
    """Budgets of nothing, a small part, half and everything: the same J and K, never more bytes than the budget."""
    flat, U, g = _case(name)
    seq = _sequence(g)[-3:]
    direct = _ctx(flat, U)
    ref = [direct.jk_direct(P, TAU) for P in seq]
    full = _ctx(flat, U, budget=BIG)
    for P, r in zip(seq, ref):
        _bitwise(full.jk_direct(P, TAU), r, "everything")
    whole = full.integral_store_info()
    assert whole["items"] == whole["items_last_build"], whole          # everything fits
    for frac in (0.0, 0.02, 0.5):
        budget = int(frac * whole["bytes"])
        ctx = _ctx(flat, U, budget=budget)
        for P, r in zip(seq, ref):
            _bitwise(ctx.jk_direct(P, TAU), r, f"budget {budget}")
        info = ctx.integral_store_info()
        assert info["bytes"] <= budget, (budget, info)
        if frac == 0.0:
            assert info["items"] == 0 and info["replayed_builds"] == 0
        if frac == 0.5:
            assert 0 < info["items"] < whole["items"] and info["replayed_builds"] == len(seq) - 1, info


@pytest.mark.gpu
def test_invalidation_between_builds():
    """tuna_set_transform, tuna_set_basis, tuna_set_shard and a new budget drop the store; the results stay equal."""
    flat, U, g = _case("ne2_uhf_ccpvqz")
    seq = _sequence(g)
    direct, semi = _ctx(flat, U), _ctx(flat, U, budget=BIG)
    P = seq[-1]
    ref = direct.jk_direct(P, TAU)
    _bitwise(semi.jk_direct(P, TAU), ref)
    assert semi.integral_store_info()["bytes"] > 0

    def dropped():
        info = semi.integral_store_info()
        assert info["bytes"] == 0 and info["items"] == 0, info

    semi.set_transform(U)
    dropped()
    _bitwise(semi.jk_direct(P, TAU), ref)
    _bitwise(semi.jk_direct(P, TAU), ref)
    semi.set_basis(*flat)
    dropped()
    semi.set_transform(U)
    _bitwise(semi.jk_direct(P, TAU), ref)
    semi.set_shard(0, 2)
    dropped()
    half = semi.jk_direct(P, TAU)
    direct.set_shard(0, 2)
    _bitwise(semi.jk_direct(P, TAU), direct.jk_direct(P, TAU), "shard (0, 2)")
    _bitwise(semi.jk_direct(P, TAU), half, "shard (0, 2) replayed")
    semi.set_shard(0, 1)
    direct.set_shard(0, 1)
    semi.set_integral_store(BIG // 2)
    dropped()
    for Q in seq[:3]:
        _bitwise(semi.jk_direct(Q, TAU), direct.jk_direct(Q, TAU))
    semi.set_integral_store(0)
    dropped()
    _bitwise(semi.jk_direct(P, TAU), ref)
    assert semi.integral_store_info()["bytes"] == 0


@pytest.mark.gpu
@pytest.mark.parametrize("rank,nranks", [(1, 2), (3, 4), (5, 8)])
@pytest.mark.parametrize("name", ["n2_ccpvtz", "ne2_uhf_ccpvqz"])
def test_sharded_ranks_with_store_on_one_device(name, rank, nranks):
    """The rank of a device group, run on one device: a context sharded as (rank, nranks) with the store against one with the same shard
    without it, over builds that change the job set (nD = 1 / 2, the asymmetric split, back).  Its light class jobs share grouped launches,
    whose units are dealt to ranks by their flat index in the group."""
    flat, U, g = _case(name)
    direct, semi = _ctx(flat, U), _ctx(flat, U, budget=BIG)
    for c in (direct, semi):
        c.set_shard(rank, nranks)
    seq = _sequence(g)
    nbf = U.shape[0]
    P = seq[-1] if seq[-1].ndim == 2 else seq[-1][0]
    A = np.random.default_rng(rank).standard_normal((nbf, nbf))
    builds = [P, np.stack([P, seq[0] if seq[0].ndim == 2 else seq[0][1]]), P, P + 1e-6 * (A - A.T), P, seq[-2]]
    for i, Q in enumerate(builds):
        _bitwise(semi.jk_direct(Q, TAU), direct.jk_direct(Q, TAU), f"rank {rank}/{nranks} build {i}")
        assert semi.counts()["evaluated_last_direct"] == direct.counts()["evaluated_last_direct"]
    info = semi.integral_store_info()
    assert info["items"] > 0 and info["replayed_builds"] >= 3, info


@pytest.mark.gpu
@pytest.mark.parametrize("n", [2, 4, 8])
@pytest.mark.parametrize("name", ["n2_ccpvtz", "ne2_uhf_ccpvqz", "et100"])
def test_group_with_store_bitwise_equals_one_device(name, n):
    import tuna_b200
    if _gpus() < n:
        pytest.skip(f"needs {n} GPUs")
    flat, U, g = _case(name)
    solo = _ctx(flat, U)
    group = tuna_b200.DeviceGroup(list(range(n)))
    group.set_basis(*flat)
    group.set_transform(U)
    group.set_integral_store(BIG)
    for i, P in enumerate(_sequence(g)[:4]):
        _bitwise(group.jk_direct(P, TAU), solo.jk_direct(P, TAU), f"build {i}")
    info = group.integral_store_info()
    assert info["items"] > 0 and info["replayed_builds"] == 3, info
    assert all(c.integral_store_info()["items"] > 0 for c in group.contexts)
    group.close()
    solo.close()


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["ne2_uhf_ccpvqz", "et100"])
def test_provider_scf_with_the_store(name):
    """The restated SCF in direct mode with the store reproduces the golden energy and iteration count, bitwise equal to the run
    without it; afterwards the handle can still be materialised (the post-HF path), which gives the store's memory back."""
    from oracle import scf_oracle
    from test_reference_on_gpu import provider_eri, provider_jk
    import tuna_b200
    from tuna_b200 import provider
    g = load_golden(name)
    saved = dict(provider._settings), provider._devices, provider._store_fraction
    try:
        results = {}
        for frac in (0.0, 0.5):
            tuna_b200.configure(mode="direct", device=0, store_fraction=frac)
            eri = provider_eri(tuna_b200, g)
            energy, iterations, _ = scf_oracle.run_scf(provider_jk(tuna_b200, eri, []), g)
            assert abs(energy - float(g["energy"])) < 1e-10 and iterations == int(g["n_iterations"]), (frac, energy, iterations)
            results[frac] = energy
            info = eri.ctx.integral_store_info()
            if frac > 0:
                assert info["bytes"] > 0 and info["replayed_builds"] > 0, info
                # the next geometry's mode is decided with the store's memory given back; the finished handle then runs direct
                eri2 = provider_eri(tuna_b200, g)
                assert eri.ctx.integral_store_info()["bytes"] == 0 and eri2.mode == "direct"
                P = np.array(g["P_final"]) if not bool(g["unrestricted"]) else np.array(g["P_alpha_final"])
                assert np.array_equal(tuna_b200.calculate_coulomb_matrix(P, eri), eri.ctx.jk_direct(P, provider._settings["tau"])[0])
                dense = np.asarray(eri)
                assert dense.shape == (int(g["nbf"]),) * 4
                assert eri.ctx.integral_store_info()["bytes"] == 0
            else:
                assert info["bytes"] == 0
        assert results[0.5] == results[0.0]
    finally:
        provider._settings.clear()
        provider._settings.update(saved[0])
        provider._devices, provider._store_fraction = saved[1], saved[2]
