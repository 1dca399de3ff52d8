"""Direct J/K from device-resident densities of any real P (tuna_jk_direct_general_dev, tuna_jk_direct_group_general_dev,
Context.jk_direct_general_dev, DeviceGroup.jk_direct_general_dev, and the asymmetric branch of FockBuilder.build).

The host entry points split a non-symmetric stack into its symmetric and antisymmetric parts and set the pre-screening bound from max|P|
(density_split.hpp).  The general device entry points take the same two maxima on the device, reach the same decision and split with the
same arithmetic, so their J and K must be BITWISE equal to tuna_jk_direct / tuna_jk_direct_group for the same P.

CPU: the shared plan compiled for the host against the rule restated here; the new symbols are exported; no source names the batched
copy family.
GPU (`-m gpu`): bitwise against the host entry point on N2/cc-pVTZ, Ne2 UHF/cc-pVQZ and ET100 for symmetric, slightly and strongly
asymmetric, large and mixed stacks; against the oracle's dense J/K; the defect of tuna_jk_direct_dev on an asymmetric P; the integral
store; sharded contexts and device groups; the per-component kernel; FockBuilder; bad arguments."""
import ctypes
import os
import re
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)

from util import basis_objects, load_golden, oracle_basis  # noqa: E402

TAU = 1e-16
BIG = 1 << 50          # integral store budget "everything": the library clamps it to the free device memory


# ---------------------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------------------
@pytest.fixture(scope="module")
def emul_density(tmp_path_factory):
    so = str(tmp_path_factory.mktemp("emul") / "libemul_density.so")
    src = os.path.join(HERE, "host_emul", "emul_density.cpp")
    subprocess.run(["g++", "-O2", "-fPIC", "-shared", "-x", "c++", "-o", so, src, "-lm"], check=True)
    return ctypes.CDLL(so)


def _plan(lib, P):
    P = np.ascontiguousarray(P, dtype=np.float64)
    nD, n = P.shape[0], P.shape[1]
    ext = np.zeros(2)
    nDrun, mask, bound = ctypes.c_int(), ctypes.c_uint(), ctypes.c_double()
    dp = ctypes.POINTER(ctypes.c_double)
    lib.emul_plan_density(P.ctypes.data_as(dp), nD, n, ext.ctypes.data_as(dp), ctypes.byref(nDrun), ctypes.byref(mask), ctypes.byref(bound))
    return float(ext[0]), float(ext[1]), nDrun.value, mask.value, bound.value


def _restated_rule(P):
    """What tuna_jk_direct did before the rule moved into density_split.hpp: max|P|, max|P - P^T|, a split stack when the second exceeds
    1e-15 times the first (the antisymmetric parts after the symmetric ones, marked in anti_mask), and dens_bound = max(1e3, 1e3 max|P|)."""
    nD = P.shape[0]
    pmax = float(np.abs(P).max())
    amax = float(np.abs(P - P.transpose(0, 2, 1)).max())
    general = amax > 1e-15 * pmax
    mask = sum(1 << (nD + d) for d in range(nD)) if general else 0
    return pmax, amax, 2 * nD if general else nD, mask, max(1e3, 1e3 * pmax)


def _stacks(n, seed=3):
    rng = np.random.default_rng(seed)
    S = rng.standard_normal((3, n, n))
    S = (S + S.transpose(0, 2, 1)) / 2
    A = rng.standard_normal((3, n, n))
    A = A - A.transpose(0, 2, 1)
    return {
        "symmetric": S,
        "asym_1e-8": S + 1e-8 * A,
        "asym_O(1)": S + A,
        "zero": np.zeros((2, n, n)),
        "mixed": np.stack([S[0], S[1] + 1e-8 * A[1]]),
        "scaled_1e3": 1e3 * S[:1],
        "eight": np.concatenate([S, S, S[:2]]) + np.concatenate([np.zeros((7, n, n)), 1e-12 * A[:1]]),
        "round_off_asym": S[:1] + 1e-17 * np.abs(S[:1]).max() * A[:1],
    }


@pytest.mark.parametrize("n", [1, 7, 60])
def test_host_plan_matches_the_restated_rule(emul_density, n):
    for name, P in _stacks(n).items():
        got, ref = _plan(emul_density, P), _restated_rule(P)
        assert got == ref, (name, got, ref)
    assert _plan(emul_density, _stacks(n)["zero"])[2:4] == (2, 0)
    if n > 1:
        assert _plan(emul_density, _stacks(n)["asym_1e-8"])[2:4] == (6, 0b111000)
        assert _plan(emul_density, _stacks(n)["eight"])[2:4] == (16, 0xff00)


def test_new_symbols_are_exported():
    from tuna_b200 import _lib
    from tuna_b200.build import build
    build()
    lib = _lib.load()
    for name in ("tuna_jk_direct_general_dev", "tuna_jk_direct_group_general_dev"):
        assert name in _lib.EXPORTS and hasattr(lib, name), name
    header = open(os.path.join(ROOT, "include", "tuna_b200.h")).read()
    assert "int tuna_jk_direct_general_dev(" in header and "int tuna_jk_direct_group_general_dev(" in header


def test_no_source_names_the_batched_copy_family():
    """Copies go through cudaMemcpyAsync / cudaMemcpyPeerAsync only (the pattern is assembled so that this file does not name them)."""
    pattern = re.compile("(cu|cuda)Memcpy(3D)?" + "Batch")
    hits = []
    for top in ("tuna_b200", "include", "tests", "tools", "oracle"):
        for dirpath, _, files in os.walk(os.path.join(ROOT, top)):
            for f in files:
                if f.endswith((".cu", ".cuh", ".hpp", ".h", ".cpp", ".c", ".py", ".sh")) or f == "Makefile":
                    path = os.path.join(dirpath, f)
                    with open(path, errors="replace") as fh:
                        if pattern.search(fh.read()):
                            hits.append(os.path.relpath(path, ROOT))
    for f in ("bench.py", "__graft_entry__.py"):
        with open(os.path.join(ROOT, f)) as fh:
            if pattern.search(fh.read()):
                hits.append(f)
    assert not hits, hits


# ---------------------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------------------
def _gpus():
    import torch
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


def _case(name):
    """(flattened basis, U, the recorded final density stack (symmetric; UHF: alpha and beta), the recorded guess density stack).
    The guess densities are asymmetric at ~1e-16 relative: below the split threshold, so they run as they are."""
    from tuna_b200.basis import flatten
    g = load_golden(name)
    if bool(g["unrestricted"]):
        P = np.stack([np.array(g["P_alpha_final"]), np.array(g["P_beta_final"])])
        G = np.stack([np.array(g["P_guess_alpha"]), np.array(g["P_guess_beta"])])
    else:
        P, G = np.array(g["P_final"])[None], np.array(g["P_guess"])[None]
    return flatten(basis_objects(g)), np.array(g["U"]), P, G


def _ctx(flat, U, device=0, shard=None, budget=0):
    import tuna_b200
    ctx = tuna_b200.Context(device)
    ctx.set_basis(*flat)
    ctx.set_transform(U)
    if shard:
        ctx.set_shard(*shard)
    if budget:
        ctx.set_integral_store(budget)
    return ctx


def _general_dev(obj, P, tau=TAU, device=0, want_j=True):
    """obj.jk_direct_general_dev on torch device buffers; the caller's density must come back unchanged."""
    import torch
    dev = torch.device("cuda", device)
    dP = torch.from_numpy(np.ascontiguousarray(P)).to(dev)
    dJ, dK = torch.full_like(dP, float("nan")), torch.full_like(dP, float("nan"))
    torch.cuda.synchronize(dev)                     # the context's own stream does not order after torch's
    obj.jk_direct_general_dev(P.shape[0], dP.data_ptr(), dJ.data_ptr() if want_j else 0, dK.data_ptr(), tau)
    torch.cuda.synchronize(dev)
    assert np.array_equal(dP.cpu().numpy(), P)
    return (dJ.cpu().numpy() if want_j else None), dK.cpu().numpy()


def _variants(P, G=None, seed=5):
    """The density stacks every workload runs, from its symmetric stack P (nD = 1 or 2) and its guess stack G."""
    nD, n = P.shape[0], P.shape[1]
    A = np.random.default_rng(seed).standard_normal((nD, n, n))
    A = A - A.transpose(0, 2, 1)
    two = P if nD == 2 else np.stack([P[0], 0.5 * P[0]])
    return [("symmetric", P), ("asym_1e-8", P + 1e-8 * A), ("asym_O(1)", P + A), ("symmetric_x1e3", 1e3 * P),
            ("mixed_asym_first", np.stack([two[0] + 1e-8 * A[0], two[1]])), ("mixed_asym_second", np.stack([two[0], two[1] + A[-1]]))] + \
        ([("guess", G)] if G is not None else [])


def _bitwise(got, ref, what):
    for a, b, name in zip(got, ref, "JK"):
        if a is None:
            continue
        assert np.array_equal(a, b), f"{what} {name}: max |general_dev - host| = {np.abs(a - b).max():.3e}"


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["n2_ccpvtz", "ne2_uhf_ccpvqz", "et100"])
def test_general_dev_bitwise_equals_host(name):
    flat, U, P, G = _case(name)
    assert 0.0 < np.abs(G - G.transpose(0, 2, 1)).max() <= 1e-15 * np.abs(G).max()
    host, dev = _ctx(flat, U), _ctx(flat, U)
    for what, Q in _variants(P, G):
        _bitwise(_general_dev(dev, Q), host.jk_direct(Q, TAU), f"{name} {what}")
        assert dev.counts()["evaluated_last_direct"] == host.counts()["evaluated_last_direct"], what
    Q = _variants(P)[2][1]
    _bitwise(_general_dev(dev, Q, want_j=False), host.jk_direct(Q, TAU), f"{name} K only")


@pytest.mark.gpu
def test_symmetric_density_within_the_default_bound_equals_jk_direct_dev():
    """max|P| <= 1 keeps the default pre-screening bound: the general entry point then runs exactly the build of tuna_jk_direct_dev."""
    import torch
    flat, U, P, G = _case("ne2_uhf_ccpvqz")
    P = P / np.abs(P).max()
    plain, general = _ctx(flat, U), _ctx(flat, U)
    dP = torch.from_numpy(P).cuda()
    dJ, dK = torch.empty_like(dP), torch.empty_like(dP)
    torch.cuda.synchronize()
    plain.jk_direct_dev(2, dP.data_ptr(), dJ.data_ptr(), dK.data_ptr(), TAU)
    torch.cuda.synchronize()
    _bitwise(_general_dev(general, P), (dJ.cpu().numpy(), dK.cpu().numpy()), "symmetric P")


@pytest.mark.gpu
def test_against_the_oracle_and_the_defect_of_the_symmetric_device_path(oracle):
    """N2/cc-pVTZ against the oracle's dense J/K (Cartesian tensor rotated with U).  On an O(1)-asymmetric P, tuna_jk_direct_dev drops
    K[A]; the general entry point does not."""
    import torch
    g = load_golden("n2_ccpvtz")
    flat, U, P, G = _case("n2_ccpvtz")
    E = oracle.cart_to_sph_eri(oracle.eri_fill(oracle_basis(oracle, g)), U)
    ctx = _ctx(flat, U)
    for what, Q in _variants(P):
        J, K = _general_dev(ctx, Q, tau=0.0)
        for d in range(Q.shape[0]):
            Jr, Kr = oracle.coulomb(Q[d], E), oracle.exchange(Q[d], E)
            scale = max(1.0, float(np.abs(Kr).max()))
            assert np.abs(J[d] - Jr).max() < 1e-11 * scale, (what, d)
            assert np.abs(K[d] - Kr).max() < 1e-11 * scale, (what, d)
    A = np.random.default_rng(17).standard_normal(P[0].shape)
    Q = (P[0] + A - A.T)[None]
    Kr = oracle.exchange(Q[0], E)
    old = _ctx(flat, U)
    dP = torch.from_numpy(Q).cuda()
    dJ, dK = torch.empty_like(dP), torch.empty_like(dP)
    torch.cuda.synchronize()
    old.jk_direct_dev(1, dP.data_ptr(), dJ.data_ptr(), dK.data_ptr(), 0.0)
    torch.cuda.synchronize()
    scale = max(1.0, float(np.abs(Kr).max()))
    assert np.abs(dK.cpu().numpy()[0] - Kr).max() > 1e-3 * scale
    assert np.abs(_general_dev(ctx, Q, tau=0.0)[1][0] - Kr).max() < 1e-11 * scale


@pytest.mark.gpu
def test_with_the_integral_store():
    """The store pass and the replayed builds of a context with the integral store equal the host call on one without it."""
    flat, U, P, G = _case("n2_ccpvtz")
    host, semi = _ctx(flat, U), _ctx(flat, U, budget=BIG)
    builds = [Q for _, Q in _variants(P)][1:3]
    for i, Q in enumerate(builds + builds + [builds[0]]):
        _bitwise(_general_dev(semi, Q), host.jk_direct(Q, TAU), f"build {i}")
    info = semi.integral_store_info()
    assert info["items"] > 0 and info["replayed_builds"] >= 2, info


@pytest.mark.gpu
@pytest.mark.parametrize("rank,nranks", [(1, 2), (3, 4)])
@pytest.mark.parametrize("name", ["n2_ccpvtz", "ne2_uhf_ccpvqz"])
def test_sharded_rank_on_one_device(name, rank, nranks):
    flat, U, P, G = _case(name)
    host, dev = _ctx(flat, U, shard=(rank, nranks)), _ctx(flat, U, shard=(rank, nranks))
    for what, Q in _variants(P):
        _bitwise(_general_dev(dev, Q), host.jk_direct(Q, TAU), f"rank {rank}/{nranks} {what}")


@pytest.mark.gpu
@pytest.mark.parametrize("n", [2, 4, 8])
def test_device_group(n):
    import tuna_b200
    if _gpus() < n:
        pytest.skip(f"needs {n} GPUs")
    flat, U, P, G = _case("n2_ccpvtz")
    solo = _ctx(flat, U)
    group = tuna_b200.DeviceGroup(list(range(n)))
    group.set_basis(*flat)
    group.set_transform(U)
    for what, Q in _variants(P):
        ref = solo.jk_direct(Q, TAU)
        _bitwise(group.jk_direct(Q, TAU), ref, f"group host {what}")
        _bitwise(_general_dev(group, Q), ref, f"group general_dev {what}")
    group.close()
    solo.close()


@pytest.mark.gpu
def test_per_component_kernel(monkeypatch):
    """TUNA_B200_DIRECT_ENGINE=generic (read at set_basis): FP64 atomics, so equal to the host call within round-off."""
    monkeypatch.setenv("TUNA_B200_DIRECT_ENGINE", "generic")
    flat, U, P, G = _case("n2_ccpvtz")
    host, dev = _ctx(flat, U), _ctx(flat, U)
    for what, Q in _variants(P):
        (J, K), (Jh, Kh) = _general_dev(dev, Q), host.jk_direct(Q, TAU)
        scale = max(1.0, float(np.abs(Kh).max()))
        assert np.abs(J - Jh).max() < 1e-11 * scale and np.abs(K - Kh).max() < 1e-11 * scale, what


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["n2_ccpvtz", "ne2_uhf_ccpvqz"])
def test_fock_builder_asymmetric_density(name):
    """FockBuilder.build of an asymmetric P runs the general device entry point; its J and K are those of the host tuna_jk_direct on the
    same shard (one rank: the whole build), as they were when that branch called it."""
    from tuna_b200.distributed import FockBuilder
    flat, U, P, G = _case(name)
    host, ctx = _ctx(flat, U), _ctx(flat, U)
    fb = FockBuilder(ctx, nD=P.shape[0], tau=TAU)
    for what, Q in _variants(P, G):
        if Q.shape[0] != P.shape[0] or "asym" not in what:      # stacks symmetric by the 1e-15 test take build_device, which did not change
            continue
        arg = Q[0] if Q.shape[0] == 1 else Q
        _bitwise(fb.build(arg), host.jk_direct(arg, TAU), f"FockBuilder {what}")
    ctx.set_stream(0)


@pytest.mark.gpu
def test_bad_arguments_leave_the_context_usable():
    import torch
    import tuna_b200
    from tuna_b200 import _lib
    lib = _lib.load()
    flat, U, P, G = _case("n2_ccpvtz")
    Q = _variants(P)[1][1]
    host, ctx = _ctx(flat, U), _ctx(flat, U)
    ref = host.jk_direct(Q, TAU)
    dP = torch.from_numpy(np.concatenate([Q] * 9)).cuda()
    dJ, dK = torch.empty_like(dP), torch.empty_like(dP)
    torch.cuda.synchronize()
    p, j, k = dP.data_ptr(), dJ.data_ptr(), dK.data_ptr()
    for nD, ptr in ((0, p), (9, p), (-1, p), (1, 0)):
        assert lib.tuna_jk_direct_general_dev(ctx._h, nD, ptr, j, k, TAU) == _lib.ERR_ARG, (nD, ptr)
    assert lib.tuna_jk_direct_general_dev(None, 1, p, j, k, TAU) == _lib.ERR_ARG
    bare = tuna_b200.Context(0)
    assert lib.tuna_jk_direct_general_dev(bare._h, 1, p, j, k, TAU) == _lib.ERR_STATE
    bare.set_basis(*flat)
    assert lib.tuna_jk_direct_general_dev(bare._h, 1, p, j, k, TAU) == _lib.ERR_STATE

    def group(ctxs, nD=1, ptr=p):
        ptrs = (ctypes.c_void_p * len(ctxs))(*[c._h.value for c in ctxs])
        return lib.tuna_jk_direct_group_general_dev(ptrs, len(ctxs), nD, ptr, j, k, TAU)

    assert group([ctx, ctx]) == _lib.ERR_ARG                       # a repeated context
    assert group([ctx], nD=9) == _lib.ERR_ARG and group([ctx], ptr=0) == _lib.ERR_ARG
    assert lib.tuna_jk_direct_group_general_dev(None, 1, 1, p, j, k, TAU) == _lib.ERR_ARG
    twin = _ctx(flat, U, shard=(1, 2))                             # a second context on device 0
    assert group([ctx, twin]) == _lib.ERR_ARG
    ctx.set_shard(0, 2)
    assert group([ctx]) == _lib.ERR_STATE                          # sharded as (0, 2) in a group of one
    ctx.set_shard(0, 1)
    assert group([bare]) == _lib.ERR_STATE                         # no transform
    torch.cuda.synchronize()
    _bitwise(_general_dev(ctx, Q), ref, "after the errors")
    ptrs = (ctypes.c_void_p * 1)(ctx._h.value)
    dQ = torch.from_numpy(Q).cuda()
    out = [torch.empty_like(dQ), torch.empty_like(dQ)]
    torch.cuda.synchronize()
    assert lib.tuna_jk_direct_group_general_dev(ptrs, 1, 1, dQ.data_ptr(), out[0].data_ptr(), out[1].data_ptr(), TAU) == _lib.OK
    torch.cuda.synchronize()
    _bitwise((out[0].cpu().numpy(), out[1].cpu().numpy()), ref, "group of one")
    for c in (twin, bare, ctx, host):
        c.close()
