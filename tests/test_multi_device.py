"""Direct J/K of one Fock build over several GPUs of ONE process (tuna_jk_direct_group, tuna_b200.DeviceGroup, configure(devices=...)).

CPU: parsing of configure(devices=...) / TUNA_B200_DEVICES, and no CPU fallback behind DeviceGroup.
GPU (`-m gpu`, each group size N skipped where the box has fewer devices): the group's J and K must be BITWISE equal to one fresh
Context on devices[0] (the ranks' 64-bit integer accumulators are summed before the conversion to FP64); with the per-component
kernel (FP64 atomics) within 1e-11 max(1, max|K|).  Invalid groups raise TunaError and leave the contexts usable.  End to end, the
restated SCF (oracle/scf_oracle.py) through the installed provider's calculate_coulomb_matrix / calculate_exchange_matrix with all
devices configured reproduces the recorded energy and iteration count, and the one-device energy exactly."""
import ctypes
import json
import os
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.join(HERE, "golden"))

from util import basis_objects, load_golden  # noqa: E402

SIZES = [1, 2, 4, 8]


def _gpus():
    import torch
    return torch.cuda.device_count() if torch.cuda.is_available() else 0


def _devices(n):
    if _gpus() < n:
        pytest.skip(f"needs {n} GPUs")
    return list(range(n))


@pytest.fixture
def provider_state():
    """configure() changes module state of tuna_b200.provider: restore it after the test."""
    from tuna_b200 import provider
    saved = dict(provider._settings), provider._devices
    yield provider
    provider._settings.clear()
    provider._settings.update(saved[0])
    provider._devices = saved[1]


# ---------------------------------------------------------------------------------------------------------------------------------
# CPU
# ---------------------------------------------------------------------------------------------------------------------------------
def test_configure_devices(provider_state):
    p = provider_state
    import tuna_b200
    tuna_b200.configure(devices=[3, 1])
    assert p.configured_devices() == [3, 1] and p._settings["device"] == 3
    tuna_b200.configure(devices="0, 2,5")
    assert p.configured_devices() == [0, 2, 5] and p._settings["device"] == 0
    tuna_b200.configure(devices="all")
    assert p._devices == "all" and p._settings["device"] == 0
    for bad in ([1, 1], "0,0", [-1], "0,-2", [], "x"):
        with pytest.raises(tuna_b200.TunaError):
            tuna_b200.configure(devices=bad)
    with pytest.raises(tuna_b200.TunaError):
        tuna_b200.configure(device=0, devices=[0, 1])
    tuna_b200.configure(device=2)
    by_device = dict(p._settings), p.configured_devices()
    tuna_b200.configure(devices=[2])
    assert (dict(p._settings), p.configured_devices()) == by_device == ({**by_device[0], "device": 2}, [2])


def _env_probe(value):
    env = {k: v for k, v in os.environ.items() if not k.startswith("TUNA_B200_")}
    if value is not None:
        env["TUNA_B200_DEVICES"] = value
    code = ("import json\nfrom tuna_b200 import provider as p\n"
            "print(json.dumps([p._settings, p._devices]))")
    return subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, cwd=ROOT, env=env, timeout=300)


def test_devices_environment_variable():
    r = _env_probe(None)
    assert r.returncode == 0, r.stderr
    assert json.loads(r.stdout) == [{"mode": "auto", "device": 0, "stored_fraction": 0.40, "tau": 1e-16}, None]
    r = _env_probe("2,0")
    assert r.returncode == 0, r.stderr
    settings, devices = json.loads(r.stdout)
    assert devices == [2, 0] and settings["device"] == 2
    r = _env_probe("all")
    assert r.returncode == 0, r.stderr
    settings, devices = json.loads(r.stdout)
    assert devices == "all" and settings["device"] == 0
    r = _env_probe("1,1")
    assert r.returncode != 0 and "TunaError" in r.stderr


def test_device_group_rejects_repeated_devices():
    import tuna_b200
    with pytest.raises(tuna_b200.TunaError):
        tuna_b200.DeviceGroup([0, 0])
    with pytest.raises(tuna_b200.TunaError):
        tuna_b200.DeviceGroup([])


def test_device_group_without_gpu():
    if _gpus() > 0:
        pytest.skip("GPU present")
    import tuna_b200
    with pytest.raises(tuna_b200.TunaError):
        tuna_b200.DeviceGroup([0, 1])


# ---------------------------------------------------------------------------------------------------------------------------------
# GPU
# ---------------------------------------------------------------------------------------------------------------------------------
def _case(name):
    """(flattened basis, U, densities) of a named case."""
    from tuna_b200 import workloads as w
    from tuna_b200.basis import flatten, from_arrays
    if name.startswith("et"):
        b = w.even_tempered_diatomic(int(name[2:]))
        bfs = from_arrays(b["origins"], b["lmn"], b["nprim"], b["exps"], b["raw_coefs"])
        return flatten(bfs), np.eye(len(bfs)), w.fixed_density(len(bfs))
    g = load_golden(name)
    U = np.array(g["U"])
    if name == "ne2_uhf_ccpvqz":
        P = np.stack([np.array(g["P_alpha_final"]), np.array(g["P_beta_final"])])
    else:
        P = w.fixed_density(U.shape[0])
    return flatten(basis_objects(g)), U, P


def _single(flat, U, device):
    import tuna_b200
    ctx = tuna_b200.Context(device)
    ctx.set_basis(*flat)
    ctx.set_transform(U)
    return ctx


def _group(flat, U, devices):
    import tuna_b200
    group = tuna_b200.DeviceGroup(devices)
    group.set_basis(*flat)
    group.set_transform(U)
    return group


def _assert_bitwise(got, ref):
    for a, b, what in zip(got, ref, "JK"):
        assert np.array_equal(a, b), f"{what}: max |group - single| = {np.abs(a - b).max():.3e}"


@pytest.mark.gpu
@pytest.mark.parametrize("n", SIZES)
@pytest.mark.parametrize("name", ["n2_ccpvtz", "ne2_uhf_ccpvqz", "et100", "et400"])
def test_group_bitwise_equals_one_device(name, n):
    devices = _devices(n)
    flat, U, P = _case(name)
    solo, group = _single(flat, U, devices[0]), _group(flat, U, devices)
    ref = solo.jk_direct(P, 1e-16)
    _assert_bitwise(group.jk_direct(P, 1e-16), ref)
    _assert_bitwise(group.jk_direct(P, 1e-16), ref)                 # a second build on the same group
    assert group.counts()["evaluated_last_direct"] == solo.counts()["evaluated_last_direct"]
    ref = solo.jk_direct(P, 1e-10)                                  # a direct SCF's threshold: the ranks drop what one device drops
    _assert_bitwise(group.jk_direct(P, 1e-10), ref)
    assert group.counts()["evaluated_last_direct"] == solo.counts()["evaluated_last_direct"]
    if name == "ne2_uhf_ccpvqz":
        from tuna_b200 import workloads as w
        g = load_golden(name)
        J, K = group.jk_direct(w.fixed_density(int(g["nbf"])), 1e-16)
        assert np.abs(J - g["Jfix"]).max() < 1e-11 and np.abs(K - g["Kfix"]).max() < 1e-11
    group.close()
    solo.close()


@pytest.mark.gpu
@pytest.mark.parametrize("n", SIZES)
def test_group_several_passes_asymmetric_density_and_device_buffers(n):
    """nD = 5 (several passes of the engine), a density with a 1e-8 antisymmetric part (symmetric / antisymmetric split), and the _dev
    entry point against tuna_jk_direct_dev, on N2/cc-pVTZ."""
    import torch
    devices = _devices(n)
    flat, U, P = _case("n2_ccpvtz")
    nbf = U.shape[0]
    rng = np.random.default_rng(7)
    stack = np.stack([P] + [(A + A.T) / 2 for A in rng.standard_normal((4, nbf, nbf))])
    A = rng.standard_normal((nbf, nbf))
    asym = P + 1e-8 * (A - A.T)
    solo, group = _single(flat, U, devices[0]), _group(flat, U, devices)
    _assert_bitwise(group.jk_direct(stack, 1e-16), solo.jk_direct(stack, 1e-16))
    _assert_bitwise(group.jk_direct(asym, 1e-16), solo.jk_direct(asym, 1e-16))
    dev = torch.device("cuda", devices[0])
    dP = torch.from_numpy(stack[:3]).to(dev)
    out = [torch.empty_like(dP) for _ in range(4)]
    torch.cuda.synchronize(dev)                                    # the contexts' own streams do not order after torch's
    solo.jk_direct_dev(3, dP.data_ptr(), out[0].data_ptr(), out[1].data_ptr(), 1e-16)
    group.jk_direct_dev(3, dP.data_ptr(), out[2].data_ptr(), out[3].data_ptr(), 1e-16)
    torch.cuda.synchronize(dev)
    _assert_bitwise((out[2].cpu().numpy(), out[3].cpu().numpy()), (out[0].cpu().numpy(), out[1].cpu().numpy()))
    group.close()
    solo.close()


@pytest.mark.gpu
def test_group_errors_leave_the_contexts_usable():
    import tuna_b200
    from tuna_b200 import _lib
    devices = list(range(min(_gpus(), 2))) or _devices(1)
    flat, U, P = _case("n2_ccpvtz")
    solo, group = _single(flat, U, devices[0]), _group(flat, U, devices)
    ref = solo.jk_direct(P, 1e-16)
    lib = _lib.load()
    nbf = U.shape[0]
    J, K = np.empty((nbf, nbf)), np.empty((nbf, nbf))

    def call(ctxs):
        ptrs = (ctypes.c_void_p * len(ctxs))(*[c._h.value for c in ctxs])
        rc = lib.tuna_jk_direct_group(ptrs, len(ctxs), 1, _lib._dp(P), _lib._dp(J), _lib._dp(K), 1e-16)
        return rc, lib.tuna_last_error(ctxs[0]._h).decode()

    twin = _single(flat, U, devices[0])                            # a second context on devices[0]
    twin.set_shard(1, 2)
    first = group.contexts[0]
    first.set_shard(0, 2)
    assert call([first, twin])[0] == _lib.ERR_ARG
    assert call([first, first])[0] == _lib.ERR_ARG
    first.set_shard(0, len(devices))
    with pytest.raises(tuna_b200.TunaError):
        tuna_b200.DeviceGroup([devices[0], devices[0]])
    last = group.contexts[-1]
    last.set_shard(0, 1)                                           # not (rank, N)
    if len(devices) == 1:
        last.set_shard(0, 2)
    with pytest.raises(tuna_b200.TunaError, match="sharded"):
        group.jk_direct(P, 1e-16)
    last.set_shard(len(devices) - 1, len(devices))
    _assert_bitwise(group.jk_direct(P, 1e-16), ref)
    if len(devices) > 1:
        other, _, _ = _case("ne2_uhf_ccpvqz")
        last.set_basis(*other)
        last.set_transform(np.eye(last.ncart))
        with pytest.raises(tuna_b200.TunaError, match="different basis"):
            group.jk_direct(P, 1e-16)
        last.set_basis(*flat)
        last.set_transform(U)
        _assert_bitwise(group.jk_direct(P, 1e-16), ref)
    twin.close()
    group.close()
    solo.close()


def _generic_child(n):
    """Per-component kernel (TUNA_B200_DIRECT_ENGINE=generic, read at set_basis): group vs single context."""
    flat, U, P = _case("n2_ccpvtz")
    solo, group = _single(flat, U, 0), _group(flat, U, list(range(n)))
    (Js, Ks), (Jg, Kg) = solo.jk_direct(P, 1e-16), group.jk_direct(P, 1e-16)
    print("RESULT " + json.dumps({"dJ": float(np.abs(Jg - Js).max()), "dK": float(np.abs(Kg - Ks).max()), "scale": max(1.0, float(np.abs(Ks).max()))}))


@pytest.mark.gpu
@pytest.mark.parametrize("n", SIZES)
def test_group_with_the_per_component_kernel(n):
    _devices(n)
    env = dict(os.environ, TUNA_B200_DIRECT_ENGINE="generic")
    r = subprocess.run([sys.executable, os.path.abspath(__file__), "generic", str(n)], capture_output=True, text=True, cwd=ROOT, env=env, timeout=900)
    lines = [line for line in r.stdout.splitlines() if line.startswith("RESULT ")]
    assert r.returncode == 0 and lines, r.stderr[-3000:]
    res = json.loads(lines[-1][len("RESULT "):])
    assert res["dJ"] < 1e-11 * res["scale"] and res["dK"] < 1e-11 * res["scale"], res


@pytest.mark.gpu
@pytest.mark.parametrize("name", ["ne2_uhf_ccpvqz", "et100"])
def test_provider_scf_over_all_devices(name, provider_state, tmp_path, monkeypatch):
    import ref_harness as rh
    from oracle import scf_oracle
    from test_reference_on_gpu import provider_eri, provider_jk, run_reference
    import tuna_b200
    if _gpus() < 2:
        pytest.skip("needs 2 GPUs")
    g = load_golden(name)
    energies = {}
    for devices in ([0], "all"):
        tuna_b200.configure(mode="direct", devices=devices)
        eri = provider_eri(tuna_b200, g)
        energy, iterations, _ = scf_oracle.run_scf(provider_jk(tuna_b200, eri, []), g)
        assert abs(energy - float(g["energy"])) < 1e-10 and iterations == int(g["n_iterations"]), (devices, energy, iterations)
        energies[str(devices)] = energy
        if devices == "all":
            assert eri._group is not None and eri._group.devices == list(range(_gpus()))
    assert energies["all"] == energies["[0]"]
    if not rh.reference_available():
        return
    line = str(g["line"])
    if "{basis_file}" in line:
        from tuna_b200 import workloads
        (tmp_path / "ET100.TUNA").write_text(workloads.even_tempered_basis_file(100))
        monkeypatch.chdir(tmp_path)
        line = line.format(basis_file="ET100.TUNA")
    energy, _ = run_reference(line, "direct", int(g["nbf"]))
    assert abs(energy - float(g["energy"])) < 1e-10, energy


if __name__ == "__main__":
    if sys.argv[1] == "generic":
        sys.path.insert(0, ROOT)
        _generic_child(int(sys.argv[2]))
