"""ctypes binding of libtuna_b200.so (C ABI declared in include/tuna_b200.h).

There is no CPU fallback: if the CUDA library is missing or no CUDA device is usable, every entry point
raises.  Build the library in-tree with `python -m tuna_b200.build` (nvcc, sm_100a).
"""
import ctypes
import os

import numpy as np

_HERE = os.path.dirname(os.path.abspath(__file__))
LIB_PATH = os.environ.get("TUNA_B200_LIB") or os.path.join(_HERE, "libtuna_b200.so")      # override: development builds only

OK, ERR_ARG, ERR_NOMEM, ERR_CUDA, ERR_STATE = 0, 1, 2, 3, 4

EXPORTS = [
    "tuna_ctx_create", "tuna_ctx_destroy", "tuna_last_error", "tuna_set_stream", "tuna_set_basis", "tuna_set_transform",
    "tuna_eri_fill_cart", "tuna_eri_cart_to_sph", "tuna_eri_fill_sph", "tuna_eri_download", "tuna_eri_upload", "tuna_eri_single", "tuna_schwarz",
    "tuna_jk_stored", "tuna_jk_stored_dev", "tuna_jk_direct", "tuna_jk_direct_dev", "tuna_set_shard", "tuna_get_counts",
    "tuna_last_kernel_ms", "tuna_algorithmic_flops", "tuna_fp64_peak_probe", "tuna_eri_transform", "tuna_eri_transform_dev",
    "tuna_eri_transform_spin_blocked", "tuna_one_electron", "tuna_cross_overlap", "tuna_jk_direct_group", "tuna_jk_direct_group_dev",
    "tuna_set_integral_store", "tuna_integral_store_info", "tuna_jk_direct_general_dev", "tuna_jk_direct_group_general_dev",
]

_lib = None


class TunaError(Exception):
    """Stand-in for the reference's TunaError (TUNA/tuna_util.py:916-944) when the reference is not importable.
    `provider.install()` swaps in the reference's own class so callers can catch the type they expect."""


error_class = TunaError


def load() -> ctypes.CDLL:
    """Load the CUDA library; raises (never falls back) if it has not been built."""
    global _lib
    if _lib is not None:
        return _lib
    if not os.path.exists(LIB_PATH):
        raise ImportError(f"{LIB_PATH} not found: the CUDA extension must be built (python -m tuna_b200.build); "
                          "tuna_b200 has no CPU fallback")
    lib = ctypes.CDLL(LIB_PATH)
    c_dp, c_ip, c_lp = ctypes.POINTER(ctypes.c_double), ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int64)
    vp, ci, cd = ctypes.c_void_p, ctypes.c_int, ctypes.c_double
    sig = {
        "tuna_ctx_create": (ci, [ci, ctypes.POINTER(vp)]),
        "tuna_ctx_destroy": (ci, [vp]),
        "tuna_last_error": (ctypes.c_char_p, [vp]),
        "tuna_set_stream": (ci, [vp, vp]),
        "tuna_set_basis": (ci, [vp, ci, c_dp, c_ip, c_ip, c_lp, c_dp, c_dp]),
        "tuna_set_transform": (ci, [vp, ci, c_dp]),
        "tuna_eri_fill_cart": (ci, [vp]),
        "tuna_eri_cart_to_sph": (ci, [vp, ci]),
        "tuna_eri_fill_sph": (ci, [vp]),
        "tuna_eri_download": (ci, [vp, ci, c_dp]),
        "tuna_eri_upload": (ci, [vp, ci, c_dp]),
        "tuna_eri_single": (ci, [vp, ci, ci, ci, ci, c_dp]),
        "tuna_schwarz": (ci, [vp, c_dp]),
        "tuna_jk_stored": (ci, [vp, ci, c_dp, c_dp, c_dp]),
        "tuna_jk_stored_dev": (ci, [vp, ci, vp, vp, vp]),
        "tuna_jk_direct": (ci, [vp, ci, c_dp, c_dp, c_dp, cd]),
        "tuna_jk_direct_dev": (ci, [vp, ci, vp, vp, vp, cd]),
        "tuna_set_shard": (ci, [vp, ci, ci]),
        "tuna_get_counts": (ci, [vp, c_lp]),
        "tuna_last_kernel_ms": (ci, [vp, ci, ctypes.POINTER(ctypes.c_float)]),
        "tuna_algorithmic_flops": (ci, [vp, c_dp, c_dp]),
        "tuna_fp64_peak_probe": (ci, [vp, c_dp]),
        "tuna_eri_transform": (ci, [vp, ci, c_dp, ci, c_dp, ci, c_dp, ci, c_dp]),
        "tuna_eri_transform_dev": (ci, [vp, ci, vp, ci, vp, ci, vp, ci, vp]),
        "tuna_eri_transform_spin_blocked": (ci, [vp, ci, c_dp, ci, c_dp, ci, c_dp]),
        "tuna_one_electron": (ci, [vp, ci, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp, c_dp]),
        "tuna_cross_overlap": (ci, [vp] + [ci, c_dp, c_ip, c_ip, c_lp, c_dp, c_dp] * 2 + [c_dp]),
        "tuna_jk_direct_group": (ci, [ctypes.POINTER(vp), ci, ci, c_dp, c_dp, c_dp, cd]),
        "tuna_jk_direct_group_dev": (ci, [ctypes.POINTER(vp), ci, ci, vp, vp, vp, cd]),
        "tuna_set_integral_store": (ci, [vp, ctypes.c_int64]),
        "tuna_integral_store_info": (ci, [vp, c_lp]),
        "tuna_jk_direct_general_dev": (ci, [vp, ci, vp, vp, vp, cd]),
        "tuna_jk_direct_group_general_dev": (ci, [ctypes.POINTER(vp), ci, ci, vp, vp, vp, cd]),
    }
    for name, (res, args) in sig.items():
        fn = getattr(lib, name)
        fn.restype, fn.argtypes = res, args
    _lib = lib
    return lib


def _dp(a):
    return a.ctypes.data_as(ctypes.POINTER(ctypes.c_double)) if a is not None else None


def _host_tensor(shape):
    """Result buffer for the large device->host copies (n^4 doubles).  Page-locked memory from torch's caching host
    allocator (plumbing: the copy then runs at PCIe/C2C speed instead of through the driver's staging buffers and the
    buffer is not page-faulted in by the copy); the ndarray keeps the torch tensor alive.  Plain np.empty when pinning fails."""
    if int(np.prod(shape)) * 8 >= (1 << 22) and os.environ.get("TUNA_B200_PINNED_RESULTS", "1") != "0":
        try:
            import torch
            return torch.empty(tuple(shape), dtype=torch.float64, pin_memory=True).numpy()
        except Exception:
            pass
    return np.empty(shape)


class Context:
    """One (device, geometry, basis): owns the pair table and any device-resident tensors."""

    KERNEL_ERI, KERNEL_SPH, KERNEL_JK_STORED, KERNEL_JK_DIRECT, KERNEL_MO_TRANSFORM, KERNEL_ONE_ELECTRON = 0, 1, 2, 3, 4, 5

    def __init__(self, device: int = 0):
        self._lib = load()
        h = ctypes.c_void_p()
        rc = self._lib.tuna_ctx_create(device, ctypes.byref(h))
        self._h = h
        if rc:
            msg = self._lib.tuna_last_error(h).decode() if h else "allocation failed"
            if h:
                self._lib.tuna_ctx_destroy(h)
                self._h = None
            self._raise(rc, msg)
        self.device = device
        self.ncart = 0
        self.nbf = 0
        self.n_stored = 0
        self.basis_flat = None      # the arrays of set_basis and the U of set_transform, for a DeviceGroup over the same basis
        self.U = None

    # -- error mapping: MemoryError like pyx:1120/1290, everything else the reference's TunaError ------------
    def _raise(self, rc, msg=None):
        msg = msg if msg is not None else self._lib.tuna_last_error(self._h).decode()
        if rc == ERR_NOMEM:
            raise MemoryError(msg)
        raise error_class(f"tuna_b200: {msg}")

    def _ck(self, rc):
        if rc:
            self._raise(rc)

    def close(self):
        if getattr(self, "_h", None):
            self._lib.tuna_ctx_destroy(self._h)
            self._h = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def set_stream(self, cuda_stream: int):
        self._ck(self._lib.tuna_set_stream(self._h, ctypes.c_void_p(cuda_stream)))

    def set_basis(self, origins_z, lmn, nprim, exps, coef_eff):
        oz = np.ascontiguousarray(origins_z, dtype=np.float64)
        lmn = np.ascontiguousarray(lmn, dtype=np.int32).reshape(-1, 3)
        nprim = np.ascontiguousarray(nprim, dtype=np.int32)
        off = np.concatenate([[0], np.cumsum(nprim)[:-1]]).astype(np.int64)
        exps = np.ascontiguousarray(exps, dtype=np.float64)
        ce = np.ascontiguousarray(coef_eff, dtype=np.float64)
        if not (len(oz) == len(lmn) == len(nprim)) or len(exps) != int(nprim.sum()) or len(ce) != len(exps):
            raise error_class("tuna_b200: inconsistent basis arrays")
        i32p, i64p = ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int64)
        self._ck(self._lib.tuna_set_basis(self._h, len(oz), _dp(oz), lmn.ctypes.data_as(i32p), nprim.ctypes.data_as(i32p),
                                          off.ctypes.data_as(i64p), _dp(exps), _dp(ce)))
        self.ncart, self.nbf, self.n_stored = len(oz), 0, 0
        self.lmn = lmn
        self.basis_flat, self.U = (oz, lmn, nprim, exps, ce), None

    def set_transform(self, U):
        U = np.ascontiguousarray(U, dtype=np.float64)
        if U.ndim != 2 or U.shape[1] != self.ncart:
            raise error_class(f"tuna_b200: transformation matrix has shape {U.shape}, expected (nbf, {self.ncart})")
        self._ck(self._lib.tuna_set_transform(self._h, U.shape[0], _dp(U)))
        self.nbf = U.shape[0]
        self.U = U

    def eri_fill_cart(self):
        self._ck(self._lib.tuna_eri_fill_cart(self._h))

    def eri_cart_to_sph(self, keep_cart: bool = False):
        self._ck(self._lib.tuna_eri_cart_to_sph(self._h, int(keep_cart)))
        self.n_stored = self.nbf

    def eri_fill_sph(self):
        """The spherical tensor as the stored tensor, without a Cartesian tensor on the engine path (tuna_eri_fill_sph)."""
        self._ck(self._lib.tuna_eri_fill_sph(self._h))
        self.n_stored = self.nbf

    def eri_download(self, which: int, out=None):
        n = self.ncart if which == 0 else self.n_stored
        if out is None:
            out = _host_tensor((n, n, n, n))
        if out.shape != (n, n, n, n) or out.dtype != np.float64 or not out.flags.c_contiguous:
            raise error_class("tuna_b200: output tensor must be C-contiguous float64 of shape (n, n, n, n)")
        self._ck(self._lib.tuna_eri_download(self._h, which, _dp(out)))
        return out

    def eri_upload(self, tensor):
        t = np.ascontiguousarray(tensor, dtype=np.float64)
        if t.ndim != 4 or len(set(t.shape)) != 1:
            raise error_class("tuna_b200: stored tensor must have shape (n, n, n, n)")
        self._ck(self._lib.tuna_eri_upload(self._h, t.shape[0], _dp(t)))
        self.n_stored = t.shape[0]

    def eri_single(self, i, j, k, l) -> float:
        out = ctypes.c_double()
        self._ck(self._lib.tuna_eri_single(self._h, i, j, k, l, ctypes.byref(out)))
        return out.value

    def schwarz(self):
        out = np.zeros((self.ncart, self.ncart))
        self._ck(self._lib.tuna_schwarz(self._h, _dp(out)))
        return out

    def eri_transform(self, C1, C2=None, so_layout=False, eri=None):
        """AO -> MO (tuna_ci.py:204-255) or spin-orbital (tuna_ci.py:143-193) transformation.  eri = None uses the
        resident stored tensor; C1 (n, n1), C2 (n, n2) (default C2 = C1).  Returns [p][r][q][s] (MO) or [p][q][r][s] (SO)."""
        C1 = np.ascontiguousarray(C1, dtype=np.float64)
        C2 = C1 if C2 is None else np.ascontiguousarray(C2, dtype=np.float64)
        if eri is not None:
            eri = np.ascontiguousarray(eri, dtype=np.float64)
            if eri.ndim != 4 or len(set(eri.shape)) != 1:
                raise error_class("tuna_b200: ERI tensor must have shape (n, n, n, n)")
            n = eri.shape[0]
        else:
            n = self.n_stored
            if n == 0:
                raise error_class("tuna_b200: no stored tensor is resident")
        if C1.ndim != 2 or C2.ndim != 2 or C1.shape[0] != n or C2.shape[0] != n:
            raise error_class(f"tuna_b200: MO coefficient matrices must have {n} rows, got {C1.shape} and {C2.shape}")
        n1, n2 = C1.shape[1], C2.shape[1]
        out = _host_tensor((n2, n1, n2, n1) if so_layout else (n2, n2, n1, n1))
        self._ck(self._lib.tuna_eri_transform(self._h, n, _dp(eri), n1, _dp(C1), n2, _dp(C2), int(bool(so_layout)), _dp(out)))
        return out

    def eri_transform_spin_blocked(self, C1, C2=None, so_layout=True):
        """Spin-orbital transformation of the spin-blocked tensor np.kron(np.eye(2), np.kron(np.eye(2), E).T) (tuna_ci.py:564-570), the
        spin-blocked tensor (16 n^4 doubles) being formed on the device from the resident stored tensor E.  C1, C2: (2n, n_so)."""
        C1 = np.ascontiguousarray(C1, dtype=np.float64)
        C2 = C1 if C2 is None else np.ascontiguousarray(C2, dtype=np.float64)
        n = self.n_stored
        if n == 0:
            raise error_class("tuna_b200: no stored tensor is resident")
        if C1.ndim != 2 or C2.ndim != 2 or C1.shape[0] != 2 * n or C2.shape[0] != 2 * n:
            raise error_class(f"tuna_b200: spin-blocked coefficient matrices must have {2 * n} rows, got {C1.shape} and {C2.shape}")
        n1, n2 = C1.shape[1], C2.shape[1]
        out = _host_tensor((n2, n1, n2, n1) if so_layout else (n2, n2, n1, n1))
        self._ck(self._lib.tuna_eri_transform_spin_blocked(self._h, n1, _dp(C1), n2, _dp(C2), int(bool(so_layout)), _dp(out)))
        return out

    def eri_transform_dev(self, n, dT, n1, dC1, n2, dC2, so_layout, d_out):
        self._ck(self._lib.tuna_eri_transform_dev(self._h, n, ctypes.c_void_p(dT), n1, ctypes.c_void_p(dC1), n2, ctypes.c_void_p(dC2),
                                                  int(bool(so_layout)), ctypes.c_void_p(d_out)))

    def one_electron(self, atom_z, atom_charge, dipole_origin):
        """(S, T, V_NE, D[3], Q[3]) of the current basis in the Cartesian basis (tuna_integral.calculate_one_electron_integrals, pyx:282-445)."""
        az = np.ascontiguousarray(atom_z, dtype=np.float64)
        ac = np.ascontiguousarray(atom_charge, dtype=np.float64)
        og = np.ascontiguousarray(dipole_origin, dtype=np.float64)
        if az.ndim != 1 or az.shape != ac.shape or og.shape != (3,) or len(az) == 0:
            raise error_class("tuna_b200: atoms must be given as equally long z / charge vectors and the origin as 3 numbers")
        n = self.ncart
        # page-locked result buffers above 4 MB (87 MB of results at ncart 1102: 55 ms into pageable memory, under 3 ms into pinned)
        S, T, V, D, Q = _host_tensor((n, n)), _host_tensor((n, n)), _host_tensor((n, n)), _host_tensor((3, n, n)), _host_tensor((3, n, n))
        self._ck(self._lib.tuna_one_electron(self._h, len(az), _dp(az), _dp(ac), _dp(og), _dp(S), _dp(T), _dp(V), _dp(D), _dp(Q)))
        return S, T, V, D, Q

    def cross_overlap(self, flat_1, flat_2):
        """S12[i, j] = <bf_1[i] | bf_2[j]> for two flattened bases (origins_z, lmn, nprim, exps, coef_eff) (pyx:626-778)."""
        i32p, i64p = ctypes.POINTER(ctypes.c_int32), ctypes.POINTER(ctypes.c_int64)
        args, keep = [], []
        for oz, lmn, nprim, exps, ce in (flat_1, flat_2):
            oz = np.ascontiguousarray(oz, dtype=np.float64)
            lmn = np.ascontiguousarray(lmn, dtype=np.int32).reshape(-1, 3)
            nprim = np.ascontiguousarray(nprim, dtype=np.int32)
            off = np.concatenate([[0], np.cumsum(nprim)[:-1]]).astype(np.int64)
            exps = np.ascontiguousarray(exps, dtype=np.float64)
            ce = np.ascontiguousarray(ce, dtype=np.float64)
            if not (len(oz) == len(lmn) == len(nprim)) or len(oz) == 0 or len(exps) != int(nprim.sum()) or len(ce) != len(exps):
                raise error_class("tuna_b200: inconsistent basis arrays")
            keep.append((oz, lmn, nprim, off, exps, ce))
            args += [len(oz), _dp(oz), lmn.ctypes.data_as(i32p), nprim.ctypes.data_as(i32p), off.ctypes.data_as(i64p), _dp(exps), _dp(ce)]
        out = np.empty((args[0], args[7]))
        self._ck(self._lib.tuna_cross_overlap(self._h, *args, _dp(out)))
        return out

    def _jk(self, fn, P, n, want_j, want_k, *extra):
        P = np.ascontiguousarray(P, dtype=np.float64)
        single = P.ndim == 2
        Ps = P[None] if single else P
        if Ps.ndim != 3 or Ps.shape[1:] != (n, n):
            raise error_class(f"tuna_b200: density matrix has shape {P.shape}, expected ({n}, {n})")
        J = np.empty_like(Ps) if want_j else None
        K = np.empty_like(Ps) if want_k else None
        self._ck(fn(self._h, Ps.shape[0], _dp(Ps), _dp(J), _dp(K), *extra))
        if single:
            return (J[0] if want_j else None), (K[0] if want_k else None)
        return J, K

    def jk_stored(self, P, want_j=True, want_k=True):
        """J_ij = sum_kl (ij|kl) P_kl, K_ij = sum_kl (il|kj) P_kl from the resident tensor (tuna_scf.py:27-72)."""
        return self._jk(self._lib.tuna_jk_stored, P, self.n_stored, want_j, want_k)

    def jk_direct(self, P, tau=1e-16, want_j=True, want_k=True):
        return self._jk(self._lib.tuna_jk_direct, P, self.nbf, want_j, want_k, ctypes.c_double(tau))

    def jk_stored_dev(self, nD, dP, dJ, dK):
        self._ck(self._lib.tuna_jk_stored_dev(self._h, nD, ctypes.c_void_p(dP), ctypes.c_void_p(dJ), ctypes.c_void_p(dK)))

    def jk_direct_dev(self, nD, dP, dJ, dK, tau=1e-16):
        self._ck(self._lib.tuna_jk_direct_dev(self._h, nD, ctypes.c_void_p(dP), ctypes.c_void_p(dJ), ctypes.c_void_p(dK), tau))

    def jk_direct_general_dev(self, nD, dP, dJ, dK, tau=1e-16):
        """jk_direct on device buffers: nD (1-8) densities of any real P at dP, J and K (either may be 0) written to dJ and dK, all
        on this context's device, enqueued on its stream.  Bitwise equal to jk_direct for the same P.  Synchronises the stream once,
        to read back max|P| and max|P - P^T|, which decide the screening bound and the symmetric / antisymmetric split
        (tuna_jk_direct_general_dev)."""
        self._ck(self._lib.tuna_jk_direct_general_dev(self._h, nD, ctypes.c_void_p(dP), ctypes.c_void_p(dJ), ctypes.c_void_p(dK),
                                                      ctypes.c_double(tau)))

    def set_shard(self, rank, nranks):
        self._ck(self._lib.tuna_set_shard(self._h, rank, nranks))

    def set_integral_store(self, budget_bytes: int):
        """Semi-direct J/K: keep up to budget_bytes of the engine's integrals on the device and replay them in later direct builds
        (0 = off, the default).  J and K stay bitwise equal to the direct build (tuna_set_integral_store)."""
        self._ck(self._lib.tuna_set_integral_store(self._h, int(budget_bytes)))

    def integral_store_info(self) -> dict:
        c = np.zeros(4, dtype=np.int64)
        self._ck(self._lib.tuna_integral_store_info(self._h, c.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))))
        return dict(zip(["bytes", "items", "items_last_build", "replayed_builds"], (int(x) for x in c)))

    def counts(self) -> dict:
        c = np.zeros(8, dtype=np.int64)
        self._ck(self._lib.tuna_get_counts(self._h, c.ctypes.data_as(ctypes.POINTER(ctypes.c_int64))))
        keys = ["ao_pairs", "unique_quartets", "surviving_quartets", "primitive_quartets", "evaluated_last_direct", "launches", "ncart", "nbf"]
        return dict(zip(keys, (int(x) for x in c)))

    def last_kernel_ms(self, which: int) -> float:
        ms = ctypes.c_float()
        self._ck(self._lib.tuna_last_kernel_ms(self._h, which, ctypes.byref(ms)))
        return ms.value

    def algorithmic_flops(self):
        a, b = ctypes.c_double(), ctypes.c_double()
        self._ck(self._lib.tuna_algorithmic_flops(self._h, ctypes.byref(a), ctypes.byref(b)))
        return a.value, b.value

    def fp64_peak_probe(self) -> float:
        t = ctypes.c_double()
        self._ck(self._lib.tuna_fp64_peak_probe(self._h, ctypes.byref(t)))
        return t.value


class DeviceGroup:
    """One direct Fock build spread over several GPUs of this process (tuna_jk_direct_group): one Context per device, rank r sharded as
    (r, len(devices)); the integer accumulators of all ranks are summed on devices[0] before the conversion to FP64, so J and K are bitwise
    equal to a single Context's.  devices[0] receives the densities and returns J and K."""

    def __init__(self, devices):
        devices = [int(d) for d in devices]
        if not devices or len(set(devices)) != len(devices) or min(devices) < 0:
            raise error_class(f"tuna_b200: a device group needs distinct non-negative device ordinals, got {devices}")
        self.devices = devices
        self.contexts = []
        try:
            for r, d in enumerate(devices):
                self.contexts.append(Context(d))
                self.contexts[-1].set_shard(r, len(devices))
        except BaseException:
            self.close()
            raise
        self._ptrs = (ctypes.c_void_p * len(devices))(*[c._h.value for c in self.contexts])
        self._lib = self.contexts[0]._lib

    @property
    def ncart(self):
        return self.contexts[0].ncart

    @property
    def nbf(self):
        return self.contexts[0].nbf

    def set_basis(self, origins_z, lmn, nprim, exps, coef_eff):
        for c in self.contexts:
            c.set_basis(origins_z, lmn, nprim, exps, coef_eff)

    def set_transform(self, U):
        for c in self.contexts:
            c.set_transform(U)

    def _ck(self, rc):
        if rc:
            self.contexts[0]._raise(rc)

    def jk_direct(self, P, tau=1e-16, want_j=True, want_k=True):
        """Same contract as Context.jk_direct: (n, n) or (nD, n, n), any real P, host arrays in and out."""
        P = np.ascontiguousarray(P, dtype=np.float64)
        n = self.nbf
        single = P.ndim == 2
        Ps = P[None] if single else P
        if Ps.ndim != 3 or Ps.shape[1:] != (n, n):
            raise error_class(f"tuna_b200: density matrix has shape {P.shape}, expected ({n}, {n})")
        J = np.empty_like(Ps) if want_j else None
        K = np.empty_like(Ps) if want_k else None
        self._ck(self._lib.tuna_jk_direct_group(self._ptrs, len(self.contexts), Ps.shape[0], _dp(Ps), _dp(J), _dp(K), ctypes.c_double(tau)))
        if single:
            return (J[0] if want_j else None), (K[0] if want_k else None)
        return J, K

    def jk_direct_dev(self, nD, dP, dJ, dK, tau=1e-16):
        """Device pointers on devices[0], enqueued on the stream of contexts[0]; symmetric densities only (tuna_jk_direct_dev).
        Any real P: jk_direct_general_dev."""
        self._ck(self._lib.tuna_jk_direct_group_dev(self._ptrs, len(self.contexts), nD, ctypes.c_void_p(dP), ctypes.c_void_p(dJ), ctypes.c_void_p(dK),
                                                    ctypes.c_double(tau)))

    def jk_direct_general_dev(self, nD, dP, dJ, dK, tau=1e-16):
        """jk_direct on device buffers on devices[0], enqueued on the stream of contexts[0]: any real P, 1 <= nD <= 8, bitwise equal to
        jk_direct and to one Context's jk_direct_general_dev.  Synchronises that stream once, after the density scan on devices[0]
        (tuna_jk_direct_group_general_dev)."""
        self._ck(self._lib.tuna_jk_direct_group_general_dev(self._ptrs, len(self.contexts), nD, ctypes.c_void_p(dP), ctypes.c_void_p(dJ),
                                                            ctypes.c_void_p(dK), ctypes.c_double(tau)))

    def set_integral_store(self, budget_bytes: int):
        """Semi-direct J/K on every rank: each stores its own share of the integrals on its own device, up to budget_bytes each."""
        for c in self.contexts:
            c.set_integral_store(budget_bytes)

    def integral_store_info(self) -> dict:
        """The ranks' store counters: bytes and items summed over the ranks, replayed builds of contexts[0]."""
        per_rank = [c.integral_store_info() for c in self.contexts]
        out = {k: sum(r[k] for r in per_rank) for k in ("bytes", "items", "items_last_build")}
        out["replayed_builds"] = per_rank[0]["replayed_builds"]
        return out

    def counts(self) -> dict:
        """Counters of contexts[0], with evaluated_last_direct summed over all ranks."""
        per_rank = [c.counts() for c in self.contexts]
        out = dict(per_rank[0])
        out["evaluated_last_direct"] = sum(c["evaluated_last_direct"] for c in per_rank)
        return out

    def close(self):
        for c in self.contexts:
            c.close()
        self.contexts = []

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass
