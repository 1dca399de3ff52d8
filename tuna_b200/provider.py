"""Drop-in ERI / Fock provider: the reference's Python call signatures over the CUDA library.

Each public function keeps the name, argument order and return convention of the reference function it
replaces (SURVEY.md section 8b); `install()` rebinds those names on the reference's flat modules so that
tuna_scf, tuna_dft (hybrid exact exchange goes through K) and the post-HF modules use this provider with
no reference edits.  The only compute path is libtuna_b200.so on a CUDA device — there is no CPU fallback.

    reference                                                             here
    tuna_integral.calculate_electron_repulsion_integrals  pyx:1267-1355   calculate_electron_repulsion_integrals
    tuna_integral.calculate_electron_repulsion_integral   pyx:1376-1414   calculate_electron_repulsion_integral
    tuna_kernel.calculate_two_electron_integrals          tuna_kernel.py:331-359
    tuna_kernel.transform_to_spherical_harmonics          tuna_kernel.py:454-529
    tuna_scf.calculate_coulomb_matrix                     tuna_scf.py:55-72
    tuna_scf.calculate_exchange_matrix                    tuna_scf.py:27-44
    tuna_ci.transform_ERI_AO_to_MO                        tuna_ci.py:204-255      (SURVEY.md 8f-2)
    tuna_ci.transform_ERI_AO_to_SO                        tuna_ci.py:143-193
    tuna_integral.calculate_one_electron_integrals        pyx:282-445             (SURVEY.md 8f-3)
    tuna_integral.calculate_cross_basis_overlap_matrix    pyx:626-778
"""
import os
import weakref

import numpy as np

from . import _lib
from .basis import flatten

DEFAULT_TAU = float(os.environ.get("TUNA_B200_TAU", "1e-16"))      # Schwarz threshold of direct mode (SURVEY.md 8d)
_settings = {"mode": os.environ.get("TUNA_B200_MODE", "auto"), "device": int(os.environ.get("TUNA_B200_DEVICE", "0")),
             "stored_fraction": 0.40, "tau": DEFAULT_TAU}
# semi-direct J/K: direct mode keeps the engine's integrals in up to this fraction of each device's free memory (0 = off)
_store_fraction = float(os.environ.get("TUNA_B200_STORE_FRACTION", "0.5"))
_devices = None      # devices of direct J/K (None: _settings["device"] alone); "all" = every visible device, resolved on first use


def _parse_devices(spec):
    """'all', a comma list '0,1,3' or a sequence of ordinals -> 'all' or a list of distinct non-negative ints."""
    if isinstance(spec, str):
        if spec.strip().lower() == "all":
            return "all"
        try:
            spec = [int(x) for x in spec.split(",") if x.strip()]
        except ValueError:
            raise _lib.error_class(f"tuna_b200: devices must be 'all' or a comma list of ordinals, got {spec!r}") from None
    devices = [int(d) for d in spec]
    if not devices or len(set(devices)) != len(devices) or min(devices) < 0:
        raise _lib.error_class(f"tuna_b200: devices must be distinct non-negative ordinals, got {devices}")
    return devices


def _set_devices(spec):
    global _devices
    _devices = _parse_devices(spec)
    _settings["device"] = 0 if _devices == "all" else _devices[0]


def configured_devices():
    """The devices direct J/K runs on; the first is the primary device (one-electron integrals, stored mode, the dense fill)."""
    global _devices
    if _devices == "all":
        import torch  # plumbing only: the number of visible devices
        n = torch.cuda.device_count()
        if n < 1:
            raise _lib.error_class("tuna_b200: devices='all' but no CUDA device is visible")
        _devices = list(range(n))
    return list(_devices) if _devices is not None else [_settings["device"]]


if os.environ.get("TUNA_B200_DEVICES", "").strip():
    _set_devices(os.environ["TUNA_B200_DEVICES"])


def configure(mode=None, device=None, tau=None, stored_fraction=None, devices=None, store_fraction=None):
    """mode: 'stored' (dense tensor on the device), 'direct' (integral-driven J/K) or 'auto' (stored when
    8*ncart^4 bytes fit in `stored_fraction` of free device memory or a post-HF consumer needs the tensor).
    devices: 'all' or a list of ordinals (or a comma list); direct-mode J/K of one Fock build is spread over all of them
    (DeviceGroup), everything else runs on devices[0].  device=d is devices=[d].
    store_fraction: direct mode keeps the integrals it evaluates in up to this fraction of each device's free memory and replays
    them in later Fock builds (semi-direct J/K, bitwise equal to the direct build); 0 = off.  Applies to handles whose first J/K call
    comes after it."""
    global _store_fraction
    if mode is not None:
        if mode not in ("stored", "direct", "auto"):
            raise _lib.error_class(f"tuna_b200: unknown mode {mode!r}")
        _settings["mode"] = mode
    if device is not None and devices is not None:
        raise _lib.error_class("tuna_b200: give either device or devices")
    if device is not None:
        _set_devices([device])
    if devices is not None:
        _set_devices(devices)
    if tau is not None:
        _settings["tau"] = float(tau)
    if stored_fraction is not None:
        _settings["stored_fraction"] = float(stored_fraction)
    if store_fraction is not None:
        if not 0.0 <= float(store_fraction) <= 1.0:
            raise _lib.error_class(f"tuna_b200: store_fraction must lie in [0, 1], got {store_fraction!r}")
        _store_fraction = float(store_fraction)


def _free_device_bytes():
    import torch  # plumbing only: device memory query
    free, _ = torch.cuda.mem_get_info(configured_devices()[0])
    return free


class ERIHandle:
    """What flows through `Integrals.ERI_AO` (TUNA/tuna_util.py:152-194) instead of a host ndarray.

    J/K consumers use the device-resident tensor (stored mode) or the pair table (direct mode) behind `ctx`.
    Post-HF consumers that need a real ndarray (tuna_ci.py:229, tuna_mp.py:632, tuna_cc.py:1851 ...) get one on
    first touch: the tensor is copied device->host once and every ndarray attribute/operator is forwarded to it.
    """

    __array_priority__ = 100.0

    def __init__(self, ctx, n, basis_kind, mode):
        self.ctx, self.n, self.basis_kind, self.mode = ctx, int(n), basis_kind, mode
        self._host = None
        self.pending_fill = False   # stored mode: the tensor is filled by transform_to_spherical_harmonics, or on first touch as an array
        self._jk_cache = []     # [(P, J, K)] most recent first
        self._group = None      # direct mode over several devices: DeviceGroup built on the first J/K call
        self._store_for = None  # direct mode: the Context / DeviceGroup whose integral store this handle has enabled
        self._store_dropped = False     # a dense tensor was materialised: the store stays off so the tensor keeps today's memory

    shape = property(lambda self: (self.n,) * 4)
    ndim = 4
    dtype = np.dtype(np.float64)
    size = property(lambda self: self.n ** 4)

    def materialise(self) -> np.ndarray:
        if self._host is None:
            if self.mode == "direct":
                self._materialise_direct()
            else:
                if self.pending_fill:
                    self.ctx.eri_fill_cart()
                    self.pending_fill = False
                self._host = self.ctx.eri_download(0 if self.basis_kind == "cart" else 1)
        return self._host

    def _materialise_direct(self):
        ctx = self.ctx
        # the integral store gives its memory back before the dense tensor's size is checked
        _release_integral_stores([t for t in (ctx, self._group) if t is not None])
        self._store_for, self._store_dropped = None, True
        if self.basis_kind == "cart" or not hasattr(ctx, "eri_fill_sph"):
            need = 8 * ctx.ncart ** 4
        else:   # the spherical fill: nbf^4 plus the engine's scratch rows, which are about as large as the unique Cartesian integrals
            need = 8 * (ctx.nbf ** 4 + ctx.ncart ** 4 // 8)
        if need > 0.8 * _free_device_bytes():
            raise MemoryError(f"tuna_b200: a dense ERI tensor was requested in direct mode but {need / 1e9:.1f} GB do not fit on the device")
        if self.basis_kind == "cart":
            ctx.eri_fill_cart()
            self._host = ctx.eri_download(0)
        else:
            _fill_spherical(ctx)
            self._host = ctx.eri_download(1)

    def __array__(self, dtype=None, copy=None):
        a = self.materialise()
        return a if dtype is None else a.astype(dtype, copy=False)

    def __getitem__(self, idx):
        return self.materialise()[idx]

    def __len__(self):
        return self.n

    def __getattr__(self, name):          # reshape, swapaxes, transpose, T, sum, ...
        if name.startswith("_"):
            raise AttributeError(name)
        return getattr(self.materialise(), name)


class SpinBlocked:
    """Lazy stand-in for the spin-blocking idiom of the reference's post-HF drivers (TUNA/tuna_ci.py:564):

        ERI_spin_block = np.kron(np.eye(2), np.kron(np.eye(2), ERI_AO).T)

    `ERIHandle.__array_function__` turns the inner `np.kron(np.eye(2), handle)` into SpinBlocked(handle, 1), `.T` into stage 2 and the
    outer kron into stage 3; `transform_ERI_AO_to_SO` recognises stage 3 and builds the 16 n^4 tensor on the device from the resident
    one.  Anything else that touches the object gets the real ndarray, computed by NumPy exactly as the reference does."""

    __array_priority__ = 100.0
    ndim = 4
    dtype = np.dtype(np.float64)

    def __init__(self, handle, stage):
        self.handle, self.stage = handle, stage
        self._host = None

    @property
    def shape(self):
        n = self.handle.n
        return {1: (n, n, 2 * n, 2 * n), 2: (2 * n, 2 * n, n, n), 3: (2 * n,) * 4}[self.stage]

    @property
    def T(self):
        return SpinBlocked(self.handle, 2) if self.stage == 1 else self.materialise().T

    def materialise(self):
        if self._host is None:
            a = np.kron(np.eye(2), self.handle.materialise())
            if self.stage >= 2:
                a = a.T
            if self.stage == 3:
                a = np.kron(np.eye(2), a)
            self._host = a
        return self._host

    def __array__(self, dtype=None, copy=None):
        a = self.materialise()
        return a if dtype is None else a.astype(dtype, copy=False)

    def __array_function__(self, func, types, args, kwargs):
        if func is np.kron and len(args) == 2 and args[1] is self and self.stage == 2 and _is_eye2(args[0]):
            return SpinBlocked(self.handle, 3)
        return func(*[a.materialise() if isinstance(a, (SpinBlocked, ERIHandle)) else a for a in args], **kwargs)

    def __getitem__(self, idx):
        return self.materialise()[idx]

    def __getattr__(self, name):
        if name.startswith("_"):
            raise AttributeError(name)
        return getattr(self.materialise(), name)


def _is_eye2(a):
    return isinstance(a, np.ndarray) and a.shape == (2, 2) and np.array_equal(a, np.eye(2))


def _handle_array_function(self, func, types, args, kwargs):
    """NumPy dispatch on ERIHandle arguments: the spin-blocking kron stays lazy (device-resident stored tensors only); every other
    function sees the materialised ndarray."""
    if (func is np.kron and len(args) == 2 and args[1] is self and _is_eye2(args[0]) and self.mode == "stored" and self.basis_kind == "sph"
            and self.ctx.n_stored == self.n):
        return SpinBlocked(self, 1)
    return func(*[a.materialise() if isinstance(a, (SpinBlocked, ERIHandle)) else a for a in args], **kwargs)


ERIHandle.__array_function__ = _handle_array_function


def _binary(op):
    def f(self, other):
        return getattr(self.materialise(), op)(np.asarray(other) if isinstance(other, ERIHandle) else other)
    return f


for _op in ("add", "radd", "sub", "rsub", "mul", "rmul", "truediv", "rtruediv", "neg", "matmul", "rmatmul", "pow"):
    if _op == "neg":
        setattr(ERIHandle, "__neg__", lambda self: -self.materialise())
    else:
        setattr(ERIHandle, f"__{_op}__", _binary(f"__{_op}__"))


_ctx_cache = []        # [(device, key, Context)] most recent first: one-electron integrals, ERIs and J/K of one geometry share a context


def _flatten_or_raise(bfs):
    try:
        return flatten(bfs)
    except ValueError as e:
        raise _lib.error_class(f"tuna_b200: {e}")


def _context_for(bfs, cached=True):
    """Context holding this basis.  With cached=True the context of the most recent identical basis (same device, byte-identical flattened
    arrays) is returned: the reference asks for the one-electron integrals, the two-electron integrals and single quartets of one geometry
    through separate calls (tuna_kernel.py:425-437), and finite-field / ionisation runs repeat them on the same geometry
    (tuna_energy.py:361-373).  The library builds the ERI pair table lazily, so a context that only serves one-electron integrals never pays
    for it.  Cached contexts are never closed here (an ERIHandle may hold them); they are released when the last reference goes."""
    flat = _flatten_or_raise(bfs)
    dev = _settings["device"]
    if cached:
        key = tuple(np.ascontiguousarray(a).tobytes() for a in flat)
        for i, (d, k, c) in enumerate(_ctx_cache):
            if d == dev and k == key and getattr(c, "_h", True):
                _ctx_cache.insert(0, _ctx_cache.pop(i))
                return c
    ctx = _lib.Context(dev)
    ctx.set_basis(*flat)
    if cached:
        _ctx_cache.insert(0, (dev, key, ctx))
        _release_integral_stores([c for _, _, c in _ctx_cache[2:]])      # a context leaving the cache keeps no store
        del _ctx_cache[2:]
    return ctx


# ---------------------------------------------------------------------------------------------------------
# tuna_integral level (pyx)
# ---------------------------------------------------------------------------------------------------------
def calculate_electron_repulsion_integrals(n_basis, ERI_AO, bfs, num_threads):
    """Fill the caller's dense (n,n,n,n) buffer in place and return it (pyx:1267-1355).  `num_threads` is advisory
    (OpenMP threads of the reference); the GPU path ignores it."""
    if len(bfs) != n_basis:
        raise _lib.error_class("tuna_b200: n_basis does not match the basis-function list")
    out = np.asarray(ERI_AO)
    if out.shape != (n_basis,) * 4 or out.dtype != np.float64:
        raise _lib.error_class("tuna_b200: ERI_AO must be a float64 array of shape (n_basis,)*4")
    ctx = _context_for(bfs, cached=False)            # the dense Cartesian tensor is only a transit buffer here: private context, closed below
    ctx.eri_fill_cart()
    if out.flags.c_contiguous:
        ctx.eri_download(0, out)
    else:
        out[...] = ctx.eri_download(0)
    ctx.close()
    return ERI_AO


def calculate_electron_repulsion_integral(bf_1, bf_2, bf_3, bf_4):
    """(12|34) for four basis functions (pyx:1376-1414)."""
    ctx = _scratch_context()                           # no context per scalar: the scratch context takes the four functions as its basis
    ctx.set_basis(*_flatten_or_raise([bf_1, bf_2, bf_3, bf_4]))
    return ctx.eri_single(0, 1, 2, 3)


# ---------------------------------------------------------------------------------------------------------
# tuna_kernel level
# ---------------------------------------------------------------------------------------------------------
def _dense_needed(calculation) -> bool:
    """True if kern.run_post_SCF_energy_calculation will hand ERI_AO to a consumer needing an ndarray
    (dispatch conditions at tuna_kernel.py:1146, :1152, :1161, :1175)."""
    m = getattr(calculation, "method", None)
    return bool(getattr(calculation, "stability_analysis", False) or getattr(m, "perturbative_method", False)
                or getattr(calculation, "MPC_prop", 0) != 0 or getattr(m, "method_base", "") == "CC"
                or getattr(m, "excited_state_method", False) or getattr(calculation, "time_dependent", False))


def _choose_mode(n_cart, calculation):
    _release_integral_stores()                 # a new geometry: earlier handles' stores give their memory back before it is measured
    mode = _settings["mode"]
    if mode != "auto":
        return mode
    need = 8 * n_cart ** 4
    if calculation is not None and _dense_needed(calculation):
        return "stored"
    return "stored" if 2.2 * need <= _settings["stored_fraction"] * _free_device_bytes() else "direct"


def calculate_two_electron_integrals(n_basis, basis_functions, calculation):
    """Cartesian two-electron integrals (tuna_kernel.py:331-359).  Returns an ERIHandle: the tensor (stored mode)
    or just the pair table (direct mode) stays on the device; timers keep the reference's names."""
    timer = _ref_timer()
    timer("Two-electron integrals", 0)
    mode = _choose_mode(n_basis, calculation)
    ctx = _context_for(basis_functions)
    handle = ERIHandle(ctx, n_basis, "cart", mode)
    handle.pending_fill = mode == "stored"     # filled straight into the spherical basis once U is known (transform_to_spherical_harmonics)
    timer("Two-electron integrals", 1)
    return handle


def _fill_spherical(ctx):
    """The spherical tensor as the stored tensor: one pass without the Cartesian tensor where the library has it, else fill + rotation."""
    if hasattr(ctx, "eri_fill_sph"):
        ctx.eri_fill_sph()
    else:
        ctx.eri_fill_cart()
        ctx.eri_cart_to_sph()


def _stored_to_spherical(handle):
    """Stored mode: the spherical tensor of a Cartesian handle, after ctx.set_transform.  A handle whose Cartesian tensor was already
    filled (touched as an array) is rotated; otherwise the tensor is filled in the spherical basis directly."""
    if handle.pending_fill:
        handle.pending_fill = False
        _fill_spherical(handle.ctx)
    else:
        handle.ctx.eri_cart_to_sph()


def transform_to_spherical_harmonics(S_cart, T_cart, V_NE_cart, D_cart, Q_cart, ERI_AO_cart, molecule, calculation, silent):
    """Cartesian -> spherical rotation of all integrals (tuna_kernel.py:454-529); the ERI part runs on the device."""
    U = np.asarray(molecule.spherical_harmonic_transformation_matrix, dtype=np.float64)
    cartharm = bool(getattr(calculation, "cartesian_harmonics", False))
    if not isinstance(ERI_AO_cart, ERIHandle):
        raise _lib.error_class("tuna_b200: transform_to_spherical_harmonics expects the ERIHandle from calculate_two_electron_integrals")
    ctx = ERI_AO_cart.ctx
    if cartharm:
        ctx.set_transform(np.eye(ctx.ncart))
        if ERI_AO_cart.mode == "stored":
            _stored_to_spherical(ERI_AO_cart)
        return S_cart, T_cart, V_NE_cart, D_cart, Q_cart, ERIHandle(ctx, ctx.ncart, "sph", ERI_AO_cart.mode)
    timer = _ref_timer()
    timer("Spherical harmonic transformation", 0)
    S = U @ S_cart @ U.T
    T = U @ T_cart @ U.T
    V_NE = U @ V_NE_cart @ U.T
    D = np.einsum("mw,awx,nx->amn", U, D_cart, U, optimize=True)
    Q = np.einsum("mw,awx,nx->amn", U, Q_cart, U, optimize=True)
    ctx.set_transform(U)
    if ERI_AO_cart.mode == "stored":
        _stored_to_spherical(ERI_AO_cart)
    handle = ERIHandle(ctx, U.shape[0], "sph", ERI_AO_cart.mode)
    timer("Spherical harmonic transformation", 1)
    return S, T, V_NE, D, Q, handle


# ---------------------------------------------------------------------------------------------------------
# tuna_scf level
# ---------------------------------------------------------------------------------------------------------
_uploaded = {}     # id(ndarray) -> (weakref, ERIHandle): dense tensors handed in by the caller, uploaded once


def _handle_for(ERI_AO):
    if isinstance(ERI_AO, ERIHandle):
        return ERI_AO
    arr = np.asarray(ERI_AO)
    if arr.ndim != 4:
        raise _lib.error_class("tuna_b200: ERI_AO must be an ERIHandle or a 4-index array")
    key = id(ERI_AO)
    hit = _uploaded.get(key)
    if hit is not None and hit[0]() is ERI_AO:
        return hit[1]
    ctx = _lib.Context(_settings["device"])
    ctx.eri_upload(arr)
    h = ERIHandle(ctx, arr.shape[0], "sph", "stored")
    h._host = arr
    try:
        _uploaded[key] = (weakref.ref(ERI_AO, lambda _r, k=key: _uploaded.pop(k, None)), h)
    except TypeError:
        pass
    return h


def coulomb_and_exchange(P, ERI_AO, want_j=True, want_k=True):
    """J and K for one density (n,n) or a stack (nD,n,n) from ONE pass over the integrals."""
    h = _handle_for(ERI_AO)
    P = np.asarray(P, dtype=np.float64)
    if h.mode == "stored":
        return h.ctx.jk_stored(P, want_j, want_k)
    # any real P: the library splits a non-symmetric density into its symmetric and antisymmetric parts (K[P] = K[S] + K[A] with
    # K[A] antisymmetric, J[P] = J[S]); the reference's guess densities are asymmetric at the 1e-8 level
    devices = configured_devices()
    if len(devices) > 1:
        if h._group is None or h._group.devices != devices:
            # the handle's own context stays unsharded (dense fill on demand, single integrals, Schwarz factors)
            group = _lib.DeviceGroup(devices)
            group.set_basis(*h.ctx.basis_flat)
            group.set_transform(h.ctx.U)
            h._group = group
        _enable_store(h, h._group, h._group.contexts)
        return h._group.jk_direct(P, _settings["tau"], want_j, want_k)
    _enable_store(h, h.ctx, [h.ctx])
    return h.ctx.jk_direct(P, _settings["tau"], want_j, want_k)


_store_holders = weakref.WeakSet()      # Contexts / DeviceGroups whose integral store a direct-mode handle turned on


def _release_integral_stores(targets=None):
    """Give back the memory of the integral stores the provider turned on (all of them, or those of `targets`).  A new geometry's mode is
    decided against the free device memory, which a finished handle's store must not hold; a handle whose store was released runs its
    later builds direct."""
    for t in list(_store_holders if targets is None else [t for t in targets if t in _store_holders]):
        if getattr(t, "_h", True):             # a closed Context has nothing left to release
            t.set_integral_store(0)
        _store_holders.discard(t)


def _enable_store(h, target, contexts):
    """Semi-direct J/K on the first direct J/K call of a handle: every context of `target` may keep up to store_fraction of its device's
    free memory (the library clamps it further and allocates only what the stored class jobs need)."""
    if h._store_for is target or h._store_dropped:
        return
    frac = _store_fraction
    if frac > 0.0:
        import torch  # plumbing only: device memory query
        for c in contexts:
            c.set_integral_store(int(frac * torch.cuda.mem_get_info(c.device)[0]))
        _store_holders.add(target)
    h._store_for = target


def _cached_jk(P, ERI_AO, which):
    h = _handle_for(ERI_AO)
    P = np.asarray(P, dtype=np.float64)
    for Pc, J, K in h._jk_cache:
        if Pc.shape == P.shape and np.array_equal(Pc, P):
            return (J if which == 0 else K).copy()
    J, K = coulomb_and_exchange(P, h)
    h._jk_cache.insert(0, (P.copy(), J, K))
    del h._jk_cache[4:]
    return (J if which == 0 else K).copy()


def calculate_coulomb_matrix(P, ERI_AO):
    """J_ij = sum_kl (ij|kl) P_kl (tuna_scf.py:55-72).  The fused kernel also produces K for the same P, which the
    reference always asks for next (tuna_scf.py:520-521, :571-577): it is kept for that call."""
    return _cached_jk(P, ERI_AO, 0)


def calculate_exchange_matrix(P, ERI_AO):
    """K_ij = sum_kl (il|kj) P_kl (tuna_scf.py:27-44)."""
    return _cached_jk(P, ERI_AO, 1)


# ---------------------------------------------------------------------------------------------------------
# tuna_ci level: AO -> MO / spin-orbital transformation (first thing every MPn / CC / CI calculation does with ERI_AO)
# ---------------------------------------------------------------------------------------------------------
_scratch = {}


def _scratch_context():
    """A basis-less context for tensors handed in as host ndarrays (e.g. the spin-blocked tensor of tuna_ci.py:564)."""
    dev = _settings["device"]
    if dev not in _scratch:
        _scratch[dev] = _lib.Context(dev)
    return _scratch[dev]


def _transform(ERI_AO, C_1, C_2, so_layout, calculation, silent):
    timer = _ref_timer()
    timer("Molecular orbital transformation", 0)
    log = _log_fn
    if log is not None and calculation is not None:
        log("\n Transforming integrals on the device (4 steps)... ", calculation, 1, end="", silent=silent)
    C_1 = np.asarray(C_1, dtype=np.float64)
    C_2 = np.asarray(C_2, dtype=np.float64)
    if isinstance(ERI_AO, SpinBlocked) and ERI_AO.stage == 3 and ERI_AO.handle.ctx.n_stored == ERI_AO.handle.n and hasattr(ERI_AO.handle.ctx, "eri_transform_spin_blocked"):
        out = ERI_AO.handle.ctx.eri_transform_spin_blocked(C_1, C_2, so_layout)     # spin-blocked on the device from the resident tensor
    elif isinstance(ERI_AO, ERIHandle) and ERI_AO.mode == "stored" and ERI_AO.basis_kind == "sph" and ERI_AO.ctx.n_stored == ERI_AO.n:
        out = ERI_AO.ctx.eri_transform(C_1, C_2, so_layout)                     # the tensor is already resident
    else:
        arr = np.asarray(ERI_AO, dtype=np.float64)
        if arr.ndim != 4 or len(set(arr.shape)) != 1:
            raise _lib.error_class("tuna_b200: ERI_AO must be an ERIHandle or an (n, n, n, n) array")
        out = _scratch_context().eri_transform(C_1, C_2, so_layout, eri=arr)
    if log is not None and calculation is not None:
        log("[Done]", calculation, 1, silent=silent)
    timer("Molecular orbital transformation", 1)
    return out


def transform_ERI_AO_to_MO(ERI_AO, C, calculation, silent):
    """ERI_MO[p,r,q,s] = sum_mknl ERI_AO[m,k,n,l] C[m,p] C[k,r] C[n,q] C[l,s] (tuna_ci.py:204-255): interleaved chemists' notation."""
    return _transform(ERI_AO, C, C, False, calculation, silent)


def transform_ERI_AO_to_SO(ERI_AO, C_1, C_2, calculation, silent):
    """ERI_SO[p,q,r,s] = sum_mknl ERI_AO[m,k,n,l] C_2[m,p] C_1[n,q] C_2[k,r] C_1[l,s] (tuna_ci.py:143-193): physicists' notation."""
    return _transform(ERI_AO, C_1, C_2, True, calculation, silent)


# ---------------------------------------------------------------------------------------------------------
# tuna_integral level: one-electron integrals (SURVEY.md 8f-3)
# ---------------------------------------------------------------------------------------------------------
def calculate_one_electron_integrals(n_basis, basis_functions, n_atoms, atoms, dipole_origin, num_threads):
    """(S_cart, T_cart, V_cart, D_cart, Q_cart) in Cartesian harmonics (pyx:282-445): overlap, kinetic, nuclear attraction,
    dipole (3, n, n) and diagonal quadrupole (3, n, n) about `dipole_origin`.  `num_threads` is advisory and ignored."""
    if len(basis_functions) != n_basis or len(atoms) != n_atoms:
        raise _lib.error_class("tuna_b200: n_basis / n_atoms do not match the lists")
    pos = np.array([np.asarray(a.origin, dtype=np.float64) for a in atoms]).reshape(n_atoms, 3)
    if np.any(pos[:, :2] != 0.0):
        raise _lib.error_class("tuna_b200: all atoms must lie on the z axis")       # as the reference's nuclear integral requires (pyx:783)
    ctx = _context_for(basis_functions)                # shared with the two-electron call that follows (tuna_kernel.py:425-437)
    return ctx.one_electron(pos[:, 2], [float(a.charge) for a in atoms], np.asarray(dipole_origin, dtype=np.float64))


def calculate_cross_basis_overlap_matrix(n_basis_1, n_basis_2, basis_functions_1, basis_functions_2, num_threads):
    """S_cross[i, j] = <bf_1[i] | bf_2[j]> between two basis sets (pyx:626-778; the minimal-basis guess projection, tuna_guess.py:281)."""
    if len(basis_functions_1) != n_basis_1 or len(basis_functions_2) != n_basis_2:
        raise _lib.error_class("tuna_b200: basis sizes do not match the lists")
    try:
        f1, f2 = flatten(basis_functions_1), flatten(basis_functions_2)
    except ValueError as e:
        raise _lib.error_class(f"tuna_b200: {e}")
    return _scratch_context().cross_overlap(f1, f2)


# ---------------------------------------------------------------------------------------------------------
# installation on the reference's modules
# ---------------------------------------------------------------------------------------------------------
_timer_fn = None
_log_fn = None


def _ref_timer():
    return _timer_fn if _timer_fn is not None else (lambda name, flag: None)


def install(tuna_integral=None, tuna_kernel=None, tuna_scf=None, tuna_util=None, tuna_ci=None):
    """Rebind the hot-path names (six of the SCF path, the two AO->MO transformations of tuna_ci, the two one-electron entry points) on the reference's (already imported) modules.  All four are module-global
    lookups at call time (SURVEY.md 8b), so no reference source is edited.  Returns a dict of the originals."""
    import sys
    global _timer_fn, _log_fn
    tuna_integral = tuna_integral or sys.modules.get("tuna_integrals.tuna_integral")
    tuna_kernel = tuna_kernel or sys.modules.get("tuna_kernel")
    tuna_scf = tuna_scf or sys.modules.get("tuna_scf")
    tuna_util = tuna_util or sys.modules.get("tuna_util")
    tuna_ci = tuna_ci or sys.modules.get("tuna_ci")
    originals = {}
    if tuna_util is not None:
        _lib.error_class = getattr(tuna_util, "TunaError", _lib.error_class)
        _timer_fn = getattr(tuna_util, "timer", None)
        _log_fn = getattr(tuna_util, "log", None)
    for mod, names in ((tuna_integral, ("calculate_electron_repulsion_integrals", "calculate_electron_repulsion_integral",
                                        "calculate_one_electron_integrals", "calculate_cross_basis_overlap_matrix")),
                       (tuna_kernel, ("calculate_two_electron_integrals", "transform_to_spherical_harmonics")),
                       (tuna_scf, ("calculate_coulomb_matrix", "calculate_exchange_matrix")),
                       (tuna_ci, ("transform_ERI_AO_to_MO", "transform_ERI_AO_to_SO"))):
        if mod is None:
            continue
        for name in names:
            originals[(mod.__name__, name)] = getattr(mod, name)
            setattr(mod, name, globals()[name])
    return originals


def uninstall(originals):
    import sys
    for (modname, name), fn in originals.items():
        setattr(sys.modules[modname], name, fn)
