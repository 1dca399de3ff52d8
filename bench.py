#!/usr/bin/env python
"""bench.py — the driver's benchmark contract for the TUNA SCF two-electron hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--workload direct:et400|stored:n2_ccpvtz|...]
                    [--dump-outputs DIR]

Headline workload (BASELINE.json configs[4], the one the metric's "1/2/4/8 B200 ... % FP64 peak" is quoted on, at its largest
point): the synthetic even-tempered N2 diatomic at nbf=800 (ncart 1102), direct ERI + J/K, one density.  The other sweep
points (nbf 100/200/400) are measured at N=1 in the same run and reported under "sweep".  A "step" is one Fock build:
every parity-surviving unique AO quartet is evaluated (Schwarz-screened) and folded into J and K.  At N GPUs the quartet
list is sharded over ranks (strong scaling) and the partial J/K are summed by one NCCL all-reduce inside the timed region.
The stored-ERI configuration (configs[1], N2 RHF/cc-pVTZ) is measured in the same run at N=1 and reported under "stored".

One JSON line on stdout (rank 0).  `value` is device-resident throughput; `e2e` goes through the public API with host
buffers (H2D of P, D2H of J and K inside the timed region); `roofline` is the dominant kernel's ALGORITHMIC flops (the
reference algorithm's count, SURVEY.md 8d) over its CUDA-event time against the FP64 pipe peak measured in this run.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

METRIC = "fock_builds_per_s"
UNIT = "Fock builds/s"

# ncu-counted FP64 work (2*DFMA + DMUL + DADD thread instructions) and DRAM traffic of one direct build, summed over all class-job
# launches: a property of the code + workload, regenerated from the ncu CSV of the round by tools/executed_from_ncu.py into
# profiles/executed_fp64.json, keyed "<workload>|<densities>|<tau>".  The RATE below always uses this run's own kernel time.
def executed_fp64_table():
    try:
        with open(os.path.join(ROOT, "profiles", "executed_fp64.json")) as f:
            return json.load(f)
    except (OSError, ValueError):
        return {}


# ----------------------------------------------------------------------------------------------------------------
# workloads
# ----------------------------------------------------------------------------------------------------------------
def load_workload(spec):
    """-> dict(name, mode, bfs, U, nbf, ncart, nD, description)."""
    from tuna_b200 import workloads as w
    from tuna_b200.basis import from_arrays
    mode, name = spec.split(":")
    if name.startswith("et"):
        nbf = int(name[2:])
        b = w.even_tempered_diatomic(nbf)
        bfs = from_arrays(b["origins"], b["lmn"], b["nprim"], b["exps"], b["raw_coefs"])
        U = make_U(b["lmn"])
        desc = f"configs[4]: synthetic even-tempered N2 (1.10 A) nbf={nbf}, {mode} ERI+J/K, RHF (1 density)"
        return dict(name=name, mode=mode, bfs=bfs, U=U, nbf=U.shape[0], ncart=len(bfs), nD=1, description=desc, raw=b)
    from util import basis_objects, load_golden
    g = load_golden(name)
    nD = 2 if bool(g["unrestricted"]) else 1
    desc = {"n2_ccpvtz": "configs[1]: N2 RHF/cc-pVTZ 1.10 A", "co_b3lyp_ccpvtz": "configs[2]: CO B3LYP/cc-pVTZ (exact-exchange K)",
            "ne2_uhf_ccpvqz": "configs[3]: Ne2 UHF/cc-pVQZ 3.1 A", "h2_631g": "configs[0]: H2 RHF/6-31G 0.74 A"}.get(name, name)
    return dict(name=name, mode=mode, bfs=basis_objects(g), U=np.array(g["U"]), nbf=int(g["nbf"]), ncart=int(g["ncart"]), nD=nD,
                description=f"{desc}, {mode} J/K, {nD} density(ies)", raw=dict(origins=g["origins"], lmn=g["lmn"], nprim=g["nprim"],
                                                                               exps=g["exps"], coefs=g["coefs"], norms=g["norms"]))


def make_U(lmn):
    """Cartesian->spherical map for full shells.  Bench inputs are synthetic, so the pure-d/f/g/h rows are generated
    from the real solid harmonics (orthonormalised per shell) instead of the reference's hard-coded tables
    (tuna_kernel.py:540-649); any full-rank (2L+1) x ncart(L) block gives the same amount of work."""
    lmn = np.asarray(lmn)
    blocks, i = [], 0
    while i < len(lmn):
        L = int(lmn[i].sum())
        nc = (L + 1) * (L + 2) // 2
        blocks.append(_sph_block(L))
        i += nc
    n_r, n_c = sum(b.shape[0] for b in blocks), sum(b.shape[1] for b in blocks)
    U = np.zeros((n_r, n_c))
    r = c = 0
    for b in blocks:
        U[r:r + b.shape[0], c:c + b.shape[1]] = b
        r += b.shape[0]
        c += b.shape[1]
    return U


_SPH_CACHE = {}


def _sph_block(L):
    if L in _SPH_CACHE:
        return _SPH_CACHE[L]
    if L <= 1:
        blk = np.eye(2 * L + 1)
    else:
        # traceless projection: remove the r^2 * (degree L-2) subspace from the Cartesian monomials of degree L
        from tuna_b200.workloads import cartesian_components
        comps = cartesian_components(L)
        low = cartesian_components(L - 2)
        idx = {c: k for k, c in enumerate(comps)}
        A = np.zeros((len(low), len(comps)))
        for r, (a, b, c) in enumerate(low):
            for d in ((2, 0, 0), (0, 2, 0), (0, 0, 2)):
                A[r, idx[(a + d[0], b + d[1], c + d[2])]] = 1.0
        # rows spanning the orthogonal complement of span(A) (dimension 2L+1), sparse-ish via QR of the null space
        _, s, Vt = np.linalg.svd(A)
        blk = Vt[len(low):]
        blk[np.abs(blk) < 1e-14] = 0.0
    _SPH_CACHE[L] = blk
    return blk


# ----------------------------------------------------------------------------------------------------------------
# helpers
# ----------------------------------------------------------------------------------------------------------------
class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region (B200_PROFILING.md recipe)."""

    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.index, self.proc, self.lines = index, None, []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "MEASURED_PEAKS.json"
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md)"


def host_threads():
    return len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)


DUMP_LIMIT_BYTES = 64 * 1024 * 1024


def dump_outputs(out_dir, arrays):
    """Writes each array as <out_dir>/<name>.npy in float64, so that two builds can be compared output for output.  Above
    DUMP_LIMIT_BYTES in all, every array is cut to a fixed, seeded sample of its flattened elements (the same elements on every
    run of the same workload), sized so that the files stay under the limit."""
    os.makedirs(out_dir, exist_ok=True)
    arrays = {k: np.ascontiguousarray(v, dtype=np.float64) for k, v in arrays.items()}
    total = sum(a.nbytes for a in arrays.values())
    budget = DUMP_LIMIT_BYTES - 4096 * len(arrays)          # room for the .npy headers
    for name, a in arrays.items():
        if total > budget:
            keep = budget * a.size // total
            a = a.ravel()[np.sort(np.random.default_rng(0).choice(a.size, size=keep, replace=False))]
        np.save(os.path.join(out_dir, f"{name}.npy"), a)


# ----------------------------------------------------------------------------------------------------------------
# CPU reference arm (oracle/_ref = the unmodified reference engine; numpy einsum = the reference's J/K, tuna_scf.py:42,70)
# ----------------------------------------------------------------------------------------------------------------
def cpu_reference(wl, budget_s=20.0):
    """Times the reference's own CPU implementation of the path on this box's host cores, on a bounded sample.
    Returns dict(value=builds/s, kind, cores, sample, quartets_per_s)."""
    from oracle import tuna_oracle as orc
    cores = host_threads()
    os.environ.setdefault("OMP_NUM_THREADS", str(cores))
    raw = wl["raw"]
    if "raw_coefs" in raw:
        fb = orc.FlatBasis.from_raw(raw["origins"], raw["lmn"], raw["nprim"], raw["exps"], raw["raw_coefs"])
    else:
        fb = orc.FlatBasis(raw["origins"], raw["lmn"], raw["nprim"], raw["exps"], raw["coefs"], raw["norms"])
    eng = orc.reference_engine()
    kind = "reference" if eng is not None else "port"
    n = fb.ncart
    full_unique, full_surv = orc.parity_surviving_quartets(fb.lmn)
    subset = None
    if n > 160:        # the reference cannot hold 8*ncart^4 beyond ~250 functions (tuna_kernel.py:392-402): sample 150 functions
        rng = np.random.default_rng(20261018)
        subset = np.sort(rng.choice(n, size=150, replace=False))
        off = fb.offsets
        sel = np.concatenate([np.arange(off[i], off[i] + fb.nprim[i]) for i in subset])
        fb = orc.FlatBasis(fb.origins[subset], fb.lmn[subset], fb.nprim[subset], fb.exps[sel], fb.coefs[sel], fb.norms[sel])
        n = fb.ncart
    _, surv = orc.parity_surviving_quartets(fb.lmn)

    def eri_once():
        if eng is not None:
            bfs = orc.reference_basis_objects(fb)
            t = time.perf_counter()
            E = np.asarray(eng.calculate_electron_repulsion_integrals(n, np.empty((n,) * 4), bfs, cores))
            return time.perf_counter() - t, E
        t = time.perf_counter()
        E = orc.eri_fill(fb, cores)
        return time.perf_counter() - t, E

    t_eri, E = eri_once()
    if t_eri < budget_s / 4:
        t_eri = min(t_eri, eri_once()[0])
    qps = surv / t_eri
    if subset is None:
        # the whole reference path: ERI build + Cartesian->spherical rotation + J + K einsums on the fixed density
        t = time.perf_counter()
        Es = orc.cart_to_sph_eri(E, wl["U"]) if wl["U"].shape[0] != wl["U"].shape[1] or not np.array_equal(wl["U"], np.eye(n)) else E
        t_sph = time.perf_counter() - t
        from tuna_b200.workloads import fixed_density
        P = fixed_density(Es.shape[0])
        reps, tJ, tK = 3, [], []
        for _ in range(reps):
            t = time.perf_counter(); orc.coulomb(P, Es); tJ.append(time.perf_counter() - t)
            t = time.perf_counter(); orc.exchange(P, Es); tK.append(time.perf_counter() - t)
        t_jk = wl["nD"] * (min(tJ) + min(tK))
        if wl["mode"] == "stored":
            value = 1.0 / t_jk
            sample = f"full workload: J+K einsums on the dense tensor, best of {reps} (ERI build {t_eri:.3f} s and rotation {t_sph:.3f} s are per-geometry, excluded as in the GPU stored figure)"
        else:
            value = 1.0 / (t_eri + t_sph + t_jk)
            sample = f"full workload: the reference has no direct mode, so one build = ERI build {t_eri:.3f} s + rotation {t_sph:.3f} s + J/K einsums {t_jk:.4f} s"
    else:
        value = qps / full_surv
        sample = (f"EXTRAPOLATED: reference ERI build on a random 150-function subset of the same basis ({surv} surviving quartets in {t_eri:.2f} s), "
                  f"scaled to the workload's {full_surv} surviving quartets; J/K einsums not included (the reference cannot hold 8*{wl['ncart']}^4 bytes)")
    return dict(value=value, unit=UNIT, cores=cores, kind=kind, sample=sample, quartets_per_s=qps)


def run_reference_arm(args, wl):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    vals, last, t0 = [], None, time.perf_counter()
    for s in range(args.warmup + args.steps):
        last = cpu_reference(wl, budget_s=10.0)
        if s >= args.warmup:
            vals.append(last["value"])
        if vals and time.perf_counter() - t0 > 150:      # keep the whole run within a few minutes
            break
    value = float(np.mean(vals))
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": len(vals), "warmup": args.warmup,
            "ms_per_step": 1e3 / value, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": wl["description"], "nbf": wl["nbf"], "ncart": wl["ncart"], "mode": wl["mode"]},
            "cpu_baseline": dict(last, value=value),
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "eri_quartets_per_s": last["quartets_per_s"], "gpu_launches": 0}
    print(json.dumps(line), flush=True)


# ----------------------------------------------------------------------------------------------------------------
# our arm
# ----------------------------------------------------------------------------------------------------------------
class L2Flush:
    """Evict L2 between timed steps: write a 256 MB buffer (> the 126 MB L2, so nothing of the previous step survives), then READ
    a second 256 MB buffer so that L2 is left holding clean lines.  Without the read pass the first ~126 MB a kernel pulls in
    would each evict a dirty line of the flush buffer, charging up to an L2's worth of HBM write-back to the timed kernel."""

    def __init__(self, torch):
        self.torch = torch
        self.a = torch.zeros(64 * 1024 * 1024, dtype=torch.float32, device="cuda")
        self.b = torch.ones(64 * 1024 * 1024, dtype=torch.float32, device="cuda")
        self.sink = None

    def __call__(self):
        self.a.add_(1.0)
        self.sink = self.torch.sum(self.b)


L2_NOTE = "flushed between steps (256 MB written, then 256 MB of a second buffer read so L2 holds clean lines)"


def time_steps(torch, stream, fn, steps, warmup, flush, dist=None):
    """W untimed + K timed steps; each timed step bracketed by CUDA events on the launching stream; L2 flushed between steps."""
    for _ in range(warmup):
        fn()
    stream.synchronize()
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    total_ms = 0.0
    for _ in range(steps):
        if flush is not None:
            flush()                               # > L2 (126 MB): evicts the previous step's lines
            torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        with torch.cuda.stream(stream):
            e0.record(stream)
            fn()
            e1.record(stream)
        e1.synchronize()
        total_ms += e0.elapsed_time(e1)
    if dist is not None:
        dist.barrier()
    torch.cuda.synchronize()
    if dist is not None:
        t = torch.tensor([total_ms], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        total_ms = float(t.item())
    return total_ms


def bench_stored(torch, wl, steps, warmup, device, outputs=None):
    """configs[1]-style: dense tensor resident, fused J+K per step.  With a dict `outputs`, J and K of the last timed step are
    stored in it as host arrays shaped like the return of coulomb_and_exchange."""
    import tuna_b200
    from tuna_b200.basis import flatten
    ctx = tuna_b200.Context(device)
    ctx.set_basis(*flatten(wl["bfs"]))
    ctx.set_transform(wl["U"])
    stream = torch.cuda.Stream()
    ctx.set_stream(stream.cuda_stream)
    t_fill, t_sph = [], []
    for _ in range(3):
        ctx.eri_fill_cart(); t_fill.append(ctx.last_kernel_ms(0))
        ctx.eri_cart_to_sph(); t_sph.append(ctx.last_kernel_ms(1))
    n, nD = wl["nbf"], wl["nD"]
    c = ctx.counts()
    P = np.stack([tuna_b200.workloads.fixed_density(n)] * nD)
    dP = torch.from_numpy(P).cuda()
    dJK = torch.empty((2, nD, n, n), dtype=torch.float64, device="cuda")
    flush = L2Flush(torch)
    l0 = ctx.counts()["launches"]
    ms = time_steps(torch, stream, lambda: ctx.jk_stored_dev(nD, dP.data_ptr(), dJK[0].data_ptr(), dJK[1].data_ptr()), steps, warmup, flush)
    if outputs is not None:
        jk = dJK.cpu().numpy()
        outputs["J"], outputs["K"] = (jk[0], jk[1]) if nD > 1 else (jk[0, 0], jk[1, 0])
    launches = ctx.counts()["launches"] - l0 - 2 * warmup * ((nD + 3) // 4)
    # per-launch kernel time from the context's own events on the same stream
    kms = []
    for _ in range(5):
        flush(); torch.cuda.synchronize()
        ctx.jk_stored_dev(nD, dP.data_ptr(), dJK[0].data_ptr(), dJK[1].data_ptr())
        kms.append(ctx.last_kernel_ms(2))
    k_ms = float(np.median(kms))
    alg_bytes = 8.0 * n ** 4 + 8.0 * n * n * (nD + 2 * nD)
    peaks, src = measured_peaks()
    # e2e through the public API with host buffers
    handle = tuna_b200.ERIHandle(ctx, n, "sph", "stored")
    Ph = P if nD > 1 else P[0]
    for _ in range(warmup):
        tuna_b200.coulomb_and_exchange(Ph, handle)
    t = time.perf_counter()
    for _ in range(steps):
        J, K = tuna_b200.coulomb_and_exchange(Ph, handle)
    e2e = steps / (time.perf_counter() - t)
    res = {"workload": wl["description"], "nbf": n, "ncart": wl["ncart"], "value": steps / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / steps,
           "l2": L2_NOTE + "; the 8*nbf^4 tensor is read from HBM",
           "eri_fill_ms": float(min(t_fill)), "cart_to_sph_ms": float(min(t_sph)),
           "eri_quartets_per_s": c["surviving_quartets"] / (min(t_fill) * 1e-3),
           "eri_fill": {"kernels": "k_shell4_multi / k_shell4_one (fill mode) + k_fill_scatter", "ms": float(min(t_fill)),
                        "tensor_write_GBps": 8.0 * wl["ncart"] ** 4 / (min(t_fill) * 1e-3) / 1e9,
                        "note": "Cartesian tensor of 8*ncart^4 bytes built by the shell-quartet engine (scratch rows of the unique integrals, then "
                                "the eight images); not HBM-bound at this size: the class jobs are short latency chains"},
           "roofline": {"bound": "hbm", "achieved": alg_bytes / (k_ms * 1e-3) / 1e9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                        "frac": alg_bytes / (k_ms * 1e-3) / 1e9 / peaks["hbm_gbs"],
                        "traffic": (executed_fp64_table().get(f"stored:{wl['name']}") or {}).get("dram_bytes_per_launch"), "peak_source": src, "kernel": "k_jk_stored_sym + k_sym_reduce (whole J/K build: both launches, CUDA events of the context)",
                        "kernel_ms": k_ms, "algorithmic_bytes": alg_bytes},
           "e2e": {"value": e2e, "unit": UNIT, "h2d_bytes_per_step": int(8 * nD * n * n), "d2h_bytes_per_step": int(16 * nD * n * n)},
           "gpu_launches": int(launches)}
    ctx.set_stream(0)
    return res, ctx


def bench_mo_transform(torch, ctx, wl, fp64_peak, flush):
    """SURVEY.md 8f-2: AO->MO transformation (tuna_ci.py:204-255) of the resident stored tensor of `ctx`, square C.
    Device-resident time = the four k_axis_gemm launches (CUDA events of the context); e2e = the provider call with the
    ERIHandle in and a host ndarray out (D2H of 8 n^4 bytes inside); CPU = the reference's four einsums on the host cores."""
    import tuna_b200
    from oracle import tuna_oracle as orc
    n = wl["nbf"]
    rng = np.random.default_rng(20261018)
    C = np.linalg.qr(rng.standard_normal((n, n)))[0]
    dC = torch.from_numpy(C).cuda()
    dOut = torch.empty((n,) * 4, dtype=torch.float64, device="cuda")
    ms = []
    for it in range(8):
        flush(); torch.cuda.synchronize()
        ctx.eri_transform_dev(n, 0, n, dC.data_ptr(), n, dC.data_ptr(), False, dOut.data_ptr())
        if it >= 3:
            ms.append(ctx.last_kernel_ms(4))
    k_ms = float(np.median(ms))
    flops = 4 * 2.0 * n ** 5
    alg_bytes = 4 * 2 * 8.0 * n ** 4
    handle = tuna_b200.ERIHandle(ctx, n, "sph", "stored")
    T = None
    for _ in range(3):          # warm-up: the page-locked result buffers come from a caching allocator (the first allocations pin 8 n^4 bytes)
        T = None
        T = tuna_b200.transform_ERI_AO_to_MO(handle, C, None, True)
    t = time.perf_counter()
    reps = 5
    for _ in range(reps):
        T = None                # the previous result is released before the next call, as a post-HF driver does with its temporaries
        T = tuna_b200.transform_ERI_AO_to_MO(handle, C, None, True)
    e2e_s = (time.perf_counter() - t) / reps
    E = ctx.eri_download(1)
    tc = []
    for _ in range(2):
        t = time.perf_counter(); ref = orc.transform_eri_ao_to_mo(E, C); tc.append(time.perf_counter() - t)
    err = float(np.abs(T - ref).max())
    return {"workload": f"AO->MO transformation of the stored tensor (nbf {n}, square C), tuna_ci.py:204-255", "value": 1e3 / k_ms, "unit": "transforms/s",
            "ms_per_step": k_ms, "max_abs_diff_vs_oracle": err,
            "roofline": {"bound": "fp64", "achieved": flops / (k_ms * 1e-3) / 1e12, "peak": fp64_peak, "unit": "TFLOP/s",
                         "frac": flops / (k_ms * 1e-3) / 1e12 / fp64_peak if fp64_peak else None,
                         "traffic": (executed_fp64_table().get(f"mo:{wl['name']}") or {}).get("dram_bytes_per_launch"), "kernel": "k_axis_gemm x4",
                         "algorithmic_flops": flops, "algorithmic_bytes": alg_bytes, "hbm_gbs": alg_bytes / (k_ms * 1e-3) / 1e9},
            "e2e": {"value": 1.0 / e2e_s, "unit": "transforms/s", "h2d_bytes_per_step": int(8 * n * n), "d2h_bytes_per_step": int(8 * n ** 4)},
            "cpu_baseline": {"value": 1.0 / min(tc), "unit": "transforms/s", "cores": host_threads(), "kind": "port",
                             "sample": "full workload: the reference's four einsums (numpy/OpenBLAS) on the same tensor, best of 2"},
            "gpu_launches": 4}


def bench_one_electron(wl, charges=(7.0, 7.0)):
    """SURVEY.md 8f-3: one-electron integrals (S, T, V_NE, dipole, quadrupole; pyx:282-445) of the workload's basis through the
    reference-signature call (host lists in, host matrices out) with the reference's compiled engine beside it."""
    import tuna_b200
    from types import SimpleNamespace
    from oracle import tuna_oracle as orc
    bfs = wl["bfs"]
    n = len(bfs)
    zs = sorted({float(np.asarray(b.origin)[2]) for b in bfs})
    atoms = [SimpleNamespace(origin=np.array([0.0, 0.0, z]), charge=float(c)) for z, c in zip(zs, charges)]
    origin = np.array([0.0, 0.0, 0.5 * (zs[0] + zs[-1])])
    tuna_b200.calculate_one_electron_integrals(n, bfs, len(atoms), atoms, origin, 1)          # warm-up (module load, tables)
    ts, ks = [], []
    for _ in range(3):
        ctx = tuna_b200.Context(0)
        from tuna_b200.basis import flatten
        ctx.set_basis(*flatten(bfs))
        t = time.perf_counter()
        got = ctx.one_electron(zs, list(charges), origin)
        ts.append(time.perf_counter() - t)
        ks.append(ctx.last_kernel_ms(5))
        ctx.close()
    out = {"workload": f"one-electron integrals, {wl['description']}", "ncart": n, "kernel_ms": float(np.median(ks)), "call_ms": 1e3 * min(ts),
           "pairs_per_s": n * (n + 1) / 2 / (np.median(ks) * 1e-3), "gpu_launches": 1}
    eng = orc.reference_engine()
    if eng is not None:
        fb = orc.FlatBasis.from_reference_objects(bfs)
        rb = orc.reference_basis_objects(fb)
        tr = []
        for _ in range(2):
            t = time.perf_counter()
            ref = eng.calculate_one_electron_integrals(n, rb, len(atoms), atoms, origin, host_threads())
            tr.append(time.perf_counter() - t)
        out["cpu_baseline"] = {"value_ms": 1e3 * min(tr), "cores": host_threads(), "kind": "reference", "sample": "full workload, best of 2"}
        out["max_abs_diff_vs_reference"] = float(max(np.abs(np.asarray(a) - b).max() for a, b in zip(ref, got)))
    return out


def parity_at_bench_size(wl, tau, builder, rank, P_timed):
    """Evidence that the timed kernels compute the reference's numbers AT THE TIMED SIZE and AT THE TIMED RANK COUNT (no dense tensor exists
    there).  (a) rank 0, single GPU, Cartesian basis: J/K from a unit-pair density P = e_k e_l^T + e_l e_k^T are single integrals,
    J_ij = (ij|kl) + (ij|lk), K_ij = (il|kj) + (ik|lj), which the oracle evaluates one by one for sampled (i, j).  (b) N > 1: the sharded,
    all-reduced build of the TIMED density (every rank takes part) against the unsharded build of the same density on rank 0.
    The oracle is the checker here, never the thing measured."""
    import tuna_b200
    from oracle import tuna_oracle as orc
    from tuna_b200.basis import flatten
    from util import pick_function, unit_pair_density
    out = None
    Jn = Kn = None
    if builder.world > 1:
        Jn, Kn = builder.build(P_timed)
    if rank != 0:
        return None
    bfs = wl["bfs"]
    fb = orc.FlatBasis.from_reference_objects(bfs)
    n = fb.ncart
    Lmax = int(np.asarray(fb.lmn).sum(axis=1).max())
    k, l = pick_function(fb, 0, Lmax, True, 0), pick_function(fb, 1, max(Lmax - 1, 0), False, 0)
    ctx = tuna_b200.Context(builder.ctx.device)
    ctx.set_basis(*flatten(bfs))
    ctx.set_transform(np.eye(n))
    J, K = ctx.jk_direct(unit_pair_density(n, k, l), tau)
    rng = np.random.default_rng(5)
    worst, ok = 0.0, True
    ns = 150
    for i, j in zip(rng.integers(0, n, ns), rng.integers(0, n, ns)):
        i, j = int(i), int(j)
        a, b = orc.eri_single(fb, i, j, k, l), orc.eri_single(fb, i, j, l, k)
        c, d = orc.eri_single(fb, i, l, k, j), orc.eri_single(fb, i, k, l, j)
        for got, ref, scale in ((J[i, j], a + b, max(abs(a), abs(b))), (K[i, j], c + d, max(abs(c), abs(d)))):
            err = abs(got - ref)
            worst = max(worst, err)
            ok = ok and err <= 2 * max(1e-12, 1e-13 * scale)
    out = {"what": "direct J/K from a unit-pair density vs single integrals of the oracle, sampled elements", "samples": 2 * ns, "pair": [k, l],
           "max_abs_diff": worst, "within_tolerance": bool(ok), "tolerance": "2 * max(1e-12, 1e-13 |ERI|) (SURVEY.md 8d)", "ranks": builder.world}
    if builder.world > 1:
        ctx.set_transform(np.asarray(wl["U"]))
        J1, K1 = ctx.jk_direct(P_timed, tau)
        scale = max(1.0, float(np.abs(K1).max()))
        d = float(max(np.abs(np.asarray(Jn) - J1).max(), np.abs(np.asarray(Kn) - K1).max()))
        out["sharded_vs_single_gpu"] = {"what": f"all-reduced build over {builder.world} ranks vs the unsharded build of the timed density on rank 0",
                                        "max_abs_diff": d, "scale": scale, "within_tolerance": bool(d <= 1e-11 * scale), "tolerance": "1e-11 * max(1, max|K|)"}
        out["within_tolerance"] = bool(out["within_tolerance"] and d <= 1e-11 * scale)
    ctx.close()
    return out


def sweep_point(torch, nbf, tau, fp64_peak, device):
    """One extra point of the even-tempered sweep at N=1: device-resident direct Fock builds, CUDA-event timed."""
    import tuna_b200
    from tuna_b200.basis import flatten
    from tuna_b200.distributed import FockBuilder
    wl = load_workload(f"direct:et{nbf}")
    ctx = tuna_b200.Context(device)
    ctx.set_basis(*flatten(wl["bfs"]))
    ctx.set_transform(wl["U"])
    fb = FockBuilder(ctx, nD=1, tau=tau)
    fb.dP.copy_(torch.from_numpy(tuna_b200.workloads.fixed_density(wl["nbf"])[None]))
    flush = L2Flush(torch)
    steps = 10
    ms = time_steps(torch, fb.stream, fb.build_device, steps, 3, flush)
    alg_eri, alg_digest = ctx.algorithmic_flops()
    c = ctx.counts()
    out = {"nbf": wl["nbf"], "ncart": wl["ncart"], "value": steps / (ms * 1e-3), "unit": UNIT, "ms_per_step": ms / steps,
           "eri_quartets_per_s": c["evaluated_last_direct"] * steps / (ms * 1e-3),
           "fp64_frac_algorithmic": (alg_eri + alg_digest) / (ms / steps * 1e-3) / 1e12 / fp64_peak if fp64_peak else None}
    ctx.set_stream(0)
    return out


def run_ours(args, wl):
    import torch
    import torch.distributed as dist
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device — tuna_b200 has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local)
    ddist = None
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        ddist = dist
    import tuna_b200
    from tuna_b200.basis import flatten
    from tuna_b200.distributed import FockBuilder

    sampler = ClockSampler(local)
    if wl["mode"] == "stored":
        if world > 1:
            raise SystemExit("stored mode is a single-GPU workload (SURVEY.md 8e); use a direct: workload for --gpus > 1")
        sampler.start()
        outputs = {} if args.dump_outputs else None
        res, ctx = bench_stored(torch, wl, args.steps, args.warmup, local, outputs)
        clocks = sampler.stop()
        if outputs is not None:
            dump_outputs(args.dump_outputs, outputs)
        line = {"metric": METRIC, "value": res["value"], "unit": UNIT, "n_gpus": 1, "steps": args.steps, "warmup": args.warmup, "ms_per_step": res["ms_per_step"],
                "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
                "config": {"workload": res["workload"], "nbf": res["nbf"], "ncart": res["ncart"], "mode": "stored", "l2": res["l2"]},
                "roofline": res["roofline"], "e2e": res["e2e"], "gpu_launches": res["gpu_launches"], "clocks": clocks,
                "eri_quartets_per_s": res["eri_quartets_per_s"], "eri_fill_ms": res["eri_fill_ms"], "cart_to_sph_ms": res["cart_to_sph_ms"]}
        line["cpu_baseline"] = cpu_reference(wl)
        print(json.dumps(line), flush=True)
        return

    # ---- direct mode (headline) ----
    ctx = tuna_b200.Context(local)
    t0 = time.perf_counter()
    ctx.set_basis(*flatten(wl["bfs"]))
    ctx.set_transform(wl["U"])
    setup_s = time.perf_counter() - t0
    n, nD = wl["nbf"], wl["nD"]
    fb = FockBuilder(ctx, nD=nD, tau=args.tau)
    P = np.stack([tuna_b200.workloads.fixed_density(n)] * nD)
    fb.dP.copy_(torch.from_numpy(P))
    flush = L2Flush(torch)
    fp64_peak = ctx.fp64_peak_probe() if rank == 0 else 0.0
    sampler.start()
    l0 = None
    for _ in range(args.warmup):
        fb.build_device()
    fb.stream.synchronize()
    l0 = ctx.counts()["launches"]
    ms = time_steps(torch, fb.stream, fb.build_device, args.steps, 0, flush, ddist)
    if args.dump_outputs and rank == 0:       # after the all-reduce every rank holds the full J and K
        jk = fb.dJK.cpu().numpy()
        dump_outputs(args.dump_outputs, {"J": jk[0], "K": jk[1]} if nD > 1 else {"J": jk[0, 0], "K": jk[1, 0]})
    launches = ctx.counts()["launches"] - l0
    k_ms = ctx.last_kernel_ms(3)
    evaluated = ctx.counts()["evaluated_last_direct"]
    # e2e: host P in, host J/K out, every step (pinned H2D + kernels + all-reduce + D2H)
    for _ in range(max(1, args.warmup // 2)):
        fb.build(P)
    if ddist is not None:
        ddist.barrier()
    torch.cuda.synchronize()
    t = time.perf_counter()
    for _ in range(args.steps):
        J, K = fb.build(P)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t
    if ddist is not None:
        tt = torch.tensor([e2e_s, float(evaluated), k_ms], dtype=torch.float64, device="cuda")
        mx = tt.clone(); ddist.all_reduce(mx, op=ddist.ReduceOp.MAX)
        sm = tt.clone(); ddist.all_reduce(sm, op=ddist.ReduceOp.SUM)
        e2e_s, evaluated, k_ms = float(mx[0]), int(sm[1].item()), float(mx[2])
    clocks = sampler.stop()
    try:       # evidence only; never allowed to take the line down (collective: every rank calls it)
        parity = parity_at_bench_size(wl, args.tau, fb, rank, P if nD > 1 else P[0])
    except Exception as e:
        parity = {"error": str(e)}
    if rank != 0:
        if ddist is not None:
            ddist.destroy_process_group()
        return
    c = ctx.counts()
    alg_eri, alg_digest = ctx.algorithmic_flops()
    # SURVEY.md 8d: screened-out quartets are not work done - the algorithmic count is scaled to the EVALUATED share of the surviving quartets
    eval_share = evaluated / max(1, c["surviving_quartets"])
    alg = (alg_eri + alg_digest * nD) * eval_share
    builds_per_s = args.steps / (ms * 1e-3)
    alg_rate = alg / world / (k_ms * 1e-3) / 1e12           # this rank's share of the algorithmic flops over its kernel time
    ex = executed_fp64_table().get(f"{wl['name']}|{nD}|{args.tau:g}")
    ex_rate = ex["fp64_flops_per_build"] / world / (k_ms * 1e-3) / 1e12 if ex else None
    roofline = {"bound": "fp64", "achieved": ex_rate, "peak": fp64_peak, "unit": "TFLOP/s",
                "frac": (ex_rate / fp64_peak) if (ex_rate is not None and fp64_peak) else None,
                "traffic": ex.get("dram_bytes_per_build") if ex else None,
                "basis": "EXECUTED FP64 flops of one build (ncu: 2*DFMA + DMUL + DADD thread instructions over all class-job launches, "
                         "profiles/executed_fp64.json) over this run's kernel time; null when no ncu count exists for this workload",
                "peak_source": "sustained FP64 DFMA stream measured in this run (tuna_fp64_peak_probe, >= 0.5 s); MEASURED_PEAKS.json has no FP64 entry",
                "kernel": "k_shell4_one (all class jobs of one build)", "kernel_ms": k_ms,
                "algorithmic": {"flops_evaluated": alg, "tflops": alg_rate, "frac": alg_rate / fp64_peak if fp64_peak else None, "evaluated_share": eval_share,
                                "note": "the reference algorithm's flop count F(a,b) (SURVEY.md 8d) + 12 flops/quartet/density of digestion, over the "
                                        "quartets that survive parity AND Schwarz screening; the engine shares Boys/R/convolution tables among all "
                                        "components of a shell quartet and therefore executes far fewer flops"}}
    if ex:
        roofline["executed"] = ex
    line = {"metric": METRIC, "value": builds_per_s, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": wl["description"], "nbf": n, "ncart": wl["ncart"], "mode": "direct", "densities": nD, "schwarz_tau": args.tau,
                       "parallelism": f"quartet list sharded over {world} GPU(s), one all-reduce of J/K per build",
                       "l2": L2_NOTE + "; inputs (pair table, P) are re-read from HBM each step",
                       "pair_table_setup_s": setup_s,
                       "parity": {"within_tolerance": parity.get("within_tolerance"), "max_abs_diff": parity.get("max_abs_diff"),
                                  "sharded_max_abs_diff": (parity.get("sharded_vs_single_gpu") or {}).get("max_abs_diff"), "error": parity.get("error")}},
            "eri_quartets_per_s": evaluated * builds_per_s, "surviving_quartets": c["surviving_quartets"], "evaluated_quartets": evaluated,
            "unique_quartets_per_s": c["unique_quartets"] * builds_per_s,
            "roofline": roofline,
            "e2e": {"value": args.steps / e2e_s, "unit": UNIT, "h2d_bytes_per_step": int(fb.h2d_bytes), "d2h_bytes_per_step": int(fb.d2h_bytes)},
            "gpu_launches": int(launches), "clocks": clocks, "parity": parity}
    if world == 1:
        line["cpu_baseline"] = cpu_reference(wl)
        if not args.no_stored:
            fb = None
            ctx.set_stream(0)
            swl = load_workload("stored:n2_ccpvtz")
            sres, sctx = bench_stored(torch, swl, max(args.steps, 20), max(args.warmup, 3), local)
            sres["cpu_baseline"] = cpu_reference(swl)
            line["stored"] = sres
            try:
                line["mo_transform"] = bench_mo_transform(torch, sctx, swl, fp64_peak, L2Flush(torch))
            except Exception as e:       # an extra (SURVEY.md 8f-2), never allowed to take the headline line down
                line["mo_transform"] = {"error": str(e)}
            sctx = None
            lwl = load_workload("stored:et100")       # the same stored kernel on a tensor well above L2 (0.8 GB): the HBM-stream regime
            lwl["description"] = "stored mode at nbf 100 (even-tempered N2, 0.8 GB tensor), 1 density"
            lres, lctx = bench_stored(torch, lwl, max(args.steps, 20), max(args.warmup, 3), local)
            line["stored_large"] = lres
            lctx = None
            line["sweep"] = [sweep_point(torch, nb, args.tau, fp64_peak, local) for nb in (100, 200, 400) if f"et{nb}" != wl["name"]]
            # extra (SURVEY.md 8f-3): in a child process, so that nothing in it can take the headline line down
            try:
                r = subprocess.run([sys.executable, os.path.abspath(__file__), "--extra-one-electron", "--workload", args.workload],
                                   capture_output=True, text=True, timeout=240)
                line["one_electron"] = json.loads(r.stdout.strip().splitlines()[-1]) if r.returncode == 0 and r.stdout.strip() else {"error": (r.stderr or "no output")[-300:]}
            except Exception as e:
                line["one_electron"] = {"error": str(e)}
    print(json.dumps(line), flush=True)
    if ddist is not None:
        ddist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=os.environ.get("TUNA_BENCH_WORKLOAD", "direct:et800"))
    ap.add_argument("--tau", type=float, default=1e-16)
    ap.add_argument("--no-stored", action="store_true", help="skip the extra stored-mode (configs[1]) and sweep measurements at N=1")
    ap.add_argument("--extra-one-electron", action="store_true", help=argparse.SUPPRESS)
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write J and K of the last timed step as DIR/J.npy and "
                                                          "DIR/K.npy (float64; a fixed, seeded sample above 64 MB in all)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs needs --impl ours")
    if args.extra_one_electron:       # child of the N=1 run: one-electron integrals of configs[1] and of the headline basis
        print(json.dumps([bench_one_electron(load_workload("stored:n2_ccpvtz")), bench_one_electron(load_workload(args.workload))]), flush=True)
        return
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    wl = load_workload(args.workload)
    if args.impl == "reference":
        run_reference_arm(args, wl)
    else:
        run_ours(args, wl)


if __name__ == "__main__":
    main()
