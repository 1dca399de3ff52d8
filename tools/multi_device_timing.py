"""Direct J/K of one Fock build over N GPUs of one process (tuna_b200.DeviceGroup) next to the torch.distributed path (bench.py under
torchrun, one process per GPU, tuna_b200.distributed.FockBuilder) at the same N and workload:

    python tools/multi_device_timing.py [out.json]

For ET800, ET400 (nD = 1, workloads.fixed_density) and Ne2 UHF/cc-pVQZ (nD = 2, the final alpha/beta densities) at every N of 1, 2, 4, 8
the box has, one JSON record with
  create_s        DeviceGroup creation + set_basis + set_transform (once per geometry), and first_build_s, the first build (job lists)
  dev_builds_s    builds/s of jk_direct_dev, P resident on devices[0]: host clock around the call ending in a device synchronise,
                  3 warm-ups, median of 10 timed builds
  host_builds_s   the same for jk_direct with host P, J, K
  rank_kernel_ms  each rank's last_kernel_ms(3) of the last build (its accumulation; the spread is the load imbalance)
  reduce_ms       last_kernel_ms(6) on devices[0]: end of the last rank's accumulation -> J/K ready (pull, sum, finish); N > 1
  bench           bench.py's JSON line for the same workload and N (torchrun for N > 1)
plus the card name and power limit.  Needs CUDA devices; there is no CPU path."""
import json
import os
import statistics
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

WORKLOADS = {"et800": ["--workload", "direct:et800"], "et400": ["--workload", "direct:et400"],
             "ne2": ["--workload", "direct:ne2_uhf_ccpvqz", "--no-stored"]}


def case(name):
    from tuna_b200 import workloads as w
    from tuna_b200.basis import flatten, from_arrays
    from util import basis_objects, load_golden
    if name == "ne2":
        g = load_golden("ne2_uhf_ccpvqz")
        return flatten(basis_objects(g)), np.array(g["U"]), np.stack([np.array(g["P_alpha_final"]), np.array(g["P_beta_final"])])
    b = w.even_tempered_diatomic(int(name[2:]))
    bfs = from_arrays(b["origins"], b["lmn"], b["nprim"], b["exps"], b["raw_coefs"])
    return flatten(bfs), np.eye(len(bfs)), w.fixed_density(len(bfs))[None]


def time_builds(fn, sync, warmup=3, steps=10):
    for _ in range(warmup):
        fn()
    sync()
    ts = []
    for _ in range(steps):
        t0 = time.perf_counter()
        fn()
        sync()
        ts.append(time.perf_counter() - t0)
    return 1.0 / statistics.median(ts)


def measure(name, devices):
    import torch
    import tuna_b200
    flat, U, P = case(name)
    dev = torch.device("cuda", devices[0])
    sync = lambda: torch.cuda.synchronize(dev)      # contexts[0]'s stream waits for every rank, so devices[0] finishing means all did
    t0 = time.perf_counter()
    group = tuna_b200.DeviceGroup(devices)
    group.set_basis(*flat)
    group.set_transform(U)
    create = time.perf_counter() - t0
    t0 = time.perf_counter()
    J, K = group.jk_direct(P, 1e-16)
    first = time.perf_counter() - t0
    nD = P.shape[0]
    dP = torch.from_numpy(np.ascontiguousarray(P)).to(dev)
    dJ, dK = torch.empty_like(dP), torch.empty_like(dP)
    sync()
    dev_rate = time_builds(lambda: group.jk_direct_dev(nD, dP.data_ptr(), dJ.data_ptr(), dK.data_ptr(), 1e-16), sync)
    host_rate = time_builds(lambda: group.jk_direct(P, 1e-16), sync)
    rank_ms = [c.last_kernel_ms(3) for c in group.contexts]
    reduce_ms = group.contexts[0].last_kernel_ms(6) if len(devices) > 1 else None
    group.close()
    return dict(workload=name, n=len(devices), nD=nD, nbf=int(U.shape[0]), create_s=create, first_build_s=first, dev_builds_s=dev_rate,
                host_builds_s=host_rate, rank_kernel_ms=rank_ms, reduce_ms=reduce_ms, checksum=[float(np.abs(J).sum()), float(np.abs(K).sum())])


def bench(name, n):
    args = ["bench.py", "--gpus", str(n), "--steps", "10", "--warmup", "3"] + WORKLOADS[name]
    cmd = ([sys.executable, "-m", "torch.distributed.run", "--nnodes=1", f"--nproc-per-node={n}", "--master-addr", "127.0.0.1",
            "--master-port", "29711"] if n > 1 else [sys.executable]) + args
    r = subprocess.run(cmd, capture_output=True, text=True, cwd=ROOT, timeout=600)
    lines = [line for line in r.stdout.splitlines() if line.startswith("{")]
    return json.loads(lines[-1]) if r.returncode == 0 and lines else {"rc": r.returncode, "stderr": r.stderr[-2000:]}


def main():
    import torch
    out = sys.argv[1] if len(sys.argv) > 1 else None
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True)
    ngpu = torch.cuda.device_count()
    if ngpu < 1:
        raise SystemExit("no CUDA device")
    records = [{"gpus": q.stdout.strip().splitlines(), "device_count": ngpu}]
    for name in WORKLOADS:
        for n in (1, 2, 4, 8):
            if n > ngpu:
                continue
            rec = measure(name, list(range(n)))
            rec["bench"] = bench(name, n)
            print(json.dumps(rec), flush=True)
            records.append(rec)
    if out:
        with open(out, "w") as f:
            json.dump(records, f, indent=1)


if __name__ == "__main__":
    main()
