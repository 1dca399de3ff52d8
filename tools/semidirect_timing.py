"""Semi-direct J/K: direct builds against builds replayed from the integral store, alternated in one process.

Per workload: one Context without the store and one with it (budget: everything that fits).  The first build of the second context is
the store pass; its time against a direct build is the store's extra cost.  Then direct and replayed builds alternate (CUDA events on the
launching stream around tuna_jk_direct_dev, L2 flushed before every build as in bench.py) and the J/K of every pair must be bitwise equal.
ET800 runs on a DeviceGroup of 8 devices when 8 are visible (host clock around tuna_jk_direct_group, which ends in a synchronise).
Prints the card name, power limit and free memory first, then one JSON line per workload (development aid).

    python tools/semidirect_timing.py [out.log] [workloads ...]      (default: n2_ccpvtz ne2_uhf_ccpvqz et200 et400 [et800 on 8 GPUs])"""
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch  # noqa: E402  (plumbing: device buffers, events, cudaMemGetInfo)
import tuna_b200  # noqa: E402
from tuna_b200 import workloads as w  # noqa: E402
from tuna_b200.basis import flatten, from_arrays  # noqa: E402
from util import basis_objects, load_golden  # noqa: E402

REPS = 5
TAU = 1e-16
BIG = 1 << 50


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,memory.total", "--format=csv,noheader"], capture_output=True, text=True, timeout=60)
        return q.stdout.strip()
    except Exception as e:      # noqa: BLE001
        return f"nvidia-smi unavailable ({e})"


def case(name):
    if name.startswith("et") and name != "et100":
        b = w.even_tempered_diatomic(int(name[2:]))
        bfs = from_arrays(b["origins"], b["lmn"], b["nprim"], b["exps"], b["raw_coefs"])
        return flatten(bfs), np.eye(len(bfs)), w.fixed_density(len(bfs))[None]
    g = load_golden(name)
    P = np.stack([g["P_alpha_final"], g["P_beta_final"]]) if bool(g["unrestricted"]) else np.array(g["P_final"])[None]
    return flatten(basis_objects(g)), np.array(g["U"]), P


class L2Flush:       # as bench.py: write 256 MB, then read another 256 MB so that L2 holds clean lines
    def __init__(self):
        self.a = torch.zeros(64 * 1024 * 1024, dtype=torch.float32, device="cuda")
        self.b = torch.ones(64 * 1024 * 1024, dtype=torch.float32, device="cuda")

    def __call__(self):
        self.a.add_(1.0)
        self.sink = torch.sum(self.b)


def one_device(name, flush):
    flat, U, P = case(name)
    nD, nbf = P.shape[0], U.shape[0]
    stream = torch.cuda.Stream()
    ctxs = []
    for budget in (0, BIG):
        c = tuna_b200.Context(0)
        c.set_basis(*flat)
        c.set_transform(U)
        c.set_integral_store(budget)
        c.set_stream(stream.cuda_stream)
        ctxs.append(c)
    dP = torch.from_numpy(np.ascontiguousarray(P)).cuda()
    outs = [[torch.empty_like(dP), torch.empty_like(dP)] for _ in ctxs]

    def build(i):
        flush()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        ctxs[i].jk_direct_dev(nD, dP.data_ptr(), outs[i][0].data_ptr(), outs[i][1].data_ptr(), TAU)
        e1.record(stream)
        e1.synchronize()
        return e0.elapsed_time(e1)

    build(0)                                     # job lists, class tables, module load (untimed)
    free_before = torch.cuda.mem_get_info(0)[0]
    t_direct0 = build(0)
    t_store = build(1)                           # the store pass
    free_after = torch.cuda.mem_get_info(0)[0]
    direct, replay = [], []
    equal = True
    for _ in range(REPS):
        direct.append(build(0))
        replay.append(build(1))
        equal &= bool(torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][1], outs[1][1]))
    info = ctxs[1].integral_store_info()
    for c in ctxs:
        c.set_stream(0)
        c.close()
    md, mr = float(np.median(direct)), float(np.median(replay))
    return {"workload": name, "nbf": nbf, "nD": nD, "devices": 1, "direct_ms": md, "replay_ms": mr, "speedup": md / mr,
            "store_pass_ms": t_store, "store_extra_ms": t_store - t_direct0, "direct_ms_all": direct, "replay_ms_all": replay,
            "store_bytes": info["bytes"], "items_stored": info["items"], "items_of_job_set": info["items_last_build"],
            "replayed_builds": info["replayed_builds"], "free_bytes_before_store": free_before, "free_bytes_after_store": free_after,
            "bitwise_equal": equal, "timing": "CUDA events on the launching stream, L2 flushed before every build, median of %d" % REPS}


def group(name, n):
    flat, U, P = case(name)
    groups = []
    for budget in (0, BIG):
        gr = tuna_b200.DeviceGroup(list(range(n)))
        gr.set_basis(*flat)
        gr.set_transform(U)
        gr.set_integral_store(budget)
        groups.append(gr)

    def build(i):
        t0 = time.perf_counter()
        r = groups[i].jk_direct(P, TAU)
        return (time.perf_counter() - t0) * 1e3, r

    build(0)
    free_before = [torch.cuda.mem_get_info(d)[0] for d in range(n)]
    t_direct0, _ = build(0)
    t_store, _ = build(1)
    free_after = [torch.cuda.mem_get_info(d)[0] for d in range(n)]
    direct, replay, equal = [], [], True
    for _ in range(REPS):
        td, rd = build(0)
        tr, rr = build(1)
        direct.append(td); replay.append(tr)
        equal &= bool(np.array_equal(rd[0], rr[0]) and np.array_equal(rd[1], rr[1]))
    info = groups[1].integral_store_info()
    for gr in groups:
        gr.close()
    md, mr = float(np.median(direct)), float(np.median(replay))
    return {"workload": name, "devices": n, "direct_ms": md, "replay_ms": mr, "speedup": md / mr, "store_pass_ms": t_store,
            "store_extra_ms": t_store - t_direct0, "store_bytes": info["bytes"], "items_stored": info["items"],
            "items_of_job_set": info["items_last_build"], "free_bytes_before_store": free_before, "free_bytes_after_store": free_after,
            "bitwise_equal": equal, "timing": "host clock around tuna_jk_direct_group (host P in, J and K out), median of %d" % REPS}


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else None
    names = sys.argv[2:] or ["n2_ccpvtz", "ne2_uhf_ccpvqz", "et200", "et400"]
    lines = [f"card: {card()}", f"free bytes on device 0 at start: {torch.cuda.mem_get_info(0)[0]}"]
    print(lines[0], flush=True); print(lines[1], flush=True)
    flush = L2Flush()
    for name in names:
        r = one_device(name, flush)
        lines.append(json.dumps(r))
        print(lines[-1], flush=True)
    if not sys.argv[2:] and torch.cuda.device_count() >= 8:
        r = group("et800", 8)
        lines.append(json.dumps(r))
        print(lines[-1], flush=True)
    if out:
        with open(out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
