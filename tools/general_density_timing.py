"""Direct J/K of device-resident densities of any real P (tuna_jk_direct_general_dev), alternated in one process against the paths it
replaces or extends:

  (a) asymmetric P (the recorded final densities + 1e-8 times a seeded antisymmetric matrix): host tuna_jk_direct (P on the host, the
      split on the host, H2D, D2H, K[S] + K[A] on the host) against tuna_jk_direct_general_dev (P, J and K on the device);
  (b) symmetric P scaled to max|P| = 1 (so both paths keep the default pre-screening bound and run the same build): tuna_jk_direct_dev
      against tuna_jk_direct_general_dev, i.e. the cost of the density scan, its read-back and the copy into the staging buffer.

Every build is bracketed by CUDA events on the launching stream (the host entry point and the general one synchronise inside; the events
still span the whole call), with L2 flushed before it as in bench.py.  Each arm has its own context; J and K of every pair must be bitwise
equal.  Prints the card name and power limit first, then one JSON line per workload (development aid).

    python tools/general_density_timing.py [out.log] [workloads ...]      (default: n2_ccpvtz ne2_uhf_ccpvqz et200)"""
import json
import os
import subprocess
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch  # noqa: E402  (plumbing: device buffers, streams, events)
import tuna_b200  # noqa: E402
from tuna_b200 import workloads as w  # noqa: E402
from tuna_b200.basis import flatten, from_arrays  # noqa: E402
from util import basis_objects, load_golden  # noqa: E402

REPS = 10
TAU = 1e-16


def card():
    try:
        q = subprocess.run(["nvidia-smi", "--id=0", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                           capture_output=True, text=True, timeout=60)
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


def run(name, flush):
    flat, U, P = case(name)
    nD, nbf = P.shape[0], U.shape[0]
    A = np.random.default_rng(7).standard_normal(P.shape)
    asym = P + 1e-8 * (A - A.transpose(0, 2, 1))
    sym = P / np.abs(P).max()
    stream = torch.cuda.Stream()
    ctxs = {}
    for arm in ("host", "general_a", "dev", "general_b"):
        c = tuna_b200.Context(0)
        c.set_basis(*flat)
        c.set_transform(U)
        c.set_stream(stream.cuda_stream)
        ctxs[arm] = c
    d_asym, d_sym = torch.from_numpy(asym).cuda(), torch.from_numpy(sym).cuda()
    out = {arm: (torch.empty_like(d_asym), torch.empty_like(d_asym)) for arm in ctxs}
    host_out = {}

    def call(arm):
        c, (dJ, dK) = ctxs[arm], out[arm]
        if arm == "host":
            host_out[arm] = c.jk_direct(asym, TAU)
        elif arm == "general_a":
            c.jk_direct_general_dev(nD, d_asym.data_ptr(), dJ.data_ptr(), dK.data_ptr(), TAU)
        elif arm == "dev":
            c.jk_direct_dev(nD, d_sym.data_ptr(), dJ.data_ptr(), dK.data_ptr(), TAU)
        else:
            c.jk_direct_general_dev(nD, d_sym.data_ptr(), dJ.data_ptr(), dK.data_ptr(), TAU)

    def timed(arm):
        flush()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        call(arm)
        e1.record(stream)
        e1.synchronize()
        return e0.elapsed_time(e1)

    for arm in ctxs:                          # job lists, class tables, module load (untimed)
        timed(arm)
    ms = {arm: [] for arm in ctxs}
    equal_a = equal_b = True
    for _ in range(REPS):
        for arm in ctxs:
            ms[arm].append(timed(arm))
        J, K = host_out["host"]
        equal_a &= bool(np.array_equal(out["general_a"][0].cpu().numpy(), J.reshape(out["general_a"][0].shape))
                        and np.array_equal(out["general_a"][1].cpu().numpy(), K.reshape(out["general_a"][1].shape)))
        equal_b &= bool(torch.equal(out["dev"][0], out["general_b"][0]) and torch.equal(out["dev"][1], out["general_b"][1]))
    for c in ctxs.values():
        c.set_stream(0)
        c.close()
    med = {arm: float(np.median(v)) for arm, v in ms.items()}
    return {"workload": name, "nbf": nbf, "nD": nD,
            "a_asymmetric": {"host_jk_direct_ms": med["host"], "general_dev_ms": med["general_a"],
                             "speedup": med["host"] / med["general_a"], "bitwise_equal": equal_a},
            "b_symmetric": {"jk_direct_dev_ms": med["dev"], "general_dev_ms": med["general_b"],
                            "extra_ms": med["general_b"] - med["dev"], "bitwise_equal": equal_b},
            "all_ms": ms,
            "timing": "CUDA events on the launching stream around the whole call, L2 flushed before every build, median of %d" % REPS}


def main():
    out = sys.argv[1] if len(sys.argv) > 1 else None
    names = sys.argv[2:] or ["n2_ccpvtz", "ne2_uhf_ccpvqz", "et200"]
    lines = [f"card: {card()}"]
    print(lines[0], flush=True)
    flush = L2Flush()
    for name in names:
        lines.append(json.dumps(run(name, flush)))
        print(lines[-1], flush=True)
    if out:
        with open(out, "w") as f:
            f.write("\n".join(lines) + "\n")


if __name__ == "__main__":
    main()
