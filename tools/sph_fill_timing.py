"""Spherical ERI tensor: eri_fill_sph (one pass, no Cartesian tensor) against eri_fill_cart + eri_cart_to_sph, alternated in one process.

Per workload and repetition: CUDA-event time of each path (tuna_last_kernel_ms: 0 = fill, 1 = rotation), host time around the call (it ends
in a device synchronise), and the peak device memory of the call, taken as the drop of cudaMemGetInfo's free bytes below the value before the
call, polled from a second thread.  Prints the card name and power limit first and one JSON line per workload (development aid)."""
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
import torch  # noqa: E402  (plumbing: cudaMemGetInfo)
import tuna_b200  # noqa: E402
from util import context_for, load_golden  # noqa: E402


def peak_bytes(fn):
    """(result of fn, largest drop of free device memory during fn, host seconds)."""
    torch.cuda.synchronize()
    free0 = torch.cuda.mem_get_info(0)[0]
    low = [free0]
    done = threading.Event()

    def poll():
        while not done.is_set():
            low[0] = min(low[0], torch.cuda.mem_get_info(0)[0])
            time.sleep(0.0002)
    t = threading.Thread(target=poll)
    t.start()
    t0 = time.perf_counter()
    r = fn()
    dt = time.perf_counter() - t0
    done.set()
    t.join()
    low[0] = min(low[0], torch.cuda.mem_get_info(0)[0])
    return r, free0 - low[0], dt


def main():
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    print(json.dumps({"card": card}), flush=True)
    reps = 5
    for name in sys.argv[1:] or ["n2_ccpvtz", "ne2_uhf_ccpvqz"]:
        g = load_golden(name)
        ctx = context_for(g)
        ctx.set_transform(g["U"])
        nbf, nc = int(ctx.nbf), int(ctx.ncart)
        out = {"name": name, "ncart": nc, "nbf": nbf, "old_ms": [], "old_fill_ms": [], "old_rot_ms": [], "new_ms": [],
               "old_host_ms": [], "new_host_ms": [], "old_peak_GB": [], "new_peak_GB": []}

        def old():
            ctx.eri_fill_cart()
            ctx.eri_cart_to_sph()

        tensors = {}
        for rep in range(reps + 1):             # repetition 0 is the warm-up (module load, first allocations)
            _, pk, dt = peak_bytes(old)
            f, r = ctx.last_kernel_ms(0), ctx.last_kernel_ms(1)
            if rep:
                out["old_fill_ms"].append(round(f, 4)); out["old_rot_ms"].append(round(r, 4)); out["old_ms"].append(round(f + r, 4))
                out["old_host_ms"].append(round(1e3 * dt, 3)); out["old_peak_GB"].append(round(pk / 1e9, 3))
            tensors["old"] = ctx.eri_download(1)
            ctx.eri_upload(np.zeros((1, 1, 1, 1)))      # release the stored tensor so that both paths start from the same free memory
            _, pk, dt = peak_bytes(ctx.eri_fill_sph)
            if rep:
                out["new_ms"].append(round(ctx.last_kernel_ms(0), 4))
                out["new_host_ms"].append(round(1e3 * dt, 3)); out["new_peak_GB"].append(round(pk / 1e9, 3))
            tensors["new"] = ctx.eri_download(1)
            ctx.eri_upload(np.zeros((1, 1, 1, 1)))
        out["tensor_GB"] = round(8 * nbf ** 4 / 1e9, 3)
        out["cart_path_model_GB"] = round(8 * (nc ** 4 + nbf * nc ** 3 + nbf ** 4) / 1e9, 3)
        out["max_abs_diff"] = float(np.abs(tensors["old"] - tensors["new"]).max())
        out["max_abs"] = float(np.abs(tensors["old"]).max())
        print(json.dumps(out), flush=True)
        ctx.close()


if __name__ == "__main__":
    main()
