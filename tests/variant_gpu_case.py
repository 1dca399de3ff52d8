"""One knob configuration of the direct engine (run by tests/test_kernel_variants.py in a child process, with the TUNA_B200_* knobs of
the configuration in its environment): direct J/K of the coverage basis and of N2/cc-pVTZ at tau = 0 and 1e-16, the two shard
partials of a two-rank split, and one engine fill of the dense tensor.  Everything goes to OUT_DIR as .npy files, with the job table
of every job set the engine built (TUNA_B200_DUMP_JOBS) as jobs_<basis>_<call>.csv; the parent compares them with the oracle."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))


def main(out_dir):
    import tuna_b200
    from tuna_b200.basis import flatten
    from test_kernel_variants import coverage_basis, densities
    from util import basis_objects, load_golden
    for name in ("coverage", "n2_ccpvtz"):
        bfs = coverage_basis() if name == "coverage" else basis_objects(load_golden(name))
        n = len(bfs)
        P = densities(n)
        ctx = tuna_b200.Context(0)
        ctx.set_basis(*flatten(bfs))
        ctx.set_transform(np.eye(n))

        def run(tag, *args):
            os.environ["TUNA_B200_DUMP_JOBS"] = os.path.join(out_dir, f"jobs_{name}_{tag}.csv")
            return ctx.jk_direct(*args) if args else ctx.eri_fill_cart()

        for tau in (0.0, 1e-16):
            J, K = run(f"tau{tau:g}", P, tau)
            np.save(os.path.join(out_dir, f"{name}_J_tau{tau:g}.npy"), J)
            np.save(os.path.join(out_dir, f"{name}_K_tau{tau:g}.npy"), K)
        for r in range(2):
            ctx.set_shard(r, 2)
            J, K = run(f"shard{r}", P, 0.0)
            np.save(os.path.join(out_dir, f"{name}_J_shard{r}.npy"), J)
            np.save(os.path.join(out_dir, f"{name}_K_shard{r}.npy"), K)
        ctx.set_shard(0, 1)
        os.environ["TUNA_B200_FILL_ENGINE"] = "1"
        run("fill")
        del os.environ["TUNA_B200_FILL_ENGINE"]
        np.save(os.path.join(out_dir, f"{name}_fill.npy"), ctx.eri_download(0))
        ctx.close()
    print("ok")


if __name__ == "__main__":
    main(sys.argv[1])
