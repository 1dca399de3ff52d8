"""A direct J/K call whose job-set build fails must leave nothing behind (run by tests/test_context_buffers.py in a child process,
with TUNA_B200_NB=4 and TUNA_B200_NB_BYTES=1000000000 in its environment).

Four quartets per batch of the coverage basis's h-shell classes do not fit the 226 KB shared-memory layout of ensure_shell4
((hh|hh) alone needs 4 x 19898 doubles), so the first jk_direct fails.  A second identical call must fail the same way without
launching anything, and once both knobs are gone (ensure_shell4 reads them on every call) the same context must give J/K bitwise
equal to a fresh context's.  Prints "ok" when all of this holds."""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))


def main():
    import tuna_b200
    from tuna_b200._lib import TunaError
    from tuna_b200.basis import flatten
    from test_kernel_variants import coverage_basis, densities
    assert os.environ.get("TUNA_B200_NB") == "4" and os.environ.get("TUNA_B200_NB_BYTES") == "1000000000"
    bfs = coverage_basis()
    n = len(bfs)
    P = densities(n)

    def context():
        ctx = tuna_b200.Context(0)
        ctx.set_basis(*flatten(bfs))
        ctx.set_transform(np.eye(n))
        return ctx

    ctx = context()
    msgs = []
    for attempt in range(2):
        launches = ctx.counts()["launches"]
        try:
            ctx.jk_direct(P, 0.0)
        except TunaError as e:
            msgs.append(str(e))
        else:
            raise AssertionError(f"call {attempt + 1}: the job-set build did not fail")
        if attempt == 1:
            assert ctx.counts()["launches"] == launches, "the failed second call launched kernels"
    assert "226 KB" in msgs[0] and msgs[1] == msgs[0], msgs
    del os.environ["TUNA_B200_NB"], os.environ["TUNA_B200_NB_BYTES"]
    J, K = ctx.jk_direct(P, 0.0)
    fresh = context()
    J0, K0 = fresh.jk_direct(P, 0.0)
    assert np.array_equal(J, J0) and np.array_equal(K, K0), "J/K after the failed build differ from a fresh context's"
    fresh.close()
    ctx.close()
    print("ok:", msgs[0])


if __name__ == "__main__":
    main()
