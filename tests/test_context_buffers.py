"""Ownership of the context's device and pinned memory (tuna_b200/csrc/devbuf.hpp).

Every buffer of tuna_b200.cu is a DevBuf / PinnedBuf: the CPU test keeps raw CUDA allocation calls and hand-kept capacity
bookkeeping out of the rest of the sources.  The GPU tests check that a failed call leaves the context usable: a job set whose
build fails is not cached, and a refused allocation leaves no buffer that claims memory it does not have."""
import os
import re
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
CSRC = os.path.join(ROOT, "tuna_b200", "csrc")


def _sources():
    for name in sorted(os.listdir(CSRC)):
        if name.endswith((".cu", ".cuh", ".hpp", ".h")):
            with open(os.path.join(CSRC, name)) as f:
                yield name, f.read()


def test_allocation_only_through_the_buffer_header():
    alloc = re.compile(r"\b(cudaMalloc|cudaMallocHost|cudaFree|cudaFreeHost)\s*\(")
    manual = re.compile(r"\b(cap_\w+|dev_alloc|dev_free|free_jobset4|basis_dev_free)\b")
    seen = []
    for name, text in _sources():
        seen.append(name)
        if name != "devbuf.hpp":
            assert not alloc.search(text), f"{name} allocates or frees outside devbuf.hpp: {alloc.findall(text)}"
        assert not manual.search(text), f"{name} keeps manual buffer bookkeeping: {sorted(set(manual.findall(text)))}"
    assert "devbuf.hpp" in seen and "tuna_b200.cu" in seen


@pytest.mark.gpu
def test_failed_jobset_build_leaves_nothing_behind():
    from test_kernel_variants import _KNOBS
    env = {k: v for k, v in os.environ.items() if k not in {"TUNA_B200_" + x for x in _KNOBS}}
    env.update(TUNA_B200_NB="4", TUNA_B200_NB_BYTES="1000000000")
    r = subprocess.run([sys.executable, os.path.join(HERE, "jobset_failure_case.py")], env=env, cwd=ROOT, capture_output=True, text=True,
                       timeout=900)
    assert r.returncode == 0 and "ok" in r.stdout, f"child failed (rc {r.returncode}):\n{r.stdout[-2000:]}{r.stderr[-4000:]}"


@pytest.mark.gpu
def test_refused_allocation_leaves_a_usable_context():
    import torch
    import tuna_b200
    n, nmo = 24, 6
    rng = np.random.default_rng(7)
    E = rng.standard_normal((n, n, n, n))
    C = rng.standard_normal((n, nmo))
    ctx = tuna_b200.Context(0)
    # n = 32768, n1 = n2 = 1: the first work buffer is n^3 doubles (~2.8e14 bytes), which cudaMalloc refuses without allocating
    big = 32768
    dT, dC1, dC2, dOut = (torch.zeros(k, dtype=torch.float64, device="cuda:0") for k in (16, big, big, 1))
    with pytest.raises(MemoryError):
        ctx.eri_transform_dev(big, dT.data_ptr(), 1, dC1.data_ptr(), 1, dC2.data_ptr(), False, dOut.data_ptr())
    got = ctx.eri_transform(C, eri=E)
    fresh = tuna_b200.Context(0)
    want = fresh.eri_transform(C, eri=E)
    assert np.array_equal(got, want)
    fresh.close()
    ctx.close()
