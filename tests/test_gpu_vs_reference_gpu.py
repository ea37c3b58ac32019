"""GPU kernel against GPU kernel: this engine vs the reference's own dpf_hybrid_kernel, compiled
unmodified for sm_100a.  Its results for these inputs are stored in tests/golden/reference_gpu_v1.npz
(tests/golden/make_reference_checks.py gpu).  Same keys, same table, results must be bit-identical."""
import os

import numpy as np
import pytest
import torch

import b200dpf
from common import random_table, seeded_keys

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def reference_gpu():
    if not torch.cuda.is_available():
        pytest.fail("GPU test selected but no CUDA device is visible")
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_gpu_v1.npz"))


@pytest.mark.parametrize("prf", [0, 1, 2, 3])
def test_same_results_as_reference_kernel(reference_gpu, prf):
    n, batch = 4096, 70
    table = random_table(n, 16, seed=prf, full_range=True)
    ka, kb, idx = seeded_keys(b200dpf.gen, n, batch, prf, seed=40 + prf)
    assert np.array_equal(idx, reference_gpu["same_idx"][prf])
    want_a, want_b = reference_gpu["same_a"][prf], reference_gpu["same_b"][prf]
    ctx = b200dpf.Context(table)
    got_a, got_b = ctx.eval(ka, prf), ctx.eval(kb, prf)
    ctx.close()
    assert np.array_equal(got_a, want_a)
    assert np.array_equal(got_b, want_b)
    assert np.array_equal((want_a.astype(np.uint32) - want_b.astype(np.uint32)).astype(np.int32), table[idx])


def test_entry_size_and_short_batch_like_reference(reference_gpu):
    n, batch, entry, prf = 1024, 5, 7, 3
    table = random_table(n, entry, seed=9)
    ka, _, idx = seeded_keys(b200dpf.gen, n, batch, prf, seed=9)
    assert np.array_equal(idx, reference_gpu["short_idx"])
    ctx = b200dpf.Context(table)
    assert np.array_equal(ctx.eval(ka, prf), reference_gpu["short_a"])
    ctx.close()
