"""Quad layout of the fused inner product: with 4 or more keys per warp, the 4 lanes of a quad
share a subtree and split the table row into 4 column slices, exchanging their leaves by
shuffle.  These cases cover what that layout has to get right and the other parity tests do
not single out: key groups that end inside a quad, lane-split warps of 4, 8 and 16 keys, the
8- and 16-uint4 row passes, and grouped bins with odd key counts.  Bit-exact against the oracle
for every PRF."""
import numpy as np
import pytest

import b200dpf
from common import random_table, seeded_keys

pytestmark = pytest.mark.gpu

ALL_PRFS = [0, 1, 2, 3]


@pytest.fixture(scope="module")
def torch_cuda():
    import torch
    if not torch.cuda.is_available():
        pytest.fail("GPU test selected but no CUDA device is visible")
    return torch


@pytest.mark.parametrize("prf", ALL_PRFS)
def test_key_groups_ending_inside_a_quad(oracle, torch_cuda, prf):
    """One key per lane; the last key group's valid keys stop in the middle of a quad."""
    n = 2048
    table = random_table(n, 16, seed=410 + prf)
    ka, kb, idx = seeded_keys(b200dpf.gen, n, 97, prf, seed=411 + prf)
    want = oracle.eval_dot(ka, prf, table)
    ctx = b200dpf.Context(table)
    for batch in (33, 35, 62, 97):
        assert np.array_equal(ctx.eval(ka[:batch], prf), want[:batch]), batch
    got_b = ctx.eval(kb, prf)
    assert np.array_equal((want.astype(np.uint32) - got_b.astype(np.uint32)).astype(np.int32), table[idx])
    ctx.close()


@pytest.mark.parametrize("prf", ALL_PRFS)
def test_lane_split_quads(oracle, torch_cuda, prf):
    """4, 8 and 16 keys per warp (the spare lanes take adjacent subtrees), full and partial quads,
    with and without the frontier."""
    n = 4096
    table = random_table(n, 16, seed=420 + prf)
    ka, _, _ = seeded_keys(b200dpf.gen, n, 16, prf, seed=421 + prf)
    want = oracle.eval_dot(ka, prf, table)
    ctx = b200dpf.Context(table)
    for frontier in (1, 0):
        ctx.set_option("frontier", frontier)
        for batch in (3, 4, 5, 6, 8, 11, 13, 16):
            assert np.array_equal(ctx.eval(ka[:batch], prf), want[:batch]), (frontier, batch)
    ctx.close()


@pytest.mark.parametrize("prf", ALL_PRFS)
@pytest.mark.parametrize("entry", [16, 17, 32, 33, 64])
def test_row_passes_under_quads(oracle, torch_cuda, prf, entry):
    """4-, 8- and 16-uint4 passes over the row, ragged last columns, one key per lane and
    lane-split warps."""
    n = 1024
    table = random_table(n, entry, seed=430 + entry)
    ka, _, _ = seeded_keys(b200dpf.gen, n, 37, prf, seed=431 + entry)
    want = oracle.eval_dot(ka, prf, table)
    ctx = b200dpf.Context(table)
    for batch in (37, 6):
        got = ctx.eval(ka[:batch], prf)
        assert got.shape == (batch, entry)
        assert np.array_equal(got, want[:batch]), batch
    ctx.close()


@pytest.mark.parametrize("prf", ALL_PRFS)
def test_grouped_bins_odd_key_counts(oracle, torch_cuda, prf):
    """Grouped evaluation: every bin's key group ends at an odd key count."""
    rng = np.random.RandomState(440 + prf)
    sizes = [1 << 10, 1 << 12, 64, 1 << 11]
    counts = [1, 3, 5, 33]
    tables = [random_table(n, 16, seed=441 + g) for g, n in enumerate(sizes)]
    ctx = b200dpf.GroupContext(tables)
    keys, bins = [], []
    for g, (n, cnt) in enumerate(zip(sizes, counts)):
        for _ in range(cnt):
            a, _ = b200dpf.gen(int(rng.randint(0, n)), n, 9500 + len(keys), prf)
            keys.append(a)
            bins.append(g)
    order = rng.permutation(len(keys))
    keys, bins = np.stack(keys)[order], np.array(bins, np.int32)[order]
    got = ctx.eval(keys, bins, prf)
    for g in range(len(sizes)):
        sel = np.nonzero(bins == g)[0]
        assert np.array_equal(got[sel], oracle.eval_dot(keys[sel], prf, tables[g])), g
    ctx.close()
