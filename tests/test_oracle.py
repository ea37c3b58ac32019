"""The CPU oracle against the golden vectors produced by the real reference.  No GPU."""
import os
import random

import numpy as np
import pytest

from common import dot_u32, formula_table

# values printed by the unmodified reference for seed 0x0123456789abcdef_fedcba9876543210 (SURVEY.md section 8c)
SURVEY_SEED = 0x0123456789ABCDEFFEDCBA9876543210
SURVEY_KAT = {
    (0, 0): 0xDA740DA740DA72CD258BF258BF259DB2, (0, 1): 0xDB97530ECA8640BD2468ACF13579CFC3,
    (1, 0): 0x5FBDA2E3F234E6B2B441D17E91810713, (1, 1): 0x96BFF27E59D21AF7115FC04F9F69A796,
    (2, 0): 0x63B38CD27C19ADE41BA01054F62962A9, (2, 1): 0x4EF8FD229FC67648B29DE9F00E19B12A,
    (3, 0): 0x13F02B85CF6357E3A3716CB94327E294, (3, 1): 0x18B5654ACFC155AA5008DAAB2FCED214,
}


def test_aes_fips197_c1(oracle):
    key = bytes(range(16))
    pt = bytes.fromhex("00112233445566778899aabbccddeeff")
    assert oracle.aes128_encrypt(key, pt).hex() == "69c4e0d86a7b0430d8cdb78070b4c55a"


def test_prf_survey_values(oracle):
    for (prf, pos), want in SURVEY_KAT.items():
        assert oracle.prf(prf, SURVEY_SEED, pos) == want


def test_prf_golden(oracle, golden):
    seeds, outs = golden["kat_seed"], golden["kat_out"]
    for si in range(seeds.shape[0]):
        s = int(seeds[si, 0]) | (int(seeds[si, 1]) << 64)
        for prf in range(4):
            for pos in (0, 1):
                want = int(outs[prf, si, pos, 0]) | (int(outs[prf, si, pos, 1]) << 64)
                assert oracle.prf(prf, s, pos) == want


def test_gen_golden(oracle, golden):
    meta = golden["case_meta"]
    for ci, (prf, n, alpha, seed32) in enumerate(meta):
        ka, kb = oracle.gen(int(alpha), int(n), int(seed32), int(prf))
        assert np.array_equal(ka, golden["keys_a"][ci])
        assert np.array_equal(kb, golden["keys_b"][ci])


def test_eval_golden(oracle, golden):
    meta = golden["case_meta"]
    for ci, (prf, n, alpha, seed32) in enumerate(meta):
        prf, n = int(prf), int(n)
        ka, kb = golden["keys_a"][ci], golden["keys_b"][ci]
        sa = oracle.eval_full(ka, prf, tree=True)
        sb = oracle.eval_full(kb, prf, tree=True)
        if n <= 1024:
            assert np.array_equal(sa, golden["share_a_%d" % ci])
            assert np.array_equal(sb, golden["share_b_%d" % ci])
            assert np.array_equal(oracle.eval_full(ka, prf, tree=False), sa)
        t = formula_table(n, 16)
        assert np.array_equal(oracle.eval_dot(ka, prf, t)[0], golden["dots_a"][ci])
        assert np.array_equal(oracle.eval_dot(kb, prf, t)[0], golden["dots_b"][ci])
        assert np.array_equal(dot_u32(sa[None, :], t)[0], golden["dots_a"][ci])


def test_shard_partials_add_up(oracle, golden):
    """Entry-range shards (SURVEY.md section 8e): partial sums over disjoint
    breadth-first leaf ranges add to the whole inner product mod 2^32."""
    meta = golden["case_meta"]
    for ci, (prf, n, alpha, seed32) in enumerate(meta):
        n = int(n)
        if n != 1024:
            continue
        t = formula_table(n, 16)
        for shards in (2, 8):
            acc = np.zeros(16, np.uint32)
            for r in range(shards):
                acc += oracle.eval_dot_shard(golden["keys_a"][ci], int(prf), t, r * n // shards, n // shards).astype(np.uint32)
            assert np.array_equal(acc.astype(np.int32), golden["dots_a"][ci])


def test_dot_range_matches_full(oracle, golden):
    ci = [i for i, m in enumerate(golden["case_meta"]) if m[1] == 1024][0]
    prf = int(golden["case_meta"][ci][0])
    t = formula_table(1024, 16)
    a = oracle.eval_dot_range(golden["keys_a"][ci], prf, t, 0, 512).astype(np.uint32)
    b = oracle.eval_dot_range(golden["keys_a"][ci], prf, t, 512, 512).astype(np.uint32)
    assert np.array_equal((a + b).astype(np.int32)[0], golden["dots_a"][ci])


# ---- against the real reference's answers (tests/golden/make_reference_checks.py cpu) ----

@pytest.fixture(scope="module")
def reference_cpu():
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_cpu_v1.npz"))


def _u128(lo_hi):
    return int(lo_hi[0]) | (int(lo_hi[1]) << 64)


def test_oracle_matches_reference_prf(oracle, reference_cpu):
    r = random.Random(7)
    seeds, outs = reference_cpu["prf_seed"], reference_cpu["prf_out"]
    assert seeds.shape[0] == 200
    for si in range(seeds.shape[0]):
        s = r.getrandbits(128)
        assert s == _u128(seeds[si])
        for prf in range(4):
            for pos in (0, 1):
                assert oracle.prf(prf, s, pos) == _u128(outs[prf, si, pos])


def test_oracle_matches_reference_gen_and_eval(oracle, reference_cpu):
    r = random.Random(11)
    meta = reference_cpu["gen_meta"]
    full = reference_cpu["eval_full_a"]
    ci, off = 0, 0
    for prf in range(4):
        for n in (2, 4, 256, 2048):
            for _ in range(3):
                alpha, seed32 = r.randrange(n), r.getrandbits(32)
                assert tuple(int(v) for v in meta[ci]) == (prf, n, alpha, seed32)
                ka, kb = oracle.gen(alpha, n, seed32, prf)
                ra, rb = reference_cpu["gen_keys_a"][ci], reference_cpu["gen_keys_b"][ci]
                assert np.array_equal(ka, ra) and np.array_equal(kb, rb)
                assert np.array_equal(oracle.eval_full(ka, prf), full[off:off + n])
                for j, idx in enumerate((0, alpha, n - 1)):
                    assert oracle.eval_flat(kb, idx, prf) == _u128(reference_cpu["eval_flat_b"][ci, j])
                ci, off = ci + 1, off + n
    assert ci == meta.shape[0] and off == full.shape[0]


def test_reference_baseline_harness(oracle, reference_cpu):
    """ref_eval_dot_mt (the --impl reference timing leg) computes the same inner product."""
    n = 512
    t = formula_table(n, 16)
    keys = np.stack([oracle.gen(i * 37 % n, n, 50 + i, 2)[0] for i in range(5)])
    assert np.array_equal(reference_cpu["harness_dot"], oracle.eval_dot(keys, 2, t))
