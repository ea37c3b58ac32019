"""Store the original project's answers that the reference-comparison tests check against.

    make -C oracle ref    && python tests/golden/make_reference_checks.py cpu
    make -C oracle refgpu && python tests/golden/make_reference_checks.py gpu   (needs a GPU)

`cpu` asks the unmodified reference CPU core (oracle/_ref/libdpfref.so) and writes
tests/golden/reference_cpu_v1.npz for tests/test_oracle.py; `gpu` asks the reference's own
GPU extension (oracle/_ref/ref_dpf_cpp.so) and writes tests/golden/reference_gpu_v1.npz for
tests/test_gpu_vs_reference_gpu.py.  Both builds need the original project's sources
(REF_ROOT); the stored files do not, so the tests run from a plain checkout.  An optional
second argument names another output path.
"""
import os
import random
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
for sub in ("gpu-dpf_b200", "oracle", "tests"):
    sys.path.insert(0, os.path.join(ROOT, sub))
import oracle as O  # noqa: E402
from common import formula_table, random_table, seeded_keys  # noqa: E402

M64 = (1 << 64) - 1


def cpu(path):
    ref = O.Ref()
    orc = O.Oracle()
    out = {}

    # PRF outputs for 200 random 128-bit seeds, both children, every PRF
    r = random.Random(7)
    seeds = [r.getrandbits(128) for _ in range(200)]
    out["prf_seed"] = np.array([(s & M64, s >> 64) for s in seeds], np.uint64)
    prf_out = np.zeros((4, len(seeds), 2, 2), np.uint64)          # [prf][seed][pos][lo, hi]
    for si, s in enumerate(seeds):
        for prf in range(4):
            for pos in (0, 1):
                v = ref.prf(prf, s, pos)
                prf_out[prf, si, pos] = (v & M64, v >> 64)
    out["prf_out"] = prf_out

    # keygen, full evaluation and single-index evaluation
    r = random.Random(11)
    meta, keys_a, keys_b, full_a, flat_b = [], [], [], [], []
    for prf in range(4):
        for n in (2, 4, 256, 2048):
            for _ in range(3):
                alpha, seed32 = r.randrange(n), r.getrandbits(32)
                ka, kb = ref.gen(alpha, n, seed32, prf)
                meta.append((prf, n, alpha, seed32))
                keys_a.append(ka)
                keys_b.append(kb)
                full_a.append(ref.eval_full(ka, prf))
                flat_b.append([(v & M64, v >> 64) for v in (ref.eval_flat(kb, idx, prf) for idx in (0, alpha, n - 1))])
    out["gen_meta"] = np.array(meta, np.int64)                       # columns: prf, n, alpha, seed32
    out["gen_keys_a"] = np.stack(keys_a)
    out["gen_keys_b"] = np.stack(keys_b)
    out["eval_full_a"] = np.concatenate(full_a)                      # case after case, n values each
    out["eval_flat_b"] = np.array(flat_b, np.uint64)                 # [case][idx 0, alpha, n-1][lo, hi]

    # the multithreaded inner product behind bench.py's `--impl reference` leg
    n = 512
    keys = np.stack([orc.gen(i * 37 % n, n, 50 + i, 2)[0] for i in range(5)])
    out["harness_dot"] = ref.eval_dot_mt(keys, 2, formula_table(n, 16), 0, n, 3)

    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


def gpu(path):
    import torch
    import b200dpf
    import refgpu
    assert torch.cuda.is_available() and refgpu.available()
    out = {}

    def run(prf, table, keys):
        ref = refgpu.RefGpuDPF(prf)
        ref.eval_init(torch.from_numpy(table))
        got = ref.eval_gpu([torch.from_numpy(k) for k in keys]).numpy()
        ref.close()
        return got

    # inputs of test_same_results_as_reference_kernel
    same_a, same_b, same_idx = [], [], []
    for prf in range(4):
        n, batch = 4096, 70
        table = random_table(n, 16, seed=prf, full_range=True)
        ka, kb, idx = seeded_keys(b200dpf.gen, n, batch, prf, seed=40 + prf)
        same_a.append(run(prf, table, ka))
        same_b.append(run(prf, table, kb))
        same_idx.append(idx)
    out["same_a"], out["same_b"], out["same_idx"] = np.stack(same_a), np.stack(same_b), np.stack(same_idx)

    # inputs of test_entry_size_and_short_batch_like_reference
    n, batch, entry, prf = 1024, 5, 7, 3
    ka, _, idx = seeded_keys(b200dpf.gen, n, batch, prf, seed=9)
    out["short_a"] = run(prf, random_table(n, entry, seed=9), ka)
    out["short_idx"] = idx

    np.savez_compressed(path, **out)
    print("wrote", path, os.path.getsize(path), "bytes")


if __name__ == "__main__":
    which = sys.argv[1]
    default = os.path.join(ROOT, "tests", "golden", "reference_%s_v1.npz" % which)
    {"cpu": cpu, "gpu": gpu}[which](sys.argv[2] if len(sys.argv) > 2 else default)
