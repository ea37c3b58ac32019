#!/usr/bin/env python
"""bench.py -- DPFs/sec of the hot path on N B200s (one process per GPU).

    python bench.py [--gpus N] [--steps K] [--warmup W]          our engine
    python bench.py --impl reference [...]                       reference CPU path

A step is one pass of the hot path over one batch: full-domain evaluation of
`batch` DPF keys fused with the inner product against an [n, 16] int32 table
(BASELINE.json metric: n = 2^20, entry_size = 16, AES128, batch 512 per GPU).

N > 1 (launched by torchrun, NCCL): the table is sharded by entry range, every
rank evaluates the whole batch over its subtree, and one NCCL reduce adds the
[B, 16] partials (SURVEY.md section 8e).  The batch grows with N (512 per GPU),
so per-GPU work is fixed: weak scaling.

Rank 0 prints ONE JSON line.  `value` is device-timed with keys resident in
HBM; `e2e` goes through the public dpf-API call with pinned HOST keys, H2D and
D2H inside the timed region.

--dump-outputs DIR saves the answers the last timed step computed (DIR/answers.npy).  Table and
keys come from fixed seeds, so two builds run with the same arguments can be compared answer for
answer.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
import gpu_dpf_b200  # noqa: E402,F401  (importable alias of gpu-dpf_b200/; makes dpf, b200dpf, dpf_cpp, sharded importable)

PRF_IDS = {"dummy": 0, "salsa20": 1, "chacha20": 2, "aes128": 3}
KEY_BYTES = 2096
BASELINE_PUBLISHED = {  # BASELINE.md section 1 (reference README.md:129-146), V100, batch 512, entry 16
    ("aes128", 1 << 14): 52536, ("aes128", 1 << 16): 15392, ("aes128", 1 << 18): 3967, ("aes128", 1 << 20): 923,
    ("salsa20", 1 << 14): 145646, ("salsa20", 1 << 16): 54892, ("salsa20", 1 << 18): 16650, ("salsa20", 1 << 20): 3894,
    ("chacha20", 1 << 14): 139590, ("chacha20", 1 << 16): 56120, ("chacha20", 1 << 18): 16086, ("chacha20", 1 << 20): 4054,
}
DUMP_MAX_BYTES = 60 << 20     # --dump-outputs: stays under 64 MB with the .npy headers


_REAL_STDOUT = None


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is not None:
        os.write(_REAL_STDOUT, data)
    else:
        sys.stdout.write(data.decode())
        sys.stdout.flush()


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference", "reference-gpu"],
                    help="reference = the reference's CPU path on the host cores; reference-gpu = the reference's "
                         "own GPU kernel compiled unmodified for sm_100a (oracle/_ref/ref_dpf_cpp.so), 1 GPU")
    ap.add_argument("--entries", "--n", dest="n", type=int, default=1 << 20, help="table size n (use --entries under torchrun: --n is ambiguous to its parser)")
    ap.add_argument("--entry", type=int, default=16)
    ap.add_argument("--prf", default="aes128", choices=sorted(PRF_IDS))
    ap.add_argument("--batch-per-gpu", type=int, default=512)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--subtree-log2", type=int, default=0)
    ap.add_argument("--strong", action="store_true",
                    help="N>1: keep the GLOBAL batch at --batch-per-gpu keys (strong scaling: each GPU still sees "
                         "every key but only 1/N of the leaves) instead of growing it with N")
    ap.add_argument("--axis", default="auto", choices=["auto", "entries", "keys"],
                    help="N>1: entry-range shards + reduce, key-split replicas + gather, or auto (by n; --strong only: "
                         "the default weak run is always entry-sharded, as BASELINE.json's metric names)")
    ap.add_argument("--no-sweep", action="store_true", help="skip the bounded n x PRF sweep / strong-scaling / config extras")
    ap.add_argument("--no-parity", action="store_true", help="skip the post-timing parity check of the timed batch")
    ap.add_argument("--reduce", default="nccl", choices=["nccl", "fused"],
                    help="N>1: NCCL reduce of the partials, or the kernel's peer-memory red.add epilogue")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the [batch, entry] result of the last timed step to DIR/answers.npy (float64, exact "
                         "for int32; a seeded sample of rows above %d MiB) so two builds can be compared" % (DUMP_MAX_BYTES >> 20))
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs applies to --impl ours")
    return args


def bytes_per_dpf(n, entry):
    """SURVEY.md section 8(d): int32 table streamed once per key + key + output."""
    return n * entry * 4 + KEY_BYTES + 4 * entry


def synthetic_table(n, entry):
    rng = np.random.RandomState(1234)
    return rng.randint(0, 2**31, size=(n, entry), dtype=np.int64).astype(np.int32)


def synthetic_keys(n, batch, prf):
    import b200dpf
    rng = np.random.RandomState(4321)
    alphas = rng.randint(0, n, size=batch).astype(np.int64)
    ka, kb = b200dpf.gen_batch(alphas, n, np.arange(batch) + 1000, prf)
    return ka, kb, alphas


def host_cores():
    """Host threads this process can really use: the scheduler affinity mask, capped by the
    cgroup CPU quota when one is set (os.cpu_count() reports the machine, not the lease)."""
    try:
        cores = len(os.sched_getaffinity(0))
    except Exception:
        cores = os.cpu_count() or 1
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            f = open(path).read().split()
            if path.endswith("cpu.max"):
                if f[0] != "max":
                    cores = min(cores, max(1, int(int(f[0]) / int(f[1]))))
            else:
                quota = int(f[0])
                period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                if quota > 0:
                    cores = min(cores, max(1, quota // period))
            break
        except Exception:
            continue
    return max(1, cores)


def cpu_model():
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                return line.split(":", 1)[1].strip()
    except Exception:
        pass
    return "unknown"


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


# ---------------------------------------------------------------------------
# clocks (B200_PROFILING.md recipe)
# ---------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
              "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
              "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu_index = gpu_index
        self.proc = None
        self.path = None

    def start(self):
        try:
            fd, self.path = tempfile.mkstemp(suffix=".csv")
            os.close(fd)
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu_index), "--query-gpu=" + self.FIELDS,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=open(self.path, "w"), stderr=subprocess.DEVNULL)
        except Exception:
            self.proc = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        if self.proc is None:
            return out
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, reasons, smax = [], set(), None
        try:
            for line in open(self.path):
                f = [x.strip() for x in line.split(",")]
                if len(f) < 9:
                    continue
                try:
                    sm.append(float(f[1]))
                    smax = float(f[2])
                except ValueError:
                    continue
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
            os.unlink(self.path)
        except Exception:
            pass
        if sm:
            top = sorted(sm)[len(sm) // 2:]          # upper half = samples taken under load
            out["sm_mhz"] = float(np.median(top))
            out["samples"] = len(sm)
        out["sm_max_mhz"] = smax
        out["reasons"] = sorted(reasons)
        return out


# ---------------------------------------------------------------------------
# reference CPU path (oracle/_ref when the reference compiled, else the oracle port)
# ---------------------------------------------------------------------------
def cpu_reference_runner(n, entry, prf, table):
    """Returns (kind, cores, sample_desc, step_fn) where step_fn() runs one bounded
    sample and returns the number of DPF-equivalents it evaluated."""
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle as O
    cores = host_cores()
    orc = O.Oracle()
    rng = np.random.RandomState(99)
    keys = np.stack([orc.gen(int(rng.randint(0, n)), n, 2000 + i, prf)[0] for i in range(cores)])
    depth = n.bit_length() - 1
    per_index_us = {0: 0.01, 1: 0.08, 2: 0.08, 3: 1.4}[prf] * depth
    idx_count = int(min(n, max(1024, 1.5e6 / per_index_us)))       # about 1.5 s per thread
    idx_count = 1 << (idx_count.bit_length() - 1)
    frac = idx_count / n
    if O.Ref.available():
        ref = O.Ref()
        kind = "reference"

        def step():
            ref.eval_dot_mt(keys, prf, table, 0, idx_count, cores)
            return cores * frac
    else:
        kind = "port"

        def step():
            th = [threading.Thread(target=orc.eval_dot_range, args=(keys[i:i + 1], prf, table, 0, idx_count))
                  for i in range(cores)]
            [t.start() for t in th]
            [t.join() for t in th]
            return cores * frac
    sample = ("%d keys (one per host thread) x %d of %d indices each via per-index EvaluateFlat + int32 dot, "
              "scaled by n/indices" % (cores, idx_count, n))
    return kind, cores, sample, step


def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    prf = PRF_IDS[args.prf]
    n, entry = args.n, args.entry
    table = synthetic_table(n, entry)
    kind, cores, sample, step = cpu_reference_runner(n, entry, prf, table)
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    units = 0.0
    for _ in range(args.steps):
        units += step()
    dt = time.perf_counter() - t0
    value = units / dt
    line = {
        "impl": "reference", "metric": "DPFs/sec", "value": value, "unit": "DPFs/sec", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * dt / max(args.steps, 1),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": {"workload": "n=%d entry_size=%d %s, reference CPU path (dpf_base EvaluateFlat per index) on host cores"
                               % (n, entry, args.prf.upper()), "n": n, "entry_size": entry, "prf": args.prf.upper()},
        "cpu_baseline": {"value": value, "unit": "DPFs/sec", "cores": cores, "kind": kind, "sample": sample,
                         "cpu_model": cpu_model()},
        "e2e": {"value": value, "unit": "DPFs/sec", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    emit(line)


def run_reference_gpu(args):
    """The reference's dpf_hybrid_kernel on this box, measured the way its benchmark.py does
    (dpf.py:286-320): wall clock around `steps` eval_gpu calls of 512 host key tensors."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import torch
    import refgpu
    if not refgpu.available():
        emit({"impl": "reference-gpu", "unavailable": "oracle/_ref/ref_dpf_cpp.so not built (needs the reference tree)"})
        return
    prf = PRF_IDS[args.prf]
    n, entry, batch = args.n, args.entry, args.batch_per_gpu
    table = synthetic_table(n, entry)
    keys_np, _, _ = synthetic_keys(n, batch, prf)
    keys = [torch.from_numpy(k) for k in keys_np]
    ref = refgpu.RefGpuDPF(prf)
    t0 = time.perf_counter()
    ref.eval_init(torch.from_numpy(table))
    t_init = time.perf_counter() - t0
    for _ in range(max(args.warmup, 1)):
        ref.eval_gpu(keys)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        out = ref.eval_gpu(keys)
    torch.cuda.synchronize()
    dt = time.perf_counter() - t0
    value = batch * args.steps / dt
    emit({"impl": "reference-gpu", "metric": "DPFs/sec", "value": value, "unit": "DPFs/sec", "n_gpus": 1,
          "steps": args.steps, "warmup": max(args.warmup, 1), "ms_per_step": 1e3 * dt / args.steps,
          "higher_is_better": True, "dtype": "u128", "data": "synthetic",
          "config": {"workload": "n=%d entry_size=%d %s batch=%d, reference dpf_hybrid_kernel compiled for sm_100a, "
                                 "wall clock incl. host marshalling (benchmark.py method)" % (n, entry, args.prf.upper(), batch),
                     "eval_init_s": t_init},
          "e2e": {"value": value, "unit": "DPFs/sec", "h2d_bytes_per_step": batch * 2080, "d2h_bytes_per_step": batch * 256},
          "checksum": int(out.to(torch.int64).sum().item())})
    ref.close()


# ---------------------------------------------------------------------------
# our engine
# ---------------------------------------------------------------------------
def pipe_roofline(prf_name, dpfs_per_s, n_local, sm_mhz):
    """Integer-pipe roofline from MEASURED peaks (profiles/int_peaks.json, written by
    tools/microbench/int_pipes.cu on a B200) and MEASURED per-node-pair instruction counts
    (profiles/pipe_ops.json, from ncu sm__inst_executed_pipe_* / l1tex wavefront counters of the
    evaluation kernel).  One node pair = one parent expanded into two children for a warp of 32
    keys; a DPF over n_local leaves has n_local - 1 of them."""
    try:
        peaks = json.load(open(os.path.join(ROOT, "profiles", "int_peaks.json")))
        ops = json.load(open(os.path.join(ROOT, "profiles", "pipe_ops.json")))[prf_name]
    except Exception:
        return None
    pipe = ops["binding_pipe"]                      # "alu" | "lsu"
    per_pair = float(ops["warp_inst_per_node_pair"][pipe])
    peak_per_clk_sm = float(peaks["peak_warp_inst_per_clk_sm"][pipe])
    sms = int(peaks.get("sms", 148))
    mhz = float(sm_mhz or peaks.get("sm_max_mhz", 1965.0))
    pairs_per_s = dpfs_per_s / 32.0 * max(n_local - 1, 1)
    achieved = pairs_per_s * per_pair                # warp-instructions (or wavefronts) per second
    peak = peak_per_clk_sm * sms * mhz * 1e6
    return {"pipe": ops.get("pipe_name", pipe), "warp_inst_per_node_pair": per_pair,
            "achieved_ginst_s": achieved / 1e9, "peak_ginst_s": peak / 1e9, "frac": achieved / peak,
            "peak_source": "profiles/int_peaks.json (tools/microbench/int_pipes.cu, %s/clk/SM) x %d SMs x %.0f MHz"
                           % (peak_per_clk_sm, sms, mhz),
            "ops_source": ops.get("source", "profiles/pipe_ops.json")}


try:   # DRAM bytes per launch of the evaluation kernel, measured with ncu per configuration (tools/gpu_r2_final.sh)
    TRAFFIC = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))
except Exception:
    TRAFFIC = {}


class Harness:
    """torch / process-group state shared by every measurement of one bench.py run."""

    def __init__(self, args):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.world = int(os.environ.get("WORLD_SIZE", "1"))
        self.rank = int(os.environ.get("RANK", "0"))
        self.local_rank = int(os.environ.get("LOCAL_RANK", "0"))
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device; the engine has no CPU path (use --impl reference for the CPU baseline)")
        torch.cuda.set_device(self.local_rank)
        self.dev = torch.device("cuda", self.local_rank)
        if self.world > 1:
            import datetime
            dist.init_process_group("nccl", device_id=self.dev, timeout=datetime.timedelta(seconds=600))
        assert self.world == args.gpus or self.world == 1, "launch with torchrun --nproc-per-node %d" % args.gpus
        self.flush = torch.empty(256 << 20, dtype=torch.uint8, device=self.dev)   # > 126 MB L2
        self.args = args

    def barrier(self, world=None):
        if (self.world if world is None else world) > 1:
            self.dist.barrier()

    def max_over_ranks(self, x, world=None):
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        if (self.world if world is None else world) > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def close(self):
        if self.world > 1:
            self.dist.destroy_process_group()


def parity_check(h, d, world, prf, table, keys_a, keys_b, alphas, n_oracle=4):
    """Outside every timed region: the engine's results for the batch that was just timed,
    checked (rank 0) by share reconstruction  a - b == table[alpha]  for EVERY key of the batch and
    bit-exactly against the CPU oracle for the first n_oracle keys."""
    torch = h.torch
    ka = torch.from_numpy(keys_a).to(h.dev)
    kb = torch.from_numpy(keys_b).to(h.dev)
    ra = d.eval_gpu_device(ka)
    a = ra.cpu().numpy().copy() if (world == 1 or h.rank == 0) else None
    rb = d.eval_gpu_device(kb)
    b = rb.cpu().numpy().copy() if (world == 1 or h.rank == 0) else None
    if a is None:
        return None
    rec = (a.astype(np.uint32) - b.astype(np.uint32)).astype(np.int32)
    bad = int((rec != table[alphas]).any(axis=1).sum())
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import oracle as O
    orc = O.Oracle()
    want = [None] * n_oracle

    def one(i):
        want[i] = orc.eval_dot(keys_a[i:i + 1], prf, table)[0]
    th = [threading.Thread(target=one, args=(i,)) for i in range(n_oracle)]
    [t.start() for t in th]
    [t.join() for t in th]
    bad_oracle = sum(0 if np.array_equal(a[i], want[i]) else 1 for i in range(n_oracle))
    return {"keys_reconstructed": int(len(alphas)), "reconstruct_mismatches": bad, "keys_vs_oracle": n_oracle,
            "oracle_mismatches": bad_oracle, "ok": bad == 0 and bad_oracle == 0,
            "checksum": int(a.astype(np.int64).sum() & 0xFFFFFFFF)}


def measure(h, prf_name, n, entry, batch, steps, warmup, world=None, axis="entries", reduce="nccl",
            e2e=True, parity=4, settle_s=0.0, subtree_log2=0, sampler=None, keep_output=False):
    """One configuration: eval_init, warm-up, `steps` device-timed steps (CUDA events on the launching
    stream, max over ranks, L2 flushed before every step), optionally the end-to-end leg through the
    public host-buffer API, and the parity check of the timed batch.  world=1 on a multi-rank run
    means: this rank alone, no collectives (other ranks must not call).  keep_output: res["output"] is
    a host copy of what the last timed step returned (the complete result on rank 0 only)."""
    import dpf as dpf_mod
    from sharded import ShardedDPF
    torch = h.torch
    world = h.world if world is None else world
    prf = PRF_IDS[prf_name]
    table = synthetic_table(n, entry)
    keys_a, keys_b, alphas = synthetic_keys(n, batch, prf)
    if world > 1:
        d = ShardedDPF(prf=prf, device=h.local_rank, reduce=reduce, axis=axis)
        d.eval_init(torch.from_numpy(table))
        inner = d._dpf
        axis_used = d.axis
    else:
        d = dpf_mod.DPF(prf=prf, device=h.local_rank)
        d.eval_init(torch.from_numpy(table))
        inner = d
        axis_used = "single"
    import dpf_cpp
    if subtree_log2:
        dpf_cpp.set_subtree_log2(inner.buffers, subtree_log2)
    keys_dev = torch.from_numpy(keys_a).to(h.dev)
    out_dev = torch.empty((batch, entry), dtype=torch.int32, device=h.dev)

    def step_device():
        return d.eval_gpu_device(keys_dev, out_dev)

    nwarm = max(warmup, 3)
    t_warm = time.perf_counter()
    for _ in range(nwarm):
        h.flush.zero_()
        step_device()
    torch.cuda.synchronize()
    extra_n = 0
    if settle_s > 0:
        # keep the GPU busy for ~settle_s in total so the clock sampler sees it under load; the number
        # of extra iterations is decided on rank 0 and broadcast (collectives must match across ranks)
        per_step = (time.perf_counter() - t_warm) / nwarm
        extra = torch.tensor([int(min(2000, max(0, settle_s / max(per_step, 1e-6) - nwarm)))], dtype=torch.int64, device=h.dev)
        if world > 1:
            h.dist.broadcast(extra, src=0)
        extra_n = int(extra.item())
        for i in range(extra_n):
            h.flush.zero_()
            step_device()
            if i % 16 == 15:
                torch.cuda.synchronize()
        torch.cuda.synchronize()
    launches_per_step = dpf_cpp.last_launches(inner.buffers)
    starts = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    ends = [torch.cuda.Event(enable_timing=True) for _ in range(steps)]
    h.barrier(world)
    torch.cuda.synchronize()
    t_wall0 = time.perf_counter()
    for k in range(steps):
        h.flush.zero_()                       # cold L2 at the start of every timed step
        starts[k].record()
        last = step_device()
        ends[k].record()
    torch.cuda.synchronize()
    h.barrier(world)
    t_wall = time.perf_counter() - t_wall0
    # copied before anything else runs: the key-split path hands out a buffer that the next call reuses
    output = last.cpu().numpy().copy() if (keep_output and last is not None) else None
    clocks = sampler.stop() if sampler else None
    dev_ms = h.max_over_ranks(sum(s.elapsed_time(e) for s, e in zip(starts, ends)), world)
    # per-step times (max over ranks, step by step): the median is what the sub-millisecond extras report
    # next to the mean -- one NCCL or driver hiccup in ten 0.3 ms steps moves the mean by a third
    per_step = torch.tensor([s.elapsed_time(e) for s, e in zip(starts, ends)], dtype=torch.float64, device=h.dev)
    if world > 1:
        h.dist.all_reduce(per_step, op=h.dist.ReduceOp.MAX)
    ms_median = float(per_step.median().item())
    res = {"value": batch * steps / (dev_ms / 1e3), "ms_per_step": dev_ms / steps, "ms_per_step_median": ms_median,
           "launches_per_step": launches_per_step,
           "warmup_effective": nwarm + extra_n, "wall_s_timed_region": t_wall, "clocks": clocks, "axis": axis_used,
           "batch": batch, "e2e": None, "parity_check": None, "output": output}

    if e2e:   # end to end through the public API: pinned HOST keys in, HOST result out, every step
        keys_host = torch.from_numpy(keys_a).pin_memory()
        for _ in range(2):
            d.eval_gpu(keys_host)
        h.barrier(world)
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(steps):
            r = d.eval_gpu(keys_host)
        torch.cuda.synchronize()
        h.barrier(world)
        dt = h.max_over_ranks(time.perf_counter() - t0, world)
        copies = world if axis_used == "entries" else 1       # entry shards: every rank uploads every key
        res["e2e"] = {"value": batch * steps / dt, "unit": "DPFs/sec",
                      "h2d_bytes_per_step": int(keys_host.numel() * 4) * copies,
                      "d2h_bytes_per_step": int(batch * entry * 4)}
        if h.rank == 0 or world == 1:
            assert r is not None and tuple(r.shape) == (batch, entry)
    if parity:
        res["parity_check"] = parity_check(h, d, world, prf, table, keys_a, keys_b, alphas, n_oracle=parity)
    d.close()
    res["table"] = table
    return res


def dump_outputs(dirname, out):
    """int32 [batch, entry] answers as float64 (every int32 is exact there).  Above DUMP_MAX_BYTES a
    fixed, seeded sample of rows is kept, in row order, and the rows taken go to answer_rows.npy."""
    os.makedirs(dirname, exist_ok=True)
    max_rows = max(1, DUMP_MAX_BYTES // (8 * (out.shape[1] + 1)))
    if out.shape[0] > max_rows:
        rows = np.sort(np.random.RandomState(0).choice(out.shape[0], max_rows, replace=False))
        out = out[rows]
        np.save(os.path.join(dirname, "answer_rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(dirname, "answers.npy"), out.astype(np.float64))


def run_ours(args):
    h = Harness(args)
    world, rank = h.world, h.rank
    prf = PRF_IDS[args.prf]
    n, entry = args.n, args.entry
    batch = args.batch_per_gpu * (1 if args.strong else world)
    sampler = ClockSampler(h.local_rank) if rank == 0 else None
    if sampler:
        sampler.start()          # nvidia-smi needs a moment to produce its first sample
    axis = args.axis if (args.strong or args.axis != "auto") else "entries"
    m = measure(h, args.prf, n, entry, batch, args.steps, args.warmup, axis=axis, reduce=args.reduce,
                e2e=not args.no_e2e, parity=0 if args.no_parity else 4, settle_s=0.5,
                subtree_log2=args.subtree_log2, sampler=sampler, keep_output=bool(args.dump_outputs))
    table = m.pop("table")
    output = m.pop("output")
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, output)
    value, clocks = m["value"], m["clocks"]

    # ---- bounded sweep over the other sizes / PRFs the north star names (N = 1), the BASELINE
    # ---- configs that need 8 GPUs (N = 8), and strong scaling of ONE 512-key batch (N > 1)
    sweep, strong, configs = [], None, []
    if not args.no_sweep:
        def entry_of(tag, prf_name, nn, ee, bb, r, ww=None):
            ww = world if ww is None else ww
            alg = bb * (nn * ee * 4 // (ww if r["axis"] == "entries" else 1) // 1 + KEY_BYTES + 4 * ee)
            out = {"config": tag, "prf": prf_name.upper(), "n": nn, "entry_size": ee, "batch": bb, "n_gpus": ww,
                   "axis": r["axis"], "value": r["value"], "ms_per_step": r["ms_per_step"],
                   "ms_per_step_median": r["ms_per_step_median"],
                   "e2e": r["e2e"]["value"] if r["e2e"] else None, "launches_per_step": r["launches_per_step"],
                   "frac": (alg / (r["ms_per_step"] / 1e3) / 1e9) / (float(load_peaks().get("hbm_gbs", 6650.0)) * ww),
                   "parity_ok": r["parity_check"]["ok"] if r["parity_check"] else None}
            shards_e = ww if r["axis"] == "entries" else 1
            pr = pipe_roofline(prf_name, r["value"] / ww, nn // shards_e, (clocks or {}).get("sm_mhz")) if ee == 16 else None
            out["pipe_frac"] = pr["frac"] if pr else None
            out["traffic"] = TRAFFIC.get("%s_n%d_e%d_b%d_%dgpu" % (prf_name, nn, ee, bb, ww), {}).get("dram_bytes_per_launch")
            return out
        try:
            if world == 1:
                for prf_name in ("aes128", "salsa20", "chacha20"):
                    for nn in (1 << 14, 1 << 16, 1 << 18):
                        r = measure(h, prf_name, nn, 16, 512, 10, 3, parity=2)
                        r.pop("table")
                        sweep.append(entry_of("n=2^%d" % (nn.bit_length() - 1), prf_name, nn, 16, 512, r))
                r = measure(h, "aes128", 1 << 14, 16, 256, 20, 3, parity=2)      # BASELINE.json config 2
                r.pop("table")
                configs.append(entry_of("C2", "aes128", 1 << 14, 16, 256, r))
            else:
                # the n x PRF matrix at this GPU count: 512 keys per GPU, axis by table size (key split for
                # small tables, entry shards + reduce above 2^18), every entry parity-checked on rank 0
                for prf_name in ("aes128", "salsa20", "chacha20"):
                    for nn in (1 << 14, 1 << 16, 1 << 18):
                        r = measure(h, prf_name, nn, 16, 512 * world, 10, 3, axis="auto", parity=2)
                        r.pop("table")
                        sweep.append(entry_of("n=2^%d" % (nn.bit_length() - 1), prf_name, nn, 16, 512 * world, r))
                strong = []
                for nn in (1 << 16, 1 << 20):
                    rs = measure(h, "aes128", nn, 16, 512, 30 if nn <= (1 << 16) else 10, 3, axis="auto", parity=2)
                    rs.pop("table")
                    one = None
                    if rank == 0:          # the same batch on ONE of these GPUs, this rank alone
                        one = measure(h, "aes128", nn, 16, 512, 30 if nn <= (1 << 16) else 10, 3, world=1, e2e=False, parity=0)
                        one.pop("table")
                    h.barrier()
                    if rank == 0:
                        strong.append({"n": nn, "prf": "AES128", "batch": 512, "axis": rs["axis"], "ms_per_step": rs["ms_per_step"],
                                       "ms_per_step_median": rs["ms_per_step_median"],
                                       "value": rs["value"], "ms_per_step_1gpu": one["ms_per_step"],
                                       "ms_per_step_1gpu_median": one["ms_per_step_median"],
                                       "speedup_vs_1gpu": one["ms_per_step"] / rs["ms_per_step"],
                                       "speedup_vs_1gpu_median": one["ms_per_step_median"] / rs["ms_per_step_median"],
                                       "parity_ok": rs["parity_check"]["ok"] if rs["parity_check"] else None})
                if world == 8 and not args.strong:
                    r = measure(h, "salsa20", 1 << 24, 16, 4096, 2, 3, e2e=False, parity=2)      # config 4
                    r.pop("table")
                    configs.append(entry_of("C4", "salsa20", 1 << 24, 16, 4096, r))
                    r = measure(h, "aes128", 1 << 20, 128, 8192, 2, 3, e2e=False, parity=2)      # config 5
                    r.pop("table")
                    configs.append(entry_of("C5", "aes128", 1 << 20, 128, 8192, r))
        except Exception as exc:   # the headline line must survive a failure in the extras
            sweep.append({"error": "%s: %s" % (type(exc).__name__, exc)})

    if rank == 0:
        peaks = load_peaks()
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_kind = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback (B200_PROFILING.md)"
        # dominant kernel = the one evaluation kernel of a step; per launch it processes `batch`
        # keys over n/world leaves each
        shards = world if m["axis"] == "entries" else 1
        alg_bytes = batch * (n // shards * entry * 4 + KEY_BYTES + 4 * entry)
        launch_ms = m["ms_per_step"]
        achieved = alg_bytes / (launch_ms / 1e3) / 1e9
        # measured with ncu (dram__bytes_read.sum + dram__bytes_write.sum), per launch
        traffic = TRAFFIC.get("%s_n%d_e%d_b%d_%dgpu" % (args.prf, n, entry, batch, world), {}).get("dram_bytes_per_launch")
        roofline = {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "traffic": traffic, "peak_source": peak_kind,
                    "pipe": pipe_roofline(args.prf, value / world, n // shards, (clocks or {}).get("sm_mhz")),
                    "note": "algorithmic bytes = batch*(n*E*4/ngpu + 2096 + 4E) per launch (table streamed once "
                            "per key, SURVEY 8d); actual DRAM traffic is far lower because 32 keys share each row "
                            "load and the table stays in L2, so the HBM fraction is nominal.  `pipe` is the roofline "
                            "that binds: measured instruction count per node pair / measured pipe issue rate."}
        cpu = None
        if world == 1 and not args.no_cpu_baseline:
            kind, cores, sample, step = cpu_reference_runner(n, entry, prf, table)
            step()
            t0 = time.perf_counter()
            units = step()
            cpu = {"value": units / (time.perf_counter() - t0), "unit": "DPFs/sec", "cores": cores, "kind": kind,
                   "sample": sample, "cpu_model": cpu_model()}
        published = BASELINE_PUBLISHED.get((args.prf, n)) if (entry == 16) else None
        par = m["parity_check"]
        line = {
            "metric": "DPFs/sec", "value": value, "unit": "DPFs/sec", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "warmup_effective": m["warmup_effective"],
            "ms_per_step": m["ms_per_step"], "higher_is_better": True,
            "scaling": "strong" if args.strong else "weak",
            "vs_baseline": (value / published) if published else None, "dtype": "u32",
            "data": "synthetic",
            "config": {"workload": "n=%d entry_size=%d %s batch=%d (%s), %s over %d GPU(s)"
                                   % (n, entry, args.prf.upper(), batch,
                                      "fixed global batch" if args.strong else "%d per GPU" % args.batch_per_gpu,
                                      "batch split by keys, table replicated" if m["axis"] == "keys" else "table entry-range sharded",
                                      world),
                       "n": n, "entry_size": entry, "prf": args.prf.upper(), "global_batch": batch,
                       "parallelism": ("%s x%d + %s" % ("entry-shard" if m["axis"] == "entries" else "key-split", world,
                                       ("NCCL reduce" if args.reduce == "nccl" else "in-kernel peer-memory red.add (symmetric memory)")
                                       if m["axis"] == "entries" else "NCCL all-gather")) if world > 1 else "single GPU",
                       "l2": "256 MiB device buffer zeroed before every timed step (L2 flush); table %d MiB" % (n * entry * 4 >> 20),
                       "vs_baseline_ref": "reference README V100 number (BASELINE.md)" if published else None},
            "e2e": m["e2e"], "gpu_launches": m["launches_per_step"] * args.steps, "roofline": roofline,
            "cpu_baseline": cpu, "clocks": clocks, "wall_s_timed_region": m["wall_s_timed_region"],
            "parity_check": par,
        }
        if sweep:
            line["sweep"] = sweep
        if configs:
            line["configs"] = configs
        if strong:
            line["strong"] = strong
        emit(line)
        if par is not None and not par["ok"]:
            h.close()
            raise SystemExit("bench.py: PARITY FAILURE in the timed batch: %r" % (par,))
    h.close()


def main():
    args = parse_args()
    # Libraries (NCCL's version banner, torchrun notices) write to stdout; the contract is ONE
    # JSON line there.  Point fd 1 at stderr for the whole run and print the line on the saved fd.
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        run_reference(args)
    elif args.impl == "reference-gpu":
        run_reference_gpu(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
