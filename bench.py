#!/usr/bin/env python
"""bench.py -- pairings/sec of the batched pairing hot path on N B200s (BASELINE.json metric).

  python bench.py --gpus 1 --steps 5 --warmup 3                  # our arm (CUDA, libpbc_b200.so)
  python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 \
         --master-port P bench.py --gpus N --steps K --warmup W  # N > 1: one rank per GPU
  python bench.py --impl reference --gpus 1 --steps K --warmup W # the reference CPU path

One "step" = one pass of the hot path over one batch: 2^20 Type A (param/a.param) pairings per
GPU (BASELINE.json configs[1]), synthetic seeded inputs in the reference wire format.  The batch
shards embarrassingly: every rank owns its own 2^20 pairs (weak scaling; --scaling strong splits
one 2^20 batch instead), no collective on the data path; timing is CUDA events on the launching
stream, max over ranks.  The default run also measures the other GPU configurations of
BASELINE.json -- type F 2^20, type D159 2^18, element_prod_pairing n = 16 with 2^16 outputs split
across the ranks -- and reports them under "configs", each with its device-resident value, its
end-to-end value through the host-buffer C ABI, its executed-work roofline fraction and its parity
against oracle/_ref on a seeded random sample of THIS rank's outputs (every rank checks its shard).

`value`  : whole-job pairings/s with inputs already resident in HBM.
`e2e`    : same metric through the host-buffer C-ABI call (pbc_b200_pairings_apply) with pinned
           HOST buffers: H2D of both inputs and D2H of the outputs inside the timed region.
`roofline`: integer-multiplier pipe (SURVEY 8d): algorithmic IMAD.WIDE.U32 unit operations of the
           dominant kernel (Miller loop) / its CUDA-event duration, against the IMAD.WIDE.U32
           issue rate measured live by a microkernel; plus the (non-binding) HBM view.
`cpu_baseline`: the unmodified reference (oracle/_ref) on the host cores, bounded sample, whose
           outputs are also compared byte-for-byte with the GPU's.

--dump-outputs DIR writes each config's outputs of its last timed step to DIR/<config>.npy (see
dump_outputs); the inputs depend only on the arguments, so two builds of the library can be
compared output for output.
"""
from __future__ import annotations
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

from pbc_b200.params import PARAMS  # noqa: E402
from pbc_b200 import synth  # noqa: E402

GRID = 4096                    # inputs are drawn from a GRID x GRID grid of distinct points
SEED = 20260922
# --- workloads: BASELINE.json configs[1] (default), [2], [3], [4] ---------------------------------
# unit = one 32x32->64 multiply-accumulate (IMAD.WIDE.U32); a t-limb(64-bit) Montgomery mulmod is
# 2(2t)^2 + 2t of them: 528 for t = 8 (type a), 78 for t = 3 (types f, d)  -- SURVEY.md 8(d).
# ref_mulmods = reference-algorithm mulmods per output (SURVEY 8d probes); ref_main = the part the
# first kernel (Miller loop) stands for.  exec_unit_ops_main = what OUR first kernel executes
# (type A, nine-slot weight-(1,2) Miller loop: 11 M + 6 S per step, 159 steps, + 26 M + 8 S around the loop:
# 1775 multiplications of 528 units + 962 squarings of 408).
WORKLOADS = {
    "a": dict(param="a", mode="single", k=1, n=1 << 20, unit=528, ref_mulmods=4394, ref_main=4394 - 719,
              exec_unit_ops_main=1775 * 528 + 962 * 408, cpu_rate=1100.0, port_rate=110.0,
              name="type A (param/a.param) element_pairing, batch 2^20 (P,Q) pairs per GPU, 512-bit F_q",
              dtype="u32 limbs (16 x 32-bit = 512-bit F_q, exact integer)", kernels=("k_a_miller9", "k_batch_invert", "k_a_finalexp")),
    "f": dict(param="f", mode="single", k=1, n=1 << 20, unit=78, ref_mulmods=98183, ref_main=None,
              exec_unit_ops_main=None, exec_unit_ops_all=861455, cpu_rate=70.0, port_rate=3.0,
              name="type F (param/f.param, BN k=12) element_pairing, batch 2^20 pairs per GPU, 158-bit F_q",
              dtype="u32 limbs (5 x 32-bit = 160-bit F_q, exact integer)", kernels=("k_f_miller_s", "-", "k_f_finalexp_s")),
    "d": dict(param="d159", mode="single", k=1, n=1 << 18, unit=78, ref_mulmods=23039, ref_main=None,
              exec_unit_ops_main=None, exec_unit_ops_all=720295, cpu_rate=350.0, port_rate=10.0,
              name="type D (param/d159.param, MNT k=6) element_pairing, batch 2^18 pairs per GPU, 159-bit F_q",
              dtype="u32 limbs (5 x 32-bit = 160-bit F_q, exact integer)", kernels=("k_d_miller", "-", "k_d_finalexp")),
    "g": dict(param="g149", mode="single", k=1, n=1 << 18, unit=78, ref_mulmods=None, ref_main=None,
              exec_unit_ops_main=None, exec_unit_ops_all=2827550, cpu_rate=110.0, port_rate=3.0,
              name="type G (param/g149.param, Freeman k=10) element_pairing, batch 2^18 pairs per GPU, 149-bit F_q",
              dtype="u32 limbs (5 x 32-bit = 160-bit F_q, exact integer)", kernels=("k_g_miller", "-", "k_g_finalexp")),
    "prod16": dict(param="a", mode="prod", k=16, n=1 << 16, unit=528, ref_mulmods=41536, ref_main=41536 - 719,
                   exec_unit_ops_main=16 * (1775 * 528 + 962 * 408), cpu_rate=130.0, port_rate=8.0,
                   name="type A element_prod_pairing n=16, 2^16 outputs (2^20 Miller loops) over all GPUs",
                   dtype="u32 limbs (16 x 32-bit = 512-bit F_q, exact integer)",
                   kernels=("k_a_miller9+k_a_prod", "k_batch_invert", "k_a_finalexp")),
    "pp": dict(param="a", mode="pp", k=1, n=1 << 20, unit=528, ref_mulmods=1838 + 719, ref_main=1838,
               exec_unit_ops_main=(160 * 7 + 5) * 528 + 4 * 408, cpu_rate=400.0, port_rate=110.0,
               name="type A pairing_pp_init + pairing_pp_apply: one fixed first argument, 2^20 second arguments per GPU",
               dtype="u32 limbs (16 x 32-bit = 512-bit F_q, exact integer)",
               kernels=("k_a_pp_apply", "k_batch_invert", "k_a_finalexp")),
}
def _a1_exec_ops():
    """unit ops k_a1_miller executes per pairing: 13 M + 6 S per bit of n, 16 M + 3 S per chord;
    M = 2*34^2 + 34 (operand scanning), S = 34*35/2 + 34^2 + 34 (product scanning) IMAD.WIDE.U32"""
    n = synth.parse_param(PARAMS["a1"])["n"]
    # signed digits of n (pbc_b200/csrc/host_naf.hpp): one step per digit below the top one, one
    # chord per non-zero digit strictly between the top digit and digit 0
    dg, m = [], n
    while m:
        d = 0
        if m & 1:
            d = -1 if m & 2 else 1
            m -= d
        dg.append(d)
        m >>= 1
    steps = len(dg) - 1
    chords = sum(1 for d in dg[1:-1] if d)
    M, S = 2 * 34 * 34 + 34, 34 * 35 // 2 + 34 * 34 + 34
    return steps * (13 * M + 6 * S) + chords * (16 * M + 3 * S)


WORKLOADS["a1"] = dict(
    param="a1", mode="single", k=1, n=148 * 128 * 2, unit=2 * 34 * 34 + 34, ref_mulmods=None, ref_main=None,
    exec_unit_ops_main=_a1_exec_ops(), cpu_rate=48.0, port_rate=6.0,
    name="type A1 (param/a1.param, 1033-bit p, 1022-bit composite-order-capable n) element_pairing, "
         "batch 2 x 148 x 128 pairs per GPU",
    dtype="u32 limbs (34 x 32-bit, 1033-bit F_p, exact integer)",
    kernels=("k_a1_miller", "k_batch_invert", "k_a1_finalexp"))
WIRE = {"a1": (260, 260, 260), "a": (128, 128, 128), "f": (40, 80, 240), "d159": (40, 120, 120), "g149": (38, 190, 190)}


def make_inputs(w, n_out, offset_out=0):
    """(P, Q) numpy uint8 arrays for outputs offset_out .. offset_out+n_out-1 of workload w."""
    prm = synth.parse_param(PARAMS[w["param"]])
    if w["param"] in ("a", "a1"):
        Pb, Qb = synth.type_a_points(prm, GRID if w["param"] == "a" else 512, SEED)
    else:
        g = json.load(open(os.path.join(ROOT, "tests", "golden", w["param"] + ".json")))["pairing"]
        Pb, Qb = synth.type_fd_points(prm, [bytes.fromhex(x) for x in g["P"][:2]],
                                      [bytes.fromhex(x) for x in g["Q"][:2]], GRID)
    return synth.build_batch(Pb, Qb, n_out * w["k"], offset_out * w["k"])


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


# ------------------------------------------------------------------------------------------
# CPU reference leg (oracle/_ref = the unmodified reference; else the Python port)
# ------------------------------------------------------------------------------------------
def _ref_worker(args):
    name, mode, k, Pb, Qb, n = args
    from oracle import ref as R
    rp = R.RefPairing(PARAMS[name])
    t0, c0 = time.perf_counter(), time.process_time()
    if mode == "pp":
        out = rp.pp_pairing(Pb, Qb, n)
    else:
        out = rp.pairing(Pb, Qb, n) if mode == "single" else rp.prod_pairing(Pb, Qb, k, n)
    return out, time.perf_counter() - t0, time.process_time() - c0


def _port_worker(args):
    name, mode, k, Pb, Qb, n = args
    from oracle import pbc_oracle as O
    pr = O.pairing_from_param(PARAMS[name])
    t0, c0 = time.perf_counter(), time.process_time()
    if mode == "pp":
        out = O.pairing_batch(pr, Pb[:pr.g1_len] * n, Qb, n)
    elif mode == "single":
        out = O.pairing_batch(pr, Pb, Qb, n)
    else:
        a, b = pr.g1_len, pr.g2_len
        out = b"".join(O.prod_pairing_bytes(pr, [Pb[(i * k + j) * a:(i * k + j + 1) * a] for j in range(k)],
                                            [Qb[(i * k + j) * b:(i * k + j + 1) * b] for j in range(k)])
                       for i in range(n))
    return out, time.perf_counter() - t0, time.process_time() - c0


def cpu_kind():
    try:
        from oracle import ref as R
        if R.available():
            return "reference"
    except Exception:
        pass
    return "port"


def cpu_pairings(w, P, Q, n, cores, pool=None):
    """n outputs of workload w on `cores` processes (each with its own pairing_t: the library is
    not thread-safe, SURVEY 8b).  Returns (bytes, wall seconds, CPU seconds summed over the
    workers): CPU seconds / wall is how many cores the box actually delivered."""
    import multiprocessing as mp
    g1, g2, _ = WIRE[w["param"]]
    k = w["k"]
    kind = cpu_kind()
    worker = _ref_worker if kind == "reference" else _port_worker
    per = (n + cores - 1) // cores
    jobs = []
    for c in range(cores):
        lo, hi = c * per, min(n, (c + 1) * per)
        if lo < hi:
            pslice = bytes(P[:g1]) if w["mode"] == "pp" else bytes(P[lo * k * g1:hi * k * g1])
            jobs.append((w["param"], w["mode"], k, pslice, bytes(Q[lo * k * g2:hi * k * g2]), hi - lo))
    own = pool is None
    if own:
        pool = mp.get_context("fork").Pool(len(jobs))
    t0 = time.perf_counter()
    res = pool.map(worker, jobs)
    wall = time.perf_counter() - t0
    if own:
        pool.close()
        pool.join()
    return b"".join(r[0] for r in res), wall, sum(r[2] for r in res)


def _cgroup_cpu_quota():
    """CPUs the container may use according to its cgroup (v2 cpu.max, v1 cfs quota), or None"""
    try:
        q, p = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max" and float(p) > 0:
            return float(q) / float(p)
    except Exception:
        pass
    try:
        q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
        p = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
        if q > 0 and p > 0:
            return q / p
    except Exception:
        pass
    return None


def host_cores():
    """worker processes for the CPU legs: the CPUs this process may run on, capped by the
    container's CPU quota when it has one (more runnable processes than quota only thrash)"""
    try:
        cores = max(1, len(os.sched_getaffinity(0)))
    except Exception:
        cores = max(1, os.cpu_count() or 1)
    quota = _cgroup_cpu_quota()
    if quota:
        cores = max(1, min(cores, int(quota + 0.999)))
    return cores


def cpu_rate_guess(w, kind):
    """outputs per second per core, to size the bounded CPU sample"""
    return w["cpu_rate"] if kind == "reference" else w["port_rate"]


# ------------------------------------------------------------------------------------------
# clocks during the timed region (B200_PROFILING.md)
# ------------------------------------------------------------------------------------------
class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, dev):
        self.rows = []
        self.proc = None
        self.dev = dev

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.dev), "--query-gpu=" + self.Q,
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons, pw = [], [], set(), []
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1])); pw.append(float(f[2]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": statistics.median(sm) if sm else None,
                "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(pw) if pw else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ------------------------------------------------------------------------------------------
def reference_arm(args):
    """--impl reference: the reference's own CPU implementation on the host cores."""
    rank = env_int("RANK", 0)
    if rank != 0:
        return 0
    w = WORKLOADS[args.workload]
    n_full = args.n or w["n"]
    cores = host_cores()
    kind = cpu_kind()
    per_step = int(min(n_full, max(cores * 4, args.ref_seconds * cpu_rate_guess(w, kind) * cores)))
    import multiprocessing as mp
    P, Q = make_inputs(w, per_step)
    P, Q = P.tobytes(), Q.tobytes()
    pool = mp.get_context("fork").Pool(cores)
    for _ in range(args.warmup):
        cpu_pairings(w, P, Q, min(per_step, cores * 2), cores, pool)   # warm-up
    t0 = time.perf_counter()
    cpu_s = 0.0
    for _ in range(args.steps):
        cpu_s += cpu_pairings(w, P, Q, per_step, cores, pool)[2]
    wall = time.perf_counter() - t0
    pool.close()
    pool.join()
    val = per_step * args.steps / wall
    unit = "pairings/s" if w["mode"] in ("single", "pp") else "outputs/s"
    line = {
        "impl": "reference", "metric": "pairings/sec", "value": val, "unit": unit,
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": 1e3 * wall / args.steps, "higher_is_better": True,
        "scaling": "weak" if w["mode"] in ("single", "pp") else "strong",
        "vs_baseline": None, "dtype": w["dtype"] if kind == "port" else "u64 limbs (GMP mpn)",
        "data": "synthetic",
        "config": {"workload": w["name"], "batch_per_step": per_step, "param": w["param"] + ".param",
                   "note": "bounded sample of the workload per step; CPU only"},
        "cpu_baseline": {"value": val, "unit": unit, "cores": cores, "kind": kind,
                         "sample": "%d outputs per step x %d steps, %d processes" % (per_step, args.steps, cores),
                         "cpu_seconds": cpu_s, "effective_cores": cpu_s / max(wall, 1e-9)},
        "e2e": {"value": val, "unit": unit, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------
EXTRA_CONFIGS = ("f", "d", "prod16")          # BASELINE.json configs[2], [3], [4]
# CPU seconds (wall, on this rank's share of the host cores) the parity sample of a config may take
CPU_BUDGET = {"a": 12.0, "f": 16.0, "d": 5.0, "prod16": 6.0, "g": 6.0, "pp": 6.0, "a1": 6.0}
MIN_SAMPLE = {"f": 1 << 14}                   # VERDICT r1: at least 2^14 type F outputs per rank


def shard_size(w, world, scaling):
    """outputs per rank: single pairings scale weakly by default (each rank its own full batch);
    the product config -- and everything under --scaling strong -- is one fixed batch split by output"""
    single = w["mode"] in ("single", "pp")
    if single and scaling == "weak":
        return w["n"]
    return max(1, w["n"] // world)


def sample_indices(n, m, seed):
    """m distinct output indices of [0, n): seeded random, plus the last 256 outputs (the tail of the
    last pipeline chunk / the ragged last block)"""
    import numpy as np
    m = min(m, n)
    tail = min(256, m, n)
    rng = np.random.default_rng(seed)
    body = rng.choice(n - tail, size=m - tail, replace=False) if m > tail else np.empty(0, dtype=np.int64)
    return np.sort(np.concatenate([body.astype(np.int64), np.arange(n - tail, n, dtype=np.int64)]))


DUMP_BYTES = 60 << 20          # --dump-outputs: every .npy file of one run, all ranks together, stays below 64 * 10^6 bytes


def dump_rows(n, gt, n_configs, world):
    """outputs per config and rank that --dump-outputs writes: all n if they fit the share of
    DUMP_BYTES of one config on one of the world ranks, at one float32 per wire byte, else a
    sample of that size"""
    return max(1, min(n, DUMP_BYTES // (n_configs * world) // (4 * gt)))


def dump_outputs(out_dir, wname, dO, n, gt, m, rank, world):
    """out_dir/<config>.npy (<config>.rank<r>.npy on more than one rank): the GT elements of m
    seeded outputs of this rank's batch (sample_indices; all of them when m == n), one row per
    output, one float32 per wire byte (exact).  The same arguments give the same rows every run."""
    import numpy as np
    import torch
    idx = torch.from_numpy(sample_indices(n, m, SEED + rank)).to(dO.device)
    rows = dO.view(n, gt).index_select(0, idx).cpu().numpy()
    os.makedirs(out_dir, exist_ok=True)
    name = wname if world == 1 else "%s.rank%d" % (wname, rank)
    np.save(os.path.join(out_dir, name + ".npy"), rows.astype(np.float32))


def cpu_sample(wname, w, Ph, Qh, n, rank, world, seconds, want_cpu):
    """run the reference on a seeded sample of this rank's outputs (before CUDA is initialised: the
    workers fork).  Returns (idx, expected bytes, cpu_baseline dict)."""
    import numpy as np
    if not want_cpu:
        return None, None, None
    g1, g2, _ = WIRE[w["param"]]
    k = w["k"]
    cores = max(1, host_cores() // max(1, world))
    kind = cpu_kind()
    m = int(min(n, max(cores * 2, MIN_SAMPLE.get(wname, 0), seconds * cpu_rate_guess(w, kind) * cores)))
    idx = sample_indices(n, m, SEED + 1000 * rank + sum(map(ord, wname)))
    P2 = Ph.reshape(n * k, g1) if w["mode"] != "pp" else None
    Q2 = Qh.reshape(n * k, g2)
    rows = (idx[:, None] * k + np.arange(k)[None, :]).reshape(-1)
    Ps = Ph[:g1].tobytes() if w["mode"] == "pp" else P2[rows].tobytes()
    out, wall, cpu_s = cpu_pairings(w, Ps, Q2[rows].tobytes(), len(idx), cores)
    unit_name = "pairings/s" if w["mode"] in ("single", "pp") else "outputs/s"
    cpu = {"value": len(idx) / wall, "unit": unit_name, "cores": cores, "kind": kind,
           "sample": "%d seeded random outputs of this rank's batch (incl. its last 256), %d processes, %.1f s wall"
                     % (len(idx), cores, wall),
           "cpu_seconds": cpu_s, "effective_cores": cpu_s / max(wall, 1e-9)}
    return idx, out, cpu


def reference_benchmark_c():
    """BASELINE.json configs[0]: the reference's own benchmark/benchmark.c, unmodified
    (oracle/_ref/benchmark), single thread, for a / f / d159 -- seconds per pairing as it prints them."""
    import tempfile
    from oracle import ref as R
    out = {}
    if not os.path.exists(R.BENCH_PATH):
        return {"unavailable": "oracle/_ref/benchmark not built"}
    for name in ("a", "f", "d159"):
        try:
            with tempfile.NamedTemporaryFile("w", suffix=".param", delete=False) as f:
                f.write(PARAMS[name])
            r = subprocess.run([R.BENCH_PATH, f.name], capture_output=True, text=True, timeout=120)
            os.unlink(f.name)
            t = {}
            for line in r.stdout.splitlines():
                if line.startswith("average pairing time (preprocessed) ="):
                    t["pairing_pp_apply_s"] = float(line.split("=")[1])
                elif line.startswith("average pairing time ="):
                    t["element_pairing_s"] = float(line.split("=")[1])
            t["pairings_per_s_one_thread"] = 1.0 / t["element_pairing_s"] if t.get("element_pairing_s") else None
            out[name] = t
        except Exception as e:      # noqa: BLE001
            out[name] = {"error": str(e)[:200]}
    out["source"] = "benchmark/benchmark.c:70-99 unmodified, 10 random pairs, one thread"
    return out


class GpuRun:
    """device handles shared by the configs of one process"""

    def __init__(self, rank, world, local):
        import torch
        import torch.distributed as dist
        self.torch, self.dist = torch, dist
        self.rank, self.world, self.local = rank, world, local
        torch.cuda.set_device(local)
        self.dev = torch.device("cuda", local)
        if world > 1:
            dist.init_process_group("nccl", device_id=self.dev)
        self.st = torch.cuda.current_stream()
        self.flush_buf = None
        self.peak = None

    def barrier(self):
        self.torch.cuda.synchronize()
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, x):
        t = self.torch.tensor([x], dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(self, xs):
        t = self.torch.tensor(list(xs), dtype=self.torch.float64, device=self.dev)
        if self.world > 1:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.SUM)
        return [float(v) for v in t.tolist()]

    def flush_l2(self):
        """write a buffer larger than the 126 MB L2 (between timed steps of the small configs)"""
        if self.flush_buf is None:
            self.flush_buf = self.torch.empty(256 << 20, dtype=self.torch.uint8, device=self.dev)
        self.flush_buf.add_(1)

    def imad_peak(self):
        """IMAD.WIDE.U32 per second, measured live by the microkernel (the roofline denominator)"""
        if self.peak is None:
            from pbc_b200.pairing import bench_imad
            sms = self.torch.cuda.get_device_properties(self.local).multi_processor_count
            iters = 3000
            ims = bench_imad(sms * 8, 256, iters, 3)
            self.peak = sms * 8 * 256 * 32 * iters / (ims * 1e-3)
        return self.peak


def run_config(G, wname, args, Ph, Qh, n, idx, cpu_out, cpu, steps, warmup, per_step_flush, dump_m=0):
    """time one workload on this process's GPU (all ranks call it together).  Returns the config's
    record on rank 0 (None elsewhere).  With args.dump_outputs, dump_m outputs of the last timed
    step go to that directory (dump_outputs)."""
    import numpy as np
    from pbc_b200.pairing import Pairing, kernel_launches
    torch = G.torch
    w = WORKLOADS[wname]
    k, single = w["k"], w["mode"] in ("single", "pp")
    g1, g2, gt = WIRE[w["param"]]
    unit_name = "pairings/s" if single else "outputs/s"
    world, dev, st = G.world, G.dev, G.st
    # PBC_B200_PARAM_EXTRA: extra "b200_*" test switches for A/B runs (e.g. "b200_prod_share 4"); never set by the driver
    pr = Pairing(PARAMS[w["param"]] + "\n" + os.environ.get("PBC_B200_PARAM_EXTRA", "") + "\n")
    Pp = torch.from_numpy(Ph.copy()).pin_memory()
    Qp = torch.from_numpy(Qh.copy()).pin_memory()
    Op = torch.empty(n * gt, dtype=torch.uint8).pin_memory()
    dP, dQ = Pp.to(dev), Qp.to(dev)
    dO = torch.empty(n * gt, dtype=torch.uint8, device=dev)

    # fixed first argument: pairing_pp_init once, outside the timed region, as benchmark/benchmark.c:79-84
    # does; the handle keeps the line table on the device (pbc_b200_pp_init)
    pph = pr.pp_init(Ph[:g1].tobytes()) if w["mode"] == "pp" else None

    def step():
        if w["mode"] == "pp":
            pph.apply_device(dO.data_ptr(), dQ.data_ptr(), n, st.cuda_stream)
        elif single:
            pr.apply_device(dO.data_ptr(), dP.data_ptr(), dQ.data_ptr(), n, st.cuda_stream)
        else:
            pr.prod_apply_device(dO.data_ptr(), dP.data_ptr(), dQ.data_ptr(), k, n, st.cuda_stream)

    def host_step():
        if w["mode"] == "pp":
            pph.apply_into(Op, Qp, n)
        elif single:
            pr.apply_into(Op, Pp, Qp, n)
        else:
            pr.prod_apply_into(Op, Pp, Qp, k, n)

    # ---- device-resident timing ----
    pr.set_stage_profiling(True)
    for _ in range(warmup):
        step()
    G.barrier()
    sampler = ClockSampler(G.local)
    sampler.start()
    launches0 = kernel_launches()
    if per_step_flush:
        ms_total = 0.0
        for _ in range(steps):
            G.flush_l2()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(st)
            step()
            e1.record(st)
            torch.cuda.synchronize()
            ms_total += e0.elapsed_time(e1)
    else:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(st)
        for _ in range(steps):
            step()
        e1.record(st)
        torch.cuda.synchronize()
        ms_total = e0.elapsed_time(e1)
    launches = kernel_launches() - launches0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, wname, dO, n, gt, dump_m, G.rank, world)
    G.barrier()
    # per-kernel durations: CUDA events recorded by the library on the launching stream
    stage = [0.0, 0.0, 0.0]
    reps = min(3, steps)
    for _ in range(reps):
        step()
        torch.cuda.synchronize()
        stage = [a + b for a, b in zip(stage, pr.stage_times())]
    stage = [x / reps for x in stage]
    clocks = sampler.stop()
    ms_total = G.max_over_ranks(ms_total)
    value = world * n * steps / (ms_total * 1e-3)

    # ---- parity of the device-resident outputs against the reference, this rank's sample ----
    dO_host = dO.cpu()
    checked, bad = 0, 0
    if cpu_out is not None:
        got = dO_host.numpy().reshape(n, gt)[idx].tobytes()
        checked = len(idx)
        if got != cpu_out:
            a = np.frombuffer(got, dtype=np.uint8).reshape(-1, gt)
            b = np.frombuffer(cpu_out, dtype=np.uint8).reshape(-1, gt)
            bad = int((a != b).any(axis=1).sum())

    # ---- end to end: host buffers through the C ABI (H2D of both inputs, D2H of the outputs inside) ----
    for _ in range(2):
        host_step()
    G.barrier()
    t0 = time.perf_counter()
    for _ in range(steps):
        host_step()
    torch.cuda.synchronize()
    e2e_s = G.max_over_ranks(time.perf_counter() - t0)
    e2e_val = world * n * steps / e2e_s
    e2e_same = bool(torch.equal(Op, dO_host))            # the WHOLE output buffer, every chunk
    tot = G.sum_over_ranks([checked, bad, 0 if e2e_same else 1, 1 if cpu_out is not None else 0])

    rec = None
    if G.rank == 0:
        peak = G.imad_peak()
        unit = w["unit"]
        dom = max(range(3), key=lambda i: stage[i])
        ach_ref = None
        if w.get("exec_unit_ops_main"):
            kern, kms = w["kernels"][0], stage[0]
            exec_main = w["exec_unit_ops_main"]
            if w["mode"] == "prod" and w["param"] == "a":
                # the engine shares one Miller accumulator between M = 2 pairs of a product while four waves
                # of threads remain (engine.cu, PBC_A_PROD_SHARE): per pair 159 x (10 M + 6 S) + 23.5 M + 7 S
                # instead of 159 x (11 M + 6 S) + 26 M + 8 S
                sms = torch.cuda.get_device_properties(G.local).multi_processor_count
                if n * k // 2 >= 4 * sms * 384 and k % 2 == 0 and "b200_prod_share" not in os.environ.get("PBC_B200_PARAM_EXTRA", ""):
                    exec_main = int(k * ((159 * 10 + 23.5) * 528 + (159 * 6 + 7) * 408))
                    kern = "k_a_miller9_shared+k_a_prod"
            ach_exec = n * exec_main / (kms * 1e-3)
            if w["ref_main"] is not None:
                ach_ref = n * w["ref_main"] * unit / (kms * 1e-3)
            work = ("%d IMAD.WIDE.U32 executed per output in this kernel (counted from the slot programs; "
                    "tests/test_kernels_on_cpu_sim.py ties it to the code)" % exec_main)
        else:
            # types f, d, g: the 32x32 products of the whole kernel sequence, counted by the CPU simulator
            # of the library while it runs these kernels (tests/test_kernels_on_cpu_sim.py)
            kern, kms = "+".join(x for x in w["kernels"] if x != "-"), sum(stage)
            ach_exec = n * w["exec_unit_ops_all"] / (kms * 1e-3)
            if w["ref_mulmods"]:
                ach_ref = n * w["ref_mulmods"] * unit / (kms * 1e-3)
            work = ("%d 32x32 products executed per pairing over the whole kernel sequence; dominant kernel %s = %.0f%% of the step"
                    % (w["exec_unit_ops_all"], w["kernels"][dom], 100 * stage[dom] / max(sum(stage), 1e-9)))
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        traffic = traffic_src = None
        try:
            t = json.load(open(os.path.join(ROOT, "profiles", "ncu_traffic.json")))[w["kernels"][0].split("+")[0]]
            # one ncu --set full capture of this kernel (dram__bytes_read.sum + dram__bytes_write.sum);
            # every thread moves the same bytes, so the capture's per-pairing figure scales to this launch
            traffic = t["dram_bytes_per_pairing"] * n * k
            traffic_src = "%s (n = %d), scaled to this launch's %d Miller loops" % (t["capture"], t["capture_n"], n * k)
        except Exception:
            pass
        alg_bytes = n * (k * (g1 + g2) + gt)
        hbm_ach = alg_bytes / (sum(stage) * 1e-3) / 1e9
        frac = ach_exec / peak
        roof = {"bound": "int-mul pipe (IMAD.WIDE.U32 issue; SURVEY 8d)", "kernel": kern,
                "achieved": ach_exec / 1e12, "peak": peak / 1e12, "unit": "T IMAD.WIDE.U32/s",
                "frac": frac, "frac_is": "executed multiplier operations / measured issue peak (a pipe utilisation, <= 1)",
                "peak_source": "live microkernel k_imad_peak (MEASURED_PEAKS.json has no integer peak)",
                "work": work, "traffic": traffic, "traffic_source": traffic_src,
                "algorithmic_bytes": alg_bytes,
                "hbm": {"bound": "hbm", "achieved": hbm_ach, "peak": hbm_peak, "unit": "GB/s",
                        "frac": hbm_ach / hbm_peak, "peak_source": "MEASURED_PEAKS.json" if peaks else "fallback",
                        "note": "%d wire bytes per output: does not bound the path" % (k * (g1 + g2) + gt)}}
        if ach_ref is not None:
            roof["achieved_reference_equivalent"] = ach_ref / 1e12
            roof["frac_reference_equivalent"] = ach_ref / peak
            roof["reference_equivalent_is"] = ("the reference algorithm's mulmod count x %d unit ops per mulmod over the same "
                                               "time: above frac because these kernels execute fewer multiplications" % unit)
        # (a run under a profiler times the peak microkernel with the profiler's per-launch overhead in it: the launch-list
        # recipes set PBC_B200_UNDER_PROFILER=1, and no number printed by such a run is a bench value)
        assert frac <= 1.05 or os.environ.get("PBC_B200_UNDER_PROFILER"), \
            "roofline.frac %.3f > 1: the executed-work count or the peak is wrong" % frac
        ws_per = 704 * k if w["param"] == "a" else {"f": (61 + 30 + 240) * 4, "d159": 31 * 4, "g149": 51 * 4, "a1": 6 * 136}[w["param"]]
        rec = {
            "value": value, "unit": unit_name, "steps": steps, "warmup": warmup, "ms_per_step": ms_total / steps,
            "scaling": "weak" if (single and args.scaling == "weak") else "strong",
            "dtype": w["dtype"],
            "config": {"workload": w["name"], "param": w["param"] + ".param", "batch_per_gpu": n,
                       "global_batch": world * n, "pairings_per_output": k,
                       "parallelism": "shard%d (independent outputs, no collective)" % world,
                       "inputs": "%dx%d grid of seeded subgroup points, all pairs distinct" % ((GRID, GRID) if w["param"] != "a1" else (512, 512)),
                       "l2": ("inputs+outputs+workspace %.0f MB per step vs 126 MB L2" % ((n * (k * (g1 + g2) + gt + ws_per)) / 1e6))
                             + ("; L2 flushed (256 MB write) between timed steps" if per_step_flush else "")},
            "clocks": clocks,
            "e2e": {"value": e2e_val, "unit": unit_name, "h2d_bytes_per_step": n * k * (g1 + g2),
                    "d2h_bytes_per_step": n * gt,
                    "timer": "perf_counter around the blocking C-ABI call, pinned host buffers, max over ranks",
                    "matches_device_resident_output": tot[2] == 0,
                    "compared": "all %d output bytes of every rank" % (n * gt)},
            "gpu_launches": launches,
            "stage_ms": dict(zip(("main", "mid", "final_exp"), stage)),
            "stage_kernels": list(w["kernels"]),
            "roofline": roof,
            "cpu_baseline": cpu,
            "parity": ({"checked": int(tot[0]), "mismatches": int(tot[1]), "bit_exact": tot[1] == 0 and tot[2] == 0,
                        "ranks_checked": int(tot[3]), "against": "oracle/_ref (unmodified reference), seeded random index sample per rank + whole e2e buffer vs device buffer"}
                       if tot[3] > 0 else None),
        }
    if pph is not None:
        pph.clear()
    pr.clear()
    del dP, dQ, dO, Pp, Qp, Op
    torch.cuda.empty_cache()
    return rec


def fp_mul_report(G):
    """SURVEY 8d / north_star: F_p multiplication throughput as a fraction of the integer-pipe roofline"""
    from pbc_b200.pairing import Pairing
    torch = G.torch
    sms = torch.cuda.get_device_properties(G.local).multi_processor_count
    peak = G.imad_peak()
    out = {}
    for name, label, imad, modes in (("a", "512-bit F_q (type A), 16 x 32-bit limbs", 528, ((0, "registers, operand scanning"), (1, "through the shared-memory slot machine (what the kernels run)"))),
                                     ("f", "158-bit F_q (type F), 5 x 32-bit limbs", 55, ((0, "registers, product scanning"),))):
        pr = Pairing(PARAMS[name])
        rows = []
        for mode, what in modes:
            blocks, iters = sms * 8, 2000 if name == "a" else 20000
            ms = pr.bench_fpmul(mode, blocks, iters, 3)
            rate = blocks * 128 * iters / (ms * 1e-3)
            rows.append({"how": what, "mulmods_per_s": rate, "imad_wide_per_mulmod": imad,
                         "frac_of_imad_peak": rate * imad / peak})
        out[name] = {"field": label, "runs": rows}
        pr.clear()
    out["peak_imad_wide_per_s"] = peak
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="a", choices=sorted(WORKLOADS))
    ap.add_argument("--configs", default=None, help="comma list of extra configs measured after the headline "
                    "(default: f,d,prod16 when --workload a and no --n; 'none' to skip)")
    ap.add_argument("--scaling", default="weak", choices=["weak", "strong"],
                    help="strong: the workload's batch is split across the ranks instead of replicated")
    ap.add_argument("--n", type=int, default=0, help="outputs per GPU per step (default: the workload's)")
    ap.add_argument("--cpu-seconds", type=float, default=0.0, help="CPU parity/baseline budget per config (default: per-config table)")
    ap.add_argument("--ref-seconds", type=float, default=3.0, help="--impl reference: seconds per step")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--extra-steps", type=int, default=None, help="timed steps of each extra config (default: --steps)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write each config's outputs of its last timed step to DIR/<config>.npy "
                         "(<config>.rank<r>.npy per rank on more than one GPU; float32, one row per output, one column "
                         "per wire byte; a fixed seeded sample where all of them would exceed 64 MB over all files of "
                         "all ranks)")
    args = ap.parse_args()
    if args.steps < 1 or (args.extra_steps is not None and args.extra_steps < 1):
        ap.error("--steps and --extra-steps must be at least 1")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the GPU path's outputs (--impl b200)")
    if args.warmup < 3:
        args.warmup = 3
    if args.impl == "reference":
        return reference_arm(args)

    rank, world, local = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
    if args.configs is None:
        extras = list(EXTRA_CONFIGS) if (args.workload == "a" and not args.n) else []
    else:
        extras = [c for c in args.configs.split(",") if c and c != "none"]
    names = [args.workload] + [c for c in extras if c != args.workload]

    # ---- phase 1 (no CUDA yet): inputs and the reference's outputs on each config's sample ----
    plans = {}
    for i, wname in enumerate(names):
        w = WORKLOADS[wname]
        n = args.n if (args.n and i == 0) else shard_size(w, world, args.scaling)
        Ph, Qh = make_inputs(w, n, offset_out=rank * n)
        secs = args.cpu_seconds or CPU_BUDGET.get(wname, 6.0)
        try:
            idx, cpu_out, cpu = cpu_sample(wname, w, Ph, Qh, n, rank, world, secs, not args.no_cpu_baseline)
        except Exception as e:                      # noqa: BLE001  (an extra config must not take the headline down)
            if i == 0:
                raise
            idx = cpu_out = None
            cpu = {"error": str(e)[:300]}
        plans[wname] = (Ph, Qh, n, idx, cpu_out, cpu)
    bench_c = reference_benchmark_c() if (rank == 0 and not args.no_cpu_baseline) else None

    # ---- phase 2: the GPU ----
    from pbc_b200 import _lib as _pbc_lib
    if _pbc_lib.IS_SIMULATOR:
        raise SystemExit("bench.py measures the CUDA library; PBC_B200_LIB points at the test suite's CPU simulator")
    G = GpuRun(rank, world, local)
    recs = {}
    for i, wname in enumerate(names):
        Ph, Qh, n, idx, cpu_out, cpu = plans.pop(wname)
        dump_m = dump_rows(n, WIRE[WORKLOADS[wname]["param"]][2], len(names), world)
        if i == 0:
            recs[wname] = run_config(G, wname, args, Ph, Qh, n, idx, cpu_out, cpu, args.steps, args.warmup, False, dump_m)
        else:
            try:
                recs[wname] = run_config(G, wname, args, Ph, Qh, n, idx, cpu_out, cpu,
                                         args.extra_steps or args.steps, 3, True, dump_m)
            except Exception as e:                  # noqa: BLE001
                recs[wname] = {"error": str(e)[:300]}
        del Ph, Qh
    fpm = fp_mul_report(G) if rank == 0 else None
    if world > 1:
        G.dist.destroy_process_group()
    if rank == 0:
        h = recs[args.workload]
        line = {
            "metric": "pairings/sec", "value": h["value"], "unit": h["unit"], "n_gpus": world,
            "steps": h["steps"], "warmup": h["warmup"], "ms_per_step": h["ms_per_step"],
            "higher_is_better": True, "scaling": h["scaling"], "vs_baseline": None,
            "dtype": h["dtype"], "data": "synthetic", "config": h["config"], "clocks": h["clocks"],
            "e2e": h["e2e"], "gpu_launches": h["gpu_launches"], "stage_ms": h["stage_ms"],
            "stage_kernels": h["stage_kernels"], "roofline": h["roofline"], "cpu_baseline": h["cpu_baseline"],
            "parity": h["parity"],
            "configs": {k: v for k, v in recs.items() if k != args.workload},
            "fp_mul": fpm,
            "reference_benchmark_c": bench_c,
        }
        sys.stdout.flush()
        print(json.dumps(line), flush=True)       # the LAST line of stdout (NCCL_DEBUG output, if any, precedes it)
    return 0


if __name__ == "__main__":
    sys.exit(main())
