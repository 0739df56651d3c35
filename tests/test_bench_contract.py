"""bench.py's CPU-only legs: the reference arm (`--impl reference`) prints the contract's JSON line;
the synthetic inputs are points of the right subgroup.  The GPU arm is exercised on the B200 box."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _ref_available():
    from oracle import ref
    return ref.available()


@pytest.mark.parametrize("workload", ["a", "a1"])
def test_reference_arm_prints_the_contract_line(workload):
    # the CPU arm runs the compiled reference where oracle/_ref is built, else the Python port of it
    kind = "reference" if _ref_available() else "port"
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--workload", workload,
                          "--steps", "1", "--warmup", "1", "--ref-seconds", "0.5"],
                         capture_output=True, text=True, timeout=600, check=True)
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    assert len(lines) == 1, out.stdout
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "pairings/sec" and d["higher_is_better"] is True
    assert d["value"] > 0 and d["n_gpus"] == 1 and d["steps"] == 1 and d["gpu_launches"] == 0
    cb = d["cpu_baseline"]
    assert cb["kind"] == kind and cb["cores"] >= 1 and cb["value"] == d["value"]
    assert 0 < cb["effective_cores"] <= cb["cores"] * 1.05
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}


def test_synthetic_a1_inputs_lie_in_the_order_n_subgroup():
    sys.path.insert(0, ROOT)
    import bench
    from oracle import pbc_oracle as O
    from pbc_b200.params import PARAMS
    w = bench.WORKLOADS["a1"]
    P, Q = bench.make_inputs(w, 3)
    pr = O.pairing_from_param(PARAMS["a1"])
    for buf in (P, Q):
        for i in range(3):
            pt = pr.G1.from_bytes(bytes(buf[i * 260:(i + 1) * 260]))
            assert pt is not None and pr.E.is_valid(pt) and pr.E.mul(pr.r, pt) is None
    assert w["exec_unit_ops_main"] == 56225715      # signed-digit scan of n (PBC_A1_NAF, default since round 2)


def test_parity_sample_is_seeded_distinct_and_reaches_the_last_chunk():
    """the index sample bench.py checks against oracle/_ref on every rank: distinct, reproducible,
    different per rank, and always containing the tail of the batch"""
    sys.path.insert(0, ROOT)
    import bench
    a = bench.sample_indices(1 << 20, 20000, 7)
    b = bench.sample_indices(1 << 20, 20000, 7)
    c = bench.sample_indices(1 << 20, 20000, 8)
    assert (a == b).all() and not (a == c).all()
    assert len(set(a.tolist())) == 20000 and a[-1] == (1 << 20) - 1 and a[-256] == (1 << 20) - 256
    assert (a[:-256] < (1 << 20) - 256).all() and a[0] >= 0
    # spread over every 2^18-output pipeline chunk of the host path
    assert all(((a >> 18) == ch).sum() > 1000 for ch in range(4))
    assert list(bench.sample_indices(5, 100, 1)) == [0, 1, 2, 3, 4]


def test_shard_sizes_follow_the_scaling_mode():
    sys.path.insert(0, ROOT)
    import bench
    W = bench.WORKLOADS
    assert bench.shard_size(W["a"], 8, "weak") == 1 << 20 and bench.shard_size(W["a"], 8, "strong") == 1 << 17
    assert bench.shard_size(W["prod16"], 8, "weak") == 1 << 13 and bench.shard_size(W["d"], 2, "weak") == 1 << 18


def test_dumped_outputs_stay_within_64_mb():
    sys.path.insert(0, ROOT)
    import bench
    W = bench.WORKLOADS
    for names in (["a", "f", "d", "prod16"], ["f"], sorted(W)):
        for world in (1, 2, 8):
            for scaling in ("weak", "strong"):
                total = 0           # every rank writes one file per config
                for x in names:
                    gt = bench.WIRE[W[x]["param"]][2]
                    rows = bench.dump_rows(bench.shard_size(W[x], world, scaling), gt, len(names), world)
                    total += world * (128 + 4 * gt * rows)     # .npy header + data
                assert 32 << 20 < total <= 64 * 10 ** 6, (names, world, scaling, total)
    assert bench.dump_rows(4096, 128, 4, 1) == 4096 and bench.dump_rows(4096, 128, 4, 8) == 3840


def test_steps_below_one_are_refused():
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--steps", "0"],
                       capture_output=True, text=True, timeout=300)
    assert r.returncode == 2 and "--steps" in r.stderr


@pytest.mark.gpu
def test_dump_outputs_are_what_the_library_computes_for_the_timed_inputs(tmp_path):
    """The plumbing of bench.py --dump-outputs: the rows it writes (every output of a small headline
    config, a seeded sample of the 2^18 outputs of config d) are, byte for byte, the library's
    pairings of inputs made afresh from the same arguments, so the rows, their seeded indices and
    the float32 encoding are right; --steps sets the timed steps of every config.  Whether those
    pairings are correct is what the reference fixtures of the other GPU tests check.  Every timed
    step computes the same outputs, so this cannot tell the last step from an earlier one: the dump
    reads the output buffer right after the timed loop."""
    import numpy as np
    sys.path.insert(0, ROOT)
    import bench
    from pbc_b200.pairing import Pairing
    from pbc_b200.params import PARAMS
    out = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--gpus", "1", "--steps", "2", "--warmup", "3",
                          "--n", "4096", "--configs", "d", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                         capture_output=True, text=True, timeout=900)
    assert out.returncode == 0, out.stderr[-3000:]
    d = json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])
    assert d["steps"] == 2 and d["configs"]["d"]["steps"] == 2
    assert sorted(os.listdir(tmp_path)) == ["a.npy", "d.npy"]
    for wname, n in (("a", 4096), ("d", 1 << 18)):
        w = bench.WORKLOADS[wname]
        gt = bench.WIRE[w["param"]][2]
        got = np.load(str(tmp_path / (wname + ".npy")))
        m = bench.dump_rows(n, gt, 2, 1)
        assert got.dtype == np.float32 and got.shape == (m, gt)
        assert (m == n) == (wname == "a")
        idx = bench.sample_indices(n, m, bench.SEED)
        P, Q = bench.make_inputs(w, n)
        g1, g2 = bench.WIRE[w["param"]][:2]
        pr = Pairing(PARAMS[w["param"]])
        want = pr.apply(P.reshape(n, g1)[idx].tobytes(), Q.reshape(n, g2)[idx].tobytes(), m)
        pr.clear()
        assert got.astype(np.uint8).tobytes() == want and (got == got.astype(np.uint8)).all()
