"""Drop-in check through the reference's own C API (pbc.h): shim/_build holds programs built
against the reference headers and linked with libpbc_b200_shim.so in front of the unmodified
reference library (shim/Makefile).  They exist only where the reference sources were at hand when
the project was built; elsewhere the two tests that run them skip."""
import os
import subprocess

import pytest

from pbc_b200.params import PARAMS

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
BUILD = os.path.join(ROOT, "shim", "_build")


def _need(name):
    path = os.path.join(BUILD, name)
    if not os.path.exists(path):
        pytest.skip("shim/_build/%s not built (needs the reference headers and library: make -C shim)" % name)
    return path


@pytest.mark.parametrize("name", ["a", "f", "d159", "g149"])
def test_pbc_api_on_gpu_matches_reference_vtable(tmp_path, name):
    exe = _need("shim_test")
    pf = tmp_path / (name + ".param")
    pf.write_text(PARAMS[name])
    r = subprocess.run([exe, str(pf), "200"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert "shim_test: OK" in r.stdout


def test_reference_benchmark_program_links_unchanged_and_runs_on_gpu(tmp_path):
    """benchmark/benchmark.c, unmodified: its self-check compares pairing_pp_apply with
    element_pairing and exits 1 printing BUG! on a mismatch (benchmark/benchmark.c:93-96)."""
    exe = _need("benchmark_b200")
    r = subprocess.run([exe], input=PARAMS["a"], capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout[-2000:] + r.stderr
    assert "BUG" not in r.stdout and "average pairing time" in r.stdout
    # pairing_pp_init keeps the line table on the GPU (pbc_b200_pp_init): the preprocessed call must
    # now be the cheaper one, as it is for the reference (benchmark/benchmark.c:98-99)
    t = {}
    for line in r.stdout.splitlines():
        if line.startswith("average pairing time (preprocessed) ="):
            t["pp"] = float(line.split("=")[1])
        elif line.startswith("average pairing time ="):
            t["plain"] = float(line.split("=")[1])
    assert t["pp"] < t["plain"], t


@pytest.mark.parametrize("name", ["a", "f", "d159", "g149"])
def test_plain_c_caller_of_the_c_abi(tmp_path, name, golden):
    """examples/batch_pairing_demo.c: a C program that includes only include/pbc_b200.h"""
    exe = os.path.join(ROOT, "examples", "_build", "batch_pairing_demo")
    assert os.path.exists(exe), "examples/_build/batch_pairing_demo is missing: run `python __graft_entry__.py`"
    g = golden[name]["pairing"]
    (tmp_path / "p.param").write_text(PARAMS[name])
    (tmp_path / "P.bin").write_bytes(b"".join(bytes.fromhex(x) for x in g["P"]))
    (tmp_path / "Q.bin").write_bytes(b"".join(bytes.fromhex(x) for x in g["Q"]))
    r = subprocess.run([exe, str(tmp_path / "p.param"), str(tmp_path / "P.bin"), str(tmp_path / "Q.bin"),
                        str(tmp_path / "E.bin")], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stdout + r.stderr
    assert (tmp_path / "E.bin").read_bytes() == b"".join(bytes.fromhex(x) for x in g["e"])


@pytest.mark.parametrize("name", ["a", "f", "d159", "g149"])
def test_bls_batch_verify_example(name):
    import sys
    r = subprocess.run([sys.executable, os.path.join(ROOT, "examples", "bls_batch_verify.py"), name, "96"],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stdout + r.stderr
    assert '"rejected": [48]' in r.stdout
