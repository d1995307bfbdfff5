"""A compiled C++ consumer of include/lanczos_b200.h (SURVEY.md 8b, VERDICT r1 #9).

oracle/Makefile (target `consumer`, run by __graft_entry__.build() and by the `exes` fixture) compiles
oracle/abi_consumer.cpp -- INTEGRATION.md's `lanczos_expected_b200` binding and a `main` that fills the reference's
static planar arrays -- into oracle/_consumers/abi_consumer_*, one executable per params.h configuration, linked
against liblanczos_b200.so.  Each prints the FNV-1a-64 of its output; tests/golden/abi_consumer_hashes.txt holds the
hash of lanczos_expected's output for the same input as the CPU oracle computes it (tests/golden/make_consumer_hashes.py;
test_oracle.py::test_golden_fixtures pins the oracle to the reference's own outputs).
"""
import glob
import os
import re
import subprocess

import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
ORACLE = os.path.join(HERE, "..", "oracle")
HASHES = os.path.join(HERE, "golden", "abi_consumer_hashes.txt")


def consumers():
    return sorted(glob.glob(os.path.join(ORACLE, "_consumers", "abi_consumer_*")))


@pytest.fixture(scope="module")
def exes(lz):
    subprocess.run(["make", "-s", "-C", ORACLE, "consumer"], check=True)      # rebuilds only what is stale
    return consumers()


def expected_hashes():
    """{(config name as in the executable's file name, content): fnv1a64}"""
    want = {}
    with open(HASHES) as fh:
        for line in fh:
            if line.startswith("#") or not line.strip():
                continue
            iw, ih, ow, oh, n, d, a, c, content, h = line.split()
            want[(f"{iw}x{ih}_{ow}x{oh}_{n}_{d}_a{a}_c{c}", content)] = int(h, 16)
    return want


def test_consumers_are_built_and_link_against_the_product_library(exes):
    assert len(exes) >= 3, "run `make -C oracle` after building the library"
    for exe in exes:
        out = subprocess.run(["ldd", exe], capture_output=True, text=True).stdout
        assert "liblanczos_b200.so" in out and "not found" not in out.split("liblanczos_b200.so")[1].split("\n")[0], out


@pytest.mark.gpu
@pytest.mark.parametrize("content", ["noise", "dark"])
def test_compiled_consumer_matches_the_reference_function(exes, content):
    want = expected_hashes()
    assert len(exes) >= 3, "run `make -C oracle` after building the library"
    for exe in exes:
        cfg = os.path.basename(exe)[len("abi_consumer_"):]
        res = subprocess.run([exe, content], capture_output=True, text=True, timeout=300)
        assert res.returncode == 0, (exe, res.stdout, res.stderr)
        got = int(re.search(r"fnv1a64 ([0-9a-f]{16})", res.stdout).group(1), 16)
        assert got == want[(cfg, content)], res.stdout
