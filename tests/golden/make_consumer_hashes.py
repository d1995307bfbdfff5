"""Expected outputs of the compiled C-ABI consumers (oracle/abi_consumer.cpp, tests/test_abi_consumer.py).

For every consumer configuration of oracle/Makefile and both input kinds, regenerates the consumer's synthetic input
(xorshift64 noise, or dark noise 0..15, planar [C][H][W]) and stores the FNV-1a-64 of lanczos_expected's output for it
in tests/golden/abi_consumer_hashes.txt.  lanczos_expected is run through the CPU oracle, literal per-tap restatement and
fast path (which must agree); test_oracle.py::test_golden_fixtures pins both to the reference's own outputs on other
configurations.  The hashes are the oracle's, not outputs of the reference run on these inputs.
  python tests/golden/make_consumer_hashes.py
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import oracle_py as O  # noqa: E402

# (in_w, in_h, out_w, out_h, n, d, a, c): CONSUMERS of oracle/Makefile
CONFIGS = [(162, 89, 486, 267, 3, 1, 2, 3), (240, 135, 480, 270, 2, 1, 3, 3), (96, 54, 144, 81, 3, 2, 3, 4)]
M64 = (1 << 64) - 1


def consumer_input(cfg, content):
    """The input main() of oracle/abi_consumer.cpp fills in."""
    iw, ih, _, _, _, _, _, c = cfg
    s = 0x9E3779B97F4A7C15
    out = np.empty(c * ih * iw, np.uint8)
    for i in range(out.size):
        s ^= (s << 13) & M64
        s ^= s >> 7
        s ^= (s << 17) & M64
        out[i] = (s >> 24) & (15 if content == "dark" else 255)
    return out.reshape(c, ih, iw)


def main():
    path = os.path.join(ROOT, "tests", "golden", "abi_consumer_hashes.txt")
    lines = ["# in_w in_h out_w out_h n d a c content fnv1a64(lanczos_expected output, planar c,y,x); "
             "input = oracle/abi_consumer.cpp main(); tests/golden/make_consumer_hashes.py\n"]
    for cfg in CONFIGS:
        iw, ih, ow, oh, n, d, a, c = cfg
        for content in ("noise", "dark"):
            img = consumer_input(cfg, content)
            out = O.expected_planar(img, ow, oh, a, n, d, fast=False)
            assert np.array_equal(out, O.expected_planar(img, ow, oh, a, n, d, fast=True)), (cfg, content)
            lines.append(" ".join(str(v) for v in cfg) + f" {content} {O.fnv1a64(out):016x}\n")
            print(lines[-1].strip())
    with open(path, "w") as fh:
        fh.writelines(lines)


if __name__ == "__main__":
    main()
