"""ReadLowHashStatistics.csv written by the facade against the file the reference's own LowHash0 leaves in its working directory
(src/LowHash0.cpp:220-243)."""
import os
import sys

import numpy as np

from shasta_b200 import assembler as A

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
import make_ref_golden as RG  # noqa: E402


def test_csv_is_byte_identical_to_the_reference(tmp_path, monkeypatch, golden_dir):
    # the reference's per-read statistics and the file it wrote from them (tests/golden/make_ref_golden.py)
    monkeypatch.chdir(tmp_path)
    g = np.load(os.path.join(golden_dir, "ref_golden.npz"))
    d = RG.csv_input()
    for i, (m, _, _) in enumerate(RG.CSV_CASES):
        stats = g[f"csv_{i}_stats"]
        want = g[f"csv_{i}_text"].tobytes().decode()
        A.write_read_low_hash_statistics_csv("ours.csv", stats, d["toc"], d["flags"], m)
        got = open("ours.csv").read()
        assert got == want
        assert want.count("\n") == 301 and ",Yes," in want
