"""CPU test: the marker-finding oracle (oracle/markers_oracle.c) against the golden output of the UNMODIFIED reference
MarkerFinder on TinyTest (tests/golden/tinytest_markers.npz; inputs tests/golden/tinytest_reads.npz), and against the
reference's ReadLoader + MarkerFinder on synthetic FASTA files (tests/golden/ref_golden.npz)."""
import os
import sys

import numpy as np

from oracle import bindings as B

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import make_ref_golden as RG  # noqa: E402


def _golden():
    r = np.load(os.path.join(ROOT, "tests", "golden", "tinytest_reads.npz"))
    m = np.load(os.path.join(ROOT, "tests", "golden", "tinytest_markers.npz"))
    is_marker = np.unpackbits(r["is_marker_bitmap"].view(np.uint8), bitorder="little")
    return r, m, is_marker


def test_marker_oracle_reproduces_reference_tinytest():
    r, m, is_marker = _golden()
    assert int(r["k"]) == 10 and len(is_marker) == 4 ** 10
    toc, data = B.oracle_find_markers(r["word_offsets"], r["words"], r["base_counts"], is_marker, 10)
    assert toc[-1] == 124036                    # SURVEY.md F5
    assert np.array_equal(toc, m["toc"]) and np.array_equal(data, m["data"])


def test_marker_oracle_against_live_reference():
    g = np.load(os.path.join(ROOT, "tests", "golden", "ref_golden.npz"))
    for name in ("fasta40_s3_k8", "fasta40_s3_k10"):
        r = RG.fasta_case(g, name)
        toc, data = B.oracle_find_markers(r["word_offsets"], r["words"], r["base_counts"], r["is_marker"], r["k"])
        assert toc[-1] > 1000
        RG.assert_markers_match(g, name, toc, data)
