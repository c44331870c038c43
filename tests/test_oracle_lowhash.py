"""CPU tests: the oracle restatement (oracle/lowhash_oracle.c) against the reference's golden vectors.

Golden material (SURVEY.md section 8c / Appendix B, D):
  * MurmurHash64A / MurmurHash2 known answers computed from the reference's src/MurmurHash2.cpp;
  * the feature enumeration example of docs/ComputationalMethods.html:750-765;
  * LowHash0 outputs of the unmodified reference on TinyTest and synthetic inputs (tests/golden), with parameters of the
    configurations and away from them.
"""
import json
import os
import sys

import numpy as np
import pytest

from oracle import bindings as B
from shasta_b200 import synth

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
import make_golden as MG  # noqa: E402
import make_ref_golden as RG  # noqa: E402


def test_murmurhash64a_known_answers():
    lib = B.oracle_lib()
    k = np.array([18, 45, 71, 3, 15, 6, 21], dtype=np.uint32)
    expect = {
        0: [0xee0158aa3dfea324, 0xff91d029981e26c1, 0xcedd8a9da9aaec4b, 0x4dc4e78740063776],
        1: [0xabd0de78c17412ad, 0x5eafe47a716e671a, 0xdecc94520b564857, 0x48b46c5b6a7e273f],
        2: [0x1d489d476b40a116, 0x5363496b2da5ffa4, 0xd61878e20588c54e, 0x88dc7f6cfb55d815],
    }
    for it, hs in expect.items():
        for j, h in enumerate(hs):
            assert lib.orc_murmurhash64a(k[j:].ctypes.data, 16, 37 * it) == h
    # m = 3: 12 bytes, tail path
    assert lib.orc_murmurhash64a(k.ctypes.data, 12, 0) == 0x1803d68b59540148


def test_murmurhash2_known_answer():
    lib = B.oracle_lib()
    n = np.array([80235], dtype=np.uint64)
    assert lib.orc_murmurhash2(n.ctypes.data, 8, 13477) == 0x9e42279c


def test_thresholds():
    # src/LowHash0.cpp:109, src/AssemblerAlign3.cpp:71-72 (SURVEY.md Appendix B)
    assert int(np.float64(0.01) * np.float64(np.iinfo(np.uint64).max)) == 184467440737095520
    assert int(np.float64(0.05) * np.float64(np.iinfo(np.uint64).max)) == 922337203685477632
    assert int(0.05 * float(2**32 - 1)) == 214748364
    assert int(0.1 * float(2**32 - 1)) == 429496729


def test_reverse_complement_on_reference_markers(golden_dir):
    # The reference's MarkerFinder writes the strand-1 row as the reversed strand-0 row with
    # reverse-complemented k-mers and mirrored positions (src/MarkerFinder.cpp:92-100).
    z = np.load(os.path.join(golden_dir, "tinytest_markers.npz"))
    km, ps = synth.unpack_markers(z["data"])
    toc = z["toc"].astype(np.int64)
    lib = B.oracle_lib()
    for r in range(len(z["flags"])):
        a, b, c = toc[2 * r], toc[2 * r + 1], toc[2 * r + 2]
        assert b - a == c - b
        assert np.array_equal(synth.reverse_complement_kmer(km[a:b][::-1], 10), km[b:c])
        assert len(set((ps[a:b][::-1].astype(np.int64) + ps[b:c].astype(np.int64)).tolist())) == 1
    for x in (0, 1, 12345, (1 << 20) - 1):
        assert lib.orc_reverse_complement_kmer(x, 10) == int(synth.reverse_complement_kmer(np.array([x]), 10)[0])
        assert lib.orc_reverse_complement_kmer(lib.orc_reverse_complement_kmer(x, 10), 10) == x


@pytest.mark.parametrize("name", list(MG.LOWHASH_CASES))
def test_oracle_matches_reference_golden(name, golden_dir):
    spec, params = MG.LOWHASH_CASES[name]
    d = MG.load_input(spec)
    g = np.load(os.path.join(golden_dir, "lowhash_golden.npz"))
    meta = json.load(open(os.path.join(golden_dir, "lowhash_golden.json")))[name]
    c, s, it = B.oracle_lowhash0(d["toc"], d["data"], d["flags"], B.LowHashParams(**params))
    assert int(d["toc"][-1]) == meta["markers"]
    assert np.array_equal(c, g[name + "/candidates"])
    assert np.array_equal(s, g[name + "/stats"])
    assert np.array_equal(it, g[name + "/summary"])
    assert hex(B.candidate_digest(c)) == meta["digest"]


def test_tinytest_pin(golden_dir):
    # SURVEY.md Appendix D: 20 reads, 124 036 markers, 186 candidates, digest 0x3fc2c96e354f8733,
    # per-iteration (high frequency, total) and per-read statistics heads.
    g = np.load(os.path.join(golden_dir, "lowhash_golden.npz"))
    c = g["tiny_default/candidates"]
    assert len(c) == 186 and B.candidate_digest(c) == 0x3fc2c96e354f8733
    assert c[:4].tolist() == [[0, 2, 0], [0, 3, 1], [0, 3, 0], [0, 4, 1]]
    assert g["tiny_default/summary"].tolist() == [[127, 152], [161, 178], [165, 180], [168, 181], [170, 183],
                                                  [175, 188], [182, 192], [182, 193], [184, 193], [186, 193]]
    assert g["tiny_default/stats"][[0, 1, 3]].tolist() == [[0, 589, 14], [0, 202, 2], [0, 2114, 46]]


def test_bucket_count_too_small_raises(golden_dir):
    z = np.load(os.path.join(golden_dir, "tinytest_markers.npz"))
    with pytest.raises(RuntimeError):
        B.oracle_lowhash0(z["toc"], z["data"], z["flags"], B.LowHashParams(log2MinHashBucketCount=5))


def test_oracle_matches_live_reference_random_params(golden_dir):
    # Parameters away from the configurations, against the reference build's outputs (tests/golden/make_ref_golden.py).
    g = np.load(os.path.join(golden_dir, "ref_golden.npz"))
    d = RG.lowhash_random_input()
    for j, params in enumerate(RG.LOWHASH_RANDOM_PARAMS):
        oc, os_, oit = B.oracle_lowhash0(d["toc"], d["data"], d["flags"], B.LowHashParams(**params))
        assert np.array_equal(g[f"lowhash_{j}_candidates"], oc) and np.array_equal(g[f"lowhash_{j}_stats"], os_)
        assert np.array_equal(g[f"lowhash_{j}_summary"], oit)
