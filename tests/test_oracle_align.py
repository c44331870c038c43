"""CPU tests: the alignment oracle (oracle/align_oracle.c) against the reference's golden vectors, among them outputs of the
unmodified Align4.cpp / Alignment.cpp / compressAlignment.cpp stored in tests/golden.

The overlap DP's tie-break rule is 'parity unpinned' (SeqAn absent, SURVEY.md F4); what IS pinned here:
  * shasta::compress bytes of the reference's own test vectors (SURVEY.md Appendix D),
  * AlignmentInfo::create and compress against the compiled reference on real alignments,
  * the whole Align4 front end (cells, searches, components, band, selection) against the compiled Align4.cpp,
  * DP optimality properties that hold for any correct implementation (score = brute force, path validity).
"""
import os
import sys

import numpy as np

from oracle import bindings as B
from shasta_b200 import synth

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
import make_ref_golden as RG  # noqa: E402

# src/compressAlignment.cpp:161-192 (testAlignmentCompression): 30 ordinal pairs exercising Formats 0-4.
COMPRESSION_TEST_VECTOR = [
    (300, 200), (301, 201), (302, 202), (305, 206), (306, 207), (320, 250), (321, 251), (322, 252), (323, 253)]
GOLDEN_9 = "63091901190a73608501"


def test_compress_worked_example():
    # src/compressAlignment.hpp:28-50 example; bytes from the reference (SURVEY.md Appendix D).
    o = np.array(COMPRESSION_TEST_VECTOR, np.uint32)
    assert B.oracle_compress(o).tobytes().hex() == GOLDEN_9
    assert np.array_equal(B.oracle_decompress(B.oracle_compress(o)), o)


def test_reference_selftest_and_compress_vectors(golden_dir):
    # shasta::compress bytes of the reference for the ordinals of its own testAlignmentCompression and for seeded runs
    # (tests/golden/make_ref_golden.py)
    g = np.load(os.path.join(golden_dir, "ref_golden.npz"))
    o = g["selftest_ordinals"]
    assert np.array_equal(B.oracle_compress(o), g["selftest_compressed"])
    assert np.array_equal(B.oracle_decompress(g["selftest_compressed"]), o)
    toc = g["compress_toc"]
    for i, o in enumerate(RG.compress_cases()):
        assert np.array_equal(B.oracle_compress(o), g["compress_bytes"][int(toc[i]):int(toc[i + 1])])
        assert np.array_equal(B.oracle_decompress(B.oracle_compress(o)), o)


def _brute_score(a, b, match, mismatch, gap, band=None):
    nx, ny = len(a), len(b)
    NEG = -10**9
    H = np.full((nx + 1, ny + 1), NEG, np.int64)
    best = NEG
    for i in range(nx + 1):
        for j in range(ny + 1):
            if band is not None and not (band[0] <= i - j <= band[1]):
                continue
            if i == 0 or j == 0:
                H[i, j] = 0
            else:
                H[i, j] = max(H[i - 1, j - 1] + (match if a[i - 1] == b[j - 1] else mismatch), H[i, j - 1] + gap, H[i - 1, j] + gap)
            if j == ny or i == nx:
                best = max(best, H[i, j])
    return best


def test_overlap_dp_optimal_score_and_valid_path():
    rng = np.random.default_rng(7)
    for trial in range(60):
        nx, ny = int(rng.integers(1, 40)), int(rng.integers(1, 40))
        a = rng.integers(0, 4, nx).astype(np.uint32)
        b = rng.integers(0, 4, ny).astype(np.uint32)
        band = None
        if trial % 2:
            lo = int(rng.integers(-ny - 3, nx + 3))
            band = (lo, lo + int(rng.integers(0, 25)))
        s, path = B.overlap_align(a, b, 6, -1, -1, band)
        if band is not None and (band[1] < -ny or band[0] > nx):
            assert s is None
            continue
        assert s == _brute_score(a, b, 6, -1, -1, band)
        if len(path):
            assert (np.diff(path[:, 0].astype(int)) > 0).all() and (np.diff(path[:, 1].astype(int)) > 0).all()
            if band is not None:
                d = path[:, 0].astype(int) - path[:, 1].astype(int)
                assert (d >= band[0]).all() and (d <= band[1]).all()


def _pairs(d, cand, limit):
    toc = d["toc"].astype(np.int64)
    km = d["kmer"]
    for r0, r1, same in cand[:limit].tolist():
        o0, o1 = 2 * r0, 2 * r1 + (0 if same else 1)
        yield km[toc[o0]:toc[o0 + 1]], km[toc[o1]:toc[o1 + 1]]


def test_align4_front_end_matches_compiled_reference(golden_dir):
    # Align4 ordinals, AlignmentInfo words and compress bytes of the compiled reference on the same pairs
    # (tests/golden/make_ref_golden.py)
    g = np.load(os.path.join(golden_dir, "ref_golden.npz"))
    pairs = RG.align4_pairs()
    for j, opts in enumerate(RG.ALIGN4_OPTIONS):
        o4 = B.make_align_options(alignMethod=4, k=10, **opts)
        ctoc = g[f"align4_{j}_comp_toc"]
        nonempty = 0
        for p, (a, b) in enumerate(pairs):
            st, al, tie = B.oracle_align_pair(a, b, o4)
            rbytes = g[f"align4_{j}_comp"][int(ctoc[p]):int(ctoc[p + 1])]
            ra = B.oracle_decompress(rbytes)        # the reference's ordinals, stored in its compressed form
            if not tie:     # ties between kept components: the reference's pick depends on unordered_map order
                assert np.array_equal(al, ra)
            if len(al):
                nonempty += 1
            if len(ra):
                assert np.array_equal(B.oracle_alignment_info(ra, len(a), len(b)), g[f"align4_{j}_info"][p])
                assert np.array_equal(B.oracle_compress(ra), rbytes)
        assert nonempty > 10


def test_method3_and_method4_agree_on_clean_overlaps():
    # Both methods end in the same banded DP; on low-noise overlaps they should produce nearly the same alignment.
    d = synth.generate(synth.SynthParams(reads=100, k=10, genome_markers=6000, n50_bases=9000, min_bases=5000, seed=8, drop=0.03, ins=0.01))
    lp = B.LowHashParams(m=4, hashFraction=0.02, minHashIterationCount=6, minBucketSize=2, maxBucketSize=30, minFrequency=2)
    cand, _, _ = B.oracle_lowhash0(d["toc"], d["data"], d["flags"], lp)
    common = dict(k=10, maxSkip=100, maxDrift=100, maxTrim=100, minAlignedMarkerCount=10, minAlignedFraction=0.1)
    same = 0
    total = 0
    for a, b in _pairs(d, cand, 40):
        _, a3, _ = B.oracle_align_pair(a, b, B.make_align_options(alignMethod=3, downsamplingFactor=0.2, **common))
        _, a4, _ = B.oracle_align_pair(a, b, B.make_align_options(alignMethod=4, **common))
        if len(a3) and len(a4):
            total += 1
            same += abs(len(a3) - len(a4)) <= max(3, len(a3) // 20)
    assert total > 10 and same >= 0.8 * total


def test_compute_alignments_driver_consistency():
    # orc_compute_alignments (threaded) == per-pair calls + filters; records are in candidate order.
    d = synth.generate(synth.SynthParams(reads=80, k=10, genome_markers=5000, n50_bases=9000, min_bases=5000, seed=12))
    lp = B.LowHashParams(m=4, hashFraction=0.02, minHashIterationCount=6, minBucketSize=2, maxBucketSize=30, minFrequency=2)
    cand, _, _ = B.oracle_lowhash0(d["toc"], d["data"], d["flags"], lp)
    o = B.make_align_options(alignMethod=3, k=10, maxSkip=30, maxDrift=30, maxTrim=30, minAlignedMarkerCount=50, minAlignedFraction=0.3)
    r1, t1, c1, _ = B.oracle_compute_alignments(d["toc"], d["kmer"], cand[:120], o, threads=1)
    r4, t4, c4, _ = B.oracle_compute_alignments(d["toc"], d["kmer"], cand[:120], o, threads=4)
    assert np.array_equal(r1, r4) and np.array_equal(t1, t4) and np.array_equal(c1, c4)
    assert len(r1) > 10
    key = r1[:, 0].astype(np.int64) * (1 << 32) + r1[:, 1].astype(np.int64) * 2 + (1 - r1[:, 2].astype(np.int64))
    assert (np.diff(key) > 0).all()
    for i in range(len(r1)):
        ords = B.oracle_decompress(c1[int(t1[i]):int(t1[i + 1])])
        assert len(ords) == r1[i, 9] >= 50


def test_alignment_golden_fixtures():
    """The oracle against tests/golden/align_golden.npz: outputs of the reference's own Align4 / AlignmentInfo / compress code
    (generated by tests/golden/make_align_golden.py in the build container); needs no reference build at test time."""
    import importlib.util
    import os
    here = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
    spec = importlib.util.spec_from_file_location("make_align_golden", os.path.join(here, "make_align_golden.py"))
    MG = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(MG)
    z = np.load(os.path.join(here, "align_golden.npz"))
    for name, (synth_spec, count, opts) in MG.ALIGN_CASES.items():
        o4 = B.make_align_options(**opts)
        pairs = MG.case_pairs(synth_spec, count)
        used = z[name + "_pairs"].tolist()
        atoc, ctoc = z[name + "_align4_toc"], z[name + "_comp_toc"]
        assert len(used) >= 0.8 * count
        nonempty = 0
        for slot, p in enumerate(used):
            a, b = pairs[p]
            gold = z[name + "_align4"][int(atoc[slot]):int(atoc[slot + 1])]
            _, al, tie = B.oracle_align_pair(a, b, o4)
            assert not tie
            assert np.array_equal(al.reshape(-1, 2), gold), (name, p)
            if len(gold):
                nonempty += 1
                assert np.array_equal(B.oracle_alignment_info(gold, len(a), len(b)), z[name + "_info"][slot])
                gbytes = z[name + "_comp"][int(ctoc[slot]):int(ctoc[slot + 1])]
                assert np.array_equal(B.oracle_compress(gold), gbytes)
                assert np.array_equal(B.oracle_decompress(gbytes), gold)
        assert nonempty >= 0.8 * len(used)
