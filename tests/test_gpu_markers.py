"""GPU parity test of the device MarkerFinder (csrc/markers.cu, shb_find_markers) through the C ABI:
  * TinyTest: inputs and expected output both produced by the UNMODIFIED reference (tests/golden/tinytest_reads.npz ->
    tests/golden/tinytest_markers.npz, 124 036 markers), 7-byte records and toc bit for bit;
  * synthetic FASTA files run through the reference's own ReadLoader + MarkerFinder (tests/golden/ref_golden.npz);
  * edge cases: reads shorter than k, empty reads, one read, k-mers straddling 64-base blocks at every offset;
  * the markers left on the device feed LowHash0 directly (no shb_set_markers): same candidates as from the uploaded records."""
import os
import sys

import numpy as np
import pytest

from oracle import bindings as B

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "golden"))
import make_ref_golden as RG  # noqa: E402


@pytest.fixture(scope="module")
def ctx():
    from shasta_b200 import capi
    c = capi.Context(0)
    yield c
    c.close()


def _golden():
    r = np.load(os.path.join(ROOT, "tests", "golden", "tinytest_reads.npz"))
    m = np.load(os.path.join(ROOT, "tests", "golden", "tinytest_markers.npz"))
    return r, m


def test_tinytest_markers_bit_for_bit(ctx):
    from shasta_b200 import capi
    r, m = _golden()
    toc, data, res = ctx.find_markers(10, r["word_offsets"], r["words"], r["base_counts"], m["flags"], is_marker_bitmap=r["is_marker_bitmap"])
    assert res.markerCount == 124036 and res.readCount == 20
    assert np.array_equal(toc, m["toc"]) and np.array_equal(data, m["data"])
    # the same through a KmerInfo table (24-byte records, isMarker at byte 12) instead of the bitmap
    is_marker = np.unpackbits(r["is_marker_bitmap"].view(np.uint8), bitorder="little")
    table = np.zeros((4 ** 10, 24), np.uint8)
    table[:, 12] = is_marker
    toc2, data2, _ = ctx.find_markers(10, r["word_offsets"], r["words"], r["base_counts"], m["flags"], kmer_table=table)
    assert np.array_equal(toc2, m["toc"]) and np.array_equal(data2, m["data"])
    # the markers are resident: LowHash0 without any upload gives the TinyTest pin (186 candidates, digest 0x3fc2c96e354f8733)
    _, _, res3 = ctx.find_markers(10, r["word_offsets"], r["words"], r["base_counts"], m["flags"], is_marker_bitmap=r["is_marker_bitmap"],
                                  want_host=False)
    cand, _, _, _ = ctx.lowhash0(capi.make_lowhash_params(m=4, hashFraction=0.01, minHashIterationCount=10, minBucketSize=0,
                                                           maxBucketSize=10, minFrequency=2))
    assert len(cand) == 186 and B.candidate_digest(cand) == 0x3fc2c96e354f8733


@pytest.mark.parametrize("k", [6, 10, 14])
def test_synthetic_fasta_against_live_reference(ctx, k):
    g = np.load(os.path.join(ROOT, "tests", "golden", "ref_golden.npz"))
    name = f"fasta60_s{k}_k{k}"
    r = RG.fasta_case(g, name)
    bitmap = np.packbits(r["is_marker"], bitorder="little").view(np.uint32)
    toc, data, res = ctx.find_markers(k, r["word_offsets"], r["words"], r["base_counts"], r["flags"], is_marker_bitmap=bitmap)
    assert res.markerCount == int(g[f"fasta_{name}_toc"][-1]) > 1000
    RG.assert_markers_match(g, name, toc, data)


def _pack_reads(reads):
    """LongBaseSequences layout (src/LongBaseSequence.hpp:33-41) of a list of base arrays (values 0..3)."""
    offsets, words, counts = [0], [], []
    for b in reads:
        n = len(b)
        counts.append(n)
        blocks = (n + 63) // 64
        for blk in range(blocks):
            lo = hi = 0
            for j, v in enumerate(b[64 * blk: 64 * blk + 64]):
                lo |= (int(v) & 1) << (63 - j)
                hi |= (int(v) >> 1) << (63 - j)
            words += [lo, hi]
        offsets.append(len(words))
    return np.array(offsets, np.uint64), np.array(words, np.uint64), np.array(counts, np.uint64)


def test_edge_cases_against_oracle(ctx):
    rng = np.random.default_rng(5)
    k = 7
    is_marker = (rng.random(4 ** k) < 0.3).astype(np.uint8)
    lengths = [0, 3, 6, 7, 8, 63, 64, 65, 70, 127, 128, 129, 1000, 0, 5, 200]
    reads = [rng.integers(0, 4, n) for n in lengths]
    wo, w, bc = _pack_reads(reads)
    flags = np.zeros(len(reads), np.uint8)
    otoc, odata = B.oracle_find_markers(wo, w, bc, is_marker, k)
    bitmap = np.packbits(is_marker, bitorder="little").view(np.uint32)
    toc, data, res = ctx.find_markers(k, wo, w, bc, flags, is_marker_bitmap=bitmap)
    assert np.array_equal(toc, otoc) and np.array_equal(data, odata)
    assert toc[2] == toc[0] and toc[4] == toc[2]        # reads shorter than k have no markers
    # no reads at all
    toc0, data0, res0 = ctx.find_markers(k, np.zeros(1, np.uint64), np.zeros(0, np.uint64), np.zeros(0, np.uint64), np.zeros(0, np.uint8),
                                         is_marker_bitmap=bitmap)
    assert toc0.tolist() == [0] and len(data0) == 0 and res0.markerCount == 0
