"""The `shasta.Assembler`-shaped facade (shasta_b200/assembler.py) and the reference's Data/ file formats.

CPU part: files written by the facade's writer are byte for byte the files the reference's own MemoryMapped::Vector code
accepted with the right record types, and files written by the reference (Markers, ReadFlags, Kmers from TinyTest through
ReadLoader + MarkerFinder) are read back by the facade's reader. What the reference did is stored in tests/golden/ref_golden.npz
(tests/golden/make_ref_golden.py).
GPU part: the two entry points run on a Data/ directory with the reference's Python-script call sequence
(scripts/FindAlignmentCandidatesLowHash0.py, scripts/ComputeAlignments.py) and reproduce the TinyTest pin."""
import os
import sys

import numpy as np
import pytest

from oracle import bindings as B
from shasta_b200 import assembler as A

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
import make_ref_golden as RG  # noqa: E402


def test_writer_is_readable_by_the_reference(tmp_path, golden_dir):
    g = np.load(os.path.join(golden_dir, "ref_golden.npz"))
    for i, (size, arr) in enumerate(RG.writer_cases()):
        path = str(tmp_path / f"v{i}")
        A.mm_write_vector(path, arr, object_size=size)
        # the reference opened exactly these bytes as a Vector of `size`-byte records, with this count and payload checksum
        assert np.array_equal(RG.sha256(open(path, "rb").read()), g["writer_sha256"][i])
        assert g["writer_count"][i] == arr.nbytes // size
        assert g["writer_checksum"][i] == RG.fnv(arr.tobytes())
        back = A.mm_read_vector(path, arr.dtype, object_size=size)
        assert np.array_equal(np.asarray(back).reshape(arr.shape), arr)
    # a wrong record size is rejected, as the reference's accessExistingReadOnly rejected v0 opened as 64-byte records
    with pytest.raises(RuntimeError, match="object size"):
        A.mm_read_vector(str(tmp_path / "v0"), np.uint8, object_size=64)


@pytest.fixture(scope="module")
def tiny_data_dir(tmp_path_factory):
    """The Data/ files the reference writes for TinyTest, rebuilt from their stored headers and the golden markers. The payload
    of Kmers is not stored: the reader needs only its header and size."""
    g = np.load(os.path.join(os.path.dirname(__file__), "golden", "ref_golden.npz"))
    z = np.load(os.path.join(os.path.dirname(__file__), "golden", "tinytest_markers.npz"))
    d = tmp_path_factory.mktemp("run") / "Data"
    os.makedirs(d)
    payloads = {"Markers.toc": z["toc"], "Markers.data": z["data"], "ReadFlags": z["flags"], "Kmers": np.zeros(0, np.uint8)}
    for name, payload in payloads.items():
        key = name.replace(".", "_")
        header = g[f"datadir_{key}_header"]
        raw = header.tobytes() + bytes(4096 - header.nbytes) + payload.tobytes()
        raw += bytes(int(header[5]) - len(raw))         # header word 5: fileSize
        if name != "Kmers":
            assert np.array_equal(RG.sha256(raw), g[f"datadir_{key}_sha256"]), name
        with open(d / name, "wb") as f:
            f.write(raw)
    return str(d) + "/"


def test_reader_on_reference_written_files(tiny_data_dir, golden_dir):
    a = A.Assembler(largeDataFileNamePrefix=tiny_data_dir)
    a.accessKmers()
    assert a.k == 10
    a.accessMarkers()
    toc, data, flags = a._markers
    z = np.load(os.path.join(golden_dir, "tinytest_markers.npz"))
    assert np.array_equal(toc, z["toc"]) and np.array_equal(data, z["data"]) and np.array_equal(flags, z["flags"])
    with pytest.raises(RuntimeError, match="not accessible"):
        A.Assembler(largeDataFileNamePrefix=tiny_data_dir).checkMarkersAreOpen()


def test_companion_accessors_with_stubbed_device(tmp_path, golden_dir, monkeypatch, capsys):
    """computeSortedMarkers / accessSortedMarkers / alignOrientedReads4 (src/PythonModule.cpp:210-214,302-327): host logic only.
    The device call is replaced by a stub that records what the facade asks for."""
    from shasta_b200 import capi
    z = np.load(os.path.join(golden_dir, "tinytest_markers.npz"))
    prefix = str(tmp_path / "Data") + "/"
    os.makedirs(prefix)
    A.mm_write_vector_of_vectors(prefix + "Markers", z["toc"], z["data"], data_object_size=7)
    A.mm_write_vector(prefix + "ReadFlags", z["flags"], object_size=1)
    A.mm_write_vector(prefix + "Kmers", np.zeros((1 << 20) * 24, np.uint8), object_size=24)
    a = A.Assembler(largeDataFileNamePrefix=prefix)
    with pytest.raises(RuntimeError, match="not accessible"):
        a.computeSortedMarkers()
    a.accessKmers()
    a.accessMarkers()
    a.computeSortedMarkers(threadCount=3)
    a.accessSortedMarkers()

    seen = {}

    class StubContext:
        def set_markers(self, toc, data, flags):
            seen["markers"] = len(flags)

    def stub_align_oriented_reads(ctx, o0, o1, opts):
        seen["pair"] = (o0, o1)
        seen["opts"] = opts
        return np.zeros((321, 2), np.uint32), np.zeros(13, np.uint32)

    monkeypatch.setattr(a, "_context", lambda: StubContext())
    a._markers_on_device = False
    monkeypatch.setattr(capi, "align_oriented_reads", stub_align_oriented_reads)
    kw = dict(deltaX=200, deltaY=10, minEntryCountPerCell=10, maxDistanceFromBoundary=100, minAlignedMarkerCount=10,
              minAlignedFraction=0.1, maxSkip=100, maxDrift=100, maxTrim=100, maxBand=1000, matchScore=6, mismatchScore=-1, gapScore=-1)
    n = a.alignOrientedReads4(readId0=7, strand0=1, readId1=3, strand1=0, **kw)
    assert n == 321 and "The alignment has 321 markers." in capsys.readouterr().out
    assert seen["markers"] == 20
    assert seen["pair"] == (15, 6)            # the orientation and order the caller gave: (7,1) horizontal, (3,0) vertical
    o = seen["opts"]
    assert (o.alignMethod, o.k, o.align4DeltaX, o.align4DeltaY, o.align4MinEntryCountPerCell, o.align4MaxDistanceFromBoundary) == (4, 10, 200, 10, 10, 100)
    assert (o.maxSkip, o.maxDrift, o.maxTrim, o.maxBand, o.minAlignedMarkerCount, o.suppressContainments) == (100, 100, 100, 1000, 10, 0)
    a.alignOrientedReads4(readId0=2, strand0=1, readId1=5, strand1=1, **kw)
    assert seen["pair"] == (5, 11)


@pytest.mark.gpu
def test_script_sequence_on_reference_data_dir(tmp_path, golden_dir, monkeypatch):
    monkeypatch.chdir(tmp_path)         # like the reference, the facade leaves ReadLowHashStatistics.csv in the working directory
    # scripts/FindAlignmentCandidatesLowHash0.py + scripts/ComputeAlignments.py call sequence. The Data/ inputs are written
    # with the facade's writer from the golden TinyTest markers (the reference tree is not on the GPU box).
    z = np.load(os.path.join(golden_dir, "tinytest_markers.npz"))
    prefix = str(tmp_path / "Data") + "/"
    os.makedirs(prefix)
    A.mm_write_vector_of_vectors(prefix + "Markers", z["toc"], z["data"], data_object_size=7)
    A.mm_write_vector(prefix + "ReadFlags", z["flags"], object_size=1)
    A.mm_write_vector(prefix + "Kmers", np.zeros((1 << 20) * 24, np.uint8), object_size=24)
    a = A.Assembler(largeDataFileNamePrefix=prefix)
    a.accessKmers()
    a.accessMarkers()
    a.findAlignmentCandidatesLowHash0(m=4, hashFraction=0.01, minHashIterationCount=10, alignmentCandidatesPerRead=20.,
                                      minBucketSize=0, maxBucketSize=10, minFrequency=2, threadCount=0)
    b = A.Assembler(largeDataFileNamePrefix=prefix)
    b.accessKmers()
    b.accessMarkers()
    b.accessAlignmentCandidates()
    cands = b.getAlignmentCandidates()
    assert len(cands) == 186 and cands[0].readIds == [0, 2] and cands[0].isSameStrand is False
    assert B.candidate_digest(b._candidates) == 0x3fc2c96e354f8733
    opts = A.AlignOptions()
    opts.minAlignedMarkerCount = 100
    opts.minAlignedFraction = 0.4
    b.computeAlignments(opts, 0)
    c = A.Assembler(largeDataFileNamePrefix=prefix)
    c.accessAlignmentData()
    c.accessCompressedAlignments()
    rec = c._alignment_data
    toc, data = c._compressed
    assert len(rec) > 20 and len(toc) == len(rec) + 1
    # against the oracle
    kmer = np.ascontiguousarray(np.asarray(z["data"]).reshape(-1, 7)[:, :4]).view("<u4").reshape(-1)
    oo = B.make_align_options(alignMethod=3, k=10, maxSkip=30, maxDrift=30, maxTrim=30, minAlignedMarkerCount=100,
                              minAlignedFraction=0.4, downsamplingFactor=0.1, bandExtend=10, maxBand=1000)
    orec, otoc, odata, _ = B.oracle_compute_alignments(z["toc"], kmer, b._candidates, oo, threads=4)
    assert np.array_equal(rec, orec) and np.array_equal(toc, otoc) and np.array_equal(data, odata)
    table_toc = A.mm_read_vector(prefix + "AlignmentTable.toc", np.uint32, object_size=4)
    assert len(table_toc) == 2 * 20 + 1 and int(table_toc[-1]) == 4 * len(rec)
    # srcMain/main.cpp:717-741 (ReadGraph.creationMethod 0): createReadGraph continues from the alignments
    kept = b.createReadGraph(maxAlignmentCount=3, maxTrim=30)
    wrec, wkeep, wedges, wtoc, wdata = B.oracle_create_read_graph(rec, 20, 3)
    assert kept == int(wkeep.sum()) and 0 < kept < len(rec)
    e = A.Assembler(largeDataFileNamePrefix=prefix)
    e.accessAlignmentData()
    assert np.array_equal(e._alignment_data, wrec)
    edges = np.asarray(A.mm_read_vector(prefix + "ReadGraphEdges", np.uint32, object_size=16)).reshape(-1, 4)
    ctoc = np.asarray(A.mm_read_vector(prefix + "ReadGraphConnectivity.toc", np.uint32, object_size=4))
    cdata = np.asarray(A.mm_read_vector(prefix + "ReadGraphConnectivity.data", np.uint32, object_size=4))
    assert np.array_equal(edges, wedges) and np.array_equal(ctoc, wtoc) and np.array_equal(cdata, wdata)
    # ... and ReadGraph.creationMethod 2 (srcMain/main.cpp:731-739), the one the May2022 configurations select
    f = A.Assembler(largeDataFileNamePrefix=prefix)
    f.accessMarkers()
    f.accessAlignmentData()
    kept2 = f.createReadGraph2(3, 0.015, 0.12, 0.12, 0.12, 0.015)
    crit2, wrec2, wkeep2, wedges2, wtoc2, wdata2 = B.oracle_create_read_graph2(rec, 20, 3, (0.015, 0.12, 0.12, 0.12, 0.015))
    assert kept2 == int(wkeep2.sum()) and f.readGraph2Criteria == crit2
    edges2 = np.asarray(A.mm_read_vector(prefix + "ReadGraphEdges", np.uint32, object_size=16)).reshape(-1, 4)
    assert np.array_equal(edges2, wedges2)
    # srcMain/main.cpp:706: computeCandidateTable after the candidates are known
    b.computeCandidateTable()
    ct_toc = np.asarray(A.mm_read_vector(prefix + "CandidateTable.toc", np.uint64, object_size=8))
    ct_data = np.asarray(A.mm_read_vector(prefix + "CandidateTable.data", np.uint64, object_size=8))
    otoc2, otable2 = B.oracle_compute_candidate_table(b._candidates, 20)
    assert np.array_equal(ct_toc, otoc2) and np.array_equal(ct_data, otable2)
    # single pair, in the orientation given (scripts/AlignOrientedReads4.py): against the oracle's Align4 on the same rows
    toc0 = np.asarray(z["toc"])
    r0, r1, same = [int(x) for x in b._candidates[0]]
    for (s0, s1) in ((0, 0 if same else 1), (1, 1 if same else 0)):
        for (ra, sa, rb, sb) in ((r0, s0, r1, s1), (r1, s1, r0, s0)):
            n4 = b.alignOrientedReads4(ra, sa, rb, sb, deltaX=200, deltaY=10, minEntryCountPerCell=10, maxDistanceFromBoundary=100,
                                       minAlignedMarkerCount=10, minAlignedFraction=0.1, maxSkip=100, maxDrift=100, maxTrim=100,
                                       maxBand=1000, matchScore=6, mismatchScore=-1, gapScore=-1)
            oa, ob = 2 * ra + sa, 2 * rb + sb
            o4 = B.make_align_options(alignMethod=4, k=10, maxSkip=100, maxDrift=100, maxTrim=100, minAlignedMarkerCount=10,
                                      minAlignedFraction=0.1, maxBand=1000)
            _, want, _ = B.oracle_align_pair(kmer[int(toc0[oa]):int(toc0[oa + 1])], kmer[int(toc0[ob]):int(toc0[ob + 1])], o4)
            assert n4 == len(want) and np.array_equal(b._last_alignment, want)
    with pytest.raises(RuntimeError, match="unreasonably small"):
        b.findAlignmentCandidatesLowHash0(m=4, hashFraction=0.01, minHashIterationCount=10, alignmentCandidatesPerRead=20.,
                                          minBucketSize=0, maxBucketSize=10, minFrequency=2, log2MinHashBucketCount=3)
