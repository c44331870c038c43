"""createReadGraph (ReadGraph.creationMethod 0) oracle against a direct statement of src/AssemblerReadGraph.cpp:35-175:
per read, the maxAlignmentCount largest (markerCount, alignmentId) pairs; edges and connectivity in the reference's order."""
import os
import sys

import numpy as np

from oracle import bindings as B

sys.path.insert(0, os.path.join(os.path.dirname(__file__), "golden"))
import make_ref_golden as RG  # noqa: E402

_records = RG.records


def _direct(rec, reads, k):
    n = len(rec)
    keep = np.zeros(n, np.uint8)
    for r in range(reads):
        ids = [a for a in range(n) if rec[a, 0] == r or rec[a, 1] == r]
        best = sorted(((int(rec[a, 9]), a) for a in ids), reverse=True)[:k]
        for _, a in best:
            keep[a] = 1
    edges = []
    for a in range(n):
        if keep[a]:
            o0, o1 = 2 * int(rec[a, 0]), 2 * int(rec[a, 1]) + (0 if rec[a, 2] else 1)
            edges.append((o0, o1, a, 0))
            edges.append((o0 ^ 1, o1 ^ 1, a, 0))
    conn = [[] for _ in range(2 * reads)]
    for i, e in enumerate(edges):
        conn[e[0]].append(i)
        conn[e[1]].append(i)
    toc = np.zeros(2 * reads + 1, np.uint32)
    toc[1:] = np.cumsum([len(c) for c in conn])
    data = np.array([i for c in conn for i in c], np.uint32)
    return keep, np.array(edges, np.uint32).reshape(-1, 4), toc, data


def test_against_direct_statement():
    rng = np.random.default_rng(3)
    for n, reads, k in [(0, 5, 3), (1, 4, 6), (60, 12, 3), (300, 25, 6), (300, 25, 1), (200, 10, 0), (150, 8, 1000)]:
        rec = _records(rng, n, reads)
        out, keep, edges, toc, data = B.oracle_create_read_graph(rec, reads, k)
        dkeep, dedges, dtoc, ddata = _direct(rec, reads, k)
        assert np.array_equal(keep, dkeep), (n, reads, k)
        assert np.array_equal(edges, dedges) and np.array_equal(toc, dtoc) and np.array_equal(data, ddata)
        assert np.array_equal(out[:, 15] & 1, keep) and np.array_equal(out[:, :15], rec[:, :15])
        # an edge joins (r0, 0) with (r1, 0 / 1) and is ordered (src/AssemblerReadGraph.cpp:129,137)
        assert np.all(edges[:, 0] < edges[:, 1]) if len(edges) else True


_quality_records = RG.quality_records


def test_histogram2_and_indicators_against_the_reference_classes(golden_dir):
    # Thresholds of the reference's Histogram2 and its AlignmentInfo accessors (tests/golden/make_ref_golden.py)
    g = np.load(os.path.join(golden_dir, "ref_golden.npz"))
    cases, rng = RG.hist2_cases()
    for i, (start, stop, bins, x) in enumerate(cases):
        for fraction, want in zip(RG.HIST2_FRACTIONS, g["hist2_thresholds"][i]):
            got = B.oracle_histogram2_threshold(x, start, stop, bins, fraction)
            assert want == got or (np.isnan(want) and np.isnan(got)), (start, stop, bins, i, fraction)
    rec = _quality_records(rng, 200, 30)
    for r, want in zip(rec, g["hist2_indicators"]):
        d0, d1 = r[3:6].astype(np.int64), r[6:9].astype(np.int64)
        frac = min(r[9] / (d0[2] + 1 - d0[1]), r[9] / (d1[2] + 1 - d1[1]))
        trim = max(min(d0[1], d1[1]), min(d0[0] - 1 - d0[2], d1[0] - 1 - d1[2]))
        assert np.array_equal(want, np.array([frac, r[9], r[14], r[13], trim], np.float64))


def test_creation_method_2_against_direct_statement():
    rng = np.random.default_rng(8)
    pc = (0.015, 0.12, 0.12, 0.12, 0.015)      # ReadGraph.*Percentile defaults (src/AssemblerOptions.cpp)
    for n, reads, k in [(0, 4, 6), (400, 30, 6), (3000, 120, 6), (3000, 120, 2)]:
        rec = _quality_records(rng, n, reads)
        crit, out, keep, edges, toc, data = B.oracle_create_read_graph2(rec, reads, k, pc)
        ok = np.zeros(n, bool)
        for a in range(n):
            r = rec[a]
            d0, d1 = r[3:6].astype(np.int64), r[6:9].astype(np.int64)
            frac = min(r[9] / (d0[2] + 1 - d0[1]), r[9] / (d1[2] + 1 - d1[1]))
            trim = max(min(d0[1], d1[1]), min(d0[0] - 1 - d0[2], d1[0] - 1 - d1[2]))
            ok[a] = not (frac < crit["minAlignedFraction"] or r[9] < crit["minAlignedMarkerCount"] or r[14] > crit["maxDrift"]
                         or r[13] > crit["maxSkip"] or trim > crit["maxTrim"])
        if n:
            assert 0 < ok.sum() < n
        # the selection of method 0 restricted to the alignments that pass: compare through the sub-table
        sub = rec[ok]
        _, skeep, _, _, _ = B.oracle_create_read_graph(sub, reads, k)
        want = np.zeros(n, np.uint8)
        want[np.flatnonzero(ok)[skeep.astype(bool)]] = 1
        assert np.array_equal(keep, want)
        dkeep, dedges, dtoc, ddata = _direct(rec[:, :], reads, 0)      # edges / connectivity from the keep flags
        kept = np.flatnonzero(keep)
        assert np.array_equal(edges[0::2, 2], kept) and np.array_equal(edges[1::2, 2], kept)
        assert np.array_equal(out[:, 15] & 1, keep)
