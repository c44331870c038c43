"""Generates ref_golden.npz: what the UNMODIFIED reference build (oracle/_ref/libshasta_ref.so) returns on the inputs of the
tests that compare the oracle, the facade and the device path with it, so that those tests run without the reference tree.

Build oracle/_ref first (`make -C oracle ref SHASTA_REF_SRC=<reference>/src`), then:
    python tests/golden/make_ref_golden.py <reference source tree>
(the tree is read only for tests/TinyTest.fasta.gz).

Inputs are regenerated from seeds by the functions below, which the tests call too. The fixture holds, per case:
  writer_*     the reference's accessExistingReadOnly on files written by the facade's mm_write_vector: object count, payload
               checksum and the SHA-256 of the exact file it accepted; and that it rejects the first file as 64-byte records
  datadir_*    header words and SHA-256 of each file the reference writes for TinyTest (Markers.toc/.data, ReadFlags, Kmers);
               the payloads of the first three are tinytest_markers.npz, that of Kmers (25 MB) is not stored
  selftest_*   the ordinals of the reference's testAlignmentCompression and the reference's shasta::compress bytes for them
  compress_*   shasta::compress bytes for the seeded ordinal runs of compress_cases()
  align4_*     AlignmentInfo words and compress bytes of the Align4 ordinals for the pairs of align4_pairs() (the ordinals
               themselves are stored in that compressed form)
  lowhash_*    LowHash0 candidates, per-read statistics and per-iteration summary for LOWHASH_RANDOM_PARAMS
  fasta_*      ReadLoader (RLE) + MarkerFinder on the seeded FASTA files of FASTA_CASES: SHA-256 of the RLE reads (which
               rle_reads() regenerates), read flags, the isMarker bit of every k-mer of the reads (read_kmers() order), and the
               markers (toc, SHA-256 of the 7-byte records)
  hist2_*      Histogram2 thresholds for hist2_cases(), and the AlignmentInfo indicators of quality_records()
  csv_*        per-read statistics and ReadLowHashStatistics.csv as LowHash0 leaves it, for CSV_CASES
"""
import gzip
import hashlib
import os
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
from oracle import bindings as B  # noqa: E402
from shasta_b200 import assembler as A  # noqa: E402
from shasta_b200 import synth  # noqa: E402

GOLDEN = os.path.join(HERE, "ref_golden.npz")


def sha256(raw):
    return np.frombuffer(hashlib.sha256(bytes(raw)).digest(), np.uint8)


def fnv(raw):
    h = 1469598103934665603
    for b in bytes(raw):
        h = ((h ^ b) * 1099511628211) & 0xFFFFFFFFFFFFFFFF
    return h


def writer_cases():
    """(record size, array) pairs written with the facade's mm_write_vector."""
    rng = np.random.default_rng(1)
    return [(12, rng.integers(0, 1000, (1000, 3)).astype(np.uint32)), (64, rng.integers(0, 2**31, (77, 16)).astype(np.uint32)),
            (24, rng.integers(0, 2**40, (50, 3)).astype(np.uint64)), (1, rng.integers(0, 255, 5000).astype(np.uint8)),
            (8, rng.integers(0, 2**50, 4097).astype(np.uint64)), (4, np.zeros(0, np.uint32))]


DATADIR_FILES = ("Markers.toc", "Markers.data", "ReadFlags", "Kmers")


def compress_cases():
    """Ordinal runs with streaks and skips spanning all five formats of shasta::compress, and a Format 4 run with a negative skip."""
    rng = np.random.default_rng(1)
    out = []
    for trial in range(200):
        n = int(rng.integers(1, 60))
        scale = [3, 7, 500, 500000, 3000000][trial % 5]
        x = np.cumsum(rng.integers(1, scale + 1, n)).astype(np.uint32)
        y = np.cumsum(rng.integers(1, scale + 1, n)).astype(np.uint32)
        run = rng.integers(0, 2, n).astype(bool)
        for i in range(1, n):
            if run[i]:
                x[i:] -= x[i] - x[i - 1] - 1
                y[i:] -= y[i] - y[i - 1] - 1
        out.append(np.stack([x, y], 1))
    out.append(np.array([[2000000, 5], [2000001, 6], [2000010, 1000000]], np.uint32))
    return out


ALIGN4_OPTIONS = (dict(maxSkip=100, maxDrift=100, maxTrim=100, minAlignedMarkerCount=10, minAlignedFraction=0.1),
                  dict(maxSkip=30, maxDrift=30, maxTrim=30, minAlignedMarkerCount=60, minAlignedFraction=0.4,
                       align4DeltaX=100, align4DeltaY=5, align4MinEntryCountPerCell=4, align4MaxDistanceFromBoundary=50, maxBand=300))


def align4_pairs(limit=60):
    """Marker k-mer id sequences of the first oracle LowHash0 candidates on a seeded synthetic read set."""
    d = synth.generate(synth.SynthParams(reads=150, k=10, genome_markers=9000, n50_bases=9000, min_bases=5000, seed=5))
    lp = B.LowHashParams(m=4, hashFraction=0.02, minHashIterationCount=6, minBucketSize=2, maxBucketSize=30, minFrequency=2)
    cand, _, _ = B.oracle_lowhash0(d["toc"], d["data"], d["flags"], lp)
    toc = d["toc"].astype(np.int64)
    km = d["kmer"]
    pairs = []
    for r0, r1, same in cand[:limit].tolist():
        o0, o1 = 2 * r0, 2 * r1 + (0 if same else 1)
        pairs.append((km[toc[o0]:toc[o0 + 1]], km[toc[o1]:toc[o1 + 1]]))
    return pairs


LOWHASH_RANDOM_PARAMS = (dict(m=2, hashFraction=0.03, minHashIterationCount=3, minBucketSize=0, maxBucketSize=5, minFrequency=1),
                         dict(m=7, hashFraction=0.1, minHashIterationCount=2, minBucketSize=3, maxBucketSize=40, minFrequency=2))


def lowhash_random_input():
    return synth.generate(synth.SynthParams(reads=150, k=10, genome_markers=20000, n50_bases=12000, min_bases=6000, seed=99))


def synthetic_reads(reads, seed):
    """Bases (0..3 = ACGT) of the seeded synthetic reads."""
    rng = np.random.default_rng(seed)
    out = []
    for _ in range(reads):
        n = int(rng.integers(10000, 14000))
        # homopolymer runs of random length so that the run-length encoding has something to do
        out.append(np.repeat(rng.integers(0, 4, n), rng.integers(1, 4, n))[:n])
    return out


def write_synthetic_fasta(path, reads, seed):
    with open(path, "w") as f:
        for i, bases in enumerate(synthetic_reads(reads, seed)):
            f.write(f">read{i}\n" + "".join("ACGT"[b] for b in bases) + "\n")


def rle_reads(reads):
    """The run-length representation of reads in LongBaseSequences layout (src/LongBaseSequence.hpp: per 64-base block a word
    of the low base bits, then a word of the high base bits, first base in bit 63): (word_offsets, words, base_counts)."""
    offsets, words, counts = [0], [], []
    weights = np.uint64(1) << np.arange(63, -1, -1, dtype=np.uint64)
    for b in reads:
        b = b[np.concatenate([[True], b[1:] != b[:-1]])].astype(np.uint64)
        n = len(b)
        blocks = np.zeros(-(-n // 64) * 64, np.uint64)
        blocks[:n] = b
        blocks = blocks.reshape(-1, 64)
        w = np.stack([((blocks & np.uint64(1)) * weights).sum(1, dtype=np.uint64), ((blocks >> np.uint64(1)) * weights).sum(1, dtype=np.uint64)], 1)
        words.append(w.reshape(-1))
        counts.append(n)
        offsets.append(offsets[-1] + w.size)
    return np.array(offsets, np.uint64), np.concatenate(words), np.array(counts, np.uint64)


# name -> (reads, seed, k); min_read_length 1000, marker probability 0.1, seed 231
FASTA_CASES = {"fasta40_s3_k8": (40, 3, 8), "fasta40_s3_k10": (40, 3, 10),
               "fasta60_s6_k6": (60, 6, 6), "fasta60_s10_k10": (60, 10, 10), "fasta60_s14_k14": (60, 14, 14)}


def fasta_case(z, name):
    """The MarkerFinder inputs of a FASTA case as the reference loads them: dict(word_offsets, words, base_counts, flags,
    is_marker uint8[4^k], k). The reads are regenerated and checked against the reference's; is_marker is the reference's
    k-mer table on every k-mer of the reads and their reverse complements, and 0 elsewhere."""
    reads, seed, k = FASTA_CASES[name]
    wo, w, bc = rle_reads(synthetic_reads(reads, seed))
    assert np.array_equal(sha256(wo.tobytes() + w.tobytes() + bc.tobytes()), z[f"fasta_{name}_reads_sha256"]), name
    present = read_kmers(wo, w, bc, k)
    is_marker = np.zeros(4 ** k, np.uint8)
    is_marker[present] = np.unpackbits(z[f"fasta_{name}_marker_bits"], count=len(present))
    return dict(word_offsets=wo, words=w, base_counts=bc, flags=z[f"fasta_{name}_flags"], is_marker=is_marker, k=k)


def assert_markers_match(z, name, toc, data):
    """toc / data (7-byte records) against the reference's markers of a FASTA case."""
    assert np.array_equal(toc, z[f"fasta_{name}_toc"]), name
    assert len(data) == 7 * int(toc[-1]) and np.array_equal(sha256(data), z[f"fasta_{name}_data_sha256"]), name


def read_kmers(word_offsets, words, base_counts, k):
    """Every k-mer id of the RLE reads in LongBaseSequences layout, and of their reverse complements. A k-mer id is the k high
    bits of its bases followed by their k low bits, first base most significant in each (src/ShortBaseSequence.hpp)."""
    out = []
    j = np.arange(64, dtype=np.uint64)
    for r in range(len(base_counts)):
        w = words[int(word_offsets[r]):int(word_offsets[r + 1])].reshape(-1, 2)
        n = int(base_counts[r])
        if n < k:
            continue
        lo_bits, hi_bits = (((w[:, p][:, None] >> (np.uint64(63) - j)) & np.uint64(1)).reshape(-1)[:n] for p in (0, 1))
        lo = np.zeros(n - k + 1, np.uint64)
        hi = np.zeros(n - k + 1, np.uint64)
        for i in range(k):
            lo = (lo << np.uint64(1)) | lo_bits[i:n - k + 1 + i]
            hi = (hi << np.uint64(1)) | hi_bits[i:n - k + 1 + i]
        out.append((hi << np.uint64(k)) | lo)
    ids = np.unique(np.concatenate(out)).astype(np.uint32)
    return np.union1d(ids, synth.reverse_complement_kmer(ids, k).astype(np.uint32))


HIST2_RANGES = ((0, 1, 100), (0, 3000, 300), (0, 100, 100))
HIST2_FRACTIONS = (0.015, 0.12, 0.5, 0.88, 0.985, 1.0)


def hist2_cases():
    """(start, stop, binCount, values) for the Histogram2 comparison: in range, on the upper edge and beyond it."""
    rng = np.random.default_rng(5)
    out = []
    for (start, stop, bins) in HIST2_RANGES:
        for trial in range(20):
            n = int(rng.integers(0, 400))
            x = rng.uniform(start, stop * rng.choice([0.5, 1.0, 1.7]), n)
            if n and trial % 3 == 0:
                x[rng.integers(0, n)] = stop
            x = np.round(x, 2) if stop > 1 else x
            out.append((start, stop, bins, x))
    return out, rng


def records(rng, n, reads):
    """AlignmentData records: read pair, strand, markerCount and a stale isInReadGraph flag."""
    rec = np.zeros((n, 16), np.uint32)
    a = rng.integers(0, reads, n)
    b = rng.integers(0, reads, n)
    same = a == b
    b[same] = (a[same] + 1) % reads
    rec[:, 0] = np.minimum(a, b)
    rec[:, 1] = np.maximum(a, b)
    rec[:, 2] = rng.integers(0, 2, n)
    rec[:, 9] = rng.integers(10, 14, n)         # few distinct marker counts: ties are decided by the alignment id
    rec[:, 15] = rng.integers(0, 2, n)          # stale flags must be overwritten
    return rec


def quality_records(rng, n, reads):
    """AlignmentData with plausible AlignmentInfo words: Data{markerCount, firstOrdinal, lastOrdinal} x 2, markerCount, offsets,
    maxSkip, maxDrift."""
    rec = records(rng, n, reads)
    for side in (0, 1):
        total = rng.integers(200, 5000, n)
        first = rng.integers(0, 150, n)
        last = total - 1 - rng.integers(0, 150, n)
        rec[:, 3 + 3 * side] = total
        rec[:, 4 + 3 * side] = first
        rec[:, 5 + 3 * side] = np.maximum(last, first)
    span = np.minimum(rec[:, 5] - rec[:, 4], rec[:, 8] - rec[:, 7]) + 1
    rec[:, 9] = np.maximum(1, (span * rng.uniform(0.2, 1.0, n)).astype(np.uint32))       # markerCount: up to ~4800 (beyond 3000)
    rec[:, 13] = rng.integers(0, 140, n)        # maxSkip: some beyond the histogram's 100
    rec[:, 14] = rng.integers(0, 120, n)        # maxDrift
    return rec


# (m, minBucketSize, maxBucketSize) on csv_input()
CSV_CASES = ((4, 2, 30), (3, 5, 8))


def csv_input():
    return synth.generate(synth.SynthParams(reads=300, k=10, genome_markers=30000, n50_bases=12000, min_bases=6000, seed=17,
                                            palindromic_every=23))


def csv_params(m, min_bucket, max_bucket):
    return B.LowHashParams(m=m, hashFraction=0.02, minHashIterationCount=6, minBucketSize=min_bucket, maxBucketSize=max_bucket,
                           minFrequency=2)


def _concat(parts, dtype):
    toc = np.zeros(len(parts) + 1, np.uint64)
    toc[1:] = np.cumsum([len(p) for p in parts])
    return toc, np.concatenate(parts).astype(dtype) if parts else np.zeros(0, dtype)


def main(reference_tree):
    assert B.have_ref(), "oracle/_ref/libshasta_ref.so is required"
    out = {}
    with tempfile.TemporaryDirectory() as tmp:
        # the facade's writer, opened by the reference
        counts, sums, shas = [], [], []
        for i, (size, arr) in enumerate(writer_cases()):
            path = os.path.join(tmp, f"v{i}")
            A.mm_write_vector(path, arr, object_size=size)
            n, h = B.ref_open_vector(path, size)
            counts.append(n)
            sums.append(h)
            shas.append(sha256(open(path, "rb").read()))
        try:
            B.ref_open_vector(os.path.join(tmp, "v0"), 64)
            rejected = False
        except RuntimeError:
            rejected = True
        out.update(writer_count=np.array(counts, np.uint64), writer_checksum=np.array(sums, np.uint64), writer_sha256=np.stack(shas),
                   writer_rejects_v0_as_64=np.array(rejected))

        # the Data/ directory the reference writes for TinyTest
        fasta = os.path.join(tmp, "TinyTest.fasta")
        with open(fasta, "wb") as f:
            f.write(gzip.open(os.path.join(reference_tree, "tests", "TinyTest.fasta.gz")).read())
        prefix = os.path.join(tmp, "Data") + "/"
        os.makedirs(prefix)
        B.ref_write_data_dir(fasta, prefix, k=10)
        for name in DATADIR_FILES:
            raw = open(prefix + name, "rb").read()
            key = name.replace(".", "_")
            out[f"datadir_{key}_header"] = np.frombuffer(raw[:64], np.uint64).copy()
            assert not any(raw[64:4096]), name
            out[f"datadir_{key}_sha256"] = sha256(raw)

        # ReadLoader + MarkerFinder on seeded FASTA files
        for name, (reads, seed, k) in FASTA_CASES.items():
            path = os.path.join(tmp, name + ".fasta")
            write_synthetic_fasta(path, reads=reads, seed=seed)
            r = B.ref_reads_from_fasta(path, k=k, min_read_length=1000)
            m = B.ref_markers_from_fasta(path, k=k, min_read_length=1000)
            present = read_kmers(r["word_offsets"], r["words"], r["base_counts"], k)
            out.update({f"fasta_{name}_reads_sha256": sha256(r["word_offsets"].tobytes() + r["words"].tobytes() + r["base_counts"].tobytes()),
                        f"fasta_{name}_flags": m["flags"], f"fasta_{name}_marker_bits": np.packbits(r["is_marker"][present]),
                        f"fasta_{name}_toc": m["toc"], f"fasta_{name}_data_sha256": sha256(m["data"])})
            case = fasta_case(out, name)
            assert np.array_equal(case["words"], r["words"]), name
            toc, data = B.oracle_find_markers(case["word_offsets"], case["words"], case["base_counts"], case["is_marker"], k)
            assert np.array_equal(toc, m["toc"]) and np.array_equal(data, m["data"]), name

        # ReadLowHashStatistics.csv as the reference's LowHash0 leaves it
        d = csv_input()
        for i, case in enumerate(CSV_CASES):
            keep = os.path.join(tmp, f"csv{i}")
            os.makedirs(keep)
            os.environ["SHB_REF_KEEP_CSV"] = keep
            _, stats, _, _ = B.ref_lowhash0(d["toc"], d["data"], d["flags"], csv_params(*case), threads=2)
            del os.environ["SHB_REF_KEEP_CSV"]
            out[f"csv_{i}_stats"] = stats
            out[f"csv_{i}_text"] = np.frombuffer(open(os.path.join(keep, "ReadLowHashStatistics.csv"), "rb").read(), np.uint8)

    # shasta::compress
    lib = B._rlib()
    assert lib.ref_test_alignment_compression() == 0
    selftest = np.array([(300, 200), (301, 201), (302, 202), (305, 206), (306, 207), (320, 250), (321, 251), (322, 252), (323, 253),
                         (325, 255), (326, 256), (350, 257), (351, 258), (352, 259), (353, 260), (354, 261), (1000, 400), (1001, 401),
                         (1002, 402), (600000, 500000), (600001, 500001), (500000, 500005), (500001, 500007), (500002, 500008),
                         (500003, 500009), (500004, 500010), (500005, 500011), (500006, 500012), (500007, 500013), (500008, 500014)],
                        np.uint32)
    out.update(selftest_ordinals=selftest, selftest_compressed=B.ref_compress(selftest))
    out["compress_toc"], out["compress_bytes"] = _concat([B.ref_compress(o) for o in compress_cases()], np.uint8)

    # Align4, AlignmentInfo and compress on the same pairs
    pairs = align4_pairs()
    for j, opts in enumerate(ALIGN4_OPTIONS):
        o4 = B.make_align_options(alignMethod=4, k=10, **opts)
        infos, comps = [], []
        for a, b in pairs:
            ra = B.ref_align4(a, b, o4)
            infos.append(B.ref_alignment_info(ra, len(a), len(b)) if len(ra) else np.zeros(12, np.uint32))
            comps.append(B.ref_compress(ra) if len(ra) else np.zeros(0, np.uint8))
            assert np.array_equal(B.oracle_decompress(comps[-1]).reshape(-1, 2), ra.reshape(-1, 2))     # how the test reads them
        out[f"align4_{j}_info"] = np.stack(infos).astype(np.uint32)
        out[f"align4_{j}_comp_toc"], out[f"align4_{j}_comp"] = _concat(comps, np.uint8)

    # LowHash0
    d = lowhash_random_input()
    for j, params in enumerate(LOWHASH_RANDOM_PARAMS):
        c, s, it, _ = B.ref_lowhash0(d["toc"], d["data"], d["flags"], B.LowHashParams(**params), threads=3)
        out.update({f"lowhash_{j}_candidates": c, f"lowhash_{j}_stats": s, f"lowhash_{j}_summary": it})

    # Histogram2 and the AlignmentInfo indicators
    cases, rng = hist2_cases()
    out["hist2_thresholds"] = np.array([[B.ref_histogram2_threshold(x, start, stop, bins, f) for f in HIST2_FRACTIONS]
                                        for (start, stop, bins, x) in cases], np.float64)
    out["hist2_indicators"] = np.stack([B.ref_alignment_indicators(r) for r in quality_records(rng, 200, 30)])

    np.savez_compressed(GOLDEN, **out)
    for key, v in out.items():
        print(f"{key:40s} {str(v.dtype):8s} {v.shape}")
    print(f"{GOLDEN}: {os.path.getsize(GOLDEN)} bytes")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit(__doc__)
    main(sys.argv[1])
