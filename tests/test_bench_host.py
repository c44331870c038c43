"""CPU tests of bench.py's host-side helpers (nothing here touches a GPU)."""
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import bench  # noqa: E402


def test_alignment_roofline_arithmetic():
    r = bench.alignment_roofline(dp_cells=3e12, dp_ms=3000.0, sm_mhz=1965.0)
    assert r["bound"] == "alu" and r["unit"] == "G cell updates/s"
    assert abs(r["achieved"] - 1000.0) < 1e-6
    assert abs(r["peak"] - 148 * 64 * 1.965e9 / bench.ALU_OPS_PER_CELL / 1e9) < 1e-6 and bench.ALU_OPS_PER_CELL == 5
    assert abs(r["frac"] - r["achieved"] / r["peak"]) < 1e-12
    assert bench.alignment_roofline(0, 0.0, 1965.0) is None
    assert bench.alignment_roofline(1e9, 1.0, None)["peak"] == r["peak"]      # falls back to the B200's 1965 MHz


def test_workloads_name_the_baseline_configuration():
    wl = bench.WORKLOADS["nanopore-may2022-1M"]
    assert wl["reads"] == 1000000
    assert bench.MINHASH_MAY2022["m"] == 4 and bench.MINHASH_MAY2022["minHashIterationCount"] == 10
    assert bench.ALIGN_MAY2022["alignMethod"] == 3 and bench.ALIGN_MAY2022["downsamplingFactor"] == 0.05


def test_effective_cpus_and_placement_helpers():
    import os
    n = bench.effective_cpus()
    assert 1 <= n <= len(os.sched_getaffinity(0))

    class NoCuda:           # a torch stand-in without a device: the helper must answer "unknown", never raise
        class cuda:
            @staticmethod
            def get_device_properties(i):
                raise RuntimeError("no device")
    assert bench.gpu_numa_cpus(NoCuda, 0) == (None, None)


def test_dump_outputs_stays_within_64_mb_at_every_world_size(tmp_path):
    import numpy as np
    rng = np.random.default_rng(0)
    cand = rng.integers(0, 2**31, (3_000_000, 3)).astype(np.uint32)
    stats = rng.integers(0, 2**40, (1_000_000, 3)).astype(np.uint64)
    rec = rng.integers(0, 2**32, (300_000, 16), dtype=np.uint64).astype(np.uint32)
    ctoc = np.concatenate([[0], np.cumsum(rng.integers(20, 400, len(rec)))]).astype(np.uint64)
    cdata = rng.integers(0, 256, int(ctoc[-1])).astype(np.uint8)
    for world in (1, 2, 8):
        root = tmp_path / f"w{world}"
        for rank in range(world):       # as bench.py calls it: the statistics come from one rank
            bench.dump_outputs(str(root / f"rank{rank}"), cand, stats if rank == 0 else None, rec, ctoc, cdata, world=world)
        total = sum(f.stat().st_size for f in root.rglob("*.npy"))
        assert total <= 64_000_000, (world, total)
    z = np.load(tmp_path / "w1" / "rank0" / "read_lowhash_statistics.npy")
    assert z.dtype == np.float64 and z.shape == (bench.DUMP_STATS_ROWS, 3)
    assert np.array_equal(z, stats[bench._sample_rows(len(stats), bench.DUMP_STATS_ROWS, 3)].astype(np.float64))
    again = tmp_path / "again"
    bench.dump_outputs(str(again), cand, stats, rec, ctoc, cdata)
    for f in (tmp_path / "w1" / "rank0").iterdir():
        assert np.array_equal(np.load(f), np.load(again / f.name)), f.name
