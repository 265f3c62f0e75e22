"""bench.py contract checks that need no GPU: the workload plan, the `config` object shared by both arms and
the reference arm itself (the unmodified reference CLI on a tiny dataset, numpy generator)."""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import bench
import ref_lib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_plan_batches_weak_and_strong():
    # weak: every rank its own dataset of the full size; the first batch of rank 0 carries the config's base seed
    p0 = bench.plan_batches(2, 200_000, 8, 0, False, 2)
    p3 = bench.plan_batches(2, 200_000, 8, 3, False, 2)
    assert sum(n for _, n, _ in p0) == 200_000 and sum(n for _, n, _ in p3) == 200_000 and len(p0) == 2
    assert p0[0][2] == bench.SEED0 + 2 and {s for _, _, s in p0}.isdisjoint({s for _, _, s in p3})
    assert len(bench.plan_batches(5, 2_000_000, 1, 0, False)) == 5  # > 400 000 reads: several batches
    # strong: ONE dataset, every batch on exactly one rank, same seeds whatever the world size
    for world in (1, 2, 4, 8):
        seen = {}
        for r in range(world):
            for j, n, s in bench.plan_batches(4, 1_000_000, world, r, True):
                assert j not in seen
                seen[j] = (n, s)
        assert len(seen) == bench.STRONG_BATCHES and sum(n for n, _ in seen.values()) == 1_000_000
        assert seen == {j: (n, s) for j, n, s in bench.plan_batches(4, 1_000_000, 1, 0, True)}


def test_config_object_is_a_pure_function_of_the_command_line():
    a = bench.static_config(2, 200_000, False)
    assert a == bench.static_config(2, 200_000, False) and a != bench.static_config(2, 200_000, True)
    assert "config[1]" in a["workload"] and a["cli"] == "-x ont" and a["reads"] == 200_000


def test_dump_outputs_writes_float64_and_samples_to_the_limit(tmp_path):
    from tgsfilter_b200 import _capi
    rng = np.random.default_rng(3)
    reads = np.zeros(5000, dtype=_capi.READ_RESULT_DTYPE)
    pieces = np.zeros(7000, dtype=_capi.PIECE_DTYPE)
    reads["sum_q"] = rng.integers(0, 1 << 40, reads.size)
    pieces["start"] = np.arange(pieces.size)
    counters = np.arange(100, dtype=np.uint64)
    bench.dump_outputs(str(tmp_path / "all"), [0], [(reads, pieces)], counters)
    r = np.load(tmp_path / "all" / "batch0_reads.npy")
    assert r.dtype == np.float64 and r.shape == (5000, 1 + len(bench.READ_COLUMNS))
    assert np.array_equal(r[:, 1], reads["sum_q"].astype(np.float64))
    assert np.array_equal(np.load(tmp_path / "all" / "counters.npy"), counters.astype(np.float64))
    limit = 200_000
    for d in ("s1", "s2"):
        bench.dump_outputs(str(tmp_path / d), [0], [(reads, pieces)], counters, limit=limit)
    assert sum(f.stat().st_size for f in (tmp_path / "s1").iterdir()) <= limit + 3 * 128  # + the .npy headers
    p1, p2 = (np.load(tmp_path / d / "batch0_pieces.npy") for d in ("s1", "s2"))
    assert 0 < len(p1) < pieces.size and np.array_equal(p1, p2)  # the same seeded sample every time
    assert np.array_equal(p1[:, 0], p1[:, 3])  # row index column = the rows' own `start` here


@pytest.mark.skipif(not ref_lib.available(), reason="oracle/_ref not present")
def test_reference_arm_prints_the_contract_line():
    pr = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--config", "1",
                         "--reads", "1500", "--steps", "1", "--warmup", "1"], stdout=subprocess.PIPE,
                        stderr=subprocess.PIPE, timeout=600, env=dict(os.environ, CUDA_VISIBLE_DEVICES=""))
    assert pr.returncode == 0, pr.stderr.decode()[-800:]
    line = json.loads([l for l in pr.stdout.decode().splitlines() if l.startswith("{")][-1])
    assert line["impl"] == "reference" and line["metric"] == "filtered Gbases/s" and line["unit"] == "Gbases/s"
    assert line["config"] == bench.static_config(1, 1500, False)
    assert line["cpu_baseline"]["kind"] == "reference" and line["cpu_baseline"]["value"] == line["value"] > 0
    assert "the whole dataset" in line["cpu_baseline"]["sample"]
    assert line["e2e"] == {"value": line["value"], "unit": "Gbases/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
