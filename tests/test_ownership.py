"""Device memory comes back: contexts created and destroyed over and over, the stateless entry points called over and
over, and a contaminant set that fails after its table was built leave free device memory where it was.

Free memory is read with torch.cuda.mem_get_info (cudaMemGetInfo of the whole device).  Each check first runs its
work once, so that lazily loaded kernels and the runtime's own reservations are in place before the baseline is read.
"""
import numpy as np
import pytest

import golden_lib
from tgsfilter_b200 import _capi, prepass, synth
from tgsfilter_b200.engine import FilterEngine, align_hw, fold_detect
from tgsfilter_b200.params import ADAPTER_LIB

pytestmark = pytest.mark.gpu

CYCLES = 20
TOLERANCE = 4 << 20  # bytes of free device memory a check may lose over all its repetitions


def _free() -> int:
    import torch
    torch.cuda.synchronize()
    return torch.cuda.mem_get_info(0)[0]


def _long_read_batch(length: int):
    rng = np.random.default_rng(17)
    seq = np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, length)].tobytes()
    return synth.pack_reads([seq], [bytes(rng.integers(38, 70, length).astype(np.uint8))])


def test_repeated_contexts_return_their_memory():
    """One cycle: a context with deflate blocks, two slots, a contaminant set and the fold-back screen; the set is
    replaced once; a batch that overflows the region pool and a read longer than max_read_len (so the counter block
    grows) are submitted and collected; the context is destroyed.

    Measured on a B200 (1000 W power limit): one cycle holds 1728 MiB of device memory before its context is
    destroyed, and 20 cycles after a warm-up cycle leave free memory exactly where it was (drift 0 bytes)."""
    from test_gpu_parity import _pool_overflow_case
    params, pool = _pool_overflow_case()
    params.gz_blocks = True
    params.n_slots = 2
    params.max_read_len = 5000
    long_read = _long_read_batch(40_000)
    sets = [synth.make_contaminant(20_000, seed=s) for s in (1, 2)]

    def cycle() -> int:
        start = _free()
        with FilterEngine(params) as eng:
            eng.set_contaminants([sets[0]], k=17)
            eng.set_foldback(True)
            eng.set_contaminants([sets[1]], k=17)
            before = eng.layout.max_bins
            reads, _ = eng.run(pool)
            assert int(reads["n_mid"].sum()) > 65536  # the pool overflowed and the tail was re-run
            eng.run(long_read)
            assert eng.counters().layout.max_bins > before
            footprint = start - _free()
        return footprint

    _free()
    cycle()  # warm-up
    base = _free()
    footprints = [cycle() for _ in range(CYCLES)]
    drift = base - _free()
    print(f"cycle footprint {min(footprints) / 2**20:.1f} MiB, drift after {CYCLES} cycles {drift / 2**20:.3f} MiB")
    assert min(footprints) > 10 * TOLERANCE
    assert drift <= TOLERANCE, f"{drift} bytes of device memory not returned after {CYCLES} cycles"


def _prepass():
    z = np.load(golden_lib.HERE + "/prepass.npz")
    return lambda: prepass.device_prepass(z["ends5p"], z["ends3p"], ADAPTER_LIB, 0.9)


def _end_kmers():
    rows = np.frombuffer(b"ACGT", dtype=np.uint8)[np.random.default_rng(3).integers(0, 4, (2000, 150))]
    return lambda: prepass.device_end_kmers(rows, 12, 60)


def _align():
    rng = np.random.default_rng(4)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    pairs = [(acgt[rng.integers(0, 4, q)].tobytes(), acgt[rng.integers(0, 4, 400)].tobytes(), q // 5)
             for q in rng.integers(10, 600, 500)]
    return lambda: align_hw(pairs)


def _fold():
    rng = np.random.default_rng(5)
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    seqs = [acgt[rng.integers(0, 4, int(n))].tobytes() for n in rng.integers(100, 20_000, 200)]
    return lambda: fold_detect(seqs)


@pytest.mark.parametrize("make", [_prepass, _end_kmers, _align, _fold], ids=["prepass", "end_kmer_counts", "align_hw",
                                                                           "fold_detect"])
def test_stateless_entry_points_return_their_memory(make):
    call = make()
    _free()
    call()  # warm-up
    base = _free()
    for _ in range(CYCLES):
        call()
    drift = base - _free()
    print(f"drift after {CYCLES} calls {drift / 2**20:.3f} MiB")
    assert drift <= TOLERANCE, f"{drift} bytes of device memory not returned after {CYCLES} calls"


def test_contaminant_set_failing_after_its_table_is_built():
    """A set whose bytes hold no valid k-mer is rejected only after its table was allocated and built: the call
    fails with TGSF_ERR_INVALID, the installed set keeps screening as before, and the table is freed."""
    genome = synth.make_contaminant(48_502)
    batch = synth.mix_contaminants(synth.make_config(1, 200), genome, 0.08, 0.04, seed=1)[0]
    params = synth.config_params(1)
    with FilterEngine(params) as eng:
        eng.set_contaminants([genome], k=17)
        _, want = eng.run(batch)
        assert (want["status"] == _capi.PIECE_CONTAM).any()
        no_kmer = [b"N" * (1 << 20)]  # a 32 MiB table

        def fail():
            with pytest.raises(_capi.TgsfError) as e:
                eng.set_contaminants(no_kmer, k=17)
            assert e.value.code == _capi.TGSF_ERR_INVALID

        fail()  # warm-up
        base = _free()
        for _ in range(CYCLES):
            fail()
        drift = base - _free()
        _, got = eng.run(batch)
    print(f"drift after {CYCLES} failed sets {drift / 2**20:.3f} MiB")
    assert np.array_equal(got, want)
    assert drift <= TOLERANCE, f"{drift} bytes of device memory not returned after {CYCLES} failed sets"
