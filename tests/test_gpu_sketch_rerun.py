"""GPU parity tests for the exact re-run of flagged sketch units (a table that overflowed, or fewer than s survivors under
the threshold although k-mers were dropped): the unit goes through the first pass's kernels again, alone, with a larger
threshold, until it passes.  Every case compares with the oracle and checks that a re-run really happened."""
import numpy as np
import pytest

from fixtures import synth_genome
from test_gpu_sketch import _reads, assert_sketch_equal
from test_gpu_screen import check, run_screen

pytestmark = pytest.mark.gpu


def sketch_with_reruns(gpu, recs, p, **kw):
    before = gpu.stats()["exact_reruns"]
    out = gpu.sketch(recs, p, counts=True, **kw)
    assert gpu.stats()["exact_reruns"] > before
    return out


def assert_counts_equal(out, u, oracle_c):
    assert np.array_equal(out[3][u, :out[1][u]], oracle_c)


def test_repetitive_unit_between_normal_units_with_counts(gpu, oracle):
    # k = 8: 4^8 k-mers, a few copies of every final hash, so the top-of-heap counting quirk applies.  The re-run unit sits
    # between two ordinary units: it rewrites its own outputs only.
    k, s = 8, 500
    p = gpu.params(k=k, s=s)
    po = oracle.params(k=k)
    units = [[bytes(synth_genome(61, 30_000))],
             [bytes(np.tile(synth_genome(62, 3_000), 200))],          # 600 kbp, ~3000 distinct 8-mers
             [bytes(synth_genome(63, 25_000)), bytes(synth_genome(64, 9_000))]]
    recs = [r for rs in units for r in rs]
    uor = [u for u, rs in enumerate(units) for _ in rs]
    out = sketch_with_reruns(gpu, recs, p, unit_of_record=uor, n_units=len(units))
    for u, rs in enumerate(units):
        oh, oc, olen = oracle.sketch_unit(rs, po, s=s, counts=True)
        assert out[2][u] == olen
        assert_sketch_equal(out, u, oh)
        assert_counts_equal(out, u, oc)


def test_rerun_table_beyond_shared_memory_sort(gpu, oracle):
    # s = 5000: the re-run's table exceeds the 2^14 slots select_kernel sorts in shared memory and goes through the segmented sort
    s = 5000
    p = gpu.params(k=21, s=s)
    po = oracle.params(k=21)
    recs = [bytes(synth_genome(71, 200_000)), bytes(np.tile(synth_genome(72, 20_000), 50))]     # the second: 1 Mbp, ~20 000 distinct k-mers
    out = sketch_with_reruns(gpu, recs, p)
    for u, r in enumerate(recs):
        oh, oc, olen = oracle.sketch_unit([r], po, s=s, counts=True)
        assert out[2][u] == olen
        assert_sketch_equal(out, u, oh)
        assert_counts_equal(out, u, oc)


def test_min_copies_low_coverage_unit(gpu, oracle):
    # `-m 2` on reads at ~1x coverage: few hashes are seen twice, so the threshold pass ends with fewer than s qualified hashes
    m, s = 2, 300
    p = gpu.params(k=21, s=s, min_copies=m)
    po = oracle.params(k=21)
    reads = _reads(81, 60_000, 400)
    out = sketch_with_reruns(gpu, reads, p, unit_of_record=[0] * len(reads), n_units=1)
    oh, oc, _ = oracle.sketch_unit_m(reads, po, s=s, min_copies=m, counts=True)
    assert_sketch_equal(out, 0, oh)
    assert_counts_equal(out, 0, oc)


def test_screen_rerun_ignores_min_copies(gpu, oracle):
    # The screen mixture is a plain bottom-s heap: `-m` does not apply to it, in the first pass or in a re-run.  A chunk of a
    # 200x tiled block plus a few kbp of unique sequence has too few distinct hashes under the first threshold and is re-run.
    s = 1000
    po = oracle.params(k=21)
    block, unique = synth_genome(91, 3_000), synth_genome(92, 4_000)
    genomes = [block, unique, synth_genome(93, 50_000)]
    ref = np.full((len(genomes), s), np.uint64(2**64 - 1)); ref_n = np.zeros(len(genomes), np.uint32)
    for i, g in enumerate(genomes):
        h, _, _ = oracle.sketch_unit([bytes(g)], po, s=s)
        ref[i, :h.size] = h; ref_n[i] = h.size
    chunks = [b"*" + bytes(np.tile(block, 200)) + b"*" + bytes(unique)]
    want = oracle.screen(ref, ref_n, chunks, po, s=s)
    for m in (1, 3):
        before = gpu.stats()["exact_reruns"]
        res = run_screen(gpu, ref, ref_n, gpu.params(k=21, s=s, min_copies=m), chunks)
        assert gpu.stats()["exact_reruns"] > before
        check(res, want)
    assert want["shared"][0] > 0 and want["shared"][1] > 0
