"""Validate the plain-C restatement against the reference's own hash + heap object code
(oracle/_ref/libmash_ref.so, built in place from the reference's sources by oracle/Makefile).  Its answers for the inputs
below are stored in tests/golden/ref_objcode.npz (`ref`, see fixtures.ReferenceAnswers); `pytest --record-reference` where
oracle/_ref is built computes them again with the reference."""
import numpy as np
import pytest

from fixtures import synth_genome

REFERENCE_ANSWERS = "ref_objcode"


def reference():
    from oracle.pyoracle import RefLib
    return RefLib()


def test_get_hash_matches_reference(oracle, ref):
    rng = np.random.Generator(np.random.PCG64(11))
    cases = []
    for k in range(1, 33):
        for _ in range(50):
            kmer = bytes(rng.integers(33, 127, k, dtype=np.uint8))
            seed = int(rng.integers(0, 2**32))
            for use64 in (True, False):
                cases.append((kmer, seed, use64))
    want = ref("get_hash", lambda lib: np.array([lib.get_hash(*c) for c in cases], np.uint64))
    assert want.size == len(cases)
    for c, w in zip(cases, want):
        assert oracle.get_hash(*c) == int(w), c


@pytest.mark.parametrize("k,s,noncanonical", [(21, 1000, False), (16, 400, False), (11, 50, False), (32, 1000, False),
                                                (21, 10, True), (8, 50, False), (3, 1000, False)])
def test_sketch_unit_matches_reference(oracle, ref, k, s, noncanonical):
    p = oracle.params(k=k, seed=42, noncanonical=noncanonical)
    recs = [bytes(synth_genome(100 + i, n, n_runs=3, lower_frac=0.05)) for i, n in enumerate([200_000, 5, k, k - 1, 70_000])]
    recs.append(b"ACGTNNNNacgtacgtacgtacgtacgtRYacgtacgtacgtacgtacgtacgtacgt*ACGTACGTACGTACGTACGTACGTA")
    ho, co, lo = oracle.sketch_unit(recs, p, s=s, counts=True)
    hr, cr, lr = ref(f"sketch_unit_k{k}_s{s}_nc{int(noncanonical)}", lambda lib: lib.sketch_unit(recs, p, s=s, counts=True))
    assert lo == lr
    assert np.array_equal(ho, hr)
    assert np.array_equal(co, cr)     # includes the top-of-heap multiplicity quirk (k=8, k=3 cases)


def test_reads_mode_length_matches_reference(oracle, ref):
    p = oracle.params(k=21, seed=42)
    recs = [bytes(synth_genome(5, 50_000))]
    assert oracle.sketch_unit(recs, p, s=100, reads=True)[2] == ref("reads_mode_length", lambda lib: lib.sketch_unit(recs, p, s=100, reads=True)[2])


def test_hash_sequence_matches_reference(oracle, ref):
    p = oracle.params(k=21, seed=42)
    g = synth_genome(3, 120_000)
    ref_h, _, _ = oracle.sketch_unit([bytes(g)], p, s=500)
    reads = [bytes(g[a:a + 150]) for a in range(0, 100_000, 97)]
    reads[3] = reads[3][:60] + b"N" + reads[3][61:]
    chunk = b"".join(b"*" + r for r in reads)
    res = oracle.screen(ref_h[None, :], np.array([ref_h.size], np.uint32), [chunk], p, s=500)

    def reference_hash_sequence(lib):
        counts = np.zeros(res["keys"].size, np.uint32)
        mix = lib.hash_sequence(res["keys"], counts, chunk, p, s=500)
        return counts, mix

    counts, mix = ref("hash_sequence", reference_hash_sequence)
    assert np.array_equal(counts, res["counts"])
    assert np.array_equal(mix, res["mixture"])


def test_reference_cpu_path_from_files_reproduces_the_goldens(reflib, golden, tmp_path):
    # the whole CPU arm as `mash sketch` runs it -- the reference's own parser (kseq.h), the restated addMinHashes loop and the
    # reference's hash + heap object code -- on the reference's test genomes (gzipped, as gzread takes them) must give
    # test/ref/genomes.json: this is the code bench.py times as cpu_baseline / --impl reference
    import os
    from fixtures import GOLDEN
    from oracle.pyoracle import Oracle
    p = Oracle().params(k=21, seed=42)
    paths = [os.path.join(GOLDEN, f"genome{i}.fna.gz") for i in (1, 2, 3)]
    h, n, lens = reflib.sketch_files(paths, p, s=1000, threads=3)
    for i in range(3):
        want, length, _, _ = golden.golden_sketch(i)
        assert n[i] == 1000 and np.array_equal(h[i], want) and int(lens[i]) == length


def test_file_path_equals_in_memory_path(oracle, ref, tmp_path):
    p = oracle.params(k=21, seed=42)
    g = synth_genome(77, 300_000, n_runs=4, lower_frac=0.05)
    path = tmp_path / "g.fa"
    with open(path, "wb") as f:
        f.write(b">g some comment\n")
        for a in range(0, g.size, 70):
            f.write(bytes(g[a:a + 70]) + b"\n")
        f.write(b">tiny\nACGT\n")                      # shorter than k: skipped, not counted in the length
    h, n, lens = ref("file_path", lambda lib: lib.sketch_files([str(path)], p, s=500, threads=1))
    hm, lm = ref("in_memory_path", lambda lib: lib.sketch_unit([bytes(g), b"ACGT"], p, s=500)[::2])
    assert int(lens[0]) == lm == g.size and np.array_equal(h[0, :n[0]], hm)
    ho, _, lo = oracle.sketch_unit([bytes(g), b"ACGT"], p, s=500)
    assert lo == lm and np.array_equal(ho, hm)


def test_ref_screen_many_matches_oracle(oracle, ref):
    """The multi-threaded CPU arm of bench.py's screen leg (reference hash + heap object code, the reference's robin_hood table
    type) against the plain-C oracle: same counters, same mixture bottom-s."""
    from fixtures import synth_genome
    p = oracle.params(k=21)
    g = [synth_genome(40 + i, 60_000) for i in range(3)]
    refs = np.full((3, 200), np.uint64(2**64 - 1)); refs_n = np.zeros(3, np.uint32)
    for i, gg in enumerate(g):
        h, _, _ = oracle.sketch_unit([bytes(gg)], p, s=200)
        refs[i, :h.size] = h; refs_n[i] = h.size
    rng = np.random.Generator(np.random.PCG64(9))
    chunks = []
    for c in range(7):
        reads = []
        for _ in range(300):
            gg = g[int(rng.integers(0, 2))]
            a = int(rng.integers(0, gg.size - 150))
            reads.append(bytes(gg[a:a + 150]))
        chunks.append(b"".join(b"*" + r for r in reads))
    want = oracle.screen(refs, refs_n, chunks, p, s=200)

    def reference_screen_many(lib):
        t = lib.screen_table(want["keys"])
        try:
            mix = lib.screen_many(t, chunks, p, s=200, threads=3)
            counts = lib.screen_table_counts(t, want["keys"])
        finally:
            lib.screen_table_free(t)
        return counts, mix

    counts, mix = ref("screen_many", reference_screen_many)
    assert np.array_equal(counts, want["counts"]) and np.array_equal(mix, want["mixture"])


def _read_set(seed, genome_len, n_reads, err=0.01):
    from fixtures import synth_genome
    g = synth_genome(seed, genome_len)
    rng = np.random.Generator(np.random.PCG64(seed + 1))
    reads = []
    acgt = np.frombuffer(b"ACGT", np.uint8)
    for _ in range(n_reads):
        a = int(rng.integers(0, g.size - 100))
        r = g[a:a + 100].copy()
        m = rng.random(100) < err
        r[m] = acgt[rng.integers(0, 4, int(m.sum()))]
        if rng.random() < 0.05:
            r[int(rng.integers(0, 100))] = ord("N")
        reads.append(bytes(r))
    return reads


@pytest.mark.parametrize("m,s,k,cov", [(2, 200, 21, 8), (3, 100, 16, 12), (2, 50, 11, 3), (5, 300, 21, 6), (2, 1000, 21, 1)])
def test_min_copies_heap_oracle_equals_reference_object_code(oracle, ref, m, s, k, cov):
    """`-m`: the oracle's restated pending-set logic against the reference's own MinHashHeap(use64, s, m, 0): same bottom-s,
    same multiplicities (incl. the top-of-heap quirk), same -r length."""
    p = oracle.params(k=k)
    reads = _read_set(100 + m + s, 20_000, 200 * cov)
    oh, oc, ol = oracle.sketch_unit_m(reads, p, s=s, min_copies=m, counts=True)
    rh, rc, rl = ref(f"sketch_unit_m_m{m}_s{s}_k{k}_cov{cov}", lambda lib: lib.sketch_unit_m(reads, p, s=s, min_copies=m, counts=True))
    assert np.array_equal(oh, rh) and np.array_equal(oc, rc) and ol == rl
    # order-independent characterisation used by the GPU path: the s smallest hashes seen at least m times
    allh = np.concatenate([oracle.all_hashes(r, p) for r in reads if len(r) >= k])
    u, c = np.unique(allh, return_counts=True)
    want = u[c >= m][:s]
    assert np.array_equal(oh, want)
    assert np.all(oc[:-1] == c[np.searchsorted(u, oh[:-1])]) if oh.size else True
    assert oh.size == 0 or m <= oc[-1] <= c[np.searchsorted(u, oh[-1])]


@pytest.mark.parametrize("m,c,s,cov", [(1, 3.0, 200, 10), (2, 4.0, 100, 12), (1, 50.0, 200, 4), (3, 3.5, 300, 20), (2, 2.0, 50, 6)])
def test_target_coverage_stop_oracle_equals_reference_object_code(oracle, ref, m, c, s, cov):
    """`-c`: the record loop stops after the first read that brings the heap's average multiplicity to the target (Sketch.cpp:1258-1262)."""
    p = oracle.params(k=21)
    reads = _read_set(500 + m + s, 20_000, 200 * cov, err=0.005)
    oh, oc, ol, ou = oracle.sketch_unit_mc(reads, p, s=s, min_copies=m, target_cov=c, counts=True)
    rh, rc, rl, ru = ref(f"sketch_unit_mc_m{m}_c{c}_s{s}_cov{cov}", lambda lib: lib.sketch_unit_mc(reads, p, s=s, min_copies=m, target_cov=c, counts=True))
    assert ou == ru and np.array_equal(oh, rh) and np.array_equal(oc, rc) and ol == rl
    if c < 20:
        assert 0 < ou < len(reads)                     # stopped early
        assert oc.sum() / oc.size >= c
    else:
        assert ou == len(reads)
