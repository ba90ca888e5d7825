"""GPU parity tests for hot path 1 (sketching), through the C ABI, against the oracle and the
reference's golden files.  Bit-exact: hashes, sketch sets, lengths."""
import numpy as np
import pytest

from fixtures import synth_genome, mutate

pytestmark = pytest.mark.gpu


def assert_sketch_equal(gpu_out, u, oracle_h):
    h, n, _ = gpu_out[:3]
    assert n[u] == oracle_h.size
    assert np.array_equal(h[u, :n[u]], oracle_h)


@pytest.mark.parametrize("k", list(range(1, 33)))
@pytest.mark.parametrize("noncanonical", [False, True])
def test_every_window_hash_matches_oracle(gpu, oracle, k, noncanonical):
    # getHash over every window, all k, both strands modes, with N runs / lower case / junk bytes
    seq = synth_genome(1000 + k, 20_000, n_runs=4, lower_frac=0.1)
    seq[5000:5003] = np.frombuffer(b"*-\x00", np.uint8)
    seq[17000] = 200
    p = gpu.params(k=k, s=100, noncanonical=noncanonical)
    po = oracle.params(k=k, noncanonical=noncanonical)
    assert p.use64 == po.use64
    h, v = gpu.hash_windows(seq, p)
    want = oracle.all_hashes(bytes(seq), po)
    assert int(v.sum()) == want.size
    assert np.array_equal(h[v], want)


def test_preserve_case_skips_lower_case(gpu, oracle):
    seq = synth_genome(77, 30_000, lower_frac=0.02)
    p = gpu.params(k=21, s=100, preserve_case=True)
    po = oracle.params(k=21, preserve_case=True)
    h, v = gpu.hash_windows(seq, p)
    want = oracle.all_hashes(bytes(seq), po)
    assert int(v.sum()) == want.size and np.array_equal(h[v], want)


def test_golden_genomes_bit_exact(gpu, golden):
    # BASELINE config 1: `mash sketch genome1.fna genome2.fna genome3.fna` -> test/ref/genomes.json
    p = gpu.params(k=21, s=1000, seed=42)
    recs, uor = [], []
    for u, (_, rs) in enumerate(golden.genomes):
        for r in rs:
            recs.append(r[2]); uor.append(u)
    h, n, length = gpu.sketch(recs, p, unit_of_record=uor, n_units=3)
    for i in range(3):
        gh, glen, _, _ = golden.golden_sketch(i)
        assert length[i] == glen
        assert n[i] == 1000 and np.array_equal(h[i], gh)


def test_golden_reads_sketch_bit_exact(gpu, golden):
    # `mash sketch -r reads1.fastq reads2.fastq`: one unit over all reads; length = estimateSetSize (host formula)
    p = gpu.params(k=21, s=1000, seed=42)
    reads = golden.reads_round_robin()
    h, n, _ = gpu.sketch(reads, p, unit_of_record=[0] * len(reads), n_units=1)
    gh, glen = golden.golden_reads_sketch()
    assert n[0] == 1000 and np.array_equal(h[0], gh)
    est = int(np.uint64(2.0 ** 64 * float(n[0]) / float(h[0, n[0] - 1])))     # MinHashHeap.h:45
    assert est == glen


@pytest.mark.parametrize("k,s", [(21, 1000), (16, 400), (11, 10), (32, 1000), (21, 10), (17, 2000), (8, 50), (3, 1000), (1, 5)])
def test_synthetic_units_match_oracle(gpu, oracle, k, s):
    # ragged batch: big / tiny / empty / shorter-than-k records, multi-record units, soft-masking, N runs
    p = gpu.params(k=k, s=s)
    po = oracle.params(k=k)
    g0 = synth_genome(1, 300_000, n_runs=5, lower_frac=0.05)
    units = [
        [bytes(g0)],
        [bytes(mutate(g0, 0.01, 2))],
        [bytes(synth_genome(3, 50_000)), b"ACGT", bytes(synth_genome(4, 1234)), b""],   # multi record
        [b"A" * 5000],                                                                    # one k-mer repeated
        [b"ACGTACGTAC" * 300],                                                            # few distinct k-mers
        [b"N" * 1000],                                                                    # nothing valid
        [b"ACG"],                                                                         # shorter than k (for k > 3)
        [bytes(synth_genome(5, 700))],                                                    # fewer k-mers than s
        [],                                                                               # unit without records
    ]
    recs, uor = [], []
    for u, rs in enumerate(units):
        for r in rs:
            recs.append(r); uor.append(u)
    out = gpu.sketch(recs, p, unit_of_record=uor, n_units=len(units), counts=True)
    for u, rs in enumerate(units):
        oh, oc, olen = oracle.sketch_unit(rs, po, s=s, counts=True)
        assert out[2][u] == olen
        assert_sketch_equal(out, u, oh)


@pytest.mark.parametrize("k,s,n", [(8, 50, 100_000), (3, 20, 5_000), (21, 200, 60_000), (11, 1000, 400_000), (16, 64, 30_000)])
def test_counts_match_reference_heap_semantics(gpu, oracle, k, s, n):
    # Multiplicities as MinHashHeap produces them (HashSet counts), INCLUDING the quirk that an occurrence equal to the
    # top of a full heap is not counted (MinHashHeap.cpp:70-74; SURVEY.md 8 a5) -- the oracle restates it and is pinned
    # to the reference's object code for it (tests/test_oracle_vs_ref.py).  High-coverage inputs make the quirk bite.
    p = gpu.params(k=k, s=s)
    po = oracle.params(k=k)
    g = synth_genome(9 + k, n)
    units = [[bytes(g)],
             [bytes(g[a:a + 150]) for a in np.random.Generator(np.random.PCG64(k)).integers(0, n - 150, 4 * n // 150)],   # "reads", ~4x coverage
             [bytes(np.tile(g[:n // 8], 8))]]
    recs, uor = [], []
    for u, rs in enumerate(units):
        recs += rs; uor += [u] * len(rs)
    h, cnt_n, _, c = gpu.sketch(recs, p, unit_of_record=uor, n_units=len(units), counts=True)
    hit = 0
    for u, rs in enumerate(units):
        oh, oc, _ = oracle.sketch_unit(rs, po, s=s, counts=True)
        m = cnt_n[u]
        assert np.array_equal(h[u, :m], oh)
        assert np.array_equal(c[u, :m], oc), (u, c[u, m - 1], oc[-1])
    # the quirk must actually have been exercised somewhere in this parametrisation (true count > reported count)
    true_last = [int(np.sum(oracle.all_hashes(b"\x00".join(rs), po) == h[u, cnt_n[u] - 1])) for u, rs in enumerate(units)]
    if k in (8, 3):
        assert any(t > int(c[u, cnt_n[u] - 1]) for u, t in enumerate(true_last))


def test_one_unit_per_record_order_preserved(gpu, oracle):
    # `-i` mode: one sketch per record, outputs in input order (ThreadPool ordering contract)
    p = gpu.params(k=21, s=200)
    po = oracle.params(k=21)
    recs = [bytes(synth_genome(100 + i, 20_000 + 997 * i)) for i in range(40)]
    out = gpu.sketch(recs, p)
    for u, r in enumerate(recs):
        oh, _, olen = oracle.sketch_unit([r], po, s=200)
        assert out[2][u] == olen
        assert_sketch_equal(out, u, oh)


def test_highly_repetitive_unit_takes_exact_rerun(gpu, oracle):
    # a long unit with few distinct k-mers: the threshold pass finds < s survivors and the exact re-run must kick in
    p = gpu.params(k=21, s=1000)
    po = oracle.params(k=21)
    unit = bytes(np.tile(synth_genome(5, 3000), 200))           # 600 kbp, ~3000 distinct k-mers
    before = gpu.stats()["exact_reruns"]
    out = gpu.sketch([unit], p)
    oh, _, _ = oracle.sketch_unit([unit], po, s=1000)
    assert_sketch_equal(out, 0, oh)
    assert gpu.stats()["exact_reruns"] > before


def test_union_property_full_size(gpu):
    # size-independent property at BASELINE's unit size (5 Mbp): bottom-s(A ++ B) == bottom-s(bottom-s(A) U bottom-s(B))
    p = gpu.params(k=21, s=1000)
    a = synth_genome(20260923, 5_000_000)
    b = synth_genome(20260924, 5_000_000)
    h, n, _ = gpu.sketch([bytes(a), bytes(b), bytes(a), bytes(b)], p, unit_of_record=[0, 1, 2, 2], n_units=3)
    assert n[0] == n[1] == n[2] == 1000
    merged = np.unique(np.concatenate([h[0], h[1]]))[:1000]
    assert np.array_equal(h[2], merged)
    assert np.all(np.diff(h[2].astype(object)) > 0)      # ascending, distinct


PROTEIN = "ACDEFGHIKLMNPQRSTVWY"


def synth_protein(seed, n):
    rng = np.random.Generator(np.random.PCG64(seed))
    a = np.frombuffer((PROTEIN + "XBZ*acdefg").encode(), np.uint8)
    w = np.array([1.0] * 20 + [0.02, 0.01, 0.01, 0.01] + [0.05] * 6)
    return a[rng.choice(a.size, n, p=w / w.sum())]


@pytest.mark.parametrize("k,alphabet,preserve_case", [(9, PROTEIN, False), (7, PROTEIN, False), (9, PROTEIN, True), (21, "ACGTN", False),
                                                       (12, "ACGU", False), (32, PROTEIN, False), (1, "AB", False), (5, "acgt", True)])
def test_byte_alphabets_every_window(gpu, oracle, k, alphabet, preserve_case):
    # `mash sketch -a` (protein, k=9) and `-z <alphabet>`: non-canonical, any byte alphabet (sketchParameterSetup.cpp:79-95)
    p = gpu.params(k=k, s=100, alphabet=alphabet, noncanonical=True, preserve_case=preserve_case)
    po = oracle.params(k=k, alphabet=alphabet, noncanonical=True, preserve_case=preserve_case)
    assert p.use64 == po.use64 and bytes(p.alphabet) == bytes(po.alphabet)
    seq = synth_protein(k, 30_000) if "D" in alphabet else synth_genome(k, 30_000, n_runs=5, lower_frac=0.2)
    if alphabet == "ACGU":
        seq = seq.copy(); seq[seq == ord("T")] = ord("U")
    h, v = gpu.hash_windows(seq, p)
    want = oracle.all_hashes(bytes(seq), po)
    assert int(v.sum()) == want.size and np.array_equal(h[v], want)


@pytest.mark.parametrize("k,s", [(9, 1000), (7, 400), (5, 50)])
def test_protein_sketches_match_oracle(gpu, oracle, k, s):
    p = gpu.params(k=k, s=s, alphabet=PROTEIN, noncanonical=True)
    po = oracle.params(k=k, alphabet=PROTEIN, noncanonical=True)
    units = [[bytes(synth_protein(1, 400_000))], [bytes(synth_protein(2, 3_000)), b"MKV", bytes(synth_protein(3, 50_000))], [b"M" * 2000], []]
    recs, uor = [], []
    for u, rs in enumerate(units):
        recs += rs; uor += [u] * len(rs)
    out = gpu.sketch(recs, p, unit_of_record=uor, n_units=len(units), counts=True)
    for u, rs in enumerate(units):
        oh, oc, olen = oracle.sketch_unit(rs, po, s=s, counts=True)
        assert out[2][u] == olen
        assert_sketch_equal(out, u, oh)
        assert np.array_equal(out[3][u, :out[1][u]], oc)
    # murmur KAT from the reference object code (SURVEY.md 8c): MKVLAAGIV, k=9 -> 10212611784005380714
    h, v = gpu.hash_windows(b"MKVLAAGIV", gpu.params(k=9, s=1, alphabet=PROTEIN, noncanonical=True))
    assert v[0] and int(h[0]) == 10212611784005380714


def test_canonical_needs_nucleotide_alphabet(gpu):
    import mash_b200
    p = gpu.params(k=9, s=100, alphabet=PROTEIN, noncanonical=False)
    with pytest.raises(mash_b200.MashGpuError) as e:
        gpu.sketch([b"MKVLAAGIVALLLAAGCSSAPQ"], p)
    assert e.value.code == 3


def test_packed_feed_path_equals_ascii_path(gpu, oracle, monkeypatch):
    # MASHGPU_HOST_PACK=1: mashgpu_sketch_batch packs to 2 bits/base (+ invalid runs) on the host and the scan kernel
    # stages from the packed stream; default: pinned ASCII copy.  Same sketches either way.
    p = gpu.params(k=21, s=500)
    po = oracle.params(k=21)
    g = synth_genome(31, 1_000_037, n_runs=40, lower_frac=0.07)
    g[123456] = ord("*"); g[0] = ord("n"); g[-1] = 0
    recs = [bytes(g), bytes(synth_genome(32, 33)), b"ACGTACGTACGTACGTACGTACGTACGTNNACGT", bytes(synth_genome(33, 777_777))]
    uor = [0, 0, 1, 2]
    ascii_ = gpu.sketch(recs, p, unit_of_record=uor, n_units=3, counts=True)
    monkeypatch.setenv("MASHGPU_HOST_PACK", "1")
    packed = gpu.sketch(recs, p, unit_of_record=uor, n_units=3, counts=True)
    monkeypatch.delenv("MASHGPU_HOST_PACK")
    for a, b in zip(packed, ascii_):
        assert np.array_equal(a, b)
    for u, rs in enumerate([[recs[0], recs[1]], [recs[2]], [recs[3]]]):
        oh, _, olen = oracle.sketch_unit(rs, po, s=500)
        assert packed[2][u] == olen
        assert_sketch_equal(packed, u, oh)


@pytest.mark.parametrize("pack", ["0", "1"])
def test_multi_wave_batch(gpu, oracle, monkeypatch, pack):
    # more than one wave (2^31 stream positions each): 3 units of ~0.9 Gbp would be slow for the oracle, so the wave
    # size is not reachable here; instead check a batch whose units straddle many tiles and records
    monkeypatch.setenv("MASHGPU_HOST_PACK", pack)
    p = gpu.params(k=21, s=300)
    po = oracle.params(k=21)
    recs, uor = [], []
    for u in range(12):
        for r in range(1 + u % 3):
            recs.append(bytes(synth_genome(500 + 10 * u + r, 40_000 + 7919 * u)))
            uor.append(u)
    out = gpu.sketch(recs, p, unit_of_record=uor, n_units=12)
    for u in range(12):
        oh, _, olen = oracle.sketch_unit([r for r, x in zip(recs, uor) if x == u], po, s=300)
        assert out[2][u] == olen
        assert_sketch_equal(out, u, oh)


@pytest.mark.parametrize("mode", ["hybrid", "ascii", "packed"])
def test_feed_scheduler_many_waves_pinned_buffers(gpu, oracle, monkeypatch, mode):
    # The two feed paths of mashgpu_sketch_batch side by side: records in page-locked memory (eligible for the direct ASCII
    # copy), waves cut small (MASHGPU_WAVE_BYTES / MASHGPU_WAVE_UNITS are test hooks) so that the ASCII producer and the host
    # packer both claim waves of one batch; some units are made of small records, which only the packer (or, ASCII only, the
    # pinned staging buffer) takes.  Same sketches whichever producer fed a wave.
    import torch
    monkeypatch.setenv("MASHGPU_WAVE_BYTES", str(700_000))
    monkeypatch.setenv("MASHGPU_WAVE_UNITS", "3")
    if mode != "hybrid":
        monkeypatch.setenv("MASHGPU_HOST_PACK", "0" if mode == "ascii" else "1")
    p = gpu.params(k=21, s=400)
    po = oracle.params(k=21)
    recs, uor, keep = [], [], []
    for u in range(14):
        n_rec = 1 if u % 4 else 3
        for r in range(n_rec):
            ln = (300_000 + 4099 * u) if n_rec == 1 else (5_000 + 911 * r)
            g = synth_genome(900 + 10 * u + r, ln, n_runs=2 if u % 3 == 0 else 0, lower_frac=0.03 if u % 5 == 0 else 0.0)
            t = torch.from_numpy(g.copy()).pin_memory()
            keep.append(t)
            recs.append(t.numpy()); uor.append(u)
    out = gpu.sketch(recs, p, unit_of_record=uor, n_units=14, counts=True)
    for u in range(14):
        oh, oc, olen = oracle.sketch_unit([bytes(r) for r, x in zip(recs, uor) if x == u], po, s=400, counts=True)
        assert out[2][u] == olen
        assert_sketch_equal(out, u, oh)
        assert np.array_equal(out[3][u, :out[1][u]], oc)


def test_large_sketch_size_goes_through_global_sort(gpu, oracle):
    # s = 5000: the unit's candidate table (2^16 slots) does not fit select_kernel's shared-memory sort, so the unit goes
    # through the segmented radix sort -- same answer, `mash sketch -s 5000`
    p = gpu.params(k=21, s=5000)
    po = oracle.params(k=21)
    g = bytes(synth_genome(1234, 400_000))
    short = bytes(synth_genome(1235, 3_000))          # fewer k-mers than s
    out = gpu.sketch([g, short], p, counts=True)
    for u, r in enumerate((g, short)):
        oh, oc, olen = oracle.sketch_unit([r], po, s=5000, counts=True)
        assert out[2][u] == olen
        assert_sketch_equal(out, u, oh)
        assert np.array_equal(out[3][u, :out[1][u]], oc)


def _reads(seed, genome_len, n_reads, err=0.01, read_len=100):
    g = synth_genome(seed, genome_len)
    rng = np.random.Generator(np.random.PCG64(seed + 1))
    acgt = np.frombuffer(b"ACGT", np.uint8)
    out = []
    for _ in range(n_reads):
        a = int(rng.integers(0, g.size - read_len))
        r = g[a:a + read_len].copy()
        m = rng.random(read_len) < err
        r[m] = acgt[rng.integers(0, 4, int(m.sum()))]
        if rng.random() < 0.05:
            r[int(rng.integers(0, read_len))] = ord("N")
        out.append(bytes(r))
    return out


@pytest.mark.parametrize("m,s,k,cov", [(2, 200, 21, 8), (3, 100, 16, 12), (2, 50, 11, 3), (5, 300, 21, 6), (2, 1000, 21, 1), (2, 400, 21, 30)])
def test_min_copies_filter_matches_reference_heap(gpu, oracle, m, s, k, cov):
    # `mash sketch -r -m m` (MinHashHeap.cpp:96-144, pinned to the reference's object code in tests/test_oracle_vs_ref.py): a hash
    # enters the sketch at its m-th occurrence.  Hash set, multiplicities (incl. the top-of-heap quirk, now on the m-th
    # occurrence) and units that end with fewer than s qualified hashes (low coverage: exact re-run up to keep-all).
    p = gpu.params(k=k, s=s, min_copies=m)
    po = oracle.params(k=k)
    units = [_reads(300 + 7 * u + m + s, 20_000 + 1000 * u, 200 * cov) for u in range(3)]
    recs = [r for u in units for r in u]
    uor = [u for u, rs in enumerate(units) for _ in rs]
    out = gpu.sketch(recs, p, unit_of_record=uor, n_units=3, counts=True)
    plain = gpu.sketch(recs, gpu.params(k=k, s=s), unit_of_record=uor, n_units=3)
    for u, rs in enumerate(units):
        oh, oc, _ = oracle.sketch_unit_m(rs, po, s=s, min_copies=m, counts=True)
        assert_sketch_equal(out, u, oh)
        assert np.array_equal(out[3][u, :out[1][u]], oc)
    assert any(not np.array_equal(out[0][u, :out[1][u]], plain[0][u, :plain[1][u]]) for u in range(3))     # the filter really bites


@pytest.mark.parametrize("wave_bytes", [None, "300000"])
def test_caller_packed_stream_equals_ascii_batch(gpu, oracle, monkeypatch, wave_bytes):
    # mashgpu_sketch_batch_packed: the caller keeps its collection 2-bit packed (+ invalid runs, the format of mashgpu_host_pack)
    # and sketches units of that stream; many waves (the 32-position alignment of a wave's first unit is the delicate part)
    if wave_bytes:
        monkeypatch.setenv("MASHGPU_WAVE_BYTES", wave_bytes)
        monkeypatch.setenv("MASHGPU_WAVE_UNITS", "2")
    p = gpu.params(k=21, s=300)
    po = oracle.params(k=21)
    recs, uor = [], []
    for u in range(9):
        for r in range(1 + u % 3):
            recs.append(bytes(synth_genome(2000 + 10 * u + r, 60_000 + 7919 * u + 13 * r, n_runs=u % 2, lower_frac=0.02)))
            uor.append(u)
    recs.append(b"ACGTNACGT"); uor.append(9)                       # a unit without any k-mer
    codes, runs, starts = gpu.host_pack(recs, p, threads=3)
    unit_first = [uor.index(u) for u in range(10)]
    unit_start = np.array([starts[i] for i in unit_first] + [starts[-1]], np.uint64)
    h, n, c = gpu.sketch_packed(codes, int(starts[-1]), runs, unit_start, p, counts=True)
    ref = gpu.sketch(recs, p, unit_of_record=uor, n_units=10, counts=True)
    assert np.array_equal(n, ref[1]) and np.array_equal(h, ref[0]) and np.array_equal(c, ref[3])
    for u in (0, 4, 8):
        oh, _, _ = oracle.sketch_unit([r for r, x in zip(recs, uor) if x == u], po, s=300)
        assert np.array_equal(h[u, :n[u]], oh)
    assert n[9] == 0


@pytest.mark.parametrize("m,c,s,n_reads,glen", [(1, 3.0, 300, 60_000, 300_000), (2, 4.0, 200, 50_000, 200_000), (1, 1e9, 300, 30_000, 400_000),
                                               (3, 2.5, 100, 45_000, 150_000), (1, 1.5, 1000, 50_000, 1_000_000), (1, 0.0, 300, 5_000, 100_000)])
def test_reads_mode_target_coverage_stop_is_exact(gpu, oracle, m, c, s, n_reads, glen):
    # `mash sketch -r -m m -c c`: the sketch is the heap as it stood after the first read that brought the average multiplicity
    # to c (Sketch.cpp:1258-1262) -- order dependent.  The engine finds that read exactly (position bands bounded by exact
    # prefix sketches, events replayed through the heap logic on the device); oracle pinned to the reference's heap object code
    # in tests/test_oracle_vs_ref.py.  Several bands (streams above 2^21 positions), early and late stops, no stop at all.
    p = gpu.params(k=21, s=s, min_copies=m, target_cov=c)
    po = oracle.params(k=21)
    reads = _reads(4000 + m + s, glen, n_reads, err=0.004)
    reads[7] = b"ACGT"                                       # shorter than k: skipped, not counted as used
    h, cnt, used = gpu.sketch_reads(reads, p, counts=True)
    oh, oc, _, ou = oracle.sketch_unit_mc(reads, po, s=s, min_copies=m, target_cov=c, counts=True)
    assert used == ou
    assert np.array_equal(h, oh) and np.array_equal(cnt, oc)
    if 0 < c < 100:
        assert 0 < used < n_reads - 1                        # the stop really happened inside the stream
    else:
        assert used == n_reads - 1
