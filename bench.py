#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200-native MinHash engine.

Contract (see the task statement): `python bench.py --gpus N --steps K --warmup W` prints ONE JSON line on rank 0.

  metric   Gbp/s sketched on BASELINE.json configs[1]: 10 000 synthetic 5 Mbp genomes, k=21, s=1000 (per GPU; weak
           scaling: every rank sketches its own 10 000 genomes, no data-path collective -- sketching shards by record).
           A "step" is one pass of hot path 1 (scan -> hash -> bottom-s) over the whole batch, inputs resident in HBM.
  e2e      the same metric through mashgpu_sketch_batch with HOST (pinned) buffers: H2D of every genome and D2H of the
           sketches are inside the timed region.
  dist     (extra object) sketch-pairs/s of hot path 2 on configs[2]: all-vs-all of 100 000 synthetic s=1000 sketches
           (10^10 ordered pairs, dense numer/denom/distance/p-value/pass materialised in HBM tile by tile); at N>1 the
           reference axis is sharded per rank and the query sketches are NCCL-broadcast from their owners.  The timed run
           uses the engine's default (tile prefilter + merge + dense p-value pass, results identical to merging every
           pair); `prefilter` reports how many (query, tile) combinations reached the merge, `side_measurements` the
           rate with the prefilter off and with the sketches in random order, `triangle` the `mash triangle` enumeration.
  screen   (extra object) Gbp/s of hot path 3 on configs[3]: 100 000-sketch reference table, 50 M 150 bp reads sampled
           from 50 of the configs[1] genomes (their sketches are in the table), chunks resident in HBM.
  roofline the scan kernel against the measured HBM peak (algorithmic bytes = 1 B/base of ASCII input), plus the
           integer-issue fraction that actually bounds it (DESIGN.md).
  dist5    (extra object) BASELINE.json configs[4]: all-vs-all of 1 000 000 s=1000 sketches (10^12 ordered pairs), reference axis
           sharded over the ranks, dictionary built by the sharded sample sort (mash_b200/shard.py), `-d 0.05` pass list returned
           to the host tile by tile.  ONE pass, timed from the raw hashes to the last list on the host: dictionary build, exchange
           and every kernel are inside the figure.
  cpu_baseline / --impl reference: the reference's own hash+heap object code (oracle/_ref) on the host cores the process
           may use (the faster of one thread per usable CPU -- cgroup quota -- and one per visible CPU; both reported), input
           in memory; `with_fasta_parse` = the same with the reference's kseq.h parser reading FASTA files from tmpfs;
           `.dist` = compare / compareSketches (CommandDistance.cpp:195-232, 306-448 restated in oracle/) over 4096-pair jobs of
           a 4000 x 4000 subset; `.screen` = hashSequence (CommandScreen.cpp:484-599) on 10^6 reads with the reference's own
           hash, heap and robin_hood table code.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

K, S, SEED = 21, 1000, 42
GENOME_LEN = 5_000_000
N_GENOMES = 10_000
N_SKETCHES = 100_000
SCAN_INSTR_PER_KMER = None   # filled from profiles/ when known (see DESIGN.md); used for the int-issue fraction


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--units", type=int, default=N_GENOMES, help="genomes per rank per step (default: the BASELINE config; lower only for profiling)")
    ap.add_argument("--genome-len", type=int, default=GENOME_LEN)
    ap.add_argument("--sketches", type=int, default=N_SKETCHES, help="sketches in the dist workload (default: the BASELINE config)")
    ap.add_argument("--e2e-units", type=int, default=0, help="genomes per e2e step (0 = as many of --units as pinned host memory allows)")
    ap.add_argument("--reads", type=int, default=50_000_000, help="150 bp reads in the screen workload (default: the BASELINE config)")
    ap.add_argument("--sketches5", type=int, default=1_000_000, help="sketches in the configs[4] dist workload (dist5)")
    ap.add_argument("--skip-dist5", action="store_true")
    ap.add_argument("--skip-dist", action="store_true")
    ap.add_argument("--skip-screen", action="store_true")
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-cli", action="store_true")
    ap.add_argument("--cli-files", type=int, default=1000, help="FASTA files in the file -> .msh side measurement of the host shim")
    ap.add_argument("--cli-dist-sketches", type=int, default=6000, help="sketches in the `mash dist` wall-clock side measurement of the host shim")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed sketch step returned on rank 0 to DIR/*.npy (see dump_sketch_outputs)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_UNITS = 2048       # sketches whose hashes --dump-outputs writes: 2048 x 1000 hashes x 2 halves x 8 B = 33 MB


def dump_sketch_outputs(out_dir, d_hashes, d_n):
    """--dump-outputs: the result of the last timed sketch step, as float64 .npy files that hold every value exactly, so that two
    builds can be compared output for output.  sketch_n_hashes = hashes in each unit's sketch (all units); for a fixed, seeded
    sample of units (sketch_units, ascending), sketch_hashes_hi / _lo = the high and low 32 bits of their hashes (a uint64 does
    not fit a float64).  Positions past a unit's count hold no result and are written as 0."""
    os.makedirs(out_dir, exist_ok=True)
    n = d_n.cpu().numpy().astype(np.int64)
    units = np.sort(np.random.Generator(np.random.PCG64(7)).choice(n.size, min(n.size, DUMP_UNITS), replace=False))
    h = d_hashes.cpu().numpy().view(np.uint64)[units]
    h[np.arange(h.shape[1])[None, :] >= n[units][:, None]] = 0
    np.save(os.path.join(out_dir, "sketch_units.npy"), units.astype(np.float64))
    np.save(os.path.join(out_dir, "sketch_n_hashes.npy"), n.astype(np.float64))
    np.save(os.path.join(out_dir, "sketch_hashes_hi.npy"), (h >> np.uint64(32)).astype(np.float64))
    np.save(os.path.join(out_dir, "sketch_hashes_lo.npy"), (h & np.uint64(0xFFFFFFFF)).astype(np.float64))


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)), "measured"
        except Exception:
            pass
    return {"hbm_gbs": 6650.0, "sm_max_mhz": 1965.0}, "fallback"


class ClockSampler:
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe)."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown," \
        "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "200", "-i", str(index)],
                                      stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if self.p is None:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [l.strip().split(", ") for l in open(self.f.name) if l.strip()]
        os.unlink(self.f.name)
        sm, reasons = [], set()
        for r in rows:
            if len(r) < 9:
                continue
            try:
                sm.append(float(r[1])); out["sm_max_mhz"] = float(r[2])
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[5:9]):
                if v.strip().lower() == "active":
                    reasons.add(name)
        if sm:
            out["sm_mhz"] = float(np.median(sm))
        out["reasons"] = sorted(reasons)
        out["samples"] = len(sm)
        return out


# ------------------------------------------------------------------------------------------------------------------
# synthetic data (device side, torch is plumbing only)
# ------------------------------------------------------------------------------------------------------------------
def make_genomes_device(torch, dev, n_units, genome_len, seed):
    """Flat stream: n_units genomes of genome_len iid uniform ACGT bytes, one 0 separator after each; every 10th genome
    gets 20 N-runs (length U[1,1000]) and 5% lower-case soft-masking (SURVEY.md 8(d) Config 2)."""
    span = genome_len + 1
    total = n_units * span
    stream = torch.empty(total + 64, dtype=torch.uint8, device=dev)
    stream[total:] = 0
    lut = torch.tensor(list(b"ACGT"), dtype=torch.uint8, device=dev)
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    chunk_units = max(1, (1 << 28) // span)
    for u0 in range(0, n_units, chunk_units):
        u1 = min(n_units, u0 + chunk_units)
        idx = torch.randint(0, 4, ((u1 - u0) * span,), generator=g, device=dev, dtype=torch.uint8)
        view = stream[u0 * span:u1 * span]
        view.copy_(lut[idx.long()])
        del idx
    stream[:total].view(n_units, span)[:, genome_len] = 0
    rng = np.random.Generator(np.random.PCG64(seed))
    for u in range(0, n_units, 10):
        base = u * span
        starts = rng.integers(0, genome_len, 20)
        lens = rng.integers(1, 1001, 20)
        for a, l in zip(starts, lens):
            b = min(genome_len, int(a) + int(l))
            stream[base + int(a):base + b] = ord("N")
        m = torch.rand(genome_len, generator=g, device=dev) < 0.05
        stream[base:base + genome_len] |= (m.to(torch.uint8) * 0x20)
        del m
    unit_start = np.arange(n_units + 1, dtype=np.uint64) * np.uint64(span)
    return stream, unit_start


def make_sketches_device(torch, dev, n, s, seed, n_families=100, length=5_000_000):
    """SURVEY.md 8(d) Config 3: family base sets of sorted distinct draws in [0, 2^64 s/L); members keep a fraction j of the
    base entries and redraw the rest; lengths U[4e6, 6e6]."""
    g = torch.Generator(device=dev)
    g.manual_seed(seed)
    hi = int(2 ** 64 * s / length)
    per = (n + n_families - 1) // n_families
    H = torch.empty((n, s), dtype=torch.int64, device=dev)
    jac = [1.0, 0.98, 0.95, 0.9, 0.8, 0.5, 0.1, 0.0]
    for f in range(n_families):
        r0, r1 = f * per, min(n, (f + 1) * per)
        if r0 >= r1:
            break
        m = r1 - r0
        base = torch.randint(0, hi, (2 * s,), generator=g, device=dev, dtype=torch.int64)
        fresh = torch.randint(0, hi, (m, 2 * s), generator=g, device=dev, dtype=torch.int64)
        keep_p = torch.tensor(jac, device=dev)[torch.randint(0, len(jac), (m,), generator=g, device=dev)]
        keep = torch.rand((m, 2 * s), generator=g, device=dev) < keep_p[:, None]
        v = torch.where(keep, base[None, :].expand(m, -1), fresh)
        v, _ = torch.sort(v, dim=1)
        # make strictly increasing (duplicates are vanishingly rare in a 2^51 range; bump them)
        dup = torch.zeros_like(v, dtype=torch.bool)
        dup[:, 1:] = v[:, 1:] <= v[:, :-1]
        v = v + torch.cumsum(dup.to(torch.int64), dim=1)
        H[r0:r1] = v[:, :s]
    N = torch.full((n,), s, dtype=torch.int32, device=dev)
    L = torch.randint(4_000_000, 6_000_000, (n,), generator=g, device=dev, dtype=torch.int64)
    return H, N, L


# ------------------------------------------------------------------------------------------------------------------
# CPU baseline (reference object code on host cores)
# ------------------------------------------------------------------------------------------------------------------
def host_genomes(n_units, genome_len, seed):
    """configs[1] genomes in host memory: iid uniform ACGT; every 10th with 20 N-runs (U[1,1000]) and 5 % lower case."""
    rng = np.random.Generator(np.random.PCG64(seed))
    acgt = np.frombuffer(b"ACGT", np.uint8)
    out = []
    for u in range(n_units):
        g = acgt[rng.integers(0, 4, genome_len, dtype=np.uint8)]
        if u % 10 == 0:
            for a, l in zip(rng.integers(0, genome_len, 20), rng.integers(1, 1001, 20)):
                g[int(a):min(genome_len, int(a) + int(l))] = ord("N")
            g[rng.random(genome_len) < 0.05] |= 0x20
        out.append(g)
    return out


def host_sketches(n, s, seed, n_families, length=5_000_000):
    """The configs[2] generator (make_sketches_device) in numpy, for the CPU arms."""
    rng = np.random.Generator(np.random.PCG64(seed))
    hi = int(2 ** 64 * s / length)
    per = (n + n_families - 1) // n_families
    H = np.empty((n, s), np.uint64)
    jac = np.array([1.0, 0.98, 0.95, 0.9, 0.8, 0.5, 0.1, 0.0])
    for f in range(n_families):
        r0, r1 = f * per, min(n, (f + 1) * per)
        if r0 >= r1:
            break
        m = r1 - r0
        base = rng.integers(0, hi, 2 * s, dtype=np.uint64)
        fresh = rng.integers(0, hi, (m, 2 * s), dtype=np.uint64)
        keep = rng.random((m, 2 * s)) < jac[rng.integers(0, jac.size, m)][:, None]
        v = np.sort(np.where(keep, base[None, :], fresh), axis=1)
        dup = np.zeros(v.shape, bool)
        dup[:, 1:] = v[:, 1:] <= v[:, :-1]
        v = v + np.cumsum(dup, axis=1, dtype=np.uint64)
        H[r0:r1] = v[:, :s]
    N = np.full(n, s, np.uint32)
    L = rng.integers(4_000_000, 6_000_000, n).astype(np.uint64)
    return H, N, L


def cpu_dist_rate(threads, n_sub=4000, seed=55):
    """compare (CommandDistance.cpp:306-334) over the reference's <= 4096-pair jobs (:195-232), one job per pool thread at a
    time, on an n_sub x n_sub subset of the configs[2] generator.  compareSketches / pValue are the oracle's restatement
    (CommandDistance.cpp does not compile here: GSL/Boost and the capnp header are absent).  Returns (pairs/s, seconds)."""
    import ctypes as C
    from concurrent.futures import ThreadPoolExecutor
    from oracle.pyoracle import Oracle, PairOutput, u64p, u32p
    orc = Oracle()
    H, N, L = host_sketches(n_sub, S, seed, n_families=max(1, n_sub // 100))
    out = (PairOutput * (n_sub * n_sub))()
    rows_per_job = max(1, 4096 // n_sub)
    ks = 4.0 ** K

    def job(q0):
        orc.lib.mo_compare_all(out, H.ctypes.data_as(u64p), N.ctypes.data_as(u32p), L.ctypes.data_as(u64p), n_sub, S,
                               H.ctypes.data_as(u64p), N.ctypes.data_as(u32p), L.ctypes.data_as(u64p), n_sub, S,
                               S, K, ks, 1.0, 1.0, q0, min(n_sub, q0 + rows_per_job))

    t0 = time.perf_counter()
    with ThreadPoolExecutor(threads) as ex:
        list(ex.map(job, range(0, n_sub, rows_per_job)))
    dt = time.perf_counter() - t0
    return n_sub * n_sub / dt, dt


def cpu_screen_rate(threads, n_reads=1_000_000, n_table=10_000, seed=66):
    """hashSequence (CommandScreen.cpp:484-599) on n_reads 150 bp reads in 1 MiB '*'-joined chunks (:224-262), the reference's
    own getHash / MinHashHeap object code and its robin_hood table type (oracle/_ref), `threads` workers.  The table holds
    n_table synthetic sketches plus the sketches of the 4 genomes the reads are sampled from.  Returns (Gbp/s, seconds, kind)."""
    from oracle.pyoracle import Oracle, RefLib
    if not RefLib.available():
        return None
    ref = RefLib()
    p = Oracle().params(k=K, seed=SEED)
    H, N, L = host_sketches(n_table, S, seed, n_families=max(1, n_table // 1000))
    src = host_genomes(4, 2_000_000, seed + 1)
    sk, sk_n = ref.sketch_many(src, p, s=S, threads=min(4, threads))
    keys = np.unique(np.concatenate([H.reshape(-1), sk.reshape(-1)]))
    rng = np.random.Generator(np.random.PCG64(seed + 2))
    pool = np.concatenate(src)
    starts = rng.integers(0, pool.size - 150, n_reads)
    reads = pool[starts[:, None] + np.arange(150)[None, :]]
    err = rng.random(reads.shape) < 0.005
    reads[err] = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, int(err.sum()))]
    reads[rng.random(reads.shape) < 0.001] = ord("N")
    joined = np.concatenate([np.full((n_reads, 1), ord("*"), np.uint8), reads], axis=1).reshape(-1)
    per_chunk = (1 << 20) // 151 * 151
    chunks = [joined[o:o + per_chunk] for o in range(0, joined.size, per_chunk)]
    t = ref.screen_table(keys)
    try:
        t0 = time.perf_counter()
        ref.screen_many(t, chunks, p, s=S, threads=threads)
        dt = time.perf_counter() - t0
    finally:
        ref.screen_table_free(t)
    return n_reads * 150 / dt / 1e9, dt, "reference"


WORKLOAD_SKETCH = ("configs[1]: {units} synthetic genomes x {glen} bp per GPU, k=%d s=%d seed=%d, canonical, ASCII input "
                   "(every 10th genome with 20 N-runs and 5%% lower case)" % (K, S, SEED))


def cpu_arms(threads):
    """dist and screen CPU arms (bounded samples), as sub-objects of cpu_baseline."""
    d_rate, d_dt = cpu_dist_rate(threads)
    out = {"dist": {"value": d_rate, "unit": "pairs/s", "cores": threads, "kind": "port",
                    "sample": f"4000 x 4000 sketches of the configs[2] generator (s={S}), compare over <= 4096-pair jobs on {threads} threads, {d_dt:.1f} s wall; "
                              "compareSketches/pValue restated in oracle/mash_oracle.c (CommandDistance.cpp needs GSL/Boost, absent here)"}}
    sc = cpu_screen_rate(threads)
    if sc is not None:
        out["screen"] = {"value": sc[0], "unit": "Gbp/s", "cores": threads, "kind": sc[2],
                         "sample": f"10^6 synthetic 150 bp reads in 1 MiB chunks against a 10 004-sketch table on {threads} threads, {sc[1]:.1f} s wall; "
                                   "reference getHash/MinHashHeap object code and robin_hood table (oracle/_ref), restated hashSequence loop"}
    return out


def usable_cpus():
    """CPUs this process may really use: visible count, affinity mask and the container's CPU quota (cgroup v2 cpu.max)."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except (AttributeError, OSError):
        pass
    try:
        quota, period = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if quota != "max":
            n = min(n, max(1, -(-int(quota) // int(period))))
    except (OSError, ValueError):
        pass
    return n


def best_cpu_sketch_rate(n_units, genome_len, seed=123):
    """The CPU arm at its best on this host: once with one thread per usable CPU (the quota), once with one per visible CPU --
    oversubscribing a quota can go either way -- and the faster of the two counts.  Returns (Gbp/s, kind, seconds, threads, tried)."""
    tried = {}
    for th in sorted({usable_cpus(), os.cpu_count() or 1}):
        r, kind, dt = cpu_sketch_rate(n_units, genome_len, th, seed)
        tried[th] = (r, kind, dt)
    th = max(tried, key=lambda t: tried[t][0])
    r, kind, dt = tried[th]
    return r, kind, dt, th, {str(t): round(v[0], 4) for t, v in tried.items()}


def cpu_sketch_rate(n_units, genome_len, threads, seed=123):
    """Times the reference's hash + MinHashHeap object code (oracle/_ref, restated scan loop) on `threads` host threads.
    Falls back to the plain-C oracle port when oracle/_ref is absent. Returns (Gbp/s, kind, seconds)."""
    from oracle.pyoracle import Oracle, RefLib
    orc = Oracle()
    p = orc.params(k=K, seed=SEED)
    seqs = host_genomes(n_units, genome_len, seed)
    if RefLib.available():
        ref = RefLib()
        t0 = time.perf_counter()
        ref.sketch_many(seqs, p, s=S, threads=threads)
        dt = time.perf_counter() - t0
        kind = "reference"
    else:
        from concurrent.futures import ThreadPoolExecutor
        t0 = time.perf_counter()
        with ThreadPoolExecutor(threads) as ex:
            list(ex.map(lambda q: orc.sketch_unit([q], p, s=S), seqs))
        dt = time.perf_counter() - t0
        kind = "port"
    return n_units * genome_len / dt / 1e9, kind, dt


def cpu_sketch_rate_from_files(n_units, genome_len, threads, seed=321):
    """The CPU arm with the parse included, as `mash sketch -p threads *.fna` runs it: uncompressed 70-column FASTA files on
    tmpfs, the reference's own kseq.h parser + hash + heap object code (oracle/_ref).  Returns (Gbp/s, seconds) or None."""
    from oracle.pyoracle import Oracle, RefLib
    if not RefLib.available():
        return None
    ref = RefLib()
    if not hasattr(ref.lib, "ref_sketch_files"):
        return None
    p = Oracle().params(k=K, seed=SEED)
    seqs = host_genomes(n_units, genome_len, seed)
    base = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else None
    with tempfile.TemporaryDirectory(dir=base) as d:
        paths = write_fasta_files(seqs, d)
        t0 = time.perf_counter()
        ref.sketch_files(paths, p, s=S, threads=threads)
        dt = time.perf_counter() - t0
    return n_units * genome_len / dt / 1e9, dt


def write_fasta_files(seqs, d):
    """uncompressed 70-column FASTA, one file per genome"""
    paths = []
    for i, q in enumerate(seqs):
        a = np.frombuffer(q, np.uint8)
        full = (a.size // 70) * 70
        lines = np.concatenate([a[:full].reshape(-1, 70), np.full((full // 70, 1), 10, np.uint8)], axis=1).tobytes()
        path = os.path.join(d, f"g{i}.fna")
        with open(path, "wb") as f:
            f.write(b">g%d synthetic\n" % i + lines + a[full:].tobytes() + b"\n")
        paths.append(path)
    return paths


def cli_sketch_rate(n_files, genome_len, threads, seed=4321):
    """File -> .msh wall clock of the host shim: `mash sketch -p threads -o out -l list` on n_files uncompressed FASTA files on tmpfs
    (process start, CUDA context, parse, sketch, .msh write all inside).  Returns dict or None."""
    mash = os.path.join(ROOT, "mash_b200", "host", "mash")
    base = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else None
    if not os.path.exists(mash) or base is None:
        return None
    try:
        st = os.statvfs(base)
        room = st.f_bavail * st.f_frsize
    except OSError:
        return None
    n_files = int(min(n_files, max(0, room // 2) // (genome_len + genome_len // 70 + 64)))
    if n_files < 8:
        return None
    with tempfile.TemporaryDirectory(dir=base) as d:
        paths = []
        for c0 in range(0, n_files, 64):
            seqs = host_genomes(min(64, n_files - c0), genome_len, seed + c0)
            sub = os.path.join(d, f"b{c0}")
            os.mkdir(sub)
            paths += write_fasta_files(seqs, sub)
        lst = os.path.join(d, "list.txt")
        open(lst, "w").write("\n".join(paths) + "\n")
        out = os.path.join(d, "out")
        t0 = time.perf_counter()
        pr = subprocess.run([mash, "sketch", "-p", str(threads), "-o", out, "-l", lst], capture_output=True, text=True, env=dict(os.environ, MASHGPU_TRACE="1"))
        dt = time.perf_counter() - t0
        sys.stderr.write("cli trace:\n" + "\n".join(l for l in (pr.stderr or "").splitlines() if l.startswith("[mash")) + "\n")
        if pr.returncode != 0 or not os.path.exists(out + ".msh"):
            return {"error": (pr.stderr or "")[-300:]}
        size = os.path.getsize(out + ".msh")
    return {"value": n_files * genome_len / dt / 1e9, "unit": "Gbp/s", "seconds": dt, "files": n_files, "threads": threads, "msh_bytes": size,
            "command": f"mash sketch -p {threads} -o out -l list.txt  ({n_files} uncompressed 70-column FASTA files of {genome_len} bp on tmpfs)",
            "note": "wall clock of the whole process: start-up and CUDA context creation, FASTA parse on the host threads, sketching on the GPU, "
                    ".msh (Cap'n Proto) write"}


def cli_dist_rate(n_sketches, contig_len, threads, seed=8765):
    """Wall clock of `mash dist -p threads x.msh x.msh > /dev/null` through the host shim (process start, CUDA context, .msh load,
    dictionary, kernels, D2H, and the text of every pair -- one line per pair as the reference prints them).  The sketches come from
    `mash sketch -l list` over n_sketches small FASTA files.  Never raises: returns a dict with an "error" key instead."""
    try:
        mash = os.path.join(ROOT, "mash_b200", "host", "mash")
        base = "/dev/shm" if os.path.isdir("/dev/shm") and os.access("/dev/shm", os.W_OK) else None
        if not os.path.exists(mash) or base is None:
            return None
        with tempfile.TemporaryDirectory(dir=base) as d:
            paths = []
            for c0 in range(0, n_sketches, 1000):
                seqs = host_genomes(min(1000, n_sketches - c0), contig_len, seed + c0)
                sub = os.path.join(d, f"b{c0}")
                os.mkdir(sub)
                paths += write_fasta_files(seqs, sub)
            lst = os.path.join(d, "list.txt")
            with open(lst, "w") as f:
                f.write("\n".join(paths) + "\n")
            out = os.path.join(d, "x")
            pr = subprocess.run([mash, "sketch", "-p", str(threads), "-o", out, "-l", lst], capture_output=True, text=True, timeout=300)
            if pr.returncode != 0 or not os.path.exists(out + ".msh"):
                return {"error": "sketch: " + (pr.stderr or "")[-300:]}
            res = {}
            for label, th in (("threads_1", 1), (f"threads_{threads}", threads)):
                with open(os.devnull, "wb") as null:
                    t0 = time.perf_counter()
                    pr = subprocess.run([mash, "dist", "-p", str(th), out + ".msh", out + ".msh"], stdout=null, stderr=subprocess.PIPE, text=True, timeout=600)
                    dt = time.perf_counter() - t0
                if pr.returncode != 0:
                    return {"error": "dist: " + (pr.stderr or "")[-300:]}
                res[label] = {"seconds": dt, "pairs_per_s": n_sketches * n_sketches / dt}
                if th == threads:
                    break
        res.update({"pairs": n_sketches * n_sketches, "unit": "pairs/s, wall clock of the whole process",
                    "command": f"mash dist -p T x.msh x.msh > /dev/null  ({n_sketches} sketches, s=1000: one output line per pair, {n_sketches * n_sketches} lines)",
                    "note": "process start, CUDA context, .msh load, dictionary, kernels, D2H and the formatting of every line (host/fastout.hpp) inside; "
                            "the reference prints ~1e6 lines/s from one thread (cout << ... << endl per pair)"})
        return res
    except Exception as e:          # a side measurement must not take the bench line down
        return {"error": repr(e)[:300]}


def run_reference_arm(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    n_units = max(128, 2 * (os.cpu_count() or 1))
    rates = []
    cores, tried, kind = 1, {}, "port"
    for i in range(args.warmup + args.steps):
        r, kind, dt, cores, tried = best_cpu_sketch_rate(n_units, args.genome_len, seed=1000 + i)
        if i >= args.warmup:
            rates.append((r, dt))
    value = float(np.mean([r for r, _ in rates]))
    arms = cpu_arms(cores)
    line = {
        "impl": "reference", "metric": "Gbp_per_s_sketched", "value": value, "unit": "Gbp/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": float(np.mean([dt for _, dt in rates]) * 1e3),
        "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64", "data": "synthetic",
        "config": {"workload": WORKLOAD_SKETCH.format(units=args.units, glen=args.genome_len),
                   "k": K, "s": S, "units_per_gpu": args.units, "genome_len": args.genome_len,
                   "sample": f"{n_units} genomes of the batch per step (CPU arm: bounded sample of the same workload)"},
        "cpu_baseline": {"value": value, "unit": "Gbp/s", "cores": cores, "kind": kind,
                         "visible_cpus": os.cpu_count(), "usable_cpus": usable_cpus(), "gbp_per_s_by_threads": tried,
                         "sample": f"{n_units} genomes x {args.genome_len} bp per step, one job per genome on {cores} threads (the faster of one "
                                   "thread per usable CPU and one per visible CPU); "
                                   "reference MurmurHash3/hash/MinHashHeap object code, restated addMinHashes loop, in-memory input (no FASTA parse)"},
        "e2e": {"value": value, "unit": "Gbp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "dist": dict(arms["dist"], metric="sketch_pairs_per_s"),
        "screen": dict(arms["screen"], metric="Gbp_per_s_screened") if "screen" in arms else None,
    }
    line["cpu_baseline"]["dist"] = arms["dist"]
    line["cpu_baseline"]["screen"] = arms.get("screen")
    emit_json_line(line)


# ------------------------------------------------------------------------------------------------------------------
def emit_json_line(line):
    """The contract is ONE JSON line on stdout; libraries (NCCL's version banner, torchrun) also write to fd 1, so main()
    points fd 1 at stderr for the whole run and the result line is written to the saved real stdout."""
    data = (json.dumps(line) + "\n").encode()
    fd = _REAL_STDOUT if _REAL_STDOUT is not None else 1
    os.write(fd, data)


_REAL_STDOUT = None


def main():
    global _REAL_STDOUT
    args = parse_args()
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        return run_reference_arm(args)

    import torch
    import mash_b200

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    dist_on = world > 1
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU path); use --impl reference for the CPU arm")
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if dist_on:
        import torch.distributed as td
        td.init_process_group("nccl", device_id=dev)

    def barrier():
        if dist_on:
            td.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if not dist_on:
            return x
        t = torch.tensor([x], dtype=torch.float64, device=dev)
        td.all_reduce(t, op=td.ReduceOp.MAX)
        return float(t.item())

    # host side of a rank: the CPUs (and with them the memory) of the NUMA node next to its GPU -- before any pinned allocation
    from mash_b200.shard import bind_to_gpu_numa_node
    cpus_before_binding = usable_cpus()
    affinity_before_binding = os.sched_getaffinity(0)
    numa = None if os.environ.get("MASHGPU_BENCH_NUMA", "1") == "0" else bind_to_gpu_numa_node(local)
    # host packer threads of the hybrid feed path: the ranks of one node share its CPUs (an equal share of what the process may
    # use, counted before the binding narrowed the affinity mask to one socket)
    local_world_n = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
    os.environ.setdefault("MASHGPU_PACK_THREADS", str(max(1, cpus_before_binding // max(1, local_world_n) - 1)))
    # feed of the drop-in sketch call: with 8 ranks on a 2-socket host the host memory system is the bound, and the packer's own
    # reads and writes (1.25 B per base it packs) cost more than the PCIe bytes they save -- measured at N = 8 with the ranks bound
    # to their sockets: ASCII copies only 397 Gbp/s, both producers 294 (profiles/r02_e2e_n8_ab.json); with 1-2 ranks per host the
    # two producers win (81 against 52 Gbp/s at N = 1).  The library's default stays "both"; the launcher decides per deployment.
    feed_note = None
    if local_world_n >= 8 and "MASHGPU_HOST_PACK" not in os.environ:
        os.environ["MASHGPU_HOST_PACK"] = "0"
        feed_note = f"ASCII DMA only: chosen by bench.py for {local_world_n} ranks per host (host memory bound; the library default is the hybrid feed)"
    eng = mash_b200.Engine(local)
    eng_sm_count = torch.cuda.get_device_properties(local).multi_processor_count
    p = eng.params(k=K, s=S, seed=SEED)
    peaks, peak_kind = measured_peaks()
    W, Ksteps = args.warmup, args.steps
    # a non-default torch stream: its handle is passed to the C ABI so that torch's CUDA events bracket our kernels
    st = torch.cuda.Stream(device=dev)
    torch.cuda.set_stream(st)
    st_ptr = st.cuda_stream
    assert st_ptr != 0

    # ---------------- hot path 1: sketch, inputs resident in HBM -------------------------------------------------
    n_units, glen = args.units, args.genome_len
    stream, unit_start = make_genomes_device(torch, dev, n_units, glen, seed=20260923 + rank)
    d_hashes = torch.zeros((n_units, S), dtype=torch.int64, device=dev)
    d_n = torch.zeros(n_units, dtype=torch.int32, device=dev)
    bases_per_step = n_units * glen

    def sketch_step():
        eng.sketch_stream_dev(p, stream.data_ptr(), unit_start, d_hashes.data_ptr(), d_n.data_ptr(), stream=st_ptr)

    for _ in range(W):
        sketch_step()
    eng.set_timing(True)
    eng.stats(reset=True)
    barrier()
    sampler = ClockSampler(local) if rank == 0 else None
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(st)
    for _ in range(Ksteps):
        sketch_step()
    e1.record(st)
    barrier()
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    clocks = sampler.stop() if sampler else None
    stats = eng.stats(reset=True)
    eng.set_timing(False)
    ms_per_step = ms_total / Ksteps
    value = world * bases_per_step / (ms_per_step * 1e-3) / 1e9
    scan_ms = stats["scan_kernel_ms"] / max(1, stats["scan_kernel_launches"])
    scan_gbs = bases_per_step * 1.0 / (scan_ms * 1e-3) / 1e9                 # 1 B/base ASCII
    roofline = {"bound": "hbm", "kernel": "scan_kernel<21,canonical>", "achieved": scan_gbs, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                "frac": scan_gbs / peaks["hbm_gbs"], "traffic": None, "peak_source": peak_kind,
                "algorithmic_bytes_per_launch": bases_per_step, "launch_ms": scan_ms,
                "note": "integer-issue bound by the exact MurmurHash3_x64_128 per k-mer, not HBM bound; see int_issue and DESIGN.md 2.4"}
    model_path = os.path.join(ROOT, "profiles", "r01_scan_model.json")
    if os.path.exists(model_path):
        model = json.load(open(model_path))
        # DRAM traffic per launch: bytes/base measured by one `ncu --set full` capture of this kernel, scaled to this launch
        roofline["traffic"] = model["dram_bytes_per_base"] * bases_per_step
        roofline["traffic_source"] = "profiles/r01_scan_kernel_ncu.csv (dram__bytes_read+write per base at 400 units) x bases per launch"
        sm_hz = (clocks or {}).get("sm_mhz") or peaks.get("sm_max_mhz", 1965.0)
        sm_hz *= 1e6
        issue_peak = eng_sm_count * 4 * sm_hz                       # warp instructions / s (1 per SM sub-partition per clock)
        warp_inst = bases_per_step / 32 * model["warp_instructions_per_32_kmers"] / (scan_ms * 1e-3)
        roofline["int_issue"] = {"warp_instructions_per_32_kmers": model["warp_instructions_per_32_kmers"],
                                 "achieved_warp_inst_per_s": warp_inst, "peak_warp_inst_per_s": issue_peak, "frac": warp_inst / issue_peak,
                                 "alu_pipe_frac": warp_inst * model["alu_pipe_share"] / (issue_peak / 2),
                                 "note": "ALU pipe (SHF/LOP3/IADD3/PRMT) issues one warp instruction per 2 clocks per sub-partition; instruction mix from the ncu source page"}
    sanity = {"sketches_full": int((d_n == S).sum().item()), "units": n_units}
    if args.dump_outputs and rank == 0:
        dump_sketch_outputs(args.dump_outputs, d_hashes, d_n)

    # ---------------- e2e: host buffers through mashgpu_sketch_batch --------------------------------------------------
    e2e = None
    if not args.skip_e2e:
        avail = 0
        try:
            for l in open("/proc/meminfo"):
                if l.startswith("MemAvailable"):
                    avail = int(l.split()[1]) * 1024
        except Exception:
            pass
        local_world = int(os.environ.get("LOCAL_WORLD_SIZE", str(world)))
        budget = max(1 << 30, int(avail * 0.35 / max(1, local_world)))
        e2e_units = args.e2e_units or max(1, min(n_units, budget // (glen + 1)))
        span = glen + 1
        host = torch.empty(e2e_units * span, dtype=torch.uint8, pin_memory=True)
        host.copy_(stream[:e2e_units * span])
        torch.cuda.synchronize()
        hnp = host.numpy()
        recs = [hnp[u * span:u * span + glen] for u in range(e2e_units)]
        import ctypes as C
        ptrs = (C.c_void_p * e2e_units)(*[r.ctypes.data for r in recs])
        lens = np.full(e2e_units, glen, np.uint64)
        out_h = torch.empty((e2e_units, S), dtype=torch.int64, pin_memory=True).numpy().view(np.uint64)
        out_n = np.zeros(e2e_units, np.uint32)
        out_len = np.zeros(e2e_units, np.uint64)
        u64p, u32p = C.POINTER(C.c_uint64), C.POINTER(C.c_uint32)

        def e2e_step():
            eng._check(eng.lib.mashgpu_sketch_batch(eng.h, C.byref(p), e2e_units, C.cast(ptrs, C.c_void_p), lens.ctypes.data_as(u64p), None,
                                                    e2e_units, out_h.ctypes.data_as(u64p), None, out_n.ctypes.data_as(u32p), out_len.ctypes.data_as(u64p)))

        for _ in range(W):
            e2e_step()
        barrier()
        t0 = time.perf_counter()
        for _ in range(Ksteps):
            e2e_step()
        torch.cuda.synchronize()
        dt = max_over_ranks(time.perf_counter() - t0)
        same = bool(np.array_equal(out_h[: min(e2e_units, n_units)], d_hashes[:e2e_units].cpu().numpy().view(np.uint64)))
        e2e = {"value": world * e2e_units * glen * Ksteps / dt / 1e9, "unit": "Gbp/s",
               "h2d_bytes_per_step": int(e2e_units * span), "d2h_bytes_per_step": int(e2e_units * (S * 8 + 4)),
               "units_per_step": e2e_units, "ms_per_step": dt / Ksteps * 1e3, "matches_device_path": same,
               "feed": feed_note or {"0": "ASCII DMA only (MASHGPU_HOST_PACK=0)", "1": "host 2-bit packer only (MASHGPU_HOST_PACK=1)"}.get(
                   os.environ.get("MASHGPU_HOST_PACK", ""), "hybrid: ASCII DMA and host 2-bit packer side by side (default)"),
               "api": "mashgpu_sketch_batch (host pinned buffers; H2D + kernels + D2H inside the timed region)"}
        # ---- the same batch from a collection the caller keeps 2-bit packed (mashgpu_sketch_batch_packed): packing is done once,
        # outside the timed region (that is the premise: a cached packed collection); per step 0.25 B/base cross PCIe
        e2e_packed = None
        try:
            total_pos = e2e_units * span
            pk_codes = torch.empty((total_pos + 31) // 32, dtype=torch.int64, pin_memory=True)
            cap_runs = 1 << 22
            pk_runs = torch.empty(2 * cap_runs, dtype=torch.int64, pin_memory=True)
            n_runs = C.c_uint64(0)
            t_pack = time.perf_counter()
            eng._check(eng.lib.mashgpu_host_pack(C.byref(p), e2e_units, C.cast(ptrs, C.c_void_p), lens.ctypes.data_as(u64p), usable_cpus(),
                                                 C.cast(pk_codes.data_ptr(), u64p), C.cast(pk_runs.data_ptr(), u64p), cap_runs, C.byref(n_runs)))
            t_pack = time.perf_counter() - t_pack
            if n_runs.value <= cap_runs:
                ustart = (np.arange(e2e_units + 1, dtype=np.uint64) * np.uint64(span))
                out_h2 = torch.empty((e2e_units, S), dtype=torch.int64, pin_memory=True).numpy().view(np.uint64)

                def packed_step():
                    eng._check(eng.lib.mashgpu_sketch_batch_packed(eng.h, C.byref(p), C.cast(pk_codes.data_ptr(), u64p), total_pos, C.cast(pk_runs.data_ptr(), u64p),
                                                                   n_runs.value, ustart.ctypes.data_as(u64p), e2e_units, out_h2.ctypes.data_as(u64p), None,
                                                                   out_n.ctypes.data_as(u32p)))

                for _ in range(min(W, 2)):
                    packed_step()
                barrier()
                t0 = time.perf_counter()
                for _ in range(Ksteps):
                    packed_step()
                torch.cuda.synchronize()
                dtp = max_over_ranks(time.perf_counter() - t0)
                e2e_packed = {"value": world * e2e_units * glen * Ksteps / dtp / 1e9, "unit": "Gbp/s", "ms_per_step": dtp / Ksteps * 1e3,
                              "h2d_bytes_per_step": int(pk_codes.numel() * 8 + n_runs.value * 16), "d2h_bytes_per_step": int(e2e_units * (S * 8 + 4)),
                              "matches_ascii_path": bool(np.array_equal(out_h2, out_h)), "one_off_pack_seconds": t_pack, "pack_threads": usable_cpus(),
                              "api": "mashgpu_sketch_batch_packed (caller-packed 2-bit stream + invalid runs in pinned host memory; H2D + kernels + D2H inside)"}
            del pk_codes, pk_runs
        except AttributeError:
            e2e_packed = None
        e2e["packed_collection"] = e2e_packed
        del host

    # ---------------- hot path 2: dist ---------------------------------------------------------------------------
    dist_obj = None
    dist5_obj = None
    screen_obj = None
    if not args.skip_dist:
        # configs[3] samples its reads from 50 of the configs[1] genomes: keep those genomes and their sketches for the screen step
        n_src = min(50, n_units)
        screen_src = stream[: n_src * (glen + 1)].clone()
        screen_src_hashes = d_hashes[:n_src].clone()
        del stream
        torch.cuda.empty_cache()
        n_sk = args.sketches
        # every rank owns n_sk/world sketches: its reference shard (resident), and its share of the queries
        shard = (n_sk + world - 1) // world
        H, N, L = make_sketches_device(torch, dev, shard, S, seed=1000 + rank, n_families=max(1, 100 // world))
        if dist_on:
            from mash_b200.shard import sharded_dictionary, DictOps, warm_collectives
            warm_collectives(dev)                 # communicator channel set-up is a process start-up cost, not part of a pass
        torch.cuda.synchronize()
        barrier()
        # ---- one-off work of a job, timed: dictionary build (+ the exchange step at N > 1) ----
        t_open = time.perf_counter()
        enc = None
        if dist_on:
            # exchange step: sample sort of the hashes by hash range (all-to-all) + all-gather of the encoded rows (4 B per hash)
            rows, n_eff, lens_all, counts, dstat = sharded_dictionary(DictOps(eng, st_ptr), H, N, L, S)
            b0 = sum(counts[:rank])
            enc = (rows, n_eff, lens_all)
            job = eng.dist_open_encoded(rows.data_ptr(), n_eff.data_ptr(), lens_all.data_ptr(), rows.shape[0], b0, counts[rank],
                                        sketch_size=S, k=K, kmer_space=p.kmer_space, keepalive=enc)
        else:
            dstat = None
            ref_set = mash_b200._capi._Set(H.data_ptr(), N.data_ptr(), L.data_ptr(), on_device=True, n=H.shape[0], stride=S)
            job = mash_b200._capi.DistJob(eng, ref_set, None, None, None, None, None, S, K, p.kmer_space, 1.0, 1.0)
        torch.cuda.synchronize()
        open_ms = max_over_ranks((time.perf_counter() - t_open) * 1e3)
        n_ref, n_qry = job.n_ref, job.n_qry
        q_tile = max(1, min(n_qry, (1 << 29) // max(1, n_ref)))   # 2^29 pairs = 13.4 GB of dense outputs per launch
        o_numer = torch.empty(q_tile * n_ref, dtype=torch.int32, device=dev)
        o_denom = torch.empty(q_tile * n_ref, dtype=torch.int32, device=dev)
        o_dist = torch.empty(q_tile * n_ref, dtype=torch.float64, device=dev)
        o_p = torch.empty(q_tile * n_ref, dtype=torch.float64, device=dev)
        o_pass = torch.empty(q_tile * n_ref, dtype=torch.uint8, device=dev)

        def dist_step():
            for q0 in range(0, n_qry, q_tile):
                qc = min(q_tile, n_qry - q0)
                job.run_dev(q0, qc, o_numer.data_ptr(), o_denom.data_ptr(), o_dist.data_ptr(), o_p.data_ptr(), o_pass.data_ptr(), stream=st_ptr)

        dW = min(W, 1) if n_ref * n_qry >= 10 ** 9 else W
        barrier()
        e0.record(st)
        dist_step()                               # the first pass of the job (also the first warm-up step)
        e1.record(st)
        barrier()
        first_pass_ms = max_over_ranks(e0.elapsed_time(e1))
        for _ in range(max(0, dW - 1)):
            dist_step()
        eng.set_timing(True); eng.stats(reset=True)
        barrier()
        e0.record(st)
        for _ in range(Ksteps):
            dist_step()
        e1.record(st)
        barrier()
        dms = max_over_ranks(e0.elapsed_time(e1)) / Ksteps
        dstats = eng.stats(reset=True)
        eng.set_timing(False)
        pairs_per_rank = n_ref * n_qry
        total_pairs = pairs_per_rank * world
        last_shared_nonzero = int((o_numer[: min(q_tile, n_qry) * n_ref] > 0).sum().item())
        pf = job.prefilter_stats()

        def one_tile_rate(j, reps=2):
            """pairs/s of this rank on the first query tile only (side measurements: merge-only and shuffled order)."""
            qc = min(q_tile, j.n_qry)
            j.run_dev(0, qc, o_numer.data_ptr(), o_denom.data_ptr(), o_dist.data_ptr(), o_p.data_ptr(), o_pass.data_ptr(), stream=st_ptr)
            torch.cuda.synchronize()
            a0 = torch.cuda.Event(enable_timing=True); a1 = torch.cuda.Event(enable_timing=True)
            a0.record(st)
            for _ in range(reps):
                j.run_dev(0, qc, o_numer.data_ptr(), o_denom.data_ptr(), o_dist.data_ptr(), o_p.data_ptr(), o_pass.data_ptr(), stream=st_ptr)
            a1.record(st); torch.cuda.synchronize()
            return qc * j.n_ref / (a0.elapsed_time(a1) / reps * 1e-3)

        side = {}
        if rank == 0:
            side["first_query_tile_as_timed"] = one_tile_rate(job)
            job.set_prefilter(0)
            side["first_query_tile_merge_every_pair"] = one_tile_rate(job)
            job.set_prefilter(-1)
        tri = None
        if world == 1:
            # `mash triangle` enumeration of the same set (BASELINE configs[2] quotes it: n(n-1)/2 ~ 5e9 unordered pairs)
            job.set_triangle(True)
            dist_step(); torch.cuda.synchronize()
            a0 = torch.cuda.Event(enable_timing=True); a1 = torch.cuda.Event(enable_timing=True)
            a0.record(st); dist_step(); a1.record(st); torch.cuda.synchronize()
            tri_pairs = n_ref * (n_ref - 1) // 2
            tri = {"enumeration": "lower triangle, row i vs rows 0..i-1 (CommandTriangle.cpp:200-214)", "pairs": tri_pairs,
                   "ms": a0.elapsed_time(a1), "pairs_per_s": tri_pairs / (a0.elapsed_time(a1) * 1e-3)}
            job.set_triangle(False)
        dist_obj = {"metric": "sketch_pairs_per_s", "value": total_pairs / (dms * 1e-3), "unit": "pairs/s", "ms_per_step": dms,
                    "steps": Ksteps, "warmup": dW, "pairs_per_step": total_pairs, "enumeration": "all ordered pairs (full Q x R grid)",
                    "workload": f"configs[2]: {n_sk} synthetic s={S} sketches all-vs-all, 100 families stored family by family (SURVEY.md 8d generator); "
                                f"reference axis sharded over {world} rank(s), every rank compares all {n_sk} queries with its shard",
                    "outputs": "dense numer,denom (u32), distance,pvalue (f64), pass (u8) = 25 B/pair written to an HBM tile buffer that is reused per query tile",
                    "algorithm": "tile prefilter (cuckoo filter per 32-reference tile; closed form for pairs without shared hashes) + sorted merge of the "
                                 "rest + dense p-value pass; results identical to merging every pair (tests/test_gpu_dist_prefilter.py)",
                    "prefilter": {"query_tile_combinations_probed": pf["combos_probed"], "sent_to_merge": pf["combos_flagged"],
                                  "fraction_merged": (pf["combos_flagged"] / pf["combos_probed"]) if pf["combos_probed"] else None,
                                  "pairs_merged_from_pair_lists": pf["pairs_from_lists"]},
                    "one_off_ms": open_ms, "first_pass_ms": first_pass_ms,
                    "value_first_pass_incl_one_off": total_pairs / ((open_ms + first_pass_ms) * 1e-3),
                    "one_off": ("dictionary build inside mashgpu_dist_open (radix sort of all hashes)" if not dist_on else
                                "sharded dictionary build: local sort, all-to-all by hash range, ranking, all-to-all back, all-gather of the encoded rows "
                                "(mash_b200/shard.py sharded_dictionary), then mashgpu_dist_open_encoded; wall clock, max over ranks"),
                    "sharded_dictionary": dstat,
                    "kernel_ms_per_step": dstats["dist_kernel_ms"] / Ksteps, "gpu_launches": int(dstats["kernel_launches"]),
                    "pairs_with_shared_hashes_in_last_tile": last_shared_nonzero,
                    "roofline": {"bound": "hbm", "achieved": (total_pairs / world * 25 + (n_ref + n_qry) * S * 4) / (dstats["dist_kernel_ms"] / Ksteps * 1e-3) / 1e9,
                                 "peak": peaks["hbm_gbs"], "unit": "GB/s",
                                 "note": "algorithmic bytes = 25 B/pair written + the rank rows read once; the probe kernel is ALU-pipe bound and the merge "
                                         "kernel shared-memory bound, not HBM bound (DESIGN.md 3.3)"}}
        dist_obj["roofline"]["frac"] = dist_obj["roofline"]["achieved"] / peaks["hbm_gbs"]
        job.close()
        if rank == 0:
            # the same sketches in random order: related sketches no longer sit in the same reference tile, more tiles reach the merge
            perm = torch.randperm(H.shape[0], device=dev, generator=torch.Generator(device=dev).manual_seed(3))
            Hs = H[perm].contiguous(); Ls = L[perm].contiguous()
            sset = mash_b200._capi._Set(Hs.data_ptr(), N.data_ptr(), Ls.data_ptr(), on_device=True, n=Hs.shape[0], stride=S)
            sjob2 = mash_b200._capi.DistJob(eng, sset, None, None, None, None, None, S, K, p.kmer_space, 1.0, 1.0)
            side["first_query_tile_shuffled_order"] = one_tile_rate(sjob2)
            sjob2.set_prefilter(0)
            side["first_query_tile_shuffled_order_merge_every_pair"] = one_tile_rate(sjob2)
            sjob2.close()
            del Hs, Ls, sset
            side["note"] = ("pairs/s of rank 0 on one query tile of its own shard (self comparison), outside the timed region; 'merge_every_pair' = prefilter off "
                            "(the reference's algorithm for every pair)")
        dist_obj["side_measurements"] = side
        dist_obj["triangle"] = tri

        # ---------------- configs[4]: 1 M sketches all-vs-all, one pass from raw hashes to pass lists on the host ----------
        if not args.skip_dist5:
            del o_numer, o_denom, o_dist, o_p, o_pass, enc
            torch.cuda.empty_cache()
            import ctypes as C
            n5 = args.sketches5
            shard5 = (n5 + world - 1) // world
            H5, N5, L5 = make_sketches_device(torch, dev, shard5, S, seed=5000 + rank, n_families=max(1, shard5 // 1000))
            cap5 = 1 << 22
            l_idx = torch.empty(cap5, dtype=torch.int64, pin_memory=True); l_num = torch.empty(cap5, dtype=torch.int32, pin_memory=True)
            l_den = torch.empty(cap5, dtype=torch.int32, pin_memory=True); l_dist = torch.empty(cap5, dtype=torch.float64, pin_memory=True)
            l_pv = torch.empty(cap5, dtype=torch.float64, pin_memory=True)
            max_d5 = 0.05
            eng.set_timing(True); eng.stats(reset=True)
            torch.cuda.synchronize()
            barrier()
            t0 = time.perf_counter()
            if dist_on:
                rows5, neff5, lens5, counts5, dstat5 = sharded_dictionary(DictOps(eng, st_ptr), H5, N5, L5, S)
                job5 = eng.dist_open_encoded(rows5.data_ptr(), neff5.data_ptr(), lens5.data_ptr(), rows5.shape[0], sum(counts5[:rank]), counts5[rank],
                                             sketch_size=S, k=K, kmer_space=p.kmer_space, max_distance=max_d5, max_pvalue=1.0, keepalive=(rows5, neff5, lens5))
            else:
                dstat5 = None
                set5 = mash_b200._capi._Set(H5.data_ptr(), N5.data_ptr(), L5.data_ptr(), on_device=True, n=H5.shape[0], stride=S)
                job5 = mash_b200._capi.DistJob(eng, set5, None, None, None, None, None, S, K, p.kmer_space, max_d5, 1.0)
            torch.cuda.synchronize()
            t_dict = time.perf_counter() - t0
            n_ref5, n_qry5 = job5.n_ref, job5.n_qry
            q_tile5 = max(1, min(n_qry5, (1 << 29) // max(1, n_ref5)))
            n_pass_total, n_tiles5, max_tile_pass = 0, 0, 0
            npass = C.c_uint64(0)
            u64p, u32p, f64p = C.POINTER(C.c_uint64), C.POINTER(C.c_uint32), C.POINTER(C.c_double)
            for q0 in range(0, n_qry5, q_tile5):
                qc = min(q_tile5, n_qry5 - q0)
                eng._check(eng.lib.mashgpu_dist_run_list(job5.h, q0, qc, cap5, C.cast(l_idx.data_ptr(), u64p), C.cast(l_num.data_ptr(), u32p),
                                                         C.cast(l_den.data_ptr(), u32p), C.cast(l_dist.data_ptr(), f64p), C.cast(l_pv.data_ptr(), f64p), C.byref(npass)))
                if npass.value > cap5:
                    raise SystemExit(f"dist5: pass list of a tile ({npass.value}) exceeds the capacity {cap5}")
                n_pass_total += npass.value; n_tiles5 += 1; max_tile_pass = max(max_tile_pass, npass.value)
            torch.cuda.synchronize()
            t_rank = time.perf_counter() - t0
            barrier()
            dt5 = max_over_ranks(t_rank)
            t_dict = max_over_ranks(t_dict)
            st5 = eng.stats(reset=True)
            eng.set_timing(False)
            pf5 = job5.prefilter_stats()
            pass_all = n_pass_total
            if dist_on:
                tt = torch.tensor([n_pass_total], dtype=torch.int64, device=dev)
                td.all_reduce(tt)
                pass_all = int(tt.item())
            last_ok = bool(npass.value == 0 or (l_dist[:npass.value] <= max_d5).all().item())
            pairs5 = n_ref5 * n_qry5 * world
            dist5_obj = {"metric": "sketch_pairs_per_s", "value": pairs5 / dt5, "unit": "pairs/s", "seconds": dt5,
                         "workload": f"configs[4]: {shard5 * world} synthetic s={S} sketches all-vs-all ({shard5 * world // 1000} families of 1000, configs[2] generator), "
                                     f"reference axis sharded over {world} rank(s), every rank compares all queries with its {shard5} references",
                         "pairs": pairs5, "enumeration": "all ordered pairs (full Q x R grid)",
                         "timed_region": "ONE pass from the raw uint64 hashes in HBM to the last pass list in pinned host memory: dictionary build "
                                         f"({'sharded sample sort + all-gather of encoded rows' if dist_on else 'mashgpu_dist_open'}), probe + merge + p-value kernels for every "
                                         "query tile, list sort by pair index, D2H of the lists; wall clock, max over ranks",
                         "outputs": f"compacted pass list of `-d {max_d5}` (pair index, numer, denom, distance, p-value = 32 B per passing pair) in the reference's "
                                    "output order per query tile (CommandDistance.cpp:247-304 prints only passing pairs); dense outputs would be 25 TB",
                         "dictionary_and_exchange_seconds": t_dict, "kernel_seconds_this_rank": st5["dist_kernel_ms"] / 1e3,
                         "query_tiles": n_tiles5, "queries_per_tile": q_tile5, "passing_pairs": pass_all, "largest_tile_list": max_tile_pass,
                         "last_list_within_max_distance": last_ok, "gpu_launches": int(st5["kernel_launches"]),
                         "prefilter": {"query_tile_combinations_probed": pf5["combos_probed"], "sent_to_merge": pf5["combos_flagged"],
                                       "fraction_merged": (pf5["combos_flagged"] / pf5["combos_probed"]) if pf5["combos_probed"] else None,
                                       "pairs_merged_from_pair_lists": pf5["pairs_from_lists"]},
                         "sharded_dictionary": dstat5,
                         "hbm_roofline_note": "algorithmic HBM bytes = rank rows read once per reference tile pass (L2-resident re-reads) + 32 B per passing pair: "
                                              "far below the HBM roofline; the probe kernel's shared-memory lookups bound this workload (DESIGN.md 3.3)"}
            job5.close()
            del H5, N5, L5, l_idx, l_num, l_den, l_dist, l_pv
            if dist_on:
                del rows5, neff5, lens5
            torch.cuda.empty_cache()

        # ---------------- hot path 3: screen (configs[3], rank 0's sketches as the reference .msh) -----------------
        if not args.skip_screen:
            if args.skip_dist5:
                del o_numer, o_denom, o_dist, o_p, o_pass
            torch.cuda.empty_cache()
            if dist_on:
                from mash_b200.shard import _all_gather
                QH = _all_gather(H, world).view(-1, S); QL = _all_gather(L, world).view(-1)
                QN = torch.full((QH.shape[0],), S, dtype=torch.int32, device=dev)
            else:
                QH, QN, QL = H, N, L
            n_reads, read_len = args.reads, 150
            span_r = read_len + 1
            # reads: '*' + 150 bases drawn as substrings of the genome pool (0.5 % substitutions, 0.1 % N), all on the device
            g = torch.Generator(device=dev); g.manual_seed(4242 + rank)
            lut = torch.tensor(list(b"ACGT"), dtype=torch.uint8, device=dev)
            chunk_reads = min(n_reads, 2_000_000)
            # reads are sampled from rank 0's first 50 genomes (configs[3]); the sketches of those genomes replace the first 50
            # rows of the reference table, so that the table probe and the hit counters see real hits
            pool = screen_src
            if dist_on:
                td.broadcast(pool, src=0); td.broadcast(screen_src_hashes, src=0)
            QH = QH.clone(); QL = QL.clone()
            QH[:n_src] = screen_src_hashes
            QL[:n_src] = glen
            idx = torch.arange(read_len, device=dev)[None, :]
            # the reference table is replicated: every rank screens its reads against ALL sketches (QH = the gathered set)
            sset = mash_b200._capi._Set(QH.data_ptr(), QN.data_ptr(), QL.data_ptr(), on_device=True, n=QH.shape[0], stride=S)
            n_chunks = max(1, n_reads // chunk_reads)
            chunk_bytes = chunk_reads * span_r
            chunk_pitch = (chunk_bytes + 64 + 255) // 256 * 256
            chunks = torch.zeros((n_chunks, chunk_pitch), dtype=torch.uint8, device=dev)       # n_chunks DISTINCT chunks, resident in HBM

            def make_chunk(c):
                starts = torch.randint(0, pool.numel() - read_len, (chunk_reads,), generator=g, device=dev)
                body = pool[(starts[:, None] + idx)]
                err = torch.rand((chunk_reads, read_len), generator=g, device=dev) < 0.005
                body = torch.where(err, lut[torch.randint(0, 4, (chunk_reads, read_len), generator=g, device=dev, dtype=torch.uint8).long()], body)
                body = torch.where(torch.rand((chunk_reads, read_len), generator=g, device=dev) < 0.001, torch.full_like(body, ord("N")), body)
                v = chunks[c, :chunk_bytes].view(chunk_reads, span_r)
                v[:, 0] = ord("*")
                v[:, 1:] = body

            for c in range(n_chunks):
                make_chunk(c)
            torch.cuda.synchronize()          # the chunks are written on torch's stream, the engine reads them on its own
            if dist_on:
                from mash_b200.shard import screen_allreduce

            def screen_pass(job, feed, n):
                """n chunks through `feed`, then the cross-rank reduce and finish(); returns (seconds max over ranks, result, per-feed ms, finish ms)"""
                barrier()
                t0 = time.perf_counter()
                feed_ms = []
                for c in range(n):
                    tf = time.perf_counter()
                    feed(job, c)
                    feed_ms.append((time.perf_counter() - tf) * 1e3)
                t_fin = time.perf_counter()
                if dist_on:
                    screen_allreduce(job)                                 # reads sharded over ranks: sum the counters, merge the mixtures
                res = job.finish()
                torch.cuda.synchronize()
                fin_ms = (time.perf_counter() - t_fin) * 1e3
                return max_over_ranks(time.perf_counter() - t0), res, feed_ms, fin_ms

            # ---- value: chunks resident in HBM
            sjob = mash_b200._capi.ScreenJob(eng, sset, None, p)
            for c in range(2):
                sjob.feed_dev(chunks[c].data_ptr(), chunk_bytes)          # warm-up (counts towards the counters; the timed pass below re-opens the job)
            sjob.close()
            sjob = mash_b200._capi.ScreenJob(eng, sset, None, p)
            eng.set_timing(True); eng.stats(reset=True)
            dt, res, feed_ms, fin_ms = screen_pass(sjob, lambda j, c: j.feed_dev(chunks[c].data_ptr(), chunk_bytes), n_chunks)
            sstats = eng.stats(reset=True)
            eng.set_timing(False)
            sjob.close()
            bases = n_chunks * chunk_reads * read_len
            # ---- e2e: the same chunks from pinned host memory through mashgpu_screen_feed (H2D inside, two-buffer pipeline)
            host_chunks = torch.empty((n_chunks, chunk_bytes), dtype=torch.uint8, pin_memory=True)
            host_chunks.copy_(chunks[:, :chunk_bytes])
            torch.cuda.synchronize()
            hnp = host_chunks.numpy()
            def host_pass(mode):
                """mode None: the library's default (ASCII copies); "0" / "1" force ASCII copies / the host 2-bit packer"""
                if mode is None:
                    os.environ.pop("MASHGPU_SCREEN_HOST_PACK", None)
                else:
                    os.environ["MASHGPU_SCREEN_HOST_PACK"] = mode
                wjob = mash_b200._capi.ScreenJob(eng, sset, None, p)     # warm-up pass of the host path (staging buffers, first-use costs), like the resident one
                for c in range(3):
                    wjob.feed(hnp[c])
                wjob.finish()
                wjob.close()
                ejob = mash_b200._capi.ScreenJob(eng, sset, None, p)
                out = screen_pass(ejob, lambda j, c: j.feed(hnp[c]), n_chunks)
                ejob.close()
                os.environ.pop("MASHGPU_SCREEN_HOST_PACK", None)
                return out

            dt_e, res_e, feed_e, fin_e = host_pass(None)
            dt_a, res_a, _, _ = host_pass("0")
            dt_p, res_p, _, _ = host_pass("1")
            same_e2e = bool(all(np.array_equal(r["shared"], res["shared"]) and r["set_size"] == res["set_size"] for r in (res_e, res_a, res_p)))
            screen_obj = {"metric": "Gbp_per_s_screened", "value": world * bases / dt / 1e9, "unit": "Gbp/s",
                          "workload": f"configs[3]: {QH.shape[0]}-sketch reference table ({int(QN.sum().item())} hashes) vs {n_chunks * chunk_reads} synthetic 150 bp reads "
                                      f"per rank in {n_chunks} distinct '*'-joined chunks of {chunk_reads} reads resident in HBM; "
                                      f"{'counters all-reduced over NCCL + mixtures merged on the device, ' if dist_on else ''}finish() included",
                          "ms_total": dt * 1e3, "scan_kernel_ms": sstats["scan_kernel_ms"],
                          "host_ms": {"feed_first": feed_ms[0], "feed_median": float(np.median(feed_ms)), "feed_max": max(feed_ms), "allreduce_and_finish": fin_ms}, "gpu_launches": int(sstats["kernel_launches"]),
                          "e2e": {"value": world * bases / dt_e / 1e9, "unit": "Gbp/s", "h2d_bytes": int(n_chunks * chunk_bytes),
                                  "host_chunk_bytes": int(n_chunks * chunk_bytes), "ms_total": dt_e * 1e3,
                                  "feed_median_ms": float(np.median(feed_e)), "feed_max_ms": float(max(feed_e)), "allreduce_and_finish_ms": fin_e, "matches_device_path": same_e2e,
                                  "ascii_copies_only": world * bases / dt_a / 1e9, "host_packer_only": world * bases / dt_p / 1e9,
                                  "pack_threads": int(os.environ.get("MASHGPU_PACK_THREADS", "0")),
                                  "api": "mashgpu_screen_feed with pinned host chunks (default feed: ASCII copies, the copy of chunk i+1 overlaps the kernels of chunk i; "
                                         "host_packer_only = MASHGPU_SCREEN_HOST_PACK=1: host 2-bit packer + invalid mask, 0.375 B/base over PCIe); finish() and its D2H inside"},
                          "set_size": int(res["set_size"]), "references_hit": int((res["shared"] > 0).sum()), "exact_reruns": int(sstats["exact_reruns"]),
                          "source_genomes": n_src, "median_multiplicity_of_hit_references": float(np.median(res["median"][res["shared"] > 0])) if (res["shared"] > 0).any() else 0.0,
                          "mean_identity_of_source_genomes": float(np.mean(res["identity"][:n_src]))}
            del host_chunks, hnp
            if rank == 0:
                # ---- side measurement: a reference .msh that also holds small genomes.  Their sketches are ALL their k-mers, i.e. hashes
                # spread over the whole 64-bit range, so the largest reference hash no longer filters anything: every k-mer of the
                # mixture is a table candidate.  With and without the value-indexed bitmap in front of the table.
                n_small = 2000
                gs = torch.Generator(device=dev); gs.manual_seed(99)
                v = torch.randint(-2 ** 63, 2 ** 63 - 1, (n_small, S), generator=gs, device=dev, dtype=torch.int64)
                sign = torch.tensor(-2 ** 63, dtype=torch.int64, device=dev)
                v = (torch.sort(v ^ sign, dim=1)[0]) ^ sign                  # ascending as unsigned
                WH = torch.cat([QH, v]); WN = torch.cat([QN, torch.full((n_small,), S, dtype=torch.int32, device=dev)])
                WL = torch.cat([QL, torch.full((n_small,), 1020, dtype=QL.dtype, device=dev)])
                wset = mash_b200._capi._Set(WH.data_ptr(), WN.data_ptr(), WL.data_ptr(), on_device=True, n=WH.shape[0], stride=S)
                side = {}
                n_side = min(n_chunks, 8)
                for label, env in (("bitmap", "1"), ("no_bitmap", "0")):
                    os.environ["MASHGPU_SCREEN_BITMAP"] = env
                    wjob = mash_b200._capi.ScreenJob(eng, wset, None, p)
                    wjob.feed_dev(chunks[0].data_ptr(), chunk_bytes)
                    torch.cuda.synchronize()
                    tw = time.perf_counter()
                    for c in range(n_side):
                        wjob.feed_dev(chunks[c].data_ptr(), chunk_bytes)
                    torch.cuda.synchronize()
                    side[label] = n_side * chunk_reads * read_len / (time.perf_counter() - tw) / 1e9
                    wjob.close()
                os.environ.pop("MASHGPU_SCREEN_BITMAP", None)
                screen_obj["whole_range_table"] = {"Gbp_per_s_with_bitmap": side["bitmap"], "Gbp_per_s_without_bitmap": side["no_bitmap"], "chunks": n_side,
                                                   "table": f"the {QH.shape[0]} sketches above + {n_small} sketches of genomes shorter than s k-mers (hashes uniform over "
                                                            "the whole 64-bit range): the largest reference hash is ~2^64, every k-mer is a table candidate",
                                                   "note": "rank 0, chunks resident in HBM, outside the timed region of `value`"}
                del WH, WN, WL, v
        else:
            screen_obj = None

    # ---------------- CPU baseline on rank 0 --------------------------------------------------------------------------
    cpu = None
    os.sched_setaffinity(0, affinity_before_binding)       # the CPU arms (and the CLI run) get every CPU the process was given
    if rank == 0 and world == 1 and not args.skip_cpu:
        n_cpu = max(128, 2 * (os.cpu_count() or 1))
        rate, kind, dt, cores, tried = best_cpu_sketch_rate(n_cpu, glen)
        parsed = cpu_sketch_rate_from_files(max(32, 2 * usable_cpus()), glen, cores)
        cpu = {"value": rate, "unit": "Gbp/s", "cores": cores, "kind": kind,
               "visible_cpus": os.cpu_count(), "usable_cpus": usable_cpus(), "gbp_per_s_by_threads": tried,
               "with_fasta_parse": None if parsed is None else
               {"value": parsed[0], "unit": "Gbp/s", "threads": cores,
                "note": f"same threads, one job per file: uncompressed 70-column FASTA on tmpfs through the reference's kseq.h parser (oracle/_ref), {parsed[1]:.1f} s wall"},
               "sample": f"{n_cpu} genomes x {glen} bp, one job per genome on {cores} threads (the faster of one thread per usable CPU -- the "
                         f"container's quota -- and one per visible CPU), {dt:.1f} s wall; reference MurmurHash3/hash/MinHashHeap "
                         "object code (oracle/_ref), restated addMinHashes loop, in-memory input"}
        cpu.update(cpu_arms(cores))
        if not args.skip_cli:
            cpu["gpu_cli_file_to_msh"] = cli_sketch_rate(args.cli_files, glen, usable_cpus())
            cpu["gpu_cli_dist"] = cli_dist_rate(args.cli_dist_sketches, 20000, usable_cpus())

    if rank == 0:
        line = {"metric": "Gbp_per_s_sketched", "value": value, "unit": "Gbp/s", "n_gpus": world, "steps": Ksteps, "warmup": W,
                "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64",
                "data": "synthetic",
                "config": {"workload": WORKLOAD_SKETCH.format(units=n_units, glen=glen),
                           "k": K, "s": S, "units_per_gpu": n_units, "genome_len": glen,
                           "l2": "inputs larger than L2 (one step streams %.1f GB)" % (bases_per_step / 1e9),
                           "parallelism": f"records sharded over {world} rank(s), no data-path collective",
                           "host_binding": (f"rank 0 bound to NUMA node {numa[0]} of its GPU ({numa[1]} CPUs allowed)" if numa else "no NUMA topology visible / single node: not bound")},
                "clocks": clocks, "e2e": e2e, "gpu_launches": int(stats["kernel_launches"]),
                "roofline": roofline, "cpu_baseline": cpu, "dist": dist_obj, "dist5": dist5_obj, "screen": screen_obj, "sanity": sanity,
                "exact_reruns": int(stats["exact_reruns"])}
        emit_json_line(line)
    if dist_on:
        td.destroy_process_group()


if __name__ == "__main__":
    main()
