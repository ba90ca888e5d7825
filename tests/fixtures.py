"""Test helpers: golden fixtures, a kseq-semantics FASTA/FASTQ reader, synthetic generators."""
import gzip
import json
import os

import numpy as np

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def read_fastx(path):
    """Records as kseq_read delivers them (kseq.h:170-208): header at '>'/'@', name = up to first
    whitespace, comment = rest of the line, sequence = only isgraph() bytes; FASTQ quality skipped."""
    opener = gzip.open if path.endswith(".gz") else open
    data = opener(path, "rb").read()
    recs = []
    i, n = 0, len(data)
    while i < n and data[i] not in b">@":
        i += 1
    while i < n:
        eol = data.find(b"\n", i)
        if eol < 0:
            eol = n
        header = data[i + 1:eol]
        parts = header.split(None, 1)
        name = parts[0] if parts else b""
        comment = header[len(name):].lstrip(b" \t") if len(parts) > 1 else b""
        i = eol + 1
        seq = bytearray()
        while i < n and data[i] not in b">+@":
            eol = data.find(b"\n", i)
            if eol < 0:
                eol = n
            seq += bytes(c for c in data[i:eol] if 33 <= c <= 126)
            i = eol + 1
        if i < n and data[i:i + 1] == b"+":
            eol = data.find(b"\n", i)
            i = eol + 1
            need = len(seq)
            q = 0
            while i < n and q < need:
                if 33 <= data[i] <= 127:
                    q += 1
                i += 1
            while i < n and data[i] not in b">@":
                i += 1
        recs.append((name.decode(), comment.decode(), bytes(seq)))
    return recs


class Golden:
    """The reference's golden outputs (tests/golden/ref_*, copied from /root/reference/test/ref)."""

    def __init__(self):
        self.genomes_json = json.load(open(os.path.join(GOLDEN, "ref_genomes.json")))
        self.reads_json = json.load(open(os.path.join(GOLDEN, "ref_reads.json")))
        self.dist_lines = [l.rstrip("\n").split("\t") for l in open(os.path.join(GOLDEN, "ref_genomes.dist"))]
        self.screen_lines = [l.rstrip("\n").split("\t") for l in open(os.path.join(GOLDEN, "ref_screen"))]
        self.murmur_kat = json.load(open(os.path.join(GOLDEN, "murmur_kat.json")))
        self.pvalue_cases = json.load(open(os.path.join(GOLDEN, "pvalue_mpmath.json")))
        self._genomes = None
        self._reads = None

    @property
    def genomes(self):
        """[(file name, [(name, comment, seq)])] for genome1..3.fna"""
        if self._genomes is None:
            self._genomes = [(f"genome{i}.fna", read_fastx(os.path.join(GOLDEN, f"genome{i}.fna.gz"))) for i in (1, 2, 3)]
        return self._genomes

    @property
    def reads(self):
        """reads1.fastq, reads2.fastq record lists"""
        if self._reads is None:
            self._reads = [read_fastx(os.path.join(GOLDEN, f"reads{i}.fastq.gz")) for i in (1, 2)]
        return self._reads

    def reads_round_robin(self):
        """Record order of sketchFile/screen over several files: round robin (Sketch.cpp:1202-1270)."""
        a, b = self.reads
        out = []
        for i in range(max(len(a), len(b))):
            if i < len(a):
                out.append(a[i][2])
            if i < len(b):
                out.append(b[i][2])
        return out

    def golden_sketch(self, i):
        s = self.genomes_json["sketches"][i]
        return np.array(s["hashes"], dtype=np.uint64), s["length"], s["name"], s["comment"]

    def golden_reads_sketch(self):
        s = self.reads_json["sketches"][0]
        return np.array(s["hashes"], dtype=np.uint64), s["length"]


class ReferenceAnswers:
    """What the reference's own code answered for the inputs of a test module, stored in tests/golden/<name>.npz so that the
    comparison runs in every checkout.  `answers(key, compute)` returns the stored answer; when recording (reference given,
    `pytest --record-reference`), it returns compute(reference) instead and save() writes the file.  Changing a test's inputs
    means recording again where the reference can be built (oracle/Makefile)."""

    def __init__(self, name, reference=None):
        self.path = os.path.join(GOLDEN, name + ".npz")
        self.reference = reference
        self.stored = dict(np.load(self.path)) if os.path.exists(self.path) else {}

    def __call__(self, key, compute):
        if self.reference is not None:
            out = compute(self.reference)
            for i, v in enumerate(out if isinstance(out, tuple) else (out,)):
                self.stored[f"{key}.{i}"] = np.asarray(v)
            return out
        if f"{key}.0" not in self.stored:
            raise KeyError(f"{self.path} holds no answer for {key!r}: record it with `pytest --record-reference`")
        out = []
        while f"{key}.{len(out)}" in self.stored:
            v = self.stored[f"{key}.{len(out)}"]
            out.append(v.item() if v.ndim == 0 else v)
        return tuple(out) if len(out) > 1 else out[0]

    def save(self):
        if self.reference is not None:
            np.savez_compressed(self.path, **self.stored)


def fmt_g(x):
    """iostream default formatting of a double: %g with 6 significant digits."""
    return "%g" % x


def synth_genome(seed, length, n_runs=0, lower_frac=0.0, alphabet=b"ACGT"):
    """SURVEY.md section 8(d) Config-2 style generator (PCG64, iid uniform ACGT, optional N-runs and
    lower-case soft-masking)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    seq = np.frombuffer(alphabet, np.uint8)[rng.integers(0, len(alphabet), length)]
    seq = seq.copy()
    for _ in range(n_runs):
        a = int(rng.integers(0, max(1, length)))
        l = int(rng.integers(1, 1001))
        seq[a:a + l] = ord("N")
    if lower_frac > 0:
        m = rng.random(length) < lower_frac
        seq[m] |= 0x20
    return seq


def mutate(seq, rate, seed):
    rng = np.random.Generator(np.random.PCG64(seed))
    out = seq.copy()
    m = rng.random(seq.size) < rate
    sub = np.frombuffer(b"ACGT", np.uint8)[rng.integers(0, 4, int(m.sum()))]
    out[m] = sub
    return out


def synth_sketches(n, s, seed, n_families=4, length=5_000_000, ragged=False):
    """SURVEY.md 8(d) Config-3 style sketch synthesis: family base sets of sorted distinct draws in
    [0, 2^64*s/L); members replace a fraction of entries. Returns (hashes (n x s) u64, n_hashes u32, lengths u64)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    hi = int(2**64 * s / length)
    fams = [np.unique(rng.integers(0, hi, 2 * s, dtype=np.uint64))[: 2 * s] for _ in range(n_families)]
    H = np.full((n, s), np.uint64(0xFFFFFFFFFFFFFFFF), dtype=np.uint64)
    N = np.zeros(n, np.uint32)
    lens = rng.integers(4_000_000, 6_000_000, n).astype(np.uint64)
    for g in range(n):
        base = fams[g % n_families]
        keep = rng.random(base.size) < rng.choice([1.0, 0.95, 0.8, 0.5, 0.1])
        fresh = rng.integers(0, hi, base.size, dtype=np.uint64)
        v = np.unique(np.where(keep, base, fresh))
        m = s
        if ragged and g % 5 == 0:
            m = int(rng.integers(0, s + 1))
        v = v[:m]
        H[g, :v.size] = v
        N[g] = v.size
    return H, N, lens


class NumpyDictOps:
    """Test double for mash_b200.shard.DictOps (the four device steps of the sharded dictionary build) in numpy, so that the
    exchange protocol of shard.sharded_dictionary can run under gloo without a GPU.  Same contracts as mashgpu_dict_*."""

    @staticmethod
    def _neff(n_hashes, stride, s):
        return np.minimum(np.minimum(n_hashes.astype(np.int64), s + 1), stride)

    def local_sort(self, hashes, n_hashes, sketch_size):
        import torch
        H = hashes.numpy().view(np.uint64)
        ne = self._neff(n_hashes.numpy(), H.shape[1], sketch_size)
        P = sketch_size + 1
        keys, slots = [], []
        for r in range(H.shape[0]):
            keys.append(H[r, :ne[r]])
            slots.append(r * P + np.arange(ne[r], dtype=np.int64))
        keys = np.concatenate(keys) if keys else np.zeros(0, np.uint64)
        slots = np.concatenate(slots) if slots else np.zeros(0, np.int64)
        o = np.argsort(keys, kind="stable")
        return torch.from_numpy(keys[o].view(np.int64).copy()), torch.from_numpy(slots[o].astype(np.int32))

    def split(self, keys, splitters):
        k = keys.numpy().view(np.uint64)
        pos = [int(np.searchsorted(k, sp, side="left")) for sp in splitters]
        edges = [0] + pos + [k.size]
        return [edges[i + 1] - edges[i] for i in range(len(edges) - 1)]

    def rank(self, keys):
        import torch
        k = keys.numpy().view(np.uint64)
        u, inv = np.unique(k, return_inverse=True)
        return torch.from_numpy(inv.astype(np.int32)), int(u.size)

    def scatter(self, codes, slots, seg_counts, seg_base, hashes, n_hashes, sketch_size):
        import torch
        m, stride = hashes.shape
        P = sketch_size + 1
        rows = np.full(m * P, 0xFFFFFFFF, np.uint32)
        base = np.repeat(np.asarray(seg_base, np.int64), np.asarray(seg_counts, np.int64))
        rows[slots.numpy().astype(np.int64)] = (codes.numpy().astype(np.int64) + base).astype(np.uint32)
        ne = self._neff(n_hashes.numpy(), stride, sketch_size)
        return torch.from_numpy(rows.view(np.int32).reshape(m, P).copy()), torch.from_numpy(ne.astype(np.int32))


def dense_rank_rows(H, N, sketch_size):
    """What every dictionary build must produce: rows of sketch_size+1 codes = rank of each hash among the distinct hashes of
    the whole collection, padding 0xFFFFFFFF."""
    P = sketch_size + 1
    ne = np.minimum(np.minimum(N.astype(np.int64), P), H.shape[1])
    valid = np.arange(H.shape[1])[None, :] < ne[:, None]
    u = np.unique(H[valid])
    rows = np.full((H.shape[0], P), 0xFFFFFFFF, np.uint32)
    w = min(P, H.shape[1])
    codes = np.searchsorted(u, H[:, :w]).astype(np.uint32)
    rows[:, :w] = np.where(valid[:, :w], codes, np.uint32(0xFFFFFFFF))
    return rows, ne.astype(np.uint32)
