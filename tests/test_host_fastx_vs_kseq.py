"""Differential test of the product's FASTA/FASTQ reader (mash_b200/host/fastx.hpp, the host feed path of SURVEY.md 8f
row 1) against the REFERENCE's own parser: kseq.h compiled in place into oracle/_ref/kseq_dump (oracle/ref_kseq_dump.cpp,
KSEQ_INIT(gzFile, gzread) as in Sketch.cpp).  Record by record: name, comment, sequence bytes and the final return code
must agree on the reference's test files and on seeded fuzz (odd white space, '>' '@' '+' inside sequences, CRLF, missing
final newline, empty records, short / long / missing quality strings, non-graph bytes, gzip).  The SHA-256 of kseq_dump's
output for each input is stored in tests/golden/ref_kseq.npz (`ref`, see fixtures.ReferenceAnswers); `pytest
--record-reference` where oracle/_ref is built runs kseq_dump again."""
import gzip
import hashlib
import os
import subprocess

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KSEQ_DUMP = os.path.join(ROOT, "oracle", "_ref", "kseq_dump")
GOLDEN = os.path.join(ROOT, "tests", "golden")
REFERENCE_ANSWERS = "ref_kseq"


def reference():
    if not os.path.exists(KSEQ_DUMP):
        raise FileNotFoundError(f"{KSEQ_DUMP} is not built: the reference's sources are needed to record its answers")
    return KSEQ_DUMP


def kseq_dump_digest(kseq_dump, path):
    r = subprocess.run([kseq_dump, path], capture_output=True, timeout=60)
    if r.returncode < 0:
        # the reference's kseq_read writes through a null pointer when the FIRST record of a file has a header and no
        # sequence byte at all (seq.s is only allocated once a sequence byte arrives, kseq.h:193-204) -- `mash` itself
        # crashes on such a file; there is nothing to compare with (the product returns an empty record, skipped as l < k)
        return ""
    assert r.returncode == 0
    return hashlib.sha256(r.stdout).hexdigest()


@pytest.fixture(scope="module")
def tools(tmp_path_factory):
    out = tmp_path_factory.mktemp("fastx") / "fastx_dump"
    subprocess.check_call(["g++", "-O2", "-std=c++17", os.path.join(ROOT, "tools", "fastx_dump.cpp"), "-o", str(out), "-lz"])
    return str(out), tmp_path_factory.mktemp("fastx_inputs")


def both(tools, ref, key, path):
    """(our reader's dump, SHA-256 of the reference's dump or None where the reference crashes)"""
    ours = subprocess.run([tools[0], path], capture_output=True, timeout=60)
    assert ours.returncode == 0
    digest = ref(key, lambda kseq_dump: kseq_dump_digest(kseq_dump, path))
    return ours.stdout, digest or None


def test_reference_test_files(tools, ref):
    for f in ("genome1.fna.gz", "genome2.fna.gz", "reads1.fastq.gz", "reads2.fastq.gz"):
        ours, digest = both(tools, ref, f, os.path.join(GOLDEN, f))            # gzipped input, as gzread handles it
        assert hashlib.sha256(ours).hexdigest() == digest and ours.count(b"\nE -1") == 1


def fuzz_file(rng):
    alpha = b"ACGTNacgtn"
    parts = []
    fastq = rng.random() < 0.5
    nl = b"\r\n" if rng.random() < 0.15 else b"\n"
    if rng.random() < 0.2:
        parts.append(rng.choice([b"", b"junk before the first header" + nl, nl + nl, b"  \t" + nl]))
    for _ in range(int(rng.integers(0, 9))):
        head = b"@" if fastq and rng.random() < 0.9 else b">"
        name = bytes(rng.choice(list(b"abcXYZ019_.|:-"), int(rng.integers(0, 12))).tolist())
        comment = b""
        r = rng.random()
        if r < 0.4:
            comment = rng.choice([b" ", b"\t", b"  "]) + bytes(rng.choice(list(b"abc def\tghi>@+"), int(rng.integers(0, 20))).tolist())
        parts.append(head + name + comment + nl)
        n = int(rng.integers(0, 400)) if rng.random() < 0.9 else int(rng.integers(60_000, 140_000))      # some records cross the 64 KiB / 1 MiB buffers
        seq = bytes(np.frombuffer(alpha, np.uint8)[rng.integers(0, len(alpha), n)].tolist())
        lines = []
        width = int(rng.choice([0, 60, 70, 80, 7]))
        if width:
            lines = [seq[i:i + width] for i in range(0, len(seq), width)]
        else:
            lines = [seq]
        body = b""
        for ln in lines:
            if rng.random() < 0.03:
                ln = ln + rng.choice([b" ", b"\t", b"\x01", b"\x7f", b"*", b"-", b"."])          # non-graph / odd bytes inside the sequence
            if rng.random() < 0.01:
                ln = ln[:len(ln) // 2] + rng.choice([b">", b"@"]) + ln[len(ln) // 2:]             # a header byte in mid-line ends the record (kseq)
            body += ln + (nl if rng.random() < 0.97 else b"")
        parts.append(body)
        if fastq and head == b"@":
            if rng.random() < 0.95:
                parts.append(b"+" + (name if rng.random() < 0.3 else b"") + nl)
                qn = n
                r = rng.random()
                if r < 0.05:
                    qn = max(0, n - int(rng.integers(1, 5)))        # truncated quality -> -2
                elif r < 0.08:
                    qn = n + int(rng.integers(1, 5))
                qual = bytes(rng.integers(33, 127, qn).astype(np.uint8).tolist())
                if width:
                    qual = nl.join(qual[i:i + width] for i in range(0, len(qual), width))
                parts.append(qual + (nl if rng.random() < 0.95 else b""))
    if rng.random() < 0.1:
        parts.append(rng.choice([b">", b"@", b">last", b">last no newline", b"+"]))
    return b"".join(parts)


def test_fuzzed_inputs(tools, ref):
    rng = np.random.Generator(np.random.PCG64(20260923))
    _, d = tools
    mismatches = []
    crashed = 0
    for i in range(400):
        data = fuzz_file(rng)
        path = os.path.join(str(d), f"f{i}" + (".gz" if i % 5 == 0 else ""))
        with (gzip.open(path, "wb") if i % 5 == 0 else open(path, "wb")) as f:
            f.write(data)
        ours, digest = both(tools, ref, f"fuzz{i}", path)
        if digest is None:
            crashed += 1
        elif hashlib.sha256(ours).hexdigest() != digest:
            mismatches.append((i, data[:200], ours[:300]))
    assert not mismatches, mismatches[:3]
    assert crashed < 40          # the comparison must cover almost all of the inputs
