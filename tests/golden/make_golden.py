#!/usr/bin/env python
"""Regenerate tests/golden/ from the reference tree (run in the build container only).

  * copies the reference's own golden outputs   test/ref/{genomes.json,reads.json,genomes.dist,screen}
  * gzips the reference's test inputs           test/genome{1,2,3}.fna, test/reads{1,2}.fastq
    (data, not source; needed because /root/reference does not exist on the GPU box)
  * murmur_kat.json: MurmurHash3 known answers produced by the reference's OWN object code
    (oracle/_ref/libmash_ref.so -> getHash, hash.cpp:10-38)
  * pvalue_mpmath.json: 50-digit mpmath values of P[Bin(n, r) >= x] = I_r(x, n-x+1), the quantity
    gsl_cdf_binomial_Q(x-1, r, n) evaluates (CommandDistance.cpp:446, CommandScreen.cpp:613)
  * ref_objcode.npz, ref_kseq.npz: the answers of the reference's object code (oracle/_ref/libmash_ref.so) and of its parser
    (oracle/_ref/kseq_dump) for the inputs of tests/test_oracle_vs_ref.py and tests/test_host_fastx_vs_kseq.py, recorded by
    running those tests with --record-reference
"""
import gzip
import json
import os
import shutil
import subprocess
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
REF = "/root/reference"


def main():
    for f in ("genomes.json", "reads.json", "genomes.dist", "screen"):
        shutil.copyfile(os.path.join(REF, "test/ref", f), os.path.join(HERE, "ref_" + f))
    for f in ("genome1.fna", "genome2.fna", "genome3.fna", "reads1.fastq", "reads2.fastq"):
        with open(os.path.join(REF, "test", f), "rb") as src, gzip.GzipFile(os.path.join(HERE, f + ".gz"), "wb", 9, mtime=0) as dst:
            shutil.copyfileobj(src, dst)

    from oracle.pyoracle import RefLib
    ref = RefLib()
    import numpy as np
    rng = np.random.Generator(np.random.PCG64(7))
    kat = []
    fixed = [(b"A" * 21, 42, True), (b"AGCTTTTCATTCTGACTGCAA", 42, True), (b"AGCTTTTCATTCTGACTGCAA", 0, True),
             (b"ACGT" * 4, 42, False), (b"ACGT" * 8, 42, True), (b"MKVLAAGIV", 42, True)]
    for kmer, seed, use64 in fixed:
        kat.append(dict(kmer=kmer.decode(), seed=seed, use64=use64, hash=str(ref.get_hash(kmer, seed, use64))))
    for k in range(1, 33):
        for _ in range(4):
            kmer = bytes(rng.choice(np.frombuffer(b"ACGT", np.uint8), k))
            seed = int(rng.integers(0, 2**32))
            use64 = k > 16
            kat.append(dict(kmer=kmer.decode(), seed=seed, use64=use64, hash=str(ref.get_hash(kmer, seed, use64))))
    json.dump(kat, open(os.path.join(HERE, "murmur_kat.json"), "w"), indent=0)

    import mpmath as mp
    mp.mp.dps = 60
    cases = []
    # the six golden lines (genomes.dist / screen) + a grid
    grid = []
    for n in (1, 2, 10, 37, 400, 1000, 5000, 10000):
        for k in (11, 16, 21, 32):
            for L in (5e3, 1e5, 4.6e6, 5e8):
                K = 4.0 ** k
                pX = 1.0 / (1.0 + K / L)
                r = pX * pX / (pX + pX - pX * pX)
                for x in sorted(set([1, 2, 3, max(1, n // 10), max(1, n // 2), max(1, n - 1), n])):
                    if x <= n:
                        grid.append((x, r, n))
    for r in (0.001, 0.1, 0.5, 0.9, 0.999):
        for n in (10, 1000):
            for x in (1, n // 4 + 1, n // 2, n):
                grid.append((x, r, n))
    seen = set()
    for x, r, n in grid:
        if (x, r, n) in seen:
            continue
        seen.add((x, r, n))
        v = mp.betainc(x, n - x + 1, 0, mp.mpf(r), regularized=True)
        cases.append(dict(x=x, r=repr(float(r)), n=n, p=mp.nstr(v, 25)))
    json.dump(cases, open(os.path.join(HERE, "pvalue_mpmath.json"), "w"), indent=0)

    subprocess.check_call([sys.executable, "-m", "pytest", "-q", "--record-reference",
                           "tests/test_oracle_vs_ref.py", "tests/test_host_fastx_vs_kseq.py"], cwd=ROOT)
    print("golden fixtures written:", sorted(os.listdir(HERE)))


if __name__ == "__main__":
    main()
