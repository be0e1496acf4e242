"""The device half of `self_align` (uncalled_b200/csrc/unc_selfalign.cuh) and its host sampler, run on the CPU
through the emulator library, against the oracle (itself pinned to the reference in test_index_params.py).
The repetitive multi-sequence index below exercises what the random genomes do not: paths far longer than the
staging depth (re-walked in pass 2), sequences shorter than a k-mer, ambiguous bases, paths cut by the end of
their sequence."""
import ctypes as C
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tools")]


def repeat_index(dirname):
    """FASTA with a 3x tandem repeat, a tiny sequence, one with N runs and a low-complexity one; index built
    by the product's own (bwa-identical) builder."""
    from uncalled_b200 import _native as N
    rng = np.random.default_rng(5)
    unit = "".join("ACGT"[i] for i in rng.integers(0, 4, 700))
    rnd = "".join("ACGT"[i] for i in rng.integers(0, 4, 3000))
    seqs = [("rep", unit * 3 + rnd[:500]), ("tiny", "ACG"), ("amb", rnd[:900] + "N" * 37 + rnd[900:2000] + "NNACGTN"),
            ("low", "A" * 150 + "AC" * 100 + rnd[2000:2300])]
    fa = os.path.join(dirname, "rep.fa")
    with open(fa, "w") as f:
        for name, s in seqs:
            f.write(">%s\n" % name)
            for i in range(0, len(s), 70):
                f.write(s[i:i + 70] + "\n")
    prefix = os.path.join(dirname, "rep")
    assert N.lib().unc_index_build(fa.encode(), prefix.encode()) == 0
    return prefix


def test_glibc_rand_restatement_matches_libc():
    import emulib
    libc = C.CDLL("libc.so.6")
    for seed in (0, 1, 2, 12345, 0x7FFFFFFF, 0xFFFFFFFF):
        libc.srand(seed)
        want = [libc.rand() for _ in range(3000)]
        assert list(emulib.glibc_rand(seed, 3000)) == want, seed


@pytest.mark.parametrize("which,sample_dist", [("g200k", 4), ("g200k", 1), ("g1m", 20), ("example", 1)])
def test_emulated_self_align_matches_oracle(which, sample_dist):
    import emulib
    import orclib
    import test_index_params as tip
    prefix = tip.prefix_of(which)
    a, b = emulib.self_align(prefix, sample_dist), orclib.self_align(prefix, sample_dist)
    assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1])


def test_repeats_short_and_ambiguous_sequences(tmp_path):
    import emulib
    import orclib
    prefix = repeat_index(str(tmp_path))
    for sd in (1, 3):
        a, b = emulib.self_align(prefix, sd), orclib.self_align(prefix, sd)
        assert np.array_equal(a[0], b[0]) and np.array_equal(a[1], b[1]), sd
        lens = np.diff(a[0].astype(np.int64))
        assert lens.max() > 1000 and lens.min() >= 1           # repeats: far beyond the staging depth of 48
    from make_reference_checks_golden import sa_digest
    gold = orclib.reference_checks("self_align_repeats")       # and the oracle against the reference's own self_align
    for sd in (1, 3):
        assert sa_digest(*orclib.self_align(prefix, sd)) == gold[str(sd)], sd
