"""CPU tier: the product's bwa-compatible index builder (unc_index_build) writes byte-identical
files to `bwa index` (the shipped example index is the golden vector; the comparison is repeated against
digests of what bwa_idx_build itself writes for a synthetic genome)."""
import os

import numpy as np

import orclib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _lib():
    from uncalled_b200 import _native as N
    return N.lib()


def test_example_index_bytes(tmp_path):
    z = np.load(os.path.join(ROOT, "tests", "golden", "example_index_files.npz"))
    fa = tmp_path / "example_ref.fa"
    z["fasta"].tofile(str(fa))
    prefix = str(tmp_path / "mine")
    assert _lib().unc_index_build(str(fa).encode(), prefix.encode()) == 0
    for ext in ("pac", "ann", "amb", "bwt", "sa"):
        assert open(prefix + "." + ext, "rb").read() == z[ext].tobytes(), ext


def test_ambiguous_bases_and_multiple_sequences(tmp_path):
    """N runs (lrand48 replacement, .amb holes) and several contigs: structure checks."""
    fa = tmp_path / "t.fa"
    fa.write_text(">c1 first contig\nACGTNNNNACGTTTGACCA\nGGGTTTAAACCC\n>c2\nNACGTACGTRYACGT\n")
    prefix = str(tmp_path / "t")
    assert _lib().unc_index_build(str(fa).encode(), prefix.encode()) == 0
    ann = open(prefix + ".ann").read().split("\n")
    assert ann[0] == "46 2 11" and ann[1] == "0 c1 first contig" and ann[2] == "0 31 1" and ann[3] == "0 c2 (null)"
    amb = open(prefix + ".amb").read().split("\n")
    assert amb[0] == "46 2 4" and amb[1] == "4 4 N" and amb[2] == "31 1 N"
    O = orclib.Oracle.__new__(orclib.Oracle)   # only the loader is needed: write a dummy .uncl
    open(prefix + ".uncl", "w").write("default\t-10,-3\t0.1\t1\n")
    O2 = orclib.Oracle(prefix)
    assert O2.lib.orc_fmi_size(O2.idx) == 92


def test_against_bwa_idx_build(tmp_path):
    """bwa_idx_build itself (oracle/_ref) on the same genome: digests of its files in tests/golden/reference_checks.json
    (tools/make_reference_checks_golden.py)."""
    import hashlib
    import synth
    g = synth.genome(30011, seed=5)
    fa = str(tmp_path / "g.fa")
    synth.write_fasta(fa, g, name="chrS some comment")
    mine = str(tmp_path / "mine")
    assert _lib().unc_index_build(fa.encode(), mine.encode()) == 0
    want = orclib.reference_checks("index_build")["sha256"]
    for ext in ("pac", "ann", "amb", "bwt", "sa"):
        assert hashlib.sha256(open(mine + "." + ext, "rb").read()).hexdigest() == want[ext], ext
