"""Mapping against a reference with SEVERAL sequences (and ambiguous bases): bns_pos2rid / translate_loc
(reference submods/bwa/bntseq.c:354-368, src/bwa_index.hpp:213-220) turn an FM coordinate into (contig, offset).
The index is built end to end by the product's own `uncalled index` (FM builder + self-alignments on the emulated device
+ parameter search); reads from every contig and both strands are mapped by the emulated kernels, the oracle and the
reference's own code (its records stored in tests/golden/reference_checks.json)."""
import os
import sys

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tools")]

CONTIGS = (("chrA", 60000, 1), ("chrB", 90000, 2), ("chrC", 50000, 3))


def build_multi_contig_index(dirname, self_align_fn):
    """FASTA with three contigs (the middle one carrying two N runs) -> <dir>/multi.{bwt,sa,ann,amb,pac,uncl}."""
    import synth
    from uncalled_b200 import index as UI
    gens = []
    fa = os.path.join(dirname, "multi.fa")
    with open(fa, "w") as f:
        for name, n, seed in CONTIGS:
            g = synth.genome(n, seed)
            gens.append(g)
            s = np.frombuffer(b"ACGT", dtype=np.uint8)[g].tobytes().decode()
            if name == "chrB":
                s = s[:30000] + "N" * 23 + s[30023:70000] + "N" * 5 + s[70005:]
            f.write(">%s some description\n" % name)
            for i in range(0, len(s), 80):
                f.write(s[i:i + 80] + "\n")
    prefix = os.path.join(dirname, "multi")
    UI.index_cmd(fa, prefix, self_align_fn=self_align_fn)
    return prefix, gens


def contig_reads(gens, per_contig=3, n_samples=3000):
    import synth
    sigs = []
    for k, g in enumerate(gens):
        sig, _ = synth.reads(g, per_contig, n_samples, seed=40 + k, frac_random=0.0)
        sigs += [sig[i] for i in range(per_contig)]
    edge, _ = synth.reads(gens[0][-1200:], 1, n_samples, seed=77, frac_random=0.0)     # ends at the contig boundary
    rnd, _ = synth.reads(gens[0], 1, n_samples, seed=78, frac_random=1.0)              # maps nowhere
    return sigs + [edge[0], rnd[0]]


def test_reads_map_to_the_right_contig(tmp_path):
    import emulib
    import orclib
    import test_emul_kernel as T
    prefix, gens = build_multi_contig_index(str(tmp_path), emulib.self_align)
    sigs = contig_reads(gens)
    E, O = emulib.Emu(prefix), orclib.Oracle(prefix)
    recs, _, _, _ = T._check(E, O, sigs)
    hit = [(r.rid, int(r.rf_len)) for r in recs if r.mapped]
    lens = {i: n for i, (_, n, _) in enumerate(CONTIGS)}
    assert len(hit) >= 7 and len(set(h[0] for h in hit)) == 3 and all(lens[rid] == rl for rid, rl in hit)
    assert [r.rid for r in recs[:9] if r.mapped] == sorted(r.rid for r in recs[:9] if r.mapped)   # reads 0-2 -> chrA, 3-5 -> chrB, ...
    assert not recs[-1].mapped
    want = orclib.reference_checks("multi_contig")["paf"]       # the reference's own Mapper on this index
    assert [list(orclib.paf_tuple(O.map_read(np.ascontiguousarray(s, np.float32)))) for s in sigs] == want
