"""CPU tier: the exact-ties kernel (k2_map_exact: the reference's unstable pdqsort run serially on the event's keys,
uncalled_b200/csrc/unc_pdqsort.cuh) under the emulator, against PAF records computed by the UNMODIFIED reference itself
(tests/golden/synth_paf_golden.json, tools/make_synth_paf_golden.py) -- including the two reads of that set which the
reference maps differently from its own stable-sort build -- and against the oracle's restated pdqsort (mode 1)."""
import json
import os

import numpy as np
import pytest

import emulib
import orclib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.fixture(scope="module")
def setup():
    import sys
    sys.path.insert(0, os.path.join(ROOT, "tools"))
    import make_synth_paf_golden as M
    gold = json.load(open(os.path.join(ROOT, "tests", "golden", "synth_paf_golden.json")))
    name, n, ns, seed, frac = M.SETS[1]
    prefix, sig = M.signals(name, n, ns, seed, frac)
    yield emulib.Emu(prefix), orclib.Oracle(prefix), sig, gold, name
    emulib.lib().emu_set_tie_order(0)


def _counts(r):
    return (r.n_children, r.n_sources, r.n_seeds, r.n_clusters)


def test_exact_ties_kernel_gives_the_unmodified_references_records(setup):
    E, O, sig, gold, name = setup
    differ = gold["differ"][name]
    assert differ == [64, 137]
    ids = differ + [3, 150]
    sigs = [np.ascontiguousarray(sig[i], np.float32) for i in ids]
    try:
        E.set_tie_order(1)
        exact = E.map_batch(sigs)[0]
    finally:
        E.set_tie_order(0)
    plain = E.map_batch(sigs)[0]
    O.lib.orc_set_child_sort(1)
    try:
        pdq = [O.map_read(s) for s in sigs]
    finally:
        O.lib.orc_set_child_sort(0)
    for j, i in enumerate(ids):
        assert list(emulib.paf_tuple(exact[j])) == gold["reference"][name][i], i             # the reference as it is
        assert list(emulib.paf_tuple(plain[j])) == gold["reference_stable_sort"][name][i], i   # ... with a stable sort
        assert (emulib.paf_tuple(exact[j]), _counts(exact[j])) == (orclib.paf_tuple(pdq[j]), _counts(pdq[j])), i
        assert exact[j].status == 0
    assert all(emulib.paf_tuple(exact[j]) != emulib.paf_tuple(plain[j]) for j in range(2))


def test_exact_ties_on_a_small_buffer_and_odd_cta_shapes(setup):
    """max_paths 300 on the 200 kb index: short arrays (insertion sort only) up to the cap; 2- and 5-warp CTAs."""
    import synth
    import synthdata
    prefix, g = synthdata.get_index("g200k")
    E, O = emulib.Emu(prefix), orclib.Oracle(prefix)
    sig, _ = synth.reads(g, 6, 2500, seed=13, frac_random=0.3)
    sigs = [np.ascontiguousarray(sig[i], np.float32) for i in range(6)]
    O.lib.orc_set_child_sort(1)
    try:
        E.set_tie_order(1)
        for max_paths, n_warps in ((10000, 8), (300, 2), (300, 5)):
            E.params.max_paths = O.params.max_paths = max_paths
            recs = E.map_batch(sigs, n_warps=n_warps)[0]
            for i, s in enumerate(sigs):
                w = O.map_read(s)
                assert (emulib.paf_tuple(recs[i]), _counts(recs[i])) == (orclib.paf_tuple(w), _counts(w)), (max_paths, i)
    finally:
        E.set_tie_order(0)
        O.lib.orc_set_child_sort(0)


def test_both_exact_modes_together_equal_the_unmodified_references_long_lived_mapper():
    """No oracle in between: ONE Mapper of the reference's own code (oracle/_ref, pdqsort as vendored; its records stored
    in tests/golden/reference_checks.json) over four reads in order, against the emulated exact-ties kernel driven by the
    ordered-mode host logic.  The default configuration differs on exactly the two reads DESIGN.md section 2 explains
    (36: tie order, 589: flags left by 588)."""
    import synth
    import synthdata
    want = orclib.reference_checks("divergences")["one_mapper_36_588_589_590"]
    prefix, g = synthdata.get_index("g4m7")
    sig, _ = synth.reads(g, 600, 4000, seed=7, frac_random=0.15)
    ids = [36, 588, 589, 590]                             # 36: tie order decides a seed; 589: depends on what 588 leaves set
    sigs = [np.ascontiguousarray(sig[i], np.float32) for i in ids]
    E = emulib.Emu(prefix)
    E.set_tie_order(1)
    try:
        exact, _, n_re, _ = E.map_ordered(sigs)
    finally:
        E.set_tie_order(0)
    plain = E.map_batch(sigs)[0]
    assert [ids[i] for i in range(4) if list(emulib.paf_tuple(exact[i])) != want[i]] == [] and n_re == 1
    assert [ids[i] for i in range(4) if list(emulib.paf_tuple(plain[i])) != want[i]] == [36, 589]


def test_streaming_path_with_exact_ties(setup):
    """k2_map_stream_exact: chunk-wise mapping with the reference's child sort reproduced, against the streaming oracle in
    pdqsort mode (the reference's own streaming Mapper also sorts with pdqsort) -- reads following each other on channels."""
    import synth
    import synthdata
    import test_stream_emul as TS
    prefix, g = synthdata.get_index("g200k")
    E, O = emulib.Emu(prefix), orclib.Oracle(prefix)
    sig, _ = synth.reads(g, 4, 5000, seed=5, frac_random=0.3)
    O.lib.orc_set_child_sort(1)
    try:
        E.set_tie_order(1)
        st = TS._check(E, O, [sig[i][:5000 - 37 * i] for i in range(4)], 2, 450)
        assert (2, 0) in st
        E.params.max_paths = O.params.max_paths = 300
        TS._check(E, O, [sig[i] for i in range(3)], 3, 450, max_chunks=4, n_warps=3)
    finally:
        E.set_tie_order(0)
        O.lib.orc_set_child_sort(0)


def test_both_exact_modes_on_a_small_buffer_and_a_5_warp_cta():
    """Ordered mode and exact ties together, against one Mapper of the oracle with the reference's child sort: max_paths
    300 and a 5-warp CTA.  The sources_added_ words the four reads leave behind match too."""
    import synth
    import synthdata
    prefix, g = synthdata.get_index("g200k")
    E, O = emulib.Emu(prefix), orclib.Oracle(prefix)
    E.params.max_paths = O.params.max_paths = 300
    sig, _ = synth.reads(g, 40, 2000, seed=21, frac_random=0.4)
    sigs = [np.ascontiguousarray(sig[i], np.float32) for i in (5, 6, 0, 1)]
    flat = np.concatenate(sigs)
    lens = np.full(4, 2000, np.uint32)
    offs = (np.arange(4, dtype=np.uint64) * 2000).astype(np.uint64)
    O.lib.orc_set_child_sort(1)
    try:
        E.set_tie_order(1)
        want = O.map_reads_one_mapper(flat, offs, lens)
        recs, carry, n_re, _ = E.map_ordered(sigs, n_warps=5)
        for i in range(4):
            assert (emulib.paf_tuple(recs[i]), _counts(recs[i])) == (orclib.paf_tuple(want[i]), _counts(want[i])), i
        prev = np.zeros(32, np.uint32)
        for s in sigs:
            _, prev = O.map_read_flags(s, prev)
        assert np.array_equal(carry, prev) and n_re >= 1
    finally:
        E.L.emu_set_tie_order(0)
        O.lib.orc_set_child_sort(0)
