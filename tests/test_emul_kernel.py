"""CPU tier: the DEVICE source (uncalled_b200/csrc/unc_device.cuh), compiled for the host with
-DUNC_EMUL and run under the lockstep CTA emulator (tests/emul/warp_emul.hpp), against the
oracle.  This exercises the exact kernel logic -- warp scans, the chunk-local extension, the
segment radix sort, the look-back prefix, the tracker's blocked cluster list -- without a GPU.
(It is a test vehicle: the shipped library contains only the CUDA build.)"""
import numpy as np
import pytest

import emulib
import orclib
import synth
import synthdata


def _check(E, O, sigs, **kw):
    recs, ev, nm, mel = E.map_batch(sigs, **kw)
    for i, s in enumerate(sigs):
        w = O.map_read(s)
        assert orclib.paf_tuple(w) == emulib.paf_tuple(recs[i]), i
        assert (w.n_children, w.n_sources, w.n_seeds, w.n_clusters) == \
               (recs[i].n_children, recs[i].n_sources, recs[i].n_seeds, recs[i].n_clusters), i
        assert recs[i].status == 0
    return recs, ev, nm, mel


def test_example_read_events_and_paf(example_prefix, golden_read):
    E, O = emulib.Emu(example_prefix), orclib.Oracle(example_prefix)
    raw = golden_read["raw"]
    recs, ev, nm, mel = _check(E, O, [raw, raw[:4000]])
    assert np.array_equal(ev[0], golden_read["ev_mean"]) and np.array_equal(nm[0], golden_read["normed"])
    assert mel[0] == golden_read["mean_event_len"]
    assert emulib.paf_tuple(recs[0])[6:12] == (106, 73, 106, 6938, 6976, 10000)


@pytest.fixture(scope="module")
def g200k():
    prefix, g = synthdata.get_index("g200k")
    return prefix, g


def test_synthetic_reads_and_ragged_batch(g200k):
    prefix, g = g200k
    E, O = emulib.Emu(prefix), orclib.Oracle(prefix)
    sig, _ = synth.reads(g, 6, 12000, seed=5)
    lens = [12000, 5, 40, 300, 4000, 7777]
    _check(E, O, [sig[i, :L] for i, L in enumerate(lens)])


@pytest.mark.parametrize("n_warps", [2, 3, 5, 14, 16])      # 14 = the shape the GPU build runs (K2_WARPS)
def test_cta_shapes(g200k, n_warps):
    prefix, g = g200k
    E, O = emulib.Emu(prefix), orclib.Oracle(prefix)
    sig, _ = synth.reads(g, 3, 3000, seed=3)
    _check(E, O, [sig[i] for i in range(3)], n_warps=n_warps)


@pytest.mark.parametrize("max_paths", [300, 77])
def test_full_buffer_semantics(g200k, max_paths):
    """tiny max_paths: the full-buffer break, the source caps and the stale sources_added_
    flags are hit on almost every event."""
    prefix, g = g200k
    E, O = emulib.Emu(prefix), orclib.Oracle(prefix)
    E.params.max_paths = O.params.max_paths = max_paths
    sig, _ = synth.reads(g, 4, 2500, seed=13)
    _check(E, O, [sig[i] for i in range(4)])
    sig, _ = synth.reads(g, 3, 3000, seed=3)
    _check(E, O, [sig[i][:2500] for i in range(3)])


def test_i16_calibration_path(g200k):
    prefix, g = g200k
    E, O = emulib.Emu(prefix), orclib.Oracle()
    rng = np.random.default_rng(3)
    i16 = rng.integers(200, 1200, 3000).astype(np.int16)
    i16[100:110] = -5
    cal = (1467.61, 10.0, 8192.0)
    pa = (np.float32(cal[0]) * (i16.astype(np.uint16).astype(np.float32) + np.float32(cal[1]))) / np.float32(cal[2])
    recs, ev, nm, mel = E.map_batch([i16], run_k2=False, dtype=1, cal=cal)
    m, s, l, omel = O.detect(pa.astype(np.float32))
    assert np.array_equal(ev[0], m) and mel[0] == omel


def test_bench_scale_reads_on_the_4m7_index():
    """The shipped kernel at the bench workload's scale (4.7 Mb index, max_paths 10 000, 4000-sample reads): one read that
    maps and one that never does and extends ~4 M children through every phase at the buffer cap (3 radix passes,
    deferred window walks, full-buffer cuts)."""
    prefix, g = synthdata.get_index("g4m7")
    E, O = emulib.Emu(prefix), orclib.Oracle(prefix)
    sig, _ = synth.reads(g, 120, 4000, seed=7, frac_random=0.15)
    recs, _, _, _ = _check(E, O, [sig[100], sig[99]])
    assert recs[0].mapped and not recs[1].mapped and recs[1].n_children > 3000000


def test_kmer_ranges_that_overlap_share_a_bucket(g200k):
    """get_base_range's start (L2[b], not L2[b]+1) lets a k-mer's FM range begin on its predecessor's last row; children of
    the two k-mers then interleave in the sorted order (first seen on the B200: read 30 of this set, event 63 -- two gap
    sources short).  The second worker structure keeps such k-mers in one bucket and walks it as the reference does."""
    prefix, g = g200k
    sig, _ = synth.reads(g, 31, 4000, seed=7)
    E = emulib.Emu(prefix)
    O = orclib.Oracle(prefix)
    st, en = O.kmer_ranges()
    ne = st <= en
    order = np.argsort(st[ne], kind="stable")
    s, e = st[ne][order], en[ne][order]
    assert (s[1:] <= e[:-1]).sum() >= 1          # the index has overlapping k-mer ranges
    recs = E.map_batch([sig[30]])[0]
    w = O.map_read(sig[30])
    assert emulib.paf_tuple(recs[0]) == orclib.paf_tuple(w)
    assert (recs[0].n_children, recs[0].n_sources, recs[0].n_seeds, recs[0].n_clusters) == (w.n_children, w.n_sources, w.n_seeds, w.n_clusters)
