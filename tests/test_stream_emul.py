"""CPU tier: the STREAMING device path (unc_stream.cuh front end + the mapper kernel resuming from and
saving to per-channel state, driven by the same host bookkeeping as unc_stream_step) under the warp
emulator, against the oracle's streaming restatement (which is pinned to the reference's own streaming
Mapper, tests/test_oracle_stream.py)."""
import numpy as np
import pytest

import emulib
import orclib
import synth
import synthdata


@pytest.fixture(scope="module")
def g200k():
    prefix, g = synthdata.get_index("g200k")
    return prefix, g


def _check(E, O, sigs, n_channels, chunk_len, max_chunks=1000000, n_warps=8):
    ES = emulib.EmuStream(E, n_channels, chunk_len, max_chunks=max_chunks, n_warps=n_warps)
    res = ES.map_reads(sigs, chunk_len)
    ES.close()
    states = []
    for c in range(n_channels):
        idxs = list(range(c, len(sigs), n_channels))
        want = O.stream_channel([sigs[i] for i in idxs], chunk_len, max_chunks)   # the channel's Mapper persists
        for i, (rec, nu, en) in zip(idxs, want):
            r = res[i]
            if nu == 0:
                assert r is None, i
                continue
            assert (emulib.paf_tuple(r[3]), r[2], r[1]) == (orclib.paf_tuple(rec), nu, en), i
            assert (r[3].n_children, r[3].n_sources, r[3].n_seeds) == (rec.n_children, rec.n_sources, rec.n_seeds), i
            assert r[0] == (2 if rec.mapped else 3)
            states.append((r[0], r[1]))
    return states


def test_reads_following_each_other_on_shared_channels(g200k):
    """450-sample chunks (chunk_time 0.1125 s); two reads per channel: the streaming normaliser's statistics
    and sources_added_ carry over from a channel's previous read."""
    prefix, g = g200k
    E, O = emulib.Emu(prefix), orclib.Oracle(prefix)
    sig, _ = synth.reads(g, 4, 5000, seed=5, frac_random=0.3)
    sigs = [sig[i][:5000 - 37 * i] for i in range(4)] + [sig[0][:300]]      # the last one is shorter than a chunk
    st = _check(E, O, sigs, 2, 450)
    assert (2, 0) in st
    _check(E, O, [sig[i] for i in range(3)], 3, 450, max_chunks=4, n_warps=3)   # one read per channel, a 3-warp CTA


def test_max_chunks_and_one_second_chunks(g200k):
    prefix, g = g200k
    E, O = emulib.Emu(prefix), orclib.Oracle(prefix)
    sig, _ = synth.reads(g, 5, 5000, seed=5, frac_random=0.3)
    st = _check(E, O, [sig[i] for i in range(5)], 5, 450, max_chunks=4)
    assert (3, 1) in st                                  # gave up when the signal (max_chunks) ran out: ended
    _check(E, O, [sig[i][:4500] for i in range(2)], 2, 4000, n_warps=2)   # chunk_time 1.0 s, a 2-warp CTA


def test_max_events_and_small_path_buffer(g200k):
    """max_events reached in the middle of a chunk (FAILURE + ended) and a tiny max_paths (full-buffer cut)."""
    prefix, g = g200k
    E, O = emulib.Emu(prefix), orclib.Oracle(prefix)
    E.params.max_events = O.params.max_events = 150
    E.params.max_paths = O.params.max_paths = 300
    sig, _ = synth.reads(g, 6, 5000, seed=9, frac_random=0.5)
    st = _check(E, O, [sig[i] for i in range(6)], 2, 450, n_warps=5)
    assert (3, 1) in st and (2, 0) in st


def test_bench_stream_job_logic(g200k):
    """bench.py --workload stream: the pass/count/timing loop (stream_job), driven with the emulated device."""
    import os
    import sys
    sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
    import bench
    prefix, g = g200k
    E = emulib.Emu(prefix)
    sig, _ = synth.reads(g, 2, 1500, seed=5)

    class SM:
        def __init__(self):
            self.es = emulib.EmuStream(E, 2, 450)
            self.step = self.es.step

        def map_reads(self, sigs):
            from uncalled_b200.stream import feed_reads
            return feed_reads(self.step, 2, sigs, 450)
    sm = SM()
    calls = []
    ms, counters, res, lat = bench.stream_job(sm, [sig[0], sig[1]], 1, 1, lambda: calls.append("b"), lambda: calls.append("s"))
    assert calls == ["s", "b", "b"] and ms > 0
    assert 2 <= counters["chunks"] <= 6 and counters["steps"] >= 2 and counters["bytes"] >= counters["chunks"] * 450 * 4
    assert len(res) == 2 and all(r is not None and r[0] in (2, 3) for r in res)


@pytest.mark.parametrize("seed,length", [(334826472, 2996), (297309666, 5699)])
def test_max_events_reached_exactly_at_the_end_of_a_chunk(g200k, seed, length):
    """event_i_ gets to max_events with the chunk's last event: map_chunk notices only at its next call, and the fully
    mapped chunk lets try_add_chunk hand over one more chunk first -- it goes through the detector and the normaliser,
    none of its events is mapped, then the read fails as ended (3 chunks, not 2; found by tools/emul_stream_sweep.py and
    confirmed with the reference's own Mapper: oracle/_ref gives (0, 151, 255, 150), 3 chunks, ended, for the first)."""
    prefix, g = g200k
    E, O = emulib.Emu(prefix), orclib.Oracle(prefix)
    E.params.max_events = O.params.max_events = 150
    E.params.max_paths = O.params.max_paths = 77
    sig, _ = synth.reads(g, 3, length, seed=seed, frac_random=0.35)
    st = _check(E, O, [sig[i] for i in range(3)], 1, 450)
    assert (3, 1) in st
