"""The device seed tracker (trk_add_seed of unc_device.cuh: blocked sorted set with a directory, clusters rewritten in place,
search reused for the insert, directory in a fast copy that moves to the workspace when it outgrows it) alone under the warp
emulator, seed by seed against the oracle's tracker -- which is itself pinned, seed by seed, to what the reference's own
SeedTracker (src/seed_tracker.cpp:129-143,157-232) returns.  After every seed: clusters in the set, max_map, get_final, multiset size."""
import ctypes as C

import numpy as np
import pytest

import emulib
import orclib

u32p = C.POINTER(C.c_uint32)
u64p = C.POINTER(C.c_uint64)


def _streams(kind, n, rng):
    """(ref_en, ref_len, evt): evt non-decreasing as in a read."""
    evt = np.sort(rng.integers(0, max(2, n // 8), n)).astype(np.uint32) + 22
    ln = rng.integers(12, 23, n).astype(np.uint32)
    if kind == "scattered":            # false-positive seeds all over a 9.4 Mb index: inserts, block splits
        en = rng.integers(100, 9_400_000, n).astype(np.uint64)
    elif kind == "loci":               # a few loci followed event by event (the tail of a mapping read): in-place updates,
        base = rng.integers(10_000, 9_000_000, 6)       # duplicates, neighbours one base apart
        which = rng.integers(0, 6, n)
        en = (base[which] + evt + rng.integers(-2, 3, n)).astype(np.uint64)
    elif kind == "mixed":
        en = rng.integers(100, 9_400_000, n).astype(np.uint64)
        base = rng.integers(10_000, 9_000_000, 3)
        m = rng.random(n) < 0.5
        en[m] = (base[rng.integers(0, 3, n)] + evt + rng.integers(-1, 2, n))[m].astype(np.uint64)
    else:                              # dense: everything within a few hundred bases -> many clusters inside every window
        en = (50_000 + rng.integers(0, 400, n) + evt).astype(np.uint64)
    return en, ln, evt


def _oracle(en, ln, evt, prm):
    out = np.zeros((len(en), 6), np.uint32)
    L = orclib.orc()
    L.orc_tracker_run.argtypes = [C.POINTER(orclib.OrcParams), u64p, u32p, u32p, C.c_uint32, u32p]
    assert L.orc_tracker_run(C.byref(prm), en.ctypes.data_as(u64p), ln.ctypes.data_as(u32p), evt.ctypes.data_as(u32p), len(en),
                             out.ctypes.data_as(u32p)) == 0
    return out


def _emul(en, ln, evt, prm, max_blocks, fast_cap):
    out = np.zeros((len(en), 6), np.uint32)
    L = emulib.lib()
    L.emu_tracker_run.argtypes = [C.c_uint32, C.c_float, C.c_float, u32p, u32p, u32p, C.c_uint32, u32p, C.c_uint32, C.c_uint32]
    en32 = en.astype(np.uint32)
    rc = L.emu_tracker_run(prm.min_map_len, prm.min_mean_conf, prm.min_top_conf, en32.ctypes.data_as(u32p), ln.ctypes.data_as(u32p),
                           evt.ctypes.data_as(u32p), len(en), out.ctypes.data_as(u32p), max_blocks, fast_cap)
    return out, rc


def _params():
    prm = orclib.OrcParams()
    orclib.orc().orc_params_default(C.byref(prm))
    return prm


@pytest.mark.parametrize("kind", ["scattered", "loci", "mixed", "dense"])
@pytest.mark.parametrize("fast_cap", [0, 3, 1024])
def test_device_tracker_equals_the_oracle_seed_by_seed(kind, fast_cap):
    rng = np.random.default_rng(hash((kind, fast_cap)) & 0xFFFF)
    prm = _params()
    for n in (1, 40, 700, 3000):
        en, ln, evt = _streams(kind, n, rng)
        want = _oracle(en, ln, evt, prm)
        got, rc = _emul(en, ln, evt, prm, max_blocks=2048, fast_cap=fast_cap)
        assert not (rc & 1)
        bad = np.nonzero((want != got).any(axis=1))[0]
        assert len(bad) == 0, (kind, n, int(bad[0]), want[bad[0]].tolist(), got[bad[0]].tolist())
        if kind == "scattered" and n == 3000 and fast_cap == 3:
            assert rc & 2                      # > 3 blocks: the directory has moved to the workspace


def test_directory_outgrows_its_fast_copy_in_the_middle_of_a_read():
    """40 000 scattered seeds: ~1800 blocks, so a 1024-entry fast copy (the size the kernel has) is outgrown."""
    rng = np.random.default_rng(5)
    prm = _params()
    en, ln, evt = _streams("scattered", 40000, rng)
    en = rng.integers(100, 4_000_000_000, len(en)).astype(np.uint64)      # a chr1-sized coordinate space: hardly any seed joins a cluster
    want = _oracle(en, ln, evt, prm)
    assert want[-1, 0] > 30000
    got, rc = _emul(en, ln, evt, prm, max_blocks=4096, fast_cap=1024)
    assert rc == 2
    assert np.array_equal(want, got)


def test_block_store_overflow_is_reported():
    rng = np.random.default_rng(6)
    en, ln, evt = _streams("scattered", 3000, rng)
    got, rc = _emul(en, ln, evt, _params(), max_blocks=16, fast_cap=1024)
    assert rc & 1


KINDS = ["scattered", "loci", "mixed", "dense"]


def reference_streams(kind):
    """(n, streams) of the comparison with the reference's SeedTracker"""
    rng = np.random.default_rng(11)
    for n in (40, 3000):
        yield n, _streams(kind, n, rng)


@pytest.mark.parametrize("kind", KINDS)
def test_oracle_tracker_equals_the_reference_seed_tracker(kind):
    """Against the reference's SeedTracker run on the same streams (tests/golden/reference_checks.npz,
    tools/make_reference_checks_golden.py)."""
    g = np.load(orclib.REFERENCE_CHECKS_NPZ)
    prm = _params()
    for n, (en, ln, evt) in reference_streams(kind):
        want = g["tracker/%s_%d" % (kind, n)]
        got = _oracle(en, ln, evt, prm)
        bad = np.nonzero((want != got).any(axis=1))[0]
        assert want.shape == (n, 6) and len(bad) == 0, (kind, n, int(bad[0]), want[bad[0]].tolist(), got[bad[0]].tolist())
