"""DTW (SURVEY 8(f) rank 4; reference src/dtw.hpp): the oracle's restatement against what the reference's own DTWr94p / DTWr94d
return (stored in tests/golden/reference_checks.npz), the device routine under the emulator against the oracle, and -- on the GPU -- unc_dtw_batch
through the Python classes against the oracle.  Bit-exact: path, score, mean score."""
import ctypes as C

import numpy as np
import pytest

import emulib
import orclib

u64p = C.POINTER(C.c_uint64)
u16p = C.POINTER(C.c_uint16)
f32p = C.POINTER(C.c_float)
TAB = np.fromfile(orclib.MODEL_TABLE, dtype=np.float32)
PRESETS = [(2, 1, 100), (10, 1, 1000), (1, 1, 1), (1.5, 0.75, 3.25)]


def _template_model():
    L = orclib.orc()
    M = orclib.OrcModel()
    L.orc_model_init(C.byref(M), TAB.ctypes.data_as(f32p), 0)
    return M


def _problem(rng, nr, nc, walk=True):
    km = rng.integers(0, 1024, nr).astype(np.uint16)
    if walk:      # events that follow the k-mers (with stays and noise), as an aligned read would
        idx = np.clip((np.arange(nc) * nr) // max(nc, 1), 0, nr - 1)
        means = (TAB[2 * km[idx].astype(np.int64)] + rng.normal(0, 2.5, nc)).astype(np.float32)
    else:
        means = rng.uniform(55, 135, nc).astype(np.float32)
    return means, km


def _oracle(M, kind, sub, w, means, km):
    L = orclib.orc()
    L.orc_dtw.argtypes = [C.POINTER(orclib.OrcModel), C.c_int, C.c_int, C.c_float, C.c_float, C.c_float, f32p, C.c_uint32, u16p, C.c_uint32,
                          u64p, u64p, f32p]
    p = np.zeros(2 * (len(means) + len(km)), np.uint64)
    n, s = C.c_uint64(), C.c_float()
    assert L.orc_dtw(C.byref(M), kind, sub, w[0], w[1], w[2], means.ctypes.data_as(f32p), len(means), km.ctypes.data_as(u16p), len(km),
                     p.ctypes.data_as(u64p), C.byref(n), C.byref(s)) == 0
    return p[:2 * n.value].reshape(-1, 2).copy(), s.value


def dtw_problems():
    """400 random problems: (kind, sub, weights, event means, k-mers)"""
    rng = np.random.default_rng(1)
    for t in range(400):
        nr, nc = int(rng.integers(1, 70)), int(rng.integers(1, 70))
        kind, sub, w = int(rng.integers(0, 2)), int(rng.integers(0, 3)), PRESETS[int(rng.integers(0, 4))]
        means, km = _problem(rng, nr, nc, rng.random() < 0.7)
        yield kind, sub, w, means, km


def test_oracle_dtw_equals_the_reference_classes():
    """Against the paths and scores of the reference's DTWr94p / DTWr94d on the same problems
    (tests/golden/reference_checks.npz, tools/make_reference_checks_golden.py)."""
    g = np.load(orclib.REFERENCE_CHECKS_NPZ)
    want_path, want_len = g["dtw/path"].astype(np.uint64), g["dtw/path_len"]
    want_score, want_mean = g["dtw/score"], g["dtw/mean_score"]
    assert len(want_len) == 400
    M = _template_model()
    at = 0
    for t, (kind, sub, w, means, km) in enumerate(dtw_problems()):
        n = int(want_len[t])
        want = want_path[at:at + 2 * n]
        at += 2 * n
        path, score = _oracle(M, kind, sub, w, means, km)
        assert len(path) == n and score == want_score[t] and np.array_equal(path.ravel(), want), (t, kind, sub, len(km), len(means))
        assert np.float32(score) / np.float32(len(path)) == want_mean[t]
        if kind == 1 and all(float(x).is_integer() for x in w):
            assert score == int(score)                 # abs() of the truncated difference: whole numbers (integer weights)
    assert at == len(want_path)


def _emul(kind, sub, w, probs, n_threads):
    L = emulib.lib()
    L.emu_dtw_batch.argtypes = [f32p, C.c_int, C.c_int, C.c_float, C.c_float, C.c_float, C.c_uint32, f32p, u64p, u16p, u64p, u64p, u64p, u64p,
                                f32p, C.c_int]
    n = len(probs)
    moff = np.zeros(n + 1, np.uint64); koff = np.zeros(n + 1, np.uint64); poff = np.zeros(n + 1, np.uint64)
    moff[1:] = np.cumsum([len(m) for m, _ in probs]); koff[1:] = np.cumsum([len(k) for _, k in probs])
    poff[1:] = np.cumsum([len(m) + len(k) for m, k in probs])
    am = np.concatenate([m for m, _ in probs]); ak = np.concatenate([k for _, k in probs])
    path = np.zeros(2 * int(poff[-1]), np.uint64); plen = np.zeros(n, np.uint64); score = np.zeros(n, np.float32)
    assert L.emu_dtw_batch(TAB.ctypes.data_as(f32p), kind, sub, w[0], w[1], w[2], n, am.ctypes.data_as(f32p), moff.ctypes.data_as(u64p),
                           ak.ctypes.data_as(u16p), koff.ctypes.data_as(u64p), path.ctypes.data_as(u64p), poff.ctypes.data_as(u64p),
                           plen.ctypes.data_as(u64p), score.ctypes.data_as(f32p), n_threads) == 0
    return [(path[2 * int(poff[i]):2 * (int(poff[i]) + int(plen[i]))].reshape(-1, 2), float(score[i])) for i in range(n)]


@pytest.mark.parametrize("kind", [0, 1])
@pytest.mark.parametrize("sub", [0, 1, 2])
def test_device_dtw_under_the_emulator_equals_the_oracle(kind, sub):
    M = _template_model()
    rng = np.random.default_rng(10 * kind + sub)
    for w in PRESETS:
        shapes = [(1, 1), (1, 9), (9, 1), (2, 2), (33, 31), (64, 65), (7, 120), (130, 5), (97, 101)]
        probs = [_problem(rng, nr, nc, rng.random() < 0.7) for nr, nc in shapes]
        probs = [(m, k) for m, k in probs]
        got = _emul(kind, sub, w, probs, n_threads=32 if sub == 0 else 96)
        for (means, km), (path, score) in zip(probs, got):
            wp, ws = _oracle(M, kind, sub, w, means, km)
            assert score == ws and np.array_equal(path, wp), (kind, sub, w, len(km), len(means))


def test_path_properties():
    """Size-independent checks: monotone path, the end cells each sub-sequence mode allows, score = sum of weighted costs."""
    M = _template_model()
    rng = np.random.default_rng(3)
    for sub in (0, 1, 2):
        means, km = _problem(rng, 300, 420)
        path, score = _oracle(M, 0, sub, (2, 1, 100), means, km)
        j, i = path[:, 0].astype(np.int64), path[:, 1].astype(np.int64)
        assert np.all(np.diff(j) <= 0) and np.all(np.diff(i) <= 0) and np.all((np.diff(j) != 0) | (np.diff(i) != 0))
        if sub != 1:
            assert i[0] == 299 and i[-1] == 0
        if sub != 2:
            assert j[0] == 419 and j[-1] == 0


@pytest.mark.gpu
@pytest.mark.parametrize("cost", ["r94p", "r94d"])
def test_gpu_dtw_batch_equals_the_oracle(cost):
    from uncalled_b200 import dtw as D
    M = _template_model()
    rng = np.random.default_rng(21)
    kind = 0 if cost == "r94p" else 1
    for prm in (D.DTW_EVENT_GLOB, D.DTW_EVENT_QSUB, D.DTW_EVENT_RSUB, D.DTW_RAW_GLOB, D.DTWParams(D.DTWSubSeq.NONE, 1, 1, 1)):
        shapes = [(1, 1), (1, 40), (40, 1), (33, 31), (257, 255), (300, 700), (900, 650), (64, 2000)] + \
            [(int(rng.integers(1, 400)), int(rng.integers(1, 400))) for _ in range(40)]
        probs = [_problem(rng, nr, nc, rng.random() < 0.7) for nr, nc in shapes]
        got = D.dtw_batch(probs, prm, cost)
        for (means, km), (path, score) in zip(probs, got):
            wp, ws = _oracle(M, kind, prm.subseq, (prm.dw, prm.hw, prm.vw), means, km)
            assert score == ws and np.array_equal(path, wp), (cost, prm.subseq, len(km), len(means))


@pytest.mark.gpu
def test_gpu_dtw_classes_and_errors():
    from uncalled_b200 import dtw as D
    import uncalled_b200._native as N
    M = _template_model()
    rng = np.random.default_rng(22)
    means, km = _problem(rng, 500, 800)
    d = D.DTWr94p(means, km, D.DTW_EVENT_GLOB)
    wp, ws = _oracle(M, 0, 0, (2, 1, 100), means, km)
    assert d.get_path() == [(int(a), int(b)) for a, b in wp] and d.score() == ws
    assert d.mean_score() == float(np.float32(ws) / np.float32(len(wp)))
    d2 = D.DTWr94d(means, km, D.DTW_EVENT_RSUB)
    wp, ws = _oracle(M, 1, 1, (2, 1, 100), means, km)
    assert d2.get_path() == [(int(a), int(b)) for a, b in wp] and d2.score() == ws
    with pytest.raises(N.UncError):
        D.dtw_batch([(means, np.array([5, 2000], np.uint16))], D.DTW_EVENT_GLOB)       # k-mer code out of range
    with pytest.raises(N.UncError):
        D.dtw_batch([(np.zeros(0, np.float32), km)], D.DTW_EVENT_GLOB)                 # no events


@pytest.mark.gpu
def test_gpu_dtw_through_the_uncalled_module():
    """`_uncalled.DTWr94p(means, kmers, _uncalled.DTW_EVENT_GLOB)` as the reference's Python package would call it."""
    import os
    import sys
    import uncalled_b200._native as N
    N.build_pymodule()
    pkg = os.path.dirname(N.__file__)
    if pkg not in sys.path:
        sys.path.insert(0, pkg)
    import _uncalled as U
    M = _template_model()
    rng = np.random.default_rng(23)
    means, km = _problem(rng, 200, 260)
    for cls, kind in ((U.DTWr94p, 0), (U.DTWr94d, 1)):
        for prm, sub in ((U.DTW_EVENT_GLOB, 0), (U.DTW_EVENT_QSUB, 2), (U.DTW_EVENT_RSUB, 1)):
            d = cls(means.tolist(), km.tolist(), prm)
            wp, ws = _oracle(M, kind, sub, (2, 1, 100), means, km)
            assert d.get_path() == [(int(a), int(b)) for a, b in wp] and d.score() == ws
            assert d.mean_score() == float(np.float32(ws) / np.float32(len(wp)))


def test_dtw_fails_loudly_without_a_gpu():
    """No CPU path: without a CUDA device the call reports UNC_E_NO_DEVICE (it must never fall back to the oracle)."""
    import uncalled_b200._native as N
    from uncalled_b200 import dtw as D
    if N.lib().unc_device_count() > 0:
        pytest.skip("a CUDA device is present")
    with pytest.raises(N.UncError, match="no CUDA device"):
        D.DTWr94p(np.array([80.0, 90.0], np.float32), np.array([1, 2, 3], np.uint16), D.DTW_EVENT_GLOB)
