"""CPU tier: uncalled_b200/csrc/unc_pdqsort.cuh (the exact-ties kernels' serial sort) against pdqsort ITSELF -- the
reference's vendored submods/pdqsort/pdqsort.h compiled into oracle/_ref (ref_pdqsort_keys) -- on arbitrary key arrays:
random keys with many ties, and the patterns that drive pdqsort through partition_left, the partial insertion sorts,
its pattern-breaking swaps; and the heapsort fallback (libstdc++'s make_heap + sort_heap) directly.  Byte-for-byte equality of
the sorted arrays (the tag word tracks where equal keys land), through the committed digests that this file's
`python tests/test_pdqsort.py` makes with the real header."""
import ctypes as C
import hashlib
import json
import os

import numpy as np

import emulib
import orclib

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden", "pdqsort_digests.json")
SIZES = (0, 1, 2, 5, 23, 24, 25, 100, 128, 129, 130, 1000, 5000, 20000)


def patterns(n, rng):
    """name -> (start, end, prob) columns; few distinct values so that ties are everywhere"""
    r = lambda hi: rng.integers(0, hi, n).astype(np.uint32)           # noqa: E731
    asc = np.arange(n, dtype=np.uint32)
    probs = (rng.integers(0, 4, n).astype(np.float32) - 2.5)
    half = n // 2
    out = {
        "random_few_values": (r(16), r(3), probs),
        "random_many_values": (r(1 << 20), r(1 << 20), rng.standard_normal(n).astype(np.float32)),
        "all_equal": (np.full(n, 7, np.uint32), np.full(n, 9, np.uint32), np.full(n, -1.25, np.float32)),
        "ascending": (asc, asc, probs),
        "descending": (asc[::-1].copy(), asc[::-1].copy(), probs),
        "pipe_organ": (np.concatenate([asc[:half], asc[:n - half][::-1]]), r(2), probs),
        "push_front": (np.concatenate([asc[1:], asc[:1]]) if n else asc, r(2), probs),
        "push_middle": (np.concatenate([asc[:half], asc[half + 1:], asc[half:half + 1]]) if n else asc, r(2), probs),
        "sawtooth": ((asc % 7).astype(np.uint32), (asc % 3).astype(np.uint32), probs),
        "blocks_of_equal": ((asc // 50)[::-1].copy().astype(np.uint32), np.zeros(n, np.uint32), np.zeros(n, np.float32)),
    }
    return out


def keys_of(cols):
    st, en, pr = cols
    n = len(st)
    k = np.zeros((n, 4), np.uint32)
    k[:, 0], k[:, 1], k[:, 2], k[:, 3] = st, en, np.asarray(pr, np.float32).view(np.uint32), np.arange(n, dtype=np.uint32)
    return k


def cases():
    rng = np.random.default_rng(20240923)
    for n in SIZES:
        for name, cols in patterns(n, rng).items():
            yield "%s/%d" % (name, n), keys_of(cols)
    # inputs that exhaust pdqsort's budget of highly unbalanced partitions, so that the sort itself falls back to heapsort
    # (found by hill climbing on the smallest budget reached, tests/golden/pdqsort_killers.json): as they are, and with
    # every value doubled up (ties) -- the latter need not reach the fallback
    killers = json.load(open(os.path.join(ROOT, "tests", "golden", "pdqsort_killers.json")))
    for n, vals in killers.items():
        v = np.array(vals, np.uint32)
        z = np.zeros(len(v), np.float32)
        yield "killer/%s" % n, keys_of((v, np.zeros(len(v), np.uint32), z))
        yield "killer_ties/%s" % n, keys_of((v // 2, np.zeros(len(v), np.uint32), z))


def emu_sort(k):
    L = emulib.lib()
    L.emu_pdq_sort.argtypes = [C.c_void_p, C.c_uint32, C.c_uint32]
    out = np.ascontiguousarray(k.copy())
    assert L.emu_pdq_sort(out.ctypes.data, len(out), 256) == 0
    return out


def test_device_pdqsort_equals_the_vendored_header_on_patterns():
    gold = json.load(open(GOLD))
    L = emulib.lib()
    L.emu_pdq_heapsorts.restype = C.c_ulong
    h0 = L.emu_pdq_heapsorts()
    for name, k in cases():
        got = emu_sort(k)
        assert hashlib.sha256(got.tobytes()).hexdigest() == gold[name], name
        srt = got[:, :3]
        assert sorted(map(tuple, k.tolist())) == sorted(map(tuple, got.tolist())), name      # a permutation
        f = got[:, 2].view(np.float32)
        for i in range(1, len(got)):                                                       # ... in operator< order
            a, b = got[i - 1], got[i]
            assert (a[0], a[1]) < (b[0], b[1]) or ((a[0], a[1]) == (b[0], b[1]) and not (f[i] < f[i - 1])), (name, i)
    # no mapped read exhausts pdqsort's budget of unbalanced partitions (the oracle counts its fallbacks); besides the
    # killer inputs the fallback routine is pinned on its own: pq_heapsort == libstdc++'s make_heap + sort_heap
    assert L.emu_pdq_heapsorts() - h0 >= 3          # the killer inputs went through the fallback inside the sort
    L.emu_pdq_heapsort.argtypes = [C.c_void_p, C.c_uint32]
    for name, k in cases():
        got = np.ascontiguousarray(k.copy())
        L.emu_pdq_heapsort(got.ctypes.data, len(got))
        assert hashlib.sha256(got.tobytes()).hexdigest() == gold["heap/" + name], name


if __name__ == "__main__":      # regenerate the digests with the REAL pdqsort (needs oracle/_ref)
    R = orclib.ref()
    R.ref_pdqsort_keys.argtypes = [C.c_void_p, C.c_uint32]
    R.ref_heapsort_keys.argtypes = [C.c_void_p, C.c_uint32]
    d = {}
    for name, k in cases():
        want = np.ascontiguousarray(k.copy())
        R.ref_pdqsort_keys(want.ctypes.data, len(want))
        d[name] = hashlib.sha256(want.tobytes()).hexdigest()
        want = np.ascontiguousarray(k.copy())
        R.ref_heapsort_keys(want.ctypes.data, len(want))
        d["heap/" + name] = hashlib.sha256(want.tobytes()).hexdigest()
    json.dump(d, open(GOLD, "w"), indent=0)
    print("wrote", GOLD, len(d))
