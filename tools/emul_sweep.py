"""Randomised CPU sweep of the emulated kernels (minutes; not part of the test suite): random read lengths, max_paths in
{10000, 1000, 300, 77}, max_events in {30000, 200}, 2..16-warp CTAs on the 200 kb and 1 Mb indexes -- the default kernel
against the oracle (stable order, new Mapper per read), and the exact-ties kernel under the ordered-mode host logic
against the oracle's pdqsort one-Mapper chain; PAF fields and the children / sources / seeds / clusters counters.
    python tools/emul_sweep.py [seed [configs per index]]"""
import sys, time
import os
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools"), ROOT]
import numpy as np, emulib, orclib, synth, synthdata
rng = np.random.default_rng(int(sys.argv[1]) if len(sys.argv) > 1 else 5)
cnt = lambda r: (r.n_children, r.n_sources, r.n_seeds, r.n_clusters)
key = lambda r, P: (P.paf_tuple(r), cnt(r))
bad = 0; total = 0; t0 = time.time()
for name in ("g200k", "g1m"):
    prefix, g = synthdata.get_index(name)
    E = emulib.Emu(prefix)
    O = orclib.Oracle(prefix)
    for rep in range(int(sys.argv[2]) if len(sys.argv) > 2 else 10):
        mp = int(rng.choice([10000, 1000, 300, 77])); me = int(rng.choice([30000, 30000, 200]))
        E.params.max_paths = O.params.max_paths = mp
        E.params.max_events = O.params.max_events = me
        n = 6
        L = int(rng.integers(500, 6000))
        sig, _ = synth.reads(g, n, L, seed=int(rng.integers(1, 1 << 30)), frac_random=0.3)
        sigs = [np.ascontiguousarray(sig[i][:int(rng.integers(L // 2, L + 1))], np.float32) for i in range(n)]
        nw = int(rng.choice([2, 3, 5, 8, 16]))
        # default kernel vs oracle (stable)
        recs = E.map_batch(sigs, n_warps=nw)[0]
        want = [O.map_read(s) for s in sigs]
        d1 = [i for i in range(n) if key(recs[i], emulib) != key(want[i], orclib)]
        # exact ties + ordered vs oracle pdq one-Mapper chain
        flat = np.concatenate(sigs); lens = np.array([len(s) for s in sigs], np.uint32)
        offs = np.concatenate([[0], np.cumsum(lens[:-1], dtype=np.uint64)]).astype(np.uint64)
        O.lib.orc_set_child_sort(1)
        chain = O.map_reads_one_mapper(flat, offs, lens)
        O.lib.orc_set_child_sort(0)
        E.set_tie_order(1)
        ex, _, nre, _ = E.map_ordered(sigs, n_warps=nw)
        E.set_tie_order(0)
        d2 = [i for i in range(n) if key(ex[i], emulib) != key(chain[i], orclib)]
        total += 2 * n
        if d1 or d2:
            bad += 1
            print("MISMATCH", name, mp, me, L, nw, d1, d2, flush=True)
    print(name, "done %.0fs" % (time.time() - t0), flush=True)
print("SWEEP total", total, "bad configs", bad)
