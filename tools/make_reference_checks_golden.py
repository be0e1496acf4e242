#!/usr/bin/env python
"""Generates tests/golden/reference_checks.json and tests/golden/reference_checks.npz: what the REFERENCE's own code
(oracle/_ref, built by `make -C oracle ref` from a reference source tree, and the reference's uncalled/pafstats.py) returns
on the seeded inputs of the tests that compare the oracle, the emulated kernels and the index builder with it.  The tests
rebuild the same inputs from their seeds and compare against these records, so they run wherever the repository is.
One section per process (the reference keeps its index in process-global statics, and one of its two builds per process):
    python tools/make_reference_checks_golden.py [REFERENCE_TREE]     # the tree is needed for the pafstats section"""
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import tempfile

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools"), ROOT]
import numpy as np  # noqa: E402

OUT_JSON = os.path.join(ROOT, "tests", "golden", "reference_checks.json")
OUT_NPZ = os.path.join(ROOT, "tests", "golden", "reference_checks.npz")
u16p, u32p, u64p, f32p = (C.POINTER(t) for t in (C.c_uint16, C.c_uint32, C.c_uint64, C.c_float))


def _paf(r):
    import orclib
    return [int(v) for v in orclib.paf_tuple(r)]


def _map_reads(R, sigs):
    """fresh Mapper per read (ref_map_read)"""
    import orclib
    out = []
    for s in sigs:
        s = np.ascontiguousarray(s, np.float32)
        rec = orclib.RefPaf()
        R.ref_map_read(orclib.fp(s), len(s), C.byref(rec))
        out.append(_paf(rec))
    return out


def _one_mapper(R, sigs):
    """ONE long-lived Mapper over the reads in order (ref_map_batch_mt on one thread)"""
    import orclib
    n = len(sigs)
    flat = np.ascontiguousarray(np.concatenate(sigs), np.float32)
    lens = np.array([len(s) for s in sigs], np.uint32)
    offs = np.concatenate([[0], np.cumsum(lens[:-1], dtype=np.uint64)]).astype(np.uint64)
    out = (orclib.RefPaf * n)()
    R.ref_map_batch_mt(orclib.fp(flat), offs.ctypes.data_as(u64p), lens.ctypes.data_as(u32p), n, 1, out)
    return [_paf(r) for r in out]


def _loaded(prefix, stable_sort=False):
    import orclib
    R = orclib.ref(stable_sort=stable_sort)
    assert R.ref_load(prefix.encode(), b"default") == 0
    return R


def sa_digest(off, val):
    return {"n_paths": int(len(off) - 1), "n_values": int(len(val)),
            "offsets_sha256": hashlib.sha256(np.ascontiguousarray(off, "<u8").tobytes()).hexdigest(),
            "values_sha256": hashlib.sha256(np.ascontiguousarray(val, "<u8").tobytes()).hexdigest()}


def synthetic_reads():
    """test_oracle_pinned: 96 reads on the 200 kb index; events, normaliser, model and thresholds of the reference."""
    import orclib
    import synth
    import synthdata
    prefix, g = synthdata.get_index("g200k")
    sig, _ = synth.reads(g, 96, 4000, seed=11)
    R = _loaded(prefix)
    ev, st, ln, mel = np.zeros(4001, np.float32), np.zeros(4001, np.uint32), np.zeros(4001, np.uint32), C.c_float()
    ne = R.ref_get_events(orclib.fp(sig[0]), 4000, orclib.fp(ev), st.ctypes.data_as(u32p), ln.ctypes.data_as(u32p), C.byref(mel))
    nm = np.zeros(ne, np.float32)
    R.ref_normalize(orclib.fp(ev[:ne].copy()), ne, orclib.fp(nm))
    probs = np.array([[R.ref_match_prob(e, k) for k in range(1024)] for e in (61.5, 90.25, 118.0)], np.float32)
    return {"paf": _map_reads(R, sig)}, {
        "ev_mean": ev[:ne], "ev_start": st[:ne], "ev_len": ln[:ne], "mean_event_len": np.float32(mel.value),
        "normed": nm, "match_prob": probs, "prob_thresh": np.array([R.ref_prob_thresh(b) for b in range(64)], np.float32)}


def g4m7_sets():
    import synth
    import synthdata
    prefix, g = synthdata.get_index("g4m7")
    a, _ = synth.reads(g, 600, 4000, seed=7, frac_random=0.15)
    b, _ = synth.reads(g, 2400, 4000, seed=123, frac_random=0.15)
    return prefix, a, b


def divergences():
    """test_oracle_pinned / test_exact_ties_emul: the unmodified reference on the 4.7 Mb index."""
    prefix, a, b = g4m7_sets()
    R = _loaded(prefix)
    return {"one_mapper_575_595": _one_mapper(R, [a[i] for i in range(575, 595)]),
            "one_mapper_36_588_589_590": _one_mapper(R, [a[i] for i in (36, 588, 589, 590)]),
            "fresh_30_40": _map_reads(R, [a[i] for i in range(30, 40)]),
            "fresh_second_set": _map_reads(R, [b[i] for i in (64, 137, 1395, 1598, 1971)])}, {}


def stable_sort():
    """test_oracle_pinned: the reference's code with its child sort made stable."""
    prefix, a, b = g4m7_sets()
    R = _loaded(prefix, stable_sort=True)
    return {"fresh": _map_reads(R, [a[i] for i in range(30, 40)] + [b[i] for i in (64, 137, 1395, 1598)])}, {}


def stream():
    """test_oracle_stream: the reference's streaming Mapper on fresh reads."""
    import orclib
    import synth
    import synthdata
    prefix, g = synthdata.get_index("g200k")
    R = _loaded(prefix)
    sig, _ = synth.reads(g, 10, 9000, seed=77, frac_random=0.3)
    rows = []
    for i in range(10):
        s = np.ascontiguousarray(sig[i], np.float32)
        for ct, mc in ((0.1125, 1000000), (0.1125, 7), (0.25, 3)):
            out, nu, en = orclib.RefPaf(), C.c_uint32(), C.c_int32()
            R.ref_stream_read(orclib.fp(s), len(s), ct, mc, C.byref(out), C.byref(nu), C.byref(en))
            rows.append({"read": i, "chunk_time": ct, "max_chunks": mc, "paf": _paf(out), "chunks": nu.value, "ended": en.value})
    return {"rows": rows}, {}


def dtw():
    """test_dtw: the reference's DTWr94p / DTWr94d on 400 random problems."""
    import orclib
    import test_dtw as T
    R = orclib.ref()
    R.ref_dtw.argtypes = [C.c_int, C.c_int, C.c_float, C.c_float, C.c_float, f32p, C.c_uint32, u16p, C.c_uint32, u64p, u64p, f32p, f32p]
    paths, lens, scores, means = [], [], [], []
    for kind, sub, w, m, km in T.dtw_problems():
        want = np.zeros(2 * (len(m) + len(km)), np.uint64)
        n, s, ms = C.c_uint64(), C.c_float(), C.c_float()
        R.ref_dtw(kind, sub, w[0], w[1], w[2], m.ctypes.data_as(f32p), len(m), km.ctypes.data_as(u16p), len(km), want.ctypes.data_as(u64p),
                  C.byref(n), C.byref(s), C.byref(ms))
        paths.append(want[:2 * n.value].astype(np.uint16))
        lens.append(n.value)
        scores.append(s.value)
        means.append(ms.value)
    return {}, {"path": np.concatenate(paths), "path_len": np.array(lens, np.uint32),
                "score": np.array(scores, np.float32), "mean_score": np.array(means, np.float32)}


def tracker():
    """test_tracker_emul: the reference's SeedTracker seed by seed."""
    import orclib
    import test_tracker_emul as T
    prm = T._params()
    R = orclib.ref()
    R.ref_tracker_run.argtypes = [C.c_uint32, C.c_float, C.c_float, u64p, u32p, u32p, C.c_uint32, u32p]
    arrays = {}
    for kind, n, (en, ln, evt) in ((k, n, x) for k in T.KINDS for n, x in T.reference_streams(k)):
        want = np.zeros((n, 6), np.uint32)
        assert R.ref_tracker_run(prm.min_map_len, prm.min_mean_conf, prm.min_top_conf, en.ctypes.data_as(u64p), ln.ctypes.data_as(u32p),
                                 evt.ctypes.data_as(u32p), n, want.ctypes.data_as(u32p)) == 0
        arrays["%s_%d" % (kind, n)] = want
    return {}, arrays


def index_build():
    """test_index_build: bwa_idx_build itself on a 30 kb synthetic genome."""
    import orclib
    import synth
    d = tempfile.mkdtemp()
    fa = os.path.join(d, "g.fa")
    synth.write_fasta(fa, synth.genome(30011, seed=5), name="chrS some comment")
    orclib.ref().ref_index_build(fa.encode(), os.path.join(d, "ref").encode())
    return {"sha256": {ext: hashlib.sha256(open(os.path.join(d, "ref." + ext), "rb").read()).hexdigest()
                       for ext in ("pac", "ann", "amb", "bwt", "sa")}}, {}


def self_align_g200k():
    """test_index_params: the reference's self_align on the 200 kb index."""
    import orclib
    import synthdata
    prefix = synthdata.get_index("g200k")[0]
    return {str(sd): sa_digest(*orclib.ref_self_align(prefix, sd)) for sd in (1, 7, 250)}, {}


def self_align_repeats():
    """test_selfalign_emul: the reference's self_align on the repetitive multi-sequence index."""
    import orclib
    import test_selfalign_emul as T
    prefix = T.repeat_index(tempfile.mkdtemp())
    return {str(sd): sa_digest(*orclib.ref_self_align(prefix, sd)) for sd in (1, 3)}, {}


def multi_contig():
    """test_multi_contig: the reference's Mapper on the three-contig index that `uncalled index` of the product builds."""
    import emulib
    import test_multi_contig as T
    prefix, gens = T.build_multi_contig_index(tempfile.mkdtemp(), emulib.self_align)
    return {"paf": _map_reads(_loaded(prefix), T.contig_reads(gens))}, {}


def pafstats(tree):
    """test_pafstats: what the reference's uncalled/pafstats.py prints for the test's two PAF files."""
    import test_pafstats as T
    d = tempfile.mkdtemp()
    q, r = os.path.join(d, "q.paf"), os.path.join(d, "r.paf")
    open(q, "w").write(T.QRY)
    open(r, "w").write(T.REF)
    code = ("import sys, types; sys.modules['_uncalled'] = types.ModuleType('_uncalled'); sys.path.insert(0, %r);"
            "import pafstats, argparse; p = argparse.ArgumentParser(); pafstats.add_opts(p); pafstats.run(p.parse_args(%r))"
            % (os.path.join(tree, "uncalled"), [q, "-r", r]))
    out = subprocess.run([sys.executable, "-W", "ignore", "-c", code], capture_output=True, text=True, timeout=120, check=True)
    return {"stdout": out.stdout.replace(d + os.sep, "")}, {}


SECTIONS = [synthetic_reads, divergences, stable_sort, stream, dtw, tracker, index_build, self_align_g200k, self_align_repeats,
            multi_contig]


def main():
    tree = sys.argv[1] if len(sys.argv) > 1 else None
    gold, arrays = {}, {}
    tmp = tempfile.mkdtemp()
    for fn in SECTIONS + ([pafstats] if tree else []):
        out = os.path.join(tmp, fn.__name__)
        code = ("import sys, json, numpy as np; sys.path[:0] = %r; import make_reference_checks_golden as M\n"
                "j, a = M.%s(%s)\njson.dump(j, open(%r + '.json', 'w')); np.savez(%r + '.npz', **a)"
                % (sys.path[:3], fn.__name__, repr(tree) if fn is pafstats else "", out, out))
        subprocess.run([sys.executable, "-c", code], check=True, cwd=ROOT)
        gold[fn.__name__] = json.load(open(out + ".json"))
        for k, v in np.load(out + ".npz").items():
            arrays[fn.__name__ + "/" + k] = v
        print(fn.__name__, "done", flush=True)
    if not tree:                                     # keep the stored pafstats output
        gold["pafstats"] = json.load(open(OUT_JSON))["pafstats"]
    json.dump(gold, open(OUT_JSON, "w"), indent=0, sort_keys=True)
    np.savez_compressed(OUT_NPZ, **arrays)
    print("wrote", OUT_JSON, OUT_NPZ)


if __name__ == "__main__":
    main()
