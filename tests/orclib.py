"""ctypes bindings for the CHECKERS: oracle/libunc_oracle.so (C restatement) and
oracle/_ref/libuncalled_ref.so (the reference's own mapper sources, unmodified).

Test infrastructure only -- imported by tests/, __graft_entry__.smoke() and bench.py's
cpu_baseline / --impl reference legs, never by the product package.
"""
import ctypes as C
import os
import subprocess
import tempfile

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
ORACLE_DIR = os.path.join(ROOT, "oracle")
GOLDEN = os.path.join(ROOT, "tests", "golden")
MODEL_TABLE = os.path.join(ROOT, "uncalled_b200", "data", "r94_5mer_template.f32")
# what the reference's own code returns on the tests' seeded inputs (tools/make_reference_checks_golden.py)
REFERENCE_CHECKS_JSON = os.path.join(GOLDEN, "reference_checks.json")
REFERENCE_CHECKS_NPZ = os.path.join(GOLDEN, "reference_checks.npz")

u8p = C.POINTER(C.c_uint8)
f32p = C.POINTER(C.c_float)
u32p = C.POINTER(C.c_uint32)
u64p = C.POINTER(C.c_uint64)


class OrcParams(C.Structure):
    _fields_ = [(n, C.c_uint32) for n in
                ("seed_len", "min_rep_len", "max_rep_copy", "max_paths", "max_consec_stay", "max_events")] + \
               [("max_stay_frac", C.c_float), ("min_seed_prob", C.c_float),
                ("min_map_len", C.c_uint32), ("min_mean_conf", C.c_float), ("min_top_conf", C.c_float),
                ("window_length1", C.c_uint32), ("window_length2", C.c_uint32),
                ("threshold1", C.c_float), ("threshold2", C.c_float), ("peak_height", C.c_float),
                ("min_mean", C.c_float), ("max_mean", C.c_float),
                ("bp_per_sec", C.c_float), ("sample_rate", C.c_float)]


class OrcModel(C.Structure):
    _fields_ = [("lv_mean", C.c_float * 1024), ("lv_var2", C.c_float * 1024), ("lognorm", C.c_float * 1024),
                ("model_mean", C.c_float), ("model_stdv", C.c_float)]


class OrcPaf(C.Structure):
    _fields_ = [("mapped", C.c_int32), ("fwd", C.c_int32), ("rid", C.c_int32),
                ("n_events", C.c_uint32), ("events_used", C.c_uint32), ("matches", C.c_uint32),
                ("rd_len", C.c_uint64), ("rd_st", C.c_uint64), ("rd_en", C.c_uint64),
                ("rf_st", C.c_uint64), ("rf_en", C.c_uint64), ("rf_len", C.c_uint64),
                ("map_ms", C.c_float),
                ("n_children", C.c_uint64), ("n_sources", C.c_uint64), ("n_neighbor_calls", C.c_uint64),
                ("n_occ_blocks", C.c_uint64), ("n_sa_steps", C.c_uint64), ("n_seeds", C.c_uint64),
                ("max_paths_seen", C.c_uint32), ("n_clusters", C.c_uint32)]


class RefPaf(C.Structure):
    _fields_ = [("mapped", C.c_int32), ("fwd", C.c_int32), ("rid", C.c_int32),
                ("n_events", C.c_uint32), ("events_used", C.c_uint32), ("matches", C.c_uint32),
                ("rd_len", C.c_uint64), ("rd_st", C.c_uint64), ("rd_en", C.c_uint64),
                ("rf_st", C.c_uint64), ("rf_en", C.c_uint64), ("rf_len", C.c_uint64),
                ("map_ms", C.c_float)]


PAF_KEYS = ("mapped", "fwd", "rid", "n_events", "events_used", "matches",
            "rd_len", "rd_st", "rd_en", "rf_st", "rf_en", "rf_len")


def paf_tuple(r):
    """Comparable PAF fields.  Unmapped records compare on (mapped, rd_len, n_events, events_used)."""
    if not r.mapped:
        return (0, int(r.rd_len), int(r.n_events), int(r.events_used))
    return tuple(int(getattr(r, k)) for k in PAF_KEYS)


def build_oracle():
    """Compile the C restatement."""
    subprocess.run(["make", "-C", ORACLE_DIR, "libunc_oracle.so"], check=True, capture_output=True)


def reference_checks(section):
    """The stored records of one section of tests/golden/reference_checks.json."""
    import json
    with open(REFERENCE_CHECKS_JSON) as f:
        return json.load(f)[section]


_orc = None


def orc():
    global _orc
    if _orc is None:
        path = os.path.join(ORACLE_DIR, "libunc_oracle.so")
        if not os.path.exists(path):
            build_oracle()
        lib = C.CDLL(path)
        lib.orc_params_default.argtypes = [C.POINTER(OrcParams)]
        lib.orc_model_init.argtypes = [C.POINTER(OrcModel), f32p, C.c_int]
        lib.orc_match_prob.argtypes = [C.POINTER(OrcModel), C.c_float, C.c_uint16]
        lib.orc_match_prob.restype = C.c_float
        lib.orc_detect_events.argtypes = [C.POINTER(OrcParams), f32p, C.c_uint32, f32p, u32p, u32p, f32p]
        lib.orc_detect_events.restype = C.c_uint32
        lib.orc_normalize.argtypes = [C.POINTER(OrcModel), f32p, C.c_uint32, f32p]
        lib.orc_index_load.argtypes = [C.c_char_p, C.c_char_p, C.POINTER(C.c_void_p)]
        lib.orc_index_free.argtypes = [C.c_void_p]
        lib.orc_fmi_size.argtypes = [C.c_void_p]
        lib.orc_fmi_size.restype = C.c_uint64
        lib.orc_sa.argtypes = [C.c_void_p, C.c_uint64]
        lib.orc_sa.restype = C.c_uint64
        lib.orc_kmer_range.argtypes = [C.c_void_p, C.c_uint16, u64p, u64p]
        lib.orc_get_neighbor.argtypes = [C.c_void_p, C.c_uint64, C.c_uint64, C.c_uint8, u64p, u64p]
        lib.orc_prob_thresh.argtypes = [C.c_void_p, C.c_int]
        lib.orc_prob_thresh.restype = C.c_float
        lib.orc_n_seqs.argtypes = [C.c_void_p]
        lib.orc_seq_name.argtypes = [C.c_void_p, C.c_int]
        lib.orc_seq_name.restype = C.c_char_p
        lib.orc_seq_len.argtypes = [C.c_void_p, C.c_int]
        lib.orc_seq_len.restype = C.c_uint64
        lib.orc_map_read.argtypes = [C.c_void_p, C.POINTER(OrcModel), C.POINTER(OrcParams), f32p, C.c_uint32,
                                     C.POINTER(OrcPaf)]
        lib.orc_map_batch_mt.argtypes = [C.c_void_p, C.POINTER(OrcModel), C.POINTER(OrcParams), f32p, u64p, u32p,
                                         C.c_uint32, C.c_int, C.POINTER(OrcPaf)]
        lib.orc_stream_map_read.argtypes = [C.c_void_p, C.POINTER(OrcModel), C.POINTER(OrcParams), f32p, C.c_uint32,
                                            C.c_uint32, C.c_uint32, C.POINTER(OrcPaf), C.POINTER(C.c_uint32),
                                            C.POINTER(C.c_int32)]
        lib.orc_stream_map_channel.argtypes = [C.c_void_p, C.POINTER(OrcModel), C.POINTER(OrcParams), f32p, u64p, u32p,
                                               C.c_uint32, C.c_uint32, C.c_uint32, C.POINTER(OrcPaf),
                                               C.POINTER(C.c_uint32), C.POINTER(C.c_int32)]
        _orc = lib
    return _orc


def fp(a):
    return a.ctypes.data_as(f32p)


class Oracle:
    """Convenience wrapper over the C restatement."""

    def __init__(self, prefix=None, preset="default"):
        self.lib = orc()
        self.params = OrcParams()
        self.lib.orc_params_default(C.byref(self.params))
        self.model = OrcModel()
        tab = np.fromfile(MODEL_TABLE, dtype=np.float32)
        assert tab.size == 2048
        self.lib.orc_model_init(C.byref(self.model), fp(tab), 1)
        self.idx = C.c_void_p()
        if prefix is not None:
            rc = self.lib.orc_index_load(prefix.encode(), preset.encode(), C.byref(self.idx))
            if rc != 0:
                raise RuntimeError("orc_index_load failed: %d" % rc)

    def match_probs(self, event):
        return np.array([self.lib.orc_match_prob(C.byref(self.model), float(event), k) for k in range(1024)],
                        dtype=np.float32)

    def detect(self, raw):
        raw = np.ascontiguousarray(raw, dtype=np.float32)
        n = raw.size
        means = np.zeros(n + 1, np.float32)
        starts = np.zeros(n + 1, np.uint32)
        lens = np.zeros(n + 1, np.uint32)
        mel = C.c_float()
        ne = self.lib.orc_detect_events(C.byref(self.params), fp(raw), n, fp(means),
                                        starts.ctypes.data_as(u32p), lens.ctypes.data_as(u32p), C.byref(mel))
        return means[:ne].copy(), starts[:ne].copy(), lens[:ne].copy(), np.float32(mel.value)

    def normalize(self, ev):
        ev = np.ascontiguousarray(ev, dtype=np.float32)
        out = np.zeros(ev.size, np.float32)
        self.lib.orc_normalize(C.byref(self.model), fp(ev), ev.size, fp(out))
        return out

    def map_read(self, raw):
        raw = np.ascontiguousarray(raw, dtype=np.float32)
        rec = OrcPaf()
        self.lib.orc_map_read(self.idx, C.byref(self.model), C.byref(self.params), fp(raw), raw.size, C.byref(rec))
        return rec

    def stream_read(self, raw, chunk_len, max_chunks=1000000):
        """The streaming path (Mapper::process_chunk / map_chunk) over one read; returns (rec, chunks used, ended)."""
        raw = np.ascontiguousarray(raw, dtype=np.float32)
        rec, nu, en = OrcPaf(), C.c_uint32(), C.c_int32()
        self.lib.orc_stream_map_read(self.idx, C.byref(self.model), C.byref(self.params), fp(raw), raw.size,
                                     int(chunk_len), int(max_chunks), C.byref(rec), C.byref(nu), C.byref(en))
        return rec, nu.value, en.value

    def stream_channel(self, signals, chunk_len, max_chunks=1000000):
        """Reads one after the other on one channel (persistent Mapper); returns [(rec, chunks, ended)]."""
        flat = np.ascontiguousarray(np.concatenate(signals), dtype=np.float32)
        lens = np.array([len(s) for s in signals], np.uint32)
        offs = np.concatenate([[0], np.cumsum(lens[:-1], dtype=np.uint64)]).astype(np.uint64)
        n = len(signals)
        out, nu, en = (OrcPaf * n)(), (C.c_uint32 * n)(), (C.c_int32 * n)()
        self.lib.orc_stream_map_channel(self.idx, C.byref(self.model), C.byref(self.params), fp(flat),
                                        offs.ctypes.data_as(u64p), lens.ctypes.data_as(u32p), n, int(chunk_len),
                                        int(max_chunks), out, nu, en)
        return [(out[i], nu[i], en[i]) for i in range(n)]

    def map_batch(self, samples, offsets, lens, threads=1):
        samples = np.ascontiguousarray(samples, dtype=np.float32)
        offsets = np.ascontiguousarray(offsets, dtype=np.uint64)
        lens = np.ascontiguousarray(lens, dtype=np.uint32)
        out = (OrcPaf * len(lens))()
        self.lib.orc_map_batch_mt(self.idx, C.byref(self.model), C.byref(self.params), fp(samples),
                                  offsets.ctypes.data_as(u64p), lens.ctypes.data_as(u32p), len(lens), threads, out)
        return list(out)

    def map_reads_one_mapper(self, samples, offsets, lens):
        """One long-lived Mapper over the reads in order (`uncalled map -t 1`): sources_added_ carried between reads."""
        n = len(lens)
        out = (OrcPaf * n)()
        self.lib.orc_map_reads_one_mapper.argtypes = [C.c_void_p, C.POINTER(OrcModel), C.POINTER(OrcParams), f32p, u64p, u32p,
                                                      C.c_uint32, C.POINTER(OrcPaf)]
        samples = np.ascontiguousarray(samples, np.float32)
        offsets = np.ascontiguousarray(offsets, np.uint64)
        lens = np.ascontiguousarray(lens, np.uint32)
        self.lib.orc_map_reads_one_mapper(self.idx, C.byref(self.model), C.byref(self.params), fp(samples),
                                          offsets.ctypes.data_as(u64p), lens.ctypes.data_as(u32p), n, out)
        return list(out)

    def map_read_flags(self, raw, flags_in=None):
        """One read with explicit sources_added_ flags (32 words) before; returns (rec, flags after)."""
        raw = np.ascontiguousarray(raw, dtype=np.float32)
        rec = OrcPaf()
        fi = None if flags_in is None else np.ascontiguousarray(flags_in, np.uint32)
        fo = np.zeros(32, np.uint32)
        self.lib.orc_map_read_flags.argtypes = [C.c_void_p, C.POINTER(OrcModel), C.POINTER(OrcParams), f32p, C.c_uint32,
                                                C.c_void_p, C.c_void_p, C.POINTER(OrcPaf)]
        self.lib.orc_map_read_flags(self.idx, C.byref(self.model), C.byref(self.params), fp(raw), raw.size,
                                    None if fi is None else fi.ctypes.data, fo.ctypes.data, C.byref(rec))
        return rec, fo

    def kmer_ranges(self):
        st = np.zeros(1024, np.uint64)
        en = np.zeros(1024, np.uint64)
        a, b = C.c_uint64(), C.c_uint64()
        for k in range(1024):
            self.lib.orc_kmer_range(self.idx, k, C.byref(a), C.byref(b))
            st[k], en[k] = a.value, b.value
        return st, en


_ref = None


def ref_available():
    return os.path.exists(os.path.join(ORACLE_DIR, "_ref", "libuncalled_ref.so"))


def ref(stable_sort=False):
    """oracle/_ref: the reference's own code.  One index per process (static state), and one of the two builds per
    process: stable_sort=True loads the build whose child sort is stable (oracle/ref_build/stubs_stable/pdqsort.h)."""
    global _ref
    if _ref is None:
        lib = C.CDLL(os.path.join(ORACLE_DIR, "_ref", "libuncalled_ref_stable.so" if stable_sort else "libuncalled_ref.so"))
        lib.ref_load.argtypes = [C.c_char_p, C.c_char_p]
        lib.ref_set_max_events.argtypes = [C.c_uint32]
        lib.ref_fmi_size.restype = C.c_uint64
        lib.ref_sa.argtypes = [C.c_uint64]
        lib.ref_sa.restype = C.c_uint64
        lib.ref_kmer_range.argtypes = [C.c_uint16, u64p, u64p]
        lib.ref_get_neighbor.argtypes = [C.c_uint64, C.c_uint64, C.c_uint8, u64p, u64p]
        lib.ref_prob_thresh.argtypes = [C.c_int]
        lib.ref_prob_thresh.restype = C.c_float
        lib.ref_match_prob.argtypes = [C.c_float, C.c_uint16]
        lib.ref_match_prob.restype = C.c_float
        lib.ref_model_mean.restype = C.c_float
        lib.ref_model_stdv.restype = C.c_float
        lib.ref_seq_name.argtypes = [C.c_int]
        lib.ref_seq_name.restype = C.c_char_p
        lib.ref_seq_len.argtypes = [C.c_int]
        lib.ref_seq_len.restype = C.c_uint64
        lib.ref_get_events.argtypes = [f32p, C.c_uint32, f32p, u32p, u32p, f32p]
        lib.ref_get_events.restype = C.c_uint32
        lib.ref_normalize.argtypes = [f32p, C.c_uint32, f32p]
        lib.ref_map_read.argtypes = [f32p, C.c_uint32, C.POINTER(RefPaf)]
        lib.ref_map_batch_mt.argtypes = [f32p, u64p, u32p, C.c_uint32, C.c_int, C.POINTER(RefPaf)]
        lib.ref_stream_channel.argtypes = [f32p, u64p, u32p, C.c_uint32, C.c_float, C.c_uint32, C.POINTER(RefPaf),
                                           C.POINTER(C.c_uint32), C.POINTER(C.c_int32)]
        lib.ref_stream_channels_mt.argtypes = [f32p, u64p, u32p, C.c_uint32, C.c_uint32, C.c_float, C.c_uint32, C.c_int,
                                               C.POINTER(RefPaf), C.POINTER(C.c_uint32), C.POINTER(C.c_int32)]
        lib.ref_stream_read.argtypes = [f32p, C.c_uint32, C.c_float, C.c_uint32, C.POINTER(RefPaf),
                                        C.POINTER(C.c_uint32), C.POINTER(C.c_int32)]
        lib.ref_index_build.argtypes = [C.c_char_p, C.c_char_p]
        lib.ref_self_align.argtypes = [C.c_char_p, C.c_uint32, u64p]
        lib.ref_self_align.restype = C.c_uint64
        lib.ref_self_align_copy.argtypes = [C.c_void_p, C.c_void_p]
        _ref = lib
    return _ref


def self_align(prefix, sample_dist):
    """The oracle's self_align as CSR (offsets[n+1], values): FM range lengths of the sampled paths."""
    lib = orc()
    lib.orc_self_align.argtypes = [C.c_void_p, C.c_char_p, C.c_uint32, u64p, u64p, C.c_void_p, C.c_void_p]
    idx = C.c_void_p()
    if lib.orc_index_load(prefix.encode(), b"-", C.byref(idx)) != 0:
        raise RuntimeError("oracle index load failed: " + prefix)
    try:
        a, b = C.c_uint64(), C.c_uint64()
        lib.orc_self_align(idx, prefix.encode(), sample_dist, C.byref(a), C.byref(b), None, None)
        off, val = np.zeros(a.value + 1, np.uint64), np.zeros(max(b.value, 1), np.uint64)
        lib.orc_self_align(idx, prefix.encode(), sample_dist, C.byref(a), C.byref(b), off.ctypes.data, val.ctypes.data)
        return off, val[:b.value]
    finally:
        lib.orc_index_free(idx)


def ref_self_align(prefix, sample_dist):
    """oracle/_ref: the reference's own self_align (src/self_align_ref.cpp), same CSR form."""
    R = ref()
    nv = C.c_uint64()
    n = R.ref_self_align(prefix.encode(), sample_dist, C.byref(nv))
    off, val = np.zeros(n + 1, np.uint64), np.zeros(max(nv.value, 1), np.uint64)
    R.ref_self_align_copy(off.ctypes.data, val.ctypes.data)
    return off, val[:nv.value]


def materialise_example_index(dst_dir):
    """Write the shipped example index (tests/golden/example_index_files.npz) into dst_dir."""
    z = np.load(os.path.join(GOLDEN, "example_index_files.npz"))
    prefix = os.path.join(dst_dir, "example_ref")
    for ext in ("bwt", "sa", "ann", "amb", "pac", "uncl"):
        z[ext].tofile(prefix + "." + ext)
    z["fasta"].tofile(os.path.join(dst_dir, "example_ref.fa"))
    return prefix


def run_in_subprocess(code, timeout=600):
    """oracle/_ref holds static state (one index per process): run such checks in a child."""
    import sys
    r = subprocess.run([sys.executable, "-c", code], capture_output=True, text=True, timeout=timeout, cwd=ROOT)
    if r.returncode != 0:
        raise RuntimeError("child failed:\n" + r.stdout + "\n" + r.stderr)
    return r.stdout
