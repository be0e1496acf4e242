"""ctypes binding of tests/emul/libunc_emul.so: the DEVICE source run on the CPU under the
32-fiber warp emulator (test vehicle; see tests/emul/warp_emul.hpp)."""
import ctypes as C
import os
import subprocess

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
EMUL_DIR = os.path.join(ROOT, "tests", "emul")
MODEL_TABLE = os.path.join(ROOT, "uncalled_b200", "data", "r94_5mer_template.f32")


class UncParams(C.Structure):
    _fields_ = [(n, C.c_uint32) for n in
                ("seed_len", "min_rep_len", "max_rep_copy", "max_paths", "max_consec_stay", "max_events")] + \
               [("max_stay_frac", C.c_float), ("min_seed_prob", C.c_float),
                ("min_map_len", C.c_uint32), ("min_mean_conf", C.c_float), ("min_top_conf", C.c_float),
                ("window_length1", C.c_uint32), ("window_length2", C.c_uint32),
                ("threshold1", C.c_float), ("threshold2", C.c_float), ("peak_height", C.c_float),
                ("min_mean", C.c_float), ("max_mean", C.c_float),
                ("bp_per_sec", C.c_float), ("sample_rate", C.c_float)]


class UncReadDesc(C.Structure):
    _fields_ = [("offset", C.c_uint64), ("n_samples", C.c_uint32), ("dtype", C.c_uint32),
                ("cal_range", C.c_float), ("cal_offset", C.c_float), ("cal_digit", C.c_float)]


class UncPaf(C.Structure):
    _fields_ = [("mapped", C.c_int32), ("fwd", C.c_int32), ("rid", C.c_int32), ("status", C.c_int32),
                ("n_events", C.c_uint32), ("events_used", C.c_uint32), ("matches", C.c_uint32),
                ("n_clusters", C.c_uint32),
                ("rd_len", C.c_uint64), ("rd_st", C.c_uint64), ("rd_en", C.c_uint64),
                ("rf_st", C.c_uint64), ("rf_en", C.c_uint64), ("rf_len", C.c_uint64),
                ("n_children", C.c_uint64), ("n_sources", C.c_uint64), ("n_occ_blocks", C.c_uint64),
                ("n_sa_steps", C.c_uint64), ("n_seeds", C.c_uint64)]


def default_params():
    p = UncParams()
    (p.seed_len, p.min_rep_len, p.max_rep_copy, p.max_paths, p.max_consec_stay, p.max_events) = (22, 0, 50, 10000, 8, 30000)
    p.max_stay_frac, p.min_seed_prob = 0.5, -3.75
    p.min_map_len, p.min_mean_conf, p.min_top_conf = 25, 6.0, 1.85
    p.window_length1, p.window_length2 = 3, 6
    p.threshold1, p.threshold2, p.peak_height, p.min_mean, p.max_mean = 1.4, 9.0, 0.2, 0, 400
    p.bp_per_sec, p.sample_rate = 450, 4000
    return p


def make_descs(lens, dtype=0, cal=(1.0, 0.0, 1.0)):
    n = len(lens)
    d = (UncReadDesc * n)()
    off = 0
    for i, L in enumerate(lens):
        d[i].offset, d[i].n_samples, d[i].dtype = off, int(L), dtype
        d[i].cal_range, d[i].cal_offset, d[i].cal_digit = cal
        off += int(L)
    return d


def build():
    """Compiles the device source for the host."""
    src = os.path.join(EMUL_DIR, "emul_main.cpp")
    out = os.path.join(EMUL_DIR, "libunc_emul.so")
    deps = [src, os.path.join(EMUL_DIR, "warp_emul.hpp")] + \
           [os.path.join(ROOT, "uncalled_b200", "csrc", f) for f in
            ("unc_device.cuh", "unc_k2v2.cuh", "unc_dtw.cuh", "unc_k1.cuh", "unc_stream.cuh", "unc_stream_logic.hpp", "unc_ordered_logic.hpp", "unc_pdqsort.cuh", "unc_warp.cuh", "unc_host_index.hpp", "unc_host_params.hpp",
             "unc_selfalign.cuh", "unc_selfalign_host.hpp")]
    if os.path.exists(out) and all(os.path.getmtime(out) >= os.path.getmtime(d) for d in deps):
        return out
    subprocess.run(["g++", "-O2", "-g", "-std=c++17", "-ffp-contract=off", "-DUNC_EMUL", "-fPIC", "-shared",
                    "-I" + EMUL_DIR, "-I" + os.path.join(ROOT, "uncalled_b200", "csrc"), "-o", out, src],
                   check=True, capture_output=True)
    return out


_lib = None


def _bind(L):
    """argtypes of one loaded emulator library"""
    L.emu_index_load.restype = C.c_void_p
    L.emu_index_load.argtypes = [C.c_char_p, C.c_char_p, C.c_char_p]
    L.emu_index_free.argtypes = [C.c_void_p]
    L.emu_kmer_range.argtypes = [C.c_void_p, C.c_uint32, C.POINTER(C.c_uint64), C.POINTER(C.c_uint64)]
    L.emu_map_batch.argtypes = [C.c_void_p, C.POINTER(UncParams), C.POINTER(UncReadDesc), C.c_uint32, C.c_void_p,
                                C.POINTER(UncPaf), C.c_uint32, C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p,
                                C.c_int, C.c_uint32, C.c_int]
    L.emu_map_batch_ordered.argtypes = [C.c_void_p, C.POINTER(UncParams), C.POINTER(UncReadDesc), C.c_uint32, C.c_void_p,
                                        C.c_void_p, C.POINTER(UncPaf), C.POINTER(C.c_uint32), C.POINTER(C.c_uint32),
                                        C.c_uint32, C.c_int]
    L.emu_set_tie_order.argtypes = [C.c_int]
    L.emu_match_probs.argtypes = [C.c_void_p, C.c_float, C.c_void_p]
    L.emu_self_align.argtypes = [C.c_char_p, C.c_uint32, C.POINTER(C.c_uint64), C.POINTER(C.c_void_p), C.POINTER(C.c_void_p)]
    L.emu_glibc_rand.argtypes = [C.c_uint, C.c_uint32, C.c_void_p]
    L.emu_free.argtypes = [C.c_void_p]
    L.emu_free.restype = None
    L.emu_sa.argtypes = [C.c_void_p, C.c_uint64]
    L.emu_sa.restype = C.c_uint64
    L.emu_k1_stats.argtypes = [C.c_void_p]
    L.emu_stream_create.restype = C.c_void_p
    L.emu_stream_create.argtypes = [C.c_void_p, C.POINTER(UncParams), C.c_uint32, C.c_uint32, C.c_uint32, C.c_uint32]
    L.emu_stream_free.argtypes = [C.c_void_p]
    L.emu_stream_step.argtypes = [C.c_void_p, C.c_void_p, C.c_uint32, C.c_void_p, C.c_void_p, C.c_int]
    return L


def lib():
    """The emulator library."""
    global _lib
    if _lib is None:
        _lib = _bind(C.CDLL(build()))
    return _lib


class Emu:
    def __init__(self, prefix, preset="default"):
        self.L = lib()
        self.idx = self.L.emu_index_load(prefix.encode(), preset.encode(), MODEL_TABLE.encode())
        if not self.idx:
            raise RuntimeError("emu_index_load failed")
        self.params = default_params()

    def map_batch(self, signals, run_k2=True, max_blocks=4096, dtype=0, cal=(1.0, 0.0, 1.0), n_warps=8):
        """signals: list of 1-D arrays.  Returns (recs, events list, normed list, mean_event_len)."""
        lens = [len(s) for s in signals]
        npdt = np.float32 if dtype == 0 else np.int16
        flat = np.ascontiguousarray(np.concatenate(signals).astype(npdt))
        n = len(lens)
        d = make_descs(lens, dtype, cal)
        stride = max(lens)
        out = (UncPaf * n)()
        ev = np.zeros((n, stride), np.float32)
        nm = np.zeros((n, stride), np.float32)
        ne = np.zeros(n, np.uint32)
        mel = np.zeros(n, np.float32)
        rc = self.L.emu_map_batch(self.idx, C.byref(self.params), d, n, flat.ctypes.data, out, stride,
                                  ev.ctypes.data, nm.ctypes.data, ne.ctypes.data, mel.ctypes.data,
                                  1 if run_k2 else 0, max_blocks, n_warps)
        if rc != 0:
            raise RuntimeError("emu_map_batch rc=%d" % rc)
        return list(out), [ev[i, :ne[i]].copy() for i in range(n)], [nm[i, :ne[i]].copy() for i in range(n)], mel


    def set_tie_order(self, mode):
        """1: the exact-ties kernel (the reference's pdqsort reproduced), 0: the default kernel."""
        self.L.emu_set_tie_order(int(mode))

    def map_ordered(self, signals, carry=None, max_blocks=4096, n_warps=8):
        """unc_map_batch_ordered under the emulator: (recs, carry after, reads mapped again, extra rounds)."""
        lens = [len(s) for s in signals]
        flat = np.ascontiguousarray(np.concatenate(signals).astype(np.float32))
        n = len(lens)
        d = make_descs(lens)
        out = (UncPaf * n)()
        carry = np.zeros(32, np.uint32) if carry is None else np.array(carry, dtype=np.uint32, copy=True)
        nre, nro = C.c_uint32(), C.c_uint32()
        rc = self.L.emu_map_batch_ordered(self.idx, C.byref(self.params), d, n, flat.ctypes.data, carry.ctypes.data, out,
                                          C.byref(nre), C.byref(nro), max_blocks, n_warps)
        if rc != 0:
            raise RuntimeError("emu_map_batch_ordered rc=%d" % rc)
        return list(out), carry, nre.value, nro.value


def stream_reads(step, n_channels, signals, chunk_len, max_chunks=1000000):
    """The chunk-feeding policy of the product's python layer (uncalled_b200/stream.py feed_reads; pure python)."""
    from uncalled_b200.stream import feed_reads
    return feed_reads(step, n_channels, signals, chunk_len, max_chunks)


class EmuStream:
    """The streaming path under the emulator (tests/emul/emul_main.cpp emu_stream_*)."""

    def __init__(self, emu, n_channels, max_chunk_len, max_chunks=1000000, max_blocks=4096, n_warps=8):
        self.emu, self.n_channels, self.n_warps = emu, n_channels, n_warps
        self.h = emu.L.emu_stream_create(emu.idx, C.byref(emu.params), n_channels, max_chunk_len, max_chunks, max_blocks)
        self.max_chunks = max_chunks

    def step(self, descs, n, flat, res):
        rc = self.emu.L.emu_stream_step(self.h, descs, n, flat.ctypes.data, res, self.n_warps)
        if rc != 0:
            raise RuntimeError("emu_stream_step rc=%d" % rc)

    def map_reads(self, signals, chunk_len):
        return stream_reads(self.step, self.n_channels, signals, chunk_len, self.max_chunks)

    def close(self):
        if self.h:
            self.emu.L.emu_stream_free(self.h)
            self.h = None


def k1_stats():
    """(tiles, FSM re-run rounds, re-run lanes, reads flagged for the serial routine) of the last emu_map_batch."""
    a = (C.c_uint32 * 4)()
    lib().emu_k1_stats(a)
    return tuple(a)


PAF_KEYS = ("mapped", "fwd", "rid", "n_events", "events_used", "matches",
            "rd_len", "rd_st", "rd_en", "rf_st", "rf_en", "rf_len")


def paf_tuple(r):
    if not r.mapped:
        return (0, int(r.rd_len), int(r.n_events), int(r.events_used))
    return tuple(int(getattr(r, k)) for k in PAF_KEYS)


def self_align(prefix, sample_dist):
    """unc_selfalign.cuh on the CPU: (offsets, values) as numpy arrays."""
    import numpy as np
    L = lib()
    n, po, pv = C.c_uint64(), C.c_void_p(), C.c_void_p()
    if L.emu_self_align(prefix.encode(), sample_dist, C.byref(n), C.byref(po), C.byref(pv)) != 0:
        raise RuntimeError("emu_self_align failed")
    off = np.ctypeslib.as_array(C.cast(po, C.POINTER(C.c_uint64)), (n.value + 1,)).copy()
    val = np.ctypeslib.as_array(C.cast(pv, C.POINTER(C.c_uint64)), (max(int(off[-1]), 1),)).copy()[:int(off[-1])]
    L.emu_free(po); L.emu_free(pv)
    return off, val


def glibc_rand(seed, n):
    import numpy as np
    out = np.zeros(n, np.int32)
    lib().emu_glibc_rand(seed, n, out.ctypes.data)
    return out
