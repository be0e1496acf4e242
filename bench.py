#!/usr/bin/env python
"""bench.py -- reads/sec mapped on the headline workload of BASELINE.json.

Workload (configs[1]): E. coli-sized (4.7 Mb) index, 10 000 synthetic r9.4 reads x 4000 raw
samples per GPU (synthetic genome + reads from tools/synth.py, FM index from the product's own
bwa-compatible builder, .uncl thresholds from the committed reference fixture).  A "step" is
one pass of the whole hot path (event detection + normalisation kernel, mapper kernel) over
that batch.  With --gpus N every rank maps its own 10 000 reads (reads shard with no data-path
collective; torch.distributed is used only for the barrier and the max-over-ranks time).

  value  reads/s with the samples already resident in HBM (unc_map_batch_device)
  e2e    reads/s through the C-ABI call a MapPool makes, samples in pinned HOST memory,
         H2D of the samples and D2H of the PAF records inside the timed region
  --impl reference   the reference's own CPU mapper (oracle/_ref, else the oracle port) on
         all host cores over a bounded sample of the same workload

The benchmark writes nothing into the source tree (which may be read-only): the synthetic index is
built in a temporary directory that is removed at exit.
"""
import argparse
import atexit
import json
import os
import shutil
import subprocess
import sys
import tempfile
import threading
import time

sys.dont_write_bytecode = True
ROOT = os.path.dirname(os.path.abspath(__file__))
for p in (ROOT, os.path.join(ROOT, "tests"), os.path.join(ROOT, "tools")):
    sys.path.insert(0, p)

import numpy as np  # noqa: E402

METRIC = "reads/sec mapped (E. coli, 4k-sample reads) at 1/2/4/8 B200 vs CPU ref"
GENOME = "g4m7"
N_READS = 10000
N_SAMPLES = 4000
NOISE_MULT = 1.5          # SURVEY.md 8(d): noise N(0, 1.5 * level_stdv)
DUMP_BYTES = 64 << 20     # --dump-outputs writes at most this much

_data_dir = None


def data_dir():
    """Per-process scratch directory for the synthetic index, removed at exit."""
    global _data_dir
    if _data_dir is None:
        _data_dir = tempfile.mkdtemp(prefix="uncalled_b200_bench_")
        atexit.register(shutil.rmtree, _data_dir, True)
    return _data_dir


def workload(rank, n_reads=N_READS):
    import synth
    import synthdata
    prefix, g = synthdata.get_index(GENOME, data_dir())
    sig, truth = synth.reads(g, n_reads, N_SAMPLES, seed=7 + 1000 * rank, noise_mult=NOISE_MULT)
    return prefix, sig


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region."""

    def __init__(self, gpu):
        self.gpu, self.rows, self.proc = gpu, [], None

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            pass
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 7 for i in range(4) if r[3 + i] == "Active"})
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


def host_cpus():
    """CPUs this process can really use: the scheduler affinity capped by the cgroup CPU quota (a GPU lease is often a
    slice of the host: 128 CPUs visible, a quota of 16)."""
    import math
    aff = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    quota = None
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()[:2]
        if q != "max":
            quota = float(q) / float(per)
    except Exception:
        try:
            q = float(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                quota = q / per
        except Exception:
            pass
    usable = aff if quota is None else max(1, min(aff, int(math.ceil(quota))))
    return {"usable": usable, "affinity": aff, "cpu_count": os.cpu_count(), "cgroup_quota_cpus": quota}


def cpu_sample_size(threads, n_avail):
    """Reads of one CPU step: >= 48 per thread so that the last reads' tail stays a few percent, bounded so that a
    step is about 20 s on either kind of host."""
    return int(min(n_avail, min(4096, max(256, 48 * threads))))


def cpu_reference_run(prefix, sig, threads, budget_reads):
    """The reference CPU mapper (one long-lived Mapper per thread, as MapPool keeps them) over the first `budget_reads`
    reads; returns (reads/s, kind, seconds, mapped, PAF keys per read)."""
    import ctypes as C
    import orclib
    n = min(budget_reads, len(sig))
    flat = np.ascontiguousarray(sig[:n]).ravel()
    offs = (np.arange(n, dtype=np.uint64) * N_SAMPLES)
    lens = np.full(n, N_SAMPLES, np.uint32)
    if orclib.ref_available():
        R = orclib.ref()
        R.ref_load(prefix.encode(), b"default")
        out = (orclib.RefPaf * n)()
        t = time.time()
        R.ref_map_batch_mt(orclib.fp(flat), offs.ctypes.data_as(orclib.u64p), lens.ctypes.data_as(orclib.u32p), n,
                           threads, out)
        dt = time.time() - t
        return n / dt, "reference", dt, int(sum(r.mapped for r in out)), [orclib.paf_tuple(r) for r in out]
    O = orclib.Oracle(prefix)
    O.lib.orc_set_child_sort(1)          # the reference's pdqsort order (oracle/unc_oracle.c)
    t = time.time()
    out = O.map_batch(flat, offs, lens, threads)
    dt = time.time() - t
    return n / dt, "port", dt, int(sum(r.mapped for r in out)), [orclib.paf_tuple(r) for r in out]


def cpu_fresh_mapper_keys(prefix, sig, ids):
    """PAF keys of single reads mapped by the reference with a FRESH Mapper (ref_map_read): what a read gives when
    it is the first on its thread."""
    import orclib
    res = {}
    if orclib.ref_available():
        R = orclib.ref()
        for i in ids:
            rec = orclib.RefPaf()
            a = np.ascontiguousarray(sig[i])
            R.ref_map_read(orclib.fp(a), len(a), rec)
            res[i] = orclib.paf_tuple(rec)
    else:
        O = orclib.Oracle(prefix)
        O.lib.orc_set_child_sort(1)
        for i in ids:
            res[i] = orclib.paf_tuple(O.map_read(np.ascontiguousarray(sig[i])))
    return res


def parity_report(prefix, sig, ref_keys, gpu_default, gpu_exact):
    """In-bench parity gate: the GPU records of the CPU sample's reads against the reference's records of the same
    reads.  The timed reference run keeps one Mapper per thread, so a read may inherit sources_added_ flags from its
    thread's previous read (thread timing decides which); such reads are re-mapped with a fresh Mapper before they
    count as a mismatch.  The exact-ties kernel must then equal the reference on every read; the default kernel may
    differ only where the exact-ties kernel differs from it too (the reference's unstable sort decided a tie)."""
    import uncalled_b200 as U
    n = len(ref_keys)
    kd = [U.paf_key(gpu_default[i]) for i in range(n)]
    ke = [U.paf_key(gpu_exact[i]) for i in range(n)] if gpu_exact is not None else None
    diff_d = [i for i in range(n) if kd[i] != ref_keys[i]]
    diff_e = [i for i in range(n) if ke is not None and ke[i] != ref_keys[i]]
    fresh = cpu_fresh_mapper_keys(prefix, sig, sorted(set(diff_d) | set(diff_e)))
    bad_e = [i for i in diff_e if ke[i] != fresh[i]]
    carry = [i for i in diff_d if kd[i] == fresh[i]]
    tie = [i for i in diff_d if kd[i] != fresh[i] and ke is not None and ke[i] == fresh[i]]
    bad_d = [i for i in diff_d if i not in carry and i not in tie]
    rep = {"reads": n,
           "default_kernel": {"identical": n - len(diff_d), "differing_ids": diff_d[:32],
                              "explained_by_mapper_carry": len(carry), "explained_by_tie_order": len(tie),
                              "unexplained": bad_d[:32]},
           "exact_ties_kernel": None if ke is None else {"identical": n - len(diff_e), "differing_ids": diff_e[:32],
                                                         "explained_by_mapper_carry": len(diff_e) - len(bad_e),
                                                         "unexplained": bad_e[:32]},
           "fields": "mapped, strand, rid, events, matches, rd_len/st/en, rf_st/en/len",
           "ok": not bad_d and not bad_e}
    return rep


def run_reference_arm(args, rank, world):
    if rank != 0:
        return
    cpus = host_cpus()
    threads = cpus["usable"]
    prefix, sig = workload(0, n_reads=cpu_sample_size(threads, N_READS))
    sample = len(sig)
    times = []
    for i in range(args.warmup + args.steps):
        rps, kind, dt, mapped, _ = cpu_reference_run(prefix, sig, threads, sample)
        if i >= args.warmup:
            times.append(dt)
    ms = 1e3 * float(np.mean(times))
    value = sample / (ms / 1e3)
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "reads/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32/f64+u64", "data": "synthetic",
            "config": {"workload": "configs[1]: E. coli-sized 4.7 Mb synthetic index, %d synthetic r9.4 reads x %d "
                                   "samples per GPU, noise %.1f x level stdv (SURVEY 8d)" % (N_READS, N_SAMPLES, NOISE_MULT),
                       "reads_per_gpu": N_READS, "samples_per_read": N_SAMPLES,
                       "reads_per_step": sample, "note": "each step is a bounded sample (the first reads) of that workload, on the host CPUs this "
                                                         "process can use; rank 0 only"},
            "cpu_baseline": {"value": value, "unit": "reads/s", "cores": threads, "kind": kind, "host_cpus": cpus,
                             "reads_per_s_per_thread": value / threads,
                             "sample": "%d reads x %d samples per step, %d threads (one long-lived Mapper per thread, as MapPool)" % (sample, N_SAMPLES, threads)},
            "e2e": {"value": value, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def stream_job(sm, sigs, steps, warmup, barrier, on_timed_start=None):
    """W untimed + K timed passes of all reads through a stream mapper (anything with .step and .map_reads);
    returns (total ms of the K passes, per-pass counters of the C-ABI steps, the last pass's results, step latencies)."""
    counters = {"steps": 0, "chunks": 0, "bytes": 0}
    lat = []
    inner = sm.step

    def counting_step(descs, n, flat, res):
        counters["steps"] += 1
        counters["chunks"] += sum(1 for i in range(n) if descs[i].n_samples)
        counters["bytes"] += int(flat.nbytes)
        inner(descs, n, flat, res)
        if hasattr(sm, "last_step_ms"):
            lat.append(sm.last_step_ms())
    sm.step = counting_step
    for _ in range(warmup):
        sm.map_reads(sigs)
    for k in counters:
        counters[k] = 0
    del lat[:]
    if on_timed_start:
        on_timed_start()
    barrier()
    t0 = time.perf_counter()
    res = None
    for _ in range(steps):
        res = sm.map_reads(sigs)
    barrier()
    ms = (time.perf_counter() - t0) * 1e3
    sm.step = inner
    return ms, counters, res, lat


def cpu_stream_run(prefix, sigs, n_channels, chunk_len, threads):
    """The reference's streaming path on the CPU (oracle/_ref: one Mapper per channel, chunk by chunk through
    Mapper::new_read / add_chunk / process_chunk / map_chunk, channels on `threads` worker threads) over the same reads."""
    import ctypes as C
    import orclib
    n = len(sigs)
    flat = np.ascontiguousarray(np.concatenate(sigs), np.float32)
    lens = np.array([len(x) for x in sigs], np.uint32)
    offs = np.concatenate([[0], np.cumsum(lens[:-1], dtype=np.uint64)]).astype(np.uint64)
    if not orclib.ref_available():
        return None
    R = orclib.ref()
    R.ref_load(prefix.encode(), b"default")
    out = (orclib.RefPaf * n)()
    nch = (C.c_uint32 * n)()
    en = (C.c_int32 * n)()
    t = time.time()
    R.ref_stream_channels_mt(orclib.fp(flat), offs.ctypes.data_as(orclib.u64p), lens.ctypes.data_as(orclib.u32p), n, n_channels,
                             chunk_len / float(bench_sample_rate()), 1000000, threads, out, nch, en)
    dt = time.time() - t
    keys = [(orclib.paf_tuple(out[i]), int(nch[i]), int(en[i])) for i in range(n)]
    return n / dt, dt, int(sum(nch)), keys


def bench_sample_rate():
    return 4000.0


def run_stream_workload(args, rank, local_rank, world):
    """configs[4]: chunk streaming (450-sample chunks = chunk_time 0.1125 s) over 512 channels of one flow cell with
    persistent per-channel device state (unc_stream_step), reads following each other on every channel; with --gpus N the
    channels are dealt out c -> rank c mod N (64 per GPU at N = 8).  A step of the metric = all reads of the workload
    streamed to completion.  Every chunk crosses the host boundary (host buffer -> H2D inside unc_stream_step), so there is
    only an end-to-end number: `value` repeats it and says so.  Also reported: chunks/s and the per-step wall-clock time
    (the decision latency a ReadUntil client sees for every chunk of the step)."""
    import torch
    import torch.distributed as dist
    import synth
    import synthdata
    import uncalled_b200 as U
    total_channels, chunk_len = 512, 450
    n_channels = (total_channels + world - 1 - rank) // world       # channel c lives on rank c % world
    n_reads = n_channels * args.reads_per_channel
    prefix, g = synthdata.get_index(GENOME, data_dir())
    sig, _ = synth.reads(g, n_reads, N_SAMPLES, seed=7 + 1000 * rank, noise_mult=NOISE_MULT)
    sigs = [sig[i] for i in range(n_reads)]
    idx = U.Index(prefix, device=local_rank)
    sm = U.StreamMapper(idx, n_channels, chunk_len)
    sampler = ClockSampler(local_rank)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()
    ms, counters, res, lat = stream_job(sm, sigs, args.steps, args.warmup, barrier, sampler.start if rank == 0 else None)
    clocks = sampler.stop() if rank == 0 else None
    v = torch.tensor([ms], dtype=torch.float64, device="cuda")
    tot = torch.tensor([float(n_reads), float(counters["chunks"]) / args.steps], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(v, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    ms = float(v[0]) / args.steps
    all_reads, all_chunks = float(tot[0]), float(tot[1])
    value = all_reads / (ms / 1e3)
    if rank == 0:
        mapped = sum(1 for r in res if r is not None and r[0] == 2)
        la = np.array(lat) if lat else np.zeros(1)
        line = {"metric": METRIC, "value": value, "unit": "reads/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "f32/f64 events, u32 FM index", "data": "synthetic",
                "config": {"workload": "configs[4]: chunk streaming, %d channels x %d-sample chunks (%d channels on this GPU), %d reads x %d "
                                       "samples per channel, 4.7 Mb synthetic index, noise %.1f x level stdv"
                                       % (total_channels, chunk_len, n_channels, args.reads_per_channel, N_SAMPLES, NOISE_MULT),
                           "timing": "wall clock around the whole streamed job, barrier + cuda.synchronize on both sides "
                                     "(every step is a synchronous C-ABI call); value == e2e (no device-resident variant)",
                           "chunk_steps_per_job": counters["steps"] / args.steps, "chunks_per_job": all_chunks,
                           "mapped_fraction": mapped / n_reads},
                "chunks_per_s": all_chunks / (ms / 1e3),
                "step_latency_ms": {"p50": float(np.percentile(la, 50)), "p99": float(np.percentile(la, 99)), "max": float(la.max()),
                                    "note": "wall clock of one unc_stream_step on rank 0 (H2D of the chunks, event detection + mapping of all "
                                            "their events, D2H of the results): every chunk of the step gets its decision after this long"},
                "e2e": {"value": value, "unit": "reads/s", "h2d_bytes_per_step": int(counters["bytes"] / args.steps),
                        "d2h_bytes_per_step": int(counters["chunks"] / args.steps * 160), "ms_per_step": ms},
                "gpu_launches": int(2 * counters["steps"]), "clocks": clocks}
        if not args.no_cpu_baseline and world == 1:
            cpus = host_cpus()
            nsub = min(n_channels, max(16, 2 * cpus["usable"]))          # a bounded number of whole channels
            sub = [sigs[i] for i in range(n_reads) if i % n_channels < nsub]
            r = cpu_stream_run(prefix, sub, nsub, chunk_len, cpus["usable"])
            if r is not None:
                rps, dt, nchunks, keys = r
                import orclib
                # parity on the same channels, both sides starting from fresh per-channel state (the timed passes above
                # reuse one stream, whose channels carry their normaliser statistics and flags from pass to pass)
                sm2 = U.StreamMapper(idx, nsub, chunk_len)
                gpu = sm2.map_reads(sub)
                sm2.close()
                bad = [j for j in range(len(sub)) if gpu[j] is None or (U.paf_key(gpu[j][3]), int(gpu[j][2]), int(gpu[j][1])) != keys[j]]
                line["cpu_baseline"] = {"value": rps, "unit": "reads/s", "chunks_per_s": nchunks / dt, "cores": cpus["usable"], "kind": "reference",
                                        "host_cpus": cpus, "sample": "%d channels x %d reads (the first channels of the same workload), %d threads, "
                                                                     "%.1f s; one Mapper per channel as RealtimePool" % (nsub, args.reads_per_channel, cpus["usable"], dt)}
                line["parity"] = {"reads": len(sub), "identical": len(sub) - len(bad), "differing_ids": bad[:32],
                                  "fields": "PAF fields, chunks used, ended; default kernel vs the unmodified reference (tie order may differ, DESIGN.md section 2)"}
        print(json.dumps(line), flush=True)
    sm.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def run_fast5_workload(args, rank, local_rank, world):
    """configs[2]/[3] as written: multi-read fast5 files (4000 reads x 4000 samples each, gzip int16; bench_data/
    bench_reads_4000x4000.fast5 from tools/make_bench_fast5.py) -> the product's own fast5 reader on the host threads ->
    int16 over PCIe -> calibration + event detection + mapping on the GPU -> PAF records, through the public MapPool
    (uncalled_b200/api.py: what `python -m uncalled_b200 map` drives).  With --gpus N the files are dealt out round-robin
    to the ranks (one process per GPU, no collective), --files is the TOTAL number of files (x 4000 reads).  The same
    file is queued repeatedly: decode work and PCIe traffic are real every time.  A step = all files once."""
    import torch
    import torch.distributed as dist
    import synthdata
    import uncalled_b200 as U
    from uncalled_b200 import api
    from uncalled_b200.fast5 import Fast5File
    path = os.path.join(ROOT, "bench_data", "bench_reads_4000x4000.fast5")
    if not os.path.exists(path):
        raise SystemExit("bench_data/bench_reads_4000x4000.fast5 is missing: run tools/make_bench_fast5.py where /root/reference exists")
    prefix, _ = synthdata.get_index(GENOME, data_dir())
    cpus = host_cpus()
    threads = max(1, cpus["usable"] // world)
    my_files = [path for i in range(args.files) if i % world == rank]
    n_mine = 4000 * len(my_files)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def one_pass():
        conf = api.Conf()
        conf.bwa_prefix, conf.threads, conf.device, conf.batch_reads = prefix, threads, local_rank, args.batch_reads
        pool = api.MapPool(conf)
        for f in my_files:
            pool.add_fast5(f)
        n = mapped = 0
        while pool.running():
            for p in pool.update():
                n += 1
                mapped += 1 if p.is_mapped() else 0
        pool.stop()
        return n, mapped
    for _ in range(min(args.warmup, 1)):
        one_pass()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    barrier()
    t0 = time.perf_counter()
    n = mapped = 0
    for _ in range(args.steps):
        a, b = one_pass()
        n += a
        mapped += b
    barrier()
    ms = (time.perf_counter() - t0) * 1e3
    clocks = sampler.stop() if rank == 0 else None
    assert n == n_mine * args.steps
    # decode alone on this rank's threads (the host stage's capacity)
    t1 = time.perf_counter()
    F = Fast5File(path)
    F.load(0, F.n_reads, threads=threads)
    F.close()
    decode_rps = 4000 / (time.perf_counter() - t1)
    v = torch.tensor([ms], dtype=torch.float64, device="cuda")
    w = torch.tensor([float(n), float(mapped), decode_rps], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(v, op=dist.ReduceOp.MAX)
        dist.all_reduce(w, op=dist.ReduceOp.SUM)
    ms = float(v[0]) / args.steps
    total = float(w[0]) / args.steps
    value = total / (ms / 1e3)
    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "reads/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": ms, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
                "dtype": "i16 DAC in, f32/f64 events, u32 FM index", "data": "synthetic",
                "config": {"workload": "configs[2]/[3]: %d multi-read fast5 files x 4000 reads x 4000 samples (%d reads) through MapPool: host fast5 "
                                       "decode (%d threads per rank) -> i16 over PCIe -> GPU; 4.7 Mb synthetic index, noise 1.5 x level stdv"
                                       % (args.files, int(total), threads),
                           "timing": "wall clock around the whole job incl. file reading and inflate, barrier + cuda.synchronize on both sides",
                           "batch_reads": args.batch_reads, "mapped_fraction": float(w[1]) / float(w[0])},
                "e2e": {"value": value, "unit": "reads/s", "h2d_bytes_per_step": int(total * 8000), "d2h_bytes_per_step": int(total * 120), "ms_per_step": ms},
                "stages": {"host_decode_reads_per_s_all_ranks": float(w[2]), "host_cpus": cpus,
                           "note": "decode capacity measured alone on the same threads; the GPU stage's capacity is the default workload's `value`; "
                                   "the slower of the two bounds this number"},
                "gpu_launches": int(4 * ((n_mine + args.batch_reads - 1) // args.batch_reads)) * world, "clocks": clocks}
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def dump_outputs(out_dir, recs):
    """The PAF records a caller of the timed path receives, one DIR/paf_<field>.npy per field (float64 holds every
    field exactly), and DIR/read_index.npy naming their reads: all of them, or a fixed seeded sample when all of them
    would take more than DUMP_BYTES."""
    fields = recs.dtype.names
    per_read = 8 * (len(fields) + 1)
    ids = np.arange(len(recs))
    budget = (DUMP_BYTES - 128 * (len(fields) + 1)) // per_read        # 128 bytes: the header of a .npy file
    if len(recs) > budget:
        ids = np.sort(np.random.default_rng(0).choice(len(recs), budget, replace=False))
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "read_index.npy"), ids.astype(np.float64))
    for f in fields:
        np.save(os.path.join(out_dir, "paf_%s.npy" % f), recs[f][ids].astype(np.float64))


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--reads", type=int, default=N_READS)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-extras", action="store_true", help="skip the side modes (two-pool overlap, ordered, exact ties) that ride along at N=1")
    ap.add_argument("--overlap", action="store_true",
                    help="additionally time the steps with two pools used alternately (unc_map_batch_submit / _wait): the "
                         "next batch's CTAs fill the SMs that the previous batch's tail leaves idle; reported under 'overlap'")
    ap.add_argument("--ordered", action="store_true",
                    help="additionally time unc_map_batch_ordered (`uncalled map -t 1` semantics: one long-lived Mapper, reads in "
                         "order, resolved by re-mapping the reads whose predecessor left flags set); reported under 'ordered'")
    ap.add_argument("--exact-ties", action="store_true",
                    help="additionally time the exact-ties kernel (unc_pool_set_tie_order(1): the reference's unstable pdqsort "
                         "reproduced serially per event); reported under 'exact_ties'")
    ap.add_argument("--workload", default="batch", choices=["batch", "stream", "fast5"],
                    help="batch: configs[1] (the headline); stream: chunk streaming over 512 channels (configs[4]); "
                         "fast5: multi-read fast5 files through MapPool, decode included (configs[2]/[3] as written)")
    ap.add_argument("--files", type=int, default=16, help="fast5 workload: total number of 4000-read files (all ranks together)")
    ap.add_argument("--batch-reads", type=int, default=8000, help="fast5 workload: reads per GPU batch")
    ap.add_argument("--reads-per-channel", type=int, default=2)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="batch workload: after the timed steps, write the PAF records of the last timed step (rank 0) to "
                         "DIR as float64 .npy files, one per field, for comparing two builds on identical inputs")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or args.workload != "batch"):
        ap.error("--dump-outputs is available for the batch workload of --impl ours only")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        run_reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import uncalled_b200 as U

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product has no CPU path")
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))

    if args.workload == "stream":
        run_stream_workload(args, rank, local_rank, world)
        return
    if args.workload == "fast5":
        run_fast5_workload(args, rank, local_rank, world)
        return

    n_reads = args.reads
    prefix, sig = workload(rank, n_reads)
    descs = U.make_descs([N_SAMPLES] * n_reads)
    idx = U.Index(prefix, device=local_rank)
    bm = U.BatchMapper(idx, max_reads=n_reads, max_samples=n_reads * N_SAMPLES)
    host = torch.from_numpy(sig.reshape(-1)).pin_memory()
    dev = host.to("cuda:%d" % local_rank)
    torch.cuda.synchronize()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps):
        """K steps bracketed by barrier+synchronize; returns (max-over-ranks device ms, wall ms, timings)."""
        barrier()
        t0 = time.time()
        dev_ms, tms = 0.0, []
        for _ in range(steps):
            fn()
            tm = bm.timing()          # CUDA events recorded on the launching stream
            dev_ms += tm["total_ms"]
            tms.append(tm)
        barrier()
        wall_ms = (time.time() - t0) * 1e3
        v = torch.tensor([dev_ms, wall_ms], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(v, op=dist.ReduceOp.MAX)
        return float(v[0]), float(v[1]), tms

    out_holder = {}

    def step_device():
        out_holder["o"] = bm.map_device(dev.data_ptr(), descs)

    def step_host():
        out_holder["o"] = bm.map(host.numpy(), descs)

    timed(step_device, args.warmup)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
    dev_ms, wall_ms, tms = timed(step_device, args.steps)
    out_dev = out_holder["o"].copy()
    timed(step_host, 1)
    e2e_ms, e2e_wall, tms_h = timed(step_host, args.steps)
    clocks = sampler.stop() if rank == 0 else None
    out_host = out_holder["o"]
    assert np.array_equal(out_dev, out_host), "device-resident and host-buffer paths disagree"
    assert int((out_dev["status"] != 0).sum()) == 0, "a read overflowed its device workspace"

    # the side modes ride along at N=1 with their own bounded step counts (the flags force them at N>1 as well)
    extras = world == 1 and not args.no_extras
    x_steps = max(1, min(args.steps, 3))
    overlap = None
    if args.overlap or extras:
        bm2 = U.BatchMapper(idx, max_reads=n_reads, max_samples=n_reads * N_SAMPLES)
        pools = [bm, bm2]

        def pipelined(steps):
            barrier()
            t0 = time.time()
            outs = []
            pools[0].record(0)                                   # device-side start mark
            pools[0].submit(dev.data_ptr(), descs, on_device=True)
            for k in range(1, steps):
                pools[k % 2].submit(dev.data_ptr(), descs, on_device=True)
                outs.append(pools[(k - 1) % 2].wait())
            pools[0].record(1)
            pools[1].record(1)                                   # end marks behind the last batch of either pool
            outs.append(pools[(steps - 1) % 2].wait())
            dev_span = max(pools[0].elapsed_ms(0, pools[0], 1), pools[0].elapsed_ms(0, pools[1], 1))
            barrier()
            w = torch.tensor([dev_span, (time.time() - t0) * 1e3], dtype=torch.float64, device="cuda")
            if world > 1:
                dist.all_reduce(w, op=dist.ReduceOp.MAX)
            return float(w[0]), float(w[1]), outs
        ov_steps = max(2, min(args.steps, 4))
        pipelined(2)
        ov_ms, ov_wall, outs = pipelined(ov_steps)
        assert all(np.array_equal(o_, out_dev) for o_ in outs), "pipelined batches disagree with the single-pool result"
        overlap = {"value": world * n_reads * ov_steps / (ov_ms / 1e3), "unit": "reads/s", "pools": 2, "steps": ov_steps,
                   "ms_per_step": ov_ms / ov_steps, "wall_ms_per_step": ov_wall / ov_steps,
                   "note": "CUDA events from the first submit to the end of the last batch on either pool, max over ranks; "
                           "the last step's tail is not hidden"}
        bm2.close()

    ordered = None
    if args.ordered or extras:
        oh = {}

        def step_ordered():
            oh["r"] = bm.map_ordered(dev.data_ptr(), descs, on_device=True)
        timed(step_ordered, 1)
        od_ms, od_wall, _ = timed(step_ordered, x_steps)
        recs_o, _, n_re, n_ro = oh["r"]
        ordered = {"value": world * n_reads / (od_ms / x_steps / 1e3), "unit": "reads/s", "steps": x_steps, "ms_per_step": od_ms / x_steps,
                   "wall_ms_per_step": od_wall / x_steps, "reads_mapped_again": n_re, "extra_rounds": n_ro,
                   "records_differing_from_plain_batch": int((recs_o != out_dev).sum()),
                   "note": "device-resident samples; sum of the CUDA-event times of all rounds, max over ranks"}

    exact_ties = None
    recs_e = None
    if args.exact_ties or extras:
        bm.set_tie_order(1)
        try:
            ex_ms, ex_wall, _ = timed(step_device, 1)      # one step: this mode is a verification mode, several times slower
            recs_e = out_holder["o"].copy()
        finally:
            bm.set_tie_order(0)
        paf_fields = ["mapped", "fwd", "rid", "events_used", "matches", "rd_st", "rd_en", "rf_st", "rf_en"]
        exact_ties = {"value": world * n_reads / (ex_ms / 1e3), "unit": "reads/s", "steps": 1, "ms_per_step": ex_ms,
                      "reads_with_a_PAF_field_differing_from_default_kernel": int(np.any([recs_e[k] != out_dev[k] for k in paf_fields], axis=0).sum()),
                      "note": "k2_map_exact, device-resident samples, CUDA events, max over ranks"}

    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, out_dev)

    ms_per_step = dev_ms / args.steps
    value = world * n_reads / (ms_per_step / 1e3)
    e2e_value = world * n_reads / (e2e_ms / args.steps / 1e3)

    if rank == 0:
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak = float(peaks.get("hbm_gbs", 6650.0))
        peak_kind = "measured (MEASURED_PEAKS.json hbm_gbs)" if "hbm_gbs" in peaks else "fallback 6.65 TB/s"
        k2_ms = float(np.mean([t["k2_ms"] for t in tms]))
        k1_ms = float(np.mean([t["k1_events_ms"] for t in tms]))          # the event-detection kernel alone
        k1_all_ms = float(np.mean([t["k1_ms"] for t in tms]))            # + serial-redo + normaliser launches
        # algorithmic bytes of the mapper kernel (DESIGN.md, SURVEY.md 8(d)): exact counters
        o = out_dev
        k2_bytes = 64.0 * float(o["n_occ_blocks"].sum()) + 8.0 * float(o["n_seeds"].sum()) + \
            2 * 56.0 * float(o["n_children"].sum() + o["n_sources"].sum())
        k1_bytes = 4.0 * n_reads * N_SAMPLES + 4.0 * float(o["n_events"].sum())
        achieved = k2_bytes / (k2_ms / 1e3) / 1e9
        traffic = None
        try:
            traffic = json.load(open(os.path.join(ROOT, "profiles", "k2_traffic.json"))).get("dram_bytes_per_launch")
        except Exception:
            pass
        line = {
            "metric": METRIC, "value": value, "unit": "reads/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32/f64 events, u32 FM index", "data": "synthetic",
            "config": {"workload": "configs[1]: E. coli-sized 4.7 Mb synthetic index, %d synthetic r9.4 reads x %d "
                                   "samples per GPU, noise %.1f x level stdv (SURVEY 8d)" % (n_reads, N_SAMPLES, NOISE_MULT),
                       "reads_per_gpu": n_reads, "samples_per_read": N_SAMPLES, "parallelism": "reads sharded, replicas x%d" % world,
                       "l2": "inputs (%.0f MB/GPU) larger than L2; per-warp path state (GBs) streams through HBM" % (n_reads * N_SAMPLES * 4 / 1e6),
                       "mapped_fraction": float(o["mapped"].mean())},
            "e2e": {"value": e2e_value, "unit": "reads/s", "h2d_bytes_per_step": int(tms_h[-1]["h2d_bytes"]),
                    "d2h_bytes_per_step": int(tms_h[-1]["d2h_bytes"]), "ms_per_step": e2e_ms / args.steps},
            "gpu_launches": int(sum(t["kernel_launches"] for t in tms)),
            "wall_ms_per_step": wall_ms / args.steps,
            "overlap": overlap,
            "ordered": ordered,
            "exact_ties": exact_ties,
            "clocks": clocks,
            "roofline": {"kernel": "k2_map", "bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "peak_kind": peak_kind,
                         "algorithmic_bytes_per_launch": k2_bytes, "launch_ms": k2_ms,
                         "note": "latency/L2-bound graph kernel; Occ blocks of the 7 MB index are L2 hits"},
            "roofline_k1": {"kernel": "k1_events", "bound": "hbm", "achieved": k1_bytes / (k1_ms / 1e3) / 1e9, "peak": peak,
                            "unit": "GB/s", "frac": k1_bytes / (k1_ms / 1e3) / 1e9 / peak, "launch_ms": k1_ms,
                            "all_k1_launches_ms": k1_all_ms, "k1_stats(tiles,fsm_rerun_rounds,rerun_lanes,serial_reads)": list(bm.k1_stats()),
                            "algorithmic_bytes_per_launch": k1_bytes},
        }
        if not args.no_cpu_baseline and world == 1:
            cpus = host_cpus()
            threads = cpus["usable"]
            sample = cpu_sample_size(threads, n_reads)
            rps, kind, dt, mapped, ref_keys = cpu_reference_run(prefix, sig, threads, sample)
            line["cpu_baseline"] = {"value": rps, "unit": "reads/s", "cores": threads, "kind": kind, "host_cpus": cpus,
                                    "reads_per_s_per_thread": rps / threads,
                                    "sample": "first %d reads of the same workload, %d threads (one long-lived Mapper per thread, "
                                              "as MapPool), %.1f s" % (sample, threads, dt)}
            # parity gate: the same reads, both arms, on this box
            line["parity"] = parity_report(prefix, sig, ref_keys, out_dev, recs_e)
            if not line["parity"]["ok"]:
                print(json.dumps(line), flush=True)
                raise SystemExit("parity gate failed: GPU records differ from the reference's beyond the documented tie / carry cases")
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
