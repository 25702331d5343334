#!/usr/bin/env python
"""bench.py -- the driver's measurement contract for the k-mer hot path.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

--dump-outputs DIR writes what the timed path hands its caller after the last of the K timed steps (and the final
all-reduce), as float64 .npy files: hist.npy (the int64 histogram the K steps accumulate into) and status.npy (the
status words).  The inputs depend only on the arguments, so two builds run with the same arguments can be compared
file by file.  A histogram of more than 2^21 bins is written as a fixed, seeded sample of 2^21 bins, with their
indices in hist_index.npy, which keeps the dump under 64 MB.

A "step" is one pass of the fused hot path (FASTQ chunk bytes -> 2-bit codes -> k=31 rolling hash -> bincount) over
one batch of synthetic 150 bp reads that is already resident in HBM (BASELINE.json configs[1]: 10 M x 150 bp per GPU,
3.17 GB -- far larger than the 126 MB L2, so no L2 flush is needed between steps).  Batches accumulate into one
histogram per GPU; N > 1 is BASELINE configs[4] sharded (every rank counts its own record range, weak scaling) and the
timed region ends with the ONE NCCL all-reduce of the final histogram north_star describes (its duration is reported
separately).  Timing: CUDA events on the launching stream around exactly K steps (+ that all-reduce), barrier +
synchronize on both sides, max over ranks.

The JSON line also carries
  roofline      achieved algorithmic GB/s of the dominant kernel (event-timed per launch) vs the measured HBM peak
  headline_2^24 the same workload into 2^24 buckets (SURVEY 8d's default for the hashed-bucket extension)
  extra         BASELINE configs 3 (100 M reads, minimizers), 4 (a sample of sacCer3.fa, k=21), the materialising get_kmers mode,
                k=5 exact; each min/median over >= 10 repetitions (3 for the 100 M-read one)
  oracle_check  the 10 M-read headline table compared bin by bin with oracle/kmer_oracle.c (untimed)
  e2e           the same metric through the host-buffer C-ABI call (pinned host chunk -> sliced H2D overlapped with
                the count -> D2H of the histogram), every step
  e2e_api       the same through the kept reader API: for chunk in bnp.open(path).read_chunks(): count_kmers_hashed(...)
  cpu_baseline  the oracle's NumPy port of the reference path on a bounded sample (rank 0, N=1); the single-core
                figure is the primary one (the reference is single-threaded)
`--impl reference` times that CPU port on all host cores instead (the reference itself cannot be imported: its
npstructures dependency is absent, see DESIGN.md).
"""
import argparse
import json
import multiprocessing as mp
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

READ_LEN = 150
RECORD_BYTES = 317
METRIC = "Gbases/s k=31 hash+count on 150bp reads"
KERNEL_NAME = "bnpk::ws::tile_ws_kernel (fused split+encode+hash+count, warp-specialised, TMA ring)"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--reads", type=int, default=10_000_000, help="reads per GPU and step")
    ap.add_argument("--k", type=int, default=31)
    ap.add_argument("--buckets", type=int, default=1 << 14,
                    help="histogram bins: hash mod buckets (2^14 = the shared-memory-privatised table)")
    ap.add_argument("--window", type=int, default=0, help="minimizer window in bases (0 = plain k-mers)")
    ap.add_argument("--e2e-steps", type=int, default=10)
    ap.add_argument("--reps", type=int, default=10, help="repetitions of the secondary configurations")
    ap.add_argument("--no-extra", action="store_true", help="skip the secondary configurations")
    ap.add_argument("--config3-reads", type=int, default=100_000_000)
    ap.add_argument("--cpu-sample-reads", type=int, default=200_000)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the timed path's outputs as DIR/<name>.npy")
    return ap.parse_args()


def host_cores():
    try:
        return len(os.sched_getaffinity(0))
    except AttributeError:  # pragma: no cover
        return os.cpu_count() or 1


# ------------------------------------------------------------------------------------------------
# CPU baseline = the oracle's NumPy port of the reference path (test infrastructure; timed, not shipped)
# ------------------------------------------------------------------------------------------------
_CPU_CHUNK = None


def _cpu_init(chunk_reads):
    """Every worker builds one ~4.8 MB synthetic chunk once (not timed)."""
    global _CPU_CHUNK
    from oracle import bnp_oracle as oracle
    _CPU_CHUNK = oracle.synthetic_fastq((os.getpid() % 1000) * chunk_reads, chunk_reads)


def _cpu_worker(job):
    k, buckets, window = job
    from oracle import bnp_oracle as oracle
    t0 = time.perf_counter()
    hist, size, n_bases = oracle.fastq_chunk_kmer_counts(_CPU_CHUNK, k, buckets, True, window_size=window)
    return time.perf_counter() - t0, n_bases, int(hist.sum())


def cpu_baseline(k, buckets, window, sample_reads, n_procs):
    """The reference op sequence (oracle port) on `n_procs` processes, each over ~4.8 MB chunks (bionumpy's default
    min_chunk_size, io/parser.py:96), input already in RAM.  Returns (Gbases/s, bases, wall seconds)."""
    chunk_reads = 15_000
    n_jobs = max(n_procs, sample_reads // chunk_reads)
    jobs = [(k, buckets, window)] * n_jobs
    if n_procs == 1:
        _cpu_init(chunk_reads)
        _cpu_worker(jobs[0])
        res = [_cpu_worker(j) for j in jobs]
        wall = sum(r[0] for r in res)
    else:
        with mp.get_context("fork").Pool(n_procs, initializer=_cpu_init, initargs=(chunk_reads,)) as pool:
            pool.map(_cpu_worker, jobs[:n_procs], chunksize=1)          # warm up (imports, page faults)
            t0 = time.perf_counter()
            res = pool.map(_cpu_worker, jobs, chunksize=1)
            wall = time.perf_counter() - t0
    bases = sum(r[1] for r in res)
    return bases / wall / 1e9, bases, wall


# ------------------------------------------------------------------------------------------------
def sample_clocks(stop_evt, out):
    """nvidia-smi clocks/throttle reasons during the timed region (B200_PROFILING.md recipe), every GPU."""
    q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
         "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
    try:
        p = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100"],
                             stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
    except Exception:
        return
    lines = []

    def reader():
        for line in p.stdout:
            lines.append(line)
    t = threading.Thread(target=reader, daemon=True)
    t.start()
    stop_evt.wait()
    p.terminate()
    t.join(timeout=2)
    out.extend(lines)


def summarize_clocks(lines, gpu_index):
    sm, mx, reasons = [], [], set()
    for ln in lines:
        f = [x.strip() for x in ln.split(",")]
        if len(f) < 9 or f[0] != str(gpu_index):
            continue
        try:
            sm.append(float(f[1]))
            mx.append(float(f[2]))
        except ValueError:
            continue
        for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
            if v.lower().startswith("active"):
                reasons.add(name)
    if not sm:
        return None
    sm.sort()
    return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": max(mx), "reasons": sorted(reasons), "samples": len(sm)}


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


def traffic_from_profiles(key):
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get(key)
        except Exception:
            return None
    return None


# ------------------------------------------------------------------------------------------------
def run_reference(args, rank, world):
    """--impl reference: the reference's CPU path (oracle port, all host cores) on the same config."""
    if rank != 0:
        return
    cores = host_cores()
    vals = []
    sample = max(args.cpu_sample_reads, 15_000 * cores * 2)      # at least two ~4.8 MB chunks per core and step
    for i in range(args.warmup + args.steps):
        v, bases, wall = cpu_baseline(args.k, args.buckets, args.window, sample, cores)
        if i >= args.warmup:
            vals.append((v, wall))
    value = sum(v for v, _ in vals) / len(vals)
    ms = 1e3 * sum(w for _, w in vals) / len(vals)
    v1, _, _ = cpu_baseline(args.k, args.buckets, args.window, 60_000, 1)
    line = {
        "impl": "reference", "metric": METRIC, "value": round(value, 4), "unit": "Gbases/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": round(ms, 2), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "int64", "data": "synthetic",
        "config": {"workload": f"synthetic {args.reads}x150bp FASTQ per GPU, k={args.k}, hash mod {args.buckets} bincount"
                               + (f", minimizer window {args.window}" if args.window else ""),
                   "sample": f"same 317-byte records and metric; each step samples {sample} reads in ~4.8 MB chunks (the "
                             f"reference's default min_chunk_size) instead of holding {args.reads} reads resident"},
        "cpu_baseline": {"value": round(value, 4), "unit": "Gbases/s", "cores": cores, "kind": "port",
                         "sample": f"{sample} reads x {args.steps} steps, one process per core "
                                   f"(len(os.sched_getaffinity(0)) = {cores})",
                         "single_core_value": round(v1, 4)},
        "e2e": {"value": round(value, 4), "unit": "Gbases/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0,
    }
    print(json.dumps(line), flush=True)


DUMP_MAX_BINS = 1 << 21


def dump_outputs(out_dir, hist, status):
    """hist.npy and status.npy as float64 (exact: counts stay far below 2^53); a histogram of more than DUMP_MAX_BINS
    bins as the same seeded sample of bins on every run, indices in hist_index.npy."""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    h = hist.cpu().numpy()
    if h.size > DUMP_MAX_BINS:
        idx = np.sort(np.random.default_rng(0).choice(h.size, DUMP_MAX_BINS, replace=False))
        np.save(os.path.join(out_dir, "hist_index.npy"), idx.astype(np.float64))
        h = h[idx]
    np.save(os.path.join(out_dir, "hist.npy"), h.astype(np.float64))
    np.save(os.path.join(out_dir, "status.npy"), status.cpu().numpy().astype(np.float64))


def timed(fn, reps, warm=2):
    """min / median of `reps` event-timed calls (ms)."""
    import torch
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    ts = []
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        torch.cuda.synchronize()
        ts.append(a.elapsed_time(b))
    return min(ts), statistics.median(ts)


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return

    import ctypes
    import numpy as np
    import torch
    import torch.distributed as dist
    from bionumpy_b200 import ops, _native as nv
    from bionumpy_b200.distributed import all_reduce_histogram

    assert torch.cuda.is_available(), "bench.py needs a CUDA device"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    assert world == args.gpus or world == 1, "launch with torchrun --nproc-per-node == --gpus"

    lib = nv.lib()
    n = args.reads
    first_record = rank * n                       # shard = disjoint record range (weak scaling)
    chunk = ops.synth_fastq(n, first_record=first_record, device=dev)
    n_bytes = chunk.numel()
    hist = torch.zeros(args.buckets, dtype=torch.int64, device=dev)
    status = nv.new_status(dev)
    per_read = READ_LEN - (args.window or args.k) + 1
    peak, peak_src = measured_peak_gbs()

    def step():
        ops.chunk_kmer_count(chunk, args.k, args.buckets, hist=hist, window_size=args.window, status=status)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    warm = max(args.warmup, 3)
    for _ in range(warm):
        step()
    if world > 1:
        all_reduce_histogram(hist.clone())        # NCCL communicator set-up outside the timed region
    barrier()
    # correctness guard on the measured configuration: every k-mer of every warm-up batch landed in exactly one bin
    st = ops.read_status(status)
    assert st.n_records == n and st.n_values == warm * n * per_read, st.words
    assert int(hist.sum().item()) == warm * n * per_read
    hist.zero_()
    nv.check(lib.bnpk_status_init(nv.ptr(status), nv.stream_ptr()))

    stop_evt, clock_lines = threading.Event(), []
    clk_thread = None
    if local_rank == 0:
        clk_thread = threading.Thread(target=sample_clocks, args=(stop_evt, clock_lines), daemon=True)
        clk_thread.start()
        time.sleep(0.3)

    lib.bnpk_profile_enable(1)
    launches0 = lib.bnpk_launch_count()
    barrier()
    ev0, ev1, ev2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    ev0.record()
    for _ in range(args.steps):
        step()
    ev1.record()
    all_reduce_histogram(hist)                    # the ONE collective: the final histogram
    ev2.record()
    barrier()
    elapsed_ms = ev0.elapsed_time(ev2)
    allreduce_ms = ev1.elapsed_time(ev2)
    launches = lib.bnpk_launch_count() - launches0
    tot_ms, n_l = ctypes.c_double(0), ctypes.c_uint64(0)
    lib.bnpk_profile_read(ctypes.byref(tot_ms), ctypes.byref(n_l))
    lib.bnpk_profile_enable(0)
    if local_rank == 0:
        time.sleep(0.2)
        stop_evt.set()
        clk_thread.join(timeout=3)
    kern_ms = tot_ms.value / max(n_l.value, 1)
    t = torch.tensor([elapsed_ms, allreduce_ms, kern_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    elapsed_ms, allreduce_ms, kern_ms_max = (float(x) for x in t.tolist())
    ms_per_step = elapsed_ms / args.steps
    value = world * n * READ_LEN / (ms_per_step * 1e-3) / 1e9
    assert int(hist.sum().item()) == world * args.steps * n * per_read
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, hist, status)
    # clocks of every GPU of the box (one sampler), gathered as text
    clocks_all = None
    if local_rank == 0:
        clocks_all = {str(g): summarize_clocks(clock_lines, g) for g in range(max(world, 1))}

    # roofline of the dominant kernel: algorithmic bytes per launch / event-timed duration of that launch
    alg_bytes = n_bytes + 16 * n + 8 * args.buckets       # SURVEY 8d: chunk once + row vector + histogram
    achieved = alg_bytes / (kern_ms * 1e-3) / 1e9
    roofline = {"bound": "hbm", "achieved": round(achieved, 1), "peak": peak, "unit": "GB/s",
                "frac": round(achieved / peak, 4), "traffic": traffic_from_profiles("tile_kernel_dram_bytes_per_10M_reads"),
                "kernel": KERNEL_NAME, "kernel_ms": round(kern_ms, 4), "kernel_ms_max_over_ranks": round(kern_ms_max, 4),
                "algorithmic_bytes_per_launch": alg_bytes, "peak_source": peak_src,
                "kernel_share_of_step": round(kern_ms / ms_per_step, 3)}

    line = {
        "metric": METRIC, "value": round(value, 3), "unit": "Gbases/s", "n_gpus": world, "steps": args.steps,
        "warmup": warm, "ms_per_step": round(ms_per_step, 4), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8->u32 codes, int64 counts", "data": "synthetic",
        "config": {"workload": f"synthetic {n}x150bp FASTQ per GPU and step ({n_bytes / 1e9:.2f} GB resident in HBM, > L2 so no "
                               f"flush between steps; splitmix64-keyed generator, bit-identical to oracle.synthetic_fastq), "
                               f"2-bit encode + k={args.k} rolling hash + bincount(hash mod {args.buckets})"
                               + (f", minimizer window {args.window}" if args.window else ""),
                   "reads_per_gpu_and_step": n, "k": args.k, "buckets": args.buckets, "window": args.window,
                   "parallelism": f"reads sharded over {world} GPU(s); {args.steps} batches accumulate per GPU, then ONE NCCL "
                                  f"all-reduce of the int64 histogram ({args.buckets * 8} bytes) inside the timed region"},
        "roofline": roofline, "gpu_launches": int(launches),
        "allreduce_ms": round(allreduce_ms, 4),
    }
    if clocks_all:
        line["clocks"] = clocks_all.get(str(local_rank)) or next((c for c in clocks_all.values() if c), None)
        if world > 1:
            line["clocks_per_gpu"] = clocks_all

    def roof(ms, alg):
        return {"ms": round(ms, 4), "achieved_GB/s": round(alg / (ms * 1e-3) / 1e9, 1), "frac": round(alg / (ms * 1e-3) / 1e9 / peak, 4)}

    if world == 1 and not args.no_extra:
        # ---- the headline table compared with the oracle, bin by bin (untimed) ----------------------------------
        try:
            from oracle import bnp_oracle as oracle
            so = os.path.join(ROOT, "oracle", "_build", "liboracle.so")
            co = ctypes.CDLL(so)
            co.oracle_fastq_kmer_hist.restype = ctypes.c_int64
            co.oracle_fastq_kmer_hist.argtypes = [ctypes.c_void_p, ctypes.c_size_t, ctypes.c_int, ctypes.c_char_p, ctypes.c_int,
                                                  ctypes.c_int, ctypes.c_uint64, ctypes.c_void_p, ctypes.c_void_p]
            host = chunk.cpu().numpy()
            want = np.zeros(args.buckets, dtype=np.int64)
            stats = np.zeros(3, dtype=np.int64)
            t0 = time.perf_counter()
            r = co.oracle_fastq_kmer_hist(host.ctypes.data, host.size, 4, b"ACGT", args.k, args.window, args.buckets,
                                          want.ctypes.data, stats.ctypes.data)
            dt = time.perf_counter() - t0
            h1 = torch.zeros(args.buckets, dtype=torch.int64, device=dev)
            ops.chunk_kmer_count(chunk, args.k, args.buckets, hist=h1, window_size=args.window)
            same = bool(np.array_equal(h1.cpu().numpy(), want))
            line["oracle_check"] = {"identical": same, "records": int(r), "bins": args.buckets,
                                    "oracle": "oracle/kmer_oracle.c, one thread, %.1f s = %.4f Gbases/s" % (dt, n * READ_LEN / dt / 1e9)}
            assert same and r == n, "headline histogram differs from the oracle"
            del host, h1
        except OSError as exc:  # pragma: no cover
            line["oracle_check"] = {"error": repr(exc)}

        # ---- second headline: 2^24 buckets ---------------------------------------------------------------------------
        b24 = 1 << 24
        h24 = torch.zeros(b24, dtype=torch.int64, device=dev)
        lib.bnpk_profile_enable(1)
        mn, med = timed(lambda: ops.chunk_kmer_count(chunk, args.k, b24, hist=h24, status=status), args.reps)
        lib.bnpk_profile_read(ctypes.byref(tot_ms), ctypes.byref(n_l))
        lib.bnpk_profile_enable(0)
        k24 = tot_ms.value / max(n_l.value, 1)
        alg24 = n_bytes + 16 * n + 8 * b24
        line["headline_2^24"] = {"buckets": b24, "ms_per_step_min": round(mn, 4), "ms_per_step_median": round(med, 4),
                                 "value": round(n * READ_LEN / med / 1e6, 2), "unit": "Gbases/s",
                                 "roofline": {"bound": "hbm (the kernel itself is bound by L2 atomics: 1.2 G RED per step)",
                                              "kernel_ms": round(k24, 4), "achieved": round(alg24 / (k24 * 1e-3) / 1e9, 1),
                                              "peak": peak, "unit": "GB/s", "frac": round(alg24 / (k24 * 1e-3) / 1e9 / peak, 4)}}
        del h24

        extra = {}
        # ---- k = 5 exact (4^5 bins: what the reference itself can histogram, BASELINE configs[0]'s operation) --------
        h5 = torch.zeros(4 ** 5, dtype=torch.int64, device=dev)
        mn, med = timed(lambda: ops.chunk_kmer_count(chunk, 5, 4 ** 5, hist=h5, status=status), args.reps)
        extra["k5_exact_4^5_bins"] = {"min_ms": round(mn, 4), "median_ms": round(med, 4), "Gbases/s": round(n * READ_LEN / med / 1e6, 2),
                                      "frac_of_hbm_roofline": roof(med, n_bytes + 16 * n + 8 * 4 ** 5)["frac"]}
        # ---- minimizers on the headline batch ----------------------------------------------------------------------------
        hm = torch.zeros(1 << 14, dtype=torch.int64, device=dev)
        mn, med = timed(lambda: ops.chunk_kmer_count(chunk, args.k, 1 << 14, hist=hm, window_size=41, status=status), args.reps)
        extra["minimizers_w41_buckets_2^14_10M_reads"] = {"min_ms": round(mn, 4), "median_ms": round(med, 4),
                                                          "Gbases/s": round(n * READ_LEN / med / 1e6, 2),
                                                          "frac_of_hbm_roofline": roof(med, n_bytes + 16 * n + 8 * (1 << 14))["frac"]}
        del h5, hm
        # ---- materialising mode: get_kmers(k=31) writes 8 bytes per k-mer (SURVEY 8d: 8.62 B/base) ------------------
        try:
            starts, lens, _ = ops.line_split(chunk, 4, 1, 0, ord("@"), True, -1, max_rows=n)
            offsets = ops.row_offsets(lens, args.k - 1)
            total = int(offsets[-1].item())
            out = torch.empty(total, dtype=torch.int64, device=dev)

            def materialise():
                nv.check(lib.bnpk_rows_kmer_hash(nv.ptr(chunk), n_bytes, nv.ptr(starts), nv.ptr(lens), n, nv.ENC_ASCII_ACGT, None,
                                                 args.k, nv.ptr(offsets), nv.ptr(out), nv.ptr(status), nv.stream_ptr()))
            mn, med = timed(materialise, args.reps)
            algm = n_bytes + 16 * n + 8 * total
            extra["materialised_get_kmers_k31"] = {"min_ms": round(mn, 4), "median_ms": round(med, 4), "kmers": total,
                                                    "Gbases/s": round(n * READ_LEN / med / 1e6, 2),
                                                    "algorithmic_bytes": algm, "frac_of_hbm_roofline": roof(med, algm)["frac"],
                                                    "note": "bnpk_rows_kmer_hash over the row-offset vector of bnpk_line_split "
                                                            "(line_split itself: %.3f ms)" % timed(lambda: ops.line_split(chunk, 4, 1, 0, ord("@"), True, -1, max_rows=n), 3)[1]}
            del starts, lens, offsets, out
        except Exception as exc:  # pragma: no cover
            extra["materialised_get_kmers_k31"] = {"error": repr(exc)}
        # ---- BASELINE configs[3]: every sacCer3 chromosome (50 kbases each), k=21 (long ragged rows) -------------------
        try:
            extra["config4_sacCer3_k21"] = bench_saccer3(dev, peak)
        except Exception as exc:  # pragma: no cover
            extra["config4_sacCer3_k21"] = {"error": repr(exc)}
        line["extra"] = extra

    # ---- end to end through the host-buffer C-ABI call -----------------------------------------------
    e2e = None
    try:
        host = torch.empty(n_bytes, dtype=torch.uint8).pin_memory()
        host.copy_(chunk)
        torch.cuda.synchronize()
        pipe = ops.HostPipeline(n_bytes, slice_bytes=32 << 20)
        res_host = torch.empty(args.buckets, dtype=torch.int64).pin_memory()

        def e2e_step():
            hist.zero_()
            pipe.kmer_count(host, args.k, hist, window_size=args.window)     # H2D slices overlapped with the count
            res_host.copy_(hist)                                             # the step's result back on the host
            torch.cuda.synchronize()

        e2e_step()
        barrier()
        dts = []
        for _ in range(args.e2e_steps):
            t0 = time.perf_counter()
            e2e_step()
            dts.append(time.perf_counter() - t0)
        barrier()
        dt = sum(dts) / len(dts)
        t = torch.tensor([dt], device=dev, dtype=torch.float64)
        if world > 1:
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt = float(t.item())
        assert int(res_host.sum().item()) == n * per_read
        e2e = {"value": round(world * n * READ_LEN / dt / 1e9, 3), "unit": "Gbases/s",
               "h2d_bytes_per_step": n_bytes, "d2h_bytes_per_step": args.buckets * 8 + 128,
               "ms_per_step": round(dt * 1e3, 3), "ms_min": round(min(dts) * 1e3, 3), "ms_median": round(statistics.median(dts) * 1e3, 3),
               "steps": args.e2e_steps, "h2d_GB/s": round(n_bytes / dt / 1e9, 2),
               "api": "bnpk_pipeline_kmer_count_host_on (pinned host chunk -> sliced H2D || fused count -> D2H histogram); "
                      "per GPU, no collective"}
        pipe.close()
        # ---- the same through the kept reader API on a real file ---------------------------------------------------------
        if world == 1 and not args.no_extra:
            try:
                line["e2e_api"] = bench_api(host, n, args, dev)
            except Exception as exc:  # pragma: no cover
                line["e2e_api"] = {"error": repr(exc)}
        del host
    except Exception as exc:  # pragma: no cover
        e2e = {"error": repr(exc)}
    line["e2e"] = e2e

    # ---- BASELINE configs[2]: 100 M reads, k=31 minimizers (11 k-mers per window = window_size 41) -------------------
    if world == 1 and not args.no_extra and args.config3_reads > 0:
        try:
            del chunk
            torch.cuda.empty_cache()
            n3 = args.config3_reads
            big = ops.synth_fastq(n3, device=dev)
            res = {}
            for b in (1 << 14, 1 << 24):
                hb = torch.zeros(b, dtype=torch.int64, device=dev)
                mn, med = timed(lambda: ops.chunk_kmer_count(big, args.k, b, hist=hb, window_size=41, status=status), 3, warm=1)
                assert int(hb.sum().item()) == 4 * n3 * (READ_LEN - 41 + 1)
                res[f"buckets_2^{b.bit_length() - 1}"] = {"min_ms": round(mn, 3), "median_ms": round(med, 3),
                                                          "Gbases/s": round(n3 * READ_LEN / med / 1e6, 2),
                                                          "frac_of_hbm_roofline": roof(med, big.numel() + 16 * n3 + 8 * b)["frac"]}
                del hb
            res["reads"] = n3
            res["resident_GB"] = round(big.numel() / 1e9, 2)
            line.setdefault("extra", {})["config3_minimizers_w41"] = res
            del big
        except Exception as exc:  # pragma: no cover
            line.setdefault("extra", {})["config3_minimizers_w41"] = {"error": repr(exc)}

    # ---- CPU baseline: the reference path's NumPy port on this box's host cores (rank 0, N = 1) -------
    if rank == 0 and world == 1:
        cores = host_cores()
        v1, bases1, wall1 = cpu_baseline(args.k, args.buckets, args.window, 120_000, 1)
        n_sample = 15_000 * cores * 4                         # four ~4.8 MB chunks per core
        vN, basesN, wallN = cpu_baseline(args.k, args.buckets, args.window, n_sample, cores)
        line["cpu_baseline"] = {"value": round(v1, 4), "unit": "Gbases/s", "cores": 1, "kind": "port",
                                "sample": f"120000 synthetic reads in ~4.8 MB chunks on ONE core ({wall1:.1f} s): the reference is "
                                          f"single-threaded (its own benchmark runs --cores 1)",
                                "all_cores_value": round(vN, 4), "all_cores": cores,
                                "all_cores_sample": f"{n_sample} reads = {basesN / 1e9:.2f} Gbases, one process per core "
                                                    f"(len(os.sched_getaffinity(0)) = {cores}), {wallN:.1f} s wall"}
    if rank == 0:
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


def bench_saccer3(dev, peak):
    """BASELINE configs[3] in miniature: tests/golden/sacCer3_sample.fa.gz (the first 50 kbases of every chromosome of
    the reference's example_data/sacCer3.fa) through the kept API: bnp.open(...).read_chunks() ->
    count_kmers_hashed(k=21, 2^24 buckets); plus the device-only time of the count."""
    import gzip
    import tempfile
    import numpy as np
    import torch
    import bionumpy_b200 as bnp
    src = os.path.join(ROOT, "tests", "golden", "sacCer3_sample.fa.gz")
    raw = gzip.open(src).read()
    tmp = tempfile.NamedTemporaryFile(suffix=".fa", delete=False)
    tmp.write(raw)
    tmp.close()
    B = 1 << 24
    try:
        def run():
            hist = torch.zeros(B, dtype=torch.int64, device=dev)
            n_bases = 0
            for chunk in bnp.open(tmp.name).read_chunks(min_chunk_size=1 << 24):
                hist += bnp.count_kmers_hashed(chunk.sequence, 21, B)
                n_bases += int(chunk.sequence.lengths.sum().item()) if hasattr(chunk.sequence, "lengths") else 0
            torch.cuda.synchronize()
            return hist, n_bases
        hist, n_bases = run()
        ts = []
        for _ in range(5):
            t0 = time.perf_counter()
            run()
            ts.append(time.perf_counter() - t0)
        # device-only: the whole genome as one resident buffer
        whole = (raw if raw.endswith(b"\n") else raw + b"\n") + b">"          # what the reader hands over for the last chunk
        buf = bnp.MultiLineFastaBuffer.from_raw_buffer(np.frombuffer(whole, dtype=np.uint8))
        seq = buf.get_data().sequence
        mn, med = timed(lambda: bnp.count_kmers_hashed(seq, 21, B), 10)
        n_kmers = int(hist.sum().item())
        return {"file_bytes": len(raw), "bases": n_bases, "kmers": n_kmers, "distinct_buckets": int((hist > 0).sum().item()),
                "api_ms_median": round(statistics.median(ts) * 1e3, 2), "api_Gbases/s": round(n_bases / statistics.median(ts) / 1e9, 3),
                "count_only_ms_median": round(med, 3), "count_only_Gbases/s": round(n_bases / med / 1e6, 2),
                "count_only_frac_of_hbm_roofline": round((n_bases + 8 * B) / (med * 1e-3) / 1e9 / peak, 4),
                "note": "17 rows of 50 kbases; bit-exact check incl. np.unique in "
                        "tests/test_gpu_round2.py::test_saccer3_whole_genome_k21"}
    finally:
        os.unlink(tmp.name)


def bench_api(host_chunk, n_reads, args, dev):
    """for chunk in bnp.open(path).read_chunks(min_chunk_size): hist += count_kmers_hashed(chunk.sequence, k, B) on a
    real FASTQ file (a prefix of the synthetic batch written to local disk; it stays in the page cache)."""
    import tempfile
    import numpy as np
    import torch
    import bionumpy_b200 as bnp
    n_file = min(n_reads, 4_000_000)
    tmp = tempfile.NamedTemporaryFile(suffix=".fq", delete=False)
    tmp.write(host_chunk[: n_file * RECORD_BYTES].numpy().tobytes())
    tmp.close()
    out = {"file_reads": n_file, "file_bytes": n_file * RECORD_BYTES}
    try:
        for label, mcs in (("min_chunk_size_5MB", 5_000_000), ("min_chunk_size_256MB", 256 << 20)):
            def run():
                hist = torch.zeros(args.buckets, dtype=torch.int64, device=dev)
                with bnp.open(tmp.name) as f:
                    for chunk in f.read_chunks(min_chunk_size=mcs):
                        hist += bnp.count_kmers_hashed(chunk.sequence, args.k, args.buckets)
                res = hist.cpu()
                return res
            res = run()
            assert int(res.sum().item()) == n_file * (READ_LEN - args.k + 1)
            ts = []
            for _ in range(5):
                t0 = time.perf_counter()
                run()
                ts.append(time.perf_counter() - t0)
            med = statistics.median(ts)
            out[label] = {"ms_median": round(med * 1e3, 2), "ms_min": round(min(ts) * 1e3, 2),
                          "Gbases/s": round(n_file * READ_LEN / med / 1e9, 3), "file_GB/s": round(n_file * RECORD_BYTES / med / 1e9, 2)}
        return out
    finally:
        os.unlink(tmp.name)


if __name__ == "__main__":
    main()
