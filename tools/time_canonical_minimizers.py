"""Canonical minimizer counts on the bench workload (10 M synthetic 150 bp reads, 3.17 GB): the fused chunk count
(bnpk_chunk_minimizer_count_canonical: the wsmc build for CTA-private tables and windows of up to 12 k-mers, the
register-staged kernel otherwise) against the row route (line_split + rows_minimizer_count_canonical), with the plain
fused minimizer count at the same arguments as the reference point.  One process, CUDA-event timed, best of --reps
launches after --warmup launches of every case.  Check: for every case the fused and the row-route tables are
identical and hold (151 - w) values per read; the script exits non-zero otherwise.

    python tools/time_canonical_minimizers.py [--reads N] [--reps R] [--warmup W] [--json PATH]
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

from bionumpy_b200 import _native as nv, ops  # noqa: E402

CASES = [(31, 41, 1 << 14), (31, 41, 1 << 24), (15, 25, 1 << 14)]     # (k, window_size, bins)


def timed(fn, reps, warmup):
    for _ in range(warmup):
        fn()
    torch.cuda.synchronize()
    best = float("inf")
    for _ in range(reps):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        fn()
        b.record()
        b.synchronize()
        best = min(best, a.elapsed_time(b))
    return best


def gpu_settings():
    """Power limit, current and maximum SM clock of this device (read-only query)."""
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit,clocks.sm,clocks.max.sm", "--format=csv,noheader",
                              "-i", str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout
        return out.strip() or "unknown"
    except (OSError, subprocess.SubprocessError):
        return "unknown"


def main():
    p = argparse.ArgumentParser()
    p.add_argument("--reads", type=int, default=10_000_000)
    p.add_argument("--reps", type=int, default=5)
    p.add_argument("--warmup", type=int, default=2)
    p.add_argument("--json", default=None)
    args = p.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("time_canonical_minimizers.py needs a CUDA device")
    n = args.reads
    chunk = ops.synth_fastq(n)
    N = chunk.numel()
    dev = chunk.device
    status = nv.new_status(dev)
    n_bases = 150 * n
    settings = gpu_settings()
    print(f"device: {torch.cuda.get_device_name(dev)}, power limit / SM clock / max SM clock: {settings}; "
          f"{n} reads x 150 bp = {N / 1e9:.2f} GB")
    rows = []

    def report(name, k, w, bins, ms):
        r = {"case": name, "k": k, "window_size": w, "bins": bins, "ms": round(ms, 4),
             "gbases_s": round(n_bases / ms / 1e6, 1)}
        rows.append(r)
        print(f"{name:<38} k={k:<2} w={w:<2} bins=2^{bins.bit_length() - 1:<2} {ms:8.3f} ms  {r['gbases_s']:7.1f} Gbases/s")

    ok = True
    for k, w, bins in CASES:
        hist = torch.zeros(bins, dtype=torch.int64, device=dev)
        plain = lambda: ops.chunk_kmer_count(chunk, k, bins, hist=hist, window_size=w, status=status)  # noqa: E731
        fused = lambda: ops.chunk_minimizer_count_canonical(chunk, k, w, 3, bins, hist=hist, status=status)  # noqa: E731

        def rows_route():
            starts, lens, _ = ops.line_split(chunk, max_rows=n)
            ops.rows_minimizer_count_canonical(chunk, starts, lens, nv.ENC_ASCII_ACGT, k, w, 3, bins, hist=hist,
                                               status=status)
        t_plain = timed(plain, args.reps, args.warmup)
        t_fused = timed(fused, args.reps, args.warmup)
        t_rows = timed(rows_route, args.reps, args.warmup)
        report("plain minimizers fused", k, w, bins, t_plain)
        report("canonical minimizers fused", k, w, bins, t_fused)
        report("canonical minimizers line_split + rows", k, w, bins, t_rows)
        # check: one fresh table from each route
        a, _ = ops.chunk_minimizer_count_canonical(chunk, k, w, 3, bins)
        starts, lens, _ = ops.line_split(chunk, max_rows=n)
        b, _ = ops.rows_minimizer_count_canonical(chunk, starts, lens, nv.ENC_ASCII_ACGT, k, w, 3, bins)
        same = bool(torch.equal(a, b)) and int(a.sum().item()) == (151 - w) * n
        ok &= same
        print(f"  tables identical: {same}; canonical/plain fused = {t_fused / t_plain:.3f}, "
              f"fused/rows = {t_fused / t_rows:.3f}")
    summary = {"device": torch.cuda.get_device_name(dev), "power_limit_sm_clock_max_sm_clock": settings, "reads": n,
               "chunk_bytes": N, "reps": args.reps, "warmup": args.warmup, "rows": rows, "tables_identical": ok}
    print(json.dumps(summary))
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            json.dump(summary, f, indent=1)
    if not ok:
        raise SystemExit("canonical minimizer fused and row-route tables differ")


if __name__ == "__main__":
    main()
