"""Canonical k-mer counts on the bench workload (10 M synthetic 150 bp reads, 3.17 GB): the fused chunk count
(bnpk_chunk_kmer_count_canonical) against the row route it replaces (line_split + rows_kmer_count_canonical), with the
plain fused count as the reference point.  One process, CUDA-event timed, best of --reps launches after --warmup
launches of every case.  Oracle check: for every case the fused and the row-route tables are identical.

    python tools/time_canonical.py [--reads N] [--reps R] [--warmup W] [--json PATH]
"""
import argparse
import json
import os
import subprocess
import sys

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

import torch  # noqa: E402

from bionumpy_b200 import _native as nv, ops  # noqa: E402

PEAK_GBS = 6575.8          # measured device-to-device copy bandwidth of the B200 (DESIGN.md §3)
CASES = [(31, 1 << 14), (31, 1 << 24), (15, 1 << 14)]


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


def power_limit():
    try:
        out = subprocess.run(["nvidia-smi", "--query-gpu=power.limit", "--format=csv,noheader", "-i",
                              str(torch.cuda.current_device())], capture_output=True, text=True, timeout=30).stdout
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
        raise SystemExit("time_canonical.py needs a CUDA device")
    n = args.reads
    chunk = ops.synth_fastq(n)
    N = chunk.numel()
    dev = chunk.device
    status = nv.new_status(dev)
    n_bases = 150 * n
    print(f"device: {torch.cuda.get_device_name(dev)}, power limit {power_limit()}; {n} reads x 150 bp = {N / 1e9:.2f} GB")
    rows = []

    def report(name, k, bins, ms):
        alg = N + 16 * n + 8 * bins                                    # algorithmic bytes (SURVEY §8d)
        r = {"case": name, "k": k, "bins": bins, "ms": round(ms, 4), "gbases_s": round(n_bases / ms / 1e6, 1),
             "alg_GBs": round(alg / ms / 1e6, 1), "of_peak": round(alg / ms / 1e6 / PEAK_GBS, 4)}
        rows.append(r)
        print(f"{name:<34} k={k:<2} bins=2^{bins.bit_length() - 1:<2} {ms:8.3f} ms  {r['gbases_s']:7.1f} Gbases/s  "
              f"{r['alg_GBs']:7.1f} GB/s alg = {r['of_peak']:.4f} of {PEAK_GBS} GB/s")

    hist = torch.zeros(1 << 14, dtype=torch.int64, device=dev)
    report("plain fused", 31, 1 << 14,
           timed(lambda: ops.chunk_kmer_count(chunk, 31, 1 << 14, hist=hist, status=status), args.reps, args.warmup))
    ok = True
    for k, bins in CASES:
        hist = torch.zeros(bins, dtype=torch.int64, device=dev)
        fused = lambda: ops.chunk_kmer_count_canonical(chunk, k, 3, bins, hist=hist, status=status)  # noqa: E731

        def rows_route():
            starts, lens, _ = ops.line_split(chunk, max_rows=n)
            ops.rows_kmer_count_canonical(chunk, starts, lens, nv.ENC_ASCII_ACGT, k, 3, bins, hist=hist, status=status)
        t_fused = timed(fused, args.reps, args.warmup)
        t_rows = timed(rows_route, args.reps, args.warmup)
        report("canonical fused", k, bins, t_fused)
        report("canonical line_split + rows", k, bins, t_rows)
        # oracle check: one fresh table from each route
        a, st = ops.chunk_kmer_count_canonical(chunk, k, 3, bins)
        starts, lens, _ = ops.line_split(chunk, max_rows=n)
        b, _ = ops.rows_kmer_count_canonical(chunk, starts, lens, nv.ENC_ASCII_ACGT, k, 3, bins)
        same = bool(torch.equal(a, b)) and int(a.sum().item()) == (151 - k) * n
        ok &= same
        print(f"  tables identical: {same}; fused/rows time = {t_fused / t_rows:.3f}")
    summary = {"device": torch.cuda.get_device_name(dev), "power_limit": power_limit(), "reads": n, "chunk_bytes": N,
               "reps": args.reps, "warmup": args.warmup, "rows": rows, "tables_identical": ok}
    print(json.dumps(summary))
    if args.json:
        os.makedirs(os.path.dirname(os.path.abspath(args.json)), exist_ok=True)
        with open(args.json, "w") as f:
            json.dump(summary, f, indent=1)
    if not ok:
        raise SystemExit("canonical fused and row-route tables differ")


if __name__ == "__main__":
    main()
