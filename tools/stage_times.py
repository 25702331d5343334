"""Development: per-stage latencies of the warp-specialised count (needs BNPK_WS_DEBUG with bit 16 set)."""
import sys, os
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import torch
from bionumpy_b200 import ops, _native as nv
n = 10_000_000
chunk = ops.synth_fastq(n); N = chunk.numel()
status = nv.new_status(chunk.device); ws = nv.workspace(N, chunk.device)
hist = torch.zeros(1 << 14, dtype=torch.int64, device="cuda")
for _ in range(2):
    ops.chunk_kmer_count(chunk, 31, 1 << 14, hist=hist, status=status)
torch.cuda.synchronize()
a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
a.record(); ops.chunk_kmer_count(chunk, 31, 1 << 14, hist=hist, status=status); b.record(); torch.cuda.synchronize()
w = ws.view(torch.int64)[:16].cpu().tolist()
tiles, chunks = max(w[10], 1), max(w[11], 1)
f = 1.0 / 1.965e3   # cycles -> us at 1965 MHz
print("ms %.3f | per tile (us): copy %.2f  scan %.2f  phase check + push %.2f | per chunk: queue wait %.2f  chunk %.2f | P waits for a free slot %.2f us per tile | tiles %d chunks %d" % (
    a.elapsed_time(b), w[4] / tiles * f, w[5] / tiles * f, w[6] / tiles * f, w[7] / chunks * f, w[8] / chunks * f, w[9] / tiles * f, tiles, chunks))
