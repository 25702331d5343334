// misc_kernels.cu -- byte census, ragged offsets (single-pass scan), standalone bincount,
// synthetic FASTQ generator, and the small C-ABI entry points.
#include <mutex>
#include <utility>
#include <vector>
#include "bnpk_host.h"

namespace bnpk {

std::atomic<uint64_t> g_launches{0};
static thread_local char g_err[512] = "";

int set_err(int code, const char *msg) {
    snprintf(g_err, sizeof(g_err), "%s", msg);
    return code;
}
int cuda_fail(cudaError_t e, const char *what) {
    snprintf(g_err, sizeof(g_err), "CUDA error %d (%s) in %s", (int)e, cudaGetErrorString(e), what);
    cudaGetLastError();
    return (int)e;
}
// ---- optional timing of the tile kernel (CUDA events on the launching stream) ----------------
static std::mutex g_prof_mu;
static bool g_prof_on = false;
static std::vector<std::pair<cudaEvent_t, cudaEvent_t>> g_prof_events;
static std::vector<cudaEvent_t> g_prof_pool;
static cudaEvent_t prof_event() {
    if (!g_prof_pool.empty()) { cudaEvent_t e = g_prof_pool.back(); g_prof_pool.pop_back(); return e; }
    cudaEvent_t e;
    cudaEventCreate(&e);
    return e;
}
void profile_before(cudaStream_t st) {
    std::lock_guard<std::mutex> l(g_prof_mu);
    if (!g_prof_on) return;
    cudaEvent_t a = prof_event(), b = prof_event();
    cudaEventRecord(a, st);
    g_prof_events.emplace_back(a, b);
}
void profile_after(cudaStream_t st) {
    std::lock_guard<std::mutex> l(g_prof_mu);
    if (!g_prof_on || g_prof_events.empty()) return;
    cudaEventRecord(g_prof_events.back().second, st);
}

int ensure_dyn_smem(const void *kernel, int bytes) {
    static std::mutex mu;
    static std::vector<std::pair<const void *, int>> done;                // (kernel, device) pairs already raised
    int dev = 0;
    BNPK_CUDA(cudaGetDevice(&dev));
    std::lock_guard<std::mutex> l(mu);
    for (const auto &e : done)
        if (e.first == kernel && e.second == dev) return 0;
    BNPK_CUDA(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes));
    done.emplace_back(kernel, dev);
    return 0;
}

int sm_count() {
    static thread_local int cached_dev = -1, cached = 0;
    int dev = 0;
    if (cudaGetDevice(&dev) != cudaSuccess) return 148;
    if (dev != cached_dev) {
        cudaDeviceGetAttribute(&cached, cudaDevAttrMultiProcessorCount, dev);
        cached_dev = dev;
    }
    return cached > 0 ? cached : 148;
}

// ------------------------------------------------------------------------------------------
__global__ void status_init_kernel(int64_t *status) {
    const int i = threadIdx.x;
    if (i < BNPK_ST_WORDS) {
        int64_t v = 0;
        if (i == BNPK_ST_BAD_HEADER_ENTRY || i == BNPK_ST_BAD_PLUS_ENTRY || i == BNPK_ST_BAD_BASE) v = INT64_MAX;
        status[i] = v;
    }
}

// ------------------------------------------------------------------------------------------
// K0: how many bytes equal `value`
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) count_byte_kernel(const uint8_t *chunk, size_t n, uint32_t pattern,
                                                         unsigned long long *out) {
    const size_t n_units = n / 16;
    const bool aligned = (reinterpret_cast<uintptr_t>(chunk) & 15) == 0;
    unsigned long long c = 0;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t u = (size_t)blockIdx.x * blockDim.x + threadIdx.x; u < n_units; u += stride) {
        const uint4 q = aligned ? ld_stream(reinterpret_cast<const uint4 *>(chunk) + u)
                                : load_unit_guarded(chunk, n, (int64_t)u * 16);
        c += __popc(__vcmpeq4(q.x, pattern) & 0x01010101u) + __popc(__vcmpeq4(q.y, pattern) & 0x01010101u) +
             __popc(__vcmpeq4(q.z, pattern) & 0x01010101u) + __popc(__vcmpeq4(q.w, pattern) & 0x01010101u);
    }
    if (blockIdx.x == 0 && threadIdx.x == 0)
        for (size_t p = n_units * 16; p < n; ++p) c += (chunk[p] == (uint8_t)pattern);
    c = warp_sum_u64(c);
    if ((threadIdx.x & 31) == 0 && c) atomicAdd(out, c);
}

// ------------------------------------------------------------------------------------------
// ragged offsets: exclusive prefix sum of max(len - shrink, 0), single pass (look-back)
// ------------------------------------------------------------------------------------------
constexpr int kScanThreads = 256;
constexpr int kScanItems = 8;
constexpr int kScanTile = kScanThreads * kScanItems;

__global__ void __launch_bounds__(kScanThreads) row_offsets_kernel(const int32_t *lens, size_t n, int shrink,
                                                                   int64_t *offsets, uint64_t *ws) {
    __shared__ uint64_t s_warp[kScanThreads / 32 + 1];
    __shared__ int64_t s_tile;
    __shared__ uint64_t s_base;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    uint64_t *state = ws + kWsHeaderWords;
    const int64_t n_tiles = (int64_t)((n + kScanTile - 1) / kScanTile);
    while (true) {
        if (tid == 0) s_tile = (int64_t)atomicAdd((unsigned long long *)(ws + kWsTicket), 1ull);
        __syncthreads();
        const int64_t tile = s_tile;
        if (tile >= n_tiles) break;
        const size_t r0 = (size_t)tile * kScanTile + (size_t)tid * kScanItems;
        uint64_t v[kScanItems];
        uint64_t sum = 0;
#pragma unroll
        for (int i = 0; i < kScanItems; ++i) {
            int64_t l = 0;
            if (r0 + i < n) l = (int64_t)lens[r0 + i] - shrink;
            v[i] = l > 0 ? (uint64_t)l : 0;
            sum += v[i];
        }
        uint64_t inc = sum;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint64_t t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += t;
        }
        if (lane == 31) s_warp[warp] = inc;
        __syncthreads();
        if (warp == 0) {
            uint64_t w = lane < kScanThreads / 32 ? s_warp[lane] : 0;
            uint64_t winc = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint64_t t = __shfl_up_sync(0xffffffffu, winc, o);
                if (lane >= o) winc += t;
            }
            const uint64_t total = __shfl_sync(0xffffffffu, winc, kScanThreads / 32 - 1);
            if (lane < kScanThreads / 32) s_warp[lane] = winc - w;
            const uint64_t excl = lookback_exclusive(state, tile, total, lane);
            if (lane == 0) {
                s_base = excl;
                if (tile == n_tiles - 1) offsets[n] = (int64_t)(excl + total);
            }
        }
        __syncthreads();
        uint64_t run = s_base + s_warp[warp] + inc - sum;
#pragma unroll
        for (int i = 0; i < kScanItems; ++i) {
            if (r0 + i < n) offsets[r0 + i] = (int64_t)run;
            run += v[i];
        }
        __syncthreads();
    }
}

// ------------------------------------------------------------------------------------------
// K5: standalone bincount
// ------------------------------------------------------------------------------------------
template <bool SMEM_HIST>
__global__ void __launch_bounds__(512) bincount_kernel(const int64_t *values, size_t n, uint64_t n_bins,
                                                       unsigned long long *hist, int64_t *status) {
    extern __shared__ uint32_t s_hist[];
    if (SMEM_HIST) {
        for (uint32_t b = threadIdx.x; b < n_bins; b += blockDim.x) s_hist[b] = 0;
        __syncthreads();
    }
    const uint64_t mask = (n_bins & (n_bins - 1)) == 0 ? n_bins - 1 : 0;
    const size_t stride = (size_t)gridDim.x * blockDim.x;
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += stride) {
        const int64_t v = values[i];
        if (v < 0) {
            atomicMin((long long *)&status[BNPK_ST_BAD_BASE], (long long)i);
            continue;
        }
        const uint64_t b = mask ? ((uint64_t)v & mask) : ((uint64_t)v % n_bins);
        if (SMEM_HIST) atomicAdd(s_hist + (uint32_t)b, 1u);
        else atomicAdd(hist + b, 1ull);
    }
    if (SMEM_HIST) {
        __syncthreads();
        for (uint32_t b = threadIdx.x; b < n_bins; b += blockDim.x) {
            const uint32_t c = s_hist[b];
            if (c) atomicAdd(hist + b, (unsigned long long)c);
        }
    }
}

// K5': per-row bincount (count_encoded(axis=-1)); one warp per row
__global__ void __launch_bounds__(256) bincount_rows_kernel(const int64_t *values, const int64_t *offsets, size_t n_rows,
                                                            uint64_t n_bins, unsigned long long *out, int64_t *status) {
    const int lane = threadIdx.x & 31;
    const size_t warp_global = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const size_t n_warps = ((size_t)gridDim.x * blockDim.x) >> 5;
    for (size_t r = warp_global; r < n_rows; r += n_warps) {
        const int64_t b = offsets[r], e = offsets[r + 1];
        for (int64_t i = b + lane; i < e; i += 32) {
            const int64_t v = values[i];
            if (v < 0) { atomicMin((long long *)&status[BNPK_ST_BAD_BASE], (long long)i); continue; }
            atomicAdd(out + r * n_bins + ((uint64_t)v % n_bins), 1ull);
        }
    }
}


// ------------------------------------------------------------------------------------------
// Multi-line FASTA bookkeeping (io/multiline_buffer.py:46-62,89-106) over the per-line (start, len) arrays of K1:
//   flags    : is the line a header ('>'), does an entry start right after its newline, '\r' trimming;
//              out[0] = max index of a line that is followed by an entry start + 1 (0: none), out[1] = 1 if one of the
//              first ten lines ends in '\r'
//   entries  : with hdr_before = exclusive scan of the header flags (bnpk_row_offsets): header fields, the compacted
//              sequence-line list and the per-entry sequence lengths
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) multiline_flags_kernel(const uint8_t *chunk, size_t n, const int64_t *starts, const int32_t *lens,
                                                              size_t n_lines, int32_t *is_header, int64_t *out) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_lines; i += (size_t)gridDim.x * blockDim.x) {
        const int64_t s = starts[i], e = s + lens[i];                 // e = position of the line's '\n'
        is_header[i] = (i == 0 || chunk[s] == '>') ? 1 : 0;
        const size_t nxt = (size_t)min((long long)(e + 1), (long long)n - 1);
        if (chunk[nxt] == '>') atomicMax((unsigned long long *)&out[0], (unsigned long long)i + 1ull);
        if (i < 10 && e > 0 && chunk[e - 1] == 13) out[1] = 1;
    }
}
__global__ void __launch_bounds__(256) multiline_entries_kernel(const uint8_t *chunk, const int64_t *starts, const int32_t *lens,
                                                                const int32_t *is_header, const int64_t *hdr_before, size_t keep,
                                                                int trim_cr, int64_t *h_starts, int32_t *h_lens, int64_t *s_starts,
                                                                int32_t *s_lens, unsigned long long *entry_lens) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < keep; i += (size_t)gridDim.x * blockDim.x) {
        const int64_t s = starts[i];
        int32_t L = lens[i];
        if (trim_cr && L > 0 && chunk[s + L - 1] == 13) L -= 1;       // _modify_ends_for_carriage_returns (:103-106)
        const int64_t e = hdr_before[i] + is_header[i] - 1;           // entry of this line
        if (is_header[i]) {
            h_starts[e] = s + 1;
            h_lens[e] = max(L - 1, 0);
        } else {
            const int64_t pos = (int64_t)i - (e + 1);                 // sequence lines before this one
            s_starts[pos] = s;
            s_lens[pos] = L;
            atomicAdd(entry_lens + e, (unsigned long long)L);
        }
    }
}

// ------------------------------------------------------------------------------------------
// Indexed FASTA (io/indexed_fasta.py:101-206): sequence positions -> file bytes, skipping the line ends.
// Row r = bases [row_start[r], row_start[r] + row_len[r]) of the contig whose first base is file byte
// contig_offset[r], written with lenc[r] bases per line of lenb[r] bytes.  One warp per row, coalesced writes.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) fasta_gather_kernel(const uint8_t *file, size_t file_bytes, size_t n_rows,
                                                           const int64_t *contig_offset, const int64_t *row_start,
                                                           const int64_t *row_len, const int32_t *lenc, const int32_t *lenb,
                                                           const int64_t *out_offsets, uint8_t *out, int64_t *status) {
    const int lane = threadIdx.x & 31;
    const size_t warp_global = ((size_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const size_t n_warps = ((size_t)gridDim.x * blockDim.x) >> 5;
    for (size_t r = warp_global; r < n_rows; r += n_warps) {
        const int64_t base = contig_offset[r], s = row_start[r], L = row_len[r], o = out_offsets[r];
        const int64_t c = lenc[r], b = lenb[r];
        for (int64_t i = lane; i < L; i += 32) {
            const int64_t p = s + i;
            const int64_t byte = base + (p / c) * b + p % c;
            uint8_t v = 0;
            if (byte >= 0 && (size_t)byte < file_bytes) v = file[byte];
            else atomicMin((long long *)&status[BNPK_ST_BAD_BASE], (long long)(((int64_t)r << 32) | i));
            out[o + i] = v;
        }
    }
}

// ------------------------------------------------------------------------------------------
// Bloom filter over k-mer hashes (sequence/bloom_filter.py:15-42): bit j of the filter is the byte mask[j];
// hash function i is v ^ offsets[i], reduced mod the mask size.
// ------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) bloom_insert_kernel(const int64_t *values, size_t n, const int64_t *offsets, int n_hash,
                                                           uint8_t *mask, uint64_t mask_size) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const int64_t v = values[i];
        for (int h = 0; h < n_hash; ++h) mask[(uint64_t)(v ^ offsets[h]) % mask_size] = 1;
    }
}
__global__ void __launch_bounds__(256) bloom_query_kernel(const int64_t *values, size_t n, const int64_t *offsets, int n_hash,
                                                          const uint8_t *mask, uint64_t mask_size, uint8_t *out) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x) {
        const int64_t v = values[i];
        uint8_t all = 1;
        for (int h = 0; h < n_hash; ++h) all &= mask[(uint64_t)(v ^ offsets[h]) % mask_size];
        out[i] = all;
    }
}

// ------------------------------------------------------------------------------------------
// synthetic FASTQ (bit-identical to oracle/bnp_oracle.py:synthetic_fastq)
// ------------------------------------------------------------------------------------------
__device__ __forceinline__ uint64_t splitmix64(uint64_t x) {
    uint64_t z = x + 0x9E3779B97F4A7C15ull;
    z = (z ^ (z >> 30)) * 0xBF58476D1CE4E5B9ull;
    z = (z ^ (z >> 27)) * 0x94D049BB133111EBull;
    return z ^ (z >> 31);
}

__global__ void __launch_bounds__(256) synth_fastq_kernel(uint8_t *out, uint64_t first_record, uint64_t n_records,
                                                          uint64_t seed) {
    const int lane = threadIdx.x & 31;
    const uint64_t warp_global = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint64_t n_warps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    for (uint64_t i = warp_global; i < n_records; i += n_warps) {
        const uint64_t r = first_record + i;
        uint8_t *rec = out + i * 317ull;
        const uint64_t key = seed * (1ull << 40) + r * 5ull;
        for (int j = lane; j < 317; j += 32) {
            uint8_t c;
            if (j == 0) c = '@';
            else if (j == 1) c = 'r';
            else if (j < 12) {
                uint64_t d = r;
                for (int t = 0; t < 11 - j; ++t) d /= 10;
                c = (uint8_t)('0' + d % 10);
            } else if (j == 12 || j == 163 || j == 165 || j == 316) c = '\n';
            else if (j < 163) {
                const int b = j - 13;
                const uint64_t z = splitmix64(key + (uint64_t)(b >> 5));
                c = "ACGT"[(z >> (2 * (b & 31))) & 3];
            } else if (j == 164) c = '+';
            else c = 'I';
            rec[j] = c;
        }
    }
}

}  // namespace bnpk

using namespace bnpk;

extern "C" {

int bnpk_abi_version(void) { return BNPK_ABI_VERSION; }
const char *bnpk_last_error(void) { return g_err; }
int bnpk_sm_count(void) { return sm_count(); }
uint64_t bnpk_launch_count(void) { return g_launches.load(); }

int bnpk_profile_enable(int on) {
    std::lock_guard<std::mutex> l(g_prof_mu);
    g_prof_on = on != 0;
    return 0;
}

int bnpk_profile_read(double *total_ms, uint64_t *n_launches) {
    std::lock_guard<std::mutex> l(g_prof_mu);
    double total = 0;
    uint64_t n = 0;
    for (auto &p : g_prof_events) {
        float ms = 0;
        cudaEventSynchronize(p.second);
        if (cudaEventElapsedTime(&ms, p.first, p.second) == cudaSuccess) { total += ms; ++n; }
        g_prof_pool.push_back(p.first);
        g_prof_pool.push_back(p.second);
    }
    g_prof_events.clear();
    if (total_ms) *total_ms = total;
    if (n_launches) *n_launches = n;
    return 0;
}

int bnpk_status_init(int64_t *status, void *stream) {
    status_init_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(status);
    BNPK_LAUNCHED("status_init_kernel");
    return 0;
}

int bnpk_count_byte(const uint8_t *chunk, size_t n, uint8_t value, int64_t *count_out, void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    BNPK_CUDA(cudaMemsetAsync(count_out, 0, sizeof(int64_t), st));
    if (n == 0) return 0;
    const size_t want = (n / 16 + 255) / 256;
    const unsigned grid = (unsigned)std::max<size_t>(1, std::min<size_t>(want, (size_t)sm_count() * 8));
    const uint32_t pattern = 0x01010101u * value;
    count_byte_kernel<<<grid, 256, 0, st>>>(chunk, n, pattern, (unsigned long long *)count_out);
    BNPK_LAUNCHED("count_byte_kernel");
    return 0;
}

size_t bnpk_tile_workspace_bytes(size_t n) { return tile_workspace_bytes(n); }

int bnpk_tile_workspace_reset(void *workspace, size_t workspace_bytes, void *stream) {
    BNPK_CUDA(cudaMemsetAsync(workspace, 0, workspace_bytes, (cudaStream_t)stream));
    return 0;
}

int bnpk_line_split(const uint8_t *chunk, size_t n, int lines_per_entry, int field_line, int start_offset,
                    uint8_t header_char, int check_plus, int trim_cr, int64_t *starts, int32_t *lens, size_t max_rows,
                    int64_t *status, void *workspace, size_t workspace_bytes, void *stream) {
    return line_split_impl(chunk, n, lines_per_entry, field_line, start_offset, header_char, check_plus, trim_cr,
                           starts, lens, max_rows, status, workspace, workspace_bytes, (cudaStream_t)stream);
}

int bnpk_chunk_kmer_count(const uint8_t *chunk, size_t n, size_t slice_begin, size_t slice_end, int final_slice,
                          int lines_per_entry, uint8_t header_char, int check_plus, int trim_cr, int enc_mode,
                          const uint8_t *lut256, int k, int window_size, int64_t n_bins, int hist_mode, int64_t *hist,
                          int64_t *status, void *workspace, size_t workspace_bytes, void *stream) {
    return chunk_kmer_count_impl(chunk, n, slice_begin, slice_end, final_slice, lines_per_entry, header_char,
                                 check_plus, trim_cr, enc_mode, lut256, k, window_size, n_bins, hist_mode, hist, status,
                                 workspace, workspace_bytes, (cudaStream_t)stream);
}

int bnpk_chunk_kmer_count_canonical(const uint8_t *chunk, size_t n, size_t slice_begin, size_t slice_end, int final_slice,
                                    int lines_per_entry, uint8_t header_char, int check_plus, int trim_cr, int enc_mode,
                                    const uint8_t *lut256, int k, int complement_xor, int64_t n_bins, int hist_mode,
                                    int64_t *hist, int64_t *status, void *workspace, size_t workspace_bytes, void *stream) {
    if (complement_xor < 1 || complement_xor > 3) return set_err(BNPK_E_BADARG, "complement_xor must be 1, 2 or 3");
    return chunk_kmer_count_impl(chunk, n, slice_begin, slice_end, final_slice, lines_per_entry, header_char,
                                 check_plus, trim_cr, enc_mode, lut256, k, 0, n_bins, hist_mode, hist, status,
                                 workspace, workspace_bytes, (cudaStream_t)stream, canon_pattern(complement_xor));
}

int bnpk_chunk_minimizer_count_canonical(const uint8_t *chunk, size_t n, size_t slice_begin, size_t slice_end,
                                         int final_slice, int lines_per_entry, uint8_t header_char, int check_plus,
                                         int trim_cr, int enc_mode, const uint8_t *lut256, int k, int window_size,
                                         int complement_xor, int64_t n_bins, int hist_mode, int64_t *hist,
                                         int64_t *status, void *workspace, size_t workspace_bytes, void *stream) {
    if (complement_xor < 1 || complement_xor > 3) return set_err(BNPK_E_BADARG, "complement_xor must be 1, 2 or 3");
    if (window_size < 1) return set_err(BNPK_E_WINDOW, "window_size must be positive");
    return chunk_kmer_count_impl(chunk, n, slice_begin, slice_end, final_slice, lines_per_entry, header_char,
                                 check_plus, trim_cr, enc_mode, lut256, k, window_size, n_bins, hist_mode, hist, status,
                                 workspace, workspace_bytes, (cudaStream_t)stream, canon_pattern(complement_xor));
}

int bnpk_row_offsets(const int32_t *lens, size_t n_rows, int shrink, int64_t *offsets, void *workspace,
                     size_t workspace_bytes, void *stream) {
    cudaStream_t st = (cudaStream_t)stream;
    if (n_rows == 0) {
        BNPK_CUDA(cudaMemsetAsync(offsets, 0, sizeof(int64_t), st));
        return 0;
    }
    const size_t n_tiles = (n_rows + kScanTile - 1) / kScanTile;
    const size_t need = (kWsHeaderWords + n_tiles) * sizeof(uint64_t);
    if (workspace_bytes < need) return set_err(BNPK_E_WORKSPACE, "workspace too small");
    BNPK_CUDA(cudaMemsetAsync(workspace, 0, need, st));
    const unsigned grid = (unsigned)std::min<size_t>(n_tiles, (size_t)sm_count() * 4);
    row_offsets_kernel<<<grid, kScanThreads, 0, st>>>(lens, n_rows, shrink, offsets, (uint64_t *)workspace);
    BNPK_LAUNCHED("row_offsets_kernel");
    return 0;
}

int bnpk_bincount(const int64_t *values, size_t n, int64_t n_bins, int hist_mode, int64_t *hist, int64_t *status,
                  void *stream) {
    if (n_bins < 1) return set_err(BNPK_E_BINS, "n_bins must be positive");
    if (hist_mode == BNPK_HIST_SMEM && n_bins > kSmemMaxBins) return set_err(BNPK_E_BINS, "too many bins for the shared-memory histogram");
    if (n == 0) return 0;
    cudaStream_t st = (cudaStream_t)stream;
    const bool sm = use_smem_hist(n_bins, hist_mode);
    const size_t want = (n + 511) / 512;
    if (sm) {
        BNPK_DYN_SMEM(bincount_kernel<true>, 200 * 1024);
        const size_t smem = (size_t)n_bins * 4;
        int per_sm = 1;
        BNPK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, bincount_kernel<true>, 512, smem));
        const unsigned grid = (unsigned)std::max<size_t>(1, std::min<size_t>(want, (size_t)sm_count() * std::max(per_sm, 1)));
        bincount_kernel<true><<<grid, 512, smem, st>>>(values, n, (uint64_t)n_bins, (unsigned long long *)hist, status);
    } else {
        const unsigned grid = (unsigned)std::max<size_t>(1, std::min<size_t>(want, (size_t)sm_count() * 4));
        bincount_kernel<false><<<grid, 512, 0, st>>>(values, n, (uint64_t)n_bins, (unsigned long long *)hist, status);
    }
    BNPK_LAUNCHED("bincount_kernel");
    return 0;
}

int bnpk_bincount_rows(const int64_t *values, const int64_t *offsets, size_t n_rows, int64_t n_bins, int64_t *out,
                       int64_t *status, void *stream) {
    if (n_bins < 1) return set_err(BNPK_E_BINS, "n_bins must be positive");
    if (n_rows == 0) return 0;
    const size_t want = (n_rows + 7) / 8;
    const unsigned grid = (unsigned)std::max<size_t>(1, std::min<size_t>(want, (size_t)sm_count() * 8));
    bincount_rows_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(values, offsets, n_rows, (uint64_t)n_bins,
                                                                 (unsigned long long *)out, status);
    BNPK_LAUNCHED("bincount_rows_kernel");
    return 0;
}

int bnpk_multiline_flags(const uint8_t *chunk, size_t n, const int64_t *line_starts, const int32_t *line_lens, size_t n_lines,
                         int32_t *is_header, int64_t *out2, void *stream) {
    if (n_lines == 0 || n == 0) return 0;
    const unsigned grid = (unsigned)std::max<size_t>(1, std::min<size_t>((n_lines + 255) / 256, (size_t)sm_count() * 8));
    multiline_flags_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(chunk, n, line_starts, line_lens, n_lines, is_header, out2);
    BNPK_LAUNCHED("multiline_flags_kernel");
    return 0;
}

int bnpk_multiline_entries(const uint8_t *chunk, const int64_t *line_starts, const int32_t *line_lens, const int32_t *is_header,
                           const int64_t *hdr_before, size_t keep, int trim_cr, int64_t *h_starts, int32_t *h_lens,
                           int64_t *s_starts, int32_t *s_lens, int64_t *entry_lens, void *stream) {
    if (keep == 0) return 0;
    const unsigned grid = (unsigned)std::max<size_t>(1, std::min<size_t>((keep + 255) / 256, (size_t)sm_count() * 8));
    multiline_entries_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(chunk, line_starts, line_lens, is_header, hdr_before, keep, trim_cr,
                                                                     h_starts, h_lens, s_starts, s_lens,
                                                                     (unsigned long long *)entry_lens);
    BNPK_LAUNCHED("multiline_entries_kernel");
    return 0;
}

int bnpk_fasta_gather(const uint8_t *file, size_t file_bytes, size_t n_rows, const int64_t *contig_offset,
                      const int64_t *row_start, const int64_t *row_len, const int32_t *lenc, const int32_t *lenb,
                      const int64_t *out_offsets, uint8_t *out, int64_t *status, void *stream) {
    if (n_rows == 0) return 0;
    const size_t want = (n_rows + 7) / 8;
    const unsigned grid = (unsigned)std::max<size_t>(1, std::min<size_t>(want, (size_t)sm_count() * 8));
    fasta_gather_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(file, file_bytes, n_rows, contig_offset, row_start, row_len, lenc,
                                                                lenb, out_offsets, out, status);
    BNPK_LAUNCHED("fasta_gather_kernel");
    return 0;
}

int bnpk_bloom_insert(const int64_t *values, size_t n, const int64_t *offsets, int n_hash, uint8_t *mask, size_t mask_size,
                      void *stream) {
    if (n_hash < 1 || mask_size == 0) return set_err(BNPK_E_BADARG, "bloom filter needs hash functions and a mask");
    if (n == 0) return 0;
    const unsigned grid = (unsigned)std::max<size_t>(1, std::min<size_t>((n + 255) / 256, (size_t)sm_count() * 16));
    bloom_insert_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(values, n, offsets, n_hash, mask, (uint64_t)mask_size);
    BNPK_LAUNCHED("bloom_insert_kernel");
    return 0;
}

int bnpk_bloom_query(const int64_t *values, size_t n, const int64_t *offsets, int n_hash, const uint8_t *mask, size_t mask_size,
                     uint8_t *out, void *stream) {
    if (n_hash < 1 || mask_size == 0) return set_err(BNPK_E_BADARG, "bloom filter needs hash functions and a mask");
    if (n == 0) return 0;
    const unsigned grid = (unsigned)std::max<size_t>(1, std::min<size_t>((n + 255) / 256, (size_t)sm_count() * 16));
    bloom_query_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(values, n, offsets, n_hash, mask, (uint64_t)mask_size, out);
    BNPK_LAUNCHED("bloom_query_kernel");
    return 0;
}

int bnpk_synth_fastq(uint8_t *out, uint64_t first_record, uint64_t n_records, uint64_t seed, void *stream) {
    if (n_records == 0) return 0;
    const uint64_t want = (n_records + 7) / 8;
    const unsigned grid = (unsigned)std::max<uint64_t>(1, std::min<uint64_t>(want, (uint64_t)sm_count() * 16));
    synth_fastq_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(out, first_record, n_records, seed);
    BNPK_LAUNCHED("synth_fastq_kernel");
    return 0;
}

}  // extern "C"
