// row_kernels.cu -- kernels driven by a row-offset vector (starts[R], lens[R]) over a byte buffer:
// the general EncodedRaggedArray form (io/file_buffers.py:335-338).  One warp per read row; rows
// longer than one staging segment are walked in overlapping segments by the same warp.
//   K2 rows_encode      change_encoding            encoded_array.py:655-695
//   K3 rows_kmer_hash   get_kmers/_get_dna_kmers   sequence/kmers.py:36-126
//   K4 rows_minimizers  get_minimizers             sequence/minimizers.py:20-54
//   K3/K4+K5 rows_kmer_count   count_kmers         sequence/kmers.py:129-145
// plus the clean-up passes of the fused chunk count (long rows, trailing incomplete entry).
#include <climits>
#include "bnpk_host.h"

namespace bnpk {

constexpr int kRowThreads = 256;
constexpr int kRowWarps = kRowThreads / 32;
constexpr int kSegUnits = 128;               // 2 KiB staged per warp and segment
constexpr int kSegBytes = kSegUnits * 16;
constexpr int kWarpWords = 2 * kSegUnits + 4;

enum { RM_ENCODE = 0, RM_HASH = 1, RM_MINIMIZER = 2, RM_COUNT = 3, RM_COUNT_MIN = 4 };

struct RowArgs {
    const uint8_t *base;
    size_t base_bytes;
    const int64_t *starts;
    const int32_t *lens;
    size_t n_rows;
    const uint8_t *lut;
    int k, window;
    const int64_t *offsets;
    void *out;
    uint64_t n_bins;
    unsigned long long *hist;
    int64_t *status;
    // deferred (long-row) mode
    const uint64_t *deferred_count;
    const uint64_t *deferred;
    size_t deferred_cap;
    int lpe;
    uint64_t canon_xor;          // != 0: canonical k-mers, or canonical minimizers with a window
};

template <int RM, int ENC, bool SMEM_HIST>
__device__ void warp_row(const RowArgs &a, uint32_t *w_codes, uint32_t *w_flags, const uint8_t *s_lut,
                         const HistTarget &ht, int64_t start, int64_t L, int64_t r, int64_t out_off, int lane,
                         uint64_t &acc_values) {
    constexpr bool MINZ = (RM == RM_MINIMIZER || RM == RM_COUNT_MIN);
    const int span = MINZ ? a.window : (RM == RM_ENCODE ? 1 : a.k);
    const uint64_t kmask = (1ull << (2 * a.k)) - 1;
    int64_t seg_start = 0;
    bool reported = false;
    while (seg_start < L) {
        const int64_t g0 = start + seg_start;
        const int off = (int)((reinterpret_cast<uintptr_t>(a.base) + g0) & 15);
        const int64_t ua = g0 - off;
        const int seg_len = (int)min(L - seg_start, (int64_t)(kSegBytes - off));
        const int n_units = (off + seg_len + 15) >> 4;
        for (int u = lane; u < n_units; u += 32) {
            const uint4 q = load_unit_guarded(a.base, a.base_bytes, ua + 16 * (int64_t)u);
            uint32_t c, f;
            encode_unit<ENC>(q, s_lut, c, f);
            w_codes[u] = c;
            w_flags[u] = f;
        }
        if (lane < 4) w_codes[n_units + lane] = 0;
        __syncwarp();
        if (!reported && !(RM == RM_ENCODE && ENC == BNPK_ENC_LUT)) {
            const int bad = find_invalid(w_flags, off, off + seg_len, lane);
            if (bad >= 0) {
                reported = true;
                if (lane == 0)
                    atomicMin((long long *)&a.status[BNPK_ST_BAD_BASE], (long long)((r << 32) | (seg_start + bad - off)));
            }
        }
        if constexpr (RM == RM_ENCODE) {
            uint8_t *out = reinterpret_cast<uint8_t *>(a.out) + out_off + seg_start;
            if constexpr (ENC == BNPK_ENC_LUT) {
                // any alphabet size: the full LUT value is the code, 255 = invalid
                // (AlphabetEncoding._encode, encodings/alphabet_encoding.py:34-46)
                int first_bad = INT_MAX;
                for (int p = lane; p < seg_len; p += 32) {
                    const uint8_t code = s_lut[a.base[g0 + p]];
                    out[p] = code;
                    if (code == 255 && p < first_bad) first_bad = p;
                }
#pragma unroll
                for (int o = 16; o; o >>= 1) first_bad = min(first_bad, __shfl_xor_sync(0xffffffffu, first_bad, o));
                if (first_bad != INT_MAX && !reported) {
                    reported = true;
                    if (lane == 0)
                        atomicMin((long long *)&a.status[BNPK_ST_BAD_BASE], (long long)((r << 32) | (seg_start + first_bad)));
                }
            } else {
                for (int p = lane; p < seg_len; p += 32) {
                    const int b = off + p;
                    out[p] = (uint8_t)((w_codes[b >> 4] >> (2 * (b & 15))) & 3u);
                }
            }
        } else if constexpr (RM == RM_HASH) {
            int64_t *out = reinterpret_cast<int64_t *>(a.out) + out_off + seg_start;
            const int npos = seg_len - span + 1;
            for (int p = lane; p < npos; p += 32) {
                uint64_t h = stream_64(w_codes, (uint32_t)(off + p)) & kmask;
                if (a.canon_xor) h = canonical_hash(h, a.k, a.canon_xor);
                out[p] = (int64_t)h;
            }
            if (npos > 0) acc_values += (uint64_t)((npos - lane + 31) / 32);
        } else if constexpr (RM == RM_MINIMIZER) {
            int64_t *out = reinterpret_cast<int64_t *>(a.out) + out_off + seg_start;
            const int w = a.window - a.k + 1;
            const int nout = seg_len - a.window + 1;
            const int nh = seg_len - a.k + 1;
            if (w <= 32) {
                const int step = 32 - (w - 1);
                for (int base = 0; base < nout; base += step) {
                    const int p = base + lane;
                    uint64_t h = ~0ull;                       // lanes past the last hash keep the sentinel
                    if (p < nh) {
                        h = stream_64(w_codes, (uint32_t)(off + p)) & kmask;
                        if (a.canon_xor) h = canonical_hash(h, a.k, a.canon_xor);
                    }
                    const uint64_t m = warp_sliding_min(h, w);
                    if (lane < step && p < nout) { out[p] = (int64_t)m; ++acc_values; }
                }
            } else {
                for (int j = lane; j < nout; j += 32) {
                    uint64_t m = ~0ull;
                    for (int i = 0; i < w; ++i) {
                        uint64_t h = stream_64(w_codes, (uint32_t)(off + j + i)) & kmask;
                        if (a.canon_xor) h = canonical_hash(h, a.k, a.canon_xor);
                        m = h < m ? h : m;
                    }
                    out[j] = (int64_t)m;
                    ++acc_values;
                }
            }
        } else {
            if (seg_len >= span)
                acc_values += row_count<SMEM_HIST, MINZ>(w_codes, off, seg_len, a.k, a.window, ht, lane);
        }
        __syncwarp();
        if (seg_start + seg_len >= L) break;
        seg_start += seg_len - (span - 1);
    }
}

template <int RM, int ENC, bool SMEM_HIST, bool DEFERRED>
__global__ void __launch_bounds__(kRowThreads) rows_kernel(const RowArgs a) {
    extern __shared__ __align__(16) uint32_t smem[];
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    uint32_t *w_codes = smem + warp * kWarpWords;
    uint32_t *w_flags = w_codes + kSegUnits + 4;
    uint8_t *s_lut = reinterpret_cast<uint8_t *>(smem + kRowWarps * kWarpWords);
    uint32_t *s_hist = reinterpret_cast<uint32_t *>(s_lut + 256);
    if (ENC == BNPK_ENC_LUT && tid < 256) s_lut[tid] = a.lut[tid];
    constexpr bool COUNTING = (RM == RM_COUNT || RM == RM_COUNT_MIN);
    if (COUNTING && SMEM_HIST)
        for (uint32_t b = tid; b < a.n_bins; b += kRowThreads) s_hist[b] = 0;
    HistTarget ht;
    ht.global = a.hist;
    ht.smem = s_hist;
    ht.n_bins = a.n_bins;
    ht.mask = (a.n_bins & (a.n_bins - 1)) == 0 ? a.n_bins - 1 : 0;
    ht.delta = 1ull;
    ht.canon_xor = a.canon_xor;
    __syncthreads();

    uint64_t acc_values = 0, acc_bases = 0, acc_long = 0;
    size_t n_rows = a.n_rows;
    int64_t n_records = 0;
    bool cr = false;
    if (DEFERRED) {
        n_rows = (size_t)min((unsigned long long)*a.deferred_count, (unsigned long long)a.deferred_cap);
        n_records = a.status[BNPK_ST_N_RECORDS];
        cr = a.status[BNPK_ST_CR] != 0;
    }
    for (size_t row = (size_t)blockIdx.x * kRowWarps + warp; row < n_rows; row += (size_t)gridDim.x * kRowWarps) {
        int64_t start, L, r, out_off = 0;
        if (DEFERRED) {
            start = (int64_t)a.deferred[2 * row];
            const uint64_t rw = a.deferred[2 * row + 1];
            r = (int64_t)(rw & ~kDeferredResolved);
            if (r >= n_records) continue;                     // belongs to a trailing incomplete entry
            L = warp_line_len(a.base, a.base_bytes, start, lane);
            if (L < 0) continue;
            const int64_t end = start + L;                    // its newline
            if (cr && L > 0 && a.base[start + L - 1] == '\r') L -= 1;
            // a row of a tile the ws resolve pass walked is a long row only if the in-tile walk would have deferred it:
            // its newline past the tile's slot, or more than kWsRowMax bytes
            const int64_t slot_end = ((start - 1) & ~(int64_t)(kTileBytes - 1)) + kWsSlotBytes;
            if (lane == 0 && (!(rw & kDeferredResolved) || end >= slot_end || L > kWsRowMax)) ++acc_long;
        } else {
            start = a.starts[row];
            L = a.lens[row];
            r = (int64_t)row;
            if (a.offsets) out_off = a.offsets[row];
        }
        if (L <= 0) continue;
        if (lane == 0) acc_bases += (uint64_t)L;
        warp_row<RM, ENC, SMEM_HIST>(a, w_codes, w_flags, s_lut, ht, start, L, r, out_off, lane, acc_values);
    }
    if (COUNTING && SMEM_HIST) {
        __syncthreads();
        for (uint32_t b = tid; b < a.n_bins; b += kRowThreads) {
            const uint32_t c = s_hist[b];
            if (c) atomicAdd(a.hist + b, (unsigned long long)c);
        }
    }
    acc_values = warp_sum_u64(acc_values);
    acc_bases = warp_sum_u64(acc_bases);
    acc_long = warp_sum_u64(acc_long);
    if (lane == 0) {
        if (acc_values) atomicAdd((unsigned long long *)&a.status[BNPK_ST_N_VALUES], acc_values);
        if (acc_bases) atomicAdd((unsigned long long *)&a.status[BNPK_ST_N_BASES], acc_bases);
        if (acc_long) atomicAdd((unsigned long long *)&a.status[BNPK_ST_N_LONG_ROWS], acc_long);
    }
}

// Un-count the sequence line of a trailing incomplete entry: the fused pass counts every
// terminated sequence line it meets; the reference only keeps entries with all their lines
// (io/one_line_buffer.py:67).  One warp.
template <int ENC, bool MINZ>
__global__ void uncount_kernel(const RowArgs a) {
    extern __shared__ __align__(16) uint32_t smem[];
    const int lane = threadIdx.x & 31;
    const int64_t n_lines = a.status[BNPK_ST_N_LINES];
    const int64_t n_records = n_lines / a.lpe;
    if (n_lines % a.lpe < 2) return;                          // its sequence line was never terminated
    if (a.status[BNPK_ST_LAST_ROW_INDEX] - 1 != n_records) return;  // that line was not counted in-tile
    const int64_t start = a.status[BNPK_ST_LAST_ROW_START] - 1;
    int64_t L = warp_line_len(a.base, a.base_bytes, start, lane);
    if (L < 0) return;
    if (a.status[BNPK_ST_CR] != 0 && L > 0 && a.base[start + L - 1] == '\r') L -= 1;
    uint32_t *w_codes = smem;
    uint32_t *w_flags = w_codes + kSegUnits + 4;
    uint8_t *s_lut = reinterpret_cast<uint8_t *>(smem + kWarpWords);
    if (ENC == BNPK_ENC_LUT)
        for (int i = lane; i < 256; i += 32) s_lut[i] = a.lut[i];
    __syncwarp();
    HistTarget ht;
    ht.global = a.hist;
    ht.smem = nullptr;
    ht.n_bins = a.n_bins;
    ht.mask = (a.n_bins & (a.n_bins - 1)) == 0 ? a.n_bins - 1 : 0;
    ht.delta = ~0ull;                                          // -1
    ht.canon_xor = a.canon_xor;                                // the values the fused pass counted
    uint64_t produced = 0;
    // the BAD_BASE slot must not be touched by this row: point validation at a scratch word
    RowArgs b = a;
    __shared__ int64_t scratch_status[BNPK_ST_WORDS];
    if (lane < BNPK_ST_WORDS) scratch_status[lane] = INT64_MAX;
    __syncwarp();
    b.status = scratch_status;
    warp_row<MINZ ? RM_COUNT_MIN : RM_COUNT, ENC, false>(b, w_codes, w_flags, s_lut, ht, start, L, n_records, 0, lane, produced);
    produced = warp_sum_u64(produced);
    if (lane == 0) {
        atomicAdd((unsigned long long *)&a.status[BNPK_ST_N_VALUES], 0ull - produced);
        atomicAdd((unsigned long long *)&a.status[BNPK_ST_N_BASES], 0ull - (unsigned long long)L);
    }
}


// ---------------------------------------------------------------------------------------------
// Generic alphabets (size != 4): h = sum_j code[i+j] * A^j in int64 arithmetic, the reference's
// KmerEncoder dot product (sequence/kmers.py:17-27, sequence/rollable.py:49-66).  One warp per row,
// one lane per window; codes come from a 256-byte LUT (or are the bytes themselves).
// ---------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) rows_generic_hash_kernel(const uint8_t *base, size_t base_bytes, const int64_t *starts,
                                                                const int32_t *lens, size_t n_rows, const uint8_t *lut,
                                                                int alphabet_size, int k, const int64_t *offsets,
                                                                int64_t *out, int64_t *status) {
    __shared__ uint8_t s_lut[256];
    __shared__ unsigned long long s_pow[64];
    const int tid = threadIdx.x, lane = tid & 31;
    if (tid < 256) s_lut[tid] = lut ? lut[tid] : (uint8_t)tid;
    if (tid == 0) {
        unsigned long long p = 1;
        for (int j = 0; j < 64; ++j) { s_pow[j] = p; p *= (unsigned long long)alphabet_size; }
    }
    __syncthreads();
    const size_t warp_global = ((size_t)blockIdx.x * blockDim.x + tid) >> 5;
    const size_t n_warps = ((size_t)gridDim.x * blockDim.x) >> 5;
    for (size_t r = warp_global; r < n_rows; r += n_warps) {
        const int64_t start = starts[r], L = lens[r], o = offsets[r];
        for (int64_t i = lane; i < L; i += 32) {                    // validity of every symbol of the row
            const uint8_t c = s_lut[base[start + i]];
            if (c >= alphabet_size) atomicMin((long long *)&status[BNPK_ST_BAD_BASE], (long long)(((int64_t)r << 32) | i));
        }
        for (int64_t i = lane; i + k <= L; i += 32) {
            unsigned long long h = 0;
            for (int j = 0; j < k; ++j) h += (unsigned long long)s_lut[base[start + i + j]] * s_pow[j];
            out[o + i] = (int64_t)h;
        }
    }
}

// get_reverse_complement (sequence/dna.py:36-65): out row r = lut[row r read backwards]; one warp per row,
// coalesced writes.  The 256-byte lut is the reference's complement Lookup for the array's encoding.
__global__ void __launch_bounds__(256) rows_reverse_complement_kernel(const uint8_t *base, const int64_t *starts, const int32_t *lens,
                                                                      size_t n_rows, const uint8_t *lut, const int64_t *offsets,
                                                                      uint8_t *out) {
    __shared__ uint8_t s_lut[256];
    const int tid = threadIdx.x, lane = tid & 31;
    s_lut[tid] = lut[tid];
    __syncthreads();
    const size_t warp_global = ((size_t)blockIdx.x * blockDim.x + tid) >> 5;
    const size_t n_warps = ((size_t)gridDim.x * blockDim.x) >> 5;
    for (size_t r = warp_global; r < n_rows; r += n_warps) {
        const int64_t start = starts[r], L = lens[r], o = offsets[r];
        for (int64_t i = lane; i < L; i += 32) out[o + i] = s_lut[base[start + L - 1 - i]];
    }
}

static size_t rows_smem_bytes(bool counting, bool smem_hist, uint64_t n_bins) {
    size_t b = (size_t)kRowWarps * kWarpWords * 4 + 256;
    if (counting && smem_hist) b += n_bins * 4;
    return b;
}

template <int RM, int ENC, bool SMEM_HIST, bool DEFERRED>
static int launch_rows_t(const RowArgs &a, size_t est_rows, cudaStream_t st) {
    auto kern = rows_kernel<RM, ENC, SMEM_HIST, DEFERRED>;
    constexpr bool COUNTING = (RM == RM_COUNT || RM == RM_COUNT_MIN);
    const size_t smem = rows_smem_bytes(COUNTING, SMEM_HIST, a.n_bins);
    BNPK_DYN_SMEM(kern, 200 * 1024);
    int per_sm = 1;
    BNPK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kRowThreads, smem));
    if (per_sm < 1) return set_err(BNPK_E_BINS, "rows kernel does not fit shared memory");
    const size_t want = (est_rows + kRowWarps - 1) / kRowWarps;
    const size_t cap = (size_t)sm_count() * per_sm;
    const unsigned grid = (unsigned)std::max<size_t>(1, std::min(want, cap));
    kern<<<grid, kRowThreads, smem, st>>>(a);
    BNPK_LAUNCHED("rows_kernel");
    return 0;
}

template <int RM, bool SMEM_HIST, bool DEFERRED>
static int launch_rows_enc(const RowArgs &a, int enc_mode, size_t est_rows, cudaStream_t st) {
    switch (enc_mode) {
        case BNPK_ENC_ASCII_ACGT: return launch_rows_t<RM, BNPK_ENC_ASCII_ACGT, SMEM_HIST, DEFERRED>(a, est_rows, st);
        case BNPK_ENC_ASCII_ACTG: return launch_rows_t<RM, BNPK_ENC_ASCII_ACTG, SMEM_HIST, DEFERRED>(a, est_rows, st);
        case BNPK_ENC_CODES: return launch_rows_t<RM, BNPK_ENC_CODES, SMEM_HIST, DEFERRED>(a, est_rows, st);
        case BNPK_ENC_LUT: return launch_rows_t<RM, BNPK_ENC_LUT, SMEM_HIST, DEFERRED>(a, est_rows, st);
    }
    return set_err(BNPK_E_BADARG, "bad enc_mode");
}

static int check_common(int enc_mode, const uint8_t *lut256, int k, int window) {
    if (k < 1 || k > 31) return set_err(BNPK_E_K, "k must be larger than 0 and smaller than 32");
    if (window != 0 && window < k) return set_err(BNPK_E_WINDOW, "kmer size must be smaller than window size");
    if (window > kSegBytes / 2) return set_err(BNPK_E_WINDOW, "window_size above 1024 is not supported");
    if (enc_mode < 0 || enc_mode > 3) return set_err(BNPK_E_BADARG, "bad enc_mode");
    if (enc_mode == BNPK_ENC_LUT && !lut256) return set_err(BNPK_E_BADARG, "lut256 required");
    return 0;
}

template <bool MINZ>
static int launch_uncount(const RowArgs &a, int enc_mode, cudaStream_t st) {
    const size_t smem = kWarpWords * 4 + 256;
    switch (enc_mode) {
        case BNPK_ENC_ASCII_ACGT: uncount_kernel<BNPK_ENC_ASCII_ACGT, MINZ><<<1, 32, smem, st>>>(a); break;
        case BNPK_ENC_ASCII_ACTG: uncount_kernel<BNPK_ENC_ASCII_ACTG, MINZ><<<1, 32, smem, st>>>(a); break;
        case BNPK_ENC_CODES: uncount_kernel<BNPK_ENC_CODES, MINZ><<<1, 32, smem, st>>>(a); break;
        default: uncount_kernel<BNPK_ENC_LUT, MINZ><<<1, 32, smem, st>>>(a); break;
    }
    BNPK_LAUNCHED("uncount_kernel");
    return 0;
}

int count_fixups_impl(const uint8_t *chunk, size_t n, int lpe, int enc_mode, const uint8_t *lut256, int k,
                      int window, int64_t n_bins, int64_t *hist, int64_t *status, const uint64_t *deferred_count,
                      const uint64_t *deferred, size_t deferred_cap, cudaStream_t st, uint64_t canon_xor) {
    RowArgs a{};
    a.base = chunk; a.base_bytes = n; a.lut = lut256; a.k = k; a.window = window;
    a.n_bins = (uint64_t)n_bins; a.hist = (unsigned long long *)hist; a.status = status;
    a.deferred_count = deferred_count; a.deferred = deferred; a.deferred_cap = deferred_cap; a.lpe = lpe;
    a.canon_xor = canon_xor;                                   // long rows and the un-count count canonical values too
    // long rows: a modest fixed grid; the kernel reads the row count on the device
    const size_t est = (size_t)sm_count() * kRowWarps * 2;
    int rc = window ? launch_rows_enc<RM_COUNT_MIN, false, true>(a, enc_mode, est, st)
                    : launch_rows_enc<RM_COUNT, false, true>(a, enc_mode, est, st);
    if (rc) return rc;
    return window ? launch_uncount<true>(a, enc_mode, st) : launch_uncount<false>(a, enc_mode, st);
}

}  // namespace bnpk

using namespace bnpk;

extern "C" {

int bnpk_rows_encode(const uint8_t *base, size_t base_bytes, const int64_t *starts, const int32_t *lens, size_t n_rows,
                     int enc_mode, const uint8_t *lut256, const int64_t *offsets, uint8_t *codes_out,
                     int64_t *status, void *stream) {
    if (int rc = check_common(enc_mode, lut256, 1, 0)) return rc;
    if (n_rows == 0) return 0;
    RowArgs a{};
    a.base = base; a.base_bytes = base_bytes; a.starts = starts; a.lens = lens; a.n_rows = n_rows; a.lut = lut256;
    a.k = 1; a.offsets = offsets; a.out = codes_out; a.n_bins = 1; a.status = status;
    return launch_rows_enc<RM_ENCODE, false, false>(a, enc_mode, n_rows, (cudaStream_t)stream);
}

int bnpk_rows_kmer_hash(const uint8_t *base, size_t base_bytes, const int64_t *starts, const int32_t *lens, size_t n_rows,
                        int enc_mode, const uint8_t *lut256, int k, const int64_t *offsets, int64_t *hashes_out,
                        int64_t *status, void *stream) {
    if (int rc = check_common(enc_mode, lut256, k, 0)) return rc;
    if (n_rows == 0) return 0;
    RowArgs a{};
    a.base = base; a.base_bytes = base_bytes; a.starts = starts; a.lens = lens; a.n_rows = n_rows; a.lut = lut256;
    a.k = k; a.offsets = offsets; a.out = hashes_out; a.n_bins = 1; a.status = status;
    return launch_rows_enc<RM_HASH, false, false>(a, enc_mode, n_rows, (cudaStream_t)stream);
}

int bnpk_rows_generic_hash(const uint8_t *base, size_t base_bytes, const int64_t *starts, const int32_t *lens, size_t n_rows,
                            const uint8_t *lut256, int alphabet_size, int k, const int64_t *offsets, int64_t *hashes_out,
                            int64_t *status, void *stream) {
    if (k < 1 || k > 63) return set_err(BNPK_E_K, "k must be in 1..63 for the generic hash");
    if (alphabet_size < 2 || alphabet_size > 255) return set_err(BNPK_E_BADARG, "alphabet_size must be in 2..255");
    if (n_rows == 0) return 0;
    const size_t want = (n_rows + 7) / 8;
    const unsigned grid = (unsigned)std::max<size_t>(1, std::min<size_t>(want, (size_t)sm_count() * 8));
    rows_generic_hash_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(base, base_bytes, starts, lens, n_rows, lut256,
                                                                    alphabet_size, k, offsets, hashes_out, status);
    BNPK_LAUNCHED("rows_generic_hash_kernel");
    return 0;
}

int bnpk_rows_minimizers(const uint8_t *base, size_t base_bytes, const int64_t *starts, const int32_t *lens, size_t n_rows,
                         int enc_mode, const uint8_t *lut256, int k, int window_size, const int64_t *offsets,
                         int64_t *mins_out, int64_t *status, void *stream) {
    if (window_size < 1) return set_err(BNPK_E_WINDOW, "window_size must be positive");
    if (int rc = check_common(enc_mode, lut256, k, window_size)) return rc;
    if (n_rows == 0) return 0;
    RowArgs a{};
    a.base = base; a.base_bytes = base_bytes; a.starts = starts; a.lens = lens; a.n_rows = n_rows; a.lut = lut256;
    a.k = k; a.window = window_size; a.offsets = offsets; a.out = mins_out; a.n_bins = 1; a.status = status;
    return launch_rows_enc<RM_MINIMIZER, false, false>(a, enc_mode, n_rows, (cudaStream_t)stream);
}

int bnpk_rows_kmer_count(const uint8_t *base, size_t base_bytes, const int64_t *starts, const int32_t *lens, size_t n_rows,
                         int enc_mode, const uint8_t *lut256, int k, int window_size, int64_t n_bins, int hist_mode,
                         int64_t *hist, int64_t *status, void *stream) {
    if (int rc = check_common(enc_mode, lut256, k, window_size)) return rc;
    if (n_bins < 1) return set_err(BNPK_E_BINS, "n_bins must be positive");
    if (hist_mode == BNPK_HIST_SMEM && n_bins > kSmemMaxBins) return set_err(BNPK_E_BINS, "too many bins for the shared-memory histogram");
    if (n_rows == 0) return 0;
    RowArgs a{};
    a.base = base; a.base_bytes = base_bytes; a.starts = starts; a.lens = lens; a.n_rows = n_rows; a.lut = lut256;
    a.k = k; a.window = window_size; a.n_bins = (uint64_t)n_bins; a.hist = (unsigned long long *)hist; a.status = status;
    const bool sm = use_smem_hist(n_bins, hist_mode);
    cudaStream_t st = (cudaStream_t)stream;
    if (window_size)
        return sm ? launch_rows_enc<RM_COUNT_MIN, true, false>(a, enc_mode, n_rows, st)
                  : launch_rows_enc<RM_COUNT_MIN, false, false>(a, enc_mode, n_rows, st);
    return sm ? launch_rows_enc<RM_COUNT, true, false>(a, enc_mode, n_rows, st)
              : launch_rows_enc<RM_COUNT, false, false>(a, enc_mode, n_rows, st);
}

int bnpk_rows_kmer_hash_canonical(const uint8_t *base, size_t base_bytes, const int64_t *starts, const int32_t *lens,
                                  size_t n_rows, int enc_mode, const uint8_t *lut256, int k, int complement_xor,
                                  const int64_t *offsets, int64_t *hashes_out, int64_t *status, void *stream) {
    if (int rc = check_common(enc_mode, lut256, k, 0)) return rc;
    if (complement_xor < 1 || complement_xor > 3) return set_err(BNPK_E_BADARG, "complement_xor must be 1, 2 or 3");
    if (n_rows == 0) return 0;
    RowArgs a{};
    a.base = base; a.base_bytes = base_bytes; a.starts = starts; a.lens = lens; a.n_rows = n_rows; a.lut = lut256;
    a.k = k; a.offsets = offsets; a.out = hashes_out; a.n_bins = 1; a.status = status;
    a.canon_xor = canon_pattern(complement_xor);
    return launch_rows_enc<RM_HASH, false, false>(a, enc_mode, n_rows, (cudaStream_t)stream);
}

int bnpk_rows_kmer_count_canonical(const uint8_t *base, size_t base_bytes, const int64_t *starts, const int32_t *lens,
                                   size_t n_rows, int enc_mode, const uint8_t *lut256, int k, int complement_xor,
                                   int64_t n_bins, int hist_mode, int64_t *hist, int64_t *status, void *stream) {
    if (int rc = check_common(enc_mode, lut256, k, 0)) return rc;
    if (complement_xor < 1 || complement_xor > 3) return set_err(BNPK_E_BADARG, "complement_xor must be 1, 2 or 3");
    if (n_bins < 1) return set_err(BNPK_E_BINS, "n_bins must be positive");
    if (hist_mode == BNPK_HIST_SMEM && n_bins > kSmemMaxBins) return set_err(BNPK_E_BINS, "too many bins for the shared-memory histogram");
    if (n_rows == 0) return 0;
    RowArgs a{};
    a.base = base; a.base_bytes = base_bytes; a.starts = starts; a.lens = lens; a.n_rows = n_rows; a.lut = lut256;
    a.k = k; a.n_bins = (uint64_t)n_bins; a.hist = (unsigned long long *)hist; a.status = status;
    a.canon_xor = canon_pattern(complement_xor);
    cudaStream_t st = (cudaStream_t)stream;
    return use_smem_hist(n_bins, hist_mode) ? launch_rows_enc<RM_COUNT, true, false>(a, enc_mode, n_rows, st)
                                            : launch_rows_enc<RM_COUNT, false, false>(a, enc_mode, n_rows, st);
}

int bnpk_rows_minimizers_canonical(const uint8_t *base, size_t base_bytes, const int64_t *starts, const int32_t *lens,
                                   size_t n_rows, int enc_mode, const uint8_t *lut256, int k, int window_size,
                                   int complement_xor, const int64_t *offsets, int64_t *mins_out, int64_t *status,
                                   void *stream) {
    if (complement_xor < 1 || complement_xor > 3) return set_err(BNPK_E_BADARG, "complement_xor must be 1, 2 or 3");
    if (window_size < 1) return set_err(BNPK_E_WINDOW, "window_size must be positive");
    if (int rc = check_common(enc_mode, lut256, k, window_size)) return rc;
    if (n_rows == 0) return 0;
    RowArgs a{};
    a.base = base; a.base_bytes = base_bytes; a.starts = starts; a.lens = lens; a.n_rows = n_rows; a.lut = lut256;
    a.k = k; a.window = window_size; a.offsets = offsets; a.out = mins_out; a.n_bins = 1; a.status = status;
    a.canon_xor = canon_pattern(complement_xor);
    return launch_rows_enc<RM_MINIMIZER, false, false>(a, enc_mode, n_rows, (cudaStream_t)stream);
}

int bnpk_rows_minimizer_count_canonical(const uint8_t *base, size_t base_bytes, const int64_t *starts,
                                        const int32_t *lens, size_t n_rows, int enc_mode, const uint8_t *lut256, int k,
                                        int window_size, int complement_xor, int64_t n_bins, int hist_mode,
                                        int64_t *hist, int64_t *status, void *stream) {
    if (complement_xor < 1 || complement_xor > 3) return set_err(BNPK_E_BADARG, "complement_xor must be 1, 2 or 3");
    if (window_size < 1) return set_err(BNPK_E_WINDOW, "window_size must be positive");
    if (int rc = check_common(enc_mode, lut256, k, window_size)) return rc;
    if (n_bins < 1) return set_err(BNPK_E_BINS, "n_bins must be positive");
    if (hist_mode == BNPK_HIST_SMEM && n_bins > kSmemMaxBins) return set_err(BNPK_E_BINS, "too many bins for the shared-memory histogram");
    if (n_rows == 0) return 0;
    RowArgs a{};
    a.base = base; a.base_bytes = base_bytes; a.starts = starts; a.lens = lens; a.n_rows = n_rows; a.lut = lut256;
    a.k = k; a.window = window_size; a.n_bins = (uint64_t)n_bins; a.hist = (unsigned long long *)hist; a.status = status;
    a.canon_xor = canon_pattern(complement_xor);
    cudaStream_t st = (cudaStream_t)stream;
    return use_smem_hist(n_bins, hist_mode) ? launch_rows_enc<RM_COUNT_MIN, true, false>(a, enc_mode, n_rows, st)
                                            : launch_rows_enc<RM_COUNT_MIN, false, false>(a, enc_mode, n_rows, st);
}

int bnpk_rows_reverse_complement(const uint8_t *base, size_t base_bytes, const int64_t *starts, const int32_t *lens,
                                 size_t n_rows, const uint8_t *lut256, const int64_t *offsets, uint8_t *out, void *stream) {
    (void)base_bytes;
    if (!lut256) return set_err(BNPK_E_BADARG, "lut256 required");
    if (n_rows == 0) return 0;
    const size_t want = (n_rows + 7) / 8;
    const unsigned grid = (unsigned)std::max<size_t>(1, std::min<size_t>(want, (size_t)sm_count() * 8));
    rows_reverse_complement_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(base, starts, lens, n_rows, lut256, offsets, out);
    BNPK_LAUNCHED("rows_reverse_complement_kernel");
    return 0;
}

}  // extern "C"
