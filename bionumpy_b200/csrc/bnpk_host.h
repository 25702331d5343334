// bnpk_host.h -- host-side glue shared by the translation units of libbnpk.so
#pragma once
#include <algorithm>
#include <atomic>
#include <cstdio>
#include <cstring>
#include "bnpk_device.cuh"

namespace bnpk {

extern std::atomic<uint64_t> g_launches;
int set_err(int code, const char *msg);
int cuda_fail(cudaError_t e, const char *what);
int sm_count();
// cudaFuncAttributeMaxDynamicSharedMemorySize is a per-device attribute: set it once per (kernel, device)
int ensure_dyn_smem(const void *kernel, int bytes);
#define BNPK_DYN_SMEM(kern, bytes)                                            \
    do {                                                                      \
        int rc__ = ::bnpk::ensure_dyn_smem((const void *)(kern), (int)(bytes)); \
        if (rc__) return rc__;                                                \
    } while (0)

#define BNPK_CUDA(expr)                                             \
    do {                                                            \
        cudaError_t e__ = (expr);                                   \
        if (e__ != cudaSuccess) return ::bnpk::cuda_fail(e__, #expr); \
    } while (0)

#define BNPK_LAUNCHED(name)                                         \
    do {                                                            \
        ::bnpk::g_launches.fetch_add(1, std::memory_order_relaxed); \
        cudaError_t e__ = cudaGetLastError();                       \
        if (e__ != cudaSuccess) return ::bnpk::cuda_fail(e__, name); \
    } while (0)

// optional per-launch timing of the dominant (tile) kernel, see bnpk_profile_* in bnpk.h
void profile_before(cudaStream_t st);
void profile_after(cudaStream_t st);

size_t tile_workspace_bytes(size_t n);
bool use_smem_hist(int64_t n_bins, int hist_mode);

// the complement of a 2-bit code as an XOR pattern over a whole hash (complement_xor 1..3, see canonical_hash)
inline uint64_t canon_pattern(int complement_xor) {
    return complement_xor == 3 ? ~0ull : complement_xor == 2 ? 0xAAAAAAAAAAAAAAAAull : 0x5555555555555555ull;
}

// canon_xor != 0: count canonical k-mers (window 0) or canonical minimizers (window > 0)
int chunk_kmer_count_impl(const uint8_t *chunk, size_t n, size_t slice_begin, size_t slice_end, int final_slice,
                          int lpe, uint8_t header_char, int check_plus, int trim_cr, int enc_mode,
                          const uint8_t *lut256, int k, int window, int64_t n_bins, int hist_mode, int64_t *hist,
                          int64_t *status, void *workspace, size_t workspace_bytes, cudaStream_t st,
                          uint64_t canon_xor = 0);

int line_split_impl(const uint8_t *chunk, size_t n, int lpe, int field_line, int start_offset, uint8_t header_char,
                    int check_plus, int trim_cr, int64_t *starts, int32_t *lens, size_t max_rows, int64_t *status,
                    void *workspace, size_t workspace_bytes, cudaStream_t st);

// after the last slice of a fused count: long (deferred) rows + un-count of the sequence line
// of a trailing incomplete entry
int count_fixups_impl(const uint8_t *chunk, size_t n, int lpe, int enc_mode, const uint8_t *lut256, int k,
                      int window, int64_t n_bins, int64_t *hist, int64_t *status, const uint64_t *deferred_count,
                      const uint64_t *deferred, size_t deferred_cap, cudaStream_t st, uint64_t canon_xor = 0);

}  // namespace bnpk
