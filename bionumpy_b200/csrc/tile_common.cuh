// tile_common.cuh -- pieces shared by the tile kernels (tile_kernels.cu: split + register-staged count;
// tile_tma_kernel.cu: the shared-memory-staged count): launch arguments, exact byte tests, the
// 16-byte unit encoder and the two-level decoupled look-back over the tile newline counts.
#pragma once
#include "bnpk_host.h"

namespace bnpk {

struct TileArgs {
    const uint8_t *chunk;
    size_t n;
    int64_t tile_begin, tile_end;  // tiles handled by this launch
    int lpe, lpe_shift, field_line, start_offset;
    uint32_t header_char;
    int check_plus;
    int64_t *status;
    uint64_t *ws;                  // header | tile_state[] | deferred[]
    int64_t n_tiles_total;
    uint64_t *deferred;            // long-row list (start, entry) pairs
    size_t deferred_cap;
    // split
    int64_t *starts;
    int32_t *lens;
    size_t max_rows;
    // count
    const uint8_t *lut;
    int k, window;                 // window = 0: k-mers; else minimizers over `window` bases
    uint64_t n_bins;
    unsigned long long *hist;
    uint32_t *hist32;              // optional 32-bit scratch table in the workspace (large global tables), else null
    uint64_t canon_xor;            // != 0: canonical k-mers / minimizers, the complement as an XOR pattern (canon_pattern)
};

// 256-bit streaming load (sm_100: LDG.E.256), read-only path, no L1 allocation
__device__ __forceinline__ void ld_stream_256(const uint8_t *p, uint32_t *r) {
    asm volatile("ld.global.nc.L1::no_allocate.v8.u32 {%0,%1,%2,%3,%4,%5,%6,%7}, [%8];"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "l"(p));
}

// exact per-byte "== pattern byte" flags at bit 7 of every byte
__device__ __forceinline__ uint32_t bytes_eq_msb(uint32_t w, uint32_t pattern) {
    const uint32_t v = w ^ pattern;
    return ~(((v & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | v) & 0x80808080u;
}
// bits 7,15,23,31 -> bits 0..3 (one IMAD.HI: the partial products land on distinct bits)
__device__ __forceinline__ uint32_t msb_to_nibble(uint32_t z) { return __umulhi(z, 0x02040810u) & 0xFu; }

// 16 flag bits (one per byte) of four words
__device__ __forceinline__ uint32_t eq_mask16(const uint32_t *w, uint32_t pattern) {
    const uint32_t n0 = msb_to_nibble(bytes_eq_msb(w[0], pattern)), n1 = msb_to_nibble(bytes_eq_msb(w[1], pattern));
    const uint32_t n2 = msb_to_nibble(bytes_eq_msb(w[2], pattern)), n3 = msb_to_nibble(bytes_eq_msb(w[3], pattern));
    return (n1 * 16u + n0) + (n3 * 16u + n2) * 256u;
}
__device__ __forceinline__ uint64_t eq_mask64(const uint32_t *raw, uint32_t pattern) {
    const uint32_t lo = eq_mask16(raw, pattern) | (eq_mask16(raw + 4, pattern) << 16);
    const uint32_t hi = eq_mask16(raw + 8, pattern) | (eq_mask16(raw + 12, pattern) << 16);
    return ((uint64_t)hi << 32) | lo;
}

// One 16-byte unit of sequence bytes -> 32 bits of 2-bit codes; `bad` becomes non-zero iff a byte
// selected by `seq16` is outside the alphabet (exact).
template <int ENC>
__device__ __forceinline__ uint32_t encode_unit_seq(const uint32_t *w, uint32_t seq16, const uint8_t *s_lut, uint32_t &bad) {
    uint32_t codes = 0;
    if constexpr (ENC == BNPK_ENC_ASCII_ACGT || ENC == BNPK_ENC_ASCII_ACTG) {
        uint32_t dif[4];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            uint32_t x;
            if constexpr (ENC == BNPK_ENC_ASCII_ACGT) x = ((w[j] >> 1) ^ (w[j] >> 2)) & 0x03030303u;
            else x = (w[j] >> 1) & 0x03030303u;
            codes |= bytes_2bit_to_byte(x) << (8 * j);
            // re-decode the codes (PRMT as a 4-entry byte LUT) and compare with the case-folded input
            const uint32_t y = x | (x >> 4);
            const uint32_t sel = __byte_perm(y, 0u, 0x4420);       // nibbles = the four codes
            const uint32_t letters = (ENC == BNPK_ENC_ASCII_ACGT) ? 0x74676361u : 0x67746361u;  // "acgt" / "actg"
            dif[j] = __byte_perm(letters, 0u, sel) ^ (w[j] | 0x20202020u);
        }
        if (seq16 == 0xFFFFu) {
            bad = dif[0] | dif[1] | dif[2] | dif[3];
        } else {
            bad = 0;
#pragma unroll
            for (int j = 0; j < 4; ++j) {
                const uint32_t nz = (((dif[j] & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | dif[j]) & 0x80808080u;  // byte != 0
                bad |= msb_to_nibble(nz) & (seq16 >> (4 * j)) & 0xFu;
            }
        }
    } else if constexpr (ENC == BNPK_ENC_CODES) {
        bad = 0;
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            codes |= bytes_2bit_to_byte(w[j] & 0x03030303u) << (8 * j);
            const uint32_t hi = w[j] & 0xFCFCFCFCu;
            const uint32_t nz = (((hi & 0x7F7F7F7Fu) + 0x7F7F7F7Fu) | hi) & 0x80808080u;
            bad |= msb_to_nibble(nz) & (seq16 >> (4 * j)) & 0xFu;
        }
    } else {
        bad = 0;
#pragma unroll
        for (int b = 0; b < 16; ++b) {
            const uint32_t code = s_lut[(w[b >> 2] >> (8 * (b & 3))) & 0xFFu];
            codes |= (code & 3u) << (2 * b);
            bad |= ((code >= 4u) ? 1u : 0u) & (seq16 >> b);
        }
    }
    return codes;
}

// ---- two-level look-back state in the workspace ------------------------------------------------
//   tile_state[t]  : flag|value, AGG = newlines of tile t, PREFIX = newlines of tiles 0..t
//   block_cnt[b]   : atomic (count << 56 | sum) over the 32 tiles of block b
//   block_state[b] : flag|value, AGG = newlines of the whole block, PREFIX = newlines of tiles 0..32b+31
// A tile resolves its exclusive prefix from <= 31 tile entries of its own block plus <= 32 block
// entries: two loads per lane, issued one pipeline stage before they are needed.
struct LookbackArrays {
    uint64_t *tile_state, *block_cnt, *block_state;
};
__device__ __forceinline__ LookbackArrays lookback_arrays(uint64_t *ws, int64_t n_tiles_total) {
    LookbackArrays l;
    l.tile_state = ws + kWsHeaderWords;
    const int64_t nb = (n_tiles_total >> 5) + 2;
    l.block_cnt = l.tile_state + n_tiles_total + 1;
    l.block_state = l.block_cnt + nb;
    return l;
}
__device__ __forceinline__ void lookback_publish(const LookbackArrays &l, int64_t tile, uint64_t agg) {
    st_relaxed(l.tile_state + tile, (tile == 0 ? kFlagPrefix : kFlagAgg) | agg);
    const int64_t b = tile >> 5;
    const unsigned long long old = atomicAdd((unsigned long long *)(l.block_cnt + b), (1ull << 56) | agg);
    if ((old >> 56) == 31ull)
        atomicMax((unsigned long long *)(l.block_state + b), kFlagAgg | ((old & ((1ull << 56) - 1)) + agg));
}
__device__ __forceinline__ void lookback_issue(const LookbackArrays &l, int64_t tile, int lane, uint64_t &lbA, uint64_t &lbB) {
    const int i = (int)(tile & 31);
    const int64_t b = tile >> 5;
    lbA = (lane < i) ? ld_relaxed(l.tile_state + tile - 1 - lane) : kFlagPrefix;
    lbB = (b - 1 - lane >= 0) ? ld_relaxed(l.block_state + (b - 1 - lane)) : kFlagPrefix;
}
// Warp-wide.  Returns the exclusive prefix of `tile` and publishes its inclusive prefix.
__device__ __forceinline__ uint64_t lookback_finish(const LookbackArrays &l, int64_t tile, uint64_t agg, int lane,
                                                    uint64_t lbA, uint64_t lbB) {
    const int i = (int)(tile & 31);
    int64_t b = tile >> 5;
    uint64_t excl = 0;
    bool have = false;
    // ---- my own block: tiles 32b .. tile-1 (lane 0 = tile-1).  Wait (a short loop: the waiting warp shares its
    // issue slots with the warps it waits for) until every earlier tile of the block has published something.
    {
        const bool valid = lane < i;
        while (__any_sync(0xffffffffu, valid && (lbA >> 62) == 0))
            if (valid && (lbA >> 62) == 0) lbA = ld_relaxed(l.tile_state + tile - 1 - lane);
        const unsigned pref = __ballot_sync(0xffffffffu, valid && (lbA >> 62) == 2);
        const unsigned upto = pref ? ((pref & (0u - pref)) << 1) - 1u : 0xffffffffu;     // lanes 0..first prefix
        const uint64_t v = (valid && ((1u << lane) & upto)) ? (lbA & kValueMask) : 0;
        excl = warp_sum_u64(v);
        have = pref != 0;
    }
    // ---- whole blocks before mine (lane 0 = block b-1)
    int64_t bb = b;
    while (!have) {
        const unsigned pref = __ballot_sync(0xffffffffu, (lbB >> 62) == 2);
        const unsigned zero = __ballot_sync(0xffffffffu, (lbB >> 62) == 0);
        const unsigned upto = pref ? ((pref & (0u - pref)) << 1) - 1u : 0xffffffffu;
        if (zero & upto) {
            lbB = (bb - 1 - lane >= 0) ? ld_relaxed(l.block_state + (bb - 1 - lane)) : kFlagPrefix;
            continue;
        }
        const uint64_t v = ((1u << lane) & upto) ? (lbB & kValueMask) : 0;
        excl += warp_sum_u64(v);
        if (pref) break;
        bb -= 32;                                            // more than 32 blocks back (cold start only)
        lbB = (bb - 1 - lane >= 0) ? ld_relaxed(l.block_state + (bb - 1 - lane)) : kFlagPrefix;
    }
    if (lane == 0) {
        const uint64_t incl = (excl + agg) & kValueMask;
        st_relaxed(l.tile_state + tile, kFlagPrefix | incl);
        if (i == 31) atomicMax((unsigned long long *)(l.block_state + b), kFlagPrefix | incl);
    }
    return excl;
}


// the shared-memory-staged fused count (tile_tma_kernel.cu).  Returns -1 when the launch does not
// qualify (minimizers, unaligned chunk, too many bins for its table) and the caller must fall back.
bool tma_count_eligible(const TileArgs &a, bool smem_hist);
constexpr int64_t kScratch32MaxBins = 1ll << 24;   // 64 MiB of u32 counters at the end of the workspace
int launch_tma_count(const TileArgs &a, int enc_mode, bool smem_hist, cudaStream_t st);
// the warp-specialised fused count (tile_ws_kernel.cu): same eligibility, the default
int launch_ws_count(const TileArgs &a, int enc_mode, bool smem_hist, cudaStream_t st);
bool wsm_count_eligible(const TileArgs &a, bool smem_hist);
int launch_wsm_count(const TileArgs &a, int enc_mode, bool smem_hist, cudaStream_t st);
bool wsc_count_eligible(const TileArgs &a, bool smem_hist);
int launch_wsc_count(const TileArgs &a, int enc_mode, bool smem_hist, cudaStream_t st);
int launch_wsmc_count(const TileArgs &a, int enc_mode, bool smem_hist, cudaStream_t st);   // canonical minimizers, wsm_count_eligible
// after the last launch of a chunk through one of the ws builds: line prefix, phase check, keys -> entry indices
int ws_resolve(const TileArgs &a, cudaStream_t st);

}  // namespace bnpk
