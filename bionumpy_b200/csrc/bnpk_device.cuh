// bnpk_device.cuh -- shared device helpers for the sm_100a k-mer hot path.
//
// Data model (see DESIGN.md):
//   every 16-byte unit of the raw chunk is turned, in registers, into
//     codes32 : 2 bits per byte  (byte j of the unit at bits 2j)  -> a contiguous 2-bit stream
//     flags32 : low 16 bits = "byte is '\n'", high 16 bits = "byte is a valid base"
//   and only those 8 bytes per unit are kept in shared memory.  A k-mer starting at byte b is
//   the 2k-bit field at bit 2b of the packed stream (first base in the lowest bits), which is
//   exactly the reference hash sum_j code[i+j]*4^j (sequence/kmers.py:105-126).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include "../../include/bnpk.h"

namespace bnpk {

constexpr int kTileBytes = 16384;          // bytes owned by one tile
constexpr int kHaloBytes = 2048;           // extra bytes staged so in-tile rows can finish
constexpr int kTileThreads = 512;
constexpr int kTileWarps = kTileThreads / 32;
constexpr int kTileUnits = kTileBytes / 16;                  // 1024
constexpr int kStagedUnits = (kTileBytes + kHaloBytes) / 16; // 1152
constexpr int kRowCap = 512;               // rows of one tile kept in shared memory (more: deferred)
constexpr int kSmemMaxBins = 32768;        // u32 bins that fit next to the tile staging

constexpr uint64_t kFlagAgg = 1ull << 62;
constexpr uint64_t kFlagPrefix = 2ull << 62;
constexpr uint64_t kValueMask = (1ull << 62) - 1;

// workspace header (uint64 words)
constexpr int kWsTicket = 0;        // per-launch tile ticket
constexpr int kWsDeferred = 1;      // number of deferred (long) rows
constexpr int kWsLines = 3;         // ws kernels: newlines of the whole chunk (resolve pass)
// ws kernels: labels as tile-major keys until the resolve pass turns them into entry indices (words 4..11 hold the
// development stage clocks, BNPK_WS_DEBUG).  key = tile << 14 | entry of the tile (the entry index counted from the
// tile's first line: at most (3 + 16383 + 1) >> 1 < 2^14); BAD_BASE's key = tile << 24 | entry << 10 | position in
// the row (rows counted in the tile are at most 1024 bytes).  Keys ordered by tile are ordered by line, so min / max
// over keys pick the same record as over entry indices.
constexpr int kWsKeyHeader = 12;    // min key of a bad header line (all ones: none)
constexpr int kWsKeyPlus = 13;      // min key of a bad '+' line (all ones: none)
constexpr int kWsKeyBase = 14;      // min BAD_BASE key (all ones: none)
constexpr int kWsKeyLastRow = 15;   // 1 + max key of a tile's last counted row (0: none)
constexpr int kWsHeaderWords = 16;
constexpr int kKeyEntryBits = 14, kKeyPosBits = 10;
// deferred-row entries of the ws kernels hold a key; this bit marks a row the resolve pass deferred from a tile whose
// record phase was not fixed locally (it counts as a long row only if the in-tile walk would have deferred it too)
constexpr uint64_t kDeferredResolved = 1ull << 62;
// ws kernels: per-tile word in tile_state[] = newlines of the tile | record phase guessed from its bytes << 16 |
// kTileWordAmbiguous when no single phase was left (a tile has at most 16384 newlines: 15 bits)
constexpr int kTileWordPhaseShift = 16;
constexpr uint64_t kTileWordAmbiguous = 1ull << 18;
constexpr int kWsSlotBytes = kTileBytes + 512;   // ws kernels: tile + halo staged per ring slot
constexpr int kWsRowMax = 1024;                  // ws kernels: longer rows take the deferred pass

__device__ __forceinline__ uint64_t ld_relaxed(const uint64_t *p) {
    uint64_t v;
    asm volatile("ld.relaxed.gpu.global.u64 %0, [%1];" : "=l"(v) : "l"(p) : "memory");
    return v;
}
__device__ __forceinline__ void st_relaxed(uint64_t *p, uint64_t v) {
    asm volatile("st.relaxed.gpu.global.u64 [%0], %1;" ::"l"(p), "l"(v) : "memory");
}
// streaming 16-byte load: read-only path, do not keep in L1
__device__ __forceinline__ uint4 ld_stream(const uint4 *p) {
    uint4 r;
    asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
                 : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}

__device__ __forceinline__ uint32_t warp_sum_u32(uint32_t v) {
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}
__device__ __forceinline__ uint64_t warp_sum_u64(uint64_t v) {
#pragma unroll
    for (int o = 16; o; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
    return v;
}

// Decoupled look-back (single-pass chained scan).  Called by one full warp.  Publishes this
// tile's aggregate, walks back over predecessors until an inclusive prefix is found, publishes
// the tile's inclusive prefix and returns the exclusive one.  Tiles are handed out in
// increasing order by an atomic ticket, so every predecessor is already running (or done).
// The walk keeps kLookbackDepth windows of 32 predecessors in flight per round trip.
constexpr int kLookbackDepth = 4;
__device__ __forceinline__ uint64_t lookback_exclusive(uint64_t *state, int64_t tile, uint64_t aggregate, int lane) {
    if (tile == 0) {
        if (lane == 0) st_relaxed(state, kFlagPrefix | aggregate);
        return 0;
    }
    if (lane == 0) st_relaxed(state + tile, kFlagAgg | aggregate);
    uint64_t excl = 0;
    int64_t idx = tile - 1;
    while (true) {
        uint64_t s[kLookbackDepth];
        bool pending;
        do {
            pending = false;
#pragma unroll
            for (int d = 0; d < kLookbackDepth; ++d) {
                const int64_t j = idx - 32 * d - lane;
                s[d] = (j >= 0) ? ld_relaxed(state + j) : kFlagPrefix;
            }
            // only entries up to the first inclusive prefix matter
            bool need = true;
#pragma unroll
            for (int d = 0; d < kLookbackDepth; ++d) {
                const unsigned zero = __ballot_sync(0xffffffffu, (s[d] >> 62) == 0);
                const unsigned pref = __ballot_sync(0xffffffffu, (s[d] >> 62) == 2);
                if (need) {
                    // a not-yet-published entry before the first prefix of this window?
                    const unsigned before = pref ? ((pref & (0u - pref)) - 1u) : 0xffffffffu;   // lanes closer than the first prefix
                    if (zero & before) pending = true;
                    if (pref) need = false;
                }
            }
        } while (pending);
        bool done = false;
#pragma unroll
        for (int d = 0; d < kLookbackDepth; ++d) {
            if (!done) {
                const unsigned pmask = __ballot_sync(0xffffffffu, (s[d] >> 62) == 2);
                uint64_t v = s[d] & kValueMask;
                if (pmask) {
                    const int first = __ffs(pmask) - 1;
                    if (lane > first) v = 0;
                    done = true;
                }
                excl += warp_sum_u64(v);
            }
        }
        if (done) break;
        idx -= 32 * kLookbackDepth;
    }
    if (lane == 0) st_relaxed(state + tile, kFlagPrefix | ((excl + aggregate) & kValueMask));
    return excl;
}

// ---------------------------------------------------------------------------------------------
// byte -> code / flag transforms, four bytes at a time
// ---------------------------------------------------------------------------------------------
// gather bit 0 of each byte into a nibble (bits 0..3)
__device__ __forceinline__ uint32_t bytes_lsb_to_nibble(uint32_t m01) {
    return ((m01 & 0x01010101u) * 0x00204081u >> 21) & 0xFu;
}
// gather the low 2 bits of each byte into 8 bits
__device__ __forceinline__ uint32_t bytes_2bit_to_byte(uint32_t x03) {
    return (x03 * 0x01041040u) >> 24;
}

template <int ENC>
__device__ __forceinline__ void encode_word(uint32_t w, const uint8_t *s_lut, uint32_t &code8, uint32_t &valid4) {
    if constexpr (ENC == BNPK_ENC_ASCII_ACGT || ENC == BNPK_ENC_ASCII_ACTG) {
        uint32_t x;
        if constexpr (ENC == BNPK_ENC_ASCII_ACGT)
            x = ((w >> 1) ^ (w >> 2)) & 0x03030303u;  // A0 C1 G2 T3
        else
            x = (w >> 1) & 0x03030303u;                // A0 C1 T2 G3
        code8 = bytes_2bit_to_byte(x);
        const uint32_t u = w | 0x20202020u;            // fold case (alphabet_encoding.py:24-28)
        const uint32_t eq = __vcmpeq4(u, 0x61616161u) | __vcmpeq4(u, 0x63636363u) |
                            __vcmpeq4(u, 0x67676767u) | __vcmpeq4(u, 0x74747474u);
        valid4 = bytes_lsb_to_nibble(eq);
    } else if constexpr (ENC == BNPK_ENC_CODES) {
        code8 = bytes_2bit_to_byte(w & 0x03030303u);
        valid4 = bytes_lsb_to_nibble(__vcmpeq4(w & 0xFCFCFCFCu, 0u));
    } else {
        uint32_t c = 0, v = 0;
#pragma unroll
        for (int b = 0; b < 4; ++b) {
            const uint32_t code = s_lut[(w >> (8 * b)) & 0xFFu];
            c |= (code & 3u) << (2 * b);
            v |= (code < 4u ? 1u : 0u) << b;
        }
        code8 = c;
        valid4 = v;
    }
}

// one 16-byte unit -> (codes32, flags32)
template <int ENC>
__device__ __forceinline__ void encode_unit(const uint4 q, const uint8_t *s_lut, uint32_t &codes, uint32_t &flags) {
    uint32_t c0, c1, c2, c3, v0, v1, v2, v3;
    encode_word<ENC>(q.x, s_lut, c0, v0);
    encode_word<ENC>(q.y, s_lut, c1, v1);
    encode_word<ENC>(q.z, s_lut, c2, v2);
    encode_word<ENC>(q.w, s_lut, c3, v3);
    codes = c0 | (c1 << 8) | (c2 << 16) | (c3 << 24);
    const uint32_t nl = bytes_lsb_to_nibble(__vcmpeq4(q.x, 0x0A0A0A0Au)) |
                        (bytes_lsb_to_nibble(__vcmpeq4(q.y, 0x0A0A0A0Au)) << 4) |
                        (bytes_lsb_to_nibble(__vcmpeq4(q.z, 0x0A0A0A0Au)) << 8) |
                        (bytes_lsb_to_nibble(__vcmpeq4(q.w, 0x0A0A0A0Au)) << 12);
    flags = nl | ((v0 | (v1 << 4) | (v2 << 8) | (v3 << 12)) << 16);
}

// load a 16-byte unit that may stick out of [0, n): out-of-range bytes read as 0
__device__ __forceinline__ uint4 load_unit_guarded(const uint8_t *base, size_t n, int64_t unit_byte0) {
    if (unit_byte0 >= 0 && (size_t)unit_byte0 + 16 <= n && ((reinterpret_cast<uintptr_t>(base) + unit_byte0) & 15) == 0)
        return ld_stream(reinterpret_cast<const uint4 *>(base + unit_byte0));
    uint32_t w[4] = {0, 0, 0, 0};
#pragma unroll
    for (int b = 0; b < 16; ++b) {
        const int64_t p = unit_byte0 + b;
        if (p >= 0 && (size_t)p < n) w[b >> 2] |= (uint32_t)base[p] << (8 * (b & 3));
    }
    return make_uint4(w[0], w[1], w[2], w[3]);
}

// length of the line starting at global byte `start` (distance to the next '\n'); -1 if the data
// ends first.  Warp-wide.
__device__ __forceinline__ int64_t warp_line_len(const uint8_t *base, size_t n, int64_t start, int lane) {
    const int off = (int)((reinterpret_cast<uintptr_t>(base) + start) & 15);
    int64_t u0 = start - off;
    bool first = true;
    while (u0 < (int64_t)n) {
        const int64_t ub = u0 + 16 * (int64_t)lane;
        uint32_t m = 0;
        if (ub < (int64_t)n) {
            const uint4 q = load_unit_guarded(base, n, ub);
            m = bytes_lsb_to_nibble(__vcmpeq4(q.x, 0x0A0A0A0Au)) | (bytes_lsb_to_nibble(__vcmpeq4(q.y, 0x0A0A0A0Au)) << 4) |
                (bytes_lsb_to_nibble(__vcmpeq4(q.z, 0x0A0A0A0Au)) << 8) | (bytes_lsb_to_nibble(__vcmpeq4(q.w, 0x0A0A0A0Au)) << 12);
            if (first && lane == 0) m &= 0xFFFFu << off;
        }
        const unsigned b = __ballot_sync(0xffffffffu, m != 0);
        if (b) {
            const int src = __ffs(b) - 1;
            const int64_t pos = ub + __ffs(m) - 1;
            return __shfl_sync(0xffffffffu, pos, src) - start;
        }
        first = false;
        u0 += 512;
    }
    return -1;
}

// ---------------------------------------------------------------------------------------------
// packed-stream readers
// ---------------------------------------------------------------------------------------------
// low 32 bits of the 2-bit stream starting at byte `b` (codes[] is the unit array, 32-bit words)
__device__ __forceinline__ uint32_t stream_lo32(const uint32_t *codes, uint32_t b) {
    const uint32_t bit = 2u * b;
    const uint32_t idx = bit >> 5, sh = bit & 31u;
    return __funnelshift_r(codes[idx], codes[idx + 1], sh);
}
// 64 bits of the stream starting at byte `b`
__device__ __forceinline__ uint64_t stream_64(const uint32_t *codes, uint32_t b) {
    const uint32_t bit = 2u * b;
    const uint32_t idx = bit >> 5, sh = bit & 31u;
    const uint32_t w0 = codes[idx], w1 = codes[idx + 1], w2 = codes[idx + 2];
    return ((uint64_t)__funnelshift_r(w1, w2, sh) << 32) | __funnelshift_r(w0, w1, sh);
}

// sliding minimum over `w` consecutive lanes (w <= 32): lane l gets min(v[l .. l+w-1]);
// only lanes l <= 32-w hold a complete window.
__device__ __forceinline__ uint64_t warp_sliding_min(uint64_t v, int w) {
    int span = 1;
    while (span * 2 <= w) {
        const uint64_t o = __shfl_down_sync(0xffffffffu, v, span);
        v = o < v ? o : v;
        span *= 2;
    }
    const int rest = w - span;
    if (rest) {
        const uint64_t o = __shfl_down_sync(0xffffffffu, v, rest);
        v = o < v ? o : v;
    }
    return v;
}

// min(h, hash of the reverse complement of the k-mer): bases reversed (bit reversal + swap inside each pair) and
// complemented.  cx = the complement as an XOR on every 2-bit code (ACGT order: 3 -> all ones, ACTG order: 2).
__device__ __forceinline__ uint64_t canonical_hash(uint64_t h, int k, uint64_t cx) {
    uint64_t x = __brevll(h ^ cx);
    x = ((x & 0x5555555555555555ull) << 1) | ((x >> 1) & 0x5555555555555555ull);
    x >>= (64 - 2 * k);
    return x < h ? x : h;
}

struct HistTarget {
    unsigned long long *global;  // int64 table in HBM/L2
    uint32_t *smem;              // privatised table (or nullptr)
    uint64_t n_bins;
    uint64_t mask;               // n_bins-1 when n_bins is a power of two, else 0
    unsigned long long delta;    // +1, or -1 for the un-count of an incomplete record
    uint64_t canon_xor;          // != 0: count min(h, reverse-complement hash) (see canonical_hash)
};

template <bool SMEM>
__device__ __forceinline__ void hist_add(const HistTarget &t, uint64_t value) {
    const uint64_t b = t.mask ? (value & t.mask) : (value % t.n_bins);
    if constexpr (SMEM)
        atomicAdd(t.smem + (uint32_t)b, 1u);
    else
        atomicAdd(t.global + b, t.delta);
}

// first newline at or after tile-relative byte `from`, below `limit`; -1 if none.  Warp-wide.
__device__ __forceinline__ int find_newline(const uint32_t *s_flags, int from, int limit, int lane) {
    int unit0 = from >> 4;
    const int last_unit = (limit + 15) >> 4;
    for (; unit0 < last_unit; unit0 += 32) {
        const int u = unit0 + lane;
        uint32_t m = (u < last_unit) ? (s_flags[u] & 0xFFFFu) : 0u;
        if (u == (from >> 4)) m &= 0xFFFFu << (from & 15);
        const unsigned b = __ballot_sync(0xffffffffu, m != 0);
        if (b) {
            const int src = __ffs(b) - 1;
            const int pos = (u << 4) + __ffs(m) - 1;
            const int e = __shfl_sync(0xffffffffu, pos, src);
            return e < limit ? e : -1;
        }
    }
    return -1;
}

// first invalid byte in [from, to) (tile-relative), -1 if all valid.  Warp-wide.
__device__ __forceinline__ int find_invalid(const uint32_t *s_flags, int from, int to, int lane) {
    if (to <= from) return -1;
    int unit0 = from >> 4;
    const int last_unit = (to + 15) >> 4;
    for (; unit0 < last_unit; unit0 += 32) {
        const int u = unit0 + lane;
        uint32_t bad = 0;
        if (u < last_unit) {
            bad = (~(s_flags[u] >> 16)) & 0xFFFFu;
            if (u == (from >> 4)) bad &= 0xFFFFu << (from & 15);
            if (u == ((to - 1) >> 4)) bad &= 0xFFFFu >> (15 - ((to - 1) & 15));
        }
        const unsigned b = __ballot_sync(0xffffffffu, bad != 0);
        if (b) {
            const int src = __ffs(b) - 1;
            const int pos = (u << 4) + __ffs(bad) - 1;
            return __shfl_sync(0xffffffffu, pos, src);
        }
    }
    return -1;
}

// k-mers / minimizers of one staged row -> histogram.  Warp-wide.  Returns values counted by
// this lane.  `b0` = tile-relative byte of the row's first base, L = row length.
template <bool SMEM_HIST, bool MINIMIZER>
__device__ __forceinline__ uint32_t row_count(const uint32_t *s_codes, int b0, int L, int k, int window,
                                              const HistTarget &ht, int lane) {
    uint32_t produced = 0;
    const uint64_t kmask = (k == 32) ? ~0ull : ((1ull << (2 * k)) - 1);
    if constexpr (!MINIMIZER) {
        const int npos = L - k + 1;
        // fast path: the bin index only needs the low 32 bits of the window
        if (ht.mask && ht.mask <= 0xFFFFFFFFull && !ht.canon_xor) {
            const uint32_t m32 = (uint32_t)(ht.mask & kmask);
            for (int i = lane; i < npos; i += 32) {
                const uint32_t lo = stream_lo32(s_codes, (uint32_t)(b0 + i)) & m32;
                if constexpr (SMEM_HIST) atomicAdd(ht.smem + lo, 1u);
                else atomicAdd(ht.global + lo, ht.delta);
                ++produced;
            }
        } else {
            for (int i = lane; i < npos; i += 32) {
                uint64_t h = stream_64(s_codes, (uint32_t)(b0 + i)) & kmask;
                if (ht.canon_xor) h = canonical_hash(h, k, ht.canon_xor);
                hist_add<SMEM_HIST>(ht, h);
                ++produced;
            }
        }
    } else {
        // canon_xor != 0: canonical minimizers, the minimum of the canonical hashes of the window
        const int w = window - k + 1;           // k-mers per window (minimizers.py:52)
        const int nout = L - window + 1;        // windows in the row
        const int nh = L - k + 1;               // hashes in the row
        if (w <= 32) {
            const int step = 32 - (w - 1);
            for (int base = 0; base < nout; base += step) {
                const int p = base + lane;
                uint64_t h = ~0ull;             // lanes past the last hash keep the sentinel
                if (p < nh) {
                    h = stream_64(s_codes, (uint32_t)(b0 + p)) & kmask;
                    if (ht.canon_xor) h = canonical_hash(h, k, ht.canon_xor);
                }
                const uint64_t m = warp_sliding_min(h, w);
                if (lane < step && p < nout) { hist_add<SMEM_HIST>(ht, m); ++produced; }
            }
        } else {
            for (int j = lane; j < nout; j += 32) {
                uint64_t m = ~0ull;
                for (int i = 0; i < w; ++i) {
                    uint64_t h = stream_64(s_codes, (uint32_t)(b0 + j + i)) & kmask;
                    if (ht.canon_xor) h = canonical_hash(h, k, ht.canon_xor);
                    m = h < m ? h : m;
                }
                hist_add<SMEM_HIST>(ht, m);
                ++produced;
            }
        }
    }
    return produced;
}

}  // namespace bnpk
