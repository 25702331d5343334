// tile_ws_kernel.cu -- the four builds of the warp-specialised fused count (tile_ws_kernel.inl)
#include "tile_common.cuh"

// k-mer counts: the dominant kernel of the hot path
#define BNPK_WS_NAMESPACE ws
#define BNPK_WS_NS 8
#define BNPK_WS_SG 2
#define BNPK_WS_RW 8
#define BNPK_WS_MINZ 0
#define BNPK_WS_CANON 0
#define BNPK_WS_LAUNCH launch_ws_count
#include "tile_ws_kernel.inl"
#undef BNPK_WS_NAMESPACE
#undef BNPK_WS_NS
#undef BNPK_WS_SG
#undef BNPK_WS_RW
#undef BNPK_WS_MINZ
#undef BNPK_WS_CANON
#undef BNPK_WS_LAUNCH

// minimizer counts (windows of up to 12 k-mers, CTA-private table)
#define BNPK_WS_NAMESPACE wsm
#define BNPK_WS_NS 4       // the slots are held for the front end and the encoding only (rows are staged), see kStageU
#define BNPK_WS_SG 1       // the row warps bound this build: one scan group is enough, and sixteen row warps (80 registers
#define BNPK_WS_RW 16      // per thread, no spills; 8 -> 12 -> 16 row warps: 5.5 -> 4.45 -> 3.98 ms)
#define BNPK_WS_MINZ 1
#define BNPK_WS_CANON 0
#define BNPK_WS_LAUNCH launch_wsm_count
#include "tile_ws_kernel.inl"
#undef BNPK_WS_NAMESPACE
#undef BNPK_WS_NS
#undef BNPK_WS_SG
#undef BNPK_WS_RW
#undef BNPK_WS_MINZ
#undef BNPK_WS_CANON
#undef BNPK_WS_LAUNCH

// canonical k-mer counts (min of a k-mer and its reverse complement), CTA-private table; the ring of the k-mer build
#define BNPK_WS_NAMESPACE wsc
#define BNPK_WS_NS 8
#define BNPK_WS_SG 2
#define BNPK_WS_RW 8
#define BNPK_WS_MINZ 0
#define BNPK_WS_CANON 1
#define BNPK_WS_LAUNCH launch_wsc_count
#include "tile_ws_kernel.inl"
#undef BNPK_WS_NAMESPACE
#undef BNPK_WS_NS
#undef BNPK_WS_SG
#undef BNPK_WS_RW
#undef BNPK_WS_MINZ
#undef BNPK_WS_CANON
#undef BNPK_WS_LAUNCH

// canonical minimizer counts (the minimum of min(k-mer, reverse complement) over each window); the ring, geometry and
// staging of the minimizer build
#define BNPK_WS_NAMESPACE wsmc
#define BNPK_WS_NS 4
#define BNPK_WS_SG 1
#define BNPK_WS_RW 14      // the reverse-complement words do not fit 80 registers (16 row warps: spills); 20 warps: 96, no stack
#define BNPK_WS_MINZ 1
#define BNPK_WS_CANON 1
#define BNPK_WS_LAUNCH launch_wsmc_count
#include "tile_ws_kernel.inl"

namespace bnpk {
// minimizer counts the wsm build (and, canonical, the wsmc build) takes: CTA-private table, windows of at most kMinzW
// k-mers; the rest (and global tables) stay with the register-staged kernel
bool wsm_count_eligible(const TileArgs &a, bool smem_hist) {
    if (a.window == 0 || !smem_hist || a.n_bins > (uint64_t)wsm::kMaxBins) return false;
    if (a.window - a.k + 1 > wsm::kMinzW) return false;
    if ((reinterpret_cast<uintptr_t>(a.chunk) & 15) != 0) return false;
    if (a.tile_end > 0x7FFFFFF0ll || a.n < 16) return false;
    return true;
}

// canonical k-mer counts (chunk_kmer_count_impl admits them without a window only) the wsc build takes: CTA-private
// table of at most 2^14 bins, 16-byte-aligned chunk; the rest (global tables, 2^15 bins, unaligned chunks) stay with
// the register-staged kernel
bool wsc_count_eligible(const TileArgs &a, bool smem_hist) {
    if (!smem_hist || a.n_bins > (uint64_t)wsc::kMaxBins) return false;
    if ((reinterpret_cast<uintptr_t>(a.chunk) & 15) != 0) return false;
    if (a.tile_end > 0x7FFFFFF0ll || a.n < 16) return false;
    return true;
}
}  // namespace bnpk

// ---- resolve pass: after the last launch of a chunk through the ws / wsm / wsc / wsmc builds -----------------------------
// The kernel labels entries by tile-major keys and fixes each tile's record phase from the tile's own bytes.  Here the
// tiles' newline counts are scanned (two-level: sums of 1024 tiles, then one block per 1024 tiles), every guessed phase
// is checked against the line prefix (a wrong guess means the true phase breaks a line rule inside that tile: malformed
// input, BNPK_ST_OVERFLOW), the tiles whose phase was left open are walked with the true phase (entry checks; their
// rows join the deferred list), and the keys become the entry indices of the status words and deferred rows.
namespace bnpk {
namespace {
constexpr int kResolveTiles = 1024;                    // tiles per block of the scan (one per thread)
constexpr uint64_t kKeyEntryMask = (1ull << kKeyEntryBits) - 1;

__device__ __forceinline__ uint64_t block_sum_1024(uint64_t v, uint64_t *s_part) {
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    v = warp_sum_u64(v);
    if (lane == 0) s_part[warp] = v;
    __syncthreads();
    uint64_t t = lane < (int)(blockDim.x >> 5) ? s_part[lane] : 0ull;
    t = warp_sum_u64(t);
    __syncthreads();
    return t;
}

__global__ void __launch_bounds__(kResolveTiles) ws_resolve_sum_kernel(const TileArgs a) {
    __shared__ uint64_t s_part[32];
    const int64_t t = (int64_t)blockIdx.x * kResolveTiles + threadIdx.x;
    const uint64_t *tile_state = a.ws + kWsHeaderWords;
    const uint64_t c = t < a.n_tiles_total ? (tile_state[t] & 0xFFFFull) : 0ull;
    const uint64_t s = block_sum_1024(c, s_part);
    if (threadIdx.x == 0) a.ws[kWsHeaderWords + a.n_tiles_total + 1 + blockIdx.x] = s;   // block_cnt[] of the workspace
}

// One warp walks a tile whose phase the kernel left open, now that its first line index `excl` is known: the entry
// checks of tile_head_checks and the row walk for every newline of the tile, and its sequence rows go to the deferred
// list (marked, so that rows_kernel counts as long only the rows the in-tile walk would have deferred).
__device__ void walk_open_tile(const TileArgs &a, int64_t tile, uint64_t excl, uint32_t count, int lane) {
    const uint32_t ls = (uint32_t)a.lpe_shift, pm = (1u << ls) - 1u, ph = (uint32_t)excl & pm;
    const size_t byte0 = (size_t)tile * kTileBytes, end = min(byte0 + (size_t)kTileBytes, a.n);
    const uint64_t key0 = (uint64_t)tile << kKeyEntryBits;
    unsigned long long complete = 0;
    uint32_t seen = 0;                                              // newlines of the tile before this stretch
    for (size_t off = byte0; off < end && seen < count; off += 512) {
        const size_t ub = off + 16 * (size_t)lane;
        uint32_t m = 0;
        for (int b = 0; b < 16; ++b)
            if (ub + b < end && a.chunk[ub + b] == '\n') m |= 1u << b;
        const uint32_t cnt = (uint32_t)__popc(m);
        uint32_t inc = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t v = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += v;
        }
        uint32_t j = seen + inc - cnt;
        while (m) {
            const int bit = __ffs((int)m) - 1;
            m &= m - 1;
            const size_t P = ub + (size_t)bit;
            const uint32_t line = ph + j + 1u, role = line & pm;       // the line after newline j of the tile
            const uint64_t key = key0 + (line >> ls);
            if (P + 1 < a.n) {
                const uint32_t c = a.chunk[P + 1];
                if (role == 0u && c != a.header_char) atomicMin((unsigned long long *)(a.ws + kWsKeyHeader), key);
                if (role == 2u && a.check_plus && c != '+') atomicMin((unsigned long long *)(a.ws + kWsKeyPlus), key);
                if (role == 1u) {
                    const unsigned long long d = atomicAdd((unsigned long long *)(a.ws + kWsDeferred), 1ull);
                    if (d < a.deferred_cap) {
                        a.deferred[2 * d] = P + 1;
                        a.deferred[2 * d + 1] = key | kDeferredResolved;
                    } else {
                        a.status[BNPK_ST_OVERFLOW] = 1;
                    }
                }
            }
            if (role == 0u) complete = max(complete, (unsigned long long)(P + 1));   // the newline that ends an entry
            ++j;
        }
        seen += __shfl_sync(0xffffffffu, inc, 31);
    }
#pragma unroll
    for (int o = 16; o; o >>= 1) complete = max(complete, __shfl_xor_sync(0xffffffffu, complete, o));
    if (lane == 0 && complete) atomicMax((unsigned long long *)&a.status[BNPK_ST_N_COMPLETE_BYTES], complete);
}

__global__ void __launch_bounds__(kResolveTiles) ws_resolve_tiles_kernel(const TileArgs a) {
    __shared__ uint64_t s_part[32], s_excl[kResolveTiles];
    __shared__ uint32_t s_open[kResolveTiles], s_n_open;
    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    uint64_t *tile_state = a.ws + kWsHeaderWords;
    const uint64_t *block_sums = tile_state + a.n_tiles_total + 1;
    if (tid == 0) s_n_open = 0;
    uint64_t before = 0;                                           // newlines of the blocks before this one
    for (uint32_t b = tid; b < blockIdx.x; b += kResolveTiles) before += block_sums[b];
    before = block_sum_1024(before, s_part);
    const int64_t t = (int64_t)blockIdx.x * kResolveTiles + tid;
    const uint64_t w = t < a.n_tiles_total ? tile_state[t] : 0ull;
    const uint64_t c = w & 0xFFFFull;
    // exclusive scan of the block's counts
    uint64_t inc = c;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const uint64_t v = __shfl_up_sync(0xffffffffu, inc, o);
        if (lane >= o) inc += v;
    }
    if (lane == 31) s_part[warp] = inc;
    __syncthreads();
    if (warp == 0) {
        uint64_t x = s_part[lane];
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint64_t v = __shfl_up_sync(0xffffffffu, x, o);
            if (lane >= o) x += v;
        }
        s_part[lane] = x;                                          // inclusive over the warps
    }
    __syncthreads();
    const uint64_t excl = before + (warp ? s_part[warp - 1] : 0ull) + inc - c;
    if (t < a.n_tiles_total) {
        const uint32_t pm = (1u << a.lpe_shift) - 1u;
        if (w & kTileWordAmbiguous) {
            if (c) {
                const uint32_t i = atomicAdd(&s_n_open, 1u);
                s_open[i] = (uint32_t)c << 10 | (uint32_t)tid;
            }
        } else if (((uint32_t)(w >> kTileWordPhaseShift) & 3u) != ((uint32_t)excl & pm)) {
            a.status[BNPK_ST_OVERFLOW] = 1;                        // the bytes of this tile break a line rule
        }
        s_excl[tid] = excl;
        if (t == a.n_tiles_total - 1) a.ws[kWsLines] = excl + c;
    }
    __syncthreads();
    if (t < a.n_tiles_total) tile_state[t] = excl;                 // for the labels pass
    for (uint32_t i = (uint32_t)warp; i < s_n_open; i += kResolveTiles / 32) {
        const uint32_t k = s_open[i] & (kResolveTiles - 1);
        walk_open_tile(a, (int64_t)blockIdx.x * kResolveTiles + k, s_excl[k], s_open[i] >> 10, lane);
    }
}

// keys -> entry indices: the status words (one thread) and every deferred row
__global__ void ws_resolve_labels_kernel(const TileArgs a) {
    const uint64_t *prefix = a.ws + kWsHeaderWords;                // exclusive line prefix of every tile
    const uint32_t ls = (uint32_t)a.lpe_shift;
    auto entry = [&](uint64_t key) -> uint64_t { return (prefix[key >> kKeyEntryBits] >> ls) + (key & kKeyEntryMask); };
    if (blockIdx.x == 0 && threadIdx.x == 0) {
        a.status[BNPK_ST_N_LINES] = (int64_t)a.ws[kWsLines];
        const uint64_t kh = a.ws[kWsKeyHeader], kp = a.ws[kWsKeyPlus], kb = a.ws[kWsKeyBase], kl = a.ws[kWsKeyLastRow];
        if (kh != ~0ull) atomicMin((long long *)&a.status[BNPK_ST_BAD_HEADER_ENTRY], (long long)entry(kh));
        if (kp != ~0ull) atomicMin((long long *)&a.status[BNPK_ST_BAD_PLUS_ENTRY], (long long)entry(kp));
        if (kb != ~0ull)
            atomicMin((long long *)&a.status[BNPK_ST_BAD_BASE],
                      (long long)((entry(kb >> kKeyPosBits) << 32) | (kb & ((1ull << kKeyPosBits) - 1))));
        if (kl) atomicMax((unsigned long long *)&a.status[BNPK_ST_LAST_ROW_INDEX], (unsigned long long)entry(kl - 1) + 1ull);
    }
    const uint64_t n_def = min((unsigned long long)a.ws[kWsDeferred], (unsigned long long)a.deferred_cap);
    for (uint64_t d = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; d < n_def; d += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t r = a.deferred[2 * d + 1];
        a.deferred[2 * d + 1] = entry(r & ~kDeferredResolved) | (r & kDeferredResolved);
    }
}
}  // namespace

int ws_resolve(const TileArgs &a, cudaStream_t st) {
    if (a.n_tiles_total <= 0) return 0;
    const unsigned nb = (unsigned)((a.n_tiles_total + kResolveTiles - 1) / kResolveTiles);
    ws_resolve_sum_kernel<<<nb, kResolveTiles, 0, st>>>(a);
    BNPK_LAUNCHED("ws_resolve_sum_kernel");
    ws_resolve_tiles_kernel<<<nb, kResolveTiles, 0, st>>>(a);
    BNPK_LAUNCHED("ws_resolve_tiles_kernel");
    ws_resolve_labels_kernel<<<(unsigned)sm_count(), 256, 0, st>>>(a);
    BNPK_LAUNCHED("ws_resolve_labels_kernel");
    return 0;
}
}  // namespace bnpk
