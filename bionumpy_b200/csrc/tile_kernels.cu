// tile_kernels.cu -- single-pass kernels over raw chunk bytes (K1 line split, K6 fused count).
//
// Persistent CTAs; tiles of kTileBytes (+ a halo so rows that start in a tile can finish in it)
// are handed out in order by an atomic ticket.  Thread t of a CTA owns the 64 contiguous bytes
// [64t, 64t+64) of the staged region (two 256-bit loads); the last warp owns the halo.  Per tile:
//   1. 64 B/thread -> registers; exact '\n' mask per thread (SWAR zero-byte test)
//   2. block scan of newline counts + decoupled look-back -> global line index of every byte,
//      so every thread knows which of its bytes lie on a sequence line (the row-offset vector
//      never leaves the SM: row starts/ends go to shared memory)
//   3. only sequence bytes are turned into 2-bit codes (and validated) -> packed stream in smem
//   4. four threads per read row walk the packed stream: funnel-shift = rolling 2-bit hash,
//      one shared-memory atomic per k-mer into the CTA-private histogram
//   5. at the end of the grid-stride loop the private histogram is flushed with global atomics.
// Minimizers use one warp per row and a warp-shuffle sliding minimum.
#include <cstdlib>
#include "tile_common.cuh"

namespace bnpk {



// -------------------------------------------------------------------------------------------
// init: decide '\r' trimming like OneLineBuffer._modify_for_carriage_return
// (io/one_line_buffer.py:175-182): trim iff the header line of one of the first
// `lines_per_entry` entries ends in '\r'.
// -------------------------------------------------------------------------------------------
__global__ void cr_detect_kernel(const uint8_t *chunk, size_t n, int lpe, int trim_cr, int64_t *status) {
    if (blockIdx.x != 0 || threadIdx.x >= 32) return;
    const int lane = threadIdx.x;
    int64_t cr = 0;
    if (trim_cr == 1) cr = 1;
    if (trim_cr < 0) {
        int64_t pos = 0;
        for (int line = 0; line < lpe * lpe && pos < (int64_t)n; ++line) {
            const int64_t len = warp_line_len(chunk, n, pos, lane);
            if (len < 0) break;
            if (line % lpe == 0 && len > 0 && chunk[pos + len - 1] == '\r') { cr = 1; break; }
            pos += len + 1;
        }
    }
    if (lane == 0) status[BNPK_ST_CR] = cr;
}

// -------------------------------------------------------------------------------------------
// the tile kernel.  MODE 0 = split (write starts/lens), MODE 1 = fused count.
// -------------------------------------------------------------------------------------------
constexpr int kCtaThreads = (kTileBytes + kHaloBytes) / 64;      // one thread per 64 staged bytes
constexpr int kCtaWarps = kCtaThreads / 32;
constexpr int kMainThreads = kTileBytes / 64;
constexpr int kNl0Bytes = (kCtaThreads + 4 + 15) & ~15;
static_assert(kCtaThreads % 32 == 0 && kMainThreads % 32 == 0 && kCtaWarps <= 32, "tile geometry");
// shared-memory layout of the tile kernel, in 32-bit words
constexpr int kOffCodes = 0;
constexpr int kOffRowEnd = kOffCodes + kStagedUnits + 4;
constexpr int kOffRowStart = kOffRowEnd + kRowCap;
constexpr int kOffWarp = kOffRowStart + kRowCap / 2;
constexpr int kOffMisc = kOffWarp + 32;
constexpr int kOffNl0 = kOffMisc + 16;
constexpr int kOffLut = kOffNl0 + kNl0Bytes / 4;
constexpr int kOffHist = kOffLut + 64;

// Software pipeline (per CTA): front(T+3) | look-back loads(T+1) | main(T)
//   front : take a ticket, load 64 B/thread from HBM, exact newline mask, block scan, publish the tile's count
//   main  : resolve the line prefix (loads issued one stage earlier); every thread drops the positions of its
//           newlines into a sorted shared list; ONE THREAD PER NEWLINE does validation / field publishing;
//           rows are read straight off the list (row s starts after newline jr0 + s*lpe and ends at the next one);
//           four threads per read row load the row's 16-byte units (L2 hits), encode + validate only those,
//           then walk the packed stream for the k-mers.
constexpr int kNlCap = 1024;              // newline positions of one staged tile kept in shared memory
constexpr int kNlStep = kNlCap - 8;       // window advance when a tile holds more (lines shorter than ~18 bytes)

template <int MODE, int ENC, bool SMEM_HIST, bool MINIMIZER>
__global__ void __launch_bounds__(kCtaThreads, MODE == 0 ? 4 : 3) tile_kernel(const TileArgs a) {
    extern __shared__ __align__(16) uint32_t smem[];
    // layout: [private histogram (n_bins u32, SMEM_HIST only)] [packed stream] [newline list] [small stuff]
    uint32_t *s_hist = smem;
    uint32_t *s_codes = smem + ((MODE == 1 && SMEM_HIST) ? a.n_bins : 0);          // kStagedUnits + 4
    uint16_t *s_nlpos = reinterpret_cast<uint16_t *>(s_codes + kStagedUnits + 4);  // kNlCap
    uint32_t *s_warp = reinterpret_cast<uint32_t *>(s_nlpos + kNlCap);             // 32
    uint32_t *s_misc = s_warp + 32;                                                // 16
    uint8_t *s_lut = reinterpret_cast<uint8_t *>(s_misc + 16);                     // 256
    __shared__ int64_t s_line_base;
    __shared__ int64_t s_tk[3];

    const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5;
    const LookbackArrays lb = lookback_arrays(a.ws, a.n_tiles_total);
    const bool cr = a.status[BNPK_ST_CR] != 0;

    if (MODE == 1) {
        if (ENC == BNPK_ENC_LUT && tid < 256) s_lut[tid] = a.lut[tid];
        if (SMEM_HIST)
            for (uint32_t b = tid; b < a.n_bins; b += kCtaThreads) s_hist[b] = 0;
        for (int i = tid; i < kStagedUnits + 4; i += kCtaThreads) s_codes[i] = 0;
    }
    HistTarget ht;
    ht.global = a.hist;
    ht.smem = s_hist;
    ht.n_bins = a.n_bins;
    ht.mask = (a.n_bins & (a.n_bins - 1)) == 0 ? a.n_bins - 1 : 0;
    ht.delta = 1ull;
    ht.canon_xor = a.canon_xor;
    uint64_t acc_bases = 0, acc_values = 0;     // per-thread statistics, flushed once
    // lines_per_entry is a power of two (1, 2 or 4): phases and entry indices are masks and shifts
    const uint32_t ls = (uint32_t)a.lpe_shift, pm = (1u << ls) - 1u;
    const uint32_t fl = (uint32_t)a.field_line;
    const uint32_t want = (fl - 1u) & pm;                          // phase of the newline before the field line
    const int my0 = tid * 64;                                       // first staged byte of this thread

    auto staged_len_of = [&](int64_t tile) -> int {
        const size_t byte0 = (size_t)tile * kTileBytes;
        return (MODE == 1) ? (int)min((size_t)(kTileBytes + kHaloBytes), a.n - byte0) : (int)min((size_t)kTileBytes, a.n - byte0);
    };
    auto load_raw = [&](int64_t tile, uint32_t *raw) {
        const size_t byte0 = (size_t)tile * kTileBytes;
        const int staged_len = staged_len_of(tile);
        if (my0 < staged_len) {
            const uint8_t *p = a.chunk + byte0 + my0;
            if (my0 + 64 <= staged_len && (reinterpret_cast<uintptr_t>(p) & 31) == 0) {
                ld_stream_256(p, raw);
                ld_stream_256(p + 32, raw + 8);
            } else {
#pragma unroll
                for (int u = 0; u < 4; ++u) {
                    const uint4 q = load_unit_guarded(a.chunk, a.n, (int64_t)(byte0 + my0) + 16 * u);
                    raw[4 * u] = q.x; raw[4 * u + 1] = q.y; raw[4 * u + 2] = q.z; raw[4 * u + 3] = q.w;
                }
            }
        }
    };
    // front end of one tile: newline mask, block scan, publish the tile's newline count.
    // (two __syncthreads; must be called by every thread).  tnl = newlines of the tile proper,
    // tall = newlines of the whole staged region (tile + halo).
    auto front = [&](int64_t tile, const uint32_t *raw, uint64_t &nl, uint32_t &ex, int st_slot) {
        const int staged_len = staged_len_of(tile);
        nl = 0;
        if (my0 < staged_len) {
            nl = eq_mask64(raw, 0x0A0A0A0Au);
            if (my0 + 64 > staged_len) nl &= (~0ull) >> (64 - (staged_len - my0));
        }
        const uint32_t cnt = (uint32_t)__popcll(nl);
        uint32_t inc = cnt;
#pragma unroll
        for (int o = 1; o < 32; o <<= 1) {
            const uint32_t t = __shfl_up_sync(0xffffffffu, inc, o);
            if (lane >= o) inc += t;
        }
        if (lane == 31) s_warp[warp] = inc;
        __syncthreads();
        if (warp == 0) {
            const uint32_t w = lane < kCtaWarps ? s_warp[lane] : 0;
            uint32_t winc = w;
#pragma unroll
            for (int o = 1; o < 32; o <<= 1) {
                const uint32_t t = __shfl_up_sync(0xffffffffu, winc, o);
                if (lane >= o) winc += t;
            }
            if (lane < kCtaWarps) s_warp[lane] = winc - w;           // exclusive warp prefix
            const uint32_t tile_nl_w = __shfl_sync(0xffffffffu, winc, kMainThreads / 32 - 1);   // tile proper only
            const uint32_t all_nl_w = __shfl_sync(0xffffffffu, winc, kCtaWarps - 1);
            if (lane == 0) {
                s_misc[6 + 2 * st_slot] = tile_nl_w;                 // per-stage ring: newlines of the tile proper ...
                s_misc[7 + 2 * st_slot] = all_nl_w;                  // ... and of the whole staged region
            }
        }
        __syncthreads();
        ex = s_warp[warp] + inc - cnt;
        // publish after the barrier: the round trip of its atomic (whose result only this thread needs) must not
        // hold up the other warps
        if (tid == 0) lookback_publish(lb, tile, s_misc[6 + 2 * st_slot]);
    };
    auto take_ticket = [&]() -> int64_t {
        return a.tile_begin + (int64_t)atomicAdd((unsigned long long *)(a.ws + kWsTicket), 1ull);
    };
    auto defer_row = [&](uint64_t start, uint64_t r) {
        const unsigned long long d = atomicAdd((unsigned long long *)(a.ws + kWsDeferred), 1ull);
        if (d < a.deferred_cap) {
            a.deferred[2 * d] = start;
            a.deferred[2 * d + 1] = r;
        } else {
            a.status[BNPK_ST_OVERFLOW] = 1;
        }
    };

    // ---- prologue: fill the pipeline: all three first tickets are counted and published before any
    // main stage runs, so no CTA ever waits for a neighbour's main stage ------------------------------
    if (tid == 0) { s_tk[0] = take_ticket(); s_tk[1] = take_ticket(); s_tk[2] = take_ticket(); }
    __syncthreads();
    int64_t tM = s_tk[0], tP = s_tk[1], tF = s_tk[2];
    uint32_t raw[16];
    uint64_t nlM = 0, nlP = 0, nlF = 0, lbA = kFlagPrefix, lbB = kFlagPrefix;
    uint32_t exM = 0, exP = 0, exF = 0;
    int slotM = 0;                                                  // ring slot of the main-stage tile (P: +1, F: +2 mod 3)
    if (tM < a.tile_end) { load_raw(tM, raw); front(tM, raw, nlM, exM, 0); }
    if (tP < a.tile_end) { load_raw(tP, raw); front(tP, raw, nlP, exP, 1); }
    if (tF < a.tile_end) { load_raw(tF, raw); front(tF, raw, nlF, exF, 2); }
    if (warp == 0 && tM < a.tile_end) lookback_issue(lb, tM, lane, lbA, lbB);

    while (tM < a.tile_end) {
        const int64_t tile = tM;
        const size_t byte0 = (size_t)tile * kTileBytes;
        const int staged_len = staged_len_of(tile);
        const uint32_t tile_nl = s_misc[6 + 2 * slotM], all_nl = s_misc[7 + 2 * slotM];

        // ---- 1. resolve the prefix, ask for the next ticket ------------------------------------------
        int64_t next_ticket = 0;
        if (tid == 0) next_ticket = take_ticket();
        if (warp == 0) {
            const uint64_t excl = lookback_finish(lb, tile, tile_nl, lane, lbA, lbB);
            if (lane == 0) {
                s_line_base = (int64_t)excl;
                s_misc[1] = 0; s_misc[2] = 0;
                s_tk[0] = next_ticket;
            }
        }
        const int n_rounds = all_nl > (uint32_t)kNlCap ? (int)((all_nl - 8u + kNlStep - 1) / kNlStep) : 1;
        int64_t line_base = 0, tN = 0;
        for (int round = 0; round < n_rounds; ++round) {
            // ---- 2. sorted list of the newline positions of this staged tile (window `round`) -------------
            if (round > 0) __syncthreads();
            const int win_lo = round * kNlStep;
            {
                uint64_t m = nlM;
                int li = (int)exM - win_lo;
                while (m) {
                    const int bit = __ffsll((long long)m) - 1;
                    m &= m - 1;
                    if (li >= 0 && li < kNlCap) s_nlpos[li] = (uint16_t)(my0 + bit);
                    ++li;
                }
            }
            __syncthreads();                                         // S1: prefix, ticket, list (and the previous k-mer stage) done
            if (round == 0) {
                line_base = s_line_base;
                tN = s_tk[0];
                // start the next front-end load (HBM) and the look-back loads of the pending tile
                if (tN < a.tile_end) load_raw(tN, raw);
                if (warp == 0 && tP < a.tile_end) lookback_issue(lb, tP, lane, lbA, lbB);
            }
            // 32-bit, tile-relative line arithmetic: global line = line_base + rel
            const uint32_t base_phase = (uint32_t)line_base & pm;
            const int64_t q0 = line_base >> ls;                      // entry index of the tile's first line
            const uint32_t jr0 = (want - base_phase) & pm;           // first newline (rel) that precedes a field line
            const uint32_t r_first_off = (base_phase + jr0 + 1u) >> ls;
            const int64_t r_first = q0 + r_first_off;
            const int n_rows_tile = (tile_nl > jr0) ? (int)(((tile_nl - 1u - jr0) >> ls) + 1u) : 0;
            const int n_in_win = min((int)all_nl - win_lo, kNlCap);
            // events owned by this window: newline indices [win_lo, win_lo + kNlStep) (all of them in the last window)
            const int ev_hi = (round == n_rounds - 1) ? n_in_win : kNlStep;

            // ---- 3. one thread per newline: validation, field publishing (split mode) -----------------
            for (int i = tid; i < ev_hi; i += kCtaThreads) {
                const uint32_t gi = (uint32_t)(win_lo + i);           // tile-relative newline index = rel line index
                const int p = s_nlpos[i];
                const size_t gp = byte0 + p;
                const uint32_t phase = (base_phase + gi) & pm;
                if (gi < tile_nl) {                                   // newline of the tile proper
                    if (phase == pm) {                                // last line of an entry: next byte starts a header
                        if (gp + 1 < a.n && a.chunk[gp + 1] != a.header_char)      // one_line_buffer.py:155-173
                            atomicMin((long long *)&a.status[BNPK_ST_BAD_HEADER_ENTRY],
                                      (long long)(q0 + ((base_phase + gi + 1u) >> ls)));
                    }
                    if (a.check_plus && phase == 1u) {              // fastq_buffer.py:38-45
                        if (gp + 1 < a.n && a.chunk[gp + 1] != '+')
                            atomicMin((long long *)&a.status[BNPK_ST_BAD_PLUS_ENTRY],
                                      (long long)(q0 + ((base_phase + gi) >> ls)));
                    }
                    if (MODE == 0) {
                        // split: start and end of the wanted line are published independently;
                        // lens[r] accumulates (end - start) mod 2^32 from two atomics.
                        if (phase == want) {
                            const int64_t r = q0 + ((base_phase + gi + 1u) >> ls);
                            if ((size_t)r < a.max_rows) {
                                const int64_t st = (int64_t)gp + 1 + a.start_offset;
                                a.starts[r] = st;
                                atomicSub((unsigned int *)&a.lens[r], (unsigned int)(uint64_t)st);
                            }
                        }
                        if (phase == fl) {
                            const int64_t r = q0 + ((base_phase + gi) >> ls);
                            if ((size_t)r < a.max_rows) {
                                int64_t e = (int64_t)gp;
                                if (cr && gp > 0 && a.chunk[gp - 1] == '\r') e -= 1;
                                atomicAdd((unsigned int *)&a.lens[r], (unsigned int)(uint64_t)e);
                            }
                        }
                    }
                }
            }
            // last complete entry of the tile proper: the last newline with phase pm
            if (tid == 0 && tile_nl > 0) {
                const uint32_t last = tile_nl - 1u;
                const uint32_t back = (base_phase + last - pm) & pm;  // steps back to a phase-pm newline
                if (last >= back) {
                    const int li = (int)(last - back) - win_lo;
                    if (li >= 0 && li < ev_hi)
                        atomicMax((unsigned long long *)&a.status[BNPK_ST_N_COMPLETE_BYTES],
                                  (unsigned long long)(byte0 + s_nlpos[li] + 1));
                }
            }
            if (tile == 0 && tid == 0 && round == 0) {
                if (a.n > 0 && a.chunk[0] != a.header_char)
                    atomicMin((long long *)&a.status[BNPK_ST_BAD_HEADER_ENTRY], 0ll);
                if (MODE == 0 && fl == 0 && a.max_rows > 0) {       // the first line has no newline before it
                    a.starts[0] = a.start_offset;
                    atomicSub((unsigned int *)&a.lens[0], (unsigned int)a.start_offset);
                }
            }

            // ---- 4. rows straight off the list: encode their units, then the k-mers -------------------
            if (MODE == 1) {
                // rows whose start newline index lies in this window
                const int s_lo = (win_lo > (int)jr0) ? (int)((win_lo - jr0 + pm) >> ls) : 0;
                int s_hi = n_rows_tile;
                if (round != n_rounds - 1) s_hi = min(s_hi, (int)((win_lo + kNlStep - (int)jr0 + (int)pm) >> ls));
                const uint64_t kmask = (1ull << (2 * a.k)) - 1;
                const bool fast = ht.mask && ht.mask <= 0x3FFFFFFFull && !ht.canon_xor;   // the minimum needs every bit
                const uint32_t m32x4 = (uint32_t)(ht.mask & kmask) << 2;         // byte-offset mask into the table
                const uint32_t need_bits = (uint32_t)__popcll(ht.mask & kmask);  // stream bits one table index needs
                constexpr int kGroups = MINIMIZER ? kCtaWarps : kCtaThreads / 4;  // rows handled concurrently
                const int sub = MINIMIZER ? lane : (lane & 3);
                const int nsub = MINIMIZER ? 32 : 4;
                const int grp = MINIMIZER ? warp : (tid >> 2);
                const unsigned gmask = MINIMIZER ? 0xffffffffu : (0xFu << (lane & ~3));
                for (int slot0 = s_lo; slot0 < s_hi; slot0 += kGroups) {
                    const int slot = slot0 + grp;
                    if (slot >= s_hi) continue;
                    const int li = (int)(jr0 + ((uint32_t)slot << ls)) - win_lo;   // list index of the row's start newline
                    const int b0 = (int)s_nlpos[li] + 1 + a.start_offset;
                    if ((uint32_t)(win_lo + li) + 1u >= all_nl) {   // no terminating newline in the staged region
                        if (sub == 0 && byte0 + staged_len < a.n) defer_row(byte0 + b0, (uint64_t)(r_first + slot));   // long row
                        continue;                                    // (else: unterminated last line, not an entry)
                    }
                    int e = s_nlpos[li + 1];
                    if (cr && e > b0 && a.chunk[byte0 + e - 1] == '\r') e -= 1;
                    const int L = e - b0;
                    if (sub == 0) {
                        acc_bases += (uint64_t)L;
                        atomicMax(&s_misc[1], (uint32_t)b0 + 1u);
                        atomicMax(&s_misc[2], (uint32_t)slot + 1u);
                    }
                    // encode + validate the row's 16-byte units (re-read from L2); only sequence units are touched
                    if (L > 0) {
                        const int u1 = (e - 1) >> 4;
                        for (int u = (b0 >> 4) + sub; u <= u1; u += nsub) {
                            const uint4 q = load_unit_guarded(a.chunk, a.n, (int64_t)byte0 + 16 * (int64_t)u);
                            const uint32_t w[4] = {q.x, q.y, q.z, q.w};
                            const int lo = max(b0 - 16 * u, 0), hi = min(e - 16 * u, 16);
                            const uint32_t seq16 = (0xFFFFu >> (16 - hi)) & (0xFFFFu << lo);
                            uint32_t bad;
                            s_codes[u] = encode_unit_seq<ENC>(w, seq16, s_lut, bad);
                            if (bad) {                                // rare: exact position, byte by byte
                                for (int p = 16 * u + lo; p < 16 * u + hi; ++p) {
                                    const uint32_t c = a.chunk[byte0 + p];
                                    bool okb;
                                    if (ENC == BNPK_ENC_CODES) okb = c < 4;
                                    else if (ENC == BNPK_ENC_LUT) okb = s_lut[c] < 4;
                                    else { const uint32_t uu = c | 0x20u; okb = (uu == 'a' || uu == 'c' || uu == 'g' || uu == 't'); }
                                    if (!okb) {
                                        atomicMin((long long *)&a.status[BNPK_ST_BAD_BASE],
                                                  (long long)(((r_first + slot) << 32) | (int64_t)(p - b0)));
                                        break;
                                    }
                                }
                            }
                        }
                    }
                    __syncwarp(gmask);
                    if constexpr (MINIMIZER) {
                        if (L >= a.window) acc_values += row_count<SMEM_HIST, true>(s_codes, b0, L, a.k, a.window, ht, lane);
                    } else {
                        const int npos = L - a.k + 1;
                        if (fast) {
                            // Interleaved positions: thread `sub` of the row's four takes p = sub + 4j, so the shift of
                            // k-mer j inside its 32-bit stream word is 8*(j&3) + 2*sub: the 2*sub part is folded into a
                            // per-thread rotated copy of the stream, what is left are constant byte shifts.  The stream
                            // is also pre-shifted left by two bits so that (window & mask) is the table's byte offset.
                            const uint32_t last_w = npos > 0 ? (2u * (uint32_t)(b0 + npos - 1) + need_bits - 1u) >> 5 : 0u;
                            for (int pbase = 0; pbase < npos; pbase += 128) {
                                const int nj = min((npos - pbase - sub + 3) >> 2, 32);      // my k-mers in this pass
                                if (nj <= 0) continue;
                                acc_values += (uint64_t)nj;
                                const uint32_t bit = 2u * (uint32_t)(b0 + pbase);
                                const uint32_t idx = bit >> 5, sh = bit & 31u;
                                // only words that hold bits of this row are read (neighbours may still be written)
                                uint32_t wq = idx + 2 <= last_w ? s_codes[idx + 2] : 0u;
                                const uint32_t wA = s_codes[idx], wB = idx + 1 <= last_w ? s_codes[idx + 1] : 0u;
                                uint32_t c1 = __funnelshift_r(wB, wq, sh);
                                uint32_t r0 = __funnelshift_r(__funnelshift_r(wA, wB, sh), c1, 2u * (uint32_t)sub);
                                uint32_t rp0 = r0 << 2;
#pragma unroll
                                for (int q = 0; q < 8; ++q) {
                                    if (4 * q >= nj) break;
                                    const uint32_t wn = idx + q + 3 <= last_w ? s_codes[idx + q + 3] : 0u;
                                    const uint32_t c2 = __funnelshift_r(wq, wn, sh);
                                    const uint32_t r1 = __funnelshift_r(c1, c2, 2u * (uint32_t)sub);
                                    const uint32_t rp1 = __funnelshift_l(r0, r1, 2);
                                    const int left = nj - 4 * q;
#pragma unroll
                                    for (int t = 0; t < 4; ++t) {
                                        const uint32_t v = __funnelshift_r(rp0, rp1, 8 * t) & m32x4;
                                        if (t < left) {
                                            if constexpr (SMEM_HIST) atomicAdd(reinterpret_cast<uint32_t *>(reinterpret_cast<char *>(s_hist) + v), 1u);
                                            else atomicAdd(reinterpret_cast<unsigned long long *>(reinterpret_cast<char *>(a.hist) + 2 * (size_t)v), 1ull);
                                        }
                                    }
                                    wq = wn; c1 = c2; r0 = r1; rp0 = rp1;
                                }
                            }
                        } else {
                            for (int p0 = sub * 32; p0 < npos; p0 += 128) {
                                const int n_here = min(32, npos - p0);
                                acc_values += (uint64_t)n_here;
                                for (int j = 0; j < n_here; ++j) {
                                    uint64_t h = stream_64(s_codes, (uint32_t)(b0 + p0 + j)) & kmask;
                                    if (ht.canon_xor) h = canonical_hash(h, a.k, ht.canon_xor);
                                    if (!SMEM_HIST && a.hist32)       // canonical counts into 2^22..2^24 bins
                                        atomicAdd(a.hist32 + (ht.mask ? (h & ht.mask) : (h % ht.n_bins)), 1u);
                                    else
                                        hist_add<SMEM_HIST>(ht, h);
                                }
                            }
                        }
                    }
                }
            }
        }
        // ---- 5. front end of the new tile (its bytes were requested after S1); rotate the pipeline ------
        uint64_t nlN = 0;
        uint32_t exN = 0;
        if (tN < a.tile_end) {
            front(tN, raw, nlN, exN, slotM);                         // two __syncthreads inside; reuses the finished tile's slot
        } else {
            __syncthreads();
        }
        // per-tile global bookkeeping of the tile just finished (its shared-memory atomics are ordered before
        // the barrier(s) above)
        if (tid == 0) {
            if (MODE == 1 && s_misc[1]) {
                const uint32_t base_phase = (uint32_t)line_base & pm;
                const uint32_t jr0 = (want - base_phase) & pm;
                const int64_t r_first = (line_base >> ls) + ((base_phase + jr0 + 1u) >> ls);
                atomicMax((unsigned long long *)&a.status[BNPK_ST_LAST_ROW_START], (unsigned long long)(byte0 + s_misc[1] - 1) + 1ull);
                atomicMax((unsigned long long *)&a.status[BNPK_ST_LAST_ROW_INDEX], (unsigned long long)(r_first + s_misc[2] - 1) + 1ull);
            }
            if (tile == a.n_tiles_total - 1) a.status[BNPK_ST_N_LINES] = line_base + tile_nl;
        }
        tM = tP; nlM = nlP; exM = exP;
        tP = tF; nlP = nlF; exP = exF;
        tF = tN; nlF = nlN; exF = exN;
        slotM = slotM == 2 ? 0 : slotM + 1;
    }

    // ---- flush ---------------------------------------------------------------------------------
    if (MODE == 1) {
        if (SMEM_HIST) {
            __syncthreads();
            for (uint32_t b = tid; b < a.n_bins; b += kCtaThreads) {
                const uint32_t c = s_hist[b];
                if (c) atomicAdd(a.hist + b, (unsigned long long)c);
            }
        }
        acc_bases = warp_sum_u64(acc_bases);
        acc_values = warp_sum_u64(acc_values);
        if (lane == 0) {
            if (acc_bases) atomicAdd((unsigned long long *)&a.status[BNPK_ST_N_BASES], acc_bases);
            if (acc_values) atomicAdd((unsigned long long *)&a.status[BNPK_ST_N_VALUES], acc_values);
        }
    }
}

// n_records and friends once every tile is done
__global__ void finalize_status_kernel(int64_t *status, int lpe) {
    if (threadIdx.x == 0 && blockIdx.x == 0) status[BNPK_ST_N_RECORDS] = status[BNPK_ST_N_LINES] / lpe;
}

static size_t tile_smem_bytes(int mode, uint64_t n_bins, bool smem_hist) {
    size_t bytes = (size_t)kOffHist * 4;
    if (mode == 1 && smem_hist) bytes += n_bins * 4;
    return bytes;
}

template <int MODE, int ENC, bool SMEM_HIST, bool MINIMIZER>
static int launch_tile(const TileArgs &a, cudaStream_t st) {
    auto kern = tile_kernel<MODE, ENC, SMEM_HIST, MINIMIZER>;
    const size_t smem = tile_smem_bytes(MODE, a.n_bins, SMEM_HIST);
    BNPK_DYN_SMEM(kern, 200 * 1024);
    int per_sm = 1;
    BNPK_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&per_sm, kern, kCtaThreads, smem));
    if (per_sm < 1) return set_err(BNPK_E_BINS, "tile kernel does not fit shared memory");
    const int64_t n_tiles = a.tile_end - a.tile_begin;
    if (n_tiles <= 0) return 0;
    const int64_t grid = std::min<int64_t>(n_tiles, (int64_t)sm_count() * per_sm);
    profile_before(st);
    kern<<<(unsigned)grid, kCtaThreads, smem, st>>>(a);
    profile_after(st);
    BNPK_LAUNCHED("tile_kernel");
    return 0;
}

template <int ENC>
static int launch_count_enc(const TileArgs &a, bool smem_hist, cudaStream_t st) {
    const bool mz = a.window > 0;
    if (smem_hist) return mz ? launch_tile<1, ENC, true, true>(a, st) : launch_tile<1, ENC, true, false>(a, st);
    return mz ? launch_tile<1, ENC, false, true>(a, st) : launch_tile<1, ENC, false, false>(a, st);
}

// BNPK_TILE_KERNEL selects the fused-count kernel (A/B runs, tests of every path): "reg" = register-staged
// everywhere, "tma" = the round-1 shared-memory-staged kernel, anything else = the warp-specialised one
static int tile_kernel_choice() {
    static const int choice = [] {
        const char *e = std::getenv("BNPK_TILE_KERNEL");
        if (e && e[0] == 'r') return 0;
        if (e && e[0] == 't') return 1;
        if (e && e[0] == 'w') return 3;                              // "ws": the warp-specialised kernel for every table
        return 2;
    }();
    return choice;
}
static bool tma_kernel_allowed() { return tile_kernel_choice() != 0; }

// the kernel a fused count of a global table goes to writes the 32-bit scratch table (a.hist32) when it gets one: the
// tma / ws kernels, and for canonical k-mers tile_kernel (global canonical tables always go there).  The minimizer
// walk of tile_kernel (row_count) counts into the int64 table, so canonical minimizers get no scratch.
static bool count_takes_scratch32(const TileArgs &a, bool smem_hist) {
    if (a.canon_xor) return !smem_hist && a.window == 0;
    return tma_kernel_allowed() && tma_count_eligible(a, smem_hist);
}

// *ws_labels: the launch went to one of the ws builds, whose labels the resolve pass (ws_resolve) completes
static int launch_count(const TileArgs &a, int enc_mode, bool smem_hist, cudaStream_t st, bool *ws_labels) {
    *ws_labels = false;
    if (a.canon_xor && a.window) {
        // canonical minimizers: the wsmc build where wsm would take the count (CTA-private table of up to 2^14 bins,
        // windows of up to 12 k-mers), the register-staged kernel for the rest
        if (tma_kernel_allowed() && tile_kernel_choice() != 1 && wsm_count_eligible(a, smem_hist)) {
            *ws_labels = true;
            return launch_wsmc_count(a, enc_mode, smem_hist, st);
        }
    } else if (a.canon_xor) {
        // canonical k-mers: the wsc build for CTA-private tables of up to 2^14 bins, the register-staged kernel for the
        // rest (the round-1 kernel has no canonical build)
        if (tma_kernel_allowed() && wsc_count_eligible(a, smem_hist)) {
            *ws_labels = true;
            return launch_wsc_count(a, enc_mode, smem_hist, st);
        }
    } else if (tma_kernel_allowed() && tile_kernel_choice() != 1 && wsm_count_eligible(a, smem_hist)) {
        *ws_labels = true;
        return launch_wsm_count(a, enc_mode, smem_hist, st);          // minimizers, windows of up to 12 k-mers
    } else if (tma_kernel_allowed() && tma_count_eligible(a, smem_hist)) {
        // the warp-specialised kernel for CTA-private tables; global tables are bound by L2 atomics, where the round-1
        // kernel's 21 row warps per SM keep more of them in flight (2^24 bins: 6.6 ms against 9.3 ms)
        if (tile_kernel_choice() == 1 || (!smem_hist && tile_kernel_choice() != 3)) return launch_tma_count(a, enc_mode, smem_hist, st);
        *ws_labels = true;
        return launch_ws_count(a, enc_mode, smem_hist, st);
    }
    switch (enc_mode) {
        case BNPK_ENC_ASCII_ACGT: return launch_count_enc<BNPK_ENC_ASCII_ACGT>(a, smem_hist, st);
        case BNPK_ENC_ASCII_ACTG: return launch_count_enc<BNPK_ENC_ASCII_ACTG>(a, smem_hist, st);
        case BNPK_ENC_CODES: return launch_count_enc<BNPK_ENC_CODES>(a, smem_hist, st);
        case BNPK_ENC_LUT: return launch_count_enc<BNPK_ENC_LUT>(a, smem_hist, st);
    }
    return set_err(BNPK_E_BADARG, "bad enc_mode");
}

static size_t deferred_capacity(size_t n) { return n / kHaloBytes + n / 1024 + 16; }

// workspace (uint64 words): header | tile_state[n_tiles+1] | block_cnt[nb] | block_state[nb] | deferred[2*cap]
static size_t ws_lookback_words(size_t n_tiles) { return kWsHeaderWords + (n_tiles + 1) + 2 * ((n_tiles >> 5) + 2); }
// ... | u32 scratch[2^24]: large global tables are accumulated in 32-bit counters that stay in L2 (64 MiB instead of
// 128 MiB of int64: 191 vs 60 G updates/s on B200, tools/micro/red_bench.cu) and added to the int64 table at the end
static size_t ws_core_bytes(size_t n) {
    const size_t n_tiles = (n + kTileBytes - 1) / kTileBytes;
    return (((ws_lookback_words(n_tiles) + 2 * deferred_capacity(n)) * sizeof(uint64_t)) + 255) & ~(size_t)255;
}
size_t tile_workspace_bytes(size_t n) { return ws_core_bytes(n) + (size_t)kScratch32MaxBins * sizeof(uint32_t); }

__global__ void widen_add_kernel(const uint32_t *scratch, unsigned long long *hist, size_t n_bins) {
    for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n_bins; i += (size_t)gridDim.x * blockDim.x) {
        const uint32_t c = scratch[i];
        if (c) hist[i] += c;
    }
}

bool use_smem_hist(int64_t n_bins, int hist_mode) {
    if (hist_mode == BNPK_HIST_GLOBAL) return false;
    return n_bins <= kSmemMaxBins;
}

int chunk_kmer_count_impl(const uint8_t *chunk, size_t n, size_t slice_begin, size_t slice_end, int final_slice,
                          int lpe, uint8_t header_char, int check_plus, int trim_cr, int enc_mode,
                          const uint8_t *lut256, int k, int window, int64_t n_bins, int hist_mode, int64_t *hist,
                          int64_t *status, void *workspace, size_t workspace_bytes, cudaStream_t st, uint64_t canon_xor) {
    if (k < 1 || k > 31) return set_err(BNPK_E_K, "k must be larger than 0 and smaller than 32");
    if (window != 0 && window < k) return set_err(BNPK_E_WINDOW, "kmer size must be smaller than window size");
    if (window > 1024) return set_err(BNPK_E_WINDOW, "window_size above 1024 is not supported");
    if (n_bins < 1) return set_err(BNPK_E_BINS, "n_bins must be positive");
    if (hist_mode == BNPK_HIST_SMEM && n_bins > kSmemMaxBins) return set_err(BNPK_E_BINS, "too many bins for the shared-memory histogram");
    if (enc_mode == BNPK_ENC_LUT && !lut256) return set_err(BNPK_E_BADARG, "lut256 required");
    if ((lpe != 2 && lpe != 4) || slice_end > n || slice_begin > slice_end)
        return set_err(BNPK_E_BADARG, "lines_per_entry must be 2 or 4; slice must lie inside the chunk");
    if (workspace_bytes < tile_workspace_bytes(n)) return set_err(BNPK_E_WORKSPACE, "workspace too small");
    if (n == 0) return 0;
    const int64_t n_tiles_total = (int64_t)((n + kTileBytes - 1) / kTileBytes);
    // a tile is complete once its staged region [t*T, min((t+1)*T + H, n)) is resident
    auto tiles_done_at = [&](size_t resident) -> int64_t {
        if (resident >= n) return n_tiles_total;
        if (resident < (size_t)(kTileBytes + kHaloBytes)) return 0;
        return (int64_t)((resident - kHaloBytes) / kTileBytes);
    };
    TileArgs a{};
    a.chunk = chunk; a.n = n;
    a.tile_begin = tiles_done_at(slice_begin);
    a.tile_end = final_slice ? n_tiles_total : tiles_done_at(slice_end);
    a.lpe = lpe; a.lpe_shift = lpe == 4 ? 2 : 1; a.field_line = 1; a.start_offset = 0; a.header_char = header_char;
    a.check_plus = check_plus; a.status = status; a.ws = (uint64_t *)workspace; a.n_tiles_total = n_tiles_total;
    a.deferred_cap = deferred_capacity(n);
    a.deferred = (uint64_t *)workspace + ws_lookback_words((size_t)n_tiles_total);
    a.lut = lut256; a.k = k; a.window = window; a.n_bins = (uint64_t)n_bins; a.hist = (unsigned long long *)hist;
    a.canon_xor = canon_xor;
    if (slice_begin == 0) {
        BNPK_CUDA(cudaMemsetAsync(workspace, 0, ws_lookback_words((size_t)n_tiles_total) * sizeof(uint64_t), st));
        // the ws builds' min-keys start at "none" (all ones)
        BNPK_CUDA(cudaMemsetAsync(a.ws + kWsKeyHeader, 0xFF, (kWsKeyBase - kWsKeyHeader + 1) * sizeof(uint64_t), st));
        cr_detect_kernel<<<1, 32, 0, st>>>(chunk, std::min(n, slice_end), lpe, trim_cr, status);
        BNPK_LAUNCHED("cr_detect_kernel");
    }
    BNPK_CUDA(cudaMemsetAsync(a.ws + kWsTicket, 0, sizeof(uint64_t), st));
    const bool smem_hist = use_smem_hist(n_bins, hist_mode);
    // tables between 32 MiB and 128 MiB of int64: count in the 32-bit scratch (a bin cannot overflow: n < 2^32 bytes)
    const bool scratch32 = !smem_hist && n_bins > (1ll << 22) && n_bins <= kScratch32MaxBins && n < (1ull << 32) &&
                           count_takes_scratch32(a, smem_hist);
    if (scratch32) {
        a.hist32 = reinterpret_cast<uint32_t *>(reinterpret_cast<uint8_t *>(workspace) + ws_core_bytes(n));
        if (slice_begin == 0) BNPK_CUDA(cudaMemsetAsync(a.hist32, 0, (size_t)n_bins * sizeof(uint32_t), st));
    }
    bool ws_labels = false;
    int rc = launch_count(a, enc_mode, smem_hist, st, &ws_labels);
    if (rc) return rc;
    if (final_slice && scratch32) {
        widen_add_kernel<<<sm_count() * 8, 256, 0, st>>>(a.hist32, a.hist, (size_t)n_bins);
        BNPK_LAUNCHED("widen_add_kernel");
    }
    if (final_slice) {
        if (ws_labels && (rc = ws_resolve(a, st))) return rc;
        finalize_status_kernel<<<1, 32, 0, st>>>(status, lpe);
        BNPK_LAUNCHED("finalize_status_kernel");
        rc = count_fixups_impl(chunk, n, lpe, enc_mode, lut256, k, window, n_bins, hist, status,
                               (uint64_t *)workspace + kWsDeferred, a.deferred, a.deferred_cap, st, canon_xor);
    }
    return rc;
}

int line_split_impl(const uint8_t *chunk, size_t n, int lpe, int field_line, int start_offset, uint8_t header_char,
                    int check_plus, int trim_cr, int64_t *starts, int32_t *lens, size_t max_rows, int64_t *status,
                    void *workspace, size_t workspace_bytes, cudaStream_t st) {
    if ((lpe != 1 && lpe != 2 && lpe != 4) || field_line < 0 || field_line >= lpe)
        return set_err(BNPK_E_BADARG, "lines_per_entry must be 1, 2 or 4 and 0 <= field_line < lines_per_entry");
    if (workspace_bytes < tile_workspace_bytes(n)) return set_err(BNPK_E_WORKSPACE, "workspace too small");
    if (n == 0) return 0;
    TileArgs a{};
    a.chunk = chunk; a.n = n;
    a.n_tiles_total = (int64_t)((n + kTileBytes - 1) / kTileBytes);
    a.tile_begin = 0; a.tile_end = a.n_tiles_total;
    a.lpe = lpe; a.lpe_shift = lpe == 4 ? 2 : (lpe == 2 ? 1 : 0); a.field_line = field_line; a.start_offset = start_offset;
    a.header_char = header_char; a.check_plus = check_plus; a.status = status; a.ws = (uint64_t *)workspace;
    a.starts = starts; a.lens = lens; a.max_rows = max_rows; a.n_bins = 1;
    if (max_rows) BNPK_CUDA(cudaMemsetAsync(lens, 0, max_rows * sizeof(int32_t), st));
    BNPK_CUDA(cudaMemsetAsync(workspace, 0, ws_lookback_words((size_t)a.n_tiles_total) * sizeof(uint64_t), st));
    cr_detect_kernel<<<1, 32, 0, st>>>(chunk, n, lpe, trim_cr, status);
    BNPK_LAUNCHED("cr_detect_kernel");
    int rc = launch_tile<0, BNPK_ENC_ASCII_ACGT, false, false>(a, st);
    if (rc) return rc;
    finalize_status_kernel<<<1, 32, 0, st>>>(status, lpe);
    BNPK_LAUNCHED("finalize_status_kernel");
    return 0;
}

}  // namespace bnpk
