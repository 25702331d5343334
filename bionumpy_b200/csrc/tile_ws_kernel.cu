// tile_ws_kernel.cu -- the three builds of the warp-specialised fused count (tile_ws_kernel.inl)
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

namespace bnpk {
// minimizer counts the wsm build takes: CTA-private table, windows of at most kMinzW k-mers; the rest (and global
// tables) stay with the register-staged kernel
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
