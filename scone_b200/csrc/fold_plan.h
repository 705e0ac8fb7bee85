// fold_plan.h -- which kernel path, cluster and grid run one call of the projection fold (fold.cu).
//
// Plain host-side C++: no CUDA header, no environment read, so that g++ compiles it on its own (tests/test_fold_plan.py).
// fold.cu reads the two path switches and the exchange kernel's residency, plans the call before anything is launched, and
// fold_kernel<PATH> takes its cluster, epilogue and ring shape from the path's row.
#pragma once
#include <cstdint>

#include "../../include/scone_b200.h"

#ifdef __CUDACC__
#define SCONE_HD __host__ __device__
#else
#define SCONE_HD
#endif

namespace scone {

constexpr int kBM = 128, kBN = 256, kBK = 64;  // row tile, column chunk (one TMEM accumulator), k-block
constexpr int kABytes = kBM * kBK * 2, kBBytes = kBN * kBK * 2;
constexpr int kFoldRingBytes = 4 * (kABytes + kBBytes);  // 192 KB of ring on every path
constexpr int kMaxXch = 8;                               // CTAs of a cluster that exchange row absmax (portable cluster size)

enum FoldPath : int {
    kFoldSingle,    // one CTA per 128-row tile
    kFoldPairs,     // CTA pairs on neighbouring row tiles, each multicasting half of every W tile into both
    kFoldPairTile,  // CTA pairs on one 256-row tile, tcgen05.mma.cta_group::2
    kFoldExchange,  // INT8, one cluster of n_chunks CTAs per row tile exchanging row absmax: one sweep
    kNumFoldPaths
};

struct FoldPathRow {
    int tiles;        // row tiles a cluster computes, one per CTA (the exchange: its n_chunks CTAs share one)
    int epi_warps;    // epilogue warps: groups of 8 that drain one accumulator each
    int stages, stage_bytes;
    int w_box_rows;   // rows of W one CTA loads per stage
};

SCONE_HD constexpr int fold_threads(const FoldPathRow &r) { return 64 + 32 * r.epi_warps; }

constexpr FoldPathRow kFoldPaths[kNumFoldPaths] = {
    // kFoldSingle: FP32 / INT4, where the epilogue's stores or divisions dominate (pairs measured FP32 -9 %, INT4 -2 %)
    {1, 8, 4, kABytes + kBBytes, kBN},
    // kFoldPairs: FP16 / INT8 two sweeps: the 4-stage ring was L2-fill-bound (768 KB per 6 us of tensor work per SM); sharing
    // every W tile pulls 32 KB instead of 48 KB per stage, +3-5 % (profiles/tune_r02.md section 10)
    {2, 8, 4, kABytes + kBBytes, kBN / 2},
    // kFoldPairTile: each CTA stages its own 128 rows and half of W, so the same 192 KB hold six k-blocks in flight instead of
    // four.  FP16 with K >= 512: 3.93 -> 3.11 ms at 1024 -> 4096 and 1.44 -> 1.36 ms at 768 -> 1024 (same-box A/B,
    // profiles/tune_r02.md section 22).  Not for the others: FP32 4.10 -> 4.15 ms (store-bound), INT4 3.32 -> 4.07 ms (its
    // heavier epilogue holds up both CTAs), K = 384 3 % slower.
    {2, 8, 6, kABytes + kBBytes / 2, kBN / 2},
    // kFoldExchange: INT8 with 2..8 column chunks; its epilogue (absmax, exchange, exact division) is a ~12 us latency chain
    // per tile against ~7 us of tensor work, so two groups of 8 warps take alternate row tiles
    {1, 16, 4, kABytes + kBBytes, kBN},
};

// One call of the fold, as far as the choice of path depends on it.
struct FoldCall {
    int quant;            // SCONE_QUANT_*
    int H, K;             // output width (table dim), contraction width (in_dim)
    int64_t k;            // source rows
    int sms;              // SMs of the device
    const char *sm2_env;  // SCONE_FOLD_2SM, or NULL
    const char *xch_env;  // SCONE_FOLD_XCH, or NULL
    int xch_resident;     // clusters of the exchange kernel that fit the device (0: none fits, or not queried)
};

struct FoldPlan {
    FoldPath path;
    int cluster;                              // CTAs per cluster
    int n_chunks, k_blocks, m_groups, sweeps; // m_groups: groups of `tiles` row tiles, one per cluster at a time
    int grid, threads;
};

SCONE_HD constexpr int fold_chunks(int H) { return (H + kBN - 1) / kBN; }

// INT8 rows carry one scale per row, and TMEM holds 512 of their columns: with 2..8 column chunks the CTAs of one cluster can
// each keep a chunk and exchange the row absmax (one sweep instead of two).  SCONE_FOLD_XCH=0 forces the two-sweep path.  When
// this holds, fold.cu asks the device how many such clusters fit (FoldCall::xch_resident).
inline bool fold_exchange_possible(int quant, int H, const char *xch_env) {
    const int n = fold_chunks(H);
    return quant == SCONE_QUANT_INT8 && n >= 2 && n <= kMaxXch && !(xch_env && xch_env[0] == '0');
}

inline FoldPlan plan_fold(const FoldCall &c) {
    FoldPlan pl{};
    pl.n_chunks = fold_chunks(c.H);
    pl.k_blocks = (c.K + kBK - 1) / kBK;
    const bool xch = fold_exchange_possible(c.quant, c.H, c.xch_env) && c.xch_resident > 0;
    // SCONE_FOLD_2SM=0 / 1 forces the pair tile off / on (the tests run both for every format); never inside the exchange
    const bool sm2 = !xch && (c.sm2_env ? c.sm2_env[0] == '1' : (c.quant == SCONE_QUANT_FP16 && c.K >= 512));
    pl.path = xch ? kFoldExchange : sm2 ? kFoldPairTile : (c.quant == SCONE_QUANT_FP16 || c.quant == SCONE_QUANT_INT8) ? kFoldPairs : kFoldSingle;
    const FoldPathRow &r = kFoldPaths[pl.path];
    pl.cluster = xch ? pl.n_chunks : r.tiles;
    pl.sweeps = (c.quant == SCONE_QUANT_INT8 && pl.n_chunks > 1 && !xch) ? 2 : 1;  // first sweep: row absmax only
    const int64_t m_tiles = (c.k + kBM - 1) / kBM;
    pl.m_groups = (int)((m_tiles + r.tiles - 1) / r.tiles);
    int clusters = xch ? c.xch_resident : c.sms / pl.cluster;  // persistent: one resident wave
    if (clusters > pl.m_groups) clusters = pl.m_groups;
    pl.grid = clusters * pl.cluster;
    pl.threads = fold_threads(r);
    return pl;
}

}  // namespace scone
