// embed_plan.h -- which kernel, shape, lanes per position and ring layout run one call of the fused path.
//
// Plain host-side C++: no CUDA header, no environment read, so that g++ compiles it on its own (tests/test_embed_plan.py).
// embed.cu plans a call before anything is launched; embed_inst.cu instantiates exactly the (shape row, P, ADD)
// combinations that kShapes lists, so a planned kernel always exists.
#pragma once
#include <cstdint>

#ifdef __CUDACC__
#define SCONE_HD __host__ __device__
#else
#define SCONE_HD
#endif

namespace scone {

constexpr int kMaxRing = 16;      // row-ring slots of the bulk-copy kernels
constexpr int kMaxMetaRing = 32;  // metadata-ring slots of the pipeline

// Ring geometry of embed_bulk_kernel.
struct BulkLayout {
    int ring;        // ring slots (tiles in flight per CTA)
    int slot_bytes;  // bytes reserved per position: >= max(row_stride, 2 D), multiple of 128
    int smem_bytes;  // dynamic shared memory per CTA
};

// Ring geometry of embed_pipe_kernel.
struct PipeLayout {
    int ring;        // row-ring slots (tiles staged or being consumed)
    int meta_ring;   // metadata-ring slots, a multiple of NM
    int slot_bytes;  // bytes reserved per position: table / fallback row [+ base row of a hit at add_off]
    int add_off;
    int pos_off;     // offset of the tile's block of G position rows (2 D bytes each, contiguous) from the tile's first slot, or 0
    int tile_bytes;  // G slots + the position block
    int smem_bytes;
};

// bytes of barriers + ring metadata in front of the row slots
SCONE_HD constexpr int bulk_header_bytes(int G) { return (2 * kMaxRing * 8 + kMaxRing * G * 8 + 127) / 128 * 128; }
// barriers, slot headers and the metadata ring in front of the row slots
SCONE_HD constexpr int pipe_header_bytes(int G) {
    return ((2 * kMaxRing + 2 * kMaxMetaRing) * 8 + (kMaxRing + kMaxMetaRing) * G * 9 + 127) / 128 * 128;
}

enum Family : int {
    kBulk = 0,  // embed_bulk_kernel: one ring, the matcher stages its own tile (plain path only)
    kPipe = 1,  // embed_pipe_kernel: matcher, loader and gather warps, two rings (embed_pipe.cuh)
    kLdg = 2,   // embed_kernel: rows too wide for a ring, gather warps load them into registers
};

// One launch shape.  plain / add: the P values (lanes per position, bit P) the plan may choose the shape with, without and
// with the additive combine.  They are exactly what the plan can reach for any D and row stride; embed_inst.cu compiles
// those and nothing else, and any other combination counts as not fitting.
struct ShapeRow {
    Family family;
    int nm, nl, ng;  // matcher, loader (pipeline only) and gather warps per CTA
    int minb;        // CTAs per SM
    int budget;      // bytes of shared memory for the rings
    bool stagger;    // the matchers start staggered (EmbedParams::stagger_ns)
    unsigned plain, add;
};

enum ShapeId : int {
    kBulkNarrow6, kBulkNarrow4, kBulkWide, kBulkWide3, kBulkWide2, kBulkMid,
    kPipeNarrow6, kPipeNarrow4, kPipeMid, kPipeWide,
    kRegLoad,
    kNumShapes
};

// Measured on B200: profiles/tune_r01.md and tune_r02.md.  The shape follows the traffic per position ("moved": the stored
// row, or a 2 D fallback row, in and 2 D out).
// Matcher stagger: 400-800 ns per matcher warp is worth 1.5 % on config 2 with the pre-filter (43.3 -> 42.6 us) and 3 %
// without it (46.7 -> 45.3 us); no effect on the wide shapes; below two tiles per matcher the delay would be exposed instead.
constexpr ShapeRow kShapes[kNumShapes] = {
    // ---- single ring (embed_bulk_kernel), the plain path ----
    // kBulkNarrow6: < 6 KB moved, tiny rows; needs >= 6 ring slots
    {kBulk, 6, 0, 4, 3, 70 * 1024, true, 1 | 2 | 4 | 8, 0},
    // kBulkNarrow4: < 6 KB moved, matcher-hungry
    {kBulk, 4, 0, 4, 3, 70 * 1024, true, 1 | 2 | 4 | 8, 0},
    // kBulkWide: >= 6 KB moved, store-hungry
    {kBulk, 6, 0, 12, 1, 200 * 1024, false, 4 | 8, 0},
    // kBulkWide3: wide rows when six slots do not fit
    {kBulk, 3, 0, 12, 1, 200 * 1024, false, 8, 0},
    // kBulkWide2: wide rows when three slots do not fit (two are enough)
    {kBulk, 2, 0, 12, 1, 200 * 1024, false, 8, 0},
    // kBulkMid: narrow rows when the 70 KB shapes do not fit
    {kBulk, 4, 0, 8, 2, 100 * 1024, false, 8, 0},
    // ---- three-role pipeline (embed_pipe_kernel): the row ring only needs two full-size tiles ----
    // kPipeNarrow6: config 2 + wpe: 47 us; + base row: 51 us
    {kPipe, 6, 1, 4, 3, 70 * 1024, true, 1 | 2 | 4 | 8, 4 | 8},
    // kPipeNarrow4: two loaders, the plain path with fp32 rows of 3-4 KB (D 768 / 1024)
    {kPipe, 5, 2, 4, 3, 70 * 1024, true, 1 | 2 | 4 | 8, 0},
    // kPipeMid: 110 KB x 2 CTAs/SM, two full-size tiles of narrow rows + base row + position row (config 2 "both": 56 us
    // against 70 us for the single-ring kernel and 75 us for one 200 KB CTA per SM); fp32 rows of 5-6 KB
    {kPipe, 4, 2, 8, 2, 110 * 1024, false, 1 | 2 | 4 | 8, 4 | 8},
    // kPipeWide: config 3 modes
    {kPipe, 6, 4, 12, 1, 200 * 1024, false, 1 | 2 | 4 | 8, 4 | 8},
    // ---- kRegLoad (embed_kernel, U = 4 steps in flight per lane): rows too wide for a ring ----
    {kLdg, 2, 0, 6, 4, 0, false, 1 | 2 | 4 | 8, 4 | 8},
};

// One call of the fused path, as far as the choice of kernel depends on it.
struct EmbedCall {
    int64_t D, row_stride;
    bool pos;             // position rows are added
    bool additive;        // additive combine: a hit adds its base row
    bool resolved;        // f-gram ids are given (scone_embed_gather): P = 4
    int P;                // lanes per position the vocabulary needs (lanes_per_position), when matching
    const char *pipe_env; // SCONE_EMBED_PIPE, or NULL
    int64_t T;            // positions
    int sms;              // SMs of the device
};

struct EmbedPlan {
    ShapeId row;
    int P;
    bool add;
    BulkLayout bulk;  // kBulk
    PipeLayout pipe;  // kPipe
    int stagger_ns;
    int64_t num_tiles;
    int64_t grid;
    unsigned threads;
    int smem_bytes;
};

// The ring needs at least as many slots as matchers: gather warps release tiles strictly in order, so a matcher that
// has filled tile t - NM knows every tile <= t - NM - ring is consumed; with ring >= NM that covers t - 2 ring, i.e. its
// parity wait on slot t % ring is never more than one phase ahead.
inline bool bulk_layout(int64_t D, int64_t row_stride, int G, int nm, int budget_bytes, BulkLayout &lay) {
    int64_t slot = row_stride > 2 * D ? row_stride : 2 * D;
    slot = (slot + 127) / 128 * 128;
    const int64_t per_tile = slot * G;
    int64_t ring = (budget_bytes - bulk_header_bytes(G)) / per_tile;
    if (ring > kMaxRing) ring = kMaxRing;
    if (ring < 2 || ring < nm) return false;
    lay.ring = (int)ring;
    lay.slot_bytes = (int)slot;
    lay.smem_bytes = bulk_header_bytes(G) + (int)(per_tile * ring);
    return true;
}

// false when not even two tiles of rows fit the budget
inline bool pipe_layout(int64_t D, int64_t row_stride, bool pos, bool additive, int G, int nm, int budget_bytes, PipeLayout &lay) {
    int64_t slot = row_stride > 2 * D ? row_stride : 2 * D;
    slot = (slot + 127) / 128 * 128;
    lay.pos_off = lay.add_off = 0;
    if (additive) {
        lay.add_off = (int)slot;
        slot += (2 * D + 127) / 128 * 128;
    }
    int64_t per_tile = slot * G;
    if (pos) {
        lay.pos_off = (int)per_tile;
        per_tile += (2 * D * G + 127) / 128 * 128;
    }
    if (per_tile > (1 << 20) - 16) return false;  // an mbarrier phase counts at most 2^20 - 1 bytes
    int64_t ring = (budget_bytes - pipe_header_bytes(G)) / per_tile;
    if (ring > kMaxRing) ring = kMaxRing;
    if (ring < 2) return false;
    lay.ring = (int)ring;
    lay.meta_ring = kMaxMetaRing / nm * nm;  // a multiple of NM: a metadata slot is only ever filled by one matcher
    if (lay.meta_ring > 4 * nm) lay.meta_ring = 4 * nm;
    lay.slot_bytes = (int)slot;
    lay.tile_bytes = (int)per_tile;
    lay.smem_bytes = pipe_header_bytes(G) + (int)(per_tile * ring);
    return true;
}

// Plans the call on shape row `row` with P lanes per position; false when the row is not listed for (P, additive) or its
// rings do not fit.
inline bool plan_row(const EmbedCall &c, ShapeId row, int P, EmbedPlan &pl) {
    const ShapeRow &s = kShapes[row];
    if (((c.additive ? s.add : s.plain) & (unsigned)P) == 0) return false;
    const int G = 32 / P;
    pl = EmbedPlan{};
    if (s.family == kBulk && !bulk_layout(c.D, c.row_stride, G, s.nm, s.budget, pl.bulk)) return false;
    if (s.family == kPipe && !pipe_layout(c.D, c.row_stride, c.pos, c.additive, G, s.nm, s.budget, pl.pipe)) return false;
    pl.row = row;
    pl.P = P;
    pl.add = c.additive;
    pl.num_tiles = (c.T + G - 1) / G;
    if (s.stagger && pl.num_tiles >= 2ll * s.nm * s.minb * c.sms) pl.stagger_ns = 500;
    const int64_t resident = (int64_t)c.sms * s.minb;
    pl.grid = pl.num_tiles < resident ? pl.num_tiles : resident;
    pl.threads = 32u * (unsigned)(s.nm + s.nl + s.ng);
    pl.smem_bytes = s.family == kBulk ? pl.bulk.smem_bytes : s.family == kPipe ? pl.pipe.smem_bytes : 0;
    return true;
}

// Two kernels for rows that fit a shared-memory ring (measured, profiles/tune_r02.md): the plain path runs fastest on
// embed_bulk_kernel (one ring, the matcher stages its own tile: fewest hand-offs); with extra rows per position (fused
// position add, additive combine) the three-role pipeline keeps full-size tiles and wins.
// Measured (config 2 / config 3, us per step, single ring vs pipeline): plain 38.4 / 41.5 and 1004 / 1067; + wpe 51.9 /
// 47.0 and 1530 / 1515; + base row 54.2 / 51.4 and 1625 / 1554; both 70.3 / 56.3 and 2383 / 2295.
// Plain path with fp32 rows of 2-6 KB (the reference's own row format at D 768 .. 1536): a position moves twice as many
// bytes in as out, the single ring holds two tiles or fewer for its matchers, and the pipeline wins as well (us per step
// at D 768 / 1024 / 1280 / 1536: 52.9 -> 48.2, 66.4 -> 61.1, 92.2 -> 76.8, 102.2 -> 90.9; FP16 / INT8 / INT4 rows of any
// width and fp32 rows of 8 KB stay 1-4 % faster on the single ring: profiles/tune_r02.md section 17).
// SCONE_EMBED_PIPE=0 / 1 forces one of the two on the plain path.
inline EmbedPlan plan_embed(const EmbedCall &c) {
    const bool extra_rows = c.pos || c.additive;
    int P = c.resolved ? 4 : c.P;
    if (c.additive && P < 4) P = 4;  // additive kernels exist for 4 and 8 lanes per position only
    const bool heavy_rows = c.row_stride > 2 * c.D && c.row_stride > 2048 && c.row_stride <= 6144;
    const bool pipe = extra_rows || (c.pipe_env ? c.pipe_env[0] != '0' : heavy_rows);
    const bool wide = 2 * c.D + c.row_stride >= 6144;
    EmbedPlan pl{};
    if (pipe) {
        // full-size tiles on any shape before smaller tiles: the pipeline's matchers do not depend on the row ring
        static const ShapeId plain[] = {kPipeNarrow4, kPipeNarrow6, kPipeMid, kPipeWide, kNumShapes},
                             narrow[] = {kPipeNarrow6, kPipeMid, kPipeWide, kNumShapes}, wider[] = {kPipeMid, kPipeWide, kNumShapes};
        const ShapeId *order = !extra_rows ? plain : wide ? wider : narrow;
        for (int pp = P; pp <= 8; pp <<= 1)
            for (const ShapeId *s = order; *s != kNumShapes; ++s)
                if (plan_row(c, *s, pp, pl)) return pl;
    } else {
        // a shape that does not fit with P lanes per position is retried with 2P, 4P (fewer positions per tile = smaller
        // ring slots) before the next shape is considered; the 6-matcher narrow shape only at full tile size
        static const ShapeId narrow[] = {kBulkNarrow6, kBulkNarrow4, kBulkMid, kNumShapes}, wider[] = {kBulkWide, kBulkWide3, kBulkWide2, kNumShapes};
        for (const ShapeId *s = wide ? wider : narrow; *s != kNumShapes; ++s)
            for (int pp = P; pp <= (*s == kBulkNarrow6 ? P : 8); pp <<= 1)
                if (plan_row(c, *s, pp, pl)) return pl;
    }
    plan_row(c, kRegLoad, P, pl);
    return pl;
}

}  // namespace scone
