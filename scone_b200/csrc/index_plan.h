// index_plan.h -- the f-gram index's slot formats, and the shape scone_index_create (index.cu) gives an index: which format,
// how many slots, how large the pre-filter.  Plain host-side C++ with no CUDA header and no environment read, so that g++
// compiles it on its own (tests/test_index_plan.py); index_format.cuh holds each format's device side.
#pragma once
#include <cstdint>
#include <cstring>

#include "../../include/scone_b200.h"

namespace scone {

enum SlotFormat : int32_t { kSlotWide = 0, kSlotCompact16 = 1, kSlotCompact20 = 2, kNumSlotFormats };

// A probe step reads one aligned 64-byte block (what a DRAM access fetches anyway) and checks all its slots, 64 / slot_bytes
// of them (derived, not a column); the home slot is the first slot of a block.
constexpr int kProbeStepBytes = 64;

struct SlotFormatRow {
    int slot_bytes;
    int max_n;          // longest f-gram a slot holds
    int64_t tok_limit;  // every token is below it
    int64_t n_limit;    // fewer f-grams than this: every id is below it
    const char *name;   // scone_b200.index.SLOT_FORMATS (tests/test_index_plan.py checks the two agree)
};

constexpr SlotFormatRow kSlotFormats[kNumSlotFormats] = {
    // kSlotWide: 32 bytes = one DRAM sector, id + seven int32 tokens: holds every vocabulary scone_index_create accepts
    {32, SCONE_MAX_N, 1ll << 31, 0x7FFFFFFF, "wide32"},
    // kSlotCompact16: id + six 16-bit tokens (e.g. GPT-2's 50 257 tokens, configs 1-2).  Half the index bytes per f-gram: a
    // 1 M f-gram index is 32 MB at load factor 0.5 and stays resident in the 126 MB L2.
    {16, 6, 0xFFFF, 0x7FFFFFFF, "compact16"},
    // kSlotCompact20: a 28-bit id + five 20-bit tokens, for tokens that do not fit 16 bits (V = 128 000: configs 3-5).  Config
    // 3's index goes from 1.28 GB to 0.64 GB, config 4's from 12.8 to 6.4 GB per GPU.
    {16, 5, 0xFFFFF, 0x0FFFFFFF, "compact20"},
};

// One call of scone_index_create; the entry point has checked n, max_n, the load factor and that no token is negative.
struct IndexCall {
    int64_t n;               // f-grams
    int32_t max_n;
    int32_t max_tok;         // largest token (0 for an empty vocabulary)
    double load_factor;
    const char *format_env;  // SCONE_INDEX_FORMAT, or NULL
    const char *filter_env;  // SCONE_INDEX_FILTER, or NULL
};

struct IndexPlan {
    SlotFormat format;
    uint64_t cap;            // slots: a multiple of 4, so whole probe steps of every format
    uint32_t filter_words;   // 0 = no pre-filter
    bool filter_always;      // consult the filter for every batch size, not only from kFilterMinPositions on
};

// Compact-16 slots if they fit, else compact-20 if they fit, else 32-byte slots.  SCONE_INDEX_FORMAT=wide / prefer-compact20
// force 32-byte slots / compact-20 wherever it fits, so that small test vocabularies run every format (other values: the
// automatic choice); SCONE_INDEX_FILTER=never / always: no filter / one of any size consulted for every batch (testing).
inline IndexPlan plan_index(const IndexCall &c) {
    IndexPlan pl{};
    auto fits = [&](SlotFormat f) {
        const SlotFormatRow &r = kSlotFormats[f];
        return c.max_n <= r.max_n && c.max_tok < r.tok_limit && c.n < r.n_limit;
    };
    const bool fits20 = fits(kSlotCompact20);
    pl.format = fits(kSlotCompact16) ? kSlotCompact16 : fits20 ? kSlotCompact20 : kSlotWide;
    if (c.format_env && !strcmp(c.format_env, "wide")) pl.format = kSlotWide;
    if (c.format_env && !strcmp(c.format_env, "prefer-compact20") && fits20) pl.format = kSlotCompact20;
    // default load factor 0.25 for every format: the probe chain of the slowest of the 32 lanes gates a tile (measured:
    // compact-16 at 0.5 costs config 1 a microsecond of probe chain)
    const double lf = c.load_factor > 0.0 ? c.load_factor : 0.25;
    uint64_t cap = (uint64_t)((double)c.n / lf) + 1;
    if (cap < 64) cap = 64;
    pl.cap = (cap + 3) & ~3ull;
    const bool never = c.filter_env && !strcmp(c.filter_env, "never");
    const bool always = c.filter_env && !strcmp(c.filter_env, "always");
    // pre-filter bits per f-gram: 16 up to 12 M f-grams (24 MB), 8 up to 48 M (~6 % false positives: a 10 M-f-gram filter is
    // 20 MB and still lives in the 126 MB L2 next to the streamed rows), none above: it only pays while it stays in L2
    if (c.n > 0 && !never && (always || c.n <= 48000000ll)) {
        uint64_t words = (uint64_t)(c.n <= 12000000ll ? (c.n + 1) / 2 : (c.n + 3) / 4);
        if (words < 1024) words = 1024;
        pl.filter_words = (uint32_t)((words + 31) & ~31ull);
        pl.filter_always = always;
    }
    return pl;
}

}  // namespace scone
